"""Validation on the device: the corpus-BLEU kernels (dvae_bleu_counts / dvae_bleu_score) against oracle/bleu.py,
losses.compute_bleu, TrainEngine.eval_step / eval_steps (run.py:evalstep) against the oracle's eval-mode forward and the
reference's eval golden vectors, its freedom from side effects on training, the adversarial / MI eval terms,
ConsistencyEvaluator.bleu, and data-parallel evaluation (2 GPUs)."""
import importlib
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from conftest import load_golden, golden_state_dict  # noqa: E402
from oracle import bleu as OB  # noqa: E402
from oracle import dvae_oracle as O  # noqa: E402

pytestmark = pytest.mark.gpu
SOS, EOS, PAD = 2, 3, 0


@pytest.fixture(scope="module")
def dvae():
    import __graft_entry__ as ge
    return ge.build()


@pytest.fixture(scope="module")
def engine_mod(dvae):
    return importlib.import_module("disentanglement-vae_b200.engine")


def _token_rows(rng, B, T, vocab):
    """SOS, ids from a small vocabulary (n-grams repeat, clipping matters), EOS at a random place followed by PAD or junk;
    some rows without EOS, some empty (SOS EOS)."""
    X = rng.integers(4, 4 + vocab, size=(B, T)).astype(np.int64)
    X[:, 0] = SOS
    for b in range(B):
        kind = rng.random()
        if T >= 2 and kind < 0.1:
            X[b, 1] = EOS                      # empty sentence
        elif kind < 0.3:
            continue                           # no EOS: [1:-1] drops the last token
        elif T >= 2:
            e = int(rng.integers(1, T))
            X[b, e] = EOS
            if rng.random() < 0.5:
                X[b, e + 1:] = PAD
    return X


def _check_score(score, want):
    # float64 arithmetic on the device, stored as float32
    assert abs(float(score) - float(np.float32(want))) <= 1e-12 * max(abs(want), 1e-30), (float(score), want)


# ---- 1. the kernels against the oracle ----------------------------------------------------------------------------
@pytest.mark.parametrize("B", [1, 37, 1024])
@pytest.mark.parametrize("T_ref,T_cand", [(2, 2), (9, 9), (22, 22), (64, 64), (22, 30), (64, 9)])
def test_bleu_kernels_match_oracle(dvae, B, T_ref, T_cand):
    rng = np.random.default_rng(B * 1000 + T_ref * 10 + T_cand)
    vocab = int(rng.integers(6, 21))
    ref = _token_rows(rng, B, T_ref, vocab)
    cand = _token_rows(rng, B, T_cand, vocab)
    if T_ref == T_cand:      # half the candidates copy their reference with a few edits: non-trivial precisions
        for b in range(0, B, 2):
            cand[b] = ref[b]
            cand[b, rng.integers(1, T_cand, size=2)] = rng.integers(4, 4 + vocab, size=2)
    want = OB.bleu_counts(ref, cand, EOS)
    dev = torch.device("cuda")
    r, c = torch.from_numpy(ref).to(dev), torch.from_numpy(cand).to(dev)
    counts = torch.zeros(10, device=dev, dtype=torch.int64)
    score = torch.empty(1, device=dev)
    dvae.losses.bleu_counts_(counts, r, c, EOS)
    dvae.losses.bleu_score_(score, counts)
    assert counts.tolist() == want
    _check_score(score.item(), OB.bleu_from_counts(want))
    # the counters only add: two calls on the halves give the statistics of the whole batch
    if B > 1:
        acc = torch.zeros(10, device=dev, dtype=torch.int64)
        h = B // 2
        dvae.losses.bleu_counts_(acc, r[:h], c[:h], EOS)
        dvae.losses.bleu_counts_(acc, r[h:], c[h:], EOS)
        assert acc.tolist() == want


def test_bleu_kernel_rejects_rows_longer_than_the_limit(dvae):
    x = torch.full((2, 257), 5, device="cuda", dtype=torch.int64)
    counts = torch.zeros(10, device="cuda", dtype=torch.int64)
    with pytest.raises(dvae._lib.DvaeError):
        dvae.losses.bleu_counts_(counts, x, x, EOS)
    dvae.losses.bleu_counts_(counts, x[:, :256], x[:, :256], EOS)      # the limit itself is accepted
    assert counts.tolist()[8] == 2 * 254


# ---- 2. losses.compute_bleu ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("where", ["host", "device"])
def test_compute_bleu_equals_oracle(dvae, where):
    rng = np.random.default_rng(7)
    ref = _token_rows(rng, 50, 12, 8)
    cand = ref.copy()
    cand[:, 3] = rng.integers(4, 12, size=50)
    want = OB.corpus_bleu(ref, cand, EOS)
    assert 0.0 < want < 1.0
    X, P = torch.from_numpy(ref), torch.from_numpy(cand)
    if where == "device":
        X, P = X.cuda(), P.cuda()
    _check_score(dvae.losses.compute_bleu(X, P, None, EOS), want)


# ---- 3 / 4. eval_step against the oracle ----------------------------------------------------------------------------
def _cfg(**over):
    c = dict(bow_encoder=False, embedding_dim=64, hidden_dim=64, num_rnn_layers=2, encoder_dropout=0.5, decoder_dropout=0.5,
             bidirectional_encoder=True, latent_dims={"total": 16, "polarity": 1, "uncertainty": 1}, adversarial_loss=False,
             mi_loss=False, learn_rate=3e-3, lambdas={"default": "cyclic", "polarity": 0.005, "uncertainty": 0.005},
             random_seed=10, teacher_forcing_prob=1.0)
    c.update(over)
    return c


def _batch(gen, B, T, V, names=("uncertainty", "polarity")):
    lengths = torch.randint(3, T + 1, (B,), generator=gen)
    lengths[0] = T
    X = torch.zeros(B, T, dtype=torch.long)
    for b in range(B):
        n = int(lengths[b])
        X[b, 0], X[b, n - 1] = SOS, EOS
        X[b, 1:n - 1] = torch.randint(4, V, (n - 2,), generator=gen)
    Y = {k: (torch.rand(B, 1, generator=gen) < 0.3).float() for k in names}
    return X, lengths, Y


def _oracle_eval(vae, eng, X, L, Y, dec_inputs=None):
    sd = O.cast_state_dict({k: v.detach().cpu().numpy() for k, v in vae.state_dict().items()})
    spec = O.ModelSpec(sd, list(vae.context2params.keys()), 2, 3)
    eps = eng.plan.eps.detach().cpu().numpy()
    eps_d, off = {}, 0
    for n, zs in zip(spec.space_names, spec.space_dims):
        eps_d[n] = eps[:, off:off + zs]
        off += zs
    klw = {"default": 1.0, "polarity": 0.005, "uncertainty": 0.005}       # "cyclic" -> 1.0 in evaluation
    return O.model_forward(sd, spec, X.numpy(), L.numpy(), eps_d, labels={k: y.numpy() for k, y in Y.items()},
                           kl_weights=klw, dec_inputs=dec_inputs)


@pytest.mark.parametrize("use_graph", [True, False])
def test_eval_step_forced_matches_oracle_eval_forward(dvae, engine_mod, use_graph):
    V, B, T = 400, 20, 10
    dev = torch.device("cuda")
    dvae.set_seed(10)
    vae = dvae.build_vae(_cfg(), V, None, {"uncertainty": 1, "polarity": 1}, dev, SOS, EOS)
    vae.train()
    eng = engine_mod.TrainEngine(vae, _cfg(), B, T, total_steps=40, use_graph=use_graph, seed=5)
    gen = torch.Generator().manual_seed(11)
    eng.step_host(*_batch(gen, B, T, V))            # one training step first: evaluation of trained weights
    for _ in range(2):
        X, L, Y = _batch(gen, B, T, V)
        got = eng.eval_step(X, L, Y, teacher_forcing_prob=1.0)
        fw = _oracle_eval(vae, eng, X, L, Y)
        assert abs(got["total_loss"] - fw["total_loss"]) <= 1e-5 * abs(fw["total_loss"]), (got["total_loss"], fw["total_loss"])
        assert abs(got["reconstruction_loss"] - fw["reconstruction_loss"]) <= 1e-5 * abs(fw["reconstruction_loss"])
        for n, kl in fw["kls"].items():
            assert abs(got["idv_kls"][n] - kl) <= 1e-3 * abs(kl) + 1e-7, n
        for n, dl in fw["dsc_losses"].items():
            assert abs(got["idv_dsc_losses"][n] - dl) <= 1e-5 * abs(dl) + 1e-7, n
        preds = eng.eval_predictions.cpu().numpy()
        assert (preds[:, 0] == SOS).all() and np.array_equal(preds[:, 1:], X.numpy()[:, 1:])
        assert got["bleu"] == 1.0
        assert got["bleu_counts"] == OB.bleu_counts(X.numpy(), preds, EOS)
        want_z = np.concatenate([fw["latent"][n]["z"] for n in vae.context2params.keys()], axis=1)
        assert np.abs(eng.plan.z.cpu().numpy() - want_z).max() <= 1e-4 * max(np.abs(want_z).max(), 1.0)   # dev latents
    assert eng.adam_step == 1 and eng.step_idx == 1


def test_eval_step_on_reference_eval_golden(dvae, engine_mod):
    """tiny_eval_mc: the reference's own eval-mode forward (3-class discriminator, H = 8) through the engine, eps replayed."""
    g = load_golden("tiny_eval_mc")
    sd = golden_state_dict(g)
    names = [str(s) for s in g["space_names"]]
    dims = [int(x) for x in g["space_dims"]]
    lat = {"total": sum(dims)}
    for n, zs in zip(names, dims):
        if n != "content":
            lat[n] = zs
    label_dims = {str(n): int(d) for n, d in zip(g["label_names"], g["label_dims"])}
    Le = 1 + max(int(k.split("_l")[1][0]) for k in sd if k.startswith("encoder.recurrent.weight_hh_l"))
    p = _cfg(embedding_dim=sd["encoder.embedding.weight"].shape[1], hidden_dim=sd["decoder.recurrent.weight_hh_l0"].shape[1],
             num_rnn_layers=Le, bidirectional_encoder="encoder.recurrent.weight_ih_l0_reverse" in sd, latent_dims=lat,
             lambdas={"default": "cyclic"})
    dev = torch.device("cuda")
    vae = dvae.build_vae(p, int(g["V"]), None, label_dims, dev, int(g["sos"]), int(g["eos"]))
    vae.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    X, lengths = torch.from_numpy(g["inputs"]), torch.from_numpy(g["lengths"])
    B, T = X.shape
    eng = engine_mod.TrainEngine(vae, p, B, T, total_steps=10, seed=1)
    eng.fixed_eps = torch.from_numpy(np.concatenate([g[f"eps.{n}"] for n in names], axis=1)).to(dev)
    Y = {n: torch.from_numpy(g[f"Y.{n}"]) for n in label_dims}
    got = eng.eval_step(X, lengths, Y, teacher_forcing_prob=1.0)
    assert abs(got["total_loss"] - float(g["loss.total"])) <= 1e-5 * abs(float(g["loss.total"]))
    assert abs(got["reconstruction_loss"] - float(g["loss.reconstruction"])) <= 1e-5 * float(g["loss.reconstruction"])
    for n in names:
        assert abs(got["idv_kls"][n] - float(g[f"kl.{n}"])) <= 1e-3 * float(g[f"kl.{n}"])
    for n in label_dims:
        assert abs(got["idv_dsc_losses"][n] - float(g[f"dsc_loss.{n}"])) < 1e-5
        assert abs(got["idv_dsc_accs"][n] - float(g[f"dsc_acc.{n}"])) < 1e-6
    assert got["bleu"] == pytest.approx(OB.corpus_bleu(g["inputs"], g["token_predictions"], int(g["eos"])), abs=1e-7)


@pytest.mark.parametrize("tf", [0.0, 0.5])
@pytest.mark.parametrize("use_graph", [True, False])
def test_eval_step_sampled_matches_oracle_on_sampled_tokens(dvae, engine_mod, tf, use_graph):
    V, B, T = 60, 24, 10          # a small vocabulary: sampled sentences share n-grams with the inputs
    dev = torch.device("cuda")
    dvae.set_seed(10)
    vae = dvae.build_vae(_cfg(), V, None, {"uncertainty": 1, "polarity": 1}, dev, SOS, EOS)
    vae.train()
    eng = engine_mod.TrainEngine(vae, _cfg(), B, T, total_steps=40, use_graph=use_graph, seed=5)
    gen = torch.Generator().manual_seed(12)
    sampled_steps = 0
    for _ in range(3):
        X, L, Y = _batch(gen, B, T, V)
        got = eng.eval_step(X, L, Y, teacher_forcing_prob=tf)
        preds = eng.eval_predictions.cpu().numpy()
        coins = eng.coins.cpu().numpy()
        assert (preds[:, 0] == SOS).all()
        for i in range(1, T):
            if coins[i - 1]:
                assert np.array_equal(preds[:, i], X[:, i].numpy())
            else:
                sampled_steps += 1
        if tf == 0.0:
            assert not coins[:T - 1].any()
        fw = _oracle_eval(vae, eng, X, L, Y, dec_inputs=preds[:, :T - 1])
        assert abs(got["reconstruction_loss"] - fw["reconstruction_loss"]) <= 1e-5 * abs(fw["reconstruction_loss"])
        assert abs(got["total_loss"] - fw["total_loss"]) <= 1e-5 * abs(fw["total_loss"])
        want = OB.bleu_counts(X.numpy(), preds, EOS)
        assert got["bleu_counts"] == want
        _check_score(got["bleu"], OB.bleu_from_counts(want))
    assert sampled_steps > 0
    assert eng.adam_step == 0 and eng.step_idx == 0


def test_eval_steps_pipelined_equal_eval_step(dvae, engine_mod):
    V, B, T = 300, 16, 9
    dev = torch.device("cuda")
    gen = torch.Generator().manual_seed(21)
    batches = [_batch(gen, B, T, V) for _ in range(5)]
    runs = []
    for mode in ("sync", "pipe"):
        dvae.set_seed(10)
        vae = dvae.build_vae(_cfg(), V, None, {"uncertainty": 1, "polarity": 1}, dev, SOS, EOS)
        eng = engine_mod.TrainEngine(vae, _cfg(), B, T, total_steps=40, seed=5)
        if mode == "sync":
            runs.append([eng.eval_step(*b, teacher_forcing_prob=0.5) for b in batches])
        else:
            runs.append(list(eng.eval_steps(iter(batches), teacher_forcing_prob=0.5)))
    for a, b in zip(*runs):
        assert a["bleu_counts"] == b["bleu_counts"]
        assert abs(a["total_loss"] - b["total_loss"]) <= 1e-5 * abs(a["total_loss"])
    total = np.sum([r["bleu_counts"] for r in runs[1]], axis=0).tolist()
    _check_score(dvae.losses.bleu_from_counts(total), OB.bleu_from_counts(total))


# ---- 5. no side effects on training ------------------------------------------------------------------------------------
def _train_run(dvae, engine_mod, batches, evals, V=500, B=24, T=9):
    dvae.set_seed(10)
    vae = dvae.build_vae(_cfg(), V, None, {"uncertainty": 1, "polarity": 1}, torch.device("cuda"), SOS, EOS)
    vae.train()
    eng = engine_mod.TrainEngine(vae, _cfg(), B, T, total_steps=40, use_graph=True, seed=5)
    losses = []
    for k, b in enumerate(batches):
        if k == 2 and evals:
            before = (vae._flat.clone(), eng.m.clone(), eng.v.clone(), eng.grad.clone(), eng.step_idx, eng.adam_step,
                      eng._gen.get_state().clone(), eng._pyrand.getstate())
            for X, L, Y, tf in evals:
                eng.eval_step(X, L, Y, teacher_forcing_prob=tf)
            torch.cuda.synchronize()
            after = (vae._flat, eng.m, eng.v, eng.grad, eng.step_idx, eng.adam_step, eng._gen.get_state(), eng._pyrand.getstate())
            for x, y in zip(before, after):      # parameters, moments, gradient buffer, counters, training streams
                assert (torch.equal(x, y) if torch.is_tensor(x) else x == y)
        losses.append(eng.step_host(*b)["total_loss"])
    return losses, vae._flat.detach().clone(), eng.m.clone(), eng.v.clone()


def test_eval_between_training_steps_changes_nothing(dvae, engine_mod):
    """train 2 -> eval (tf 1 and 0.5, dropout 0.5 in the config) -> train 2 against train 4 under the same seed.  The eval
    calls leave parameters, Adam moments, gradient buffer, step counters and the training random streams bit-identical.
    The four-step runs are then compared bit for bit when two plain four-step runs agree bit for bit; otherwise (atomics
    in the backward pass order their sums differently from run to run) within that run-to-run difference."""
    V, B, T = 500, 24, 9
    gen = torch.Generator().manual_seed(31)
    batches = [_batch(gen, B, T, V) for _ in range(4)]
    evals = [(*_batch(gen, B, T, V), 1.0), (*_batch(gen, B, T, V), 0.5)]
    ref = _train_run(dvae, engine_mod, batches, [])
    ref2 = _train_run(dvae, engine_mod, batches, [])
    got = _train_run(dvae, engine_mod, batches, evals)
    deterministic = ref[0] == ref2[0] and all(torch.equal(a, b) for a, b in zip(ref[1:], ref2[1:]))
    if deterministic:
        assert got[0] == ref[0]
        for a, b in zip(got[1:], ref[1:]):
            assert torch.equal(a, b)
    else:
        noise = max(abs(x - y) for x, y in zip(ref[0], ref2[0]))
        for x, y in zip(got[0], ref[0]):
            assert abs(x - y) <= max(4 * noise, 1e-4 * abs(y)), (got[0], ref[0], ref2[0])
        w0 = _train_run(dvae, engine_mod, [], [])[1]
        assert (got[1] - ref[1]).abs().mean().item() < 0.02 * (ref[1] - w0).abs().mean().item()


# ---- 6. adversarial / MI models --------------------------------------------------------------------------------------
def test_eval_step_aux_terms_equal_the_drop_in_functions(dvae, engine_mod):
    g = load_golden("tiny_adv_mi")
    sd = golden_state_dict(g)
    names = [str(s) for s in g["space_names"]]
    dims = [int(x) for x in g["space_dims"]]
    label_dims = {str(n): int(d) for n, d in zip(g["label_names"], g["label_dims"])}
    lat = {"total": sum(dims)}
    for n, zs in zip(names, dims):
        if n != "content":
            lat[n] = zs
    p = _cfg(embedding_dim=sd["encoder.embedding.weight"].shape[1], hidden_dim=sd["decoder.recurrent.weight_hh_l0"].shape[1],
             latent_dims=lat, adversarial_loss=True, mi_loss=True, lambdas={"default": "cyclic"})
    dev = torch.device("cuda")
    vae = dvae.build_vae(p, int(g["V"]), None, label_dims, dev, int(g["sos"]), int(g["eos"]))
    vae.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    X, lengths = torch.from_numpy(g["inputs"]), torch.from_numpy(g["lengths"])
    B, T = X.shape
    eng = engine_mod.TrainEngine(vae, p, B, T, total_steps=10, seed=1)
    Y = {n: torch.from_numpy(g[f"Y.{n}"]) for n in label_dims}
    got = eng.eval_step(X, lengths, Y, teacher_forcing_prob=1.0)
    from importlib import import_module
    F = import_module("disentanglement-vae_b200.functions")
    with torch.no_grad():
        latp = eng._latents(eng.plan.z.clone())
        Yd = {n: Y[n].to(dev).float() for n in label_dims}
        A = dvae.losses.compute_adversarial_losses(vae, F.adversary_logits(vae, latp), Yd)
        M = dvae.losses.compute_mi_losses(vae, latp, beta=0.01)
    assert got["total_adv_loss"] == pytest.approx(float(A["total_adv_loss"]), rel=1e-6)
    assert got["total_mi"] == pytest.approx(float(M["total_mi"]), rel=1e-6, abs=1e-9)
    assert got["idv_adv_losses"] == pytest.approx(A["idv_adv_losses"], rel=1e-6)
    assert got["idv_mi_estimates"] == pytest.approx(M["idv_mi_estimates"], rel=1e-6, abs=1e-9)
    base = got["reconstruction_loss"] + got["total_weighted_kl"] + got["total_dsc_loss"]
    assert got["total_loss"] == pytest.approx(base + got["total_adv_loss"] + got["total_mi"], rel=1e-6)
    assert eng.adam_step == 0 and not eng.last_aux


# ---- 7. ConsistencyEvaluator.bleu ------------------------------------------------------------------------------------
@pytest.mark.parametrize("use_graph", [True, False])
def test_consistency_bleu_per_resample_equals_oracle(dvae, use_graph):
    inference = importlib.import_module("disentanglement-vae_b200.inference")
    V, B, T, R = 40, 32, 10, 4
    dev = torch.device("cuda")
    dvae.set_seed(10)
    vae = dvae.build_vae(_cfg(encoder_dropout=0.0, decoder_dropout=0.0), V, None, {"uncertainty": 1, "polarity": 1}, dev, SOS, EOS)
    vae.eval()
    X, L, _ = _batch(torch.Generator().manual_seed(5), B, T, V)
    ev = inference.ConsistencyEvaluator(vae, B, T, use_graph=use_graph, seed=3)
    ev.encode_once(X, L)
    out = ev.resample(R)
    got = ev.bleu(out).cpu().numpy()
    tok = out["token_predictions"].cpu().numpy()
    assert got.shape == (R,)
    for r in range(R):
        _check_score(got[r], OB.corpus_bleu(X.numpy(), tok[r], EOS))
    ev2 = inference.ConsistencyEvaluator(vae, B, T, use_graph=use_graph, keep_tokens=False)
    ev2.encode_once(X, L)
    with pytest.raises(dvae._lib.DvaeError):
        ev2.bleu(ev2.resample(1))


# ---- 8. data-parallel evaluation ---------------------------------------------------------------------------------------
def test_data_parallel_eval_equals_one_engine_on_the_global_batch(tmp_path):
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from test_gpu_dp import _torchrun
    out = tmp_path / "eval_dp.npz"
    r = _torchrun(2, "eval_dp_worker.py", out)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    got = np.load(out)
    import eval_dp_worker as W
    one = W.run(1, 0, torch.device("cuda", 0))
    for k in ("total_loss", "reconstruction_loss", "total_kl", "total_dsc_loss"):
        assert abs(float(got[k]) - one["forced"][k]) <= 1e-5 * abs(one["forced"][k]), k
    assert float(got["bleu_forced"]) == 1.0
    # sampled decode: each rank samples its own tokens; the summed counts are those of the gathered rows
    want = OB.bleu_counts(got["inputs"], got["preds"], EOS)
    assert got["counts_sampled"].tolist() == want
    _check_score(float(got["bleu_sampled"]), OB.bleu_from_counts(want))
