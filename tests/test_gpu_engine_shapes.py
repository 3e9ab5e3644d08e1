"""TrainEngine on batches smaller than its shape: a shorter padded length T' < T (padded with PAD columns on the host),
a short batch B' < B (a cached StepPlan / graph of its own), both together, through training, evaluation, the
adversarial / MI step and data parallel; the device BLEU row bound (dvae_bleu_counts_ex); and the errors for batches
the engine cannot take."""
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
SOS, EOS = 2, 3
NAMES = ("uncertainty", "polarity")


@pytest.fixture(scope="module")
def dvae():
    import __graft_entry__ as ge
    return ge.build()


@pytest.fixture(scope="module")
def engine_mod(dvae):
    return importlib.import_module("disentanglement-vae_b200.engine")


def _cfg(**over):
    c = dict(bow_encoder=False, embedding_dim=256, hidden_dim=256, num_rnn_layers=2, encoder_dropout=0.0, decoder_dropout=0.0,
             bidirectional_encoder=True, latent_dims={"total": 16, "polarity": 1, "uncertainty": 1}, adversarial_loss=False,
             mi_loss=False, learn_rate=3e-3, lambdas={"default": "cyclic", "polarity": 0.005, "uncertainty": 0.005},
             random_seed=10, teacher_forcing_prob=1.0)
    c.update(over)
    return c


def _batch(gen, B, T, V, no_eos=0):
    """[B, T] batch padded to its own longest row (row 0 has length T); the last `no_eos` rows end without EOS."""
    lengths = torch.randint(3, T + 1, (B,), generator=gen)
    lengths[0] = T
    X = torch.zeros(B, T, dtype=torch.long)
    for b in range(B):
        n = int(lengths[b])
        X[b, 0], X[b, n - 1] = SOS, EOS
        X[b, 1:n - 1] = torch.randint(4, V, (n - 2,), generator=gen)
        if b >= B - no_eos:
            X[b, n - 1] = 4
    Y = {k: (torch.rand(B, 1, generator=gen) < 0.3).float() for k in NAMES}
    return X, lengths, Y


def _model(dvae, cfg, V):
    dvae.set_seed(10)
    vae = dvae.build_vae(cfg, V, None, {"uncertainty": 1, "polarity": 1}, torch.device("cuda"), SOS, EOS)
    vae.train()
    return vae


def _updates_agree(got, want, w0):
    """DESIGN §2's gate for two runs of the same steps: updates within 2e-3 of the largest update (Adam turns noise-level
    gradients into +-lr moves, so a few entries may differ), and in the mean within 1e-3."""
    upd_got, upd_want = got - w0, want - w0
    scale = upd_want.abs().max()
    frac_bad = ((upd_got - upd_want).abs() > 2e-3 * scale).float().mean().item()
    assert frac_bad < 2e-3, frac_bad
    assert (upd_got - upd_want).abs().mean().item() < 1e-3 * upd_want.abs().mean().item()


def _dropin_step(dvae, vae, opt, X, L, Y, eps, klw):
    """run.py:217-262 through the drop-in module: forward, compute_all_losses, backward, clip 5.0, Adam."""
    dev = torch.device("cuda")
    out = vae(X.to(dev), L.to(dev), teacher_forcing_prob=1.0, eps=eps)
    total, _ = dvae.losses.compute_all_losses(vae, out, X.to(dev), Y, L.to(dev), klw)
    total.backward()
    torch.nn.utils.clip_grad_norm_(vae.trainable_parameters(), 5.0)
    opt.step()
    opt.zero_grad()
    return float(total.detach())


def _klw(dvae, step, total):
    return {"default": dvae.losses.get_cyclic_kl_weight(step, total), "polarity": 0.005, "uncertainty": 0.005}


# ---- 1. T' < T is exact -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tf", [1.0, 0.5])
def test_narrow_batches_equal_an_engine_built_at_their_length(dvae, engine_mod, tf):
    V, B, T, Tn, total = 2000, 24, 14, 9, 40
    cfg = _cfg(teacher_forcing_prob=tf)
    gen = torch.Generator().manual_seed(5)
    batches = [_batch(gen, B, Tn, V) for _ in range(3)]
    runs = []
    for T_eng in (T, Tn):
        vae = _model(dvae, cfg, V)
        w0 = vae._flat.detach().clone()
        eng = engine_mod.TrainEngine(vae, cfg, B, T_eng, total_steps=total, seed=3)
        losses, coins, preds, eps = [], [], [], []
        for X, L, Y in batches:
            losses.append(eng.step_host(X, L, Y))
            coins.append(eng.coins[:Tn - 1].cpu().clone())
            preds.append(eng.token_predictions.cpu().clone())
            eps.append(eng.plan.eps.cpu().clone())
        runs.append((losses, coins, preds, eps, vae._flat.detach().clone(), w0, eng))
    (la, ca, pa, ea, wa, w0, eng_a), (lb, cb, pb, eb, wb, _, _) = runs
    assert eng_a.inputs.shape == (B, T) and pa[0].shape == (B, Tn)
    for s in range(3):
        assert torch.equal(ea[s], eb[s])
        assert torch.equal(ca[s], cb[s]) and torch.equal(pa[s], pb[s]), s
        for k in ("total_loss", "reconstruction_loss", "total_kl", "total_dsc_loss"):
            assert abs(la[s][k] - lb[s][k]) <= 1e-5 * abs(lb[s][k]) + 1e-9, (s, k, la[s][k], lb[s][k])
    if tf < 1.0:
        assert any(not c.all() for c in ca)
        assert bool((eng_a.coins[Tn - 1:] == 1).all())       # steps past the batch's length: forced
    _updates_agree(wa, wb, w0)


# ---- 2. B' < B against the drop-in path ----------------------------------------------------------------------------
def test_short_batches_match_the_drop_in_path_and_reuse_their_graphs(dvae, engine_mod):
    V, B, T, total, lr = 2000, 40, 12, 50, 3e-3
    cfg = _cfg(learn_rate=lr)
    gen = torch.Generator().manual_seed(8)
    shapes = [(B, T), (13, 9), (B, T), (13, 12), (1, 7)]
    batches = [_batch(gen, b, t, V) for b, t in shapes]
    eps_all = torch.randn(B, 16, generator=gen).cuda()
    vae = _model(dvae, cfg, V)
    w0 = vae._flat.detach().clone()
    eng = engine_mod.TrainEngine(vae, cfg, B, T, total_steps=total, seed=3)
    eng.fixed_eps = eps_all            # a B' step reads its first B' rows
    ref = _model(dvae, cfg, V)
    opt = torch.optim.Adam(ref.trainable_parameters(), lr=lr)
    seen = {}
    for step, (X, L, Y) in enumerate(batches):
        got = eng.step_host(X, L, Y)["total_loss"]
        want = _dropin_step(dvae, ref, opt, X, L, Y, eps_all[:X.shape[0]], _klw(dvae, step, total))
        assert abs(got - want) <= 1e-5 * abs(want), (step, got, want)
        assert eng.plan.B == X.shape[0] and eng.plan.z.shape[0] == X.shape[0]
        sh = eng._sh
        if sh.B in seen:               # the second batch of a shape replays the graph its first one captured
            assert sh is seen[sh.B][0] and sh.graphs is seen[sh.B][1]
        seen[sh.B] = (sh, sh.graphs)
        _updates_agree(vae._flat.detach(), ref._flat.detach()[:vae._flat.numel()], w0)
    assert eng.adam_step == len(batches)
    # after a full-shape step the public views are the full shape's again
    eng.step_host(*_batch(gen, B, T, V))
    assert eng.plan is eng._full.plan and eng.inputs.shape == (B, T) and eng.lengths.shape == (B,)


def test_one_row_batch_trains_on_that_row(dvae, engine_mod):
    """B' = 1 used to broadcast into all B rows; the engine must take the step of the one-row batch, i.e. what an engine
    built for one row takes."""
    V, B, T, total = 2000, 16, 10, 20
    cfg = _cfg()
    X, L, Y = _batch(torch.Generator().manual_seed(2), 1, T, V)
    eps = torch.randn(1, 16, generator=torch.Generator().manual_seed(4)).cuda()
    out = []
    for B_eng in (B, 1):
        vae = _model(dvae, cfg, V)
        w0 = vae._flat.detach().clone()
        eng = engine_mod.TrainEngine(vae, cfg, B_eng, T, total_steps=total, seed=3)
        eng.fixed_eps = eps
        out.append((eng.step_host(X, L, Y)["total_loss"], vae._flat.detach().clone(), w0))
    (la, wa, w0), (lb, wb, _) = out
    assert abs(la - lb) <= 1e-5 * abs(lb)
    _updates_agree(wa, wb, w0)


# ---- 3. one epoch through RatioSampler ---------------------------------------------------------------------------
def test_ratio_sampler_epoch_through_train_steps_matches_the_drop_in_path(dvae, engine_mod):
    data = importlib.import_module("disentanglement-vae_b200.data")
    V, B, Tmax, total, lr = 2000, 16, 14, 30, 3e-3
    gen = torch.Generator().manual_seed(21)
    rows = []
    for i in range(37 + 21):                 # two sources, 37 and 21 rows: groups of 8, the last group ragged
        long_row = i % 13 == 0               # a few long rows: batch widths differ
        n = int(torch.randint(9, Tmax + 1, (1,), generator=gen)) if long_row else int(torch.randint(3, 9, (1,), generator=gen))
        toks = [SOS] + torch.randint(4, V, (n - 2,), generator=gen).tolist() + [EOS]
        rows.append({"source": "a" if i < 37 else "b", "toks": toks,
                     "y": {k: float(torch.rand(1, generator=gen) < 0.3) for k in NAMES}})
    sampler = data.RatioSampler(rows, "source", batch_size=B, generator=torch.Generator().manual_seed(1))

    def collate(idx):                        # pad_sequence_denoising: each batch to its own longest row
        rs = [rows[int(i)] for i in idx]
        T = max(len(r["toks"]) for r in rs)
        X = torch.zeros(len(rs), T, dtype=torch.long)
        for j, r in enumerate(rs):
            X[j, :len(r["toks"])] = torch.tensor(r["toks"])
        L = torch.tensor([len(r["toks"]) for r in rs])
        return X, L, {k: torch.tensor([[r["y"][k]] for r in rs]) for k in NAMES}
    batches = [collate(idx) for idx in sampler]
    assert batches[-1][0].shape[0] < B and len({b[0].shape[1] for b in batches}) > 1
    cfg = _cfg(learn_rate=lr)
    eps_all = torch.randn(B, 16, generator=gen).cuda()
    vae = _model(dvae, cfg, V)
    eng = engine_mod.TrainEngine(vae, cfg, B, Tmax, total_steps=total, seed=3)
    eng.fixed_eps = eps_all
    got = [L["total_loss"] for L in eng.train_steps(iter(batches))]
    ref = _model(dvae, cfg, V)
    opt = torch.optim.Adam(ref.trainable_parameters(), lr=lr)
    want = [_dropin_step(dvae, ref, opt, X, L, Y, eps_all[:X.shape[0]], _klw(dvae, s, total)) for s, (X, L, Y) in enumerate(batches)]
    assert len(got) == len(batches) == eng.adam_step
    for s, (a, b) in enumerate(zip(got, want)):
        assert abs(a - b) <= 1e-5 * abs(b), (s, got, want)


# ---- 4. evaluation ---------------------------------------------------------------------------------------------------
def _oracle_eval(vae, eng, X, L, Y, dec_inputs=None):
    sd = O.cast_state_dict({k: v.detach().cpu().numpy() for k, v in vae.state_dict().items()})
    spec = O.ModelSpec(sd, list(vae.context2params.keys()), SOS, EOS)
    eps = eng.plan.eps.detach().cpu().numpy()
    eps_d, off = {}, 0
    for n, zs in zip(spec.space_names, spec.space_dims):
        eps_d[n] = eps[:, off:off + zs]
        off += zs
    klw = {"default": 1.0, "polarity": 0.005, "uncertainty": 0.005}
    return O.model_forward(sd, spec, X.numpy(), L.numpy(), eps_d, labels={k: y.numpy() for k, y in Y.items()},
                           kl_weights=klw, dec_inputs=dec_inputs)


@pytest.mark.parametrize("tf", [1.0, 0.0])
def test_eval_step_on_short_narrow_batches_matches_oracle_and_bleu(dvae, engine_mod, tf):
    V, B, T = 60, 24, 14                     # a small vocabulary: sampled sentences share n-grams with the inputs
    cfg = _cfg(embedding_dim=64, hidden_dim=64)
    vae = _model(dvae, cfg, V)
    eng = engine_mod.TrainEngine(vae, cfg, B, T, total_steps=40, seed=5)
    gen = torch.Generator().manual_seed(12)
    for Bs, Ts in ((B, T), (11, 9), (11, 6), (B, 10)):
        X, L, Y = _batch(gen, Bs, Ts, V, no_eos=3)
        got = eng.eval_step(X, L, Y, teacher_forcing_prob=tf)
        preds = eng.eval_predictions.cpu().numpy()
        assert preds.shape == (Bs, Ts) and (preds[:, 0] == SOS).all()
        if tf == 1.0:
            assert np.array_equal(preds[:, 1:], X.numpy()[:, 1:])
        fw = _oracle_eval(vae, eng, X, L, Y, dec_inputs=None if tf == 1.0 else preds[:, :Ts - 1])
        assert abs(got["reconstruction_loss"] - fw["reconstruction_loss"]) <= 1e-5 * abs(fw["reconstruction_loss"])
        assert abs(got["total_loss"] - fw["total_loss"]) <= 1e-5 * abs(fw["total_loss"]), (Bs, Ts)
        assert got["bleu_counts"] == OB.bleu_counts(X.numpy(), preds, EOS), (Bs, Ts)
    assert eng.adam_step == 0 and len(eng._sh.eval["graphs"]) == 1


@pytest.mark.parametrize("t_max", [1, 2, 9, 17, 30, 40])
def test_bleu_counts_ex_bounds_rows_at_the_device_length(dvae, t_max):
    rng = np.random.default_rng(t_max)
    B, T = 77, 30
    ref = rng.integers(4, 12, size=(B, T)).astype(np.int64)
    ref[:, 0] = SOS
    for b in range(0, B, 3):                 # a third of the rows end (EOS, then PAD), the rest have no EOS
        e = int(rng.integers(1, T))
        ref[b, e], ref[b, e + 1:] = EOS, 0
    cand = ref.copy()
    cand[:, 5] = rng.integers(4, 12, size=B)
    dev = torch.device("cuda")
    counts = torch.zeros(10, device=dev, dtype=torch.int64)
    dvae.losses.bleu_counts_(counts, torch.from_numpy(ref).to(dev), torch.from_numpy(cand).to(dev), EOS,
                             t_max=torch.tensor([t_max], dtype=torch.int32, device=dev))
    k = min(t_max, T)
    assert counts.tolist() == OB.bleu_counts(ref[:, :k], cand[:, :k], EOS)


# ---- 5. adversarial / MI ---------------------------------------------------------------------------------------------
def test_adversarial_mi_short_narrow_step_equals_an_engine_of_that_shape(dvae, engine_mod):
    g = load_golden("tiny_adv_mi")
    sd = golden_state_dict(g)
    names = [str(s) for s in g["space_names"]]
    dims = [int(x) for x in g["space_dims"]]
    label_dims = {str(n): int(d) for n, d in zip(g["label_names"], g["label_dims"])}
    lat = {"total": sum(dims)}
    for n, zs in zip(names, dims):
        if n != "content":
            lat[n] = zs
    p = dict(bow_encoder=False, embedding_dim=sd["encoder.embedding.weight"].shape[1],
             hidden_dim=sd["decoder.recurrent.weight_hh_l0"].shape[1], num_rnn_layers=2, encoder_dropout=0.0,
             decoder_dropout=0.0, bidirectional_encoder=True, latent_dims=lat, adversarial_loss=True, mi_loss=True,
             learn_rate=float(g["lr"]), lambdas={"default": 0.5}, teacher_forcing_prob=1.0, random_seed=10)
    dev = torch.device("cuda")
    X, L = torch.from_numpy(g["inputs"]), torch.from_numpy(g["lengths"])
    Y = {n: torch.from_numpy(g[f"Y.{n}"]) for n in label_dims}
    B, T = X.shape
    eps = torch.from_numpy(np.concatenate([g[f"eps.{n}"] for n in names], axis=1)).to(dev)
    out = []
    for shape in ((B + 3, T + 4), (B, T)):
        vae = dvae.build_vae(p, int(g["V"]), None, label_dims, dev, int(g["sos"]), int(g["eos"]))
        vae.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
        for n, est in vae.mi_estimators.items():
            est.load_state_dict({k[len(f"mi0.{n}."):]: torch.from_numpy(g[k]) for k in g if k.startswith(f"mi0.{n}.")})
        vae.train()
        eng = engine_mod.TrainEngine(vae, p, *shape, total_steps=10, seed=1)
        assert eng.aux and not eng.use_graph
        eng.fixed_eps = torch.cat([eps, torch.zeros(shape[0] - B, eps.shape[1], device=dev)])
        w0 = vae._flat.detach().clone()
        got = eng.step_host(X, L, Y)
        sds = {k: v.detach().clone() for k, v in vae.state_dict().items()}
        for n, est in vae.mi_estimators.items():
            sds.update({f"mi.{n}.{k}": v.detach().clone() for k, v in est.state_dict().items()})
        out.append((got, sds, w0))
    (ga, sa, w0), (gb, sb, _) = out
    for k in ("total_loss", "total_adv_loss", "total_mi", "reconstruction_loss"):
        assert abs(ga[k] - gb[k]) <= 1e-5 * abs(gb[k]) + 1e-9, (k, ga[k], gb[k])
    for n in gb["idv_adv_losses"]:
        assert abs(ga["idv_adv_losses"][n] - gb["idv_adv_losses"][n]) <= 1e-5 * abs(gb["idv_adv_losses"][n]) + 1e-9
    for k in sb:
        assert (sa[k] - sb[k]).abs().max().item() < 4e-6, k      # each engine is within 2e-6 of the reference


# ---- 6. batches the engine cannot take -----------------------------------------------------------------------------
def test_oversize_and_undersize_batches_raise(dvae, engine_mod):
    V, B, T = 300, 8, 10
    cfg = _cfg(embedding_dim=64, hidden_dim=64)
    vae = _model(dvae, cfg, V)
    eng = engine_mod.TrainEngine(vae, cfg, B, T, total_steps=20, seed=1)
    gen = torch.Generator().manual_seed(3)
    X, L, Y = _batch(gen, B, T, V)
    X9, L9, Y9 = _batch(gen, B + 1, T, V)
    bad = {
        "rows": (X9, L9, Y9),
        "length": (torch.cat([X, X[:, :1]], 1), L, Y),
        "T'<2": (X[:, :1], torch.ones(B, dtype=torch.long), Y),
        "lengths>T'": (X[:, :6], L, Y),
        "lengths rows": (X, L[:1], Y),
        "label rows": (X, L, {k: v[:1] for k, v in Y.items()}),
    }
    dev = torch.device("cuda")
    for why, (Xb, Lb, Yb) in bad.items():
        for call in (lambda: eng.step_host(Xb, Lb, Yb), lambda: list(eng.train_steps([(Xb, Lb, Yb)])),
                     lambda: eng.eval_step(Xb, Lb, Yb, 1.0), lambda: list(eng.eval_steps([(Xb, Lb, Yb)], 1.0))):
            with pytest.raises(ValueError, match=r"\(8, 10\)|expected"):
                call()
        Yd = torch.stack([Yb[n].reshape(-1) for n in eng.label_names]).to(dev)
        with pytest.raises(ValueError):
            eng.step_resident(Xb.to(dev), Lb.to(dev), Yd)
    assert eng.adam_step == 0 and eng.step_idx == 0 and not eng._extra
    eng.step_host(X[:3, :7], L[:3].clamp(max=7), {k: v[:3] for k, v in Y.items()})      # in range: accepted
    assert eng.adam_step == 1


def test_short_shape_cache_is_bounded(dvae, engine_mod):
    V, B, T = 300, 8, 10
    cfg = _cfg(embedding_dim=64, hidden_dim=64)
    vae = _model(dvae, cfg, V)
    eng = engine_mod.TrainEngine(vae, cfg, B, T, total_steps=20, seed=1)
    gen = torch.Generator().manual_seed(3)
    for b in (2, 3, 4, 3, 5):
        eng.step_host(*_batch(gen, b, T, V))
    assert list(eng._extra) == [3, 5] and len(eng._extra) == eng.MAX_EXTRA_SHAPES
    flat = vae._flat.detach().clone()
    assert torch.isfinite(flat).all()


# ---- 7. data parallel: a short step between full ones --------------------------------------------------------------
def _free_port():
    import socket
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.parametrize("exchange", ["default", "nccl_stages"])
def test_two_ranks_with_a_short_step_equal_one_engine_on_the_global_batches(tmp_path, exchange):
    import subprocess
    world = 2
    if not torch.cuda.is_available() or torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    out = tmp_path / "dp_shapes.npz"
    env = dict(os.environ, **({"DVAE_DP_NVLS": "0"} if exchange == "nccl_stages" else {}))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr",
           "127.0.0.1", "--master-port", str(_free_port()), os.path.join(ROOT, "tests", "shapes_dp_worker.py"), str(out)]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900, env=env)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    got = np.load(out)
    assert str(got["exchange"]) == {"default": "p2p", "nccl_stages": "nccl+stages"}[exchange]
    assert got["replicas_identical"][0] == 1.0
    import shapes_dp_worker as W
    vae, eng, losses, w0 = W.run(1, 0, torch.device("cuda", 0))
    for a, b in zip(got["losses"], losses):
        assert abs(a - b) <= 1e-5 * abs(b), (got["losses"], losses)
    want = vae._flat.detach()
    _updates_agree(torch.from_numpy(got["flat"]).to(want.device)[:want.numel()], want, w0)
