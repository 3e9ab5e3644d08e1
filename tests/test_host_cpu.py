"""CPU-side tests: C-ABI surface, host logic, config schema, checkpoint-key compatibility."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest
import torch

from conftest import ROOT, load_golden, golden_state_dict

HEADER = os.path.join(ROOT, "include", "dvae_b200.h")


def _declared_functions():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    out = {}
    for m in re.finditer(r"(?:const\s+char\s*\*|int64_t|int)\s+(dvae_\w+)\s*\(([^;{]*)\)\s*;", src):
        args = m.group(2).strip()
        n = 0 if args in ("", "void") else len([a for a in args.split(",") if a.strip()])
        out[m.group(1)] = n
    return out


def test_library_builds_loads_and_exports_every_declared_symbol(dvae):
    import __graft_entry__ as ge
    ge.build()
    decl = _declared_functions()
    assert len(decl) >= 20
    lib = ctypes.CDLL(dvae._lib.LIB_PATH)
    for name in decl:
        assert hasattr(lib, name), f"{name} declared in include/dvae_b200.h but not exported"
    # the ctypes binding mirrors the header one-to-one (same names, same arity)
    assert set(decl) == set(dvae._lib.SIGNATURES), set(decl) ^ set(dvae._lib.SIGNATURES)
    for name, n in decl.items():
        assert len(dvae._lib.SIGNATURES[name][1]) == n, f"{name}: header has {n} args"
    loaded = dvae._lib.load()
    assert loaded.dvae_version() >= 100
    assert loaded.dvae_lstm_state_ws_floats(4, 8, 2) == 4 * 2 * 4 * 8 + 4 * 2 * 8 * 8 + 8 * 128    # states, W_hh^T, 8 sets of per-CTA max|dG| slots
    # no undefined CUDA driver symbols: the .so must load on a box without libcuda
    nm = subprocess.run(["nm", "-D", "--undefined-only", dvae._lib.LIB_PATH], capture_output=True, text=True).stdout
    assert " cu" not in nm.replace("cuda", "")


def test_sass_is_sm100a(dvae):
    cuobjdump = "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([cuobjdump, "-lelf", dvae._lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out


def _params(**over):
    p = {"name": "t", "random_seed": 10, "data_dir": "", "combined_dataset": False, "dataset_minibatch_ratios": {},
         "checkpoint_dir": "", "glove_path": "", "num_train_examples": -1, "lowercase": True, "reverse_input": False,
         "embedding_dim": 12, "hidden_dim": 16, "num_rnn_layers": 2, "bidirectional_encoder": True, "bow_encoder": False,
         "latent_dims": {"total": 7, "polarity": 1, "uncertainty": 2}, "epochs": 3, "batch_size": 5, "learn_rate": 3e-4,
         "encoder_dropout": 0.5, "decoder_dropout": 0.5, "teacher_forcing_prob": 0.5,
         "lambdas": {"default": "cyclic", "polarity": 0.005}, "adversarial_loss": False, "mi_loss": False,
         "train": True, "validate": False, "test": False}
    p.update(over)
    return p


def test_validate_params_schema(dvae):
    dvae.validate_params(_params())
    bad = _params()
    del bad["mi_loss"]
    with pytest.raises(ValueError, match="missing 'mi_loss'"):
        dvae.validate_params(bad)
    with pytest.raises(ValueError, match="incorrect type"):
        dvae.validate_params(_params(batch_size="32"))
    with pytest.raises(ValueError):
        dvae.validate_params(_params(lambdas={"default": "sometimes"}))
    w = dvae.utils.kl_weights_for_step(_params(), 5, 100)
    assert w == {"default": 0.4, "polarity": 0.005}


def test_cyclic_schedule_matches_golden(dvae):
    for step, total, want in load_golden("cyclic_kl")["table"]:
        assert abs(dvae.losses.get_cyclic_kl_weight(int(step), int(total)) - want) < 1e-12


def test_state_dict_keys_shapes_and_flat_views(dvae):
    g = load_golden("tiny_bi")
    sd = golden_state_dict(g)
    p = _params(embedding_dim=10, hidden_dim=8)
    vae = dvae.build_vae(p, int(g["V"]), None, {"uncertainty": 1, "polarity": 1}, torch.device("cpu"), 2, 3)
    mine = vae.state_dict()
    assert list(mine.keys()) == list(sd.keys())              # same keys, same order as the reference
    for k in sd:
        assert tuple(mine[k].shape) == sd[k].shape, k
    vae.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    # parameters are views of ONE flat buffer, grouped so the fused-head kernel sees single matrices
    flat = vae._flat
    for n, prm in vae.named_parameters():
        assert prm.data.untyped_storage().data_ptr() == flat.untyped_storage().data_ptr(), n
        assert np.array_equal(prm.detach().numpy(), sd[n])
    names = [str(s) for s in g["space_names"]]
    cat = np.concatenate([sd[f"context2params.{n}.weight"] for n in names], axis=0)
    assert np.array_equal(vae._P["_c2p.weight"].numpy(), cat)
    assert vae._flat_numel % 4 == 0
    assert len(vae.trainable_parameters()) == len(sd)
    # round trip through a checkpoint file with the reference's layout (run.py:627-630)
    ck = {"model_state_dict": vae.state_dict(), "epoch": 0}
    vae2 = dvae.build_vae(p, int(g["V"]), None, {"uncertainty": 1, "polarity": 1}, torch.device("cpu"), 2, 3)
    vae2.load_state_dict(ck["model_state_dict"])
    assert all(torch.equal(a, b) for a, b in zip(vae.state_dict().values(), vae2.state_dict().values()))


def test_cpu_model_refuses_to_run(dvae):
    vae = dvae.build_vae(_params(), 30, None, {"polarity": 1}, torch.device("cpu"), 2, 3)
    with pytest.raises(dvae.DvaeError, match="no CPU fallback"):
        vae(torch.zeros(2, 5, dtype=torch.long), torch.tensor([5, 3]))
    bow = dvae.build_vae(_params(bow_encoder=True), 30, None, {"polarity": 1}, torch.device("cpu"), 2, 3)
    assert [k for k in bow.state_dict() if k.startswith("encoder.")] == ["encoder.embedding.weight"]      # vae/model.py:13-49
    assert (bow.encoder.hidden_size, bow.encoder.num_layers, bow.encoder.num_directions) == (bow.encoder.emb_dim, 1, 1)
    assert bow.context2params["content"].in_features == bow.encoder.emb_dim


# Model settings of the golden cases (tests/golden/make_golden.py): each file's `sd.*` arrays are the reference's
# state_dict right after its set_seed(10) and build_vae(), before any step.
_GOLDEN_INIT = {
    "tiny_uni": ({}, {"polarity": 1}),
    "tiny_bi": ({"bidirectional_encoder": True, "embedding_dim": 10, "hidden_dim": 8,
                 "latent_dims": {"total": 7, "polarity": 1, "uncertainty": 2}}, {"uncertainty": 1, "polarity": 1}),
    "tiny_eval_mc": ({"num_rnn_layers": 1, "embedding_dim": 6, "hidden_dim": 8, "latent_dims": {"total": 5, "modality": 2}},
                     {"modality": 3}),
    "tiny_bow": ({"bow_encoder": True, "embedding_dim": 10, "hidden_dim": 8, "latent_dims": {"total": 5, "polarity": 1}},
                 {"polarity": 1}),
    "tiny_adv_mi": ({"bidirectional_encoder": True, "embedding_dim": 10, "hidden_dim": 8, "adversarial_loss": True,
                     "mi_loss": True, "latent_dims": {"total": 9, "polarity": 1, "uncertainty": 2}},
                    {"uncertainty": 3, "polarity": 1}),
}


def _seeded_model_of_golden_case(dvae, case):
    over, label_dims = _GOLDEN_INIT[case]
    g = load_golden(case)
    p = _params(**{"embedding_dim": 12, "hidden_dim": 16, "bidirectional_encoder": False, "encoder_dropout": 0.0,
                   "decoder_dropout": 0.0, "latent_dims": {"total": 6, "polarity": 1}, **over})
    dvae.set_seed(10)
    return g, dvae.build_vae(p, int(g["V"]), None, label_dims, torch.device("cpu"), int(g["sos"]), int(g["eos"]))


def test_adversarial_and_mi_modules_match_reference_structure_and_seeded_init(dvae):
    """adversarial_loss / mi_loss: same adversary and estimator names, same state_dict keys, and -- because the
    construction order is the reference's -- bit-identical seeded initial weights (incl. the CLUB estimators, which the
    reference keeps in a plain dict outside the state_dict; stored as `mi0.*` in the golden file)."""
    g, mine = _seeded_model_of_golden_case(dvae, "tiny_adv_mi")
    assert list(mine.adversaries.keys()) == [str(n) for n in g["adv_names"]]
    assert list(mine.mi_estimators.keys()) == [str(n) for n in g["mi_names"]]
    rs, ms = golden_state_dict(g), mine.state_dict()
    assert list(rs.keys()) == list(ms.keys())
    for k in rs:
        assert np.array_equal(rs[k], ms[k].numpy()), k
    for n, est in mine.mi_estimators.items():
        a, b = golden_state_dict(g, f"mi0.{n}."), est.state_dict()
        assert list(a.keys()) == list(b.keys())
        for k in a:
            assert np.array_equal(a[k], b[k].numpy()), (n, k)
    assert [n for n, _ in mine.named_parameters() if n.startswith("adversaries")]
    assert not [q for q in mine.trainable_parameters() if any(q is w for w in mine.adversaries.parameters())]
    assert not any(n.startswith("adversaries") for n in mine._layout)      # adversaries own their optimizers


def test_same_seed_gives_reference_initialisation(dvae):
    for case in ("tiny_uni", "tiny_bi", "tiny_eval_mc", "tiny_bow"):
        g, mine = _seeded_model_of_golden_case(dvae, case)
        rs, ms = golden_state_dict(g), mine.state_dict()
        assert list(rs.keys()) == list(ms.keys()), case
        for k in rs:
            assert np.array_equal(rs[k], ms[k].numpy()), (case, k)
