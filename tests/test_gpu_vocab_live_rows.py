"""Vocabulary projection / cross-entropy over the LIVE rows only (dvae_vocab_ce_fwd_live / dvae_vocab_ce_bwd_live): the
row list, parity with the every-row calls and the float64 oracle, one captured graph over different length mixes, and
the TrainEngine step that uses them."""
import importlib
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from oracle import dvae_oracle as O  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dvae():
    import __graft_entry__ as ge
    return ge.build()


@pytest.fixture(scope="module")
def L(dvae):
    return dvae._lib


@pytest.fixture(scope="module")
def lib(L):
    return L.load()


def dev(x, dtype=torch.float32):
    return torch.as_tensor(np.ascontiguousarray(x), dtype=dtype, device="cuda")


def rel(a, b):
    a = a.detach().cpu().numpy().astype(np.float64) if torch.is_tensor(a) else np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


class Case:
    """Inputs of one vocabulary-CE call (the construction of test_gpu_kernels.py::test_vocab_ce) and its device buffers."""

    def __init__(self, lib, T1, B, H, V, lengths=None, seed=None):
        rng = np.random.default_rng(T1 + B + V if seed is None else seed)
        self.lib, self.T1, self.B, self.H, self.V = lib, T1, B, H, V
        self.N, self.T = N, T = T1 * B, T1 + 1
        self.h = rng.standard_normal((T1, B, H)).astype(np.float32) * 0.5
        self.W = rng.uniform(-1, 1, (V, H)).astype(np.float32) / np.sqrt(H) * 3
        self.b = rng.uniform(-0.1, 0.1, V).astype(np.float32)
        if lengths is None:
            lengths = rng.integers(1, T + 1, B)
            lengths[0] = T
        self.lengths = np.asarray(lengths, np.int64)
        self.targets = rng.integers(0, V, (B, T))
        self.sos = 2
        self.targets[:, 0] = self.sos
        self.targets[1 % B, 0] = 5
        self.hd, self.Wd, self.bd = dev(self.h), dev(self.W), dev(self.b)
        self.td, self.ld = dev(self.targets, torch.int64), dev(self.lengths, torch.int64)
        self.ws = torch.zeros(lib.dvae_vocab_ce_ws_floats(N, V, H), device="cuda")
        self.wsb = torch.zeros(lib.dvae_vocab_ce_bwd_ws_floats(N, V, H), device="cuda")
        self.gs = torch.tensor([1.0], device="cuda")

    def live_mask(self):      # [N] time-major: position n = t * B + b is live when t + 1 < len_b
        t = np.arange(self.T1)[:, None]
        return (t + 1 < self.lengths[None, :]).reshape(-1)

    def oracle(self):
        logits = np.zeros((self.B, self.T, self.V))
        logits[:, 0, self.sos] = 1.0
        logits[:, 1:, :] = (self.h.astype(np.float64) @ self.W.astype(np.float64).T + self.b).transpose(1, 0, 2)
        loss, cache = O.seq_ce_fwd(logits, self.targets, self.lengths)
        dl = O.seq_ce_bwd(cache)[:, 1:, :].transpose(1, 0, 2).reshape(self.N, self.V)
        return logits, loss, cache, dl

    def fwd(self, L, live, ws=None):
        ws = self.ws if ws is None else ws
        N = self.N
        out = dict(lse=torch.zeros(N, device="cuda"), nll=torch.zeros(N, device="cuda"),
                   am=torch.zeros(N, device="cuda", dtype=torch.int32), loss=torch.zeros(1, device="cuda"))
        self.fwd_into(L, live, out, ws)
        return out

    def fwd_into(self, L, live, out, ws=None):
        lib, ws = self.lib, self.ws if ws is None else ws
        fn = lib.dvae_vocab_ce_fwd_live if live else lib.dvae_vocab_ce_fwd_ex
        L.check(fn(L.ptr(self.hd), self.H, self.T1, self.B, self.H, self.V, L.ptr(self.Wd), L.ptr(self.bd), L.ptr(self.td), self.T,
                   L.ptr(self.ld), self.sos, L.ptr(out["lse"]), L.ptr(out["nll"]), L.ptr(out["am"]), L.ptr(out["loss"]), L.ptr(ws), 0,
                   L.stream_ptr()), "vocab ce fwd")

    def bwd(self, L, live, lse, fwd_ws=None):
        N, V, H = self.N, self.V, self.H
        g = dict(d_h=torch.full((N, H), 7.0, device="cuda"), d_w=torch.full((V, H), 9.0, device="cuda"),
                 d_b=torch.full((V,), 9.0, device="cuda"))
        self.bwd_into(L, live, lse, g, fwd_ws)
        return g

    def bwd_into(self, L, live, lse, g, fwd_ws=None):
        lib = self.lib
        fn = lib.dvae_vocab_ce_bwd_live if live else lib.dvae_vocab_ce_bwd
        L.check(fn(L.ptr(self.hd), self.H, self.T1, self.B, self.H, self.V, L.ptr(self.Wd), L.ptr(self.bd), L.ptr(self.td), self.T,
                   L.ptr(self.ld), L.ptr(lse), L.ptr(self.gs), L.ptr(g["d_h"]), self.H, L.ptr(g["d_w"]), L.ptr(g["d_b"]),
                   L.ptr(self.ws if live else fwd_ws) if (live or fwd_ws is not None) else None, L.ptr(self.wsb), L.stream_ptr()),
                "vocab ce bwd")

    def row_list(self):
        at = self.lib.dvae_vocab_live_rows_at(self.N, self.V, self.H)
        iv = self.ws.view(torch.int32)
        m = int(iv[at + self.N].item())
        return m, iv[at:at + m].cpu().numpy()


# ---- (a) the row list ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["all_one", "all_full", "mixed", "m_odd"])
def test_live_row_list_matches_numpy(lib, L, kind):
    T1, B, H, V = 21, 128, 256, 10000
    T = T1 + 1
    rng = np.random.default_rng(7)
    lengths = {"all_one": np.ones(B), "all_full": np.full(B, T), "mixed": rng.integers(1, T + 1, B),
               "m_odd": np.r_[np.full(B - 1, 1), 5 + 32]}[kind].astype(np.int64)
    lengths = np.minimum(lengths, T)
    c = Case(lib, T1, B, H, V, lengths=lengths)
    c.fwd(L, True)
    torch.cuda.synchronize()
    want = np.nonzero(c.live_mask())[0]
    m, rows = c.row_list()
    assert m == len(want) and np.array_equal(rows, want)
    if kind == "m_odd":
        assert m % 32 != 0 and m % 128 != 0
    if kind == "all_one":
        assert m == 0
    if kind == "all_full":
        assert m == c.N


# ---- (b) live-row calls against the every-row calls and the float64 oracle -------------------------------------------
@pytest.mark.parametrize("T1,B,H,V", [(4, 3, 8, 23), (5, 9, 12, 1000), (6, 50, 64, 3001), (19, 128, 256, 10000), (21, 128, 256, 10000),
                                      (7, 40, 1024, 2000)])
def test_vocab_ce_live_matches_full_and_oracle(lib, L, T1, B, H, V):
    c = Case(lib, T1, B, H, V)
    logits, want_loss, cache, dl = c.oracle()
    full = c.fwd(L, False, ws=torch.zeros_like(c.ws))
    live = c.fwd(L, True)
    live_n = c.live_mask()
    assert abs(live["loss"].item() - want_loss) <= 1e-5 * abs(want_loss)
    assert abs(live["loss"].item() - full["loss"].item()) <= 1e-5 * abs(want_loss)
    nll_ref = cache["nll"][:, 1:].T.reshape(-1)
    assert rel(live["nll"].cpu().numpy()[live_n], nll_ref[live_n]) < 1e-5
    assert np.array_equal(live["nll"].cpu().numpy()[live_n], full["nll"].cpu().numpy()[live_n]) or \
        rel(live["nll"].cpu().numpy()[live_n], full["nll"].cpu().numpy()[live_n]) < 1e-6
    ref_am = logits[:, 1:, :].argmax(-1).T.reshape(-1)
    got_am = live["am"].cpu().numpy()
    bad = np.nonzero((got_am != ref_am) & live_n)[0]
    if len(bad):      # only exact fp32 near-ties may differ
        flat = logits[:, 1:, :].transpose(1, 0, 2).reshape(c.N, V)
        gap = np.abs(flat[bad, got_am[bad]] - flat[bad, ref_am[bad]])
        assert gap.max() < 1e-6, f"argmax differs on {len(bad)} live rows with gap {gap.max()}"
    g = c.bwd(L, True, live["lse"])
    hf = c.h.reshape(c.N, H).astype(np.float64)
    W64 = c.W.astype(np.float64)
    assert rel(g["d_h"], dl @ W64) < 1e-4
    assert rel(g["d_w"], dl.T @ hf) < 1e-4
    assert rel(g["d_b"], dl.sum(0)) < 1e-4
    if (~live_n).any():      # masked rows of d_h are exactly zero
        assert float(g["d_h"][torch.from_numpy(~live_n).cuda()].abs().max()) == 0.0
    gf = c.bwd(L, False, full["lse"])
    for k in ("d_h", "d_w", "d_b"):
        assert rel(g[k], gf[k].cpu().numpy()) < 1e-5, k


def test_vocab_ce_live_no_live_rows(lib, L):
    """M = 0: the loss is the position-0 term alone and every gradient is zero."""
    c = Case(lib, 21, 128, 256, 10000, lengths=np.ones(128, np.int64))
    _, want_loss, _, _ = c.oracle()
    out = c.fwd(L, True)
    assert abs(out["loss"].item() - want_loss) <= 1e-5 * abs(want_loss)
    g = c.bwd(L, True, out["lse"])
    for k in ("d_h", "d_w", "d_b"):
        assert float(g[k].abs().max()) == 0.0, k


# ---- (c) one captured graph, three length distributions --------------------------------------------------------------
def test_vocab_ce_live_graph_replay(lib, L):
    T1, B, H, V = 21, 128, 256, 10000
    T = T1 + 1
    c = Case(lib, T1, B, H, V)
    rng = np.random.default_rng(3)
    _, bench_like, _ = bench.synth_batch(rng, B)
    mixes = {"all_full": np.full(B, T), "bench": np.minimum(bench_like, T), "all_two": np.full(B, 2)}
    eager = {}
    for name, lens in mixes.items():
        c.ld.copy_(dev(lens, torch.int64))
        o = c.fwd(L, True)
        gr = c.bwd(L, True, o["lse"])
        torch.cuda.synchronize()
        eager[name] = (o["loss"].clone(), {k: v.clone() for k, v in gr.items()})
    out = dict(lse=torch.zeros(c.N, device="cuda"), nll=torch.zeros(c.N, device="cuda"),
               am=torch.zeros(c.N, device="cuda", dtype=torch.int32), loss=torch.zeros(1, device="cuda"))
    grads = dict(d_h=torch.zeros(c.N, H, device="cuda"), d_w=torch.zeros(V, H, device="cuda"), d_b=torch.zeros(V, device="cuda"))
    c.ld.copy_(dev(mixes["bench"], torch.int64))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):      # warm-up off the capture
        c.fwd_into(L, True, out)
        c.bwd_into(L, True, out["lse"], grads)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        c.fwd_into(L, True, out)
        c.bwd_into(L, True, out["lse"], grads)
    for name, lens in mixes.items():
        losses = []
        for _ in range(2):
            c.ld.copy_(dev(lens, torch.int64))
            graph.replay()
            torch.cuda.synchronize()
            losses.append(out["loss"].clone())
            want_loss, want_g = eager[name]
            assert torch.equal(out["loss"], want_loss), name
            for k in grads:
                assert rel(grads[k], want_g[k].cpu().numpy()) < 1e-6, (name, k)
        assert torch.equal(losses[0], losses[1]), name
        c.lengths = np.asarray(lens, np.int64)
        _, oracle_loss, _, _ = c.oracle()
        assert abs(out["loss"].item() - oracle_loss) <= 1e-5 * abs(oracle_loss), name


# ---- (d) the engine: one graph, replayed on a full-length and a short-row batch --------------------------------------
def test_train_engine_live_rows_graph_replay_matches_oracle(dvae):
    from test_gpu_baseline_shapes import LABELS2, _cfg, _masks
    engine_mod = importlib.import_module("disentanglement-vae_b200.engine")
    device = torch.device("cuda")
    B, cfg, V, T = 128, _cfg(), bench.VOCAB, bench.SEQ_T
    dvae.set_seed(10)
    vae = dvae.build_vae(cfg, V, None, LABELS2, device, bench.SOS, bench.EOS)
    vae.train()
    eng = engine_mod.TrainEngine(vae, cfg, B, T, total_steps=bench.TOTAL_STEPS, use_graph=True, seed=10)
    assert eng.plan.live_rows
    eng.step_idx = 1234
    rng = np.random.default_rng(1000)
    X0, l0, Y0 = bench.synth_batch(rng, B)
    eng.step_host(torch.from_numpy(X0), torch.from_numpy(l0), {n: torch.from_numpy(Y0[j]).reshape(-1, 1) for j, n in enumerate(LABELS2)})
    lr = cfg["learn_rate"]
    for step, kind in enumerate(("full", "short")):
        X, lengths, Yr = bench.synth_batch(rng, B)
        lengths = np.full(B, T, lengths.dtype) if kind == "full" else np.minimum(lengths, 3)
        Y = {n: torch.from_numpy(Yr[j]).reshape(-1, 1) for j, n in enumerate(LABELS2)}
        sd0 = {k: t.detach().cpu().numpy().astype(np.float64) for k, t in vae.state_dict().items()}
        Mv, Vv = vae.grad_views(eng.m), vae.grad_views(eng.v)
        m = {k: Mv[k].detach().cpu().numpy().astype(np.float64) for k in sd0}
        v2 = {k: Vv[k].detach().cpu().numpy().astype(np.float64) for k in sd0}
        got = eng.step_host(torch.from_numpy(X), torch.from_numpy(lengths), Y)
        d = eng.plan.d
        enc_m, dec_m = _masks(dvae, eng.plan, T, B, d.E, d.D * d.H, d.Hd, d.p_enc, d.p_dec)
        klw = {"default": O.cyclic_kl_weight(1235 + step, bench.TOTAL_STEPS), "polarity": 0.005, "uncertainty": 0.005}
        spec = O.ModelSpec(sd0, list(vae.context2params.keys()), bench.SOS, bench.EOS)
        eps = eng.plan.eps.detach().cpu().numpy()
        eps_d, off = {}, 0
        for n, zs in zip(spec.space_names, spec.space_dims):
            eps_d[n] = eps[:, off:off + zs]
            off += zs
        fw = O.model_forward(sd0, spec, X, lengths, eps_d, labels={k: v.numpy() for k, v in Y.items()}, kl_weights=klw,
                             enc_masks=enc_m, dec_masks=dec_m)
        grads = O.model_backward(sd0, spec, fw)
        assert abs(got["total_loss"] - fw["total_loss"]) <= 1e-5 * abs(fw["total_loss"]), (kind, got["total_loss"], fw["total_loss"])
        am = eng.plan.argmax[:eng.plan.N].view(T - 1, B).t().cpu().numpy()
        lg = fw["decoder_logits"][:, 1:]
        srt = np.sort(lg, axis=-1)
        sel = ((srt[..., -1] - srt[..., -2]) > 1e-5) & (np.arange(1, T)[None, :] < lengths[:, None])
        assert np.array_equal(am[sel], lg.argmax(-1)[sel])
        after = {k: a.copy() for k, a in sd0.items()}
        O.clip_and_adam(after, grads, m, v2, eng.adam_step, lr)
        now = {k: t.detach().cpu().numpy().astype(np.float64) for k, t in vae.state_dict().items()}
        for k in sd0:
            sig = np.abs(grads[k]) > 1e-4 * np.abs(grads[k]).max()
            if sig.any():
                want, have = after[k] - sd0[k], now[k] - sd0[k]
                err = np.abs(want - have)[sig].max() / max(np.abs(want[sig]).max(), 1e-30)
                assert err < 2e-3, (kind, k, err)
