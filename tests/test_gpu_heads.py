"""Fused latent heads on clusters: forward and backward against float64 torch (autograd for the gradients), over shapes
that exercise the cluster split (Z and H2L not multiples of 8, B not a multiple of the rows per cluster, wide contexts,
multi-class discriminators), plus run-to-run and graph-replay bit-reproducibility of the scalars and d_ctx."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def lib(dvae):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return dvae._lib.load()


@pytest.fixture(scope="module")
def L(dvae):
    return dvae._lib


def _case(B, C, dims, dsc_out, H2L, seed):
    rng = np.random.default_rng(seed)
    S, Z, OD = len(dims), sum(dims), sum(dsc_out)
    n_w = sum(o * z for o, z in zip(dsc_out, dims))
    f = lambda a: torch.tensor(np.asarray(a, np.float32), device="cuda")
    c = dict(B=B, C=C, dims=dims, dsc_out=dsc_out, H2L=H2L, S=S, Z=Z, OD=OD)
    c["ctx"] = f(rng.standard_normal((B, C)) * 0.5)
    c["Wc"] = f(rng.uniform(-1, 1, (2 * Z, C)) / np.sqrt(C))
    c["bc"] = f(rng.uniform(-0.1, 0.1, 2 * Z))
    c["eps"] = f(rng.standard_normal((B, Z)))
    c["Wd"] = f(rng.uniform(-1, 1, max(n_w, 1)))
    c["bd"] = f(rng.uniform(-1, 1, max(OD, 1)))
    c["Wz"] = f(rng.uniform(-1, 1, (H2L, Z)) / np.sqrt(Z))
    c["bz"] = f(rng.uniform(-0.1, 0.1, H2L))
    labels = np.zeros((max(sum(1 for o in dsc_out if o > 0), 1), B), np.float32)
    i = 0
    for o in dsc_out:
        if o > 0:
            labels[i] = rng.integers(0, max(o, 2), B)
            i += 1
    c["labels"] = f(labels)
    c["klw"] = f(rng.uniform(0, 1, S))
    c["d_hid"] = f(rng.standard_normal((B, H2L)) * 0.1)
    c["d_z_x"] = f(rng.standard_normal((B, Z)) * 0.01)
    c["d_mu_x"] = f(rng.standard_normal((B, Z)) * 0.01)
    c["d_lv_x"] = f(rng.standard_normal((B, Z)) * 0.01)
    c["d_lg_x"] = f(rng.standard_normal((B, max(OD, 1))) * 0.01)
    return c


def _reference(c):
    """float64 torch forward of the heads (vae/model.py:384-411, vae/losses.py:153-196) and the autograd gradients of
    sum_s kl_w[s] kl_s + sum_s dsc_loss_s + <d_hid, hid> + the extras' inner products."""
    g = lambda k: c[k].double().clone().requires_grad_(True)
    ctx, Wc, bc, Wd, bd, Wz, bz = (g(k) for k in ("ctx", "Wc", "bc", "Wd", "bd", "Wz", "bz"))
    eps, klw, labels = c["eps"].double(), c["klw"].double(), c["labels"].double()
    B = c["B"]
    zs_, mus, lvs, kls, logits, dls, das = [], [], [], [], [], [], []
    off = woff = boff = li = 0
    for s, zs in enumerate(c["dims"]):
        p = ctx @ Wc[2 * off:2 * off + 2 * zs].T + bc[2 * off:2 * off + 2 * zs]
        mu, lv = p[:, :zs], torch.tanh(p[:, zs:])
        z = mu + eps[:, off:off + zs] * torch.exp(lv)
        zs_.append(z); mus.append(mu); lvs.append(lv)
        kls.append((0.5 * (torch.exp(lv) + mu * mu - 1 - lv)).sum(1).mean())
        o = c["dsc_out"][s]
        if o > 0:
            lg = z @ Wd[woff:woff + o * zs].reshape(o, zs).T + bd[boff:boff + o]
            y = labels[li]
            if o == 1:
                x = lg[:, 0]
                dls.append((torch.clamp(x, min=0) - x * y + torch.log1p(torch.exp(-x.abs()))).mean())
                das.append(((x > 0).double() == y).double().mean())
            else:
                dls.append(torch.nn.functional.cross_entropy(lg, y.long()))
                das.append((lg.argmax(1) == y.long()).double().mean())
            logits.append(lg)
            woff += o * zs; boff += o; li += 1
        off += zs
    z, mu, lv = torch.cat(zs_, 1), torch.cat(mus, 1), torch.cat(lvs, 1)
    hid = torch.tanh(z @ Wz.T + bz)
    lg = torch.cat(logits, 1) if logits else None
    kl = torch.stack(kls)
    total = (klw * kl).sum() + (c["d_hid"].double() * hid).sum() + (c["d_z_x"].double() * z).sum()
    total = total + (c["d_mu_x"].double() * mu).sum() + (c["d_lv_x"].double() * lv).sum()
    if dls:
        total = total + sum(dls) + (c["d_lg_x"][:, :c["OD"]].double() * lg).sum()
    total.backward()
    out = dict(z=z, mu=mu, logvar=lv, hid=hid, logits=lg, kl=kl, dls=dls, das=das,
               d_ctx=ctx.grad, d_w_c2p=Wc.grad, d_b_c2p=bc.grad, d_w_z2h=Wz.grad, d_b_z2h=bz.grad)
    if dls:
        out["d_w_dsc"], out["d_b_dsc"] = Wd.grad, bd.grad
    out["dls"], out["das"] = [t.detach() for t in dls], [t.detach() for t in das]
    return {k: (v.detach() if torch.is_tensor(v) else v) for k, v in out.items()}


def _fwd(lib, L, c, ws):
    B, Z, OD, H2L = c["B"], c["Z"], c["OD"], c["H2L"]
    o = dict(z=torch.zeros(B, Z, device="cuda"), mu=torch.zeros(B, Z, device="cuda"), logvar=torch.zeros(B, Z, device="cuda"),
             hid=torch.zeros(B, H2L, device="cuda"), logits=torch.zeros(B, max(OD, 1), device="cuda"),
             sc=torch.zeros(L.HEADS_NSCALARS, device="cuda"))
    L.check(lib.dvae_latent_heads_fwd(L.ptr(c["ctx"]), B, c["C"], c["S"], L.int_array(c["dims"]), L.int_array(c["dsc_out"]),
                                      L.ptr(c["Wc"]), L.ptr(c["bc"]), L.ptr(c["eps"]), L.ptr(c["Wd"]), L.ptr(c["bd"]),
                                      L.ptr(c["labels"]), L.ptr(c["klw"]), L.ptr(c["Wz"]), L.ptr(c["bz"]), H2L, L.ptr(o["z"]),
                                      L.ptr(o["mu"]), L.ptr(o["logvar"]), L.ptr(o["hid"]), L.ptr(o["logits"]), L.ptr(o["sc"]),
                                      L.ptr(ws), L.stream_ptr()), "heads fwd")
    return o


def _bwd(lib, L, c, f, ws):
    B, C, Z, OD, H2L = c["B"], c["C"], c["Z"], c["OD"], c["H2L"]
    n_w = sum(o * z for o, z in zip(c["dsc_out"], c["dims"]))
    g = dict(d_w_c2p=torch.zeros(2 * Z, C, device="cuda"), d_b_c2p=torch.zeros(2 * Z, device="cuda"),
             d_w_dsc=torch.zeros(max(n_w, 1), device="cuda"), d_b_dsc=torch.zeros(max(OD, 1), device="cuda"),
             d_w_z2h=torch.zeros(H2L, Z, device="cuda"), d_b_z2h=torch.zeros(H2L, device="cuda"),
             d_ctx=torch.full((B, C), float("nan"), device="cuda"))
    L.check(lib.dvae_latent_heads_bwd(L.ptr(c["ctx"]), B, C, c["S"], L.int_array(c["dims"]), L.int_array(c["dsc_out"]),
                                      L.ptr(c["Wc"]), L.ptr(c["eps"]), L.ptr(c["Wd"]), L.ptr(c["labels"]), L.ptr(c["klw"]),
                                      L.ptr(c["Wz"]), H2L, L.ptr(f["z"]), L.ptr(f["mu"]), L.ptr(f["logvar"]), L.ptr(f["hid"]),
                                      L.ptr(f["logits"]), L.ptr(c["d_hid"]), L.ptr(c["d_z_x"]), L.ptr(c["d_mu_x"]),
                                      L.ptr(c["d_lv_x"]), L.ptr(c["d_lg_x"]), L.ptr(g["d_w_c2p"]), L.ptr(g["d_b_c2p"]),
                                      L.ptr(g["d_w_dsc"]), L.ptr(g["d_b_dsc"]), L.ptr(g["d_w_z2h"]), L.ptr(g["d_b_z2h"]),
                                      L.ptr(g["d_ctx"]), L.ptr(ws), L.stream_ptr()), "heads bwd")
    return g


def _rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).abs().max() / max(float(b.abs().max()), 1e-30))


SHAPES = [
    (6, 32, [1, 2, 4], [1, 1, 0], 48),
    (128, 1024, [1, 1, 62], [1, 1, 0], 1024),      # cfg 2
    (9, 24, [2, 3], [3, 0], 48),
    (5, 16, [4], [0], 48),
    (1, 1000, [1, 1, 30], [1, 1, 0], 100),
    (130, 1000, [3, 1, 17], [4, 1, 0], 520),        # multi-class, Z = 21, B not a multiple of the rows per cluster
    (1024, 1024, [1, 1, 62], [1, 1, 0], 1024),      # cfg 5
    (128, 4096, [1, 1, 62], [1, 1, 0], 4096),       # cfg 4
]


@pytest.mark.parametrize("B,C,dims,dsc_out,H2L", SHAPES)
def test_heads_forward_backward(lib, L, B, C, dims, dsc_out, H2L):
    c = _case(B, C, dims, dsc_out, H2L, seed=B + C + H2L)
    want = _reference(c)
    S, OD = c["S"], c["OD"]
    ws = torch.zeros(lib.dvae_heads_ws_floats(B, S), device="cuda")
    f = _fwd(lib, L, c, ws)
    for k in ("z", "mu", "logvar", "hid"):
        assert _rel(f[k], want[k]) < 5e-6, k
    if OD:
        assert _rel(f["logits"][:, :OD], want["logits"]) < 5e-6
    sc = f["sc"].cpu().double()
    kl = want["kl"].cpu()
    assert (sc[3:3 + S] - kl).abs().max() < 1e-5 * max(1.0, float(kl.abs().max()))
    assert abs(float(sc[0]) - float((c["klw"].cpu().double() * kl).sum())) < 1e-5 * max(1.0, float(kl.sum()))
    assert abs(float(sc[1]) - float(kl.sum())) < 1e-5 * max(1.0, float(kl.sum()))
    i = 0
    for s, o in enumerate(dsc_out):
        if o == 0:
            assert sc[3 + S + s] == 0 and sc[3 + 2 * S + s] == 0
            continue
        assert abs(float(sc[3 + S + s]) - float(want["dls"][i])) < 1e-5
        assert abs(float(sc[3 + 2 * S + s]) - float(want["das"][i])) < 1e-6
        i += 1
    assert abs(float(sc[2]) - float(sum(want["dls"]) if want["dls"] else 0.0)) < 1e-5
    assert int(ws[:1].view(torch.int32).item()) == 0          # the arrival counter re-armed itself

    bws = torch.zeros(lib.dvae_heads_bwd_ws_floats(B, c["Z"], H2L), device="cuda")
    g = _bwd(lib, L, c, f, bws)
    torch.cuda.synchronize()
    for k in ("d_ctx", "d_w_c2p", "d_b_c2p", "d_w_z2h", "d_b_z2h"):
        assert _rel(g[k], want[k]) < 1e-4, k
    if OD:
        n_w = sum(o * z for o, z in zip(dsc_out, dims))
        assert _rel(g["d_w_dsc"][:n_w], want["d_w_dsc"]) < 1e-4
        assert _rel(g["d_b_dsc"][:OD], want["d_b_dsc"]) < 1e-4


@pytest.mark.parametrize("B,C,dims,dsc_out,H2L", [SHAPES[1], SHAPES[5]])
def test_heads_bit_reproducible_and_graph_replay(lib, L, B, C, dims, dsc_out, H2L):
    c = _case(B, C, dims, dsc_out, H2L, seed=7)
    ws = torch.zeros(lib.dvae_heads_ws_floats(B, c["S"]), device="cuda")
    bws = torch.zeros(lib.dvae_heads_bwd_ws_floats(B, c["Z"], H2L), device="cuda")
    runs = []
    for _ in range(2):
        f = _fwd(lib, L, c, ws)
        g = _bwd(lib, L, c, f, bws)
        runs.append((f["sc"].clone(), f["hid"].clone(), g["d_ctx"].clone()))
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        f = _fwd(lib, L, c, ws)         # warm-up on the capture stream (first-launch attributes)
        g = _bwd(lib, L, c, f, bws)
        side.synchronize()
        with torch.cuda.graph(graph, stream=side):
            f = _fwd(lib, L, c, ws)
            g = _bwd(lib, L, c, f, bws)
    torch.cuda.current_stream().wait_stream(side)
    for t in (f["sc"], f["hid"], g["d_ctx"]):
        t.zero_()
    graph.replay()
    torch.cuda.synchronize()
    runs.append((f["sc"].clone(), f["hid"].clone(), g["d_ctx"].clone()))
    for r in runs[1:]:
        for a, b in zip(runs[0], r):
            assert torch.equal(a, b)
    assert int(ws[:1].view(torch.int32).item()) == 0
