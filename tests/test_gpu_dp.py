"""Hardware data-parallel parity (SURVEY.md 4(iv), VERDICT r1 "next 1b"): N ranks x (B/N) rows through the data-parallel
TrainEngine must take the same optimisation steps as ONE engine on the concatenated batch, for every gradient exchange
the engine has: the repo's all-reduce kernel inside a one-graph step (peer-to-peer loads / stores at N = 2, NVSwitch
multicast at N = 4) and the NCCL fallback between four stage graphs.  Also the exchange kernel on its own, both
variants, against exact sums.  Spawns `torch.distributed.run`; skipped with < 2 GPUs."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


EXCHANGES = {                      # environment of the worker -> which exchange the engine uses
    "default": {},
    "nccl_stages": {"DVAE_DP_NVLS": "0"},
}


def _torchrun(world, script, *args, env=None, timeout=900):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(ROOT, "tests", script)] + [str(a) for a in args]
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=timeout, env=e)


@pytest.mark.parametrize("world", [2, 4])
def test_all_reduce_kernel_gives_exact_sums_on_every_rank(world):
    """csrc/nvls.cu on its own: both variants, bucket sizes from one float4 to 14 MB, unaligned tails of the slices,
    untouched guard words behind the bucket, repeated calls on the same barrier block (tests/xchg_worker.py)."""
    if not torch.cuda.is_available() or torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    r = _torchrun(world, "xchg_worker.py")
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "XCHG_OK" in r.stdout, r.stdout[-2000:]


@pytest.mark.parametrize("world,exchange", [(2, "default"), (2, "nccl_stages"), (4, "default")])
def test_n_rank_engine_equals_single_rank_on_the_global_batch(tmp_path, world, exchange):
    if not torch.cuda.is_available() or torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    out = tmp_path / f"dp{world}.npz"
    r = _torchrun(world, "dp_worker.py", out, env=EXCHANGES[exchange])
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    got = np.load(out)
    want_mode = {"default": "p2p" if world == 2 else "nvls", "nccl_stages": "nccl+stages"}[exchange]
    assert str(got["exchange"]) == want_mode, (str(got["exchange"]), want_mode)
    assert got["replicas_identical"][0] == 1.0, "ranks diverged: parameters differ after the all-reduced steps"
    import dp_worker
    vae, eng, losses = dp_worker.run(1, 0, torch.device("cuda", 0))
    want = vae._flat.detach().cpu().numpy()
    assert int(got["adam_step"]) == eng.adam_step == dp_worker.STEPS
    for a, b in zip(got["losses"], losses):
        assert abs(a - b) <= 1e-5 * abs(b), (got["losses"], losses)
    # post-Adam weights: SURVEY 4(iv) asks 2e-3; Adam turns noise-level gradients into +-lr moves, so the bound is on the
    # update relative to the largest update, over entries that moved at all
    import importlib
    dvae = importlib.import_module("disentanglement-vae_b200")
    dvae.set_seed(10)
    w0 = dvae.build_vae(dp_worker.make_cfg(), dp_worker.V, None, {"uncertainty": 1, "polarity": 1}, torch.device("cuda", 0), 2, 3)
    w0 = w0._flat.detach().cpu().numpy()[:want.size]
    upd_want, upd_got = want - w0, got["flat"][:want.size] - w0
    scale = np.abs(upd_want).max()
    frac_bad = (np.abs(upd_got - upd_want) > 2e-3 * scale).mean()
    assert frac_bad < 2e-3, frac_bad
    assert np.abs(upd_got - upd_want).mean() < 1e-3 * np.abs(upd_want).mean()
