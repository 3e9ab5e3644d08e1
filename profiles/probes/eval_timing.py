"""Cost of validation at the cfg-2 shape (B = 128, T = 22, V = 10k, E = H = 256): TrainEngine.eval_step against the
drop-in eval pattern it replaces (run.py:evalstep: vae.eval(), a no_grad forward, compute_all_losses, compute_bleu), and
the two BLEU kernels alone at B = 1024, T = 22.  CUDA events for device time; host wall clock around synchronised loops
for the per-call cost a training script sees.  Prints one JSON object (and writes it to argv[1] if given)."""
import importlib
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench as BN  # noqa: E402
import __graft_entry__ as ge  # noqa: E402

dvae = ge.build()
engine_mod = importlib.import_module("disentanglement-vae_b200.engine")
assert torch.cuda.is_available(), "eval_timing.py measures on the GPU"
dev = torch.device("cuda", 0)
N_REP, N_WALL = 200, 100


def device_ms(fn, n=N_REP):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def wall_ms(fn, n=N_WALL):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(n):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3 / n


smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
res = {"gpu": smi[0] if smi else torch.cuda.get_device_name(0), "shape": "cfg2: B=128, T=22, V=10000, E=H=256, 2-layer biLSTM"}

dvae.set_seed(10)
vae = dvae.build_vae(BN.CFG2, BN.VOCAB, None, BN.LABELS, dev, BN.SOS, BN.EOS)
vae.train()
B, T = BN.BATCH, BN.SEQ_T
rng = np.random.default_rng(5)
X, L, Y = BN.synth_batch(rng, B)
Xt, Lt = torch.from_numpy(X), torch.from_numpy(L)
Yd = {n: torch.from_numpy(Y[i]).reshape(-1, 1) for i, n in enumerate(BN.LABELS)}
eng = engine_mod.TrainEngine(vae, BN.CFG2, B, T, total_steps=BN.TOTAL_STEPS)
for _ in range(3):
    eng.step_host(Xt, Lt, Yd)
for tf in (1.0, 0.0):
    for _ in range(3):
        eng.eval_step(Xt, Lt, Yd, teacher_forcing_prob=tf)
    g = eng._eval["graphs"][tf < 1.0]
    res[f"eval_step_tf{tf:g}_graph_device_ms"] = device_ms(g.replay)
    res[f"eval_step_tf{tf:g}_call_wall_ms"] = wall_ms(lambda: eng.eval_step(Xt, Lt, Yd, teacher_forcing_prob=tf))
    res[f"eval_steps_tf{tf:g}_pipelined_wall_ms_per_batch"] = wall_ms(
        lambda: list(eng.eval_steps([(Xt, Lt, Yd)] * 20, teacher_forcing_prob=tf)), 5) / 20

# the drop-in pattern of run.py:evalstep (run.py:347-423) through the autograd module
Xd, Ld = Xt.to(dev), Lt.to(dev)
klw = {"default": 1.0, "polarity": 0.005, "uncertainty": 0.005}


def dropin(tf):
    vae.eval()
    with torch.no_grad():
        out = vae(Xd, Ld, teacher_forcing_prob=tf)
        total, Ls = dvae.losses.compute_all_losses(vae, out, Xd, Yd, Ld, klw)
        total.item()
        dvae.losses.compute_bleu(Xd, out["token_predictions"], None, BN.EOS)


for tf in (1.0, 0.0):
    for _ in range(3):
        dropin(tf)
    res[f"dropin_eval_tf{tf:g}_wall_ms"] = wall_ms(lambda: dropin(tf))
vae.train()

# the BLEU kernels alone
Bb = 1024
R = torch.from_numpy(BN.synth_batch(rng, Bb)[0]).to(dev)
C = R.clone()
C[:, 2::3] = torch.from_numpy(rng.integers(4, BN.VOCAB, size=C[:, 2::3].shape)).to(dev)
counts = torch.zeros(10, device=dev, dtype=torch.int64)
score = torch.empty(1, device=dev)


def bleu_pair():
    dvae.losses.bleu_counts_(counts, R, C, BN.EOS)
    dvae.losses.bleu_score_(score, counts)


for _ in range(10):
    bleu_pair()
res["bleu_counts_plus_score_B1024_T22_device_us"] = device_ms(bleu_pair, 1000) * 1e3
res["note"] = ("device_ms: CUDA events around back-to-back launches / graph replays; wall_ms: host clock around a "
               "synchronised loop of whole calls (includes staging, H2D / D2H copies and host work)")
print(json.dumps(res, indent=1))
if len(sys.argv) > 1:
    os.makedirs(os.path.dirname(os.path.abspath(sys.argv[1])), exist_ok=True)
    with open(sys.argv[1], "w") as f:
        json.dump(res, f, indent=1)
