"""Cost of TrainEngine's batch shapes at cfg 2 and cfg 4 (bench.py's workloads): device time of a replayed full-shape step
and of a short-batch step (B' = B/3, padded length T), host wall time of the first step of a new shape (plan
allocation, eager warm-up, capture and the step itself), and the device memory one extra shape holds (its StepPlan,
staging block and captured graph: torch's allocator, whose graph pools count as reserved).  Prints one JSON object
(and writes it to argv[1] if given), with the card's name and power limit read in the same run."""
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
assert torch.cuda.is_available(), "shape_timing.py measures on the GPU"
dev = torch.device("cuda", 0)
N_REP = 100


def device_ms(fn, n=N_REP):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
res = {"gpu": smi[0] if smi else torch.cuda.get_device_name(0)}

for wl in ("cfg2", "cfg4"):
    uni = BN.select_workload(wl)
    B, T = BN.BATCH, BN.SEQ_T
    Bs = B // 3
    dvae.set_seed(10)
    vae = dvae.build_vae(BN.CFG2, BN.VOCAB, None, BN.LABELS, dev, BN.SOS, BN.EOS)
    vae.train()
    rng = np.random.default_rng(5)

    def dev_batch(b):
        X, L, Y = BN.synth_batch(rng, b, uniform_lengths=uni)
        return torch.from_numpy(X).to(dev), torch.from_numpy(L).to(dev), torch.from_numpy(Y).to(dev)
    full, short = dev_batch(B), dev_batch(Bs)
    eng = engine_mod.TrainEngine(vae, BN.CFG2, B, T, total_steps=BN.TOTAL_STEPS)
    for _ in range(3):
        eng.step_resident(*full)
    torch.cuda.synchronize()
    r = {"B": B, "T": T, "B_short": Bs}
    r["full_step_device_ms"] = device_ms(lambda: eng.step_resident(*full))
    alloc0, resv0 = torch.cuda.memory_allocated(dev), torch.cuda.memory_reserved(dev)
    t0 = time.perf_counter()
    eng.step_resident(*short)
    torch.cuda.synchronize()
    r["first_short_step_wall_ms"] = (time.perf_counter() - t0) * 1e3
    r["extra_shape_allocated_MB"] = (torch.cuda.memory_allocated(dev) - alloc0) / 2 ** 20
    r["extra_shape_reserved_MB"] = (torch.cuda.memory_reserved(dev) - resv0) / 2 ** 20
    r["short_step_device_ms"] = device_ms(lambda: eng.step_resident(*short))
    r["full_step_after_short_device_ms"] = device_ms(lambda: eng.step_resident(*full))
    res[wl] = r
    del eng, vae
    torch.cuda.synchronize()
    torch.cuda.empty_cache()

res["note"] = ("device_ms: CUDA events around back-to-back step_resident calls (graph replays; L2 not flushed); "
               "first_short_step_wall_ms: host clock around the first step of a new shape, ending in a synchronise")
print(json.dumps(res, indent=1))
if len(sys.argv) > 1:
    os.makedirs(os.path.dirname(os.path.abspath(sys.argv[1])), exist_ok=True)
    with open(sys.argv[1], "w") as f:
        json.dump(res, f, indent=1)
