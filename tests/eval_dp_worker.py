"""Worker of tests/test_gpu_eval.py (data-parallel evaluation), launched by `python -m torch.distributed.run` with one
rank per GPU.  Every rank builds the same model and evaluates its strided shard of a seeded global batch, teacher-forced
(noise given, so comparable with one engine on the whole batch) and with sampled decoding (tf = 0).  Rank 0 writes the
all-reduced losses, BLEU and counts, and the gathered inputs and predictions."""
import importlib
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import dp_worker  # noqa: E402


def run(world, rank, dev):
    import __graft_entry__ as ge
    dvae = ge.build()
    engine_mod = importlib.import_module("disentanglement-vae_b200.engine")
    dvae_dist = importlib.import_module("disentanglement-vae_b200.dist")
    cfg = dict(dp_worker.make_cfg(), encoder_dropout=0.5, decoder_dropout=0.5)      # ignored in evaluation
    dvae.set_seed(10)
    vae = dvae.build_vae(cfg, dp_worker.V, None, {"uncertainty": 1, "polarity": 1}, dev, 2, 3)
    B = dp_worker.GLOBAL_B
    eng = engine_mod.TrainEngine(vae, cfg, B // world, dp_worker.T, total_steps=dp_worker.TOTAL)
    X, L, Y, eps = dp_worker.global_batches()[0]
    if world > 1:
        idx = dvae_dist.shard_rows(B, rank, world)
        X, L, Y = dvae_dist.shard_batch(X, L, Y, rank, world)
        eps = eps[idx]
    eng.fixed_eps = eps.to(dev)
    forced = eng.eval_step(X, L, Y, teacher_forcing_prob=1.0)
    sampled = eng.eval_step(X, L, Y, teacher_forcing_prob=0.0)
    return dict(forced=forced, sampled=sampled, inputs=X.to(dev), preds=eng.eval_predictions.clone())


def main():
    out_path = sys.argv[1]
    world = int(os.environ["WORLD_SIZE"])
    rank = int(os.environ["RANK"])
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    r = run(world, rank, dev)
    inputs = [torch.empty_like(r["inputs"]) for _ in range(world)]
    preds = [torch.empty_like(r["preds"]) for _ in range(world)]
    dist.all_gather(inputs, r["inputs"].contiguous())
    dist.all_gather(preds, r["preds"].contiguous())
    if rank == 0:
        f, s = r["forced"], r["sampled"]
        np.savez(out_path, total_loss=f["total_loss"], reconstruction_loss=f["reconstruction_loss"], total_kl=f["total_kl"],
                 total_dsc_loss=f["total_dsc_loss"], bleu_forced=f["bleu"], bleu_sampled=s["bleu"],
                 counts_sampled=np.array(s["bleu_counts"], np.int64), inputs=torch.cat(inputs).cpu().numpy(),
                 preds=torch.cat(preds).cpu().numpy())
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
