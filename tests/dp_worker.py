"""Worker of tests/test_gpu_dp.py, launched by `python -m torch.distributed.run` with one rank per GPU.

Every rank builds the same model, takes its strided shard of a seeded GLOBAL batch and runs K steps of the
data-parallel TrainEngine (CUDA graphs + bucketed gradient exchange, exactly what bench.py times at N > 1) with
dropout off and the reparameterisation noise given, so that the run is comparable with a single-process engine on the
whole batch.  Rank 0 writes the final weights and per-step losses."""
import importlib
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def make_cfg():
    return dict(bow_encoder=False, embedding_dim=256, hidden_dim=256, num_rnn_layers=2, encoder_dropout=0.0,
                decoder_dropout=0.0, bidirectional_encoder=True, latent_dims={"total": 16, "polarity": 1, "uncertainty": 1},
                adversarial_loss=False, mi_loss=False, learn_rate=3e-3, teacher_forcing_prob=1.0, random_seed=10,
                lambdas={"default": "cyclic", "polarity": 0.005, "uncertainty": 0.005})


V, T, GLOBAL_B, STEPS, TOTAL = 2000, 12, 64, 3, 40


def global_batches():
    gen = torch.Generator().manual_seed(123)
    out = []
    for _ in range(STEPS):
        lengths = torch.randint(3, T + 1, (GLOBAL_B,), generator=gen)
        lengths[0] = T
        X = torch.zeros(GLOBAL_B, T, dtype=torch.long)
        for b in range(GLOBAL_B):
            n = int(lengths[b])
            X[b, 0], X[b, n - 1] = 2, 3
            X[b, 1:n - 1] = torch.randint(4, V, (n - 2,), generator=gen)
        Y = {k: (torch.rand(GLOBAL_B, 1, generator=gen) < 0.3).float() for k in ("uncertainty", "polarity")}
        eps = torch.randn(GLOBAL_B, 16, generator=gen)
        out.append((X, lengths, Y, eps))
    return out


def run(world, rank, dev, use_graph=True):
    import __graft_entry__ as ge
    dvae = ge.build()
    engine_mod = importlib.import_module("disentanglement-vae_b200.engine")
    dvae_dist = importlib.import_module("disentanglement-vae_b200.dist")
    cfg = make_cfg()
    dvae.set_seed(10)
    vae = dvae.build_vae(cfg, V, None, {"uncertainty": 1, "polarity": 1}, dev, 2, 3)
    vae.train()
    eng = engine_mod.TrainEngine(vae, cfg, GLOBAL_B // world, T, total_steps=TOTAL, use_graph=use_graph)
    losses = []
    for X, L, Y, eps in global_batches():
        if world > 1:
            idx = dvae_dist.shard_rows(GLOBAL_B, rank, world)
            Xs, Ls, Ys = dvae_dist.shard_batch(X, L, Y, rank, world)
            eps = eps[idx]
        else:
            Xs, Ls, Ys = X, L, Y
        eng.fixed_eps = eps.to(dev)
        out = eng.step_host(Xs, Ls, Ys)
        losses.append(out["total_loss"])
    return vae, eng, losses


def main():
    out_path = sys.argv[1]
    world = int(os.environ["WORLD_SIZE"])
    rank = int(os.environ["RANK"])
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    dist.init_process_group("nccl", device_id=dev)
    vae, eng, losses = run(world, rank, dev)
    # the global loss is the mean of the shard losses (every term is a batch mean over equal shards)
    lt = torch.tensor(losses, dtype=torch.float64, device=dev)
    dist.all_reduce(lt)
    lt /= world
    # replicas must stay bit-identical: same all-reduced gradient, same Adam
    flat = vae._flat.detach()
    ref = flat.clone()
    dist.broadcast(ref, 0)
    same = torch.tensor([1.0 if torch.equal(ref, flat) else 0.0], device=dev)
    dist.all_reduce(same, op=dist.ReduceOp.MIN)
    if rank == 0:
        np.savez(out_path, flat=flat.cpu().numpy(), losses=lt.cpu().numpy(), replicas_identical=same.cpu().numpy(), exchange=np.array(eng.exchange_mode),
                 adam_step=np.int64(eng.adam_step))
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
