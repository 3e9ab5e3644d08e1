"""Worker of tests/test_gpu_engine_shapes.py, launched by `python -m torch.distributed.run` with one rank per GPU.

Every rank takes its strided shard of three seeded GLOBAL batches -- full, short and narrow (a RatioSampler epoch's last
batch, cut to a multiple of the world size), full -- through the data-parallel TrainEngine with dropout off and the
reparameterisation noise given.  Rank 0 writes the final weights, the per-step global losses and whether the replicas
are bit-identical.  `run(1, 0, dev)` is the single-engine reference on the global batches."""
import importlib
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

V, T, GLOBAL_B, TOTAL = 2000, 12, 64, 40
SHAPES = ((GLOBAL_B, T), (22, 9), (GLOBAL_B, T))


def make_cfg():
    return dict(bow_encoder=False, embedding_dim=256, hidden_dim=256, num_rnn_layers=2, encoder_dropout=0.0,
                decoder_dropout=0.0, bidirectional_encoder=True, latent_dims={"total": 16, "polarity": 1, "uncertainty": 1},
                adversarial_loss=False, mi_loss=False, learn_rate=3e-3, teacher_forcing_prob=1.0, random_seed=10,
                lambdas={"default": "cyclic", "polarity": 0.005, "uncertainty": 0.005})


def global_batches():
    gen = torch.Generator().manual_seed(321)
    out = []
    for Bg, Tg in SHAPES:
        lengths = torch.randint(3, Tg + 1, (Bg,), generator=gen)
        lengths[0] = Tg
        X = torch.zeros(Bg, Tg, dtype=torch.long)
        for b in range(Bg):
            n = int(lengths[b])
            X[b, 0], X[b, n - 1] = 2, 3
            X[b, 1:n - 1] = torch.randint(4, V, (n - 2,), generator=gen)
        Y = {k: (torch.rand(Bg, 1, generator=gen) < 0.3).float() for k in ("uncertainty", "polarity")}
        out.append((X, lengths, Y, torch.randn(Bg, 16, generator=gen)))
    return out


def run(world, rank, dev):
    import __graft_entry__ as ge
    dvae = ge.build()
    engine_mod = importlib.import_module("disentanglement-vae_b200.engine")
    dvae_dist = importlib.import_module("disentanglement-vae_b200.dist")
    dvae.set_seed(10)
    vae = dvae.build_vae(make_cfg(), V, None, {"uncertainty": 1, "polarity": 1}, dev, 2, 3)
    vae.train()
    w0 = vae._flat.detach().clone()
    eng = engine_mod.TrainEngine(vae, make_cfg(), GLOBAL_B // world, T, total_steps=TOTAL)
    eng.fixed_eps = torch.zeros(GLOBAL_B // world, 16, device=dev)      # the captured graphs read it in place
    losses = []
    for X, L, Y, eps in global_batches():
        idx = dvae_dist.shard_rows(X.shape[0], rank, world)
        Xs, Ls, Ys = dvae_dist.shard_batch(X, L, Y, rank, world) if world > 1 else (X, L, Y)
        eng.fixed_eps[:len(idx)].copy_(eps[idx])
        losses.append(eng.step_host(Xs, Ls, Ys)["total_loss"])
    return vae, eng, losses, w0


def main():
    out_path = sys.argv[1]
    world = int(os.environ["WORLD_SIZE"])
    rank = int(os.environ["RANK"])
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    vae, eng, losses, _ = run(world, rank, dev)
    lt = torch.tensor(losses, dtype=torch.float64, device=dev)      # equal shards: the global loss is the shards' mean
    dist.all_reduce(lt)
    lt /= world
    flat = vae._flat.detach()
    ref = flat.clone()
    dist.broadcast(ref, 0)
    same = torch.tensor([1.0 if torch.equal(ref, flat) else 0.0], device=dev)
    dist.all_reduce(same, op=dist.ReduceOp.MIN)
    if rank == 0:
        np.savez(out_path, flat=flat.cpu().numpy(), losses=lt.cpu().numpy(), replicas_identical=same.cpu().numpy(),
                 exchange=np.array(eng.exchange_mode))
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
