"""world_size-2 gloo test (CPU) of the data-parallel logic: strided sharding of the global batch, sum all-reduce
and 1/world scaling reproduce the single-process gradient of the global-batch loss (SURVEY.md 8e).  The per-rank
gradients come from the numpy oracle; on the GPU the same exchange runs over NCCL on the flat gradient buffer."""
import os
import socket
import sys

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import ROOT, load_golden, golden_state_dict


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    import importlib
    from oracle import dvae_oracle as O
    dvae_dist = importlib.import_module("disentanglement-vae_b200.dist")
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    g = load_golden("tiny_bi")
    sd = O.cast_state_dict(golden_state_dict(g))
    spec = O.ModelSpec(sd, [str(s) for s in g["space_names"]], int(g["sos"]), int(g["eos"]))
    X, L = torch.from_numpy(g["inputs"]), torch.from_numpy(g["lengths"])
    Y = {str(n): torch.from_numpy(g[f"Y.{n}"]) for n in g["label_names"]}
    eps_full = {n: g[f"eps.{n}"] for n in spec.space_names}
    klw = {n: float(g[f"klw.{n}"]) for n in spec.space_names}
    idx = dvae_dist.shard_rows(X.size(0), rank, world)
    Xs, Ls, Ys = dvae_dist.shard_batch(X, L, Y, rank, world)
    assert Xs.size(0) == X.size(0) // world and torch.equal(Xs, X[rank::world])
    fw = O.model_forward(sd, spec, Xs.numpy(), Ls.numpy(), {n: e[idx.numpy()] for n, e in eps_full.items()},
                         labels={k: v.numpy() for k, v in Ys.items()}, kl_weights=klw)
    grads = O.model_backward(sd, spec, fw)
    names = sorted(sd)
    flat = torch.from_numpy(np.concatenate([grads[k].reshape(-1) for k in names]))
    dvae_dist.allreduce_mean_(flat)
    loss = torch.tensor([fw["total_loss"]], dtype=torch.float64)
    dist.all_reduce(loss)
    if rank == 0:
        np.savez(os.path.join(out_dir, "ddp.npz"), flat=flat.numpy(), loss=loss.numpy() / world)
    dist.destroy_process_group()


def test_two_rank_gradient_average_equals_global_batch_gradient(tmp_path):
    from oracle import dvae_oracle as O
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    got = np.load(tmp_path / "ddp.npz")
    g = load_golden("tiny_bi")
    sd = O.cast_state_dict(golden_state_dict(g))
    spec = O.ModelSpec(sd, [str(s) for s in g["space_names"]], int(g["sos"]), int(g["eos"]))
    fw = O.model_forward(sd, spec, g["inputs"], g["lengths"], {n: g[f"eps.{n}"] for n in spec.space_names},
                         labels={str(n): g[f"Y.{n}"] for n in g["label_names"]},
                         kl_weights={n: float(g[f"klw.{n}"]) for n in spec.space_names})
    grads = O.model_backward(sd, spec, fw)
    want = np.concatenate([grads[k].reshape(-1) for k in sorted(sd)])
    assert np.abs(got["flat"] - want).max() < 1e-10 * max(1.0, np.abs(want).max())
    assert abs(float(got["loss"][0]) - fw["total_loss"]) < 1e-10
    # and the single-process result is the reference's own (golden) gradient
    ref = np.concatenate([g[f"grad.{k}"].reshape(-1) for k in sorted(sd)])
    assert np.abs(want - ref).max() < 2e-4 * np.abs(ref).max()


def test_shard_rows_rejects_uneven_split(dvae):
    import importlib
    d = importlib.import_module("disentanglement-vae_b200.dist")
    import pytest
    with pytest.raises(ValueError):
        d.shard_rows(7, 0, 2)
    assert d.shard_rows(8, 1, 4).tolist() == [1, 5]


def _bucket_worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    import importlib
    dvae = importlib.import_module("disentanglement-vae_b200")
    dvae_dist = importlib.import_module("disentanglement-vae_b200.dist")
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    p = dict(bow_encoder=False, embedding_dim=12, hidden_dim=16, num_rnn_layers=2, encoder_dropout=0.0, decoder_dropout=0.0,
             bidirectional_encoder=True, latent_dims={"total": 6, "polarity": 1}, adversarial_loss=False, mi_loss=False)
    dvae.set_seed(10)
    vae = dvae.build_vae(p, 41, None, {"polarity": 1}, torch.device("cpu"), 2, 3)      # CPU model: layout only, never run
    n = vae._flat_numel
    flat = torch.arange(n, dtype=torch.float32) * (rank + 1)
    buckets = dvae_dist.grad_buckets(vae, flat)
    dec, rest = buckets
    assert dec.numel() + sum(b.numel() for b in rest) == n                # the buckets tile the flat buffer
    named = dict(vae.named_parameters())
    assert dec.numel() >= sum(q.numel() for k, q in named.items() if k.startswith("decoder."))
    dvae_dist.allreduce_buckets_(flat, buckets)
    if rank == 0:
        np.save(os.path.join(out_dir, "buckets.npy"), flat.numpy())
    dist.destroy_process_group()


def test_bucketed_allreduce_covers_flat_gradient_exactly_once(tmp_path):
    """The engine all-reduces the decoder bucket early (overlapping encoder backward) and the rest afterwards: summed
    over 2 gloo ranks every element of the flat gradient must come out as (1 + 2) x its single-rank value."""
    world = 2
    mp.spawn(_bucket_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    got = np.load(tmp_path / "buckets.npy")
    assert np.array_equal(got, np.arange(got.size, dtype=np.float32) * 3)


def test_three_bucket_split_covers_flat_gradient_exactly_once(dvae):
    """grad_buckets3: decoder | upper encoder layers + heads | encoder embedding + layer 0 -- disjoint, complete, and every
    parameter's gradient lies in the bucket of the backward phase that produces it."""
    import importlib
    dvae_dist = importlib.import_module("disentanglement-vae_b200.dist")
    p = dict(bow_encoder=False, embedding_dim=12, hidden_dim=16, num_rnn_layers=2, encoder_dropout=0.0, decoder_dropout=0.0,
             bidirectional_encoder=True, latent_dims={"total": 7, "polarity": 1, "uncertainty": 2}, adversarial_loss=False, mi_loss=False)
    vae = dvae.build_vae(p, 29, None, {"uncertainty": 3, "polarity": 1}, torch.device("cpu"), 2, 3)
    n = vae._flat_numel
    flat = torch.zeros(n)
    buckets = dvae_dist.grad_buckets3(vae, flat)
    assert len(buckets) == 3 and all(len(b) >= 1 for b in buckets)
    for i, views in enumerate(buckets):
        for v in views:
            v += 1.0
            assert v.data_ptr() % 16 == 0
    assert torch.equal(flat, torch.ones(n))                      # every element in exactly one bucket
    named = dict(vae.named_parameters())
    marks = torch.zeros(n)
    for i, views in enumerate(buckets):
        for v in views:
            off = (v.data_ptr() - flat.data_ptr()) // 4
            marks[off:off + v.numel()] = i
    for name, off in vae._layout.items():
        want = 0 if name.startswith("decoder.") else (2 if name.startswith("encoder.embedding") or "_l0" in name else 1)
        got = marks[off:off + named[name].numel()]
        assert (got == want).all(), (name, want, got.unique())


def test_four_stage_split_puts_the_output_layer_first(dvae):
    import importlib
    dvae_dist = importlib.import_module("disentanglement-vae_b200.dist")
    p = dict(bow_encoder=False, embedding_dim=12, hidden_dim=16, num_rnn_layers=2, encoder_dropout=0.0, decoder_dropout=0.0,
             bidirectional_encoder=True, latent_dims={"total": 7, "polarity": 1, "uncertainty": 2}, adversarial_loss=False, mi_loss=False)
    vae = dvae.build_vae(p, 29, None, {"uncertainty": 3, "polarity": 1}, torch.device("cpu"), 2, 3)
    flat = torch.zeros(vae._flat_numel)
    b = dvae_dist.grad_buckets4(vae, flat)
    assert len(b) == 4
    for views in b:
        for v in views:
            v += 1.0
    assert torch.equal(flat, torch.ones_like(flat))
    named = dict(vae.named_parameters())
    n_lin = sum(named[k].numel() for k in named if k.startswith("decoder.linear."))
    assert sum(v.numel() for v in b[0]) >= n_lin and sum(v.numel() for v in b[0]) <= n_lin + 8
    off = vae._layout["decoder.linear.weight"]
    assert b[0][0].data_ptr() == flat.data_ptr() + 4 * off


def test_two_stage_split_covers_flat_gradient_exactly_once(dvae):
    """stage_buckets of a two-stage step (bag-of-words and one-layer encoders): decoder.* | everything else."""
    import importlib
    dvae_dist = importlib.import_module("disentanglement-vae_b200.dist")
    for bow, layers in ((True, 1), (False, 1)):
        p = dict(bow_encoder=bow, embedding_dim=12, hidden_dim=16, num_rnn_layers=layers, encoder_dropout=0.0,
                 decoder_dropout=0.0, bidirectional_encoder=True, latent_dims={"total": 7, "polarity": 1, "uncertainty": 2},
                 adversarial_loss=False, mi_loss=False)
        vae = dvae.build_vae(p, 29, None, {"uncertainty": 3, "polarity": 1}, torch.device("cpu"), 2, 3)
        flat = torch.zeros(vae._flat_numel)
        buckets = dvae_dist.stage_buckets(vae, flat, 2)
        assert len(buckets) == 2
        named = dict(vae.named_parameters())
        for i, views in enumerate(buckets):
            for v in views:
                v += 1.0
                off = (v.data_ptr() - flat.data_ptr()) // 4
                for name, o in vae._layout.items():
                    if off <= o < off + v.numel():
                        assert name.startswith("decoder.") == (i == 0), (bow, name, i)
        assert torch.equal(flat, torch.ones_like(flat))              # every element in exactly one bucket
        assert sum(v.numel() for v in buckets[0]) >= sum(q.numel() for k, q in named.items() if k.startswith("decoder."))
