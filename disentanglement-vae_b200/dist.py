"""Data-parallel helpers (SURVEY.md 8e): the path shards over the batch dimension, one exchange per step.

Every loss term of the reference is a batch mean (`vae/losses.py:155`, texar `average_across_batch`, BCE mean), so
with equal shards   grad(global mean) = (1/world) * sum_r grad(mean over rank r's shard).
Rank r takes rows r::world of the global batch -- a strided split keeps `RatioSampler`'s per-source ratio inside
every shard because a batch is laid out [source 0 rows..., source 1 rows...] (`vae/data_utils.py:41-46`).
"""
import torch
import torch.distributed as dist


def shard_rows(n_rows, rank, world):
    """Row indices of the global batch owned by `rank`."""
    if n_rows % world != 0:
        raise ValueError(f"global batch {n_rows} is not divisible by world size {world}")
    return torch.arange(rank, n_rows, world)


def shard_batch(inputs, lengths, labels, rank, world):
    idx = shard_rows(inputs.size(0), rank, world)
    return inputs[idx], lengths[idx], {k: v[idx] for k, v in labels.items()}


def allreduce_mean_(flat, group=None):
    """In-place average of a flat gradient buffer over the process group (SUM then 1/world)."""
    world = dist.get_world_size(group)
    dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    flat.mul_(1.0 / world)
    return flat


def grad_buckets(model, flat_grad):
    """(decoder bucket, [remaining buckets]) as views of a flat gradient buffer laid out like `model._layout`.
    decoder.* is one contiguous range (named_parameters order) and its gradients are final as soon as the decoder's
    backward has run, so their all-reduce can overlap the heads' and the encoder's backward (engine.TrainEngine)."""
    lay, named = model._layout, dict(model.named_parameters())
    dec = [n for n in lay if n.startswith("decoder.")]
    lo = min(lay[n] for n in dec)
    hi = max((lay[n] + named[n].numel() + 3) // 4 * 4 for n in dec)
    n = flat_grad.numel()
    for name, off in lay.items():        # nothing else may live inside the decoder range
        if not name.startswith("decoder.") and lo <= off < hi:
            raise AssertionError(f"{name} lies inside the decoder gradient bucket")
    rest = [flat_grad[a:b] for a, b in ((0, lo), (hi, n)) if b > a]
    return flat_grad[lo:hi], rest


def allreduce_buckets_(flat_grad, buckets, group=None):
    """All-reduce (SUM) every bucket; together they cover `flat_grad` exactly once."""
    dec, rest = buckets
    dist.all_reduce(dec, op=dist.ReduceOp.SUM, group=group)
    for b in rest:
        dist.all_reduce(b, op=dist.ReduceOp.SUM, group=group)
    return flat_grad


def grad_buckets3(model, flat_grad):
    """Three exchange steps in the order the backward pass finishes gradients (engine.TrainEngine, world > 1):
      [0] decoder.*                                   -- final after the decoder backward
      [1] encoder layers >= 1 + z2hidden + heads      -- final after the heads' and the upper encoder layers' backward
      [2] encoder embedding + encoder layer 0         -- final at the end of the backward pass
    Each entry is a list of contiguous views of `flat_grad`; together they cover it exactly once."""
    lay, named = model._layout, dict(model.named_parameters())
    n = flat_grad.numel()
    end = {name: (off + named[name].numel() + 3) // 4 * 4 for name, off in lay.items()}

    def span(pred):
        names = [k for k in lay if pred(k)]
        if not names:
            return None
        lo, hi = min(lay[k] for k in names), max(end[k] for k in names)
        for k, off in lay.items():
            if not pred(k) and lo <= off < hi:
                raise AssertionError(f"{k} lies inside a gradient bucket it does not belong to")
        return lo, hi

    dec = span(lambda k: k.startswith("decoder."))
    low = span(lambda k: k.startswith("encoder.embedding.") or (k.startswith("encoder.recurrent.") and "_l0" in k))
    if dec is None or low is None or low[0] != 0:
        d, rest = grad_buckets(model, flat_grad)
        return [[d], rest, []]
    covered = sorted([dec, low])
    gaps, pos = [], 0
    for lo, hi in covered:
        if lo > pos:
            gaps.append((pos, lo))
        pos = max(pos, hi)
    if pos < n:
        gaps.append((pos, n))
    return [[flat_grad[dec[0]:dec[1]]], [flat_grad[a:b] for a, b in gaps if b > a], [flat_grad[low[0]:low[1]]]]


def grad_buckets4(model, flat_grad):
    """grad_buckets3 with the decoder bucket split in two: [0a] decoder.linear.* (W_out and its bias: final as soon as the
    vocabulary backward has run, before any recurrence of the backward pass) and [0b] the decoder's embedding and LSTM
    gradients.  The exchange of the 10 MB W_out gradient then starts ~250 us earlier in the step."""
    b = grad_buckets3(model, flat_grad)
    lay, named = model._layout, dict(model.named_parameters())
    lin = [k for k in lay if k.startswith("decoder.linear.")]
    if len(b[0]) != 1 or not lin:
        return [[], b[0], b[1], b[2]]
    dec = b[0][0]
    base = (dec.data_ptr() - flat_grad.data_ptr()) // 4
    lo = min(lay[k] for k in lin)
    hi = max((lay[k] + named[k].numel() + 3) // 4 * 4 for k in lin)
    if hi != base + dec.numel() or lo <= base:          # decoder.linear.* must be the tail of the decoder range
        return [[], b[0], b[1], b[2]]
    return [[flat_grad[lo:hi]], [flat_grad[base:lo]], b[1], b[2]]
