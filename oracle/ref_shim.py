"""Import shim that lets the UNMODIFIED reference (`/root/reference/vae`) import on this image.

TEST INFRASTRUCTURE ONLY.  Nothing under `oracle/` is on the product path; only `tests/`,
`__graft_entry__.smoke()` and `bench.py`'s CPU-baseline legs may import it.

The reference imports two packages at module top that are not installed here
(`/root/reference/vae/losses.py:4-5`):

* `texar.torch` -- only `tx.losses.sequence_sparse_softmax_cross_entropy` is used
  (`/root/reference/vae/losses.py:138-139`), with texar-pytorch's documented defaults
  (`average_across_batch=True, sum_over_timesteps=True`): log_softmax over the vocab axis,
  NLL at the label, mask `t < sequence_length`, sum over time, mean over batch.  texar is an
  UNPINNED dependency (`/root/reference/requirements.txt:4`) that is absent from
  `/root/reference`, so this 6-line restatement of its published behaviour *is* the spec at
  that boundary ("parity unpinned" for that one function; everything else is pinned by running
  the reference itself).
* `torchtext.data.metrics.bleu_score` -- logging only (`/root/reference/vae/losses.py:133`);
  stubbed to 0.0.

The reference is not part of this repository (point DVAE_REFERENCE_ROOT at a checkout of it).  The
only caller of `load_reference()` is `tests/golden/make_golden.py`, which stores what the reference
computes under `tests/golden/`; the tests compare against those files and never import the reference.
"""
import os
import sys
import types

REFERENCE_ROOT = os.environ.get("DVAE_REFERENCE_ROOT", "/root/reference")


def _seq_sparse_softmax_xent(labels, logits, sequence_length,
                             average_across_batch=True, sum_over_timesteps=True, **_):
    import torch
    logp = torch.log_softmax(logits, dim=-1)
    nll = -logp.gather(-1, labels.unsqueeze(-1)).squeeze(-1)          # [B, T]
    steps = torch.arange(logits.size(1), device=logits.device).unsqueeze(0)
    mask = (steps < sequence_length.to(logits.device).unsqueeze(1)).to(nll.dtype)
    per_seq = (nll * mask).sum(dim=1)                                  # sum over timesteps
    return per_seq.mean()                                              # mean over batch


def install_stubs():
    if "texar.torch" not in sys.modules:
        texar = types.ModuleType("texar")
        tx = types.ModuleType("texar.torch")
        tx_losses = types.ModuleType("texar.torch.losses")
        tx_losses.sequence_sparse_softmax_cross_entropy = _seq_sparse_softmax_xent
        tx.losses = tx_losses
        texar.torch = tx
        sys.modules["texar"] = texar
        sys.modules["texar.torch"] = tx
        sys.modules["texar.torch.losses"] = tx_losses
    if "torchtext.data.metrics" not in sys.modules:
        tt = types.ModuleType("torchtext")
        ttd = types.ModuleType("torchtext.data")
        ttm = types.ModuleType("torchtext.data.metrics")
        ttm.bleu_score = lambda *a, **k: 0.0
        tt.data = ttd
        ttd.metrics = ttm
        sys.modules["torchtext"] = tt
        sys.modules["torchtext.data"] = ttd
        sys.modules["torchtext.data.metrics"] = ttm


def reference_available():
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "vae"))


def load_reference():
    """Returns the reference's (model, losses, utils) modules, imported unmodified."""
    if not reference_available():
        raise RuntimeError(f"reference not present at {REFERENCE_ROOT}")
    install_stubs()
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    import importlib
    model = importlib.import_module("vae.model")
    losses = importlib.import_module("vae.losses")
    utils = importlib.import_module("vae.utils")
    return model, losses, utils
