"""Drop-in replacement for `vae/losses.py` (loss surface of jvasilakes/disentanglement-vae).

Same function names, arguments and returned dict keys (vae/losses.py:137-242).  When handed the
outputs of this package's `VariationalSeq2Seq.forward` the heavy terms come straight from the
fused kernels: the reconstruction loss from the vocab-CE kernel (logits never materialised), the
per-space KL from the fused-heads kernel, the discriminator losses from `dvae_dsc_loss`.
"""
import math

import torch
import torch.nn as nn

from . import _lib
from .model import FusedLogits, LatentParams, DscLogits


class CLUB(nn.Module):
    """CLUB upper bound on I(X;Y) with a variational q(Y|X) (Cheng et al., ICML 2020; vae/losses.py:10-74).  The
    nn.Sequential members are parameter containers with the reference's names and initialisation; the arithmetic runs
    in the C-ABI kernels (dvae_linear, dvae_relu / dvae_act_bwd, dvae_club_mi, dvae_club_nll)."""

    def __init__(self, x_dim, y_dim, hidden_size):
        super().__init__()
        self.p_mu = nn.Sequential(nn.Linear(x_dim, hidden_size // 2), nn.ReLU(), nn.Linear(hidden_size // 2, y_dim))
        self.p_logvar = nn.Sequential(nn.Linear(x_dim, hidden_size // 2), nn.ReLU(), nn.Linear(hidden_size // 2, y_dim),
                                      nn.Tanh())
        self.optimizer = torch.optim.Adam(self.parameters(), lr=5e-4)      # vae/losses.py:41

    def optimizer_step(self, loss):
        self.optimizer.zero_grad()
        loss.backward()
        torch.nn.utils.clip_grad_norm_(self.parameters(), 1.0)
        self.optimizer.step()

    def get_mu_logvar(self, x_samples):
        from .functions import _SmallLinearFn
        h = _SmallLinearFn.apply(x_samples, self.p_mu[0].weight, self.p_mu[0].bias, 2)
        mu = _SmallLinearFn.apply(h, self.p_mu[2].weight, self.p_mu[2].bias, 0)
        h = _SmallLinearFn.apply(x_samples, self.p_logvar[0].weight, self.p_logvar[0].bias, 2)
        logvar = _SmallLinearFn.apply(h, self.p_logvar[2].weight, self.p_logvar[2].bias, 1)
        return mu, logvar

    def forward(self, x_samples, y_samples):
        from .functions import _ClubMiFn
        mu, logvar = self.get_mu_logvar(x_samples)
        return _ClubMiFn.apply(mu, logvar, y_samples)

    def loglikeli(self, x_samples, y_samples):
        return -self.learning_loss(x_samples, y_samples)

    def learning_loss(self, x_samples, y_samples):
        from .functions import _ClubNllFn
        mu, logvar = self.get_mu_logvar(x_samples)
        return _ClubNllFn.apply(mu, logvar, y_samples)


def reconstruction_loss(targets, logits, target_lengths):
    """vae/losses.py:137-140 (texar sequence_sparse_softmax_cross_entropy defaults: sum over
    time, mean over batch, positions t < length)."""
    if not isinstance(logits, FusedLogits):
        raise _lib.DvaeError("reconstruction_loss expects the `decoder_logits` returned by the B200 model "
                             "(a FusedLogits); dense logits are only available via .materialize()")
    from .functions import reconstruction_loss_fused
    return {"reconstruction_loss": reconstruction_loss_fused(logits, targets, target_lengths)}


def get_cyclic_kl_weight(step, total_steps, cycles=4, rate=0.5):
    """vae/losses.py:143-150: linear ramp over the first `rate` of each of `cycles` periods."""
    period = total_steps / cycles
    tau = (step % math.ceil(period)) / period
    return tau / rate if tau <= rate else 1


def kl_divergence(mu, logvar):
    """vae/losses.py:153-156 on arbitrary tensors (not on the fused path; kept for API parity)."""
    return (0.5 * (torch.exp(logvar) + mu * mu - 1 - logvar)).mean(0).sum()


def compute_kl_divergence_losses(model, latent_params, kl_weights_dict):
    """vae/losses.py:159-177.  One host read for all per-space values instead of one per space."""
    names = list(latent_params.keys())
    if isinstance(latent_params, LatentParams) and latent_params.kl is not None:
        kl_vec = latent_params.kl
    else:
        kl_vec = torch.stack([kl_divergence(p.mu, p.logvar) for p in latent_params.values()])
    weights = [kl_weights_dict[n] if n in kl_weights_dict else kl_weights_dict["default"] for n in names]
    w = torch.tensor(weights, dtype=torch.float32).to(kl_vec.device, non_blocking=True)
    total_weighted_kl = (kl_vec * w).sum()
    vals = kl_vec.detach().tolist()
    idv_kls = dict(zip(names, vals))
    return {"total_weighted_kl": total_weighted_kl, "total_kl": float(sum(vals)), "idv_kls": idv_kls}


def _pack_labels(names, Ybatch, device):
    rows = [Ybatch[n].to(device=device, dtype=torch.float32).reshape(-1) for n in names]
    return torch.stack(rows).contiguous()


def compute_discriminator_losses(model, discriminator_logits, Ybatch):
    """vae/losses.py:180-196."""
    names = list(discriminator_logits.keys())
    device = model.device
    if not names:
        return {"total_dsc_loss": torch.tensor(0.0, device=device), "idv_dsc_losses": {}, "idv_dsc_accs": {}}
    from .functions import _DscLossFn
    if isinstance(discriminator_logits, DscLogits) and discriminator_logits.packed is not None:
        packed, (space_dims, dsc_out) = discriminator_logits.packed, discriminator_logits.dims
    else:
        packed = torch.cat([discriminator_logits[n] for n in names], dim=1).contiguous()
        space_dims = tuple(model.discriminators[n].latent_dim for n in names)
        dsc_out = tuple(model.discriminators[n].output_dim for n in names)
    labels = _pack_labels(names, Ybatch, packed.device)
    out = _DscLossFn.apply(packed, labels, space_dims, dsc_out)
    S = len(space_dims)
    idx = [i for i, o in enumerate(dsc_out) if o > 0]
    sel = torch.tensor(idx, device=out.device)
    total = out[:S].index_select(0, sel).sum()
    vals = out.detach().tolist()
    return {"total_dsc_loss": total,
            "idv_dsc_losses": {n: vals[i] for n, i in zip(names, idx)},
            "idv_dsc_accs": {n: vals[S + i] for n, i in zip(names, idx)}}


def _single_dsc_loss(dsc, logits, targets):
    from .functions import _DscLossFn
    labels = targets.to(device=logits.device, dtype=torch.float32).reshape(1, -1).contiguous()
    out = _DscLossFn.apply(logits.contiguous(), labels, (dsc.latent_dim,), (dsc.output_dim,))
    return out[0], out[1]


def compute_adversarial_losses(model, adversary_logits, Ybatch):
    """vae/losses.py:199-223."""
    idv_adv_losses, idv_dsc_losses, idv_dsc_accs = dict(), dict(), dict()
    total_adv_loss = torch.tensor(0.0, device=model.device)
    for adv_name, adv_logits in adversary_logits.items():
        adv = model.adversaries[adv_name]
        latent_name, label_name = adv_name.split('-')
        targets = Ybatch[label_name].to(model.device)
        adv_loss = adv.compute_adversarial_loss(adv_logits)
        idv_adv_losses[adv_name] = adv_loss.item()
        total_adv_loss = total_adv_loss + adv_loss
        idv_dsc_losses[adv_name] = adv.compute_discriminator_loss(adv_logits, targets)     # updates the adversary later
        idv_dsc_accs[adv_name] = adv.compute_accuracy(adv_logits.detach(), targets).item()
    return {"total_adv_loss": total_adv_loss, "idv_adv_losses": idv_adv_losses,
            "idv_adv_dsc_losses": idv_dsc_losses, "idv_adv_dsc_accs": idv_dsc_accs}


def compute_mi_losses(model, latent_params, beta=1.0):
    """vae/losses.py:226-242."""
    idv_mi_estimates = dict()
    total_mi = torch.tensor(0.0, device=model.device)
    for name1, params1 in latent_params.items():
        for name2, params2 in latent_params.items():
            if name1 == name2:
                continue
            mi_estimator = model.mi_estimators.get(f"{name1}-{name2}")
            if mi_estimator is None:
                continue
            mi_estimate = mi_estimator(params1.z, params2.z) * beta
            idv_mi_estimates[f"{name1}-{name2}"] = mi_estimate.item()
            total_mi = total_mi + mi_estimate
    return {"total_mi": total_mi, "idv_mi_estimates": idv_mi_estimates}


def bleu_counts_(counts, refs, cands, eos_token_idx, t_max=None):
    """Adds the corpus-BLEU statistics of (refs [B,T_ref], cands [B,T_cand]), int64 device tensors, into `counts`
    (int64 [10] device tensor, see dvae_bleu_counts) on the current stream.  `t_max`: optional int32 device tensor [1]
    that bounds both row lengths (dvae_bleu_counts_ex: rows padded beyond their batch's own length)."""
    lib = _lib.load()
    args = (refs.data_ptr(), refs.stride(0), refs.size(1), cands.data_ptr(), cands.stride(0), cands.size(1), refs.size(0),
            int(eos_token_idx))
    if t_max is None:
        _lib.check(lib.dvae_bleu_counts(*args, counts.data_ptr(), _lib.stream_ptr()), "dvae_bleu_counts")
    else:
        assert t_max.dtype == torch.int32 and t_max.is_cuda
        _lib.check(lib.dvae_bleu_counts_ex(*args, t_max.data_ptr(), counts.data_ptr(), _lib.stream_ptr()),
                   "dvae_bleu_counts_ex")
    return counts


def bleu_score_(score, counts):
    """score[0] (float32 device tensor) = corpus BLEU of the statistics in `counts`, on the current stream."""
    _lib.check(_lib.load().dvae_bleu_score(counts.data_ptr(), score.data_ptr(), _lib.stream_ptr()), "dvae_bleu_score")
    return score


def bleu_from_counts(counts, device=None):
    """Corpus BLEU (float) of accumulated statistics: e.g. the sum of TrainEngine.eval_steps' "bleu_counts" over a dev
    set, which is the BLEU of the whole set, not the mean of the batches' BLEU."""
    dev = torch.device("cuda") if device is None else torch.device(device)
    with torch.cuda.device(dev):
        c = torch.as_tensor(counts, dtype=torch.int64).to(dev)
        score = torch.empty(1, device=dev, dtype=torch.float32)
        return bleu_score_(score, c).item()


def compute_bleu(Xbatch, pred_batch, idx2word, eos_token_idx):
    """vae/losses.py:128-134: corpus BLEU (torchtext 0.6 `bleu_score`, 4-grams, uniform weights) of the predicted sentences
    against the inputs, each row cut after its first EOS and stripped of its first and last token.

    Computed on the device by `dvae_bleu_counts` + `dvae_bleu_score` over token ids, with one host read.  `idx2word` is
    accepted and not used: the reference's vocabulary maps ids to distinct words (it is built from sorted unique tokens,
    run.py:491-504), so comparing ids gives the same matches as comparing the words.  Host or device int64 tensors [B,T]
    are accepted; the two may have different T."""
    if Xbatch.dim() != 2 or pred_batch.dim() != 2 or Xbatch.size(0) != pred_batch.size(0):
        raise ValueError(f"compute_bleu expects two [B,T] token tensors with the same B, got {tuple(Xbatch.shape)} "
                         f"and {tuple(pred_batch.shape)}")
    dev = pred_batch.device if pred_batch.is_cuda else (Xbatch.device if Xbatch.is_cuda else torch.device("cuda"))
    refs = Xbatch.to(dev, torch.int64).contiguous()
    cands = pred_batch.to(dev, torch.int64).contiguous()
    with torch.cuda.device(dev):
        counts = torch.zeros(10, device=dev, dtype=torch.int64)
        score = torch.empty(1, device=dev, dtype=torch.float32)
        bleu_counts_(counts, refs, cands, eos_token_idx)
        bleu_score_(score, counts)
        return score.item()


def compute_all_losses(model, model_outputs, Xbatch, Ybatch, lengths, kl_weights_dict, mi_loss_weight=0.01):
    """run.py:128-163."""
    L = dict()
    for part in (reconstruction_loss(Xbatch, model_outputs["decoder_logits"], lengths),
                 compute_kl_divergence_losses(model, model_outputs["latent_params"], kl_weights_dict),
                 compute_discriminator_losses(model, model_outputs["dsc_logits"], Ybatch),
                 compute_adversarial_losses(model, model_outputs["adv_logits"], Ybatch),
                 compute_mi_losses(model, model_outputs["latent_params"], beta=mi_loss_weight)):
        for k, v in part.items():
            L.setdefault(k, v)
    total = (L["reconstruction_loss"] + L["total_weighted_kl"] + L["total_dsc_loss"] + L["total_adv_loss"]
             + L["total_mi"])
    return total, L
