"""Encode-once / resample-R inference: the loop body of `scripts/evaluation/consistency.py:163-205` (and the
`sample()` / re-encode pattern of `run.py:286-295`) as ONE captured CUDA graph per resample.

The reference, per batch and per resample r = 1..R, runs two complete forwards:
    output     = vae(x, lengths, teacher_forcing_prob=0.0)          # encode, heads, sampled decode
    x_hat      = output["token_predictions"]; lengths_hat = T - #(EOS | PAD tokens)      (consistency.py:186-190)
    output_hat = vae(x_hat, lengths_hat, teacher_forcing_prob=0.0)  # encode, heads, sampled decode (decode unused)
and reads only `dsc_logits` of both.  Here:
  * `encode_once(x, lengths)` runs the encoder and keeps the context [B,C];
  * `resample(R)` replays, R times, a graph of: fresh eps -> fused heads (z, discriminator logits, decoder initial
    state) -> sampled decode (vocabulary projection + Gumbel-max per step, no logits in HBM) -> on-device length
    recount -> re-encode x_hat -> fused heads.  The second forward's decode, whose output nobody consumes, is not
    run.  Everything stays on the device; results come back in one D2H copy per `resample` call.
  * `reencode_each=True` re-runs the encoder on x inside every resample, as the reference does (in train mode, which
    consistency.py:151 selects, every forward draws new dropout masks); the default encodes once, so the R resamples
    share one dropout draw of the encoder and differ in eps, decoder dropout and the sampled tokens.
RNG: Philox streams keyed by a device-resident seed that the graph itself advances (no host round trip per resample).
"""
import torch

from . import _lib
from .plan import StepPlan


class ConsistencyEvaluator:
    def __init__(self, model, B, T, use_graph=True, min_length=1, seed=None, keep_tokens=True):
        model._require_cuda()
        self.model, self.B, self.T = model, B, T
        self.device = model._flat.device
        self.plan = StepPlan(model, B, T, self.device)
        self.d = d = self.plan.d
        self.use_graph = use_graph
        self.min_length = min_length
        self.keep_tokens = keep_tokens
        dev = self.device
        self.inputs = torch.zeros(B, T, device=dev, dtype=torch.int64)
        self.lengths = torch.ones(B, device=dev, dtype=torch.int64)
        self.ctx0 = torch.zeros(B, d.C, device=dev, dtype=torch.float32)
        self.preds = torch.zeros(B, T, device=dev, dtype=torch.int64)
        self.lengths_hat = torch.ones(B, device=dev, dtype=torch.int64)
        self.coins = torch.zeros(max(T - 1, 1), device=dev, dtype=torch.int32)      # 0 = every step samples (tf = 0)
        OD = max(d.OD, 1)
        self.logits = torch.zeros(B, OD, device=dev, dtype=torch.float32)
        self.logits_hat = torch.zeros(B, OD, device=dev, dtype=torch.float32)
        self.z = torch.zeros(B, d.Z, device=dev, dtype=torch.float32)
        self.z_hat = torch.zeros(B, d.Z, device=dev, dtype=torch.float32)
        g = torch.Generator().manual_seed(10 if seed is None else int(seed))
        self.plan.seed_dev.fill_(int(torch.randint(0, 2 ** 61, (1,), generator=g)))
        self._graph = {}
        self._encoded = False
        # weight planes of the decoder's LSTM matrices: every decode step multiplies by them (x_t . W_ih^T, h_{t-1} . W_hh^T);
        # the weights do not change during evaluation, so the planes are written once per resample() call
        self._wplanes, self._plane_token = [], object()
        if B >= 256 and not d.bow:
            for n, w in model._P.items():
                if n.startswith("decoder.recurrent.weight_") and w.dim() == 2 and w.numel() >= (1 << 14) and not (w.data_ptr() & 15):
                    R, C = w.shape
                    self._wplanes.append((w, torch.empty(self.plan.lib.dvae_weight_planes_floats(R, C, 0), device=dev, dtype=torch.float32)))

    def _planes_on(self, refresh):
        lib = self.plan.lib
        if not self._wplanes:
            return
        if _lib.planes_owner is not self._plane_token:
            _lib.check(lib.dvae_weight_planes_clear(), "dvae_weight_planes_clear")
            for w, pl in self._wplanes:
                _lib.check(lib.dvae_weight_planes_register(_lib.ptr(w), w.size(0), w.size(1), _lib.ptr(pl), None), "dvae_weight_planes_register")
            _lib.planes_owner = self._plane_token
        if refresh:
            _lib.check(lib.dvae_weight_planes_refresh(_lib.stream_ptr()), "dvae_weight_planes_refresh")
        _lib.check(lib.dvae_weight_planes_enable(1), "dvae_weight_planes_enable")

    def _planes_off(self):
        if self._wplanes:
            _lib.check(self.plan.lib.dvae_weight_planes_enable(0), "dvae_weight_planes_enable")

    # ------------------------------------------------------------------------------------------
    def encode_once(self, inputs, lengths):
        """inputs [B,T] int64, lengths [B] (host or device).  Runs the encoder (dropout as model.training says)."""
        self.inputs.copy_(inputs.to(self.device, torch.int64), non_blocking=True)
        self.lengths.copy_(torch.as_tensor(lengths).to(self.device, torch.int64), non_blocking=True)
        self._encode_x()
        self._encoded = True
        return self.ctx0

    def _encode_x(self):
        pl, P, m = self.plan, self.model._P, self.model
        pl.seed_dev.add_(0x9E3779B1)
        pl.encode(P, self.inputs, self.lengths, m.training)
        self.ctx0.copy_(pl.ctx)

    def _body(self, reencode):
        pl, P, m, d = self.plan, self.model._P, self.model, self.d
        if reencode:
            self._encode_x()
        pl.seed_dev.add_(0x9E3779B1)                    # new eps / decoder dropout / Gumbel noise for this resample
        pl.randn_eps(0)
        pl.heads(P, self.ctx0, pl.eps, None, None)      # z, dsc logits, decoder initial state
        self.logits.copy_(pl.dsc_logits)
        self.z.copy_(pl.z)
        self.preds.zero_()
        self.preds[:, 0].fill_(m.sos_token_idx)
        pl.decode_sampled(P, self.preds, self.coins, m.training)
        pl.recount_lengths(self.preds, self.lengths_hat, m.eos_token_idx, 0, self.min_length)
        pl.seed_dev.add_(0x9E3779B1)                    # the second forward draws its own dropout masks and eps
        pl.encode(P, self.preds, self.lengths_hat, m.training)
        pl.randn_eps(1)
        pl.heads(P, pl.ctx, pl.eps, None, None)
        self.logits_hat.copy_(pl.dsc_logits)
        self.z_hat.copy_(pl.z)

    def _run_body(self, reencode):
        if not self.use_graph:
            return self._body(reencode)
        g = self._graph.get(reencode)
        if g is None:
            s = torch.cuda.Stream(device=self.device)
            s.wait_stream(torch.cuda.current_stream())
            seed0 = self.plan.seed_dev.clone()
            with torch.cuda.stream(s):
                self._body(reencode)                     # warm-up: lazy kernel attributes, workspaces
            torch.cuda.current_stream().wait_stream(s)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=s):
                self._body(reencode)
            torch.cuda.synchronize()
            self.plan.seed_dev.copy_(seed0)
            self._graph[reencode] = g
        g.replay()

    def resample(self, R, reencode_each=False):
        """R resamples of the batch given to encode_once().  Returns a dict of device tensors:
        dsc_logits [R,B,OD], dsc_logits_hat [R,B,OD], z / z_hat [R,B,Z], lengths_hat [R,B] and (keep_tokens)
        token_predictions [R,B,T]."""
        if not self._encoded:
            raise _lib.DvaeError("call encode_once(inputs, lengths) first")
        d, B, T, dev = self.d, self.B, self.T, self.device
        OD = max(d.OD, 1)
        out = {"dsc_logits": torch.empty(R, B, OD, device=dev), "dsc_logits_hat": torch.empty(R, B, OD, device=dev),
               "z": torch.empty(R, B, d.Z, device=dev), "z_hat": torch.empty(R, B, d.Z, device=dev),
               "lengths_hat": torch.empty(R, B, device=dev, dtype=torch.int64)}
        if self.keep_tokens:
            out["token_predictions"] = torch.empty(R, B, T, device=dev, dtype=torch.int64)
        self._planes_on(refresh=True)
        try:
            with torch.no_grad():
                for r in range(R):
                    self._run_body(bool(reencode_each))
                    self._copy_out(out, r)
        finally:
            self._planes_off()
        return out

    def _copy_out(self, out, r):
        out["dsc_logits"][r].copy_(self.logits)
        out["dsc_logits_hat"][r].copy_(self.logits_hat)
        out["z"][r].copy_(self.z)
        out["z_hat"][r].copy_(self.z_hat)
        out["lengths_hat"][r].copy_(self.lengths_hat)
        if self.keep_tokens:
            out["token_predictions"][r].copy_(self.preds)

    def bleu(self, out):
        """[R] float32 device tensor: corpus BLEU (losses.compute_bleu) of every resample's token_predictions against the
        inputs given to encode_once().  Needs keep_tokens=True.  Runs after resample(), outside its graph: two kernels per
        resample into one [R,10] block of counters, no host read."""
        from .losses import bleu_counts_, bleu_score_
        if "token_predictions" not in out:
            raise _lib.DvaeError("bleu() needs the token_predictions of resample(): build the evaluator with keep_tokens=True")
        tok = out["token_predictions"]
        R = tok.size(0)
        counts = torch.zeros(R, 10, device=self.device, dtype=torch.int64)
        scores = torch.empty(R, device=self.device, dtype=torch.float32)
        for r in range(R):
            bleu_counts_(counts[r], self.inputs, tok[r], self.model.eos_token_idx)
            bleu_score_(scores[r:r + 1], counts[r])
        return scores

    def predictions(self, packed_logits):
        """{label: [..., B] int64} = Discriminator.predict (vae/model.py:204-210) on packed logits [..., B, OD]."""
        d, preds, off = self.d, {}, 0
        for n, o in zip(d.space_names, d.dsc_out):
            if o > 0:
                x = packed_logits[..., off:off + o]
                preds[n] = (x[..., 0] > 0).long() if o == 1 else x.argmax(-1)
                off += o
        return preds
