"""Kernel sequencing for one (batch, length) shape: owns every activation / workspace buffer and
issues the C-ABI calls of `include/dvae_b200.h` in forward and backward order.

Used by both host paths: the drop-in module (`model.py`, through autograd Functions) and the
graph-captured training engine (`engine.py`).  No torch compute ops on the path -- torch only
allocates memory and provides the stream.

Data layout in HBM (all fp32 unless noted), T = padded length, T1 = T-1, N = T1*B:
  x_enc   [T,B,E]            embedded (+dropout) encoder input, time-major
  e_gates [Le][D,T,B,4H]     pre-activations -> post-activation gates -> (backward) dG, in place
  e_cs    [Le][D,T,B,H]      cell states;  e_hs [Le][T,B,D*H] layer outputs (zeros at padding)
  ctx     [B,C]              concat of final hidden states, written in place by the LSTM kernels
  eps,z,mu,logvar [B,Z]; hid [B,2*H*Ld]; dsc_logits [B,OD]; scalars [27]
  x_dec   [T1,B,E]; d_gates/d_cs/d_hs as above with D=1
  lse,nll [N]; argmax [N] int32; recon [1]
"""
import torch

from . import _lib
from ._lib import ptr, ptr_array, int_array, check

SALT_ENC_EMB, SALT_DEC_EMB, SALT_ENC_LAYER, SALT_DEC_LAYER, SALT_EPS, SALT_SAMPLE = 1, 3, 16, 32, 64, 4096


class Dims:
    """Static shape information derived from the module (mirrors vae/model.py:261-321)."""

    def __init__(self, model):
        enc, dec = model.encoder, model.decoder
        self.V, self.E = enc.embedding.weight.shape
        self.H = enc.hidden_size                 # encoder hidden size (= embedding size for the BOW encoder)
        self.Hd = dec.hidden_size                # decoder hidden size
        self.bow = not hasattr(enc, "recurrent")
        self.D = enc.num_directions
        self.Le = 0 if not hasattr(enc, "recurrent") else enc.num_layers
        self.Ld = dec.num_layers
        self.C = self.H * enc.num_layers * self.D
        self.space_names = list(model.context2params.keys())
        self.space_dims = [model.context2params[n].out_features // 2 for n in self.space_names]
        self.S = len(self.space_names)
        self.Z = sum(self.space_dims)
        self.dsc_out = [model.discriminators[n].output_dim if n in model.discriminators else 0
                        for n in self.space_names]
        self.OD = sum(self.dsc_out)
        self.H2L = 2 * self.Hd * self.Ld
        self.sos, self.eos = model.sos_token_idx, model.eos_token_idx
        self.p_enc, self.p_dec = float(enc.dropout_rate), float(dec.dropout_rate)
        assert self.S <= _lib.MAX_SPACES, f"at most {_lib.MAX_SPACES} latent spaces"


class StepPlan:
    def __init__(self, model, B, T, device):
        self.lib = _lib.load()
        self.d = d = Dims(model)
        self.B, self.T, self.T1 = B, T, T - 1
        self.N = self.T1 * B
        self.device = device
        self.busy = False
        f32 = dict(device=device, dtype=torch.float32)
        H, D, E = d.H, d.D, d.E

        def buf(*shape):
            return torch.empty(*shape, **f32)

        self.x_enc = buf(T, B, E)
        self.e_gates = [buf(D, T, B, 4 * H) for _ in range(d.Le)]
        self.e_cs = [buf(D, T, B, H) for _ in range(d.Le)]
        self.e_hs = [buf(T, B, D * H) for _ in range(d.Le)]
        self.e_xin = [None] + [buf(T, B, D * H) for _ in range(1, d.Le)]   # dropped-out layer inputs
        self.ctx = buf(B, d.C)
        self.ctx_c = buf(B, d.C)
        self.eps = buf(B, d.Z)
        self.z, self.mu, self.logvar = buf(B, d.Z), buf(B, d.Z), buf(B, d.Z)
        self.hid = buf(B, d.H2L)
        self.dsc_logits = buf(B, max(d.OD, 1))
        # one small result block so a step's scalars come back in a single D2H read:
        # out[:27] = fused-head scalars (weighted KL, KL, dsc loss, per-space ...), out[27] = recon loss
        self.out = torch.zeros(_lib.HEADS_NSCALARS + 5, **f32)
        self.scalars = self.out[:_lib.HEADS_NSCALARS]
        self.heads_ws = torch.zeros(self.lib.dvae_heads_ws_floats(B, d.S), **f32)     # arrival counter must start at zero
        T1 = max(self.T1, 1)
        self.x_dec = buf(T1, B, E)
        Hd = d.Hd
        self.d_gates = [buf(1, T1, B, 4 * Hd) for _ in range(d.Ld)]
        self.d_cs = [buf(1, T1, B, Hd) for _ in range(d.Ld)]
        self.d_hs = [buf(T1, B, Hd) for _ in range(d.Ld)]
        self.d_xin = [None] + [buf(T1, B, Hd) for _ in range(1, d.Ld)]
        self.state_ws = buf(self.lib.dvae_lstm_state_ws_floats(B, max(H, Hd), D))
        self.bow_argmax = torch.zeros(B, E, device=device, dtype=torch.int32) if d.bow else None
        self.lse, self.nll = buf(max(self.N, 1)), buf(max(self.N, 1))
        self.argmax = torch.zeros(max(self.N, 1), device=device, dtype=torch.int32)
        self.recon = self.out[_lib.HEADS_NSCALARS:_lib.HEADS_NSCALARS + 1]
        self.ce_ws = buf(self.lib.dvae_vocab_ce_ws_floats(max(self.N, 1), d.V, d.Hd))
        self.sample_ws = None                      # allocated on first sampled decode
        # vocabulary kernels over the live rows only (t < len_b): vocab_ce then leaves lse / nll / argmax at masked
        # positions unwritten.  TrainEngine sets it; the drop-in path returns every position's argmax and keeps all rows.
        self.live_rows = False
        self._bwd_ready = False
        self.seed_dev = torch.zeros(1, device=device, dtype=torch.int64)
        self.labels = buf(max(sum(1 for o in d.dsc_out if o > 0), 1), B)
        self._space_dims = int_array(d.space_dims)
        self._dsc_out = int_array(d.dsc_out)
        self.train_mode = False

    # ------------------------------------------------------------------------------------------
    def _alloc_bwd(self):
        if self._bwd_ready:
            return
        d, B, T, T1 = self.d, self.B, self.T, max(self.T1, 1)
        f32 = dict(device=self.device, dtype=torch.float32)
        w = max(d.E, d.H * d.D, d.Hd)
        self.g_top = torch.empty(T1, B, d.Hd, **f32)
        self.g_dx = [torch.empty(max(T, T1), B, w, **f32) for _ in range(2)]
        self.g_dx_dec0 = torch.empty(T1, B, d.E, **f32)       # decoder layer 0's d_x, written on decode_bwd's aux_stream
        self.g_hid = torch.empty(B, d.H2L, **f32)
        self.g_ctx = torch.empty(B, d.C, **f32)
        self.heads_bwd_ws = torch.empty(self.lib.dvae_heads_bwd_ws_floats(B, d.Z, d.H2L), **f32)
        self.ce_bwd_ws = torch.empty(self.lib.dvae_vocab_ce_bwd_ws_floats(max(self.N, 1), d.V, d.Hd), **f32)
        # operand planes of x, dG and hs for the LSTM weight-gradient GEMMs: one buffer, sized for the largest layer
        need = [self.lib.dvae_lstm_bwd_planes_ws_floats(T1, B, d.E if l == 0 else d.Hd, d.Hd, 1) for l in range(d.Ld)]
        need += [self.lib.dvae_lstm_bwd_planes_ws_floats(T, B, d.E if l == 0 else d.D * d.H, d.H, d.D) for l in range(d.Le)]
        self.lstm_bwd_planes = torch.empty(max(need), **f32)
        self._bwd_ready = True

    @staticmethod
    def _enc_w(P, l, dirs):
        sfx = [f"_l{l}" + ("_reverse" if k else "") for k in range(dirs)]
        return tuple([P[f"encoder.recurrent.{n}{s}"] for s in sfx] for n in ("weight_ih", "weight_hh", "bias_ih", "bias_hh"))

    @staticmethod
    def _dec_w(P, l):
        return tuple([P[f"decoder.recurrent.{n}_l{l}"]] for n in ("weight_ih", "weight_hh", "bias_ih", "bias_hh"))

    # ------------------------------------------------------------------------------------------
    # forward pieces.  P: dict name -> parameter tensor (reference state_dict names + fused groups)
    # ------------------------------------------------------------------------------------------
    def encode(self, P, inputs, lengths, train, after_l0_proj=None):
        """a1 + a2 (vae/model.py:88-101,373-382): inputs [B,T] int64 (row stride = inputs.stride(0)).
        `after_l0_proj`: optional callable invoked once layer 0's input-projection GEMMs are enqueued and before its
        recurrence kernel is -- the point from which 84 of the 148 SMs are idle for the rest of the encoder (the engine
        forks the decoder's encoder-independent work there)."""
        lib, d, st = self.lib, self.d, _lib.stream_ptr()
        B, T = self.B, self.T
        p = d.p_enc if train else 0.0
        if d.bow:      # BOWEncoder (vae/model.py:42-49): context = max over positions of dropout(embedding)
            check(lib.dvae_bow_encoder_fwd(ptr(P["encoder.embedding.weight"]), d.E, ptr(inputs), inputs.stride(0),
                                           inputs.stride(1), T, B, p, ptr(self.seed_dev), SALT_ENC_EMB, ptr(self.ctx), d.C,
                                           ptr(self.bow_argmax), st), "dvae_bow_encoder_fwd")
            self._enc_p = p
            return self.ctx
        check(lib.dvae_embedding_fwd(ptr(P["encoder.embedding.weight"]), d.E, ptr(inputs), inputs.stride(0),
                                     inputs.stride(1), T, B, p, ptr(self.seed_dev), SALT_ENC_EMB, -1, 0,
                                     ptr(self.x_enc), st), "dvae_embedding_fwd")
        x, I = self.x_enc, d.E
        for l in range(d.Le):
            if l > 0:
                I = d.D * d.H
                if p > 0.0:
                    check(lib.dvae_dropout(ptr(self.e_hs[l - 1]), I, T * B, I, p, ptr(self.seed_dev),
                                           SALT_ENC_LAYER + l, ptr(self.e_xin[l]), I, 0, st), "dvae_dropout")
                    x = self.e_xin[l]
                else:
                    x = self.e_hs[l - 1]
            w_ih, w_hh, b_ih, b_hh = self._enc_w(P, l, d.D)
            off = l * d.D * d.H
            split = l == 0 and after_l0_proj is not None
            if split:
                check(lib.dvae_lstm_input_proj(ptr(x), I, T, B, I, d.H, d.D, ptr_array(w_ih), ptr_array(b_ih),
                                               ptr_array(b_hh), ptr(self.e_gates[l]), st), "dvae_lstm_input_proj(enc)")
                after_l0_proj()
            check(lib.dvae_lstm_seq_fwd_ex(ptr(x), I, T, B, I, d.H, d.D, ptr_array(w_ih), ptr_array(w_hh),
                                           ptr_array(b_ih), ptr_array(b_hh), None, None, 0, 0, ptr(lengths),
                                           ptr(self.e_hs[l]), d.D * d.H, self.ctx.data_ptr() + 4 * off,
                                           self.ctx_c.data_ptr() + 4 * off, d.C, d.H, ptr(self.e_gates[l]),
                                           ptr(self.e_cs[l]), ptr(self.state_ws), 1 if split else 0, st),
                  "dvae_lstm_seq_fwd(enc)")
        self._enc_p = p
        return self.ctx

    def heads(self, P, ctx, eps, labels, kl_w):
        """a3 + a4 + a5 + a8 fused.  labels: packed [n_dsc,B] float tensor or None; kl_w: [S] or None."""
        lib, d, st = self.lib, self.d, _lib.stream_ptr()
        check(lib.dvae_latent_heads_fwd(ptr(ctx), self.B, d.C, d.S, self._space_dims, self._dsc_out,
                                        ptr(P["_c2p.weight"]), ptr(P["_c2p.bias"]), ptr(eps),
                                        ptr(P.get("_dsc.weight")), ptr(P.get("_dsc.bias")), ptr(labels), ptr(kl_w),
                                        ptr(P["z2hidden.weight"]), ptr(P["z2hidden.bias"]), d.H2L, ptr(self.z),
                                        ptr(self.mu), ptr(self.logvar), ptr(self.hid), ptr(self.dsc_logits),
                                        ptr(self.scalars), ptr(self.heads_ws), st), "dvae_latent_heads_fwd")

    def decode_forced(self, P, tokens, first_token, train, hid=None):
        """a6 under teacher forcing: `tokens` [B,>=T1] supplies the decoder input at step t (t>=1 when
        first_token >= 0 overrides step 0 with <SOS>)."""
        lib, d, st = self.lib, self.d, _lib.stream_ptr()
        B, T1 = self.B, self.T1
        hid = self.hid if hid is None else hid
        p = d.p_dec if train else 0.0
        # decode_prepare() may already have embedded the inputs and projected them through layer 0's W_ih
        prepared = getattr(self, "_dec_prepared", None) == (tokens.data_ptr(), first_token, p)
        self._dec_prepared = None
        if not prepared:
            check(lib.dvae_embedding_fwd(ptr(P["decoder.embedding.weight"]), d.E, ptr(tokens), tokens.stride(0),
                                         tokens.stride(1), T1, B, p, ptr(self.seed_dev), SALT_DEC_EMB, first_token, 0,
                                         ptr(self.x_dec), st), "dvae_embedding_fwd")
        x, I = self.x_dec, d.E
        for l in range(d.Ld):
            if l > 0:
                I = d.Hd
                if p > 0.0:
                    check(lib.dvae_dropout(ptr(self.d_hs[l - 1]), I, T1 * B, I, p, ptr(self.seed_dev),
                                           SALT_DEC_LAYER + l, ptr(self.d_xin[l]), I, 0, st), "dvae_dropout")
                    x = self.d_xin[l]
                else:
                    x = self.d_hs[l - 1]
            w_ih, w_hh, b_ih, b_hh = self._dec_w(P, l)
            check(lib.dvae_lstm_seq_fwd_ex(ptr(x), I, T1, B, I, d.Hd, 1, ptr_array(w_ih), ptr_array(w_hh),
                                           ptr_array(b_ih), ptr_array(b_hh), hid.data_ptr() + 4 * l * d.Hd,
                                           hid.data_ptr() + 4 * (d.Ld + l) * d.Hd, d.H2L, 0, None, ptr(self.d_hs[l]),
                                           d.Hd, None, None, 0, 0, ptr(self.d_gates[l]), ptr(self.d_cs[l]),
                                           ptr(self.state_ws), 1 if (prepared and l == 0) else 0, st),
                  "dvae_lstm_seq_fwd(dec)")
        self._dec_p = p
        self._dec_tokens, self._dec_first = tokens, first_token
        self._dec_hid = hid
        return self.d_hs[-1]

    def decode_prepare(self, P, tokens, first_token, train):
        """The part of decode_forced() that does not depend on the encoder: input embeddings (+ dropout) and layer 0's
        input projection, and the fp16 operand planes of W_out for vocab_ce().  Call it on another stream (the engine
        runs it under the encoder) and make the stream that calls decode_forced() / vocab_ce() wait for it."""
        lib, d, st = self.lib, self.d, _lib.stream_ptr()
        B, T1 = self.B, self.T1
        p = d.p_dec if train else 0.0
        check(lib.dvae_embedding_fwd(ptr(P["decoder.embedding.weight"]), d.E, ptr(tokens), tokens.stride(0),
                                     tokens.stride(1), T1, B, p, ptr(self.seed_dev), SALT_DEC_EMB, first_token, 0,
                                     ptr(self.x_dec), st), "dvae_embedding_fwd")
        w_ih, _, b_ih, b_hh = self._dec_w(P, 0)
        check(lib.dvae_lstm_input_proj(ptr(self.x_dec), d.E, T1, B, d.E, d.Hd, 1, ptr_array(w_ih), ptr_array(b_ih),
                                       ptr_array(b_hh), ptr(self.d_gates[0]), st), "dvae_lstm_input_proj(dec)")
        self._dec_prepared = (tokens.data_ptr(), first_token, p)
        check(lib.dvae_vocab_split_w(ptr(P["decoder.linear.weight"]), max(self.N, 1), d.V, d.Hd, ptr(self.ce_ws), st),
              "dvae_vocab_split_w")
        self._w_planes_ready = P["decoder.linear.weight"].data_ptr()

    def decode_sampled(self, P, preds, coins, train, hid=None):
        """a6 / a12 with sampled inputs (vae/model.py:457-472,498-508).  `preds` [B,T] int64 is both the
        decoder-input buffer and the returned `token_predictions`: preds[:,0] = <SOS>, preds[:,i] = the forced
        token (pre-filled by the caller) when coins[i-1] is true, else the token sampled from position i's
        logits, which is written here by the sampling kernel before step i reads it.  Leaves x_dec / d_gates /
        d_cs / d_hs exactly as a whole-sequence call would, so decode_bwd / vocab_ce are shared.
        `coins`: a host sequence of bools, or an int32 DEVICE tensor [T1] (non-zero = forced): then every step
        enqueues its sampling call and the kernels themselves skip the forced steps, so the launch sequence does not
        depend on the draw and can be captured once as a CUDA graph (engine.TrainEngine with teacher forcing < 1)."""
        lib, d, st = self.lib, self.d, _lib.stream_ptr()
        B, T1 = self.B, self.T1
        hid = self.hid if hid is None else hid
        p = d.p_dec if train else 0.0
        if self.sample_ws is None:
            self.sample_ws = torch.empty(lib.dvae_vocab_ce_ws_floats(B, d.V, d.Hd), device=self.device, dtype=torch.float32)
        emb = P["decoder.embedding.weight"]
        W = [self._dec_w(P, l) for l in range(d.Ld)]
        dev_coins = torch.is_tensor(coins)
        if dev_coins:
            assert coins.dtype == torch.int32 and coins.is_cuda and coins.numel() >= T1
        # large batches: W_out is split into the vocabulary kernels' operand planes once per decode, not once per CTA and step
        w_planes = None
        if B >= 256 and d.V >= 1024 and d.Hd % 32 == 0:
            if getattr(self, "w_out_planes", None) is None:
                self.w_out_planes = torch.empty(lib.dvae_vocab_w_planes_floats(d.V, d.Hd), device=self.device, dtype=torch.float32)
            w_planes = self.w_out_planes
            check(lib.dvae_vocab_w_planes(ptr(P["decoder.linear.weight"]), d.V, d.Hd, ptr(w_planes), st), "dvae_vocab_w_planes")
        for s in range(T1):
            check(lib.dvae_embedding_fwd(ptr(emb), d.E, ptr(preds), preds.stride(0), preds.stride(1), 1, B, p,
                                         ptr(self.seed_dev), SALT_DEC_EMB, d.sos, s, ptr(self.x_dec), st),
                  "dvae_embedding_fwd(step)")
            x, I = self.x_dec, d.E
            for l in range(d.Ld):
                if l > 0:
                    I = d.Hd
                    if p > 0.0:
                        check(lib.dvae_dropout(ptr(self.d_hs[l - 1]), I, B, I, p, ptr(self.seed_dev),
                                               SALT_DEC_LAYER + l, ptr(self.d_xin[l]), I, s * B, st), "dvae_dropout(step)")
                        x = self.d_xin[l]
                    else:
                        x = self.d_hs[l - 1]
                w_ih, w_hh, b_ih, b_hh = W[l]
                check(lib.dvae_lstm_step(ptr(x), I, s, T1, B, I, d.Hd, ptr(w_ih[0]), ptr(w_hh[0]), ptr(b_ih[0]),
                                         ptr(b_hh[0]), hid.data_ptr() + 4 * l * d.Hd,
                                         hid.data_ptr() + 4 * (d.Ld + l) * d.Hd, d.H2L, ptr(self.d_hs[l]),
                                         ptr(self.d_gates[l]), ptr(self.d_cs[l]), ptr(self.state_ws), st),
                      "dvae_lstm_step")
            if dev_coins or not coins[s]:
                h_s = self.d_hs[-1].data_ptr() + 4 * s * B * d.Hd
                flag = coins.data_ptr() + 4 * s if dev_coins else None
                check(lib.dvae_vocab_sample_step_planes(h_s, d.Hd, B, d.Hd, d.V, ptr(P["decoder.linear.weight"]),
                                                        ptr(P["decoder.linear.bias"]), ptr(w_planes), ptr(self.seed_dev),
                                                        SALT_SAMPLE + s, preds.data_ptr() + 8 * (s + 1) * preds.stride(1),
                                                        preds.stride(0), flag, ptr(self.sample_ws), st), "dvae_vocab_sample_step")
        self._dec_p = p
        self._dec_tokens, self._dec_first = preds, d.sos
        self._dec_hid = hid
        return self.d_hs[-1]

    def vocab_ce(self, P, h_top, targets, lengths):
        """a7 fused with the vocabulary projection of a6."""
        lib, d, st = self.lib, self.d, _lib.stream_ptr()
        w_ready = getattr(self, "_w_planes_ready", None) == P["decoder.linear.weight"].data_ptr()
        self._w_planes_ready = None
        fwd = lib.dvae_vocab_ce_fwd_live if self.live_rows else lib.dvae_vocab_ce_fwd_ex
        check(fwd(ptr(h_top), d.Hd, self.T1, self.B, d.Hd, d.V, ptr(P["decoder.linear.weight"]),
                  ptr(P["decoder.linear.bias"]), ptr(targets), targets.stride(0), ptr(lengths),
                  d.sos, ptr(self.lse), ptr(self.nll), ptr(self.argmax), ptr(self.recon),
                  ptr(self.ce_ws), 1 if w_ready else 0, st), "dvae_vocab_ce_fwd")
        # the backward of this same step may reuse the operand planes (live rows: and the row list) the call left in ce_ws
        self._ce_planes_valid = (h_top.data_ptr(), P["decoder.linear.weight"].data_ptr(), lengths.data_ptr(), self.live_rows)
        return self.recon

    # ------------------------------------------------------------------------------------------
    # backward pieces.  G: dict name -> gradient tensor to WRITE (same names as P)
    # ------------------------------------------------------------------------------------------
    def vocab_ce_bwd(self, P, G, h_top, targets, lengths, grad_scale_dev):
        self._alloc_bwd()
        lib, d, st = self.lib, self.d, _lib.stream_ptr()
        # operand planes left by this step's forward call (same h_top, same weights): no need to split again
        valid = getattr(self, "_ce_planes_valid", None)
        reuse = valid is not None and valid[:3] == (h_top.data_ptr(), P["decoder.linear.weight"].data_ptr(), lengths.data_ptr())
        live = reuse and valid[3]          # the live-row backward needs the forward's row list: same call, same lengths
        self._ce_planes_valid = None
        # a live-row forward's lse exists at live positions only: the every-row backward reads it only where the loss
        # weight is non-zero, so it still applies (without the forward's planes, which hold the live rows only)
        bwd = lib.dvae_vocab_ce_bwd_live if live else lib.dvae_vocab_ce_bwd
        check(bwd(ptr(h_top), d.Hd, self.T1, self.B, d.Hd, d.V, ptr(P["decoder.linear.weight"]),
                  ptr(P["decoder.linear.bias"]), ptr(targets), targets.stride(0), ptr(lengths),
                  ptr(self.lse), ptr(grad_scale_dev), ptr(self.g_top), d.Hd,
                  ptr(G["decoder.linear.weight"]), ptr(G["decoder.linear.bias"]),
                  ptr(self.ce_ws) if reuse else None, ptr(self.ce_bwd_ws), st),
              "dvae_vocab_ce_bwd")
        return self.g_top

    def decode_bwd(self, P, G, g_top, emb_grad=True, aux_stream=None):
        """BPTT through the decoder stack; leaves d(hid) in self.g_hid.  With `aux_stream` layer 0's d_x GEMM (into its
        own buffer) and the embedding-gradient scatter -- nothing downstream reads either before the optimizer -- are
        enqueued there, beside the heads' and the encoder's backward; the caller makes its stream wait for `aux_stream`
        before anything reads the embedding gradient."""
        self._alloc_bwd()
        lib, d, st = self.lib, self.d, _lib.stream_ptr()
        B, T1 = self.B, self.T1
        hid = self._dec_hid
        g_in, p = g_top, self._dec_p
        for l in range(d.Ld - 1, -1, -1):
            I = d.E if l == 0 else d.Hd
            x = self.x_dec if l == 0 else (self.d_xin[l] if p > 0.0 else self.d_hs[l - 1])
            dx_aside = l == 0 and aux_stream is not None
            g_out = self.g_dx_dec0 if dx_aside else self.g_dx[l % 2]
            w_ih, w_hh, _, _ = self._dec_w(P, l)
            gw_ih, gw_hh, gb_ih, gb_hh = self._dec_w(G, l)
            need_dx = l > 0 or emb_grad
            if dx_aside:
                check(lib.dvae_lstm_bwd_dx_stream(aux_stream.cuda_stream), "dvae_lstm_bwd_dx_stream")
            try:
                check(lib.dvae_lstm_seq_bwd_ex(ptr(x), I, T1, B, I, d.Hd, 1, ptr_array(w_ih), ptr_array(w_hh),
                                            hid.data_ptr() + 4 * l * d.Hd, hid.data_ptr() + 4 * (d.Ld + l) * d.Hd,
                                            d.H2L, 0, None, ptr(self.d_hs[l]), d.Hd, ptr(self.d_gates[l]),
                                            ptr(self.d_cs[l]), ptr(g_in), d.Hd, None, None, 0, 0,
                                            ptr(g_out) if need_dx else None, I, ptr_array(gw_ih), ptr_array(gw_hh),
                                            ptr_array(gb_ih), ptr_array(gb_hh), self.g_hid.data_ptr() + 4 * l * d.Hd,
                                            self.g_hid.data_ptr() + 4 * (d.Ld + l) * d.Hd, d.H2L, 0,
                                            ptr(self.state_ws), ptr(self.lstm_bwd_planes), st), "dvae_lstm_seq_bwd(dec)")
            finally:
                if dx_aside:
                    check(lib.dvae_lstm_bwd_dx_stream(None), "dvae_lstm_bwd_dx_stream")
            if l > 0 and p > 0.0:
                check(lib.dvae_dropout(ptr(g_out), I, T1 * B, I, p, ptr(self.seed_dev), SALT_DEC_LAYER + l,
                                       ptr(g_out), I, 0, st), "dvae_dropout(bwd)")
            g_in = g_out
        if emb_grad:
            tok = self._dec_tokens
            if aux_stream is not None:      # behind layer 0's d_x GEMM, which the library ordered after the recurrence
                st = aux_stream.cuda_stream
            check(lib.dvae_embedding_bwd(ptr(g_in), d.E, ptr(tok), tok.stride(0), tok.stride(1), T1, B, p,
                                         ptr(self.seed_dev), SALT_DEC_EMB, self._dec_first, 0,
                                         ptr(G["decoder.embedding.weight"]), st), "dvae_embedding_bwd")
        return self.g_hid

    def heads_bwd(self, P, G, ctx, eps, labels, kl_w, g_hid, g_z=None, g_mu=None, g_logvar=None, g_logits=None):
        self._alloc_bwd()
        lib, d, st = self.lib, self.d, _lib.stream_ptr()
        check(lib.dvae_latent_heads_bwd(ptr(ctx), self.B, d.C, d.S, self._space_dims, self._dsc_out,
                                        ptr(P["_c2p.weight"]), ptr(eps), ptr(P.get("_dsc.weight")), ptr(labels),
                                        ptr(kl_w), ptr(P["z2hidden.weight"]), d.H2L, ptr(self.z), ptr(self.mu),
                                        ptr(self.logvar), ptr(self.hid), ptr(self.dsc_logits), ptr(g_hid),
                                        ptr(g_z), ptr(g_mu), ptr(g_logvar), ptr(g_logits), ptr(G["_c2p.weight"]),
                                        ptr(G["_c2p.bias"]), ptr(G.get("_dsc.weight")), ptr(G.get("_dsc.bias")),
                                        ptr(G["z2hidden.weight"]), ptr(G["z2hidden.bias"]), ptr(self.g_ctx),
                                        ptr(self.heads_bwd_ws), st), "dvae_latent_heads_bwd")
        return self.g_ctx

    def encode_bwd(self, P, G, inputs, lengths, g_ctx, emb_grad=True, layers=None):
        """BPTT through the encoder stack.  `layers`: optional (first, last) pair, first >= last, to run only layers
        first..last of the top-down sweep in this call (the data-parallel engine all-reduces layer 1's gradients while layer
        0 is still running); a later call continues from the gradient the earlier one left."""
        self._alloc_bwd()
        lib, d, st = self.lib, self.d, _lib.stream_ptr()
        B, T = self.B, self.T
        p = self._enc_p
        if d.bow:
            if emb_grad:
                check(lib.dvae_bow_encoder_bwd(ptr(g_ctx), d.C, ptr(self.bow_argmax), d.E, ptr(inputs), inputs.stride(0),
                                               inputs.stride(1), T, B, p, ptr(self.seed_dev), SALT_ENC_EMB,
                                               ptr(G["encoder.embedding.weight"]), st), "dvae_bow_encoder_bwd")
            return
        first, last = (d.Le - 1, 0) if layers is None else layers
        g_in = None if first == d.Le - 1 else self._enc_g_in
        for l in range(first, last - 1, -1):
            I = d.E if l == 0 else d.D * d.H
            x = self.x_enc if l == 0 else (self.e_xin[l] if p > 0.0 else self.e_hs[l - 1])
            g_out = self.g_dx[l % 2]
            w_ih, w_hh, _, _ = self._enc_w(P, l, d.D)
            gw_ih, gw_hh, gb_ih, gb_hh = self._enc_w(G, l, d.D)
            need_dx = l > 0 or emb_grad
            off = l * d.D * d.H
            check(lib.dvae_lstm_seq_bwd_ex(ptr(x), I, T, B, I, d.H, d.D, ptr_array(w_ih), ptr_array(w_hh), None, None,
                                        0, 0, ptr(lengths), ptr(self.e_hs[l]), d.D * d.H, ptr(self.e_gates[l]),
                                        ptr(self.e_cs[l]), ptr(g_in), d.D * d.H, g_ctx.data_ptr() + 4 * off, None,
                                        d.C, d.H, ptr(g_out) if need_dx else None, I, ptr_array(gw_ih),
                                        ptr_array(gw_hh), ptr_array(gb_ih), ptr_array(gb_hh), None, None, 0, 0,
                                        ptr(self.state_ws), ptr(self.lstm_bwd_planes), st), "dvae_lstm_seq_bwd(enc)")
            if l > 0 and p > 0.0:
                check(lib.dvae_dropout(ptr(g_out), I, T * B, I, p, ptr(self.seed_dev), SALT_ENC_LAYER + l,
                                       ptr(g_out), I, 0, st), "dvae_dropout(bwd)")
            g_in = g_out
        self._enc_g_in = g_in
        if emb_grad and last == 0:
            check(lib.dvae_embedding_bwd(ptr(g_in), d.E, ptr(inputs), inputs.stride(0), inputs.stride(1), T, B, p,
                                         ptr(self.seed_dev), SALT_ENC_EMB, -1, 0, ptr(G["encoder.embedding.weight"]),
                                         st), "dvae_embedding_bwd")

    def randn_eps(self, salt_offset=0):
        """N(0,1) reparameterisation noise from the step seed; `salt_offset` separates several draws under one seed."""
        check(self.lib.dvae_randn(ptr(self.eps), self.eps.numel(), ptr(self.seed_dev), SALT_EPS + salt_offset,
                                  _lib.stream_ptr()), "dvae_randn")
        return self.eps

    def recount_lengths(self, tokens, lengths_out, eos, pad=0, min_len=1):
        """scripts/evaluation/consistency.py:186-190 on the device: length = T - #(EOS or PAD tokens), at least min_len."""
        check(self.lib.dvae_recount_lengths(ptr(tokens), tokens.stride(0), tokens.stride(1), tokens.size(0), tokens.size(1),
                                            eos, pad, min_len, ptr(lengths_out), _lib.stream_ptr()), "dvae_recount_lengths")
        return lengths_out
