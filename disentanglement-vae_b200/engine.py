"""Graph-captured data-parallel training engine: the reference's train-step body
(`run.py:217-276`: forward -> compute_all_losses -> backward -> clip_grad_norm_(5.0) -> [adversary steps] ->
Adam.step -> zero_grad -> [MI-estimator steps]) as one fixed sequence of C-ABI kernel launches over pre-allocated
buffers, replayed as CUDA graphs.  The forward + backward pass is one ordered list of stages (`TrainEngine._stage_list`),
each ending where a bucket of the flat gradient buffer is final: four for a recurrent encoder of two or more layers, two
otherwise.  One GPU runs the stages back to back.  When world_size > 1, bucket k is summed over the ranks from the end of
stage k on: by the repo's all-reduce kernel inside the one step graph (four stages; peer-to-peer at two ranks, NVSwitch
multicast beyond), or by NCCL between stage graphs (two stages, or when the kernel's start-up self-test fails on any rank).

Same kernels and the same `StepPlan` as the drop-in autograd path (`functions.py`); what the engine removes is
per-op host work (autograd bookkeeping, ctypes marshalling, allocator traffic).

Variants of the step (all with the reference's semantics):
  * teacher_forcing_prob == 1: whole-sequence decoder launches (the headline path).
  * teacher_forcing_prob  < 1: one coin per decoding step from a host RNG (vae/model.py:463), uploaded as an int32
    vector; the decoder advances step by step and the vocabulary-sampling kernels skip forced steps ON THE DEVICE, so
    the captured graph is the same for every draw.
  * adversarial_loss / mi_loss models (run.py:254-276): the encoder / heads / decoder / vocabulary path runs through the
    plan as above; the small objectives on the latent spaces (adversaries, CLUB estimators) run eagerly through their
    autograd Functions (`functions.py`, C-ABI kernels) and hand d(loss)/dz to the fused heads' backward.  Single GPU,
    no graph.
  * evaluation (eval_step / eval_steps, run.py:347-423): the same forward with train=False, the losses and corpus BLEU of
    the predictions, one graph per decode regime; no backward, no optimizer, training state untouched.

Batch shapes: the engine is built for (B, T) and takes any batch [B', T'] with B' <= B and 2 <= T' <= T.  A narrower batch
is padded to T with PAD columns in the pinned staging block (exact: the encoder reads the lengths, the loss keeps position
(t, b) only when t + 1 < len_b, and the vocabulary kernels run over those positions only).  A batch with fewer rows runs
on a `_Shape` of its own at (B', T) -- plan, staging block, graphs -- built on its first batch and cached; parameters,
gradients, Adam moments, weight planes, counters and random streams are shared.  A batch of the full shape (B, T) runs
exactly the graph the engine had before any other shape was seen.
"""
import functools
import math
import os
import random
from collections import OrderedDict

import numpy as np
import torch
import torch.distributed as dist

from . import _lib
from ._lib import ptr, check
from .plan import StepPlan, Dims
from .losses import get_cyclic_kl_weight
from .dist import stage_buckets


class _Shape:
    """The per-shape state of a TrainEngine at B rows (padded length: the engine's T): its StepPlan, the device block the
    per-step host data lands in with its typed views, the pinned host blocks that fill it (one per ring slot), the
    sampled-decode prediction buffer, the captured train graph(s) and the evaluation buffers / graphs."""

    def __init__(self, eng, B):
        T, d, dev = eng.T, eng.d, eng.device
        self.B = B
        self.plan = StepPlan(eng.model, B, T, dev)
        # the vocabulary projection and its gradients run over the positions the loss keeps only (the row count is read
        # on the device, so the captured step serves every length distribution); nothing the engine returns reads
        # vocabulary outputs at masked positions
        self.plan.live_rows = True
        # Everything the host sends per step lives in ONE device block (typed views below) filled by ONE H2D copy from a ring
        # of pinned host blocks: token ids, lengths, Philox seed, labels, Adam / KL scalars, teacher-forcing coins.  An
        # asynchronous H2D copy reads host memory when it executes, so a slot is rewritten only after the event recorded
        # behind its last use has completed (ADVICE r1: un-synchronised step_resident calls saw a later step's scalars).
        # One row per field: dtype and shape.  The fields follow each other at 16-byte boundaries, except the batch's own
        # padded length T' (the BLEU kernel's row bound): word 5 of the scalar block, which the step does not read, so the
        # block keeps its size.
        fields = {"inputs": (torch.int64, (B, T)), "lengths": (torch.int64, (B,)), "seed": (torch.int64, (1,)),
                  "labels": (torch.float32, (eng.n_dsc, B)), "scal": (torch.float32, (8 + max(d.S, 1),)),
                  "coins": (torch.int32, (max(T - 1, 1),)),          # 1 = teacher-forced step
                  "tlen": (torch.int32, (1,))}
        lay, off = {}, 0
        for name, (dtype, shape) in fields.items():
            nbytes = math.prod(shape) * dtype.itemsize
            if name == "tlen":
                lay[name] = (lay["scal"][0] + 5 * 4, nbytes)
            else:
                lay[name] = (off, nbytes)
                off = (off + nbytes + 15) // 16 * 16
        self.bytes, self.lay = off, lay

        def views(buf):
            return {k: buf[o:o + n].view(fields[k][0]).view(fields[k][1]) for k, (o, n) in lay.items()}
        self.d_stage = torch.zeros(off, device=dev, dtype=torch.uint8)
        dv = views(self.d_stage)
        self.inputs, self.lengths, self.labels, self.d_scal, self.coins, self.tlen = (
            dv[k] for k in ("inputs", "lengths", "labels", "scal", "coins", "tlen"))
        self.coins.fill_(1)
        self.plan.seed_dev = dv["seed"]     # the plan's kernels read the seed from here
        self.preds = torch.zeros(B, T, device=dev, dtype=torch.int64) if eng.sampled else None
        self.h_stage = torch.zeros(eng.NSLOT, off, dtype=torch.uint8).pin_memory()
        self.hv = [{k: v.numpy() for k, v in views(h).items()} for h in self.h_stage]
        for hv in self.hv:
            hv["coins"][:] = 1
            hv["lengths"][:] = 1
            hv["tlen"][:] = T
        self.graphs = None     # captured train step: one graph, or the data-parallel stage graphs
        self.eval = None       # evaluation buffers and graphs, allocated on this shape's first eval_step


class _Carry:
    """The values one stage of a train step hands to a later one (TrainEngine._stages)."""

    def __init__(self, g_z=None):
        # extra gradient on the sampled latents [B, Z] (adversarial / MI objectives), or a callable evaluated after the forward
        self.g_z = g_z
        self.g_top = None             # d(loss)/d(decoder top-layer states): vocabulary backward -> decoder backward
        self.g_ctx = None             # d(loss)/d(encoder context): heads backward -> encoder backward
        self.side_pending = False     # the decoder's layer-0 d_x and embedding-gradient scatter still run on the hoist side stream


class TrainEngine:
    # pinned staging slots for the per-step scalar block (ring, guarded by CUDA events) = how many steps the host may run ahead
    NSLOT = max(3, int(os.environ.get("DVAE_ENGINE_SLOTS", "4")))
    # batch sizes B' < B kept besides the full shape, least recently used evicted first.  A run through RatioSampler or a
    # DataLoader with drop_last=False meets one (its last batch); evaluation over a dev set adds at most one more.
    MAX_EXTRA_SHAPES = 2

    def __init__(self, model, params, B, T, lr=None, total_steps=None, use_graph=True, max_norm=5.0,
                 process_group=None, seed=None, teacher_forcing_prob=None):
        model._require_cuda()
        self.model, self.params, self.B, self.T = model, params, B, T
        self.lib = _lib.load()
        self.device = model._flat.device
        self.d = d = Dims(model)
        self.world = dist.get_world_size(process_group) if (dist.is_available() and dist.is_initialized()) else 1
        self.rank = dist.get_rank(process_group) if self.world > 1 else 0
        self.pg = process_group
        self.max_norm = max_norm
        self.lr = float(params["learn_rate"] if lr is None else lr)
        self.total_steps = total_steps
        self.lambdas = params["lambdas"]
        if total_steps is None and any(v == "cyclic" for v in self.lambdas.values()):
            raise ValueError("a \"cyclic\" lambda needs total_steps (= epochs * len(dataloader), run.py:215-216)")
        self.tf_prob = float(params.get("teacher_forcing_prob", 1.0) if teacher_forcing_prob is None else teacher_forcing_prob)
        self.sampled = self.tf_prob < 1.0
        self.aux = bool(len(model.adversaries) or len(model.mi_estimators))
        if self.aux and self.world > 1:
            raise NotImplementedError("adversarial_loss / mi_loss models train on one GPU through the engine (their private "
                                      "optimizers are not all-reduced)")
        self.n = model._flat_numel
        f32 = dict(device=self.device, dtype=torch.float32)
        self.flat = model._flat[:self.n]
        self.use_graph = use_graph and not self.aux
        self._nvls = None
        # DVAE_DP_NVLS=0 skips the exchange kernel: the one way to run the NCCL fallback where the kernel works (tests)
        if self.world > 1 and self.use_graph and os.environ.get("DVAE_DP_NVLS", "1") != "0":
            self._setup_nvls()          # gradient buffer in multicast memory (self.grad), or None: NCCL exchanges
        if self._nvls is None:
            self.grad = torch.zeros(self.n, **f32)
        self.m = torch.zeros(self.n, **f32)
        self.v = torch.zeros(self.n, **f32)
        self.G = model.grad_views(self.grad)
        named = dict(model.named_parameters())
        for n in model._layout:
            named[n].grad = self.G[n]
        # per-step scalars live in device memory so one captured graph serves every step
        self.n_dsc = max(sum(1 for o in d.dsc_out if o > 0), 1)
        self.hyper = torch.zeros(8, **f32)           # lr, beta1, beta2, eps, step
        self.kl_w = torch.zeros(max(d.S, 1), **f32)
        self.sumsq = torch.zeros(1, **f32)
        self.red_ws = torch.zeros(1032, **f32)
        self._full = self._sh = _Shape(self, B)     # _sh: the shape of the most recent step
        self._extra = OrderedDict()                   # B' -> _Shape, least recently used first
        self._last_T = T                              # padded length of the most recent training step's batch
        self._eval_last = None                        # (shape, T') of the most recent evaluation batch
        ns = self.NSLOT
        self.h_outs = torch.zeros(ns, self._full.plan.out.numel(), dtype=torch.float32).pin_memory()
        # the evaluation result ring, shared by the shapes like h_outs (allocated on the first eval_step)
        self._eval_ring = None
        self.h_out = self.h_outs[0]
        self._slot_ev = [None] * ns
        self._slot = -1
        self.step_idx = 0          # global step: the cyclic-KL schedule's `step` (run.py:215)
        self.adam_step = 0         # optimizer steps taken (Adam bias correction); differs from step_idx after a resume
        base = int(params.get("random_seed", 10)) if seed is None else int(seed)
        if seed is None:
            base += 7919 * self.rank          # every data-parallel shard draws its own eps / dropout / coin streams
        self._gen = torch.Generator().manual_seed(base)
        self._pyrand = random.Random(base)
        # evaluation draws its eps / coins from streams of its own, so that eval_step never shifts the training streams
        self._eval_gen = torch.Generator().manual_seed(base + 0x5EED)
        self._eval_pyrand = random.Random(base + 0x5EED)
        self._stages = self._stage_list()
        if self.world > 1:          # bucket k: the gradients final once stage k has run, summed over the ranks from there
            self._buckets = stage_buckets(model, self.grad, len(self._stages))
            self._comm = torch.cuda.Stream(device=self.device)
        # step counter in device memory, from which the exchange kernels derive their barrier epochs
        self._dp_ctr = torch.zeros(1, dtype=torch.int32, device=self.device)
        self._side = None
        self.label_names = [n for n, o in zip(d.space_names, d.dsc_out) if o > 0]
        self.last_aux = {}
        self.fixed_eps = None
        self._wplanes, self._plane_token = [], object()
        if os.environ.get("DVAE_WEIGHT_PLANES", "1") != "0" and not d.bow:
            self._alloc_weight_planes()

    # ---- the per-shape state of the most recent step ------------------------------------------------------------
    # After a step on a full (B, T) batch these are the full shape's: what they have always been.
    plan = property(lambda self: self._sh.plan, doc="StepPlan of the most recent step (utils.LatentLog.append(engine.plan, "
                                                    "ids) logs its rows: B' of them after a short batch)")
    inputs = property(lambda self: self._sh.inputs, doc="[B', T] device token ids of the most recent step (PAD beyond T')")
    lengths = property(lambda self: self._sh.lengths, doc="[B'] device lengths of the most recent step")
    labels = property(lambda self: self._sh.labels, doc="[n_dsc, B'] device labels of the most recent step")
    coins = property(lambda self: self._sh.coins, doc="[T - 1] int32 device teacher-forcing coins (1 = forced)")
    preds = property(lambda self: self._sh.preds, doc="[B', T] device decoder inputs of a sampled-decode step, or None")
    d_scal = property(lambda self: self._sh.d_scal)
    _eval = property(lambda self: self._sh.eval)

    def _shape(self, B):
        """Make the shape of B rows current: the full shape, or a cached / new short one (evicting the least recently
        used beyond MAX_EXTRA_SHAPES)."""
        if B == self.B:
            sh = self._full
        else:
            sh = self._extra.pop(B, None)
            if sh is None:
                if len(self._extra) >= self.MAX_EXTRA_SHAPES:
                    torch.cuda.synchronize(self.device)      # enqueued steps may still read its graphs and blocks
                    self._extra.popitem(last=False)
                sh = _Shape(self, B)
            self._extra[B] = sh
        self._sh = sh
        return sh

    def _check_shape(self, B, T, where):
        if not (1 <= B <= self.B and 2 <= T <= self.T):
            raise ValueError(f"{where}: a batch of shape ({B}, {T}); this engine was built for ({self.B}, {self.T}) and "
                             f"takes [B', T'] batches with 1 <= B' <= {self.B} and 2 <= T' <= {self.T}")

    def _host_batch(self, inputs, lengths, labels, where):
        """Checks a HOST batch against the engine's shape; returns (inputs, lengths, per-label rows) as numpy arrays."""
        X = inputs.numpy() if torch.is_tensor(inputs) else np.asarray(inputs)
        L = lengths.numpy() if torch.is_tensor(lengths) else np.asarray(lengths)
        if X.ndim != 2:
            raise ValueError(f"{where}: inputs must be [B', T'], got shape {tuple(X.shape)}")
        B, T = X.shape
        self._check_shape(B, T, where)
        if L.shape != (B,):
            raise ValueError(f"{where}: lengths has shape {tuple(L.shape)}, expected ({B},) for inputs of shape ({B}, {T})")
        if int(L.max()) > T:
            raise ValueError(f"{where}: a length of {int(L.max())} exceeds the batch's padded length T' = {T} "
                             f"(engine shape ({self.B}, {self.T}))")
        Ys = []
        for n in self.label_names:
            y = labels[n]
            y = (y.numpy() if torch.is_tensor(y) else np.asarray(y)).reshape(-1)
            if y.shape != (B,):
                raise ValueError(f"{where}: labels['{n}'] has {y.size} elements, expected {B} (inputs of shape ({B}, {T}))")
            Ys.append(y)
        return X, L, Ys

    # ---- weight planes: fp16 (hi, lo) operand tiles of the LSTM input weights and of W_out^T, refreshed once per step ------
    def _alloc_weight_planes(self):
        """Every GEMM that reads an LSTM input weight (x . W_ih^T forward, dG . W_ih backward) or W_out as [K, N] (d_h = P . W_out)
        would otherwise re-convert the fp32 matrix in every CTA; the engine knows the weights change exactly once per step."""
        lib, P = self.lib, self.model._P
        names = [n for n in P if (".recurrent.weight_ih_" in n)]
        todo = [(n, True, True) for n in names] + [("decoder.linear.weight", False, True)]
        for n, normal, transposed in todo:
            w = P[n]
            R, C = w.shape
            if R * C < (1 << 14) or (w.data_ptr() & 15):
                continue
            mk = lambda tr: torch.empty(lib.dvae_weight_planes_floats(R, C, tr), device=self.device, dtype=torch.float32)
            self._wplanes.append((w, mk(0) if normal else None, mk(1) if transposed else None))

    def _register_weight_planes(self):
        if not self._wplanes or _lib.planes_owner is self._plane_token:
            return
        check(self.lib.dvae_weight_planes_clear(), "dvae_weight_planes_clear")
        for w, pl, plt in self._wplanes:
            check(self.lib.dvae_weight_planes_register(ptr(w), w.size(0), w.size(1), ptr(pl), ptr(plt)), "dvae_weight_planes_register")
        _lib.planes_owner = self._plane_token

    # ---- the kernel sequences ------------------------------------------------------------------
    def _hoisted(self, sampled):
        """Whether the decoder's encoder-independent work runs on the hoist side stream (self._side) in a step."""
        return os.environ.get("DVAE_HOIST", "1") != "0" and not self.d.bow and not sampled

    def _forward(self, train=True, sampled=None, preds=None):
        """Forward pass of one step up to the reconstruction loss.  The defaults are the training step; eval_step passes
        train=False (no dropout) and its own decode regime / prediction buffer."""
        pl, P, m = self.plan, self.model._P, self.model
        sampled = self.sampled if sampled is None else sampled
        preds = self.preds if preds is None else preds
        n_pl = len(self._wplanes)
        n_ih = sum(1 for w, a, b in self._wplanes if a is not None)      # LSTM input weights come first, W_out^T last
        if n_pl:               # operand planes of the weights the encoder reads first: one launch, first thing in the step
            check(self.lib.dvae_weight_planes_refresh_ex(0, n_ih, _lib.stream_ptr()), "dvae_weight_planes_refresh")
        # unpack the per-step scalar block (device-to-device, inside the graph)
        self.hyper[:5].copy_(self.d_scal[:5])
        self.kl_w.copy_(self.d_scal[8:8 + self.kl_w.numel()])
        if self.fixed_eps is not None:      # replay given reparameterisation noise (tests; forward(eps=...) of the drop-in path)
            pl.eps.copy_(self.fixed_eps[:pl.B])      # a B' < B step reads the first B' rows
        else:
            pl.randn_eps()
        # the decoder's input embeddings, its layer-0 input projection and the W_out operand planes do not depend on
        # the encoder (teacher forcing): they run on a side stream under the encoder's recurrences (64 of 148 SMs)
        cur = torch.cuda.current_stream()
        hoist = self._hoisted(sampled)
        # W_out^T planes (10 MB at cfg 2) are read by the vocabulary backward only: not refreshed for an evaluation
        refresh_wt = n_pl > n_ih and train
        fork_prep = None
        if hoist:
            if self._side is None:
                self._side = torch.cuda.Stream(device=self.device)

            def fork_prep():      # forked behind the encoder's layer-0 projection GEMMs, which fill the machine themselves
                self._side.wait_stream(cur)
                with torch.cuda.stream(self._side):
                    pl.decode_prepare(P, self.inputs, m.sos_token_idx, train)
                    if refresh_wt:
                        check(self.lib.dvae_weight_planes_refresh_ex(n_ih, n_pl - n_ih, _lib.stream_ptr()), "dvae_weight_planes_refresh")
        if refresh_wt and not hoist:
            check(self.lib.dvae_weight_planes_refresh_ex(n_ih, n_pl - n_ih, _lib.stream_ptr()), "dvae_weight_planes_refresh")
        pl.encode(P, self.inputs, self.lengths, train, after_l0_proj=fork_prep)
        pl.heads(P, pl.ctx, pl.eps, self.labels, self.kl_w)
        if hoist:
            cur.wait_stream(self._side)
        if sampled:
            # vae/model.py:457-472: position i's input is inputs[:, i] when its coin is heads, else the token sampled from
            # position i's logits; preds doubles as decoder-input buffer and as `token_predictions`
            preds.copy_(self.inputs)
            preds[:, 0].fill_(m.sos_token_idx)
            h_top = pl.decode_sampled(P, preds, self.coins, train)
        else:
            h_top = pl.decode_forced(P, self.inputs, m.sos_token_idx, train)
        pl.vocab_ce(P, h_top, self.inputs, self.lengths)
        return h_top

    # The train step's forward + backward pass is a list of stages (_stage_list); stage k ends with gradient bucket k final
    # (dist.stage_buckets), which data-parallel training sums over the ranks from there.  Stages pass values on in a _Carry.
    def _stage_list(self):
        """A recurrent encoder of two or more layers: forward + vocabulary backward (-> decoder.linear.*) | decoder
        backward (-> decoder embedding + LSTM) | heads + encoder layers Le-1..1 (-> upper encoder + heads) | encoder layer
        0 + embedding (-> the rest).  Bag-of-words or one-layer encoders: forward + vocabulary and decoder backward (->
        decoder.*) | heads + encoder (-> the rest).  Each stage is a tuple of pieces run in order."""
        d = self.d
        if d.bow or d.Le < 2:
            return ((self._fwd_vocab_bwd, self._decoder_bwd), (self._heads_encoder_bwd,))
        upper = functools.partial(self._heads_encoder_bwd, layers=(d.Le - 1, 1))
        return ((self._fwd_vocab_bwd,), (self._decoder_bwd,), (upper,), (self._encoder_l0_bwd,))

    def _fwd_vocab_bwd(self, c):
        h_top = self._forward()
        if callable(c.g_z):
            c.g_z = c.g_z()
        c.g_top = self.plan.vocab_ce_bwd(self.model._P, self.G, h_top, self.inputs, self.lengths, None)

    def _decoder_bwd(self, c):
        # weight-gradient GEMMs of each layer keep running on side streams while the next layer's recurrence starts
        check(self.lib.dvae_defer_joins(1), "dvae_defer_joins")
        c.side_pending = self._hoisted(self.sampled)
        self.plan.decode_bwd(self.model._P, self.G, c.g_top, emb_grad="decoder.embedding.weight" in self.model._layout,
                             aux_stream=self._side if c.side_pending else None)

    def _heads_encoder_bwd(self, c, layers=None):
        pl = self.plan
        check(self.lib.dvae_defer_joins(1), "dvae_defer_joins")
        c.g_ctx = pl.heads_bwd(self.model._P, self.G, pl.ctx, pl.eps, self.labels, self.kl_w, pl.g_hid, g_z=c.g_z)
        pl.encode_bwd(self.model._P, self.G, self.inputs, self.lengths, c.g_ctx,
                      emb_grad="encoder.embedding.weight" in self.model._layout, layers=layers)

    def _encoder_l0_bwd(self, c):
        check(self.lib.dvae_defer_joins(1), "dvae_defer_joins")
        self.plan.encode_bwd(self.model._P, self.G, self.inputs, self.lengths, c.g_ctx,
                             emb_grad="encoder.embedding.weight" in self.model._layout, layers=(0, 0))

    def _fwd_bwd(self, c, stages=None, after_stage=None):
        """Runs `stages` (default: all of them, the whole forward + backward pass) back to back, passing values on in the
        _Carry `c`: side-stream work stays detached until their end, where every side stream is joined.
        `after_stage(k, c)` runs at the end of stage k."""
        try:
            for k, stage in enumerate(self._stages if stages is None else stages):
                for piece in stage:
                    piece(c)
                if after_stage is not None:
                    after_stage(k, c)
        finally:
            check(self.lib.dvae_join_side_streams(_lib.stream_ptr()), "dvae_join_side_streams")
        if c.side_pending:          # the decoder's layer-0 d_x and embedding-gradient scatter are joined too
            torch.cuda.current_stream().wait_stream(self._side)
            c.side_pending = False

    def _step(self, exchange=False):
        """forward + backward + clip + Adam.  exchange (one-graph data parallel): each bucket's exchange starts inside the
        step, at the end of its stage."""
        after_stage = None
        if exchange:
            check(self.lib.dvae_counter_increment(ptr(self._dp_ctr), _lib.stream_ptr()), "dvae_counter_increment")
            after_stage = lambda k, c: self._signal(k, self._side if c.side_pending else None)      # noqa: E731
        self._fwd_bwd(_Carry(), after_stage=after_stage)
        self._optim()

    def _setup_nvls(self):
        """The flat gradient buffer as a symmetric allocation bound to an NVSwitch multicast object, plus a barrier block,
        for the repo's own all-reduce kernel (csrc/nvls.cu).  Two phases -- allocate + exchange handles, then a self-test
        on known values with a 5 s soft timeout in the kernel's barrier -- and after each the ranks agree (all-reduce MIN
        of an ok flag; no other collective sits on a path a failing rank could skip).  Unless every rank passes both, all
        ranks keep the NCCL exchange -- said loudly on stderr, never silently."""
        import sys
        import ctypes as C

        def agreed(ok, why, phase):
            flag = torch.tensor([1 if ok else 0], dtype=torch.int32, device=self.device)
            torch.cuda.synchronize()
            dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self.pg)
            if int(flag.item()) == 1:
                return True
            print(f"[dvae_b200] rank {self.rank}: in-graph gradient exchange unavailable ({phase}: {why or 'another rank failed'}); "
                  "using NCCL all-reduce between stage graphs", file=sys.stderr, flush=True)
            return False

        # two GPUs: plain peer-to-peer loads / stores move a third of the bytes of the switch detour (measured 1.35 ms per cfg2
        # step with multimem against 1.25 peer-to-peer at N = 2; multimem 1.25 against NCCL's 1.51 at N = 4)
        mode = "p2p" if self.world == 2 else "nvls"
        n_pad = (self.n + 3) // 4 * 4
        ok, why, st = True, "", {}
        try:
            import torch.distributed._symmetric_memory as symm
            grp = self.pg if self.pg is not None else dist.group.WORLD
            buf = symm.empty(n_pad, dtype=torch.float32, device=self.device)
            hb = symm.rendezvous(buf, group=grp)
            bar = symm.empty(int(self.lib.dvae_nvls_barrier_words()), dtype=torch.int32, device=self.device)
            bar.zero_()
            hbar = symm.rendezvous(bar, group=grp)
            if mode != "p2p" and not hb.multicast_ptr:
                raise RuntimeError("no multicast address (NVSwitch multicast unavailable)")
            buf.fill_(float(self.rank + 1))
            st = dict(buf=buf, bar=bar, hb=hb, hbar=hbar, mc=int(hb.multicast_ptr), mode=mode,
                      bar_ptrs=(C.c_void_p * self.world)(*[int(p) for p in hbar.buffer_ptrs]),
                      buf_ptrs=[int(p) for p in hb.buffer_ptrs])
        except Exception as e:  # noqa: BLE001 -- any failure means "use NCCL", decided by all ranks together
            ok, why = False, repr(e)[:200]
        if not agreed(ok, why, "symmetric memory"):      # also the barrier behind every rank's fill_ / zero_
            return
        try:
            one = torch.ones(1, dtype=torch.int32, device=self.device)
            err = torch.zeros(1, dtype=torch.int32, device=self.device)
            if mode == "p2p":
                peers = (C.c_void_p * self.world)(*st["buf_ptrs"])
                check(self.lib.dvae_p2p_all_reduce(peers, n_pad, st["bar_ptrs"], self.rank, self.world, ptr(one), 1, 0, 0,
                                                   5_000_000_000, ptr(err), _lib.stream_ptr()), "dvae_p2p_all_reduce")
            else:
                check(self.lib.dvae_nvls_all_reduce(st["mc"], n_pad, st["bar_ptrs"], self.rank, self.world, ptr(one), 1, 0, 0,
                                                    5_000_000_000, ptr(err), _lib.stream_ptr()), "dvae_nvls_all_reduce")
            torch.cuda.synchronize()
            want = float(self.world * (self.world + 1) // 2)
            if int(err.item()) != 0 or not bool((st["buf"] == want).all()):
                raise RuntimeError("timeout or wrong sums")
        except Exception as e:  # noqa: BLE001
            ok, why = False, repr(e)[:200]
        if not agreed(ok, why, "self-test"):
            return
        st["buf"].zero_()
        if not agreed(True, "", "zero"):                   # every rank's buffer is zero before anyone's first step writes to it
            return
        self.grad = st["buf"][:self.n]
        self._nvls = st

    # CTAs of the exchange kernel per bucket of the four-stage step: early buckets finish under hundreds of us of backward
    # pass, the last one is (nearly) exposed
    XCHG_CTAS = (16, 16, 32, 64)

    def _signal(self, k, extra=None):
        """Bucket k's gradients are final once everything enqueued so far, the detached side-stream work and `extra` have
        run: start its exchange there, beside the rest of the backward pass -- as graph nodes on the library's signal
        stream, one all-reduce kernel per view."""
        import ctypes as C
        out = C.c_void_p()
        check(self.lib.dvae_fork_after(1, extra.cuda_stream if extra is not None else None, _lib.stream_ptr(), C.byref(out)),
              "dvae_fork_after")
        nv = self._nvls
        ctas = self.XCHG_CTAS[k]
        for j, v in enumerate(self._buckets[k]):
            off = v.data_ptr() - nv["buf"].data_ptr()
            n = (v.numel() + 3) // 4 * 4
            if nv["mode"] == "p2p":
                peers = (C.c_void_p * self.world)(*[bp + off for bp in nv["buf_ptrs"]])
                check(self.lib.dvae_p2p_all_reduce(peers, n, nv["bar_ptrs"], self.rank, self.world, ptr(self._dp_ctr),
                                                   16, 2 * k + j + 1, ctas, 0, None, out.value), "dvae_p2p_all_reduce")
            else:
                check(self.lib.dvae_nvls_all_reduce(nv["mc"] + off, n, nv["bar_ptrs"], self.rank, self.world, ptr(self._dp_ctr),
                                                    16, 2 * k + j + 1, ctas, 0, None, out.value), "dvae_nvls_all_reduce")

    def _one_graph_dp(self):
        """Data parallel as ONE graph per step, the exchanges being the repo's all-reduce kernels inside it (csrc/nvls.cu):
        needs the kernel set up, graphs on and the four-bucket split.  Otherwise: stage graphs (or eager stages) with NCCL
        between them, whose ends also end the overlap of the weight-gradient GEMMs with the next recurrence."""
        return self._nvls is not None and self.use_graph and len(self._stages) == len(self.XCHG_CTAS)

    @property
    def exchange_mode(self):
        """How this engine exchanges gradients: none (one rank) | p2p | nvls (the repo's kernel inside the one-graph step,
        peer-to-peer at two ranks, NVSwitch multicast beyond) | nccl+stages (NCCL between stage graphs: the fallback)."""
        if self.world == 1:
            return "none"
        return self._nvls["mode"] if self._one_graph_dp() else "nccl+stages"

    def _optim(self):
        st = _lib.stream_ptr()
        check(self.lib.dvae_grad_sumsq(ptr(self.grad), self.n, ptr(self.sumsq), ptr(self.red_ws), st), "dvae_grad_sumsq")
        check(self.lib.dvae_clip_adam(ptr(self.flat), ptr(self.grad), ptr(self.m), ptr(self.v), self.n, ptr(self.sumsq),
                                      self.max_norm, 1.0 / self.world, ptr(self.hyper), 1, st), "dvae_clip_adam")

    # ---- adversarial / MI objectives (run.py:254-276), eager ----------------------------------------------------
    def _latents(self, z):
        from .model import Params
        pl, d, lat, off = self.plan, self.d, {}, 0
        for n, zs in zip(d.space_names, d.space_dims):
            lat[n] = Params(z[:, off:off + zs], pl.mu[:, off:off + zs], pl.logvar[:, off:off + zs])
            off += zs
        return lat

    def _run_aux(self):
        from . import losses
        from .functions import adversary_logits
        m, pl = self.model, self.plan
        box = {}

        def aux_grad():
            # the auxiliary objectives read the sampled latents; their gradient w.r.t. z joins the heads' backward
            z = pl.z.detach().clone().requires_grad_(True)
            lat = self._latents(z)
            Y = {n: self.labels[i].reshape(-1, 1) for i, n in enumerate(self.label_names)}
            A = losses.compute_adversarial_losses(m, adversary_logits(m, lat), Y)
            M = losses.compute_mi_losses(m, lat, beta=0.01)          # run.py:239: mi_loss_weight = 0.01
            aux = A["total_adv_loss"] + M["total_mi"]
            if aux.requires_grad:
                aux.backward(retain_graph=True)      # also leaves the entropy-term gradients in the adversaries' .grad (run.py:254)
            box.update(A=A, M=M, z=z)
            return z.grad.contiguous() if z.grad is not None else None

        self._fwd_bwd(_Carry(g_z=aux_grad))
        A, M, z = box["A"], box["M"], box["z"]
        for name, dsc_loss in A["idv_adv_dsc_losses"].items():      # run.py:256-260
            m.adversaries[name].optimizer_step(dsc_loss)
        self._optim()                                                # clip_grad_norm_ + optimizer.step + zero_grad
        est_losses = {}
        for pair in M["idv_mi_estimates"]:                           # run.py:264-276
            est = m.mi_estimators[pair]
            n1, n2 = pair.split('-')
            lat = self._latents(z.detach())
            mi_loss = est.learning_loss(lat[n1].z, lat[n2].z)
            est.optimizer_step(mi_loss)
            est_losses[pair] = mi_loss
        self.last_aux = {"total_adv_loss": A["total_adv_loss"], "total_mi": M["total_mi"],
                         "idv_adv_losses": A["idv_adv_losses"], "idv_adv_dsc_accs": A["idv_adv_dsc_accs"],
                         "idv_mi_estimates": M["idv_mi_estimates"], "mi_estimator_loss": est_losses}

    def weight_planes(self):
        """Context manager for callers that drive the plan's kernel sequences themselves (bench.py's per-kernel timings):
        current planes, registry on inside the block."""
        import contextlib

        @contextlib.contextmanager
        def cm():
            self._register_weight_planes()
            if self._wplanes:
                check(self.lib.dvae_weight_planes_refresh(_lib.stream_ptr()), "dvae_weight_planes_refresh")
                check(self.lib.dvae_weight_planes_enable(1), "dvae_weight_planes_enable")
            try:
                yield self
            finally:
                if self._wplanes:
                    check(self.lib.dvae_weight_planes_enable(0), "dvae_weight_planes_enable")
        return cm()

    def _run(self, body=None):
        # the registry is consulted while kernels are ENQUEUED (eager steps, graph capture): on around this engine's launches only
        self._register_weight_planes()
        if self._wplanes:
            check(self.lib.dvae_weight_planes_enable(1), "dvae_weight_planes_enable")
        try:
            return (body or self._run_inner)()
        finally:
            if self._wplanes:
                check(self.lib.dvae_weight_planes_enable(0), "dvae_weight_planes_enable")

    def _run_inner(self):
        if self.aux:
            return self._run_aux()
        if self.use_graph and self._sh.graphs is None:
            self._capture()
        if self.world == 1 or self._one_graph_dp():
            if self.use_graph:
                self._sh.graphs[0].replay()      # one graph: forward, backward (and the exchanges), clip + Adam
            else:
                self._step()
            return
        # NCCL on the communication stream between stage graphs (or eager stages), under the stages that follow
        cur = torch.cuda.current_stream()
        c = _Carry()
        for k, bucket in enumerate(self._buckets):
            if self.use_graph:
                self._sh.graphs[k].replay()
            else:
                self._fwd_bwd(c, [self._stages[k]])
            if bucket:
                self._comm.wait_stream(cur)
                with torch.cuda.stream(self._comm):
                    for v in bucket:
                        dist.all_reduce(v, op=dist.ReduceOp.SUM, group=self.pg)
        cur.wait_stream(self._comm)
        if self.use_graph:
            self._sh.graphs[-1].replay()
        else:
            self._optim()

    def _graphs(self, warm_up, bodies):
        """Runs warm_up() eagerly on a side stream (lazy module loading, cudaFuncSetAttribute, allocator, workspaces),
        synchronises, then captures each of `bodies` as a CUDA graph on that stream."""
        s = torch.cuda.Stream(device=self.device)
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            warm_up()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        graphs = []
        for body in bodies:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=s):
                body()
            graphs.append(g)
        torch.cuda.synchronize()
        return tuple(graphs)

    def _capture(self):
        """Captures the current shape's train step.  The warm-up runs no gradient exchange (data parallel: the graph holds
        it, or NCCL runs between the stage graphs), so one rank capturing a new shape never waits on another."""
        def warm_up():
            for _ in range(2):
                self._step()
        snap = (self.flat.clone(), self.m.clone(), self.v.clone())
        if self.world == 1 or self._one_graph_dp():
            bodies = [functools.partial(self._step, exchange=self.world > 1)]
        else:                 # the all-reduces sit between the graphs (NCCL on its own stream)
            c = _Carry()
            bodies = [functools.partial(self._fwd_bwd, c, [stage]) for stage in self._stages] + [self._optim]
        graphs = self._graphs(warm_up, bodies)
        # undo the warm-up updates so that capture leaves the training state untouched
        self.flat.copy_(snap[0]); self.m.copy_(snap[1]); self.v.copy_(snap[2])
        self.grad.zero_()
        self._sh.graphs = graphs

    # ---- per-step host scalars -----------------------------------------------------------------
    def _acquire_slot(self):
        self._slot = (self._slot + 1) % self.NSLOT
        ev = self._slot_ev[self._slot]
        if ev is not None:
            ev.synchronize()
        return self._slot

    def _fill_scalars(self, hv, eval_tf=None, T=None):
        """Adam hyper-parameters and step count, KL weights (cyclic value of this global step), dropout / noise seed, the
        batch's padded length T (default: the engine's) and the teacher-forcing coins of this step, written into a pinned
        host block.  eval_tf (an evaluation's teacher-forcing probability): "cyclic" KL weights are 1.0 (run.py:374-375),
        seed and coins come from the evaluation streams."""
        T = self.T if T is None else T
        hv["tlen"][0] = T
        train = eval_tf is None
        sc = hv["scal"]
        sc[0], sc[1], sc[2], sc[3], sc[4] = self.lr, 0.9, 0.999, 1e-8, float(self.adam_step + 1)
        for i, n in enumerate(self.d.space_names):
            w = self.lambdas[n] if n in self.lambdas else self.lambdas["default"]
            if w == "cyclic":
                w = get_cyclic_kl_weight(self.step_idx, self.total_steps) if train else 1.0
            sc[8 + i] = float(w)
        hv["seed"][0] = int(torch.randint(0, 2 ** 62, (1,), generator=self._gen if train else self._eval_gen))
        tf, rnd = (self.tf_prob, self._pyrand) if train else (eval_tf, self._eval_pyrand)
        if tf < 1.0:          # one coin per decoding step, shared by the batch (vae/model.py:463)
            c = hv["coins"]
            for i in range(T - 1):      # T' - 1 draws, as the reference's loop: the stream of an engine built at T'
                c[i] = 1 if rnd.random() < tf else 0
            c[T - 1:] = 1               # steps past the batch's length read PAD inputs, forced

    def _upload(self, slot, names=None):
        """H2D of a pinned block: the whole block (one copy), or only the named fields (device-resident batches)."""
        sh = self._sh
        if names is None:
            sh.d_stage.copy_(sh.h_stage[slot], non_blocking=True)
        else:
            for k in names:
                o, n = sh.lay[k]
                sh.d_stage[o:o + n].copy_(sh.h_stage[slot, o:o + n], non_blocking=True)

    def _release_slot(self, slot):
        ev = torch.cuda.Event()
        ev.record()
        self._slot_ev[slot] = ev

    def _train_step(self, slot, T, h_out=None):
        """Runs the train step on the staged batch of padded length T (and copies its result block into h_out), releases
        `slot` behind it and advances the step counters."""
        self._last_T = T
        self._run()
        if h_out is not None:
            h_out.copy_(self.plan.out, non_blocking=True)
        self._release_slot(slot)
        self.step_idx += 1
        self.adam_step += 1

    def _pipelined(self, batches, lag, enqueue, result):
        """enqueue(inputs, lengths, labels) -> slot for every batch; yields result(slot) of each, in order, `lag` batches
        behind the one being enqueued: nothing waits for the device but the read of a result `lag` steps old."""
        assert 0 <= lag < self.NSLOT
        pending = []
        for inputs, lengths, labels in batches:
            pending.append(enqueue(inputs, lengths, labels))
            if len(pending) > lag:
                slot = pending.pop(0)
                self._slot_ev[slot].synchronize()
                yield result(slot)
        for slot in pending:
            self._slot_ev[slot].synchronize()
            yield result(slot)

    # ---- public entry points -------------------------------------------------------------------
    def step_resident(self, inputs_dev, lengths_dev, labels_dev):
        """One train step on a batch already in HBM (inputs [B',T'] int64, lengths [B'], labels [n_dsc,B']); returns the
        device result block (plan.out: [0] weighted KL, [1] KL, [2] dsc loss, [3..] per space, [27] reconstruction).
        Asynchronous: may be called back to back without synchronising.  Lengths are checked against T' only when
        T' < T (one device read); a full-width batch is taken without a host round trip."""
        if inputs_dev.dim() != 2:
            raise ValueError(f"step_resident: inputs must be [B', T'], got shape {tuple(inputs_dev.shape)}")
        B, T = inputs_dev.shape
        self._check_shape(B, T, "step_resident")
        if tuple(lengths_dev.shape) != (B,):
            raise ValueError(f"step_resident: lengths has shape {tuple(lengths_dev.shape)}, expected ({B},)")
        if self.label_names and tuple(labels_dev.shape) != (self.n_dsc, B):
            raise ValueError(f"step_resident: labels has shape {tuple(labels_dev.shape)}, expected ({self.n_dsc}, {B})")
        if T < self.T and int(lengths_dev.max()) > T:
            raise ValueError(f"step_resident: a length of {int(lengths_dev.max())} exceeds the batch's padded length "
                             f"T' = {T} (engine shape ({self.B}, {self.T}))")
        sh = self._shape(B)
        slot = self._acquire_slot()
        self._fill_scalars(sh.hv[slot], T=T)
        self._upload(slot, ("seed", "scal", "coins") if self.sampled else ("seed", "scal"))
        if T == self.T:
            self.inputs.copy_(inputs_dev, non_blocking=True)
        else:
            self.inputs[:, :T].copy_(inputs_dev, non_blocking=True)
            self.inputs[:, T:].zero_()
        self.lengths.copy_(lengths_dev, non_blocking=True)
        self.labels.copy_(labels_dev, non_blocking=True)
        self._train_step(slot, T)
        return self.plan.out

    def _enqueue_host_step(self, inputs, lengths, labels, eval_tf=None, where="step_host"):
        """Stage one HOST batch [B', T'] into the next pinned block of its shape (padded to T with PAD columns), enqueue its
        single H2D copy, the step and the D2H copy of the result block; returns the slot (its event completes when the
        losses are in h_outs[slot]).  eval_tf: an evaluation step at that teacher-forcing probability instead (result
        block in the evaluation ring)."""
        X, L, Ys = self._host_batch(inputs, lengths, labels, where)
        B, T = X.shape
        sh = self._shape(B)
        if eval_tf is not None:
            self._eval_setup()
        slot = self._acquire_slot()
        hv = sh.hv[slot]
        if T == self.T:
            hv["inputs"][...] = X
        else:
            hv["inputs"][:, :T] = X
            hv["inputs"][:, T:] = 0
        hv["lengths"][...] = L
        for i, y in enumerate(Ys):
            hv["labels"][i] = y
        self._fill_scalars(hv, eval_tf, T)
        self._upload(slot)
        if eval_tf is not None:
            self._eval_last = (sh, T)
            ev = self._eval
            self._run(lambda: self._eval_run(eval_tf < 1.0))
            ev["h_out"][slot].copy_(ev["out"], non_blocking=True)
            ev["aux"][slot] = self._eval_aux() if self.aux else None
            self._release_slot(slot)
            return slot
        self._train_step(slot, T, self.h_outs[slot])
        return slot

    def step_host(self, inputs, lengths, labels):
        """End-to-end step: HOST tensors in (inputs [B',T'] int64, lengths [B'] int64, labels {name: [B',1]}; B' <= B,
        2 <= T' <= T, lengths <= T', else ValueError), python floats out.  One H2D copy of the staged block, the step, one
        D2H read of the loss block, then a wait."""
        slot = self._enqueue_host_step(inputs, lengths, labels)
        self._slot_ev[slot].synchronize()
        self.h_out = self.h_outs[slot]
        return self.losses_from(self.h_out)

    def train_steps(self, batches, lag=2):
        """Pipelined training loop over an iterable of HOST batches (inputs, lengths, labels): yields the loss dict of every
        step, in order, `lag` steps behind the step being enqueued -- batch k + 1 is staged and uploaded while the GPU runs
        step k, and nothing waits for the device except the read of a result that is `lag` steps old.  Same arithmetic as
        calling step_host() per batch (run.py:217-262), with the same batch shapes; `lag` must be smaller than NSLOT.
        Data parallel: every rank's batches have the same shapes step by step (RatioSampler's default drop_uneven=True
        gives equal shards of a short last batch); unequal shards are not supported."""
        return self._pipelined(batches, lag, functools.partial(self._enqueue_host_step, where="train_steps"),
                               lambda slot: self.losses_from(self.h_outs[slot]))

    def losses_from(self, out, aux=None):
        """The loss dict of `compute_all_losses` from a result block; `aux`: the adversarial / MI values to add (default:
        those of the last training step)."""
        S, NS = self.d.S, _lib.HEADS_NSCALARS
        aux = self.last_aux if aux is None else aux
        o = out.tolist()
        L = {"reconstruction_loss": o[NS], "total_weighted_kl": o[0], "total_kl": o[1], "total_dsc_loss": o[2],
             "idv_kls": {n: o[3 + i] for i, n in enumerate(self.d.space_names)},
             "idv_dsc_losses": {n: o[3 + S + i] for i, n in enumerate(self.d.space_names) if self.d.dsc_out[i] > 0},
             "idv_dsc_accs": {n: o[3 + 2 * S + i] for i, n in enumerate(self.d.space_names) if self.d.dsc_out[i] > 0}}
        L["total_loss"] = o[NS] + o[0] + o[2]
        if self.aux and aux:
            L["total_adv_loss"] = float(aux["total_adv_loss"].detach())
            L["total_mi"] = float(aux["total_mi"].detach())
            for k in ("idv_adv_losses", "idv_adv_dsc_accs", "idv_mi_estimates"):
                L[k] = aux[k]
            L["total_loss"] += L["total_adv_loss"] + L["total_mi"]
        return L

    # ---- evaluation: the body of run.py:evalstep (run.py:347-423) --------------------------------------------------
    # Result block (float32): [0, NS + 5) the training block's layout (heads scalars, [NS] reconstruction loss),
    # [NS + 1] corpus BLEU, then the 10 int64 BLEU counts of dvae_bleu_counts (clipped 1-4, total 1-4, cand / ref length).
    def _eval_setup(self):
        """The current shape's evaluation buffers; the result ring (h_out, aux) is the engine's, shared by the shapes."""
        sh = self._sh
        if sh.eval is not None:
            return sh.eval
        NB = sh.plan.out.numel()
        out = torch.zeros(NB + 20, device=self.device, dtype=torch.float32)
        if self._eval_ring is None:
            self._eval_ring = (torch.zeros(self.NSLOT, out.numel(), dtype=torch.float32).pin_memory(), [None] * self.NSLOT)
        sh.eval = ev = {"out": out, "counts": out[NB:].view(torch.int64), "nb": NB, "graphs": {},
                        "preds": torch.zeros(sh.B, self.T, device=self.device, dtype=torch.int64),
                        "h_out": self._eval_ring[0], "aux": self._eval_ring[1]}
        return ev

    def _eval_body(self, sampled):
        """Eval-mode forward (no dropout, one eps draw), every loss of compute_all_losses and corpus BLEU of the
        predictions against the inputs, into the evaluation result block.  No backward pass, no optimizer."""
        from .losses import bleu_counts_, bleu_score_
        ev, pl, m = self._eval, self.plan, self.model
        preds = ev["preds"]
        self._forward(train=False, sampled=sampled, preds=preds)
        if not sampled:      # teacher forcing: the predictions are the decoder inputs (vae/model.py:455)
            preds.copy_(self.inputs)
            preds[:, 0].fill_(m.sos_token_idx)
        NS, NB = _lib.HEADS_NSCALARS, ev["nb"]
        ev["out"][:NB].copy_(pl.out)
        ev["counts"].zero_()
        # rows end at the batch's own padded length T' (from the staging block): an EOS-less row loses its T'-th token
        bleu_counts_(ev["counts"], self.inputs, preds, m.eos_token_idx, t_max=self._sh.tlen)
        bleu_score_(ev["out"][NS + 1:NS + 2], ev["counts"])

    def _eval_run(self, sampled):
        graphs = self._eval["graphs"]      # the current shape's, keyed by decode regime
        body = functools.partial(self._eval_body, sampled)
        if not self.use_graph:
            body()
        else:
            if sampled not in graphs:      # nothing to undo after the warm-up
                graphs[sampled], = self._graphs(body, [body])
            graphs[sampled].replay()
        if self.world > 1:
            self._eval_all_reduce()

    def _eval_all_reduce(self):
        """Every loss term is a batch mean and the BLEU statistics are counts: scale the means by this shard's B, sum the
        block over the ranks (one all-reduce, float64 -- exact for the counts) and divide by the global batch."""
        from .losses import bleu_score_
        ev, NB, NS = self._eval, self._eval["nb"], _lib.HEADS_NSCALARS
        red = torch.cat([ev["out"][:NB].double() * self._sh.B, ev["counts"].double(),
                         torch.full((1,), float(self._sh.B), device=self.device, dtype=torch.float64)])
        dist.all_reduce(red, op=dist.ReduceOp.SUM, group=self.pg)
        ev["out"][:NB].copy_(red[:NB] / red[-1])
        ev["counts"].copy_(red[NB:NB + 10].round().long())
        bleu_score_(ev["out"][NS + 1:NS + 2], ev["counts"])

    def _eval_aux(self):
        """run.py:evalstep's adversarial / MI terms (compute_adversarial_losses / compute_mi_losses, forward only) on the
        evaluation latents in plan.z / mu / logvar."""
        from . import losses
        from .functions import adversary_logits
        m = self.model
        with torch.no_grad():
            lat = self._latents(self.plan.z)
            Y = {n: self.labels[i].reshape(-1, 1) for i, n in enumerate(self.label_names)}
            A = losses.compute_adversarial_losses(m, adversary_logits(m, lat), Y)
            M = losses.compute_mi_losses(m, lat, beta=0.01)          # compute_all_losses: mi_loss_weight = 0.01
        return {"total_adv_loss": A["total_adv_loss"], "total_mi": M["total_mi"], "idv_adv_losses": A["idv_adv_losses"],
                "idv_adv_dsc_accs": A["idv_adv_dsc_accs"], "idv_mi_estimates": M["idv_mi_estimates"]}

    def _eval_losses(self, slot):
        ev, NS, NB = self._eval, _lib.HEADS_NSCALARS, self._eval["nb"]
        h = ev["h_out"][slot]
        L = self.losses_from(h[:NB], aux=ev["aux"][slot])
        L["bleu"] = float(h[NS + 1])
        L["bleu_counts"] = h[NB:].view(torch.int64).tolist()
        return L

    def eval_step(self, inputs, lengths, labels, teacher_forcing_prob):
        """Validation step (run.py:evalstep, run.py:347-423) on HOST tensors (inputs [B',T'] int64, lengths [B'], labels
        {name: [B',1]}; the shapes step_host takes): eval-mode forward (no dropout, one eps draw), the loss dict of
        compute_all_losses with "cyclic" KL weights at 1.0 (run.py:374-375), plus "bleu" (compute_bleu of the predictions against the inputs) and
        "bleu_counts" (its 10 corpus statistics, which add over batches).  One captured graph per decode regime
        (teacher_forcing_prob == 1: forced decode; < 1: sampled decode, coins drawn per call) and batch shape, one H2D and
        one D2H copy.
        Parameters, optimizer state, step counters and the training random streams are not touched; plan.z / mu / logvar
        hold this batch afterwards (utils.LatentLog.append(engine.plan, ids) logs dev latents); eval_predictions holds
        the predicted tokens.  Data parallel: every rank passes its shard (equal shards) and gets the losses of the
        global batch."""
        slot = self._enqueue_host_step(inputs, lengths, labels, eval_tf=float(teacher_forcing_prob), where="eval_step")
        self._slot_ev[slot].synchronize()
        return self._eval_losses(slot)

    def eval_steps(self, batches, teacher_forcing_prob, lag=2):
        """eval_step over an iterable of HOST batches (inputs, lengths, labels), pipelined as train_steps: yields each
        batch's loss dict `lag` batches behind the one being enqueued.  Sum "bleu_counts" over the batches and pass them
        to losses.bleu_from_counts() for the BLEU of the whole dev set."""
        enqueue = functools.partial(self._enqueue_host_step, eval_tf=float(teacher_forcing_prob), where="eval_steps")
        return self._pipelined(batches, lag, enqueue, self._eval_losses)

    @property
    def eval_predictions(self):
        """[B',T'] token predictions of the last eval_step's batch (device tensor; overwritten by the next one)."""
        if self._eval_last is None:
            return None
        sh, T = self._eval_last
        return sh.eval["preds"][:, :T]

    @property
    def token_predictions(self):
        """[B',T'] decoder inputs of the last step's batch (vae/model.py:455-472): sampled where the coin said so."""
        T = self._last_T
        if self.sampled:
            return self.preds[:, :T]
        p = self.inputs[:, :T].clone()
        p[:, 0] = self.model.sos_token_idx
        return p

    # ---- optimizer state in the reference's checkpoint format (run.py:624-630, vae/utils.py:147-175) -------------
    def _trainable(self):
        name_of = {id(p): n for n, p in self.model.named_parameters()}
        return [(name_of[id(p)], p) for p in self.model.trainable_parameters()]

    def optimizer_state_dict(self):
        """`torch.optim.Adam(model.trainable_parameters(), lr).state_dict()` of this engine's state: what the reference
        stores under "optimizer_state_dict" (run.py:627-628), loadable by its `utils.load_latest_checkpoint`."""
        opt = torch.optim.Adam([p for _, p in self._trainable()], lr=self.lr)
        if self.adam_step > 0:
            Mv, Vv = self.model.grad_views(self.m), self.model.grad_views(self.v)
            for n, p in self._trainable():
                opt.state[p] = {"step": torch.tensor(float(self.adam_step)), "exp_avg": Mv[n].detach().clone(),
                                "exp_avg_sq": Vv[n].detach().clone()}
        return opt.state_dict()

    def load_optimizer_state_dict(self, sd):
        """Inverse of optimizer_state_dict(): accepts the state of the reference's Adam over the same model."""
        tr = self._trainable()
        groups = sd["param_groups"]
        ids = [i for g in groups for i in g["params"]]
        if len(ids) != len(tr):
            raise ValueError(f"optimizer state has {len(ids)} parameters, the model has {len(tr)} trainable ones")
        self.lr = float(groups[0]["lr"])
        Mv, Vv = self.model.grad_views(self.m), self.model.grad_views(self.v)
        self.m.zero_(); self.v.zero_()
        steps = set()
        for i, (n, p) in zip(ids, tr):
            st = sd["state"].get(i)
            if st is None:
                continue
            if tuple(st["exp_avg"].shape) != tuple(p.shape):
                raise ValueError(f"optimizer state of '{n}' has shape {tuple(st['exp_avg'].shape)}, expected {tuple(p.shape)}")
            Mv[n].copy_(st["exp_avg"].to(self.device, torch.float32).reshape(Mv[n].shape))
            Vv[n].copy_(st["exp_avg_sq"].to(self.device, torch.float32).reshape(Vv[n].shape))
            steps.add(int(float(st["step"])))
        if len(steps) > 1:
            raise ValueError(f"per-parameter Adam step counts differ: {sorted(steps)}")
        self.adam_step = steps.pop() if steps else 0

    # the engine can stand in for the reference's `optimizer` object in utils.load_latest_checkpoint / torch.save
    state_dict = optimizer_state_dict
    load_state_dict = load_optimizer_state_dict

    def save_checkpoint(self, ckpt_dir, epoch):
        """run.py:624-630: {model_state_dict, optimizer_state_dict, epoch} -> model_{epoch}.pt"""
        os.makedirs(ckpt_dir, exist_ok=True)
        path = os.path.join(ckpt_dir, f"model_{epoch}.pt")
        torch.save({"model_state_dict": self.model.state_dict(), "optimizer_state_dict": self.optimizer_state_dict(),
                    "epoch": epoch}, path)
        return path

    def load_latest_checkpoint(self, ckpt_dir, steps_per_epoch=None):
        """vae/utils.py:147-175 for this engine; returns (next_epoch, file name or None).  With `steps_per_epoch` the
        global step of the cyclic-KL schedule resumes at next_epoch * steps_per_epoch (run.py:215)."""
        from .utils import load_latest_checkpoint
        _, _, next_epoch, fname = load_latest_checkpoint(self.model, self, ckpt_dir, map_location=self.device)
        if fname is not None and steps_per_epoch is not None:
            self.step_idx = next_epoch * steps_per_epoch
        return next_epoch, fname

    @property
    def h2d_bytes_per_step(self):
        return self._sh.bytes

    @property
    def d2h_bytes_per_step(self):
        return self.h_outs.size(1) * 4
