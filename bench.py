#!/usr/bin/env python
"""Headline benchmark: device-timed training tokens/sec of the disentangled sentence VAE step
(forward + all losses + backward + [NCCL all-reduce] + clip + Adam) at BASELINE.json configs[1]
(the sfu_amazon_100k reproduction shape) on N B200s, plus roofline / CPU-baseline / end-to-end legs.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload cfg1|cfg2|cfg3|cfg4|cfg5]
                    [--dump-outputs DIR]

N > 1 is launched by torchrun (one rank per GPU, NCCL); rank 0 prints ONE JSON line.
--dump-outputs DIR: rank 0 also writes what the last timed step computed as DIR/<name>.npy (see dump_outputs), so that
two builds run with the same arguments (hence the same seeded inputs) can be compared output for output.  Two runs of one
build are not bit-identical: on one B200 (1000 W) cfg2 dumps agreed within 2e-5 of each array's largest magnitude.
Synthetic data of the reference's shape (SURVEY.md 8d), reference initialisation under seed 10.
Workloads: cfg2 = headline; cfg1 (config_example shape), cfg3 (per-GPU shard of the 8 x 64 data-parallel run),
cfg4 (scaled decoder: H 1024, V 50k, T 64), cfg5 (inference: encode + resample decoding, batch 1024) are recorded under
profiles/.
"""
import argparse
import copy
import importlib
import json
import os
import sys
import threading
import time
import zlib

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

PAD, UNK, SOS, EOS = 0, 1, 2, 3

# BASELINE.json configs[1]: reproduction_configs/sfu_amazon_100k/vae_elbo.json with "default": "cyclic"
CFG2 = {"name": "bench/sfu_amazon_100k", "random_seed": 10, "data_dir": "", "combined_dataset": True,
        "dataset_minibatch_ratios": {"sfu": 0.5, "amazon": 0.5}, "checkpoint_dir": "", "glove_path": "",
        "num_train_examples": -1, "lowercase": True, "reverse_input": False, "embedding_dim": 256,
        "hidden_dim": 256, "num_rnn_layers": 2, "bidirectional_encoder": True, "bow_encoder": False,
        "latent_dims": {"total": 64, "polarity": 1, "uncertainty": 1}, "epochs": 20, "batch_size": 128,
        "learn_rate": 3e-4, "encoder_dropout": 0.5, "decoder_dropout": 0.5, "teacher_forcing_prob": 1.0,
        "lambdas": {"default": "cyclic", "polarity": 0.005, "uncertainty": 0.005}, "adversarial_loss": False,
        "mi_loss": False, "train": True, "validate": False, "test": False}
VOCAB, SEQ_T = 10000, 22
TOTAL_STEPS = 20 * 1563          # epochs * len(dataloader) of the reproduction run (SURVEY.md 8d)
LABELS = {"uncertainty": 1, "polarity": 1}
BATCH = 128
UNIFORM_LENGTHS = None
WORKLOAD_NAME = "cfg2"
WORKLOAD = ("cfg2 sfu_amazon_100k reproduction shape: per-GPU batch 128, T=22 (SFU length histogram: min 3, mean ~10, "
            "max 22), V=10000, E=H=256, 2-layer bi-LSTM encoder, 2-layer decoder, Z=64 (uncertainty 1, polarity 1, "
            "content 62), dropout 0.5, teacher forcing 1.0, cyclic KL")


_CFG2_DEFAULTS = dict(CFG2=copy.deepcopy(CFG2), VOCAB=VOCAB, SEQ_T=SEQ_T, TOTAL_STEPS=TOTAL_STEPS, LABELS=dict(LABELS), BATCH=BATCH,
                      UNIFORM_LENGTHS=UNIFORM_LENGTHS, WORKLOAD=WORKLOAD)


def select_workload(name):
    """Rebinds the module-level workload description (BASELINE.json `configs`), always starting from the cfg2 defaults.
    Returns the uniform length range or None (SFU-like length histogram)."""
    global CFG2, VOCAB, SEQ_T, WORKLOAD, TOTAL_STEPS, LABELS, BATCH, UNIFORM_LENGTHS, WORKLOAD_NAME
    d = _CFG2_DEFAULTS
    CFG2, VOCAB, SEQ_T, TOTAL_STEPS, LABELS = copy.deepcopy(d["CFG2"]), d["VOCAB"], d["SEQ_T"], d["TOTAL_STEPS"], dict(d["LABELS"])
    BATCH, UNIFORM_LENGTHS, WORKLOAD = d["BATCH"], d["UNIFORM_LENGTHS"], d["WORKLOAD"]
    WORKLOAD_NAME = name
    if name == "cfg1":       # config_example.json shape (BASELINE configs[0]; SURVEY.md 8 table row 1)
        CFG2 = dict(CFG2, name="bench/config_example", bidirectional_encoder=False, combined_dataset=False,
                    dataset_minibatch_ratios={}, latent_dims={"total": 32, "polarity": 1}, learn_rate=5e-3, batch_size=64,
                    epochs=15, lambdas={"default": "cyclic", "polarity": 0.005})
        VOCAB, SEQ_T, LABELS, BATCH = 10000, 30, {"polarity": 1}, 64
        TOTAL_STEPS = 15 * 1563
        UNIFORM_LENGTHS = (5, 30)
        WORKLOAD = ("cfg1 config_example.json shape: per-GPU batch 64, T=30 (lengths U{5..30}, dSentences-like), V=10000, E=H=256, "
                    "2-layer uni-directional LSTM encoder, 2-layer decoder, Z=32 (polarity 1, content 31), dropout 0.5, "
                    "teacher forcing 1.0, cyclic KL, lr 5e-3 (adversarial_loss off: the ELBO + discriminator step)")
    elif name == "cfg3":     # BASELINE configs[2]: batch 512 data-parallel over 8 GPUs = 64 rows per GPU
        BATCH = 64
        WORKLOAD = WORKLOAD.replace("cfg2 sfu_amazon_100k reproduction shape: per-GPU batch 128",
                                    "cfg3 sfu_amazon_100k model, global batch 512 over 8 GPUs: per-GPU batch 64")
    elif name == "cfg4":     # scaled decoder (SURVEY.md 8 states B = 128, lengths U{16..64})
        CFG2 = dict(CFG2, name="bench/scaled_decoder", hidden_dim=1024)
        VOCAB, SEQ_T = 50000, 64
        UNIFORM_LENGTHS = (16, 64)
        WORKLOAD = ("cfg4 scaled decoder: per-GPU batch 128, T=64 (lengths U{16..64}), V=50000, E=256, H=1024, 2-layer bi-LSTM "
                    "encoder, 2-layer decoder, Z=64, dropout 0.5, teacher forcing 1.0, cyclic KL")
    elif name == "cfg5":
        BATCH = 1024
        WORKLOAD = ("cfg5 inference (consistency-evaluation shape, scripts/evaluation/consistency.py:163-205): batch 1024, T=22, "
                    "V=10000, E=H=256, model in train mode; per resample: fresh latents -> sampled decode (tf=0) -> on-device "
                    "length recount -> re-encode of the sampled sentences -> discriminator logits of both passes; 30 resamples")
    return UNIFORM_LENGTHS


def workload_config(world, graph=True):
    """The `config` object of the JSON line: identical in the b200 and the reference arm."""
    return {"workload": WORKLOAD, "global_batch": BATCH * world, "seq_len": SEQ_T, "parallelism": f"dp{world}",
            "l2": "flushed (256 MiB write) between timed steps", "cuda_graph": bool(graph),
            "tokens": "valid tokens (sum of lengths, incl. SOS/EOS)"}


def synth_batch(rng, B, T=None, V=None, uniform_lengths=None):
    """SURVEY.md 8d: rows [SOS, w..., EOS, PAD...], Zipf(1.0) body tokens, SFU-like lengths (or U{lo..hi}), 10% labels."""
    T = SEQ_T if T is None else T
    V = VOCAB if V is None else V
    if uniform_lengths is not None:
        lengths = rng.integers(uniform_lengths[0], uniform_lengths[1] + 1, B).astype(np.int64)
    else:
        lengths = np.clip(np.round(rng.gamma(9.7, 1.06, B)), 3, T).astype(np.int64)
    lengths[0] = T
    ranks = np.arange(4, V)
    pz = 1.0 / (ranks - 3.0)
    pz /= pz.sum()
    X = np.zeros((B, T), np.int64)
    for b in range(B):
        n = lengths[b]
        X[b, 0], X[b, n - 1] = SOS, EOS
        X[b, 1:n - 1] = rng.choice(ranks, size=n - 2, p=pz)
    Y = np.stack([(rng.random(B) < 0.1).astype(np.float32) for _ in LABELS])
    return X, lengths, Y


_SAMPLER_CHILD = r"""
import json, select, sys, time
idx, period = int(sys.argv[1]), float(sys.argv[2])
fake = len(sys.argv) > 3
try:
    if fake:
        read = lambda: (1965.0, 0, 250.0)
        max_mhz = 1965.0
    else:
        import pynvml as nv
        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(idx)
        max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
        reasons = nv.nvmlDeviceGetCurrentClocksEventReasons if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
            else nv.nvmlDeviceGetCurrentClocksThrottleReasons
        read = lambda: (float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)), int(reasons(h)), nv.nvmlDeviceGetPowerUsage(h) / 1000.0)
        read()
except Exception as e:
    print("fail " + repr(e)[:200], flush=True)
    sys.exit(0)
print("ready %f" % max_mhz, flush=True)
if not sys.stdin.readline().startswith("b"):
    sys.exit(0)
samples = []
while True:
    try:
        samples.append(read())
    except Exception:
        pass
    if select.select([sys.stdin], [], [], period)[0]:
        break
print(json.dumps(samples), flush=True)
"""


class ClockSampler:
    """SM clock / throttle reasons / power sampled through NVML (nvidia-ml-py) during the timed region only (the
    B200_PROFILING.md clocks line), by a HELPER PROCESS that polls every 2 ms between begin() and stop().  Sampling from
    the launch loop itself (round 2, first half) stalled rank 0's host for milliseconds at a time: invisible at N = 1 (the
    stall falls between the per-step event pairs) but at N > 1 the other ranks wait for rank 0 inside their exchange
    kernels, and the max-over-ranks step time jumped from 1.23 to 1.35-3.6 ms in half of the runs.  nvidia-smi needed
    ~0.5 s to deliver its first line, longer than the region.  Fallback: an in-process thread (no launch-loop samples)."""
    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, gpu, period_s=0.002):
        self.samples, self.live, self._stop, self.h, self.nv, self.child = [], False, False, None, None, None
        self.source = "nvml helper process"
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = int(vis.split(",")[gpu]) if vis and all(t.strip().isdigit() for t in vis.split(",")) else gpu
        try:
            import subprocess
            extra = ["fake"] if os.environ.get("DVAE_FAKE_NVML") == "1" else []
            self.child = subprocess.Popen([sys.executable, "-c", _SAMPLER_CHILD, str(idx), str(period_s)] + extra, stdin=subprocess.PIPE,
                                          stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            import select
            line = self.child.stdout.readline() if select.select([self.child.stdout], [], [], 20.0)[0] else ""
            if not line.startswith("ready"):
                raise RuntimeError(line.strip() or "no answer")
            self.max_mhz = float(line.split()[1])
            return
        except Exception:
            if self.child is not None:
                try:
                    self.child.kill()
                except Exception:
                    pass
            self.child = None
        # fallback: background thread in this process
        self.source = "nvml in-process thread"
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.h = None
            return
        self.period = 0.005
        self.t = threading.Thread(target=self._loop, daemon=True)
        self.t.start()

    def _loop(self):
        nv = self.nv
        while not self._stop:
            if self.live:
                try:
                    mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                        else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                    pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                    self.samples.append((float(mhz), int(rs), pw))
                except Exception:
                    pass
            time.sleep(self.period)

    def sample_now(self):
        """Kept for callers' sake: nothing is sampled from the launch loop any more (see the class docstring)."""
        return

    def begin(self):
        self.live = True
        if self.child is not None:
            try:
                self.child.stdin.write("b\n")
                self.child.stdin.flush()
            except Exception:
                self.child = None

    def stop(self):
        self.live = False
        self._stop = True
        if self.child is not None:
            try:
                self.child.stdin.write("e\n")
                self.child.stdin.flush()
                import select
                line = self.child.stdout.readline() if select.select([self.child.stdout], [], [], 10.0)[0] else "[]"
                self.samples = [tuple(x) for x in json.loads(line or "[]")]
                self.child.wait(timeout=5)
            except Exception:
                try:
                    self.child.kill()
                except Exception:
                    pass
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "source": self.source}
        if (self.h is None and self.child is None) or not self.samples:
            return out
        sm = [s[0] for s in self.samples]
        bits = 0
        for s in self.samples:
            bits |= s[1]
        out.update(sm_mhz=float(np.median(sm)), sm_min_mhz=float(min(sm)), sm_max_mhz=self.max_mhz,
                   reasons=[n for n, b in self.REASONS if bits & b], samples=len(sm), power_w_max=max(s[2] for s in self.samples))
        return out


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return {"hbm_gbs": float(p["hbm_gbs"]), "bf16_tflops": float(p["bf16_tflops"]),
                "bf16_tflops_sustained": float(p.get("bf16_tflops_sustained", p["bf16_tflops"])), "src": "measured"}
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "src": "fallback"}


def algorithmic_flops(B, T, cfg=None, V=None):
    """SURVEY.md 8a: GEMM flops (2 * MAC) of one TRAIN step (forward + backward = 3 x forward) over padded positions:
    encoder over B*T, decoder and vocabulary projection over B*(T-1), heads per sequence.  Returns a dict per class."""
    cfg = CFG2 if cfg is None else cfg
    V = VOCAB if V is None else V
    E, H = cfg["embedding_dim"], cfg["hidden_dim"]
    D = 2 if cfg["bidirectional_encoder"] else 1
    Le = cfg["num_rnn_layers"]
    Ld = max(Le, 2)
    Z = cfg["latent_dims"]["total"]
    C = Le * D * H
    enc_proj = D * 8 * H * E + (Le - 1) * D * 8 * H * (D * H)          # input projections, per position
    enc_rec = Le * D * 8 * H * H                                       # recurrent products, per position
    dec_proj = 8 * H * E + (Ld - 1) * 8 * H * H
    dec_rec = Ld * 8 * H * H
    vocab = 2 * H * V
    heads = 2 * C * 2 * Z + 2 * Z * 2 * H * Ld
    n_enc, n_dec = B * T, B * (T - 1)
    fwd = {"lstm_input_projections": enc_proj * n_enc + dec_proj * n_dec, "recurrence": enc_rec * n_enc + dec_rec * n_dec,
           "vocab": vocab * n_dec, "heads": heads * B}
    train = {k: 3.0 * v for k, v in fwd.items()}
    train["total"] = sum(train.values())
    train["dense_gemm_class"] = train["lstm_input_projections"] + train["vocab"]       # the launches that are plain GEMMs
    return train


# ------------------------------------------------------------------------------------------------
# CPU legs (reported baseline only): the reference's own implementation when it is installed under baseline/_ref
# (python -m pip install --target baseline/_ref /root/reference; git-ignored, travels to the GPU box), else the oracle port
# ------------------------------------------------------------------------------------------------
def _load_installed_reference():
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref_dir, "vae")):
        return None
    from oracle.ref_shim import install_stubs       # texar / torchtext import stubs (see oracle/ref_shim.py)
    install_stubs()
    if ref_dir not in sys.path:
        sys.path.insert(0, ref_dir)
    try:
        return importlib.import_module("vae.model"), importlib.import_module("vae.losses")
    except Exception as e:      # noqa: BLE001
        print(f"[bench] installed reference failed to import ({e}); falling back to the oracle port", file=sys.stderr)
        return None


def cpu_reference_steps(n_steps, warmup, B, budget_s=150.0):
    """The UNMODIFIED reference (vae/model.py + vae/losses.py from baseline/_ref) on the host cores, the train-step body of
    run.py:227-262 (forward, compute_all_losses, backward, clip_grad_norm_(5.0), Adam.step, zero_grad) on this workload;
    torch intra-op threads = all host cores; anomaly detection off (run.py:22 turns it on: favourable to the reference)."""
    mods = _load_installed_reference()
    if mods is None:
        return None
    ref_model, ref_losses = mods
    torch.set_num_threads(os.cpu_count())
    torch.manual_seed(10)
    np.random.seed(10)
    vae = ref_model.build_vae(CFG2, VOCAB, None, LABELS, torch.device("cpu"), SOS, EOS)
    vae.train()
    opt = torch.optim.Adam(vae.trainable_parameters(), lr=CFG2["learn_rate"])
    rng = np.random.default_rng(10)
    names = list(LABELS)

    def one(i, Bs):
        X, lengths, Y = synth_batch(rng, Bs, uniform_lengths=UNIFORM_LENGTHS)
        X, lengths = torch.from_numpy(X), torch.from_numpy(lengths)
        Yb = {n: torch.from_numpy(Y[j]).reshape(-1, 1) for j, n in enumerate(names)}
        klw = {k: (ref_losses.get_cyclic_kl_weight(i, TOTAL_STEPS) if v == "cyclic" else v) for k, v in CFG2["lambdas"].items()}
        t0 = time.perf_counter()
        out = vae(X, lengths, teacher_forcing_prob=CFG2["teacher_forcing_prob"])
        L = dict()                                                   # run.py:128-163 compute_all_losses
        L.update(ref_losses.reconstruction_loss(X, out["decoder_logits"], lengths))
        L.update(ref_losses.compute_kl_divergence_losses(vae, out["latent_params"], klw))
        L.update(ref_losses.compute_discriminator_losses(vae, out["dsc_logits"], Yb))
        total = L["reconstruction_loss"] + L["total_weighted_kl"] + L["total_dsc_loss"]
        total.backward()
        torch.nn.utils.clip_grad_norm_(vae.trainable_parameters(), 5.0)
        opt.step()
        opt.zero_grad()
        return time.perf_counter() - t0, int(lengths.sum())

    t_probe, _ = one(0, B)
    Bs, total = B, n_steps + max(warmup - 1, 0)
    if t_probe * total > budget_s:                       # bounded sample: shrink the batch, keep the shape
        Bs = max(8, int(B * budget_s / (t_probe * total)) // 8 * 8)
    for i in range(max(warmup - 1, 0)):
        one(i + 1, Bs)
    ts, toks = 0.0, 0
    for i in range(n_steps):
        dt, nt = one(warmup + i, Bs)
        ts += dt
        toks += nt
    sample = (f"{n_steps} train steps of the {WORKLOAD_NAME} workload at batch {Bs}: the unmodified reference (vae/model.py + vae/losses.py "
              f"installed under baseline/_ref, torch {torch.__version__} CPU, {torch.get_num_threads()} intra-op threads), step body of run.py:227-262")
    return toks / ts, ts / n_steps, sample


def cpu_port_steps(n_steps, warmup, B=128, budget_s=150.0):
    """Times `oracle/dvae_oracle.py` (numpy, float32, BLAS threads = all host cores) on the selected workload:
    forward + losses + backward + clip + Adam.  Returns (tokens/s, s/step, sample description)."""
    from oracle import dvae_oracle as O
    dvae = importlib.import_module("disentanglement-vae_b200")
    dvae.set_seed(10)
    vae = dvae.build_vae(CFG2, VOCAB, None, LABELS, torch.device("cpu"), SOS, EOS)     # weights only; never run
    sd = O.cast_state_dict({k: v.detach().numpy() for k, v in vae.state_dict().items()}, np.float32)
    spec = O.ModelSpec(sd, list(vae.context2params.keys()), SOS, EOS)
    rng = np.random.default_rng(10)
    m = {k: np.zeros_like(v) for k, v in sd.items()}
    v_ = {k: np.zeros_like(v) for k, v in sd.items()}
    names = list(LABELS)
    E, H = CFG2["embedding_dim"], CFG2["hidden_dim"]
    D = 2 if CFG2["bidirectional_encoder"] else 1

    def one(i, Bs):
        X, lengths, Y = synth_batch(rng, Bs, uniform_lengths=UNIFORM_LENGTHS)
        eps = {n: rng.standard_normal((Bs, zs)).astype(np.float32) for n, zs in zip(spec.space_names, spec.space_dims)}
        masks_e = [(rng.random((SEQ_T, Bs, w)) >= 0.5).astype(np.float32) * 2 for w in (E, D * H)]
        masks_d = [(rng.random((SEQ_T - 1, Bs, w)) >= 0.5).astype(np.float32) * 2 for w in (E, H)]
        klw = {k: (O.cyclic_kl_weight(i, TOTAL_STEPS) if v == "cyclic" else v) for k, v in CFG2["lambdas"].items()}
        t0 = time.perf_counter()
        fw = O.model_forward(sd, spec, X, lengths, eps, labels={n: Y[j].reshape(-1, 1) for j, n in enumerate(names)},
                             kl_weights=klw, enc_masks=masks_e, dec_masks=masks_d)
        g = O.model_backward(sd, spec, fw)
        O.clip_and_adam(sd, g, m, v_, i + 1, CFG2["learn_rate"])
        return time.perf_counter() - t0, int(lengths.sum())

    t_probe, _ = one(0, B)
    Bs = B
    total = n_steps + max(warmup - 1, 0)
    if t_probe * total > budget_s:                       # bounded sample: shrink the batch, keep the shape
        Bs = max(8, int(B * budget_s / (t_probe * total)) // 8 * 8)
    for i in range(max(warmup - 1, 0)):
        one(i + 1, Bs)
    ts, toks = 0.0, 0
    for i in range(n_steps):
        dt, nt = one(warmup + i, Bs)
        ts += dt
        toks += nt
    sample = f"{n_steps} train steps of the {WORKLOAD_NAME} workload at batch {Bs} (numpy float32 port of vae/model.py + vae/losses.py + run.py:254-262)"
    return toks / ts, ts / n_steps, sample


def cpu_baseline(n_steps, warmup, B, budget_s):
    """(tokens/s, s/step, sample, kind): the installed reference when present, else the oracle port."""
    r = cpu_reference_steps(n_steps, warmup, B, budget_s)
    if r is not None:
        return r + ("reference",)
    return cpu_port_steps(n_steps, warmup, B, budget_s) + ("port",)


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.workload == "cfg5":
        print(json.dumps({"impl": "reference", "unavailable": "the inference workload has no CPU reference arm (60 full forwards "
                          "of batch 1024 per step do not fit the bench budget); see cpu_baseline of the training workloads"}), flush=True)
        return
    cores = os.cpu_count()
    torch.set_num_threads(cores)          # torchrun exports OMP_NUM_THREADS=1: the CPU arm uses every host core at any N
    tps, sps, sample, kind = cpu_baseline(args.steps, args.warmup, BATCH, 150.0)
    line = {"impl": "reference", "metric": "train_tokens_per_sec", "value": tps, "unit": "tokens/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": sps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.gpus, graph=not args.no_graph),
            "cpu_baseline": {"value": tps, "unit": "tokens/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": tps, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# cfg5: inference
# ------------------------------------------------------------------------------------------------
def run_inference_workload(args):
    """cfg5: consistency-evaluation shape (scripts/evaluation/consistency.py:163-205), batch 1024, R = 30 resamples, model in
    train mode (consistency.py:151).  `value`: the encode-once / resample-R API (inference.ConsistencyEvaluator: one CUDA
    graph per resample, second forward without its unused decode).  `e2e`: the reference's call pattern -- two full module
    forwards per resample with the lengths recounted by torch ops -- with host tensors in and predictions out."""
    import __graft_entry__ as ge
    dvae = ge.build()
    inf = importlib.import_module("disentanglement-vae_b200.inference")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    B, T = BATCH, SEQ_T
    dvae.set_seed(10)
    vae = dvae.build_vae(CFG2, VOCAB, None, LABELS, dev, SOS, EOS)
    vae.train()
    rng = np.random.default_rng(5)
    X, L, _ = synth_batch(rng, B)
    Xh, Lh = torch.from_numpy(X).pin_memory(), torch.from_numpy(L).pin_memory()
    clocks = ClockSampler(0)
    ev_ = inf.ConsistencyEvaluator(vae, B, T, keep_tokens=True)
    warm = max(args.warmup, 3)
    steps = args.steps
    n0 = dvae.launch_count()
    ev_.use_graph = False
    ev_.encode_once(Xh, Lh)
    ev_.resample(1)
    torch.cuda.synchronize()
    launches = dvae.launch_count() - n0
    ev_.use_graph = True
    ev_.resample(warm)
    torch.cuda.synchronize()
    # value: R resamples of a batch whose context is already resident (device-timed with CUDA events)
    ev_.encode_once(Xh, Lh)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    clocks.begin()
    clocks.sample_now()
    a.record()
    out = ev_.resample(steps)
    b.record()
    clocks.sample_now()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b)
    clk = clocks.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {k: v[-1] for k, v in out.items()})          # the last resample
    toks = float(L.sum()) * 2 * steps
    # e2e: host tokens in -> encode once -> R resamples -> predictions of both passes back on the host (wall clock)
    t0 = time.perf_counter()
    ev_.encode_once(Xh, Lh)
    out = ev_.resample(steps)
    preds = {k: v.cpu() for k, v in ev_.predictions(out["dsc_logits"]).items()}
    preds_hat = {k: v.cpu() for k, v in ev_.predictions(out["dsc_logits_hat"]).items()}
    torch.cuda.synchronize()
    api_s = time.perf_counter() - t0

    # reference call pattern through the drop-in module surface (consistency.py:163-205)
    def pair(Xd, Ld):
        with torch.no_grad():
            o = vae(Xd, Ld, teacher_forcing_prob=0.0)
            p1 = {n: vae.discriminators[n].predict(lg).cpu() for n, lg in o["dsc_logits"].items()}
            xh = o["token_predictions"]
            lh = xh.size(1) - ((xh == EOS) | (xh == PAD)).sum(1)
            lh = lh.clamp_(min=1)
            o2 = vae(xh, lh, teacher_forcing_prob=0.0)
            p2 = {n: vae.discriminators[n].predict(lg).cpu() for n, lg in o2["dsc_logits"].items()}
            return p1, p2
    Xd, Ld = Xh.to(dev), Lh.to(dev)
    for _ in range(2):
        pair(Xd, Ld)
    torch.cuda.synchronize()
    n_ref = max(3, min(steps, 10))
    t0 = time.perf_counter()
    Xd, Ld = Xh.to(dev, non_blocking=True), Lh.to(dev, non_blocking=True)
    for _ in range(n_ref):
        pair(Xd, Ld)
    torch.cuda.synchronize()
    ref_s = time.perf_counter() - t0
    line = {"metric": "inference_tokens_per_sec", "value": toks / (ms * 1e-3), "unit": "tokens/s", "n_gpus": 1, "steps": steps,
            "warmup": warm, "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": dict(workload_config(1), tokens="valid input tokens x 2 forwards per resample (the reference's accounting)",
                           api="inference.ConsistencyEvaluator.encode_once + resample(R): host tokens in, predictions of both passes out"),
            "e2e": {"value": toks / api_s, "unit": "tokens/s", "ms_per_step": api_s * 1e3 / steps,
                    "h2d_bytes_per_step": int((Xh.numel() * 8 + Lh.numel() * 8) / steps), "d2h_bytes_per_step": int(2 * len(LABELS) * B * 8),
                    "path": "ConsistencyEvaluator: host tokens -> encode_once -> resample(R) -> predictions of both passes on the host"},
            "e2e_reference_pattern": {"value": float(L.sum()) * 2 * n_ref / ref_s, "unit": "tokens/s", "ms_per_step": ref_s * 1e3 / n_ref,
                                      "path": "the reference's loop body through the drop-in module: vae(x, tf=0) -> torch recount -> vae(x_hat, tf=0), "
                                              "predictions to the host after each forward (consistency.py:163-205)"},
            "gpu_launches": int(launches * steps), "launches_per_step": int(launches), "clocks": clk,
            "check": {"resamples": steps, "mean_pred_agreement": {k: float((preds[k] == preds_hat[k]).float().mean()) for k in preds}}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
DUMP_BYTES = 60 * 10 ** 6       # array data of one --dump-outputs directory: with the .npy headers it stays under 64 MB


def _dump_cap(sizes, budget):
    """The largest per-array size c with sum(min(s, c)) <= budget, or None when every array fits whole."""
    if sum(sizes) <= budget:
        return None
    left, rest = budget, sorted(sizes)
    for i, s in enumerate(rest):
        c = left // (len(rest) - i)
        if s > c:
            return c
        left -= s


def dump_outputs(out_dir, arrays):
    """Writes {name: tensor or array} as out_dir/<name>.npy: floating point as float32, integers as float64 (exact).
    Over DUMP_BYTES in all, the largest arrays are cut to an equal share each, a sorted sample of their flattened elements
    drawn by a generator seeded with the array's name, so the same run always writes the same elements."""
    os.makedirs(out_dir, exist_ok=True)
    host = {}
    for name, t in arrays.items():
        a = t.detach().cpu().numpy() if torch.is_tensor(t) else np.asarray(t)
        host[name] = a.astype(np.float32 if a.dtype.kind == "f" else np.float64)
    cap = _dump_cap([a.nbytes for a in host.values()], DUMP_BYTES)
    for name, a in host.items():
        if cap is not None and a.nbytes > cap:
            idx = np.random.default_rng(zlib.crc32(name.encode())).choice(a.size, cap // a.itemsize, replace=False)
            a = a.reshape(-1)[np.sort(idx)]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def train_step_outputs(vae, eng, out):
    """What a caller of TrainEngine.step_resident holds after a step: the returned loss block, the updated parameters and
    Adam's first moments (an average of the gradients, which the parameter update alone shows only scaled by lr)."""
    m = vae.grad_views(eng.m)
    arrays = {"losses": out}
    arrays.update({f"param.{n}": p for n, p in vae.named_parameters()})
    arrays.update({f"adam_exp_avg.{n}": m[n] for n in vae._layout})
    return arrays


def _events(n):
    return [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]


def _timed(fn, flush, n=10):
    evs = _events(n)
    for a, b in evs:
        flush.zero_()
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    return float(np.median([a.elapsed_time(b) for a, b in evs]))


def dropin_e2e(dvae, vae_cfg, dev, hpool, tokens, steps):
    """The reference's call pattern (run.py:227-262) through the drop-in surface INTEGRATION.md describes: build_vae ->
    forward -> compute_all_losses -> backward -> clip_grad_norm_ -> torch Adam.step -> zero_grad, host tensors in."""
    dvae.set_seed(10)
    vae = dvae.build_vae(vae_cfg, VOCAB, None, LABELS, dev, SOS, EOS)
    vae.train()
    opt = torch.optim.Adam(vae.trainable_parameters(), lr=vae_cfg["learn_rate"])

    def one(i, X, L, Y):
        Xd, Ld = X.to(dev, non_blocking=True), L.to(dev, non_blocking=True)
        klw = {k: (dvae.losses.get_cyclic_kl_weight(i, TOTAL_STEPS) if v == "cyclic" else v) for k, v in vae_cfg["lambdas"].items()}
        out = vae(Xd, Ld, teacher_forcing_prob=vae_cfg["teacher_forcing_prob"])
        total, Ls = dvae.losses.compute_all_losses(vae, out, Xd, {n: y.reshape(-1, 1) for n, y in Y.items()}, Ld, klw)
        total.backward()
        torch.nn.utils.clip_grad_norm_(vae.trainable_parameters(), 5.0)
        opt.step()
        opt.zero_grad()
        return float(total.detach())          # D2H read of the loss, as the reference's loss logger does

    for i in range(3):
        one(i, *hpool[i % len(hpool)])
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    tok = 0
    for i in range(steps):
        j = i % len(hpool)
        one(i + 3, *hpool[j])
        tok += tokens[j]
    torch.cuda.synchronize()
    return tok, time.perf_counter() - t0


def gemm_class_trace(eng, batch, steps=3):
    """Summed device time of the dense GEMM launches (tc16 / tc / SIMT linear kernels) and of the LSTM recurrence kernels
    in `steps` eager train steps, from CUPTI kernel records (torch.profiler) AFTER the timed region: explains the headline,
    is never a bench value."""
    try:
        from torch.profiler import profile, ProfilerActivity
        eng.use_graph = False
        for _ in range(2):
            eng.step_resident(*batch)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(steps):
                eng.step_resident(*batch)
            torch.cuda.synchronize()
        gemm = rec = tot = 0.0
        n_gemm = n_rec = 0
        for e in prof.events():
            if e.device_type != torch.autograd.DeviceType.CUDA:
                continue
            tot += e.device_time
            nm = e.name
            if "gemm_kernel" in nm or "linear_kernel" in nm:
                gemm += e.device_time
                n_gemm += 1
            elif "lstm_" in nm:
                rec += e.device_time
                n_rec += 1
        return {"gemm_us_per_step": gemm / steps, "gemm_launches_per_step": n_gemm / steps, "recurrence_us_per_step": rec / steps,
                "recurrence_launches_per_step": n_rec / steps, "all_kernels_us_per_step": tot / steps}
    except Exception as e:      # noqa: BLE001
        return {"error": str(e)[:200]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 50; cfg5: 30 resamples)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-trace", action="store_true", help="skip the CUPTI GEMM-class / recurrence breakdown after the timed region")
    ap.add_argument("--only-steps", action="store_true", help="warm-up + timed steps only (launch lists under ncu): no e2e / roofline legs")
    ap.add_argument("--batch", type=int, default=None, help="per-GPU batch (default: the workload's)")
    ap.add_argument("--tf", type=float, default=None, help="teacher_forcing_prob (default 1.0 = headline; 0.5 = the shipped configs' value)")
    ap.add_argument("--workload", default="cfg2", choices=["cfg1", "cfg2", "cfg3", "cfg4", "cfg5"],
                    help="cfg2 = headline (BASELINE.json configs[1]); the others are secondary configs, recorded under profiles/")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32 / float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 30 if args.workload == "cfg5" else 50
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    uniform_lengths = select_workload(args.workload)
    global BATCH, CFG2
    if args.batch is not None:
        BATCH = args.batch
    if args.tf is not None:
        CFG2 = dict(CFG2, teacher_forcing_prob=args.tf)
    if args.impl == "reference":
        return run_reference_arm(args)
    if args.workload == "cfg5":
        return run_inference_workload(args)

    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL prints its version banner on stdout at first use: keep stdout clean for the ONE JSON line
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    import __graft_entry__ as ge
    dvae = ge.build()
    engine_mod = importlib.import_module("disentanglement-vae_b200.engine")

    B, T = BATCH, SEQ_T
    clocks = ClockSampler(local) if rank == 0 else None          # sampling thread up before warm-up; samples only in the timed region
    dvae.set_seed(10)                                     # same initial weights on every rank
    vae = dvae.build_vae(CFG2, VOCAB, None, LABELS, dev, SOS, EOS)
    vae.train()
    eng = engine_mod.TrainEngine(vae, CFG2, B, T, total_steps=TOTAL_STEPS, use_graph=not args.no_graph, seed=10 + rank)
    rng = np.random.default_rng(1000 + rank)             # each rank draws its own shard of the global batch
    pool = [synth_batch(rng, B, uniform_lengths=uniform_lengths) for _ in range(8)]
    dpool = [(torch.from_numpy(X).to(dev), torch.from_numpy(L).to(dev), torch.from_numpy(Y).to(dev)) for X, L, Y in pool]
    hpool = [(torch.from_numpy(X), torch.from_numpy(L), {n: torch.from_numpy(Y[j]) for j, n in enumerate(LABELS)}) for X, L, Y in pool]
    tokens = [int(L.sum()) for _, L, _ in pool]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)     # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up (includes graph capture) ----
    n0 = dvae.launch_count()
    eng.use_graph = False
    eng.step_resident(*dpool[0])                         # one eager step: counts this library's launches per step
    torch.cuda.synchronize()
    launches_per_step = dvae.launch_count() - n0
    eng.use_graph = not args.no_graph
    for i in range(max(args.warmup, 3)):
        out = eng.step_resident(*dpool[i % len(dpool)])
    barrier()
    loss_warm = eng.losses_from(out.cpu())["total_loss"]

    # ---- timed region: K steps, device-timed per step, L2 flushed between steps ----
    ev = _events(args.steps)
    barrier()
    if clocks:
        clocks.begin()
    tok_sum = 0
    for i in range(args.steps):
        flush.zero_()
        j = (i + 1) % len(dpool)
        ev[i][0].record()
        out = eng.step_resident(*dpool[j])
        ev[i][1].record()
        tok_sum += tokens[j]
        if clocks and i % 4 == 3:
            clocks.sample_now()                          # GPU is under load here: the host runs ahead of the queued steps
    barrier()
    clk = clocks.stop() if clocks else None
    per_step = [a.elapsed_time(b) for a, b in ev]
    dev_ms = sum(per_step)
    srt = sorted(per_step)
    step_ms = {"min": srt[0], "median": srt[len(srt) // 2], "p90": srt[min(len(srt) - 1, int(0.9 * len(srt)))], "max": srt[-1],
               "note": "per-step CUDA-event times of this rank's timed region (ms_per_step is their mean, max over ranks)"}
    loss_last = eng.losses_from(out.cpu())["total_loss"]
    if args.dump_outputs and rank == 0:          # before the legs below train the same engine further
        dump_outputs(args.dump_outputs, train_step_outputs(vae, eng, out))

    if args.only_steps:
        if world > 1:
            st_ = torch.tensor([dev_ms, float(tok_sum)], dtype=torch.float64, device=dev)
            mx_ = st_.clone(); dist.all_reduce(mx_, op=dist.ReduceOp.MAX)
            dist.all_reduce(st_, op=dist.ReduceOp.SUM)
            dev_ms, tok_sum = float(mx_[0]), float(st_[1])
        if rank == 0:
            print(json.dumps({"metric": "train_tokens_per_sec", "value": tok_sum / (dev_ms * 1e-3), "unit": "tokens/s", "n_gpus": world,
                              "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": dev_ms / args.steps,
                              "config": workload_config(world, graph=not args.no_graph), "dp_exchange": eng.exchange_mode,
                              "step_ms": step_ms, "note": "--only-steps: no e2e / roofline legs"}), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- data parallel: every rank must hold bit-identical parameters after the all-reduced steps ----
    replicas_identical = None
    if world > 1:
        ref = eng.flat.detach().clone()
        dist.broadcast(ref, 0)
        same = torch.tensor([1.0 if torch.equal(ref, eng.flat) else 0.0], device=dev)
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        replicas_identical = bool(same.item() == 1.0)
        assert replicas_identical, "data-parallel replicas diverged: parameters differ across ranks after the timed steps"

    # ---- end-to-end leg: host buffers in, losses out, through the public engine API ----
    # (TrainEngine.train_steps: every step stages its HOST batch into pinned memory, ONE H2D copy, the captured step, ONE D2H
    #  read of the loss block; batch k + 1 is staged while the GPU runs step k, losses are consumed two steps behind)
    barrier()
    t0 = time.perf_counter()
    e2e_tok = sum(tokens[i % len(hpool)] for i in range(args.steps))
    e2e_losses = [L["total_loss"] for L in eng.train_steps(hpool[i % len(hpool)] for i in range(args.steps))]
    barrier()
    e2e_s = time.perf_counter() - t0
    assert len(e2e_losses) == args.steps and all(np.isfinite(e2e_losses))
    # the same, one synchronous call per step (step_host: stage, upload, step, read back, wait)
    t0 = time.perf_counter()
    for i in range(args.steps):
        eng.step_host(*hpool[i % len(hpool)])
    barrier()
    e2e_sync_s = time.perf_counter() - t0

    # ---- end-to-end through the DROP-IN plugin call pattern (INTEGRATION.md's two-import swap), rank 0 of a 1-GPU run ----
    dropin = None
    if world == 1 and args.workload != "cfg4":
        d_steps = min(args.steps, 20)
        d_tok, d_s = dropin_e2e(dvae, CFG2, dev, hpool, tokens, d_steps)
        dropin = {"value": d_tok / d_s, "unit": "tokens/s", "ms_per_step": d_s * 1e3 / d_steps, "steps": d_steps,
                  "path": "build_vae -> forward -> compute_all_losses -> backward -> clip_grad_norm_ -> torch.optim.Adam.step "
                          "(run.py:227-262 through the drop-in module surface; autograd + ctypes per op, no CUDA graph)"}

    # ---- per-kernel rooflines, each timed alone with CUDA events (L2 flushed) ----
    pl, P = eng.plan, vae._P
    d = pl.d
    N = pl.N
    _L = importlib.import_module("disentanglement-vae_b200._lib")
    planes_cm = eng.weight_planes()        # same GEMM operand staging as inside the engine's step
    planes_cm.__enter__()
    pl.vocab_ce(P, pl.d_hs[-1], eng.inputs, eng.lengths)            # leaves the fp16 operand planes in the workspace
    call_ms = _timed(lambda: pl.vocab_ce(P, pl.d_hs[-1], eng.inputs, eng.lengths), flush)      # split + kernel + finalize + loss
    k_ms = _timed(lambda: _L.check(pl.lib.dvae_vocab_ce_partials(
        _L.ptr(pl.d_hs[-1]), d.Hd, pl.T1, pl.B, d.Hd, d.V, _L.ptr(P["decoder.linear.weight"]), _L.ptr(P["decoder.linear.bias"]),
        _L.ptr(eng.inputs), eng.inputs.stride(0), _L.ptr(eng.lengths), d.sos, _L.ptr(pl.ce_ws), _L.stream_ptr()), "dvae_vocab_ce_partials"), flush)
    pl._alloc_bwd()
    ce_bwd_ms = _timed(lambda: pl.vocab_ce_bwd(P, eng.G, pl.d_hs[-1], eng.inputs, eng.lengths, None), flush)
    adam_ms = _timed(lambda: eng._optim(), flush)
    heads_ms = _timed(lambda: pl.heads(P, pl.ctx, pl.eps, eng.labels, eng.kl_w), flush)
    enc_ms = _timed(lambda: pl.encode(P, eng.inputs, eng.lengths, True), flush)

    def rec_only(enc):       # one recurrence launch alone (gates already projected): the sequential latency chain
        lib = pl.lib
        if enc:
            w_ih, w_hh, b_ih, b_hh = pl._enc_w(P, 0, d.D)
            return lambda: _L.check(lib.dvae_lstm_seq_fwd_ex(
                _L.ptr(pl.x_enc), d.E, T, B, d.E, d.H, d.D, _L.ptr_array(w_ih), _L.ptr_array(w_hh), _L.ptr_array(b_ih),
                _L.ptr_array(b_hh), None, None, 0, 0, _L.ptr(eng.lengths), _L.ptr(pl.e_hs[0]), d.D * d.H, pl.ctx.data_ptr(),
                pl.ctx_c.data_ptr(), d.C, d.H, _L.ptr(pl.e_gates[0]), _L.ptr(pl.e_cs[0]), _L.ptr(pl.state_ws), 1, _L.stream_ptr()), "rec")
        w_ih, w_hh, b_ih, b_hh = pl._dec_w(P, 0)
        return lambda: _L.check(lib.dvae_lstm_seq_fwd_ex(
            _L.ptr(pl.x_dec), d.E, pl.T1, B, d.E, d.Hd, 1, _L.ptr_array(w_ih), _L.ptr_array(w_hh), _L.ptr_array(b_ih),
            _L.ptr_array(b_hh), pl.hid.data_ptr(), pl.hid.data_ptr() + 4 * d.Ld * d.Hd, d.H2L, 0, None, _L.ptr(pl.d_hs[0]), d.Hd,
            None, None, 0, 0, _L.ptr(pl.d_gates[0]), _L.ptr(pl.d_cs[0]), _L.ptr(pl.state_ws), 1, _L.stream_ptr()), "rec")
    rec_enc_ms = _timed(rec_only(True), flush) if not d.bow else None
    rec_dec_ms = _timed(rec_only(False), flush)
    planes_cm.__exit__(None, None, None)

    trace = None
    if rank == 0 and world == 1 and not args.no_trace:
        trace = gemm_class_trace(eng, dpool[0])

    stats = torch.tensor([dev_ms, e2e_s, float(tok_sum), float(e2e_tok), e2e_sync_s], dtype=torch.float64, device=dev)
    if world > 1:
        mx = stats.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = stats.clone()
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        dev_ms, e2e_s, e2e_sync_s = float(mx[0]), float(mx[1]), float(mx[4])
        tok_sum, e2e_tok = float(sm[2]), float(sm[3])
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = load_peaks()
    ms_per_step = dev_ms / args.steps
    alg = algorithmic_flops(B, T)
    flops = 2.0 * N * d.Hd * d.V
    tf = flops / (k_ms * 1e-3) / 1e12
    alg_bytes = 4.0 * (N * d.Hd + d.V * d.Hd + d.V + 2 * N)
    traffic, traffic_src = None, None
    for fname in ("r2_ncu_traffic.json", "r1_ncu_traffic.json"):
        try:                   # dram__bytes_read + write of this kernel from the committed `ncu --set full` capture
            with open(os.path.join(ROOT, "profiles", fname)) as f:
                t = json.load(f)["vocab_ce_fwd"]
            if args.workload in ("cfg2", "cfg3"):
                traffic, traffic_src = t["dram_bytes_read"] + t["dram_bytes_write"], f"profiles/{fname} (ncu --set full, per launch, cfg2 shape)"
            break
        except Exception:
            continue
    gemm_impl = os.environ.get("DVAE_GEMM_IMPL", "")
    kname = ("tc_gemm_kernel mode 1 (TMA + tcgen05.mma.kind::tf32, 3xTF32)" if gemm_impl.startswith("t")
             else "tc16_gemm_kernel mode 1 (pre-split fp16 hi/lo operand planes by bulk copy, A rows stationary in tensor memory, tcgen05.mma.kind::f16, one TMEM accumulator, 16 epilogue warps)")
    n_par = eng.n
    Zt = d.Z
    heads_bytes = 4.0 * (B * d.C + d.C * 2 * Zt + 2 * Zt + B * Zt + 3 * B * Zt + Zt * d.H2L + B * d.H2L)      # SURVEY 8d, K2
    Dn = d.D
    enc_flops = float(B * T) * (Dn * 8 * d.H * (d.E + d.H) + Dn * 8 * d.H * (Dn * d.H + d.H))                 # SURVEY 8a, per position
    adam_bytes = 36.0 * n_par                   # sumsq reads g; clip+Adam reads p, g, m, v and writes p, m, v and the zeroed g
    step_tf = alg["total"] / (ms_per_step * 1e-3) / 1e12
    secondary = [
        {"kernel": "WHOLE TRAIN STEP (every launch of the captured graph): algorithmic GEMM flops of SURVEY.md 8a (forward + backward "
                   "= 3 x forward, padded positions) / device ms_per_step",
         "bound": "tensor", "achieved": step_tf, "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
         "frac": step_tf / peaks["bf16_tflops_sustained"], "algorithmic_flops": alg["total"], "launch_ms": ms_per_step,
         "peak_source": "MEASURED_PEAKS.json bf16 sustained; fp32-grade emulation executes 3 tensor flops per algorithmic flop (ceiling 1/3), "
                        "and the step is a dependency chain of ~100 launches with 8 strictly sequential recurrences",
         "flops_by_class": {k: v for k, v in alg.items() if k != "total"}},
        {"kernel": "vocabulary backward = softmax-gradient recompute + d_h + d_w + d_bias (dvae_vocab_ce_bwd, all launches of the call)",
         "bound": "tensor", "achieved": 2 * flops / (ce_bwd_ms * 1e-3) / 1e12, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
         "frac": 2 * flops / (ce_bwd_ms * 1e-3) / 1e12 / peaks["bf16_tflops"], "launch_ms": ce_bwd_ms, "algorithmic_flops": 2 * flops,
         "note": "algorithmic 4*N*H*V (the recomputed logits, another 2*N*H*V, are not counted)"},
        {"kernel": "sumsq_kernel + clip_adam_kernel (grad-norm clip 5.0 + Adam + zero_grad over the flat parameter buffer)",
         "bound": "hbm", "achieved": adam_bytes / (adam_ms * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
         "frac": adam_bytes / (adam_ms * 1e-3) / 1e9 / peaks["hbm_gbs"], "launch_ms": adam_ms, "algorithmic_bytes": adam_bytes},
        {"kernel": "heads_fwd_kernel (context2params, reparameterisation, KL, discriminators + losses, z2hidden: ONE launch)",
         "bound": "hbm", "achieved": heads_bytes / (heads_ms * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
         "frac": heads_bytes / (heads_ms * 1e-3) / 1e9 / peaks["hbm_gbs"], "launch_ms": heads_ms, "algorithmic_bytes": heads_bytes,
         "note": "launch/latency bound as SURVEY 8d predicts"},
        {"kernel": "encoder forward = embedding + dropout + layers x (input-projection GEMMs + 1 persistent recurrence kernel)",
         "bound": "latency", "achieved": enc_flops / (enc_ms * 1e-3) / 1e12, "peak": peaks["bf16_tflops"],
         "unit": "TFLOP/s", "frac": enc_flops / (enc_ms * 1e-3) / 1e12 / peaks["bf16_tflops"], "launch_ms": enc_ms,
         "algorithmic_flops": enc_flops, "sequential_steps": 2 * T, "us_per_sequential_step": enc_ms * 1e3 / (2 * T)},
        {"kernel": "LSTM recurrence launches alone (gates already projected): encoder layer 0 (all directions in one launch) and decoder layer 0",
         "bound": "latency", "unit": "us per sequential step",
         "encoder_l0": None if rec_enc_ms is None else {"launch_ms": rec_enc_ms, "steps": T, "us_per_step": rec_enc_ms * 1e3 / T},
         "decoder_l0": {"launch_ms": rec_dec_ms, "steps": T - 1, "us_per_step": rec_dec_ms * 1e3 / (T - 1)},
         "achieved": rec_dec_ms * 1e3 / (T - 1), "peak": None, "frac": None}]
    if trace and "gemm_us_per_step" in trace:
        g_tf = alg["dense_gemm_class"] / (trace["gemm_us_per_step"] * 1e-6) / 1e12
        secondary.insert(1, {"kernel": "GEMM CLASS aggregate: every tc16 / 3xTF32 / SIMT GEMM launch of one step (input projections, dx / dW "
                                       "GEMMs, vocabulary forward + backward): algorithmic flops / SUMMED kernel time (they overlap on side streams)",
                             "bound": "tensor", "achieved": g_tf, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s", "frac": g_tf / peaks["bf16_tflops"],
                             "algorithmic_flops": alg["dense_gemm_class"], "summed_kernel_us": trace["gemm_us_per_step"],
                             "launches": trace["gemm_launches_per_step"], "source": "CUPTI kernel records of 3 eager steps after the timed region",
                             "recurrence_kernels_summed_us": trace["recurrence_us_per_step"], "all_kernels_summed_us": trace["all_kernels_us_per_step"]})
    roof = {"kernel": kname + " = vocab-CE forward: vocabulary projection + online log-softmax / arg-max / NLL epilogue from TMEM; "
                              "the [N,V] logits are never written to HBM; ONE launch between the CUDA events (dvae_vocab_ce_partials)",
            "bound": "tensor", "achieved": tf, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s", "frac": tf / peaks["bf16_tflops"],
            "peak_source": f"MEASURED_PEAKS.json bf16 burst ({peaks['src']}); fp32-grade emulation executes 3 tensor flops per algorithmic flop",
            "traffic": traffic, "traffic_source": traffic_src,
            "launch_ms": k_ms, "call_ms": call_ms, "call": "dvae_vocab_ce_fwd = operand split x2 + this kernel + finalize + loss",
            "tensor_flops_executed": 3 * flops, "algorithmic_flops": flops, "algorithmic_bytes": alg_bytes,
            "hbm_frac": alg_bytes / (k_ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
            "share_of_step": k_ms / ms_per_step, "step_frac": step_tf / peaks["bf16_tflops_sustained"],
            "secondary": secondary}
    line = {"metric": "train_tokens_per_sec", "value": tok_sum / (dev_ms * 1e-3), "unit": "tokens/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(world, graph=not args.no_graph),
            "dp_exchange": eng.exchange_mode,      # none | p2p | nvls (repo all-reduce kernel inside the one-graph step) | nccl+...
            "step_ms": step_ms,
            "padded_tokens_per_sec": B * world * T * args.steps / (dev_ms * 1e-3),
            "e2e": {"value": e2e_tok / e2e_s, "unit": "tokens/s", "h2d_bytes_per_step": eng.h2d_bytes_per_step,
                    "d2h_bytes_per_step": eng.d2h_bytes_per_step, "ms_per_step": e2e_s * 1e3 / args.steps,
                    "path": "TrainEngine.train_steps(host batches): per step host tensors -> pinned block -> one H2D -> captured step -> "
                            "one D2H of the loss block; pipelined (losses consumed two steps behind)",
                    "ms_per_step_synchronous": e2e_sync_s * 1e3 / args.steps,
                    "synchronous_path": "TrainEngine.step_host per batch (waits for every step's losses)"},
            "e2e_dropin": dropin,
            "gpu_launches": int(launches_per_step * args.steps), "launches_per_step": int(launches_per_step),
            "roofline": roof, "clocks": clk, "loss_after_warmup": loss_warm, "loss_last": loss_last,
            "teacher_forcing_prob": CFG2["teacher_forcing_prob"]}
    if replicas_identical is not None:
        line["replicas_identical"] = replicas_identical
    if not args.no_cpu_baseline and world == 1 and args.workload in ("cfg1", "cfg2", "cfg3"):
        tps, sps, sample, kind = cpu_baseline(3, 1, B, 25.0)
        line["cpu_baseline"] = {"value": tps, "unit": "tokens/s", "cores": os.cpu_count(), "kind": kind, "sample": sample,
                                "s_per_step": sps}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
