// Fused vocabulary projection + online log-softmax + masked NLL (see include/dvae_b200.h).
//
// Forward: each CTA owns a 128-row tile of decoder outputs and a slice of the vocabulary; it walks
// its slice in 128-column tiles (fp32 SIMT tile GEMM, K = H), folds every logits tile into running
// (max, sum-exp, argmax, target-logit) registers and never writes logits.  A single-CTA finalise
// kernel merges the vocabulary slices in a fixed order -> lse, nll, argmax and the masked, batch-
// averaged loss (deterministic).
// Backward (this round): softmax tiles are recomputed from h, W and the saved lse into an
// L2-sized chunk buffer P[N, Vc] and consumed by two dense GEMMs per chunk (dh += P W, dW = P^T h).
#include <math.h>

#include "gemm_simt.cuh"
#include "tc_gemm16.cuh"
#include "tc_planes.cuh"

namespace dvae {

int linear_impl(const float* A, int64_t lda, int trans_a, const float* B, int64_t ldb, int trans_b, float* C,
                int64_t ldc, int M, int N, int K, const float* bias, const float* bias2, float beta, int act,
                cudaStream_t st);
int colsum_impl(const float* X, int64_t ldx, int M, int N, float* out, float beta, cudaStream_t st);

using GCE = GemmTile<128, 128, 16, 8, 8, true, true>;

struct CeArgs;
static bool use_tc16(int N, int V, int H, const float* h, int64_t ldh, const float* w) {
  return !force_simt_gemm() && N >= 64 && V >= 128 && H >= 32 && tc16::supported(h, ldh, 0, w, H, 0, N, V, H);
}
// pre-split operand planes pay off when both operands are re-read by many tiles and K is a whole number of k-blocks
static bool use_presplit(int N, int V, int H) { return tc16::presplit_enabled() && H % 32 == 0 && N >= 256 && V >= 1024; }

struct CeArgs {
  const float* h; int64_t ldh;
  const float* w; const float* bias;
  const int64_t* targets; int64_t tgt_stride_b;
  const int64_t* lengths;
  int N, B, H, V, sos;
  int tiles_per_split, nsplit;
  float* part;      // [nsplit][R][4]: max, sumexp, target logit, argmax value; R = N, or (live rows) rt * 128 for rt live
                    // row tiles, inside a capacity of N rounded up to whole row tiles (part_rows)
  int* part_idx;    // [nsplit][R]
  const uint64_t* gumbel_seed; uint32_t gumbel_salt;   // sampling: arg-max over logits + Gumbel noise
  const void* h_planes; const void* w_planes;          // optional pre-split fp16 operand planes (tc16::split_planes)
  const int* skip_flag;                                // optional device flag: non-zero = no-op (see tc16::Params::skip_flag)
  // live rows (dvae_vocab_ce_fwd_live): the partials cover the *m_live rows of the row list `rows` only, in the layout
  // tc16_gemm_kernel chose on the device for `live_ctas` launched CTAs (tc16::live_split)
  const int* m_live; const int* rows; int live_ctas;
};

__device__ __forceinline__ void merge_ms(float& m, float& s, float m2, float s2) {
  float M = fmaxf(m, m2);
  if (M == -INFINITY) { s = 0.f; m = M; return; }
  s = s * expf(m - M) + s2 * expf(m2 - M);
  m = M;
}

__global__ void __launch_bounds__(GCE::NT) vocab_ce_fwd_kernel(CeArgs p) {
  __shared__ __align__(16) float smem[GCE::SMEM_FLOATS];
  if (p.skip_flag && *p.skip_flag) return;
  const int m0 = blockIdx.x * GCE::BM, split = blockIdx.y;
  const int ty = threadIdx.x / GCE::TX, tx = threadIdx.x % GCE::TX;
  const int vtiles = (p.V + GCE::BN - 1) / GCE::BN;
  const int vt0 = split * p.tiles_per_split, vt1 = min(vtiles, vt0 + p.tiles_per_split);
  float rm[GCE::TM], rs[GCE::TM], rt[GCE::TM], rav[GCE::TM];
  int rai[GCE::TM], tgt[GCE::TM];
#pragma unroll
  for (int i = 0; i < GCE::TM; ++i) {
    rm[i] = -INFINITY; rs[i] = 0.f; rt[i] = 0.f; rav[i] = -INFINITY; rai[i] = 0x7fffffff;
    int n = m0 + GCE::row_of(ty, i);
    tgt[i] = -1;
    if (n < p.N && p.targets) tgt[i] = (int)p.targets[(int64_t)(n % p.B) * p.tgt_stride_b + (n / p.B) + 1];
  }
  for (int vt = vt0; vt < vt1; ++vt) {
    const int n0 = vt * GCE::BN;
    float acc[GCE::TM][GCE::TN];
#pragma unroll
    for (int i = 0; i < GCE::TM; ++i)
#pragma unroll
      for (int j = 0; j < GCE::TN; ++j) acc[i][j] = 0.f;
    GCE::run(p.h, p.ldh, m0, p.N, p.w, p.H, n0, p.V, 0, p.H, p.H, smem, acc);
    float bj[GCE::TN];
    int cj[GCE::TN];
#pragma unroll
    for (int j = 0; j < GCE::TN; ++j) {
      cj[j] = n0 + GCE::col_of(tx, j);
      bj[j] = cj[j] < p.V ? p.bias[cj[j]] : 0.f;
    }
#pragma unroll
    for (int i = 0; i < GCE::TM; ++i) {
      float tmax = -INFINITY;
      float gn[GCE::TN];
#pragma unroll
      for (int j = 0; j < GCE::TN; ++j) gn[j] = 0.f;
      if (p.gumbel_seed) {
        const uint64_t gseed = *p.gumbel_seed;
        const int n = m0 + GCE::row_of(ty, i);
#pragma unroll
        for (int j4 = 0; j4 < GCE::TN; j4 += 4) {
          float g[4];
          gumbel4(gseed, p.gumbel_salt, n, cj[j4], (p.V + 3) >> 2, g);
          gn[j4] = g[0]; gn[j4 + 1] = g[1]; gn[j4 + 2] = g[2]; gn[j4 + 3] = g[3];
        }
      }
#pragma unroll
      for (int j = 0; j < GCE::TN; ++j) {
        float v = cj[j] < p.V ? acc[i][j] + bj[j] : -INFINITY;
        acc[i][j] = v;
        tmax = fmaxf(tmax, v);
        const float vs = v + gn[j];
        if (vs > rav[i] || (vs == rav[i] && cj[j] < rai[i])) { rav[i] = vs; rai[i] = cj[j]; }
        if (cj[j] == tgt[i]) rt[i] = v;
      }
      if (tmax > rm[i]) { rs[i] *= expf(rm[i] - tmax); rm[i] = tmax; }
      if (rm[i] != -INFINITY) {
#pragma unroll
        for (int j = 0; j < GCE::TN; ++j) rs[i] += expf(acc[i][j] - rm[i]);
      }
    }
  }
  // combine the 16 threads (tx) that share each row: lanes [16*(ty&1), +16) of the warp
#pragma unroll
  for (int i = 0; i < GCE::TM; ++i) {
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) {
      float m2 = __shfl_xor_sync(0xffffffffu, rm[i], o), s2 = __shfl_xor_sync(0xffffffffu, rs[i], o);
      float t2 = __shfl_xor_sync(0xffffffffu, rt[i], o), av2 = __shfl_xor_sync(0xffffffffu, rav[i], o);
      int ai2 = __shfl_xor_sync(0xffffffffu, rai[i], o);
      merge_ms(rm[i], rs[i], m2, s2);
      rt[i] += t2;
      if (av2 > rav[i] || (av2 == rav[i] && ai2 < rai[i])) { rav[i] = av2; rai[i] = ai2; }
    }
    int n = m0 + GCE::row_of(ty, i);
    if (tx == 0 && n < p.N) {
      float4 o4 = make_float4(rm[i], rs[i], rt[i], rav[i]);
      *reinterpret_cast<float4*>(p.part + ((int64_t)split * p.N + n) * 4) = o4;
      p.part_idx[(int64_t)split * p.N + n] = rai[i];
    }
  }
}

// Merge the vocabulary splits of each row (fixed order: deterministic), write lse / nll / arg-max, and leave one
// partial NLL sum per CTA in `block_sums`; vocab_ce_loss_kernel adds them up (fixed order again) into the loss.
// Eight lanes share a row: lane `sub` folds splits sub, sub + 8, ... and three shuffle steps fold the lanes (fixed order).
// (One thread per row walked up to 56 dependent split loads; the kernel took 35 us for 3 MB of partials.)
constexpr int kFinThreads = 128, kFinMaxBlocks = 96, kFinLanes = 8;
__global__ void __launch_bounds__(kFinThreads) vocab_ce_finalize_kernel(CeArgs p, float* lse, float* nll, int32_t* argmax,
                                                                       float* block_sums) {
  __shared__ float red[kFinThreads / 32];
  const int sub = threadIdx.x % kFinLanes, slot = threadIdx.x / kFinLanes;
  constexpr int kRows = kFinThreads / kFinLanes;
  // rows of the partials: every decoder position, or (live rows) the *m_live entries of the row list, in the split count and
  // row stride the partials kernel derived from the same count
  int rows = p.N, nsplit = p.nsplit;
  int64_t stride = p.N;
  if (p.m_live) {
    rows = *p.m_live;
    const int rt = (rows + GCE::BM - 1) / GCE::BM;
    int tpc, groups;
    tc16::live_split(rt, p.live_ctas, (p.V + GCE::BN - 1) / GCE::BN, &tpc, &groups);
    nsplit = 4 * groups;      // pre-split operands: four epilogue warp sets per CTA, each a split of its own
    stride = (int64_t)rt * GCE::BM;
  }
  float local = 0.f;
  for (int k0 = blockIdx.x * kRows; k0 < rows; k0 += gridDim.x * kRows) {      // block-uniform trip count (shuffles below)
    const int k = k0 + slot;
    float m = -INFINITY, s = 0.f, t = 0.f, av = -INFINITY;
    int ai = 0x7fffffff;
    if (k < rows) {
      for (int sp = sub; sp < nsplit; sp += kFinLanes) {
        float4 q = *reinterpret_cast<const float4*>(p.part + ((int64_t)sp * stride + k) * 4);
        int qi = p.part_idx[(int64_t)sp * stride + k];
        merge_ms(m, s, q.x, q.y);
        t += q.z;
        if (q.w > av || (q.w == av && qi < ai)) { av = q.w; ai = qi; }
      }
    }
#pragma unroll
    for (int o = 1; o < kFinLanes; o <<= 1) {
      const float m2 = __shfl_xor_sync(0xffffffffu, m, o), s2 = __shfl_xor_sync(0xffffffffu, s, o);
      const float t2 = __shfl_xor_sync(0xffffffffu, t, o), av2 = __shfl_xor_sync(0xffffffffu, av, o);
      const int ai2 = __shfl_xor_sync(0xffffffffu, ai, o);
      merge_ms(m, s, m2, s2);
      t += t2;
      if (av2 > av || (av2 == av && ai2 < ai)) { av = av2; ai = ai2; }
    }
    if (sub == 0 && k < rows) {
      const int n = p.rows ? p.rows[k] : k;      // decoder position
      float l = m + logf(s), e = l - t;
      if (lse) lse[n] = l;
      if (nll) nll[n] = e;
      if (argmax) argmax[n] = ai;
      int b = n % p.B, tpos = n / p.B + 1;
      if (tpos < p.lengths[b]) local += e;
    }
  }
  local = warp_sum(local);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = local;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tot = 0.f;
    for (int i = 0; i < kFinThreads / 32; ++i) tot += red[i];
    block_sums[blockIdx.x] = tot;
  }
}

__global__ void __launch_bounds__(128) vocab_ce_loss_kernel(CeArgs p, const float* block_sums, int nblocks, float* loss) {
  __shared__ float red[4];
  float local = 0.f;
  // position 0: one-hot(1.0) pseudo-logits at <SOS> (model.py:454): lse = 1 + log(1 + (V-1)/e)
  for (int b = threadIdx.x; b < p.B; b += blockDim.x) {
    if (p.lengths[b] > 0) {
      float l0 = (float)(1.0 + log(1.0 + (double)(p.V - 1) * exp(-1.0)));
      local += l0 - (p.targets[(int64_t)b * p.tgt_stride_b] == p.sos ? 1.f : 0.f);
    }
  }
  local = warp_sum(local);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = local;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tot = red[0] + red[1] + red[2] + red[3];
    for (int i = 0; i < nblocks; ++i) tot += block_sums[i];
    loss[0] = tot / (float)p.B;
  }
}

// sampled token per row = arg-max over the vocabulary splits of (logit + Gumbel noise)
__global__ void vocab_sample_finalize_kernel(CeArgs p, int64_t* tokens, int64_t tok_stride) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= p.N || (p.skip_flag && *p.skip_flag)) return;      // forced step: the pre-filled token stays
  float av = -INFINITY;
  int ai = 0x7fffffff;
  for (int sp = 0; sp < p.nsplit; ++sp) {
    const float q = p.part[((int64_t)sp * p.N + n) * 4 + 3];
    const int qi = p.part_idx[(int64_t)sp * p.N + n];
    if (q > av || (q == av && qi < ai)) { av = q; ai = qi; }
  }
  tokens[(int64_t)n * tok_stride] = ai;
}

// P[n][v - v0] = (softmax(logits[n])[v] - [v == target_n]) * mask_n * scale / B for v in [v0, v0+vc)
struct PArgs {
  const float* h; int64_t ldh;
  const float* w; const float* bias;
  const int64_t* targets; int64_t tgt_stride_b;
  const int64_t* lengths;
  const float* lse;
  const float* grad_scale;
  int N, B, H, V, v0, vc;
  float* P; int64_t ldp;
};

__global__ void __launch_bounds__(GCE::NT) vocab_p_kernel(PArgs p) {
  __shared__ __align__(16) float smem[GCE::SMEM_FLOATS];
  const int m0 = blockIdx.y * GCE::BM, n0 = p.v0 + blockIdx.x * GCE::BN;
  const int ty = threadIdx.x / GCE::TX, tx = threadIdx.x % GCE::TX;
  float acc[GCE::TM][GCE::TN];
#pragma unroll
  for (int i = 0; i < GCE::TM; ++i)
#pragma unroll
    for (int j = 0; j < GCE::TN; ++j) acc[i][j] = 0.f;
  GCE::run(p.h, p.ldh, m0, p.N, p.w, p.H, n0, min(p.V, p.v0 + p.vc), 0, p.H, p.H, smem, acc);
  const float gs = (p.grad_scale ? p.grad_scale[0] : 1.f) / (float)p.B;
#pragma unroll
  for (int i = 0; i < GCE::TM; ++i) {
    int n = m0 + GCE::row_of(ty, i);
    if (n >= p.N) continue;
    int b = n % p.B, tpos = n / p.B + 1;
    float scale = (tpos < p.lengths[b]) ? gs : 0.f;
    int tgt = (int)p.targets[(int64_t)b * p.tgt_stride_b + tpos];
    float l = p.lse[n];
#pragma unroll
    for (int j = 0; j < GCE::TN; ++j) {
      int v = n0 + GCE::col_of(tx, j);
      if (v >= p.V || v >= p.v0 + p.vc) continue;
      float pr = scale == 0.f ? 0.f : (expf(acc[i][j] + p.bias[v] - l) - (v == tgt ? 1.f : 0.f)) * scale;
      p.P[(int64_t)n * p.ldp + (v - p.v0)] = pr;
    }
  }
}

// row capacity of each split's partials: N, or -- live rows, where the kernel re-partitions its CTAs on the device -- whole row
// tiles (groups x live row tiles <= launched CTAs, so [4 x launched splits][row tiles x 128] holds every layout it can pick)
static int64_t part_rows(const CeArgs& p) { return p.m_live ? (int64_t)ceil_div(p.N, GCE::BM) * GCE::BM : p.N; }

// per-(row, vocabulary split) partials: tensor-core kernel when the shape allows, fp32 SIMT otherwise
// On return p.nsplit / p.part_idx describe the partials that were actually written (the fp16-split kernel's two
// -- four with pre-split operands -- epilogue warp sets each emit their own split).
static int ce_partials(CeArgs& p, cudaStream_t st) {
  if (!force_simt_gemm() && p.N >= 64 && p.V >= 128 && p.H >= 32 && tc16::supported(p.h, p.ldh, 0, p.w, p.H, 0, p.N, p.V, p.H)) {
    const int launched = p.nsplit;
    p.nsplit = (p.h_planes && p.w_planes ? 4 : 2) * launched;      // pre-split operands: 16 epilogue warps, 4 column chunks
    p.part_idx = reinterpret_cast<int*>(p.part + (int64_t)p.nsplit * part_rows(p) * 4);
    if (p.m_live) p.live_ctas = ceil_div(p.N, GCE::BM) * launched;
    return tc16::ce_partials(p.h, p.ldh, p.N, p.B, p.H, p.V, p.w, p.bias, p.targets, p.tgt_stride_b, p.lengths,
                             p.tiles_per_split, launched, p.part, p.part_idx, p.gumbel_seed, p.gumbel_salt, p.h_planes,
                             p.w_planes, p.skip_flag, st, p.m_live, p.rows);
  }
  if (!force_simt_gemm() && p.N >= 64 && p.V >= 128 && p.H >= 32 && tc::tc_linear_supported(p.h, p.ldh, p.w, p.H, p.N, p.V, p.H))
    return tc::tc_ce_partials(p.h, p.ldh, p.N, p.B, p.H, p.V, p.w, p.bias, p.targets, p.tgt_stride_b, p.lengths,
                              p.tiles_per_split, p.nsplit, p.part, p.part_idx, p.gumbel_seed, p.gumbel_salt, st);
  dim3 grid(ceil_div(p.N, GCE::BM), p.nsplit);
  vocab_ce_fwd_kernel<<<grid, GCE::NT, 0, st>>>(p);
  DVAE_LAUNCH_CHECK();
  return DVAE_OK;
}

static int ce_nsplit(int N, int V, int* tiles_per_split) {
  int row_tiles = ceil_div(N, GCE::BM), vtiles = ceil_div(V, GCE::BN);
  // ONE wave of CTAs (row tiles x splits <= 148), each with a long run of vocabulary tiles: a second wave pays the
  // kernel's prologue (A rows into tensor memory, pipeline fill) again -- 2 x 147 CTAs of 6 tiles took 51 us at cfg 2
  int want = 148 / row_tiles;
  if (want < 1) want = 1;
  if (want > vtiles) want = vtiles;
  int tps = ceil_div(vtiles, want);
  *tiles_per_split = tps;
  return ceil_div(vtiles, tps);
}

static int p_chunk(int N, int V) {
  // keep the softmax chunk under ~56 MB so it stays L2-resident between producer and consumers, and make the chunks
  // equal: at cfg 2 (N = 2688, V = 10000) two chunks of 5120 / 4880 columns instead of 4608 + 4608 + a 784-column
  // remainder whose three kernels cost 43 us for 8 % of the work
  int64_t vmax = (14LL << 20) / (N > 0 ? N : 1);
  vmax = vmax / 128 * 128;
  if (vmax < 128) vmax = 128;
  const int64_t vr = (int64_t)ceil_div(V, 128) * 128;
  if (vmax >= vr) return (int)vr;
  const int64_t nc = (vr + vmax - 1) / vmax;
  const int64_t vc = ((V + nc - 1) / nc + 127) / 128 * 128;
  return (int)vc;
}

// P as fp16 operand planes in both orientations (8 bytes per element instead of 4).  Each plane set is written once and read
// once, so it may stream through HBM: ONE chunk (the whole vocabulary) up to 4 GB of planes -- 217 MB at cfg 2, 3.2 GB at
// cfg 4 -- instead of L2-sized chunks: a third fewer launches and longer K loops (measured: cfg 2 step 1.290 -> 1.237 ms with
// 1 chunk instead of 3, the backward call 247 -> 188 us; cfg 4: 9.7 -> 7.9 ms).
static int p_chunk_planes(int N, int V) {
  static const int64_t budget = [] {      // elements per chunk (8 bytes each); DVAE_VOCAB_PCHUNK_M = millions (A/B knob)
    const char* e = getenv("DVAE_VOCAB_PCHUNK_M");
    return (int64_t)(e ? atoi(e) : 512) << 20;
  }();
  int64_t vmax = budget / (N > 0 ? N : 1);
  vmax = vmax / 128 * 128;
  if (vmax < 128) vmax = 128;
  const int64_t vr = (int64_t)ceil_div(V, 128) * 128;
  if (vmax >= vr) return (int)vr;
  const int64_t nc = (vr + vmax - 1) / vmax;
  return (int)(((V + nc - 1) / nc + 127) / 128 * 128);
}
static bool tplanes_enabled() {      // DVAE_VOCAB_TPLANES=0: the gradient GEMMs convert W_out^T / h^T in every CTA
  const char* e = getenv("DVAE_VOCAB_TPLANES");
  return !(e && e[0] == '0');
}
static bool p_planes_enabled() {
  const char* e = getenv("DVAE_VOCAB_PPLANES");
  return !(e && e[0] == '0');
}


// ---- live rows: the decoder positions the loss keeps ----------------------------------------------------------------
// Position n = t * B + b (row t + 1 of the targets) enters the loss only when t + 1 < len_b: its loss weight is zero and its
// softmax gradient exactly zero otherwise.  The live-row path runs the vocabulary GEMMs over the live rows only, in
// ascending n (so the loss sums in a fixed order), with the count M known on the device only: launch grids stay sized for
// every position and tc16_gemm_kernel re-partitions its CTAs from *m_live, so one captured graph serves every length mix.

// rows[k] = position of live row k (ascending), *m_live = M.  One CTA of up to 1024 threads: per position t, a ballot over
// the batch ranks each live b among those before it.
__global__ void __launch_bounds__(1024) vocab_live_rows_kernel(const int64_t* __restrict__ lengths, int T1, int B, int* __restrict__ rows,
                                                               int* __restrict__ m_live) {
  __shared__ int wcnt[32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  int base = 0;
  for (int t = 0; t < T1; ++t) {
    for (int b0 = 0; b0 < B; b0 += blockDim.x) {
      const int b = b0 + threadIdx.x;
      const bool live = b < B && t + 1 < lengths[b];
      const unsigned bal = __ballot_sync(0xffffffffu, live);
      if (lane == 0) wcnt[w] = __popc(bal);
      __syncthreads();
      int before = 0, total = 0;
      for (int i = 0; i < nw; ++i) {
        const int c = wcnt[i];
        before += i < w ? c : 0;
        total += c;
      }
      __syncthreads();      // wcnt is rewritten by the next round
      if (live) rows[base + before + __popc(bal & ((1u << lane) - 1))] = t * B + b;
      base += total;
    }
  }
  if (threadIdx.x == 0) *m_live = base;
}

// The live rows of h [N, H] (row stride H) as operand planes, rows in row-list order:
//   a_planes: the A operand of the forward / softmax-gradient GEMMs, [M rows, K = H] (scale / lo_scale: the convention of
//             tc16::split_planes for K = H);
//   t_planes: the B operand of d_w = P^T . h, [H rows, K = positions], dual-accumulator convention (weight_planes_kernel),
//             k-blocks per row block for all N positions.
// Rows M .. the next 128-row tile of a_planes and positions M .. the next 32-position k-block of t_planes are written as
// zeros: the GEMMs read them (multiplied by zeros of P, which would not clear a stale NaN).
__global__ void __launch_bounds__(256) vocab_live_gather_kernel(const float* __restrict__ h, int N, int H, const int* __restrict__ rows,
                                                                const int* __restrict__ m_live, float a_scale, float a_lo_scale,
                                                                uint8_t* __restrict__ a_planes, uint8_t* __restrict__ t_planes) {
  const int M = *m_live;
  const int KB = (H + 31) / 32, KC = KB * 4;
  const int64_t na = (int64_t)((M + 127) / 128) * 128 * KC;
  const int HP = (H + 127) / 128 * 128, KBt = (N + 31) / 32;
  const int64_t nt = (int64_t)HP * ((M + 31) / 32 * 4);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < na + nt; i += (int64_t)gridDim.x * blockDim.x) {
    float v[8];
    if (i < na) {
      const int kc = (int)(i % KC), r = (int)(i / KC);
      if (r < M && kc * 8 + 8 <= H) {
        const float4* src = reinterpret_cast<const float4*>(h + (int64_t)__ldg(rows + r) * H + kc * 8);
        const float4 x0 = __ldg(src), x1 = __ldg(src + 1);
        v[0] = x0.x; v[1] = x0.y; v[2] = x0.z; v[3] = x0.w; v[4] = x1.x; v[5] = x1.y; v[6] = x1.z; v[7] = x1.w;
      } else {
#pragma unroll
        for (int e = 0; e < 8; ++e) v[e] = 0.f;
      }
      uint4 hi, lo;
      hi.x = tc16::pack_hi_lo(v[0], v[1], a_scale, lo.x, a_lo_scale); hi.y = tc16::pack_hi_lo(v[2], v[3], a_scale, lo.y, a_lo_scale);
      hi.z = tc16::pack_hi_lo(v[4], v[5], a_scale, lo.z, a_lo_scale); hi.w = tc16::pack_hi_lo(v[6], v[7], a_scale, lo.w, a_lo_scale);
      const int64_t off = tc16::plane_chunk_offset(r, kc * 8, KB);
      *reinterpret_cast<uint4*>(a_planes + off) = hi;
      *reinterpret_cast<uint4*>(a_planes + off + tc16::kPlaneBytes) = lo;
    } else {
      // consecutive threads: consecutive hidden units, so each of the 8 loads is a coalesced segment of one row of h
      const int64_t j = i - na;
      const int r = (int)(j % HP), k0 = (int)(j / HP) * 8;
#pragma unroll
      for (int e = 0; e < 8; ++e) v[e] = (r < H && k0 + e < M) ? __ldg(h + (int64_t)__ldg(rows + k0 + e) * H + r) : 0.f;
      tc16::store_plane_chunk(t_planes, r, k0, KBt, v, 1.f);
    }
  }
}

}  // namespace dvae

using namespace dvae;

// workspace layout (floats): [partials 4*ns*N'*5 + 8][block sums][pad to 4][operand planes of h and w]
//   [live rows: planes of h^T (B operand of d_w) | row list (N ints) | live count (1 int) | pad]      (N' = N in whole row tiles)
static int64_t ce_part_floats(int N, int V) {
  int tps;
  int ns = ce_nsplit(N, V, &tps);
  const int64_t rows = (int64_t)ceil_div(N, GCE::BM) * GCE::BM;
  return (4LL * ns * rows * 5 + 8 + kFinMaxBlocks + 3) / 4 * 4;    // x4: the fp16-split kernel writes up to four partials per (row, split)
}
static int64_t live_off(int N, int V, int H) { return ce_part_floats(N, V) + tc16::plane_floats(N, H) + tc16::plane_floats(V, H); }
extern "C" int64_t dvae_vocab_ce_ws_floats(int N, int V, int H) {
  return live_off(N, V, H) + tc16::plane_floats(H, N) + (N + 8 + 3) / 4 * 4;
}
// float offset of the row list in the forward workspace (the live count follows its N entries)
extern "C" int64_t dvae_vocab_live_rows_at(int N, int V, int H) { return live_off(N, V, H) + tc16::plane_floats(H, N); }

// (ws, w) of the last dvae_vocab_split_w call that actually wrote W planes on this host thread
static thread_local const void* g_wsplit_ws = nullptr;
static thread_local const void* g_wsplit_w = nullptr;

// The W half of the operand split of dvae_vocab_ce_fwd, as a call of its own: W_out does not depend on the step's
// activations, so a caller can run this early, on another stream, and pass flags bit 0 to dvae_vocab_ce_fwd_ex.
// N, V, H and ws as in the forward call that follows.  A no-op for shapes the pre-split kernels do not take.
extern "C" int dvae_vocab_split_w(const float* w, int N, int V, int H, float* ws, void* stream) {
  DVAE_REQUIRE(w && ws && N > 0 && V > 0 && H > 0, "dvae_vocab_split_w: bad argument");
  g_wsplit_ws = g_wsplit_w = nullptr;
  if (force_simt_gemm() || !tc16::enabled() || !use_presplit(N, V, H) || (reinterpret_cast<uintptr_t>(w) & 15)) return DVAE_OK;
  float* wp = ws + ce_part_floats(N, V) + tc16::plane_floats(N, H);
  int rc = tc16::split_planes(w, H, V, H, 1.f, wp, (cudaStream_t)stream);
  if (rc) return rc;
  g_wsplit_ws = ws; g_wsplit_w = w;
  return DVAE_OK;
}

// the live-row path runs on the pre-split kernels with the softmax gradient as operand planes; other shapes run every row
static bool live_ok(int N, int V, int H, const float* h, int64_t ldh, const float* w) {
  return use_tc16(N, V, H, h, ldh, w) && use_presplit(N, V, H) && ldh == H && (reinterpret_cast<uintptr_t>(h) & 15) == 0 &&
         (reinterpret_cast<uintptr_t>(w) & 15) == 0 && p_planes_enabled() && tplanes_enabled();
}

static int vocab_ce_fwd_impl(const float* h, int64_t ldh, int T1, int B, int H, int V, const float* w,
                             const float* bias, const int64_t* targets, int64_t tgt_stride_b,
                             const int64_t* lengths, int sos, float* lse, float* nll, int32_t* argmax,
                             float* loss, float* ws, bool w_planes_ready, bool live, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  DVAE_REQUIRE(h && w && bias && targets && lengths && loss && ws, "dvae_vocab_ce_fwd: null pointer");
  DVAE_REQUIRE(T1 > 0 && B > 0 && H > 0 && V > 0, "dvae_vocab_ce_fwd: bad shape T1=%d B=%d H=%d V=%d", T1, B, H, V);
  CeArgs p = {};
  p.h = h; p.ldh = ldh; p.w = w; p.bias = bias; p.targets = targets; p.tgt_stride_b = tgt_stride_b;
  p.lengths = lengths; p.N = T1 * B; p.B = B; p.H = H; p.V = V; p.sos = sos;
  p.nsplit = ce_nsplit(p.N, V, &p.tiles_per_split);
  p.part = ws;
  p.part_idx = reinterpret_cast<int*>(ws + (int64_t)p.nsplit * p.N * 4);
  p.gumbel_seed = nullptr; p.gumbel_salt = 0;
  p.h_planes = p.w_planes = nullptr; p.skip_flag = nullptr;
  if (use_tc16(p.N, V, H, h, ldh, w) && use_presplit(p.N, V, H)) {
    // both operands are re-read by every tile of the other dimension: split them into fp16 planes once
    float* hp = ws + ce_part_floats(p.N, V);
    float* wp = hp + tc16::plane_floats(p.N, H);
    int rc;
    if (live && live_ok(p.N, V, H, h, ldh, w)) {
      // live rows: the row list, then the live rows of h as the A planes here and as the h^T planes of the backward's d_w
      float* tp = ws + live_off(p.N, V, H);
      int* rows = reinterpret_cast<int*>(tp + tc16::plane_floats(H, p.N));
      const int nthr = min(1024, ceil_div(B, 32) * 32);
      vocab_live_rows_kernel<<<1, nthr, 0, st>>>(lengths, T1, B, rows, rows + p.N);
      DVAE_LAUNCH_CHECK();
      const bool single = tc16::single_acc_planes(H);
      const int64_t items = (tc16::plane_floats(p.N, H) + tc16::plane_floats(H, p.N)) / 16;
      const int blocks = ceil_div(items, 256) < 148 * 4 ? ceil_div(items, 256) : 148 * 4;
      vocab_live_gather_kernel<<<blocks, 256, 0, st>>>(h, p.N, H, rows, rows + p.N, single ? tc16::kSingleScale : 1.f,
                                                       single ? 1.f : tc16::kPlaneLoScale, reinterpret_cast<uint8_t*>(hp),
                                                       reinterpret_cast<uint8_t*>(tp));
      DVAE_LAUNCH_CHECK();
      p.rows = rows; p.m_live = rows + p.N;
    } else if ((rc = tc16::split_planes(h, ldh, p.N, H, 1.f, hp, st))) {
      return rc;
    }
    // W planes: skipped when the caller vouches for an earlier dvae_vocab_split_w on the same (ws, w) since the last
    // weight update, and that call did write them
    if (!(w_planes_ready && g_wsplit_ws == ws && g_wsplit_w == w) && (rc = tc16::split_planes(w, H, V, H, 1.f, wp, st))) return rc;
    p.h_planes = hp; p.w_planes = wp;
  }
  g_wsplit_ws = g_wsplit_w = nullptr;
  { int rc = ce_partials(p, st); if (rc) return rc; }
  float* block_sums = ws + (int64_t)p.nsplit * part_rows(p) * 5 + 8;      // p.nsplit: as updated by ce_partials
  const int nblk = min(kFinMaxBlocks, ceil_div(p.N, kFinThreads / kFinLanes));
  vocab_ce_finalize_kernel<<<nblk, kFinThreads, 0, st>>>(p, lse, nll, argmax, block_sums);
  DVAE_LAUNCH_CHECK();
  vocab_ce_loss_kernel<<<1, 128, 0, st>>>(p, block_sums, nblk, loss);
  DVAE_LAUNCH_CHECK();
  return DVAE_OK;
}

extern "C" int dvae_vocab_ce_fwd(const float* h, int64_t ldh, int T1, int B, int H, int V, const float* w,
                                 const float* bias, const int64_t* targets, int64_t tgt_stride_b,
                                 const int64_t* lengths, int sos, float* lse, float* nll, int32_t* argmax,
                                 float* loss, float* ws, void* stream) {
  return vocab_ce_fwd_impl(h, ldh, T1, B, H, V, w, bias, targets, tgt_stride_b, lengths, sos, lse, nll, argmax, loss, ws,
                           false, false, stream);
}

// flags bit 0: the W planes in ws are current (dvae_vocab_split_w on the same ws / w since the last weight update)
extern "C" int dvae_vocab_ce_fwd_ex(const float* h, int64_t ldh, int T1, int B, int H, int V, const float* w,
                                    const float* bias, const int64_t* targets, int64_t tgt_stride_b,
                                    const int64_t* lengths, int sos, float* lse, float* nll, int32_t* argmax,
                                    float* loss, float* ws, int flags, void* stream) {
  return vocab_ce_fwd_impl(h, ldh, T1, B, H, V, w, bias, targets, tgt_stride_b, lengths, sos, lse, nll, argmax, loss, ws,
                           (flags & 1) != 0, false, stream);
}

// dvae_vocab_ce_fwd_ex over the live rows only (positions t + 1 < len_b): lse / nll / argmax are written at live positions
// only, the loss is the same masked average.  ws keeps the row list, the live count and the h^T planes for
// dvae_vocab_ce_bwd_live.
extern "C" int dvae_vocab_ce_fwd_live(const float* h, int64_t ldh, int T1, int B, int H, int V, const float* w,
                                      const float* bias, const int64_t* targets, int64_t tgt_stride_b,
                                      const int64_t* lengths, int sos, float* lse, float* nll, int32_t* argmax,
                                      float* loss, float* ws, int flags, void* stream) {
  return vocab_ce_fwd_impl(h, ldh, T1, B, H, V, w, bias, targets, tgt_stride_b, lengths, sos, lse, nll, argmax, loss, ws,
                           (flags & 1) != 0, true, stream);
}

// softmax-gradient chunks alternate between two buffers when there is more than one chunk: the next chunk's P is then
// computed while this chunk's d_w GEMM (the longer of its two consumers) is still running
static int p_buffers(int N, int V) { return p_chunk(N, V) < V ? 2 : 1; }

// [softmax-gradient buffers][planes of h and w (when the forward call's are not reused)][planes of w^T and h^T: the
// B operands of d_h = P . W and d_w = P^T . h, which read W_out / h as [K, N]]
static int p_buffers_planes(int N, int V) { return p_chunk_planes(N, V) < V ? 2 : 1; }
// front region: the softmax-gradient chunk buffers, as fp32 [N, vc] or as operand planes in both orientations
static int64_t p_region_floats(int N, int V) {
  const int64_t a = (int64_t)p_buffers(N, V) * N * p_chunk(N, V);
  const int vcp = p_chunk_planes(N, V);
  const int64_t b = (int64_t)p_buffers_planes(N, V) * (tc16::plane_floats(N, vcp) + tc16::plane_floats(vcp, N));
  return (a > b ? a : b) + 4;
}
extern "C" int64_t dvae_vocab_ce_bwd_ws_floats(int N, int V, int H) {
  return p_region_floats(N, V) / 4 * 4 + tc16::plane_floats(N, H) + tc16::plane_floats(V, H) + tc16::plane_floats(H, V) +
         tc16::plane_floats(H, N);
}

// d_w GEMM CTA cap, A/B knob (measured: capping this one costs 17 us -- it outlasts the recurrence it runs beside)
static int dw_max_ctas() {
  static const int cap = [] { const char* e = getenv("DVAE_VOCAB_DW_MAX_CTAS"); return e ? atoi(e) : 0; }();
  return cap;
}

// planes of W_out^T [H, V] (B operand of d_h = P . W): registered by the caller, or added to `tab` to be split into tp
static const void* wT_planes_of(const float* w, int H, int V, float* tp, tc16::PlaneTable& tab, int* kbtot) {
  tc16::PlaneHit hit;
  if (tc16::find_weight_planes(w, H, 1, H, V, &hit) && hit.tile0 == 0 && hit.kb0 == 0) {
    *kbtot = hit.kbtot;
    return hit.planes;
  }
  tab.e[tab.n++] = tc16::PlaneTable::Entry{w, V, H, nullptr, tp};
  *kbtot = ceil_div(V, 32);
  return tp;
}

// The vocabulary backward with every operand as planes: per vocabulary chunk, the softmax-gradient kernel writes P as planes
// in both orientations (and adds the bias gradient), then d_h (+)= P . W and d_w = P^T . h, both bulk-copy fed.
// m_live / rows (live rows, see dvae_vocab_ce_bwd_live): P covers the live rows only, row k of d_h's GEMM is added into row
// rows[k] and d_w's K runs over the live positions; both GEMMs then accumulate into outputs cleared beforehand.
static int planes_bwd(const float* h, int64_t ldh, int N, int B, int H, int V, const float* w, const float* bias,
                      const int64_t* targets, int64_t tgt_stride_b, const int64_t* lengths, const float* lse,
                      const float* grad_scale_dev, float* d_h, int64_t lddh, float* d_w, float* d_bias, const void* h_planes,
                      const void* w_planes, const void* wT_planes, int wT_kbtot, const void* hT_planes, float a_scale, float* ws,
                      const int* m_live, const int* rows, cudaStream_t st) {
  const int vc_max = p_chunk_planes(N, V), nbuf = p_buffers_planes(N, V);
  const int64_t pa_fl = tc16::plane_floats(N, vc_max), pt_fl = tc16::plane_floats(vc_max, N);
  DVAE_CUDA(cudaMemsetAsync(d_bias, 0, sizeof(float) * V, st));
  int chunk = 0;
  const int nchunks = ceil_div(V, vc_max);
  for (int v0 = 0; v0 < V; v0 += vc_max, ++chunk) {
    const int vc = min(vc_max, V - v0);
    float* pa = ws + (int64_t)(chunk % nbuf) * (pa_fl + pt_fl);
    float* pt = pa + pa_fl;
    float* dw = d_w + (int64_t)v0 * H;
    // the softmax-gradient kernel clears d_h (once, all N rows) and this chunk's rows of d_w when they are aligned; the live-row
    // GEMMs accumulate in any case, so there a memset clears what the kernel cannot
    const bool zh = chunk == 0 && lddh == H && (((uintptr_t)d_h) & 15) == 0 && ((int64_t)N * H) % 4 == 0;
    const bool zw = (((uintptr_t)dw) & 15) == 0 && ((int64_t)vc * H) % 4 == 0;
    if (m_live && chunk == 0 && !zh) DVAE_CUDA(cudaMemsetAsync(d_h, 0, sizeof(float) * (size_t)N * H, st));      // lddh == H
    if (m_live && !zw) DVAE_CUDA(cudaMemsetAsync(dw, 0, sizeof(float) * (size_t)vc * H, st));
    int rc;
    if ((rc = tc16::softmax_grad(h, ldh, N, B, H, V, v0, vc, w, bias, targets, tgt_stride_b, lengths, lse, grad_scale_dev, nullptr,
                                 vc_max, h_planes, w_planes, zh ? d_h : nullptr, (int64_t)N * H / 4, zw ? dw : nullptr,
                                 (int64_t)vc * H / 4, st, pa, pt, d_bias + v0, a_scale, m_live, rows))) return rc;
    Fork fork(st);
    // d_h [N,H] (+)= P [N,vc] . W[v0:v0+vc, :]: A = P planes, B = planes of W_out^T, k-blocks v0/32 .. of its K = V axis
    if ((rc = tc16::linear_planes(pa, wT_planes, d_h, lddh, N, H, vc, nullptr, chunk ? 1.f : 0.f, 0, a_scale, 1.f, nullptr,
                                  m_live ? true : zh, 16, st, v0 / 32, wT_kbtot, 0, 0, 0, nullptr, 1, m_live, rows, 0))) return rc;
    // d_w[v0:v0+vc, :] = P^T [vc,N] . h [N,H]: A = transposed P planes, B = planes of h^T
    if ((rc = tc16::linear_planes(pt, hT_planes, dw, H, vc, H, N, nullptr, 0.f, 0, a_scale, 1.f, nullptr, m_live ? true : zw, 16,
                                  fork.side(0), 0, 0, dw_max_ctas(), 0, 0, nullptr, 1, m_live, nullptr, 1))) return rc;
    // main waits for the side branch only when the NEXT chunk reuses a buffer (or at the end)
    if (chunk + 1 == nchunks || chunk + 1 >= nbuf)
      if ((rc = fork.join())) return rc;
  }
  return DVAE_OK;
}

extern "C" int dvae_vocab_ce_bwd(const float* h, int64_t ldh, int T1, int B, int H, int V, const float* w,
                                 const float* bias, const int64_t* targets, int64_t tgt_stride_b,
                                 const int64_t* lengths, const float* lse, const float* grad_scale_dev,
                                 float* d_h, int64_t lddh, float* d_w, float* d_bias, const float* fwd_ws, float* ws,
                                 void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  DVAE_REQUIRE(h && w && bias && targets && lengths && lse && d_h && d_w && d_bias && ws, "dvae_vocab_ce_bwd: null pointer");
  DVAE_REQUIRE(T1 > 0 && B > 0 && H > 0 && V > 0, "dvae_vocab_ce_bwd: bad shape");
  const int N = T1 * B;
  int vc_max = p_chunk(N, V), nbuf = p_buffers(N, V);
  const int64_t front = p_region_floats(N, V) / 4 * 4;
  PArgs p;
  p.h = h; p.ldh = ldh; p.w = w; p.bias = bias; p.targets = targets; p.tgt_stride_b = tgt_stride_b;
  p.lengths = lengths; p.lse = lse; p.grad_scale = grad_scale_dev; p.N = N; p.B = B; p.H = H; p.V = V;
  p.P = ws; p.ldp = vc_max;
  // P = (softmax - onehot) * mask * grad_scale / B: |P| <= grad_scale / B, so a power-of-two scale near B brings it to
  // O(1) for the fp16-split GEMMs (exact; undone in their epilogue)
  GemmHints ph;
  ph.a_scale = 1.f;
  while (ph.a_scale * 2.f <= (float)B) ph.a_scale *= 2.f;
  const void *h_planes = nullptr, *w_planes = nullptr;
  if (use_tc16(N, min(vc_max, V), H, h, ldh, w) && use_presplit(N, V, H)) {
    if (fwd_ws) {        // the forward call's workspace still holds the fp16 planes of the same h and w
      const float* hp = fwd_ws + ce_part_floats(N, V);
      h_planes = hp; w_planes = hp + tc16::plane_floats(N, H);
    } else {
      float* hp = ws + front;
      float* wp = hp + tc16::plane_floats(N, H);
      int rc;
      if ((rc = tc16::split_planes(h, ldh, N, H, 1.f, hp, st))) return rc;
      if ((rc = tc16::split_planes(w, H, V, H, 1.f, wp, st))) return rc;
      h_planes = hp; w_planes = wp;
    }
  }
  // B operands of the two gradient GEMMs as fp16 planes, written once per call instead of converted in every CTA:
  // W_out^T [H, V] (registered by the caller, or split here) and h^T [H, N]
  const void *wT_planes = nullptr, *hT_planes = nullptr;
  int wT_kbtot = 0;
  if (h_planes && H % 32 == 0 && N >= 128 && (reinterpret_cast<uintptr_t>(w) & 15) == 0 && ldh == H && tplanes_enabled()) {
    float* tp = ws + front + tc16::plane_floats(N, H) + tc16::plane_floats(V, H);
    tc16::PlaneTable tab;
    tab.n = 0;
    wT_planes = wT_planes_of(w, H, V, tp, tab, &wT_kbtot);
    float* hp_t = tp + tc16::plane_floats(H, V);
    tab.e[tab.n++] = tc16::PlaneTable::Entry{h, N, H, nullptr, hp_t};
    hT_planes = hp_t;
    int rc = tc16::weight_planes_launch(tab, st);
    if (rc) return rc;
  }
  // P never exists as fp32: the softmax-gradient kernel writes fp16 operand planes in both orientations (and adds the bias
  // gradient), and the two gradient GEMMs are bulk-copy fed on both operands
  const bool pp = wT_planes && hT_planes && h_planes && w_planes && p_planes_enabled() && lddh % 4 == 0 &&
                  tc16::supported(h, ldh, 0, w, H, 0, N, min(vc_max, V), H);
  if (pp)
    return planes_bwd(h, ldh, N, B, H, V, w, bias, targets, tgt_stride_b, lengths, lse, grad_scale_dev, d_h, lddh, d_w, d_bias,
                      h_planes, w_planes, wT_planes, wT_kbtot, hT_planes, ph.a_scale, ws, nullptr, nullptr, st);
  int chunk = 0;
  const int nchunks = ceil_div(V, vc_max);
  for (int v0 = 0; v0 < V; v0 += vc_max, ++chunk) {
    const int vc = min(vc_max, V - v0);
    float* Pc = ws + (int64_t)(chunk % nbuf) * N * vc_max;      // this chunk's softmax-gradient buffer
    p.v0 = v0; p.vc = vc; p.P = Pc;
    int rc;
    bool dh_zeroed = false, dw_zeroed = false;
    if (!force_simt_gemm() && N >= 64 && vc >= 128 && H >= 32 && tc16::supported(h, ldh, 0, w, H, 0, N, vc, H)) {
      // the kernel also clears the outputs of this chunk's split-K GEMMs (d_h once, this chunk's rows of d_w): no memset nodes
      const bool zh = chunk == 0 && lddh == H && (((uintptr_t)d_h) & 15) == 0 && ((int64_t)N * H) % 4 == 0;
      const bool zw = (((uintptr_t)(d_w + (int64_t)v0 * H)) & 15) == 0 && ((int64_t)vc * H) % 4 == 0;
      if ((rc = tc16::softmax_grad(h, ldh, N, B, H, V, v0, vc, w, bias, targets, tgt_stride_b, lengths, lse, grad_scale_dev, Pc,
                                   vc_max, h_planes, w_planes, zh ? d_h : nullptr, (int64_t)N * H / 4,
                                   zw ? d_w + (int64_t)v0 * H : nullptr, (int64_t)vc * H / 4, st))) return rc;
      dh_zeroed = zh; dw_zeroed = zw;
    } else if (!force_simt_gemm() && N >= 64 && vc >= 128 && H >= 32 && tc::tc_linear_supported(h, ldh, w, H, N, vc, H)) {
      if ((rc = tc::tc_softmax_grad(h, ldh, N, B, H, v0, vc, w, bias, targets, tgt_stride_b, lengths, lse, grad_scale_dev, Pc,
                                    vc_max, st))) return rc;
    } else {
      dim3 grid(ceil_div(vc, GCE::BN), ceil_div(N, GCE::BM));
      vocab_p_kernel<<<grid, GCE::NT, 0, st>>>(p);
      DVAE_LAUNCH_CHECK();
    }
    // d_h [N,H] (+)= P [N,vc] . W[v0:v0+vc, :]        (B stored [K=vc][N=H])
    Fork fork(st);         // the three consumers of this chunk of P are independent of each other
    GemmHints ph_h = ph, ph_w = ph;
    ph_h.c_zeroed = dh_zeroed; ph_w.c_zeroed = dw_zeroed;
    if (wT_planes) { ph_h.b_planes = wT_planes; ph_h.b_tile0 = 0; ph_h.b_kb0 = v0 / 32; ph_h.b_kbtot = wT_kbtot; }
    if (hT_planes) { ph_w.b_planes = hT_planes; ph_w.b_tile0 = 0; ph_w.b_kb0 = 0; ph_w.b_kbtot = ceil_div(N, 32); }
    if ((rc = linear_impl_ex(Pc, vc_max, 0, w + (int64_t)v0 * H, H, 1, d_h, lddh, N, H, vc, nullptr, nullptr, chunk ? 1.f : 0.f, 0, ph_h, st))) return rc;
    // d_w[v0:v0+vc, :] = P^T [vc,N] . h [N,H]
    if ((rc = linear_impl_ex(Pc, vc_max, 1, h, ldh, 1, d_w + (int64_t)v0 * H, H, vc, H, N, nullptr, nullptr, 0.f, 0, ph_w, fork.side(0)))) return rc;
    if ((rc = colsum_impl(Pc, vc_max, N, vc, d_bias + v0, 0.f, fork.side(1)))) return rc;
    // main waits for the side branches only when the NEXT chunk reuses a buffer (or at the end): with two buffers the next
    // chunk's softmax gradient is computed under this chunk's d_w GEMM.  Side streams run their work in order, so a later
    // join covers the branches of every earlier chunk.
    if (chunk + 1 == nchunks || chunk + 1 >= nbuf)
      if ((rc = fork.join())) return rc;
  }
  return DVAE_OK;
}

// dvae_vocab_ce_bwd over the live rows of the dvae_vocab_ce_fwd_live call whose workspace is fwd_ws (same h, w, lengths,
// untouched since): the softmax gradient of the live rows only, as operand planes in both orientations; d_h = P . W with its
// row k accumulated into row rows[k] of d_h (every other row of d_h is zero) and d_w = P^T . h over the live positions.
// Shapes the live-row forward does not take were run over every row there, and are here too.
extern "C" int dvae_vocab_ce_bwd_live(const float* h, int64_t ldh, int T1, int B, int H, int V, const float* w,
                                      const float* bias, const int64_t* targets, int64_t tgt_stride_b,
                                      const int64_t* lengths, const float* lse, const float* grad_scale_dev,
                                      float* d_h, int64_t lddh, float* d_w, float* d_bias, const float* fwd_ws, float* ws,
                                      void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  DVAE_REQUIRE(h && w && bias && targets && lengths && lse && d_h && d_w && d_bias && ws && fwd_ws, "dvae_vocab_ce_bwd_live: null pointer");
  DVAE_REQUIRE(T1 > 0 && B > 0 && H > 0 && V > 0, "dvae_vocab_ce_bwd_live: bad shape");
  const int N = T1 * B;
  const bool fwd_live = live_ok(N, V, H, h, ldh, w);
  if (!fwd_live || lddh != H || (reinterpret_cast<uintptr_t>(d_h) & 15))
    // the forward's h planes hold the live rows only: the every-row path splits h itself
    return dvae_vocab_ce_bwd(h, ldh, T1, B, H, V, w, bias, targets, tgt_stride_b, lengths, lse, grad_scale_dev, d_h, lddh, d_w,
                             d_bias, fwd_live ? nullptr : fwd_ws, ws, stream);
  const float* hp = fwd_ws + ce_part_floats(N, V);
  const float* wp = hp + tc16::plane_floats(N, H);
  const float* hT_planes = fwd_ws + live_off(N, V, H);
  const int* rows = reinterpret_cast<const int*>(hT_planes + tc16::plane_floats(H, N));
  float a_scale = 1.f;      // power-of-two scale of P near B (see dvae_vocab_ce_bwd)
  while (a_scale * 2.f <= (float)B) a_scale *= 2.f;
  tc16::PlaneTable tab;
  tab.n = 0;
  int wT_kbtot;
  const void* wT_planes = wT_planes_of(w, H, V, ws + p_region_floats(N, V) / 4 * 4 + tc16::plane_floats(N, H) + tc16::plane_floats(V, H),
                                       tab, &wT_kbtot);
  int rc = tc16::weight_planes_launch(tab, st);
  if (rc) return rc;
  return planes_bwd(h, ldh, N, B, H, V, w, bias, targets, tgt_stride_b, lengths, lse, grad_scale_dev, d_h, lddh, d_w, d_bias, hp, wp,
                    wT_planes, wT_kbtot, hT_planes, a_scale, ws, rows + N, rows, st);
}

// Measurement entry (bench.py roofline, ncu): ONLY the projection + online-softmax partials kernel of dvae_vocab_ce_fwd.
// `ws` must come from an earlier dvae_vocab_ce_fwd call with the same arguments (it holds the fp16 operand planes).
extern "C" int dvae_vocab_ce_partials(const float* h, int64_t ldh, int T1, int B, int H, int V, const float* w,
                                      const float* bias, const int64_t* targets, int64_t tgt_stride_b,
                                      const int64_t* lengths, int sos, float* ws, void* stream) {
  DVAE_REQUIRE(h && w && bias && targets && lengths && ws, "dvae_vocab_ce_partials: null pointer");
  DVAE_REQUIRE(T1 > 0 && B > 0 && H > 0 && V > 0, "dvae_vocab_ce_partials: bad shape");
  CeArgs p = {};
  p.h = h; p.ldh = ldh; p.w = w; p.bias = bias; p.targets = targets; p.tgt_stride_b = tgt_stride_b;
  p.lengths = lengths; p.N = T1 * B; p.B = B; p.H = H; p.V = V; p.sos = sos;
  p.nsplit = ce_nsplit(p.N, V, &p.tiles_per_split);
  p.part = ws;
  p.part_idx = reinterpret_cast<int*>(ws + (int64_t)p.nsplit * p.N * 4);
  p.gumbel_seed = nullptr; p.gumbel_salt = 0;
  p.h_planes = p.w_planes = nullptr; p.skip_flag = nullptr;
  if (use_tc16(p.N, V, H, h, ldh, w) && use_presplit(p.N, V, H)) {
    float* hp = ws + ce_part_floats(p.N, V);
    p.h_planes = hp; p.w_planes = hp + tc16::plane_floats(p.N, H);
  }
  return ce_partials(p, (cudaStream_t)stream);
}

static int vocab_sample_step_impl(const float* h, int64_t ldh, int B, int H, int V, const float* w, const float* bias,
                                  const uint64_t* seed_dev, uint32_t salt, int64_t* tokens_out, int64_t tok_stride,
                                  const int32_t* forced_flag_dev, const float* w_planes, float* ws, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  DVAE_REQUIRE(h && w && bias && seed_dev && tokens_out && ws, "dvae_vocab_sample_step: null pointer");
  DVAE_REQUIRE(B > 0 && H > 0 && V > 0, "dvae_vocab_sample_step: bad shape");
  CeArgs p = {};
  p.h = h; p.ldh = ldh; p.w = w; p.bias = bias; p.targets = nullptr; p.tgt_stride_b = 0; p.lengths = nullptr;
  p.N = B; p.B = B; p.H = H; p.V = V; p.sos = 0;
  p.nsplit = ce_nsplit(p.N, V, &p.tiles_per_split);
  p.part = ws;
  p.part_idx = reinterpret_cast<int*>(ws + (int64_t)p.nsplit * p.N * 4);
  p.gumbel_seed = seed_dev; p.gumbel_salt = salt;
  p.h_planes = p.w_planes = nullptr;      // one decode step: h has B rows only, splitting w per step would not pay ...
  p.skip_flag = forced_flag_dev;
  if (w_planes && use_tc16(B, V, H, h, ldh, w) && use_presplit(B, V, H)) {
    // ... unless the caller split W_out once for the whole decode (dvae_vocab_w_planes): then only the step's B x H states
    // are split here (a few KB) and the projection runs as the bulk-copy-fed A-stationary kernel of the forward pass
    float* hp = ws + ce_part_floats(B, V);
    int rc2 = tc16::split_planes(h, ldh, B, H, 1.f, hp, st);
    if (rc2) return rc2;
    p.h_planes = hp; p.w_planes = w_planes;
  }
  int rc = ce_partials(p, st);
  if (rc) return rc;
  vocab_sample_finalize_kernel<<<ceil_div(B, 128), 128, 0, st>>>(p, tokens_out, tok_stride);
  DVAE_LAUNCH_CHECK();
  return DVAE_OK;
}

extern "C" int dvae_vocab_sample_step(const float* h, int64_t ldh, int B, int H, int V, const float* w, const float* bias,
                                      const uint64_t* seed_dev, uint32_t salt, int64_t* tokens_out, int64_t tok_stride,
                                      float* ws, void* stream) {
  return vocab_sample_step_impl(h, ldh, B, H, V, w, bias, seed_dev, salt, tokens_out, tok_stride, nullptr, nullptr, ws, stream);
}

extern "C" int dvae_vocab_sample_step_ex(const float* h, int64_t ldh, int B, int H, int V, const float* w, const float* bias,
                                         const uint64_t* seed_dev, uint32_t salt, int64_t* tokens_out, int64_t tok_stride,
                                         const int32_t* forced_flag_dev, float* ws, void* stream) {
  return vocab_sample_step_impl(h, ldh, B, H, V, w, bias, seed_dev, salt, tokens_out, tok_stride, forced_flag_dev, nullptr, ws, stream);
}

extern "C" int64_t dvae_vocab_w_planes_floats(int V, int H) { return tc16::plane_floats(V, H); }

extern "C" int dvae_vocab_w_planes(const float* w, int V, int H, float* planes, void* stream) {
  DVAE_REQUIRE(w && planes && V > 0 && H > 0, "dvae_vocab_w_planes: bad argument");
  return tc16::split_planes(w, H, V, H, 1.f, planes, (cudaStream_t)stream);
}

extern "C" int dvae_vocab_sample_step_planes(const float* h, int64_t ldh, int B, int H, int V, const float* w, const float* bias,
                                             const float* w_planes, const uint64_t* seed_dev, uint32_t salt, int64_t* tokens_out,
                                             int64_t tok_stride, const int32_t* forced_flag_dev, float* ws, void* stream) {
  return vocab_sample_step_impl(h, ldh, B, H, V, w, bias, seed_dev, salt, tokens_out, tok_stride, forced_flag_dev, w_planes, ws, stream);
}
