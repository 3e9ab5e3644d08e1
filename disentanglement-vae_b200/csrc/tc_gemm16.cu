// Tensor-core GEMM, second generation: C[M,N] = A . B^T with fp32 operands in HBM, computed by tcgen05.mma.kind::f16
// on fp16 (hi, lo) operand planes produced on the fly:
//     hi = fp16(x * s)            lo = fp16((x * s - hi) * 2^11)            (s = optional power-of-two operand scale)
//     D1 += A_hi * B_hi           D2 += A_hi * B_lo + A_lo * B_hi           C = (D1 + D2 * 2^-11) / (s_a * s_b)
// 22 mantissa bits per operand and fp32 accumulation in TMEM: fp32-grade results (forward-loss parity 1e-5, identical
// arg-max) for THREE K=16 MMAs per 16 k, where the 3xTF32 kernel (tc_gemm.cu) needs six K=8 ones and twice the
// shared-memory bytes per k.  Shared-memory bandwidth is what bounds both kernels, so the work is organised to
// touch SMEM as little as possible:
//   warp 5    (TMA): cp.async.bulk.tensor (no swizzle, zero fill handles every tail) of raw fp32 A / B k-blocks into a
//              3-stage landing ring, so 96 KB of loads are in flight per SM (bytes in flight, not SMEM bandwidth or
//              MMA issue, is what bounds these fp32-operand GEMMs: profiles/probes/tc16_timeline.py).
//   warps 6-13 (converters): conflict-free LDS of the landed tile, scale + split, 16-byte stores into the UMMA
//              no-swizzle K-major core-matrix layout (padded so that the stores are conflict-free too).  MN-major
//              sources (transposed operands of the backward GEMMs) are transposed on the way, so the MMA only ever
//              sees K-major tiles.
//   warp 4    (MMA): elect.sync'ed single-thread issue from a warp-uniform branch (descriptors stay in uniform
//              registers), 5-stage ring, tcgen05.commit frees ring slots and publishes accumulators.
//   warps 0-3 (epilogue): double-buffered accumulators (2 x (D1, D2) = 512 TMEM columns) so read-out, bias /
//              activation / softmax statistics and the global stores of tile i overlap the main loop of tile i+1.
// Modes are those of tc_gemm.cu: 0 plain linear (bias, tanh, beta, split-K), 1 vocab-CE forward partials (online
// log-softmax / arg-max / Gumbel-max sampling), 2 softmax-gradient chunk.
#include <cuda_fp16.h>
#include <stdlib.h>
#include <string.h>

#include "tc_gemm.cuh"
#include "tc_gemm16.cuh"
#include "tc_planes.cuh"

namespace dvae {
namespace tc16 {

using namespace tc;

constexpr int BM = 128, BN = 128, BK = 32;
// Operand ring: 6 stages of 32 KB.  A stage is filled by TMA with the raw fp32 k-block [A 128 x 32 | B 128 x 32] and then
// converted IN PLACE by the converter warps into the four fp16 planes the MMAs read, [A_hi | A_lo | B_hi | B_lo], each
// 128 x 32 in the dense core-matrix layout (8 rows x 16 B matrices, LBO 128 B along K, SBO 512 B along rows).  fp32 in,
// hi + lo out: same bytes, so landing buffers and operand planes share one ring and all of it hides TMA latency
// (a separate 2-stage landing ring + 3-stage padded plane ring delivered a k-block every 0.73 us; TMA latency under load
// is ~1.3 us, so the stages in flight, not the converters or the MMAs, set the pace).
constexpr int STAGES = 6, MAX_STAGES = 14;
constexpr int RAW_TILE = BM * BK * 4;              // one landed fp32 tile: 16 KB  (= hi + lo fp16 planes of the same tile)
constexpr int STAGE_BYTES = 2 * RAW_TILE;          // A, B
constexpr int PS_PLANE = BM * BK * 2, PS_TILE = 2 * PS_PLANE;      // one fp16 plane: 8 KB; [hi, lo] of one operand tile: 16 KB
constexpr int PS_LBO = 128, PS_SBO = 512;
static_assert(PS_TILE == RAW_TILE, "in-place conversion: fp16 hi + lo planes occupy exactly the landed fp32 tile");
constexpr int EPI_WARPS = 8, MMA_WARP = 4, TMA_WARP = 5, PROD_WARP0 = 6, PROD_WARPS = 16, EPI2_WARP0 = PROD_WARP0 + PROD_WARPS;
// warps 0-3: epilogue of tile columns 0-63; warps 22-25 (22 % 4 == 2: TMEM lane quarter = warp & 3): columns 64-127
constexpr int NUM_THREADS = (EPI2_WARP0 + 4) * 32;               // 832: <= 78 registers per thread
constexpr int CONV_BARRIER = 1;                                  // named barrier of the 512 converter threads
constexpr int EPI_SCRATCH_BYTES = 8 * 32 * 32 * 4;               // per epilogue warp: a 32 x 32 fp32 transpose tile (XOR-swizzled)
// Pre-split mode (operands already split into tile-blocked fp16 planes in global memory): no converters -- bulk copies
// deliver MMA-ready stages [A tile | B tile] straight into the ring.
// A-stationary variant (pre-split, K <= 256, no split-K: the vocabulary kernels): the CTA's A rows live in TENSOR MEMORY
// for its whole run of N tiles (A operand of tcgen05.mma from TMEM: lane = row, 128 columns per fp16 plane), and all
// three products accumulate into ONE fp32 accumulator -- the planes of this variant keep `lo = fp16(x*s - hi)` unscaled,
// with s = 2^8 so that lo stays a normal fp16 number -- which leaves TMEM as [acc 0 | acc 1 | A_hi | A_lo] x 128 columns.
// Shared memory then holds nothing but the B ring: 7 stages of 32 KB in mode 1 (no transpose scratch), 6 in mode 2
// -- ~3 us of fetch latency covered, where 128 KB of stationary A rows in shared memory left room for 6 stages and the
// ring, not the MMAs, set the pace.
// A stage of this ring is TWO k-blocks (32 KB, one bulk copy: consecutive k-blocks of a row block are contiguous in the
// planes): the full / empty handshake per stage costs the MMA-issuing thread ~0.1 us (measured: 2.05 us per tile with no
// handshakes, 2.9 with one per k-block), so it is paid per 12 MMAs instead of per 6.
#ifndef DVAE_AS_KB
#define DVAE_AS_KB 2
#endif
constexpr int AS_MAX_KB = 8, AS_KB_PER_STAGE = DVAE_AS_KB, AS_STAGE_BYTES = AS_KB_PER_STAGE * PS_TILE;
constexpr int AS_STAGES = 12 / AS_KB_PER_STAGE, AS_STAGES_NOSCRATCH = 14 / AS_KB_PER_STAGE;
constexpr uint32_t AS_T_AHI = 256, AS_T_ALO = 384;       // TMEM columns of the stationary A planes
// [operand ring 192 KB][epilogue transpose scratch 32 KB][bias tiles 2 KB][barriers]
constexpr int OFF_SCRATCH = STAGES * STAGE_BYTES;
constexpr int OFF_BIAS = OFF_SCRATCH + EPI_SCRATCH_BYTES;          // per epilogue warp: the bias values of its tile columns
constexpr int OFF_BAR = OFF_BIAS + 8 * 64 * 4;
constexpr int SMEM_BYTES = OFF_BAR + 512;
static_assert(AS_STAGES * AS_STAGE_BYTES <= OFF_SCRATCH, "A-stationary ring must end before the transpose scratch");
static_assert(AS_STAGES_NOSCRATCH * AS_STAGE_BYTES <= OFF_BIAS, "A-stationary mode-1 ring must end before the bias tiles");
static_assert(AS_STAGES_NOSCRATCH <= MAX_STAGES && (3 * MAX_STAGES + 5) * 8 + 4 <= 512, "barrier area");
static_assert(SMEM_BYTES <= 232448, "shared memory per CTA");
constexpr int TMEM_COLS = 512;
constexpr float kLoScale = 2048.f, kLoInv = 1.f / 2048.f;

// 2^x, flush-to-zero: ONE MUFU.  `__expf` without -use_fast_math wraps its ex2 in a denormal-range fix-up (FSETP + two
// predicated FMULs through a single predicate register), which serialised the 16 exponentials of an epilogue block.
__device__ __forceinline__ float ex2_ftz(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
constexpr float kLog2e = 1.4426950408889634f;

__device__ __forceinline__ unsigned long long gtime16() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
// Main-loop probes (profiles/probes/tc16_*timeline.py) are compiled in only with -DDVAE_TC16_PROBES: per-k-block marks
// and the DVAE_TC_SKIP_EPILOGUE bit switches cost instructions in the loops they observe.
#ifdef DVAE_TC16_PROBES
#define DVAE_TC16_FLAG(bit) (p.dbg_skip_epilogue & (bit))
#define DVAE_TC16_MARK(cond, i) do { if (cond) DBG16(i); } while (0)
#else
#define DVAE_TC16_FLAG(bit) false
#define DVAE_TC16_MARK(cond, i) do { } while (0)
#endif
#define DBG16(i) do { if (p.dbg && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0) p.dbg[i] = gtime16(); } while (0)

__device__ __forceinline__ float scale_from_amax(const uint32_t* amax_bits, int n, float static_scale) {
  if (!amax_bits) return static_scale;
  uint32_t mx = 0;                       // bit patterns of non-negative floats order like the floats
  for (int i = 0; i < n; ++i) mx = max(mx, __ldg(amax_bits + i));
  // 2^(13 - floor(log2 amax)): the largest element lands in [2^13, 2^14), well inside fp16 range
  int se = 267 - (int)(mx >> 23);
  se = se < 1 ? 1 : (se > 253 ? 253 : se);
  return __uint_as_float((unsigned)se << 23);
}

// One landed k-block (128 rows x 32 k, fp32) of one operand -> 8 registers per converter thread (512 threads): thread
// (row = ptid & 127, k chunk kc = ptid >> 7) owns k 8*kc .. 8*kc+7 of its row, i.e. exactly one 16-byte fp16 chunk of each plane.
//   K-major source: the tile is [128 rows][32 k] (128-byte rows) landed with TMA's 128-byte swizzle: 16-byte piece c of row r
//     sits at piece c ^ (r & 7), so the 8 lanes of a quarter warp (8 consecutive rows, same k) read 8 different bank groups.
//   MN-major source: the tile is [32 k][128 rows], un-swizzled: 8 scalar reads with the warp's lanes on consecutive rows.
__device__ __forceinline__ void load_tile(uint32_t raw, int mn_major, int ptid, float (&v)[8]) {
  const int row = ptid & 127, kc = ptid >> 7;
  if (!mn_major) {
    const uint32_t ra = raw + (uint32_t)row * 128, sw = row & 7;
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const uint4 t = lds128(ra + (((uint32_t)(2 * kc + i) ^ sw) << 4));
      v[4 * i] = __uint_as_float(t.x); v[4 * i + 1] = __uint_as_float(t.y);
      v[4 * i + 2] = __uint_as_float(t.z); v[4 * i + 3] = __uint_as_float(t.w);
    }
  } else {
    const uint32_t src = raw + (uint32_t)(8 * kc) * (BM * 4) + (uint32_t)row * 4;
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = lds32(src + j * (BM * 4));
  }
}

// scale, split into fp16 (hi, lo) and store this thread's chunk into the operand planes (hi at `tile`, lo at + PS_PLANE):
// a quarter warp writes 128 contiguous bytes (8 rows of one core matrix)
__device__ __forceinline__ void store_tile(uint32_t tile, int ptid, float s, const float (&v)[8]) {
  const int row = ptid & 127, kc = ptid >> 7;
  const uint32_t base = tile + (uint32_t)(row >> 3) * PS_SBO + (uint32_t)kc * PS_LBO + (row & 7) * 16;
  uint4 hi, lo;
  hi.x = pack_hi_lo(v[0], v[1], s, lo.x);
  hi.y = pack_hi_lo(v[2], v[3], s, lo.y);
  hi.z = pack_hi_lo(v[4], v[5], s, lo.z);
  hi.w = pack_hi_lo(v[6], v[7], s, lo.w);
  sts128(base, hi);
  sts128(base + PS_PLANE, lo);
}

// ---- CTA-pair helpers (pre-split A-stationary kernels: the B tiles are shared by the CTAs of neighbouring row blocks) ----
__device__ __forceinline__ uint32_t cluster_size() {
  uint32_t n;
  asm volatile("mov.u32 %0, %%cluster_nctaid.x;" : "=r"(n));
  return n;
}
__device__ __forceinline__ uint32_t cluster_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// one global read, delivered to the same shared-memory offset (and mbarrier) of every CTA in `mask`
__device__ __forceinline__ void bulk_load_multicast(uint32_t smem_dst, const void* src, uint32_t bytes, uint64_t* bar, uint16_t mask) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1], %2, [%3], %4;" ::"r"(smem_dst),
               "l"(src), "r"(bytes), "r"(smem_u32(bar)), "h"(mask)
               : "memory");
}
// tcgen05.commit arriving on the same mbarrier offset of every CTA in `mask`
__device__ __forceinline__ void tc_commit_multicast(uint64_t* bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
               "h"(mask)
               : "memory");
}

// contiguous global -> shared bulk copy (no tensor map), completion on an mbarrier
__device__ __forceinline__ void bulk_load(uint32_t smem_dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_dst), "l"(src),
               "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// X [R, K] fp32 (row stride ld) -> fp16 planes hi / lo, stored tile by tile exactly as the MMA reads them from shared
// memory, so that one 16 KB bulk copy delivers a k-block of a 128-row operand tile:
//   tile (rb, kb) = rows rb*128.., k kb*32..  at byte ((rb * KB + kb) * 16384), KB = ceil(K / 32): [hi plane 8 KB][lo plane 8 KB],
//   element (r, k) of a plane at ((r / 8) * 4 + k / 8) * 128 + (r % 8) * 16 + (k % 8) * 2   (core matrices: LBO 128, SBO 512).
// Rows / columns beyond R / K are zero (R padded to 128, K to 32).
__global__ void split_planes_kernel(const float* __restrict__ X, int64_t ld, int R, int K, float scale, float lo_scale,
                                    uint8_t* __restrict__ planes) {
  const int KB = (K + BK - 1) / BK, KC = KB * (BK / 8), RP = (R + BM - 1) / BM * BM;
  const int64_t total = (int64_t)RP * KC;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int kc = (int)(i % KC), r = (int)(i / KC);            // consecutive threads: consecutive 32-byte pieces of a row
    float v[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) v[e] = (r < R && kc * 8 + e < K) ? __ldg(X + (int64_t)r * ld + kc * 8 + e) : 0.f;
    uint4 h, l;
    h.x = pack_hi_lo(v[0], v[1], scale, l.x, lo_scale); h.y = pack_hi_lo(v[2], v[3], scale, l.y, lo_scale);
    h.z = pack_hi_lo(v[4], v[5], scale, l.z, lo_scale); h.w = pack_hi_lo(v[6], v[7], scale, l.w, lo_scale);
    const int64_t off = ((int64_t)(r >> 7) * KB + (kc >> 2)) * (2 * PS_PLANE) + ((r & 127) >> 3) * PS_SBO + (kc & 3) * PS_LBO + (r & 7) * 16;
    *reinterpret_cast<uint4*>(planes + off) = h;
    *reinterpret_cast<uint4*>(planes + off + PS_PLANE) = l;
  }
}

// Planes of up to kMaxPlaneEntries registered weights in ONE launch (blockIdx.y = 2 * entry + orientation):
//   orientation 0: planes of W [R, C] (K = C), as split_planes_kernel (dual-accumulator convention);
//   orientation 1: planes of W^T [C, R] (K = R): the B operand of the GEMMs that read W as [K, N] (dx = dG . W_ih, d_h = P . W_out).
//     Consecutive threads take consecutive columns of W, so each of a thread's 8 loads is a coalesced row segment.
__global__ void weight_planes_kernel(PlaneTable tab) {
  const PlaneTable::Entry e = tab.e[blockIdx.y >> 1];
  const int tr = blockIdx.y & 1;
  uint8_t* out = reinterpret_cast<uint8_t*>(tr ? e.planes_t : e.planes);
  if (!out) return;
  const int R = tr ? e.C : e.R, K = tr ? e.R : e.C;           // rows / depth of the matrix being split
  const int64_t ld = e.ld ? e.ld : e.C;
  const float sc = scale_from_amax(e.amax, e.amax_n, 1.f);
  const int KB = (K + BK - 1) / BK, KC = KB * (BK / 8), RP = (R + BM - 1) / BM * BM;
  const int64_t total = (int64_t)RP * KC;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int kc, r;
    if (!tr) { kc = (int)(i % KC); r = (int)(i / KC); }
    else { r = (int)(i % RP); kc = (int)(i / RP); }
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int k = kc * 8 + j;
      v[j] = (r < R && k < K) ? __ldg(tr ? e.w + (int64_t)k * ld + r : e.w + (int64_t)r * ld + k) : 0.f;
    }
    uint4 h, l;
    h.x = pack_hi_lo(v[0], v[1], sc, l.x); h.y = pack_hi_lo(v[2], v[3], sc, l.y);
    h.z = pack_hi_lo(v[4], v[5], sc, l.z); h.w = pack_hi_lo(v[6], v[7], sc, l.w);
    const int64_t off = ((int64_t)(r >> 7) * KB + (kc >> 2)) * (2 * PS_PLANE) + ((r & 127) >> 3) * PS_SBO + (kc & 3) * PS_LBO + (r & 7) * 16;
    *reinterpret_cast<uint4*>(out + off) = h;
    *reinterpret_cast<uint4*>(out + off + PS_PLANE) = l;
  }
}

int weight_planes_launch(const PlaneTable& tab, cudaStream_t st) {
  if (tab.n <= 0) return DVAE_OK;
  int64_t most = 1;          // 8-element items of the largest matrix: sizes the x extent (smaller entries' extra blocks exit at once)
  for (int i = 0; i < tab.n; ++i) most = max(most, (int64_t)tab.e[i].R * tab.e[i].C / 8);
  int bx = ceil_div(most, 256 * 4);
  bx = bx < 8 ? 8 : (bx > 4 * 148 ? 4 * 148 : bx);
  weight_planes_kernel<<<dim3(bx, 2 * tab.n), 256, 0, st>>>(tab);
  DVAE_LAUNCH_CHECK();
  return DVAE_OK;
}

__global__ void __launch_bounds__(NUM_THREADS, 1)
tc16_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, Params p) {
  extern __shared__ __align__(1024) uint8_t smem[];      // 1024-byte aligned (checked below): TMA 128-byte swizzle atoms
  if (p.skip_flag && *p.skip_flag) return;               // grid-uniform: nothing has been allocated or initialised yet
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + OFF_BAR);
  uint64_t* full = bars;                       // [MAX_STAGES] converters (or bulk copies, pre-split mode) -> MMA
  uint64_t* empty = bars + MAX_STAGES;         // [MAX_STAGES] MMA -> TMA   (tcgen05.commit)
  uint64_t* raw_full = bars + 2 * MAX_STAGES;  // [MAX_STAGES] TMA -> converters (transaction bytes)
  uint64_t* tmem_full = raw_full + MAX_STAGES;   // [2] MMA -> epilogue
  uint64_t* tmem_empty = tmem_full + 2;          // [2] epilogue -> MMA (one arrival per epilogue warp)
  uint64_t* a_full = tmem_empty + 2;             // [1] A-stationary mode: all A k-blocks landed
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(a_full + 1);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // pre-split vocabulary kernels: no converters are needed, so the first 8 converter warps join the epilogue (16 warps,
  // one 32-column chunk each) -- with 8 warps the exp-heavy epilogues took 4-7 us per tile against 1.7 us of MMAs
  const bool wide_epi = p.presplit && p.mode != 0;
  // CTA pair (cluster of 2 along the row blocks, launched only for the A-stationary pre-split kernels): both CTAs walk the
  // same vocabulary tiles, so each fetches HALF of every B stage and multicasts it to both -- half the L2 -> SM traffic
  const uint32_t csize = p.mcast ? cluster_size() : 1, crank = p.mcast ? cluster_rank() : 0;
  const uint16_t cmask = (uint16_t)((1u << csize) - 1);
  const bool conv_as_epi = wide_epi && warp >= PROD_WARP0 && warp < PROD_WARP0 + EPI_WARPS;
  // a programmatically-launched successor (the persistent LSTM kernels) may start its prologue now; it still waits for
  // this grid to complete (griddepcontrol.wait) before it reads anything written here
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  if (tid == 0) DBG16(0);
  if (p.zero_buf) {
    // a buffer some later split-K GEMM accumulates into (e.g. d_h of the vocabulary backward): zeroed here, spread over
    // the grid, instead of by a memset node in front of that GEMM
    float4* z4 = reinterpret_cast<float4*>(p.zero_buf);
    const int64_t nblk = (int64_t)gridDim.x * gridDim.y * gridDim.z;
    const int64_t blk = ((int64_t)blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;
    for (int64_t i = blk * NUM_THREADS + tid; i < p.zero_n4; i += nblk * NUM_THREADS) z4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (p.zero_buf2) {
      float4* y4 = reinterpret_cast<float4*>(p.zero_buf2);
      for (int64_t i = blk * NUM_THREADS + tid; i < p.zero2_n4; i += nblk * NUM_THREADS) y4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
  const int n_tiles = (p.N + BN - 1) / BN;
  const int nkb_total = (p.K + BK - 1) / BK;   // k-blocks per row block of the operand planes (addressing)
  // this CTA's (row tile, column-tile group, k split): the launch grid, or -- live rows -- the launched CTAs re-partitioned
  // over the work the device-side live count leaves.  A CTA without work has cleared its share of zero_buf above and
  // returns here, before barrier init, TMEM allocation or any wait: every CTA decides from the same *m_live, and M = 0
  // (no live row) leaves every CTA idle, i.e. the launch is a no-op apart from the clearing.
  int bx = blockIdx.x, by = blockIdx.y, bz = blockIdx.z, M = p.M, tpc = p.tiles_per_cta, kbps = p.kb_per_split;
  int kb_end = nkb_total;
  int64_t mstride = p.M;                       // mode 1: row stride of the partials
  if (p.m_live) {
    const int live = *p.m_live;
    if (p.live_k) {                            // d_w = P^T . h: K runs over the live positions, split over the launched z
      kb_end = (live + BK - 1) / BK;
      kbps = (kb_end + (int)gridDim.z - 1) / (int)gridDim.z;
      if (bz * kbps >= kb_end) return;
    } else {
      M = live;
      const int rt = (M + BM - 1) / BM;
      const int ctas = gridDim.x * gridDim.y * gridDim.z, c = (blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;
      if (rt == 0) return;
      if (p.mode != 0) {                       // vocabulary groups x tiles per CTA: one wave over the live row tiles
        int groups;
        live_split(rt, ctas, n_tiles, &tpc, &groups);
        if (c >= rt * groups) return;
        bx = c % rt; by = c / rt; bz = 0;
        mstride = (int64_t)rt * BM;
      } else {                                 // d_h: the split-K factor grows as the live row tiles shrink
        const int tiles = rt * gridDim.y;
        int splits = max(1, min(nkb_total, ctas / tiles));
        kbps = (nkb_total + splits - 1) / splits;
        splits = (nkb_total + kbps - 1) / kbps;
        if (c >= tiles * splits) return;
        bx = c % rt; by = (c / rt) % gridDim.y; bz = c / tiles;
      }
    }
  }
  const int m0 = bx * BM;
  const int nt0 = by * tpc;
  const int nt1 = min(n_tiles, nt0 + tpc);
  const int kb0 = bz * kbps;
  const int nkb = max(0, min(kb_end, kb0 + kbps) - kb0);
  const int b_tile0 = p.b_row0 / BN;          // pre-split B planes: first row block of this launch's vocabulary chunk

  if (tid == 0) {
    if (smem_u32(smem) & 1023) {
      printf("dvae tc16_gemm: dynamic shared memory base is not 1024-byte aligned\n");
      __trap();
    }
    for (int s = 0; s < MAX_STAGES; ++s) {
      // one converter group (8 warps) per k-block; hybrid: + the TMA warp's arrive.expect_tx for the bulk-copied B tile
      mbar_init(&full[s], p.presplit ? 1 : PROD_WARPS / 2 + (p.b_presplit ? 1 : 0));
      mbar_init(&empty[s], p.mcast ? csize : 1);       // CTA pair: a B stage is free once BOTH CTAs' MMAs have read it
      mbar_init(&raw_full[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tmem_full[a], 1);
      mbar_init(&tmem_empty[a], wide_epi ? 2 * EPI_WARPS : EPI_WARPS);
    }
    mbar_init(a_full, 2 * EPI_WARPS);         // A-stationary: one arrival per epilogue warp once its share of A is in TMEM
    fence_barrier_init();
  }
  if (warp == TMA_WARP && lane == 0 && !p.presplit) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
  }
  const bool a_stat = p.presplit && !p.no_astat && nkb_total <= AS_MAX_KB && gridDim.z == 1;
  const int nstages = a_stat ? (p.mode == 1 ? AS_STAGES_NOSCRATCH : AS_STAGES) : STAGES;
  const uint32_t stage_bytes = a_stat ? AS_STAGE_BYTES : STAGE_BYTES;
  // (a padding CTA of an odd row-block count in CTA-pair mode re-reads the last real block: it only keeps the protocol going)
  const int a_blk = min(bx, (M + BM - 1) / BM - 1);
  if (warp == MMA_WARP) tmem_alloc(tmem_slot, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  if (p.mcast) cluster_sync_all();      // the peer's mbarriers are initialised before anything of ours can signal them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t smem_u = smem_u32(smem);

  if (warp == TMA_WARP) {
    // ===== TMA producer: raw fp32 k-blocks into the landing ring =====
    if (DVAE_TC16_FLAG(16)) {
      // probes only: no operand traffic at all
    } else if (lane == 0 && a_stat) {
      // only B tiles stream through shared memory (the A rows go to tensor memory: see the epilogue warps' prologue)
      const uint8_t* b_planes = reinterpret_cast<const uint8_t*>(p.b_planes);
      int stage = 0, phase = 0;
      for (int nt = nt0; nt < nt1; ++nt) {
        for (int kb = 0; kb < nkb; kb += AS_KB_PER_STAGE) {
          DVAE_TC16_MARK(nt == nt0 + 1 && kb < 8, 32 + 2 * kb);
          if (!DVAE_TC16_FLAG(8)) mbar_wait(&empty[stage], phase ^ 1);
          else mbar_wait(&full[stage], phase ^ 1);      // probes only: free-running ring (previous fill of the slot has landed)
          DVAE_TC16_MARK(nt == nt0 + 1 && kb < 8, 33 + 2 * kb);
          const uint32_t dst = smem_u + stage * AS_STAGE_BYTES;
          const uint32_t bytes = (uint32_t)min(AS_KB_PER_STAGE, nkb - kb) * PS_TILE;
          mbar_expect_tx(&full[stage], bytes);
          const uint8_t* src = b_planes + ((int64_t)(nt + b_tile0) * nkb_total + kb) * PS_TILE;
          if (csize == 1) {
            bulk_load(dst, src, bytes, &full[stage]);
          } else {              // my share of the stage, to both CTAs; the peer's share lands here through ITS copy
            const uint32_t part = bytes / csize, off = crank * part;
            bulk_load_multicast(dst + off, src + off, part, &full[stage], cmask);
          }
          if (++stage == nstages) { stage = 0; phase ^= 1; }
        }
      }
      if (DVAE_TC16_FLAG(8))                            // probes only: nothing may still be in flight at exit
        for (int s2 = 0; s2 < nstages; ++s2) mbar_wait(&full[s2], s2 < stage ? phase : phase ^ 1);
    } else if (lane == 0 && p.presplit) {
      // operand planes straight into the operand ring: one 16 KB tile k-block [hi, lo] per operand
      const uint8_t* a_tiles = reinterpret_cast<const uint8_t*>(p.a_planes) +
                               ((int64_t)bx * (p.a_kbtot ? p.a_kbtot : nkb_total) + p.a_kb0) * PS_TILE;
      const uint8_t* b_planes = reinterpret_cast<const uint8_t*>(p.b_planes);
      int stage = 0, phase = 0;
      for (int nt = nt0; nt < nt1; ++nt) {
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&empty[stage], phase ^ 1);
          const uint32_t dst = smem_u + stage * STAGE_BYTES;
          mbar_expect_tx(&full[stage], STAGE_BYTES);
          bulk_load(dst, a_tiles + (int64_t)(kb0 + kb) * PS_TILE, PS_TILE, &full[stage]);
          bulk_load(dst + PS_TILE, b_planes + ((int64_t)(nt + b_tile0) * (p.b_kbtot ? p.b_kbtot : nkb_total) + p.b_kb0 + kb0 + kb) * PS_TILE,
                    PS_TILE, &full[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    } else if (lane == 0) {
      // raw fp32 k-blocks [A | B] into the ring stage the MMAs have released
      int stage = 0, phase = 0;
      for (int nt = nt0; nt < nt1; ++nt) {
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&empty[stage], phase ^ 1);
          uint8_t* dst = smem + stage * STAGE_BYTES;
          mbar_expect_tx(&raw_full[stage], p.b_presplit ? RAW_TILE : STAGE_BYTES);
          const int k0 = (kb0 + kb) * BK;
          if (!p.a_mn) tma_load_2d(dst, &tmA, k0, m0, &raw_full[stage]);
          else tma_load_2d(dst, &tmA, m0, k0, &raw_full[stage]);
          if (p.b_presplit) {
            // B is a registered weight: its MMA-ready [hi | lo] tile lands straight in the operand slot and completes on the
            // MMA's own barrier (one more arrival + 16 KB of transaction bytes); the converters only touch A
            mbar_expect_tx(&full[stage], PS_TILE);
            bulk_load(smem_u + stage * STAGE_BYTES + RAW_TILE,
                      reinterpret_cast<const uint8_t*>(p.b_planes) + ((int64_t)(nt + b_tile0) * p.b_kbtot + p.b_kb0 + kb0 + kb) * PS_TILE,
                      PS_TILE, &full[stage]);
          } else if (!p.b_mn) tma_load_2d(dst + RAW_TILE, &tmB, k0, nt * BN, &raw_full[stage]);
          else tma_load_2d(dst + RAW_TILE, &tmB, nt * BN, k0, &raw_full[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp >= PROD_WARP0 && warp < EPI2_WARP0 && !conv_as_epi) {
    // ===== converters: landed fp32 k-block -> (scale, split) -> fp16 operand planes, in place =====
    const int ptid = tid - PROD_WARP0 * 32;
    const float sa = scale_from_amax(p.a_amax, p.a_amax_n, p.a_scale), sb = scale_from_amax(p.b_amax, p.b_amax_n, p.b_scale);
    const int n_items = p.presplit ? 0 : (nt1 - nt0) * nkb;
    // Two groups of 8 warps take alternate k-blocks: one k-block's chain (wait for the landed tile, shared loads, group
    // barrier, split, stores, proxy fence, arrive) is ~0.65 us of latencies for ~100 instructions per thread, and with all
    // 16 warps in lockstep on one k-block that chain, not L2, TMA or the MMAs, set the pace of every converter-path GEMM
    // (0.7 us per k-block whether 16 or 148 SMs were busy).  A thread owns two (row, k chunk) items of each operand.
    const int grp = ptid >> 8, gtid = ptid & 255;
    for (int it = grp; it < n_items; it += 2) {
      const int stage = it % STAGES, phase = (it / STAGES) & 1;
      DVAE_TC16_MARK(ptid == 0 && it == 12, 2);
      mbar_wait(&raw_full[stage], phase);
      DVAE_TC16_MARK(ptid == 0 && it == 12, 3);
      float va0[8], va1[8], vb0[8], vb1[8];
      const uint32_t st = smem_u + stage * STAGE_BYTES;
      load_tile(st, p.a_mn, gtid, va0);
      load_tile(st, p.a_mn, gtid + 256, va1);
      if (!p.b_presplit) {
        load_tile(st + RAW_TILE, p.b_mn, gtid, vb0);
        load_tile(st + RAW_TILE, p.b_mn, gtid + 256, vb1);
      }
      // every thread of the group has its fp32 values in registers before anyone overwrites the tiles with fp16 planes
      asm volatile("bar.sync %0, %1;" ::"r"(CONV_BARRIER + grp), "n"(PROD_WARPS * 16) : "memory");
      store_tile(st, gtid, sa, va0);
      store_tile(st, gtid + 256, sa, va1);
      if (!p.b_presplit) {
        store_tile(st + PS_TILE, gtid, sb, vb0);
        store_tile(st + PS_TILE, gtid + 256, sb, vb1);
      }
      DVAE_TC16_MARK(ptid == 0 && it == 12, 4);
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(&full[stage]);
      DVAE_TC16_MARK(ptid == 0 && it == 12, 5);
    }
  } else if (warp == MMA_WARP) {
    // ===== MMA issuer =====
    // ONE elected thread runs the whole loop, and the loop body is kept to a few dozen instructions: six 128x128x16
    // MMAs are ~390 cycles of tensor-pipe work, and a single thread issues dependent scalar instructions at one per
    // 4-6 cycles -- a 145-instruction body (per-k-block elect/reconverge, descriptor re-derivation, probe marks) made
    // the issuing thread, not the tensor pipe or operand delivery, the limiter (~820 cycles per k-block).
    constexpr uint32_t idesc = (1u << 4) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);   // f16 x f16 -> f32
    if (elect_one() && nkb > 0) {
      if (a_stat) {
        mbar_wait(a_full, 0);
        tc_fence_after();
      }
      // shared-memory descriptor = constant high word | (LBO field | address >> 4): only the 14-bit address field moves
      constexpr uint32_t d_hi = ((PS_SBO >> 4) & 0x3FFF) | (1u << 14);          // SBO, descriptor version, no swizzle
      constexpr uint32_t d_lo = ((PS_LBO >> 4) & 0x3FFF) << 16;
      constexpr uint32_t kstep16 = (2 * PS_LBO) >> 4, plane16 = PS_PLANE >> 4;
      const uint32_t stage16 = stage_bytes >> 4;
      const uint32_t base16 = smem_u >> 4;
      // operand bases: ring stage [A_hi, A_lo, B_hi, B_lo], or stationary A (k-block kb) + ring stage [B_hi, B_lo]
      const uint32_t ring16 = base16;
      const uint32_t b_off16 = a_stat ? 0 : 2 * plane16;
      auto desc = [&](uint32_t addr16) { return ((uint64_t)d_hi << 32) | (uint64_t)(d_lo | (addr16 & 0x3FFF)); };
      int stage = 0, phase = 0;
      uint32_t st16 = ring16;
      for (int tile = 0; tile < nt1 - nt0; ++tile) {
        const int acc = tile & 1;
        if (tile >= 2) {
          mbar_wait(&tmem_empty[acc], ((tile >> 1) - 1) & 1);
          tc_fence_after();
        }
        const uint32_t d1 = tmem_base + (a_stat ? acc * 128 : acc * 256), d2 = d1 + 128;
        if (a_stat) {
          // A from tensor memory (k-block kb = columns 16*kb .. 16*kb+15 of each plane), one accumulator, two k-blocks per stage
          for (int kb = 0; kb < nkb; kb += AS_KB_PER_STAGE) {
            if (!DVAE_TC16_FLAG(4)) mbar_wait(&full[stage], phase);
            if (!DVAE_TC16_FLAG(2)) {
#pragma unroll
              for (int kk = 0; kk < AS_KB_PER_STAGE; ++kk) {
                if (kb + kk < nkb) {
                  const uint32_t ta = tmem_base + (uint32_t)(kb + kk) * 16, sb16 = st16 + kk * (PS_TILE >> 4);
#pragma unroll
                  for (int k = 0; k < BK / 16; ++k) {
                    const uint32_t adv = k * kstep16;
                    mma_f16_ts(d1, ta + AS_T_AHI + 8 * k, desc(sb16 + adv), idesc, (kb | kk | k) ? 1u : 0u);
                    mma_f16_ts(d1, ta + AS_T_AHI + 8 * k, desc(sb16 + plane16 + adv), idesc, 1u);
                    mma_f16_ts(d1, ta + AS_T_ALO + 8 * k, desc(sb16 + adv), idesc, 1u);
                  }
                }
              }
            }
            if (!DVAE_TC16_FLAG(8)) {
              if (csize == 1) tc_commit(&empty[stage]);
              else tc_commit_multicast(&empty[stage], cmask);
            }
            st16 += stage16;
            if (++stage == nstages) { stage = 0; phase ^= 1; st16 = ring16; }
          }
          tc_commit(&tmem_full[acc]);
          continue;
        }
        for (int kb = 0; kb < nkb; ++kb) {
          DVAE_TC16_MARK(tile == 1 && kb < 8, 48 + 2 * kb);
          // no tcgen05.fence here: the operands arrive through the async proxy (TMA) or behind the converters'
          // fence.proxy.async, and the mbarrier wait orders them
          if (!DVAE_TC16_FLAG(4)) mbar_wait(&full[stage], phase);
          DVAE_TC16_MARK(tile == 1 && kb < 8, 49 + 2 * kb);
          const uint32_t sa16 = st16, sb16 = st16 + b_off16;
          if (!DVAE_TC16_FLAG(2)) {
#pragma unroll
            for (int k = 0; k < BK / 16; ++k) {
              const uint32_t adv = k * kstep16;
              const uint32_t accum = (kb | k) ? 1u : 0u;
              mma_f16(d1, desc(sa16 + adv), desc(sb16 + adv), idesc, accum);
              mma_f16(d2, desc(sa16 + adv), desc(sb16 + plane16 + adv), idesc, accum);
              mma_f16(d2, desc(sa16 + plane16 + adv), desc(sb16 + adv), idesc, 1u);
            }
          }
          if (!DVAE_TC16_FLAG(8)) {
            if (csize == 1) tc_commit(&empty[stage]);
            else tc_commit_multicast(&empty[stage], cmask);
          }
          st16 += stage16;
          if (++stage == nstages) { stage = 0; phase ^= 1; st16 = ring16; }
        }
        tc_commit(&tmem_full[acc]);
      }
    }
    __syncwarp();
  } else {
    // ===== epilogue: 8 warps = 4 TMEM lane quarters x 2 column halves of the tile =====
    // default: warps 0-3 own column chunks {0,1}, warps 22-25 chunks {2,3}.  wide (16 warps): one chunk per warp --
    // warps 0-3 chunk 0, 6-9 chunk 1, 22-25 chunk 2, 10-13 chunk 3 (any 4 consecutive warps cover the 4 TMEM lane quarters)
    const int quarter = warp & 3, ehalf = warp >= EPI2_WARP0 ? 1 : 0;
    const int c_lo = !wide_epi ? 2 * ehalf : (conv_as_epi ? 1 + 2 * ((warp - PROD_WARP0) >> 2) : 2 * ehalf);
    const int c_hi = wide_epi ? c_lo + 1 : c_lo + 2;
    const int ew = wide_epi ? c_lo * 4 + quarter : ehalf * 4 + quarter;      // 0..15 | 0..7
    const int row = m0 + quarter * 32 + lane;      // output row owned by this thread (TMEM lane)
    const bool row_ok = row < M;
    // c_row_scale: per-output-row factor (the A planes of that row were scaled by its inverse, e.g. per-row power-of-two
    // scaling of LSTM gate gradients); applied here, before the transpose, where a thread still owns one row
    const float oscale = p.alpha * (p.alpha_dev ? *p.alpha_dev : 1.f) * ((p.c_row_scale && row_ok) ? __ldg(p.c_row_scale + row) : 1.f) /
                         (scale_from_amax(p.a_amax, p.a_amax_n, p.a_scale) * scale_from_amax(p.b_amax, p.b_amax_n, p.b_scale));
    // per-row state of the fused vocabulary epilogues
    float rm = -INFINITY, rs = 0.f, rt = 0.f, rav = -INFINITY, row_lse = 0.f, row_nlse2 = 0.f, row_scale = 0.f;
    int rai = 0x7fffffff, tgt = -1;
    if (p.mode != 0 && row_ok) {
      const int n = p.row_map ? __ldg(p.row_map + row) : row;      // decoder position of this row
      const int b = n % p.B, tpos = n / p.B + 1;
      if (p.targets) tgt = (int)p.targets[(int64_t)b * p.tgt_stride_b + tpos];
      if (p.mode == 2) {
        row_lse = p.lse[n];
        row_nlse2 = -row_lse * kLog2e;
        row_scale = (tpos < p.lengths[b]) ? (p.grad_scale ? p.grad_scale[0] : 1.f) / (float)p.B : 0.f;
        tgt -= p.v0;
      }
    }
    if (a_stat) {
      // the CTA's A rows -> tensor memory, once: this thread owns row quarter*32 + lane (= its TMEM lane) and, with the
      // three other warps of its lane quarter, the k-blocks {2*c_lo, 2*c_lo + 1}; a 16-byte chunk of a plane (8 fp16 of K)
      // is four 32-bit TMEM columns, a k-block sixteen
      const uint8_t* a_tiles = reinterpret_cast<const uint8_t*>(p.a_planes) + (int64_t)a_blk * nkb_total * PS_TILE;
      const int r = quarter * 32 + lane;
      const uint32_t roff = (uint32_t)(r >> 3) * PS_SBO + (r & 7) * 16;
      const uint32_t tlane = tmem_base + ((uint32_t)(quarter * 32) << 16);
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const int kb = 2 * c_lo + i;
        if (kb < nkb) {
          const uint8_t* t = a_tiles + (int64_t)kb * PS_TILE + roff;
#pragma unroll
          for (int pl = 0; pl < 2; ++pl) {
            uint32_t v[16];
#pragma unroll
            for (int kc = 0; kc < 4; ++kc) {
              const uint4 q = __ldg(reinterpret_cast<const uint4*>(t + pl * PS_PLANE + kc * PS_LBO));
              v[4 * kc] = q.x; v[4 * kc + 1] = q.y; v[4 * kc + 2] = q.z; v[4 * kc + 3] = q.w;
            }
            tmem_st16(tlane + (pl ? AS_T_ALO : AS_T_AHI) + kb * 16, v);
          }
        }
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(a_full);
    }
    float bias_next[2] = {0.f, 0.f};      // this warp's bias values of the next tile (vocabulary modes)
    if (p.mode != 0 && nkb > 0) {
#pragma unroll
      for (int h2 = 0; h2 < 2; ++h2) {
        const int col = nt0 * BN + (c_lo + h2) * 32 + lane;
        bias_next[h2] = (nt0 < nt1 && h2 < c_hi - c_lo && col < p.N) ? __ldg(p.bias + col) : 0.f;
      }
    }
    int tile = 0;
    for (int nt = nt0; nt < nt1 && nkb > 0; ++nt, ++tile) {
      const int n0 = nt * BN, acc = tile & 1;
      mbar_wait(&tmem_full[acc], (tile >> 1) & 1);
      tc_fence_after();
      if (tid == 0 && tile < 4) DBG16(14 + 2 * tile);
      DVAE_TC16_MARK(tid == 0 && tile == 2, 96);
      // this warp's 64 bias values (vocabulary modes) -> shared memory: broadcast reads instead of 64 global loads
      float* sbias = reinterpret_cast<float*>(smem + OFF_BIAS) + (wide_epi ? ew * 32 : ew * 64);
      const uint32_t sbias_u = smem_u + OFF_BIAS + (wide_epi ? ew * 32 : ew * 64) * 4;
      if (p.mode != 0) {
        __syncwarp();
#pragma unroll
        for (int h2 = 0; h2 < 2; ++h2)
          if (h2 < c_hi - c_lo) sbias[h2 * 32 + lane] = bias_next[h2];
        __syncwarp();
        // the next tile's bias values are fetched now: their global-load latency hides behind this tile's epilogue
#pragma unroll
        for (int h2 = 0; h2 < 2; ++h2) {
          const int col = n0 + BN + (c_lo + h2) * 32 + lane;
          bias_next[h2] = (nt + 1 < nt1 && h2 < c_hi - c_lo && col < p.N) ? __ldg(p.bias + col) : 0.f;
        }
      }
      DVAE_TC16_MARK(tid == 0 && tile == 2, 97);
#pragma unroll 1
      for (int c = c_lo; c < c_hi; ++c) {
        const int col0 = n0 + c * 32;
        if (col0 >= p.N || DVAE_TC16_FLAG(~0)) continue;                        // warp-uniform (probe builds: any switch skips the epilogue)
        const uint32_t ta = tmem_base + ((uint32_t)(quarter * 32) << 16) + (a_stat ? acc * 128 : acc * 256) + c * 32;
        if (p.mode == 2 && wide_epi) {
          // softmax-gradient chunk with 16 epilogue warps: 2 KB of transpose scratch per warp, so the chunk goes out in two
          // [32 rows x 16 cols] halves; element (r, j) of a half lives at word r * 16 + (j ^ ((r >> 1) & 15)) and store
          // instruction k writes rows 2k, 2k+1 (lanes 0-15 / 16-31): two full 64-byte segments, no bank conflicts either way
          const uint32_t sc = smem_u + OFF_SCRATCH + ew * (32 * 16 * 4);
          const int r0 = m0 + quarter * 32;
          const int nr = min(32, M - r0);
          const bool dead = row_scale == 0.f;
          DVAE_TC16_MARK(tid == 0 && tile == 2, 104);
#pragma unroll
          for (int hh = 0; hh < 2; ++hh) {
#pragma unroll
            for (int h8 = 0; h8 < 2; ++h8) {            // 8 columns at a time: 72 registers per thread is the cap here
              float v[8], w[8];
              if (a_stat) {        // single accumulator: the lo products are already in it
                tmem_ld8_pair(ta + hh * 16 + h8 * 8, ta + hh * 16 + h8 * 8, v, w);
#pragma unroll
                for (int j = 0; j < 8; ++j) w[j] = 0.f;
              } else {
                tmem_ld8_pair(ta + hh * 16 + h8 * 8, ta + 128 + hh * 16 + h8 * 8, v, w);
              }
#pragma unroll
              for (int q = 0; q < 2; ++q) {
                const uint4 t = lds128(sbias_u + (hh * 16 + h8 * 8 + 4 * q) * 4);
                const float bq[4] = {__uint_as_float(t.x), __uint_as_float(t.y), __uint_as_float(t.z), __uint_as_float(t.w)};
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) {
                  const int j = 4 * q + jj, col = col0 + hh * 16 + h8 * 8 + j;
                  const float e = ex2_ftz(fmaf(fmaf(fmaf(w[j], kLoInv, v[j]), oscale, bq[jj]), kLog2e, row_nlse2));
                  v[j] = (dead || col >= p.N) ? 0.f : (e - (col == tgt ? 1.f : 0.f)) * row_scale;
                }
              }
              // planes output: this thread's 8 columns of its row are one 16-byte chunk of each K-major plane of P (the A
              // operand of d_h = P . W); padding rows / columns carry zeros
              // (a tile reaches past the planes' last k-block when N is not a multiple of 128: those chunks do not exist)
              // (nor do the rows of a CTA pair's padding row block)
              if (p.p_planes_a && col0 + hh * 16 + h8 * 8 < p.p_kb_a * BK && m0 < (M + BM - 1) / BM * BM)
                store_plane_chunk(p.p_planes_a, row, col0 + hh * 16 + h8 * 8, p.p_kb_a, v, p.p_scale);
#pragma unroll
              for (int j = 0; j < 8; ++j) sts32(sc + (lane * 16 + ((h8 * 8 + j) ^ ((lane >> 1) & 15))) * 4, v[j]);
            }
            __syncwarp();
            if (p.p_planes_t) {
              // transposed planes (rows = vocabulary ids, K = decoder positions: the A operand of d_w = P^T . h): after the
              // transpose through shared memory a thread holds 16 consecutive rows of one column = two 16-byte chunks per
              // plane; their sum, folded over the two row halves, is this warp's share of the bias gradient
              const int cc = lane & 15, rg = lane >> 4, colw = col0 + hh * 16 + cc;
              float tv[16], ssum = 0.f;
#pragma unroll
              for (int k = 0; k < 16; ++k) {
                const int r = rg * 16 + k;
                tv[k] = lds32(sc + (r * 16 + (cc ^ ((r >> 1) & 15))) * 4);
                ssum += tv[k];
              }
              ssum += __shfl_xor_sync(0xffffffffu, ssum, 16);
              if (colw < p.N) {
                if (rg == 0 && p.p_colsum) atomicAdd(p.p_colsum + colw, ssum);
                const float lo8[8] = {tv[0], tv[1], tv[2], tv[3], tv[4], tv[5], tv[6], tv[7]};
                const float hi8[8] = {tv[8], tv[9], tv[10], tv[11], tv[12], tv[13], tv[14], tv[15]};
                if (r0 + rg * 16 < p.p_kb_t * BK) store_plane_chunk(p.p_planes_t, colw, r0 + rg * 16, p.p_kb_t, lo8, p.p_scale);
                if (r0 + rg * 16 + 8 < p.p_kb_t * BK) store_plane_chunk(p.p_planes_t, colw, r0 + rg * 16 + 8, p.p_kb_t, hi8, p.p_scale);
              }
              __syncwarp();
              continue;
            }
            const int colw = col0 + hh * 16 + (lane & 15);
            float* cp = p.C + (int64_t)(r0 + (lane >> 4)) * p.ldc + colw;
            if (colw < p.N) {
#pragma unroll
              for (int k = 0; k < 16; ++k) {
                const float val = lds32(sc + ((2 * k + (lane >> 4)) * 16 + ((lane & 15) ^ k)) * 4);
                if (2 * k + (lane >> 4) < nr) cp[(int64_t)(2 * k) * p.ldc] = val;
              }
            }
            __syncwarp();
          }
          DVAE_TC16_MARK(tid == 0 && tile == 2, 105);
          continue;
        }
        if (p.mode != 1) {
          // modes 0 / 2 store a [32 rows x 32 cols] chunk: transpose it through padded shared memory so each
          // store instruction covers 32 consecutive columns of one row (coalesced) instead of 32 different rows
          // (element (r, c) of the chunk lives at word r * 32 + (c ^ r): conflict-free both ways without padding)
          const uint32_t sc = smem_u + OFF_SCRATCH + ew * (32 * 32 * 4);
          DVAE_TC16_MARK(tid == 0 && tile == 2, 104 + 3 * (c - c_lo));
#pragma unroll
          for (int hh = 0; hh < 2; ++hh) {
            float v[16], w[16];
            tmem_ld16_pair(ta + hh * 16, ta + 128 + hh * 16, v, w);
            float x[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) x[j] = fmaf(w[j], kLoInv, v[j]) * oscale;
            if (p.mode == 2) {
              // all 16 bias values first (4 x LDS.128), then 16 independent exp chains, then the stores: a shared load
              // per element between the (volatile) stores serialised the whole block (~100 cycles per element)
              float bv[16];
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                const uint4 t = lds128(sbias_u + ((c - c_lo) * 32 + hh * 16 + 4 * q) * 4);
                bv[4 * q] = __uint_as_float(t.x); bv[4 * q + 1] = __uint_as_float(t.y);
                bv[4 * q + 2] = __uint_as_float(t.z); bv[4 * q + 3] = __uint_as_float(t.w);
              }
              const bool dead = row_scale == 0.f;
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                const int col = col0 + hh * 16 + j;
                const float e = ex2_ftz(fmaf(x[j] + bv[j], kLog2e, row_nlse2));
                x[j] = (dead || col >= p.N) ? 0.f : (e - (col == tgt ? 1.f : 0.f)) * row_scale;
              }
            }
#pragma unroll
            for (int j = 0; j < 16; ++j) sts32(sc + (lane * 32 + ((hh * 16 + j) ^ lane)) * 4, x[j]);
          }
          DVAE_TC16_MARK(tid == 0 && tile == 2, 105 + 3 * (c - c_lo));
          __syncwarp();
          const int col = col0 + lane;
          const int r0 = m0 + quarter * 32;
          const int nr = min(32, M - r0);                // valid rows of this warp's 32-row band
          if (col < p.N && nr > 0) {
            const bool split = gridDim.z > 1 || p.atomic_out;
            float badd = 0.f;
            if (p.mode == 0 && (!split || bz == 0)) {
              if (p.bias) badd += __ldg(p.bias + col);
              if (p.bias2) badd += __ldg(p.bias2 + col);
            }
            float* cp = p.C + (int64_t)r0 * p.ldc + col;
            const int64_t ldc = p.ldc;
            auto chunk_at = [&](int rr) { return lds32(sc + (uint32_t)(rr * 32 + (lane ^ rr)) * 4); };      // element (rr, lane)
            if (p.mode == 2 || (!split && p.act == 0 && p.beta == 0.f)) {
              if (nr == 32) {
#pragma unroll
                for (int rr = 0; rr < 32; ++rr) cp[rr * ldc] = chunk_at(rr) + badd;
              } else {
                for (int rr = 0; rr < nr; ++rr) cp[rr * ldc] = chunk_at(rr) + badd;
              }
            } else if (split && p.row_map) {    // live rows: row k of this GEMM is row row_map[k] of C
              for (int rr = 0; rr < nr; ++rr) atomicAdd(p.C + (int64_t)__ldg(p.row_map + r0 + rr) * ldc + col, chunk_at(rr) + badd);
            } else if (split) {
              for (int rr = 0; rr < nr; ++rr) atomicAdd(cp + rr * ldc, chunk_at(rr) + badd);   // C pre-scaled by beta
            } else {
              const float beta = p.beta;
              const bool do_tanh = p.act == 1;
              if (nr == 32 && beta != 0.f) {
                // read-modify-write of C: all 32 loads in flight before the first dependent store
#pragma unroll 1
                for (int r8 = 0; r8 < 32; r8 += 8) {
                  float old[8];
#pragma unroll
                  for (int rr = 0; rr < 8; ++rr) old[rr] = cp[(r8 + rr) * ldc];
#pragma unroll
                  for (int rr = 0; rr < 8; ++rr) {
                    float x = chunk_at(r8 + rr) + badd;
                    if (do_tanh) x = tanhf(x);
                    cp[(r8 + rr) * ldc] = fmaf(beta, old[rr], x);
                  }
                }
              } else {
                for (int rr = 0; rr < nr; ++rr) {
                  float x = chunk_at(rr) + badd;
                  if (do_tanh) x = tanhf(x);
                  if (beta != 0.f) x = fmaf(beta, cp[rr * ldc], x);
                  cp[rr * ldc] = x;
                }
              }
            }
          }
          DVAE_TC16_MARK(tid == 0 && tile == 2, 106 + 3 * (c - c_lo));
          __syncwarp();
          continue;
        }
        // mode 1: online log-softmax statistics of this row over the tile's columns (logits never leave registers)
        const bool sample = p.gumbel_seed != nullptr;
        const uint64_t gseed = sample ? *p.gumbel_seed : 0;
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          float v[16], w[16];
          DVAE_TC16_MARK(tid == 0 && tile == 2, 98 + 3 * hh);
          if (a_stat) {          // single accumulator: the lo products are already in it
            tmem_ld16(ta + hh * 16, v);
#pragma unroll
            for (int j = 0; j < 16; ++j) w[j] = 0.f;
          } else {
            tmem_ld16_pair(ta + hh * 16, ta + 128 + hh * 16, v, w);
          }
          DVAE_TC16_MARK(tid == 0 && tile == 2, 99 + 3 * hh);
          if (!row_ok) continue;
          // 16 logits of this row: everything below is a tree or independent per element (the serial running-max /
          // arg-max / sum chains of the obvious loop made this epilogue, not the MMAs, the kernel's critical path)
          const int base = col0 + hh * 16;
          float x[16], xs[16];
          {
            // bias: four 16-byte shared loads (explicit shared-space: through the generic `sbias` pointer these were
            // sixteen predicated generic LD.E, each feeding its own FFMA)
            const uint32_t ba = sbias_u + ((c - c_lo) * 32 + hh * 16) * 4;
            float bv[16];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const uint4 t = lds128(ba + q * 16);
              bv[4 * q] = __uint_as_float(t.x); bv[4 * q + 1] = __uint_as_float(t.y);
              bv[4 * q + 2] = __uint_as_float(t.z); bv[4 * q + 3] = __uint_as_float(t.w);
            }
#pragma unroll
            for (int j = 0; j < 16; ++j) x[j] = fmaf(fmaf(w[j], kLoInv, v[j]), oscale, bv[j]);
            if (base + 16 > p.N) {                           // last, partial vocabulary tile only (warp-uniform)
#pragma unroll
              for (int j = 0; j < 16; ++j)
                if (base + j >= p.N) x[j] = -INFINITY;
            }
          }
          if (sample) {
#pragma unroll
            for (int j4 = 0; j4 < 16; j4 += 4) {
              float g[4];
              gumbel4(gseed, p.gumbel_salt, row, base + j4, (p.N + 3) >> 2, g);
#pragma unroll
              for (int jj = 0; jj < 4; ++jj) xs[j4 + jj] = x[j4 + jj] + g[jj];
            }
          } else {
#pragma unroll
            for (int j = 0; j < 16; ++j) xs[j] = x[j];
          }
          float m8[8], m4[4];
#pragma unroll
          for (int j = 0; j < 8; ++j) m8[j] = fmaxf(xs[2 * j], xs[2 * j + 1]);
#pragma unroll
          for (int j = 0; j < 4; ++j) m4[j] = fmaxf(m8[2 * j], m8[2 * j + 1]);
          const float smax = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));       // max of the (noisy) scores
          if (smax > rav) {                                  // columns ascend: ties keep the earlier index
            unsigned eq = 0;
#pragma unroll
            for (int j = 0; j < 16; ++j) eq |= (xs[j] == smax ? 1u : 0u) << j;
            rav = smax;
            rai = base + __ffs(eq) - 1;
          }
          if (tgt >= base && tgt < base + 16) {
#pragma unroll
            for (int j = 0; j < 16; ++j)
              if (base + j == tgt) rt = x[j];
          }
          float tmax = smax;
          if (sample) {                                      // the softmax statistics use the noise-free logits
#pragma unroll
            for (int j = 0; j < 8; ++j) m8[j] = fmaxf(x[2 * j], x[2 * j + 1]);
#pragma unroll
            for (int j = 0; j < 4; ++j) m4[j] = fmaxf(m8[2 * j], m8[2 * j + 1]);
            tmax = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
          }
          if (tmax > rm) { rs *= ex2_ftz((rm - tmax) * kLog2e); rm = tmax; }
          const float nrm2 = -rm * kLog2e;
          float e8[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) e8[j] = ex2_ftz(fmaf(x[2 * j], kLog2e, nrm2)) + ex2_ftz(fmaf(x[2 * j + 1], kLog2e, nrm2));
          rs += ((e8[0] + e8[1]) + (e8[2] + e8[3])) + ((e8[4] + e8[5]) + (e8[6] + e8[7]));
          DVAE_TC16_MARK(tid == 0 && tile == 2, 100 + 3 * hh);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[acc]);
      if (tid == 0 && tile < 4) DBG16(15 + 2 * tile);
    }
    if (p.mode == 1 && row_ok) {      // every epilogue warp set is a separate vocabulary split for the finalize kernel
      const int64_t sp = wide_epi ? (int64_t)by * 4 + c_lo : (int64_t)by * 2 + ehalf;
      *reinterpret_cast<float4*>(p.part + (sp * mstride + row) * 4) = make_float4(rm, rs, rt, rav);
      p.part_idx[sp * mstride + row] = rai;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (p.mcast) cluster_sync_all();      // nobody leaves while the peer may still multicast into this CTA or signal its barriers
  if (warp == MMA_WARP) tmem_dealloc(tmem_base, TMEM_COLS);
  if (tid == 0) DBG16(1);
}

// ---- host ------------------------------------------------------------------------------------------
bool supported(const float* A, int64_t lda, int trans_a, const float* B, int64_t ldb, int trans_b, int M, int N, int K) {
  return enabled() && shape_ok(A, lda, trans_a, B, ldb, trans_b, M, N, K);
}

bool enabled() {
  // default; DVAE_GEMM_IMPL=tf32 keeps the 3xTF32 kernel (tc_gemm.cu) for A/B runs, =simt the fp32 SIMT kernels
  const char* e = getenv("DVAE_GEMM_IMPL");
  return !(e && (e[0] == 't' || e[0] == 's'));
}

bool shape_ok(const float* A, int64_t lda, int trans_a, const float* B, int64_t ldb, int trans_b, int M, int N, int K) {
  // TMA: 16-byte aligned bases and row strides
  if (((reinterpret_cast<uintptr_t>(A) | reinterpret_cast<uintptr_t>(B)) & 15) || lda % 4 || ldb % 4) return false;
  return M >= 1 && N >= 1 && K >= 1;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* q = nullptr;
    cudaDriverEntryPointQueryResult r;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &q, cudaEnableDefault, &r) == cudaSuccess && r == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(q);
  }
  return fn;
}
// un-swizzled 2-D fp32 map over a row-major [outer, inner] matrix with row stride ld: K-major operands land as
// [128 rows][32 k] (box 32 x 128), MN-major ones as [32 k][128 rows] (box 128 x 32)
static int make_map(CUtensorMap* m, const float* base, int64_t ld, int mn_major, int rows, int K) {
  EncodeTiledFn fn = encode_fn();
  DVAE_REQUIRE(fn != nullptr, "tc16_gemm: cuTensorMapEncodeTiled is not available from the driver");
  cuuint64_t dims[2] = {(cuuint64_t)(mn_major ? rows : K), (cuuint64_t)(mn_major ? K : rows)};
  cuuint64_t strides[1] = {(cuuint64_t)ld * sizeof(float)};
  cuuint32_t box[2] = {(cuuint32_t)(mn_major ? BM : BK), (cuuint32_t)(mn_major ? BK : BM)};
  cuuint32_t estr[2] = {1, 1};
  // K-major tiles (128-byte rows) land with the 128-byte swizzle the converters' loads expect (load_tile)
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, mn_major ? CU_TENSOR_MAP_SWIZZLE_NONE : CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  DVAE_REQUIRE(r == CUDA_SUCCESS, "tc16_gemm: cuTensorMapEncodeTiled failed (%d) rows=%d K=%d ld=%lld", (int)r, rows, K, (long long)ld);
  return DVAE_OK;
}

// 3-D map over one fp16 plane in the blocked layout of split_planes: dim0 = one core matrix (64 elements, 128 B),
// dim1 = k chunks, dim2 = 8-row groups; a box of 64 x 4 x 16 is a dense UMMA-ready 128 x 32 operand tile
// floats occupied by both fp16 planes of X [R, K] in the tile-blocked layout (R padded to 128, K to 32)
int64_t plane_floats(int R, int K) { return (int64_t)ceil_div(R, BM) * BM * ceil_div(K, BK) * BK; }

bool presplit_enabled() {
  const char* e = getenv("DVAE_VOCAB_PRESPLIT");
  return !(e && e[0] == '0');
}

// planes of the single-accumulator (A-stationary) kernels: operand scale 2^8, lo unscaled; else scale as given, lo * 2^11
bool single_acc_planes(int K) { return ceil_div(K, BK) <= AS_MAX_KB; }

int split_planes(const float* X, int64_t ld, int R, int K, float scale, void* planes, cudaStream_t st, bool force_dual) {
  const bool single = !force_dual && single_acc_planes(K);
  const float lo_scale = single ? 1.f : kLoScale;
  if (single) scale *= kSingleScale;
  DVAE_REQUIRE(X && planes && R > 0 && K > 0, "tc16 split_planes: bad argument");
  const int64_t work = (int64_t)ceil_div(R, BM) * BM * ceil_div(K, BK) * (BK / 8);
  int blocks = ceil_div(work, 256);
  if (blocks > 148 * 8) blocks = 148 * 8;
  split_planes_kernel<<<blocks, 256, 0, st>>>(X, ld, R, K, scale, lo_scale, reinterpret_cast<uint8_t*>(planes));
  DVAE_LAUNCH_CHECK();
  return DVAE_OK;
}

static int launch(const Params& p_in, dim3 grid, cudaStream_t st) {
  Params p = p_in;
  if (p.dbg)      // probes: DVAE_TC_DBG_MODE=<mode> keeps the timeline marks of that kernel flavour only
    if (const char* e = getenv("DVAE_TC_DBG_MODE"))
      if (atoi(e) != p.mode) p.dbg = nullptr;
  static bool ready = false;
  if (!ready) {
    DVAE_CUDA(cudaFuncSetAttribute(tc16_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    ready = true;
  }
  CUtensorMap ma, mb;
  int rc;
  if (p.presplit) {          // tile-blocked fp16 planes are fetched with plain bulk copies: no tensor maps
    memset(&ma, 0, sizeof(ma));
    memset(&mb, 0, sizeof(mb));
  } else {
    if ((rc = make_map(&ma, p.A, p.lda, p.a_mn, p.M, p.K))) return rc;
    if (p.b_presplit) memset(&mb, 0, sizeof(mb));
    else if ((rc = make_map(&mb, p.Bm, p.ldb, p.b_mn, p.N, p.K))) return rc;
  }
  // A-stationary pre-split kernels (vocabulary forward / softmax gradient), opt-in with DVAE_TC16_MCAST=1: CTA pairs along
  // the row blocks share their B tiles by multicast (an odd row-block count gets one padding CTA).  Measured at cfg 2:
  // correct, but no faster (tile period 3.0 vs 3.1 us, whole forward call 82.7 vs 79.7 us): the B ring is bound by the
  // ~1.3 us latency of a 16 KB fetch against 6 stages, not by L2 -> SM bytes, and the pair runs at the pace of its slower CTA.
  const char* mc_env = getenv("DVAE_TC16_MCAST");
  const bool mcast_on = mc_env && mc_env[0] == '1';
  if (mcast_on && p.presplit && ceil_div(p.K, BK) <= AS_MAX_KB && grid.z == 1 && grid.x >= 2 && !p.m_live) {
    p.mcast = 1;
    grid.x = (grid.x + 1) / 2 * 2;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = dim3(NUM_THREADS); cfg.dynamicSmemBytes = SMEM_BYTES; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    DVAE_CUDA(cudaLaunchKernelEx(&cfg, tc16_gemm_kernel, ma, mb, p));
    DVAE_LAUNCH_CHECK();
    return DVAE_OK;
  }
  tc16_gemm_kernel<<<grid, NUM_THREADS, SMEM_BYTES, st>>>(ma, mb, p);
  DVAE_LAUNCH_CHECK();
  return DVAE_OK;
}

__global__ void tc16_scale_rows_kernel(float* C, int64_t ldc, int M, int N, float beta) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)M * N) return;
  float* c = C + (i / N) * ldc + (i % N);
  *c = beta == 0.f ? 0.f : *c * beta;
}

static void apply_hints(Params& p, const GemmHints& h) {
  if (const char* e = getenv("DVAE_TC_DBG")) p.dbg = reinterpret_cast<unsigned long long*>(strtoull(e, nullptr, 0));
  if (const char* e = getenv("DVAE_TC_SKIP_EPILOGUE")) p.dbg_skip_epilogue = atoi(e);     // probes only: main-loop speed in isolation
  p.a_amax = h.a_amax_bits; p.b_amax = h.b_amax_bits; p.a_amax_n = h.a_amax_n; p.b_amax_n = h.b_amax_n;
  p.a_scale = h.a_scale; p.b_scale = h.b_scale;
  p.alpha = 1.f; p.alpha_dev = nullptr;
  p.atomic_out = h.atomic_out ? 1 : 0;
}

int linear(const float* A, int64_t lda, int trans_a, const float* B, int64_t ldb, int trans_b, float* C, int64_t ldc, int M,
           int N, int K, const float* bias, const float* bias2, float beta, int act, const GemmHints& hints, cudaStream_t st) {
  Params p = {};
  p.A = A; p.lda = lda; p.Bm = B; p.ldb = ldb;
  p.M = M; p.N = N; p.K = K; p.a_mn = trans_a ? 1 : 0; p.b_mn = trans_b ? 1 : 0; p.tiles_per_cta = 1;
  p.C = C; p.ldc = ldc; p.bias = bias; p.bias2 = bias2; p.beta = beta; p.act = act; p.mode = 0;
  apply_hints(p, hints);
  PlaneHit hit;
  if (hints.b_planes) {
    p.b_presplit = 1; p.b_planes = hints.b_planes; p.b_row0 = hints.b_tile0 * BN; p.b_kb0 = hints.b_kb0; p.b_kbtot = hints.b_kbtot;
  } else if (!hints.b_amax_bits && hints.b_scale == 1.f && find_weight_planes(B, ldb, trans_b, N, K, &hit)) {
    p.b_presplit = 1; p.b_planes = hit.planes; p.b_row0 = hit.tile0 * BN; p.b_kb0 = hit.kb0; p.b_kbtot = hit.kbtot;
  }
  // split-K (weight-gradient shapes: few output tiles, deep K): pick the split count with the smallest modelled time
  //   waves(tiles * s) * (k-blocks per split * t_kb + fixed per-CTA cost)   [us; measured orders of magnitude]
  // -- "split only when tiles <= 74" left the 80-tile dW_out GEMM of a 5120-column vocabulary chunk at one 84-k-block
  // CTA per tile on 80 of 148 SMs (128 us instead of ~60).
  const int tiles = ceil_div(M, BM) * ceil_div(N, BN), nkb = ceil_div(K, BK);
  int splits = 1;
  if (act == 0 && nkb >= 16) {
    const float t_kb = p.b_presplit ? 0.33f + 0.15f * p.a_mn : 0.5f + 0.2f * (p.a_mn + p.b_mn);
    float best = 1e30f;
    for (int s2 = 1; s2 <= 16 && s2 <= nkb / 4; ++s2) {
      const int kbs = ceil_div(nkb, s2), se = ceil_div(nkb, kbs);
      if (se != s2) continue;
      if (hints.max_ctas > 0 && s2 > 1 && tiles * se > hints.max_ctas) break;
      const int waves = ceil_div(tiles * se, 148);
      const float t = waves * (kbs * t_kb + (se > 1 ? 6.f : 4.f)) + (se > 1 ? 2.f : 0.f);
      if (t < best * 0.95f) { best = t; splits = se; }      // a larger split count has to be clearly better
    }
  }
  if (const char* e = getenv("DVAE_TC16_SPLITS_BIG_MN"))          // A/B knob: split count of the large both-transposed GEMMs (dW_out)
    if (p.a_mn && p.b_mn && tiles >= 64 && act == 0) splits = atoi(e);
  p.kb_per_split = ceil_div(nkb, splits);
  splits = ceil_div(nkb, p.kb_per_split);
  if (splits > 1 && beta != 1.f && !(beta == 0.f && hints.c_zeroed)) {
    if (beta == 0.f && ldc == N) {
      DVAE_CUDA(cudaMemsetAsync(C, 0, sizeof(float) * (size_t)M * N, st));
    } else {
      tc16_scale_rows_kernel<<<ceil_div((int64_t)M * N, 256), 256, 0, st>>>(C, ldc, M, N, beta);
      DVAE_LAUNCH_CHECK();
    }
  }
  // more tiles than SMs: a run of N tiles per CTA, so that the next tile's main loop hides this one's epilogue and the
  // grid (times the sibling GEMMs the caller runs concurrently, e.g. the two directions' input projections) is one wave
  const int conc = hints.concurrency > 1 ? hints.concurrency : 1;
  const int sm_budget = hints.max_ctas > 0 ? hints.max_ctas : 148;
  if (splits == 1 && tiles * conc > sm_budget && ceil_div(N, BN) >= 2) {
    int tpc = ceil_div(tiles * conc, sm_budget);
    if (tpc < 2) tpc = 2;
    if (tpc > ceil_div(N, BN)) tpc = ceil_div(N, BN);
    p.tiles_per_cta = tpc;
  }
  return launch(p, dim3(ceil_div(M, BM), ceil_div(ceil_div(N, BN), p.tiles_per_cta), splits), st);
}

// C[M,N] = act(A . B^T + bias) + beta * C with BOTH operands given as tile-blocked fp16 planes (dual-accumulator convention,
// see tc_planes.cuh): no tensor maps, no landing ring, no converter warps -- a k-block is two 16 KB bulk copies.  Used where
// an operand is produced on the device directly in plane format (the recurrent state of the large-H LSTM path) and the other
// is split once per call (its weights).  c_row_scale: optional per-row output factor (device, [M]).
int linear_planes(const void* a_planes, const void* b_planes, float* C, int64_t ldc, int M, int N, int K, const float* bias,
                  float beta, int act, float a_scale, float b_scale, const float* c_row_scale, bool c_zeroed, int max_splits,
                  cudaStream_t st, int b_kb0, int b_kbtot, int max_ctas, int a_kb0, int a_kbtot, const uint32_t* a_amax, int a_amax_n,
                  const int* m_live, const int* row_map, int live_k) {
  DVAE_REQUIRE(a_planes && b_planes && C && M > 0 && N > 0 && K > 0, "tc16 linear_planes: bad argument");
  // live rows: M (live_k = 0) or K (live_k = 1) is the capacity, the device count is read by the kernel; partial tiles are
  // accumulated atomically into C, which the caller has cleared (or holds the sum to add to: beta = 1)
  DVAE_REQUIRE(!m_live || ((beta == 1.f || (beta == 0.f && c_zeroed)) && act == 0 && !bias && !c_row_scale && (live_k || row_map)),
               "tc16 linear_planes: live rows need a cleared (or accumulated) C, no bias / activation, and a row map for live M");
  Params p = {};
  p.presplit = 1; p.no_astat = 1; p.a_planes = a_planes; p.b_planes = b_planes; p.a_rows = M; p.b_rows = N;
  p.M = M; p.N = N; p.K = K; p.tiles_per_cta = 1; p.C = C; p.ldc = ldc; p.bias = bias; p.beta = beta; p.act = act; p.mode = 0;
  apply_hints(p, GemmHints());
  p.a_scale = a_scale; p.b_scale = b_scale; p.c_row_scale = c_row_scale;
  p.b_kb0 = b_kb0; p.b_kbtot = b_kbtot;          // B planes wider than this GEMM's K range (a vocabulary chunk of W_out^T)
  p.a_kb0 = a_kb0; p.a_kbtot = a_kbtot;
  if (a_amax) { p.a_amax = a_amax; p.a_amax_n = a_amax_n; }      // A planes were scaled by 2^(13 - floor(log2 amax)) (weight_planes_kernel)
  if (m_live) { p.m_live = m_live; p.row_map = row_map; p.live_k = live_k; p.atomic_out = 1; }
  const int tiles = ceil_div(M, BM) * ceil_div(N, BN), nkb = ceil_div(K, BK);
  int splits = 1;
  if (act == 0 && nkb >= 8) {      // same cost model as linear(), with the bulk-copy-fed k-block time
    const float t_kb = 0.27f;
    float best = 1e30f;
    for (int s2 = 1; s2 <= max_splits && s2 <= nkb / 4; ++s2) {
      const int kbs = ceil_div(nkb, s2), se = ceil_div(nkb, kbs);
      if (se != s2) continue;
      if (max_ctas > 0 && s2 > 1 && tiles * se > max_ctas) break;
      const int waves = ceil_div(tiles * se, 148);
      const float t = waves * (kbs * t_kb + (se > 1 ? 5.f : 4.f)) + (se > 1 ? 1.5f : 0.f);
      if (t < best * 0.95f) { best = t; splits = se; }
    }
  }
  p.kb_per_split = ceil_div(nkb, splits);
  splits = ceil_div(nkb, p.kb_per_split);
  if (splits > 1 && beta != 1.f && !(beta == 0.f && c_zeroed)) {
    if (beta == 0.f && ldc == N) {
      DVAE_CUDA(cudaMemsetAsync(C, 0, sizeof(float) * (size_t)M * N, st));
    } else {
      tc16_scale_rows_kernel<<<ceil_div((int64_t)M * N, 256), 256, 0, st>>>(C, ldc, M, N, beta);
      DVAE_LAUNCH_CHECK();
    }
  }
  const int sm_budget = max_ctas > 0 ? max_ctas : 148;
  if (splits == 1 && tiles > sm_budget && ceil_div(N, BN) >= 2) {
    int tpc = ceil_div(tiles, sm_budget);
    if (tpc < 2) tpc = 2;
    if (tpc > ceil_div(N, BN)) tpc = ceil_div(N, BN);
    p.tiles_per_cta = tpc;
  }
  return launch(p, dim3(ceil_div(M, BM), ceil_div(ceil_div(N, BN), p.tiles_per_cta), splits), st);
}

int ce_partials(const float* h, int64_t ldh, int N, int B, int H, int V, const float* w, const float* bias,
                const int64_t* targets, int64_t tgt_stride_b, const int64_t* lengths, int tiles_per_split, int nsplit,
                float* part, int* part_idx, const uint64_t* gumbel_seed, uint32_t gumbel_salt, const void* h_planes,
                const void* w_planes, const int* skip_flag, cudaStream_t st, const int* m_live, const int* row_map) {
  Params p = {};
  p.skip_flag = skip_flag;
  DVAE_REQUIRE(!m_live || (h_planes && w_planes && !gumbel_seed), "tc16 ce_partials: live rows need pre-split operands");
  p.m_live = m_live; p.row_map = row_map;
  if (h_planes && w_planes) { p.presplit = 1; p.a_planes = h_planes; p.b_planes = w_planes; p.a_rows = N; p.b_rows = V; }
  p.A = h; p.lda = ldh; p.Bm = w; p.ldb = H;
  p.M = N; p.N = V; p.K = H; p.tiles_per_cta = tiles_per_split; p.bias = bias; p.mode = 1;
  p.kb_per_split = ceil_div(H, BK);
  p.targets = targets; p.tgt_stride_b = tgt_stride_b; p.lengths = lengths; p.B = B; p.part = part; p.part_idx = part_idx;
  p.gumbel_seed = gumbel_seed; p.gumbel_salt = gumbel_salt;
  apply_hints(p, GemmHints());
  if (p.presplit && single_acc_planes(H)) p.a_scale = p.b_scale = kSingleScale;      // what split_planes applied
  return launch(p, dim3(ceil_div(N, BM), nsplit, 1), st);
}

int softmax_grad(const float* h, int64_t ldh, int N, int B, int H, int V, int v0, int vc, const float* w, const float* bias,
                 const int64_t* targets, int64_t tgt_stride_b, const int64_t* lengths, const float* lse,
                 const float* grad_scale, float* P, int64_t ldp, const void* h_planes, const void* w_planes, float* zero_buf,
                 int64_t zero_n4, float* zero_buf2, int64_t zero2_n4, cudaStream_t st, void* p_planes_a, void* p_planes_t,
                 float* p_colsum, float p_scale, const int* m_live, const int* row_map) {
  Params p = {};
  DVAE_REQUIRE(!m_live || (p_planes_a && p_planes_t && h_planes && w_planes), "tc16 softmax_grad: live rows need the planes output");
  p.m_live = m_live; p.row_map = row_map;
  if (p_planes_a && p_planes_t && h_planes && w_planes) {
    p.p_planes_a = reinterpret_cast<uint8_t*>(p_planes_a); p.p_planes_t = reinterpret_cast<uint8_t*>(p_planes_t);
    p.p_colsum = p_colsum; p.p_scale = p_scale; p.p_kb_a = ceil_div(vc, BK); p.p_kb_t = ceil_div(N, BK);
  }
  p.zero_buf = zero_buf; p.zero_n4 = zero_n4; p.zero_buf2 = zero_buf2; p.zero2_n4 = zero2_n4;
  if (!p.zero_buf) { p.zero_buf = p.zero_buf2; p.zero_n4 = p.zero2_n4; p.zero_buf2 = nullptr; p.zero2_n4 = 0; }
  DVAE_REQUIRE(!(h_planes && w_planes) || v0 % BN == 0, "tc16 softmax_grad: pre-split chunks must start on a %d-row block (v0=%d)", BN, v0);
  if (h_planes && w_planes) { p.presplit = 1; p.a_planes = h_planes; p.b_planes = w_planes; p.a_rows = N; p.b_rows = V; p.b_row0 = v0; }
  p.A = h; p.lda = ldh; p.Bm = w + (int64_t)v0 * H; p.ldb = H;
  // a run of vocabulary tiles per CTA so the epilogue of one tile overlaps the main loop of the next; ~one wave of CTAs
  const int row_tiles = ceil_div(N, BM), col_tiles = ceil_div(vc, BN);
  int per_cta = ceil_div(col_tiles, max(1, 148 / row_tiles));
  if (per_cta < 1) per_cta = 1;
  p.M = N; p.N = vc; p.K = H; p.tiles_per_cta = per_cta; p.bias = bias + v0; p.mode = 2;
  p.kb_per_split = ceil_div(H, BK);
  p.targets = targets; p.tgt_stride_b = tgt_stride_b; p.lengths = lengths; p.B = B; p.lse = lse; p.grad_scale = grad_scale;
  p.v0 = v0; p.C = P; p.ldc = ldp;
  apply_hints(p, GemmHints());
  if (p.presplit && single_acc_planes(H)) p.a_scale = p.b_scale = kSingleScale;      // what split_planes applied
  return launch(p, dim3(row_tiles, ceil_div(col_tiles, per_cta), 1), st);
}

}  // namespace tc16
}  // namespace dvae

extern "C" int dvae_tc16_linear(const float* A, int64_t lda, int trans_a, const float* B, int64_t ldb, int trans_b, float* C,
                                int64_t ldc, int M, int N, int K, const float* bias, const float* bias2, float beta, int act,
                                float a_scale, float b_scale, const uint32_t* a_amax_bits, const uint32_t* b_amax_bits,
                                void* stream) {
  DVAE_REQUIRE(A && B && C && M > 0 && N > 0 && K > 0, "dvae_tc16_linear: bad argument");
  DVAE_REQUIRE(act == 0 || act == 1, "dvae_tc16_linear: unknown activation %d", act);
  DVAE_REQUIRE(dvae::tc16::shape_ok(A, lda, trans_a, B, ldb, trans_b, M, N, K),
               "dvae_tc16_linear: operands must be 16-byte aligned with ld %% 4 == 0 (TMA)");
  dvae::GemmHints h;
  h.a_scale = a_scale; h.b_scale = b_scale; h.a_amax_bits = a_amax_bits; h.b_amax_bits = b_amax_bits;
  return dvae::tc16::linear(A, lda, trans_a, B, ldb, trans_b, C, ldc, M, N, K, bias, bias2, beta, act, h, (cudaStream_t)stream);
}
