// fp16 (hi, lo)-split tensor-core GEMM (tc_gemm16.cu): argument block and host entry points.
#pragma once
#include "common.cuh"

namespace dvae {
namespace tc16 {

struct Params {
  const float* A; int64_t lda;     // [M,K] row-major (a_mn = 0) or [K,M] row-major (a_mn = 1)
  const float* Bm; int64_t ldb;    // [N,K] row-major (b_mn = 0) or [K,N] row-major (b_mn = 1)
  int M, N, K;
  int a_mn, b_mn;
  int tiles_per_cta;     // consecutive N tiles per CTA
  float* C; int64_t ldc;
  const float* bias; const float* bias2;
  float beta; int act;
  int mode;              // 0: C = act(alpha * acc + bias) + beta*C;  1: vocab-CE forward partials;  2: softmax-gradient tile
  int kb_per_split;      // k-blocks per blockIdx.z (split-K, mode 0; partial tiles are atomically accumulated)
  // power-of-two operand scales: from the bit pattern of a device-side max |x| (when given) or a host constant
  const uint32_t* a_amax; const uint32_t* b_amax; float a_scale, b_scale; int a_amax_n, b_amax_n;
  float alpha; const float* alpha_dev;
  // modes 1 / 2 (rows are decoder positions n = (t-1)*B + b, columns are vocabulary ids)
  const int64_t* targets; int64_t tgt_stride_b; const int64_t* lengths; int B;
  float* part; int* part_idx;            // mode 1: [nsplit][M][4] (max, sumexp, target logit, argmax value), [nsplit][M]
  const float* lse; const float* grad_scale; int v0;   // mode 2: C = P[:, v0:v0+N]
  const uint64_t* gumbel_seed; uint32_t gumbel_salt;   // mode 1: when set, the arg-max is taken over logits + Gumbel noise
  // pre-split mode: the operands are fp16 (hi, lo) planes in global memory (split_planes), blocked by core matrix
  float* zero_buf; int64_t zero_n4;      // optional: up to two buffers (float4 counts) the kernel clears on its way in
  float* zero_buf2; int64_t zero2_n4;    //           (outputs of later split-K GEMMs; see tc_gemm16.cu)
  int mcast;                             // A-stationary pre-split kernels launched as CTA pairs: B stages fetched half each, multicast
  int a_kbtot; int a_kb0;                 // both-operands-presplit mode: A planes wider than this GEMM's K range
  int b_presplit; int b_kbtot; int b_kb0;   // HYBRID: A through the converter ring, B (a weight) from registered planes: k-blocks per row block / first k-block
  int atomic_out;                        // mode 0: atomicAdd into C even with one k-split (C zeroed by the caller)
  int no_astat;                          // pre-split operands in the dual-accumulator convention: never the A-stationary variant
  const float* c_row_scale;              // optional per-output-row factor [M] (mode 0)
  int presplit; int b_row0;     // b_row0: first B row of this call inside the B planes (a vocabulary chunk)
  const void* a_planes; const void* b_planes; int a_rows, b_rows;      // tile-blocked fp16 planes (split_planes)
  // mode 2, pre-split kernels only: P leaves the kernel as fp16 operand planes (dual-accumulator convention, values * p_scale)
  // in both orientations instead of fp32 -- p_planes_a [M rows, K = N cols] for d_h = P . W, p_planes_t [N cols as rows, K = M]
  // for d_w = P^T . h -- and its column sums are added to p_colsum (the bias gradient): no fp32 P, no converter warps and no
  // separate column-sum kernel downstream
  uint8_t* p_planes_a; uint8_t* p_planes_t; float* p_colsum; float p_scale; int p_kb_a, p_kb_t;
  const int* skip_flag;      // optional device flag: non-zero = the whole launch is a no-op (sampled decoding: a step whose
                             // input is teacher-forced needs no vocabulary sample; decided on the device so one CUDA graph serves every step)
  // live rows (decoder positions the loss keeps; see dvae_vocab_ce_fwd_live): with m_live set, the extent that runs over
  // decoder positions comes from device memory -- M (modes 1 / 2, and mode 0 with live_k = 0) or K (mode 0, live_k = 1) --
  // and the launched CTAs are re-partitioned over the live work (live_split); row_map[k] = position of live row k (modes 1 / 2:
  // targets / lse lookups; mode 0 with live_k = 0: output row k is accumulated into C row row_map[k])
  const int* m_live; const int* row_map; int live_k;
  int dbg_skip_epilogue;     // probes only (DVAE_TC_SKIP_EPILOGUE=1): accumulators are released unread
  unsigned long long* dbg;   // optional: pipeline milestone timestamps (ns) of CTA (0,0,0), profiles/probes/tc16_timeline.py
};

// Vocabulary kernels over live rows: `ctas` launched CTAs, `row_tiles` live 128-row tiles, `col_tiles` vocabulary tiles ->
// vocabulary groups (CTAs per row tile) and tiles per CTA, by the one-wave rule of the full-N launches (ce_nsplit)
__host__ __device__ inline void live_split(int row_tiles, int ctas, int col_tiles, int* tiles_per_cta, int* groups) {
  int g = row_tiles > 0 ? ctas / row_tiles : 1;
  g = g < 1 ? 1 : (g > col_tiles ? col_tiles : g);
  const int tpc = (col_tiles + g - 1) / g;
  *tiles_per_cta = tpc;
  *groups = (col_tiles + tpc - 1) / tpc;
}

bool enabled();     // DVAE_GEMM_IMPL=f16
bool shape_ok(const float* A, int64_t lda, int trans_a, const float* B, int64_t ldb, int trans_b, int M, int N, int K);
bool supported(const float* A, int64_t lda, int trans_a, const float* B, int64_t ldb, int trans_b, int M, int N, int K);
int linear(const float* A, int64_t lda, int trans_a, const float* B, int64_t ldb, int trans_b, float* C, int64_t ldc, int M,
           int N, int K, const float* bias, const float* bias2, float beta, int act, const GemmHints& hints, cudaStream_t st);
// Operand planes: X [R, K] fp32 -> fp16 hi / lo planes (blocked by core matrix, zero padded to 8 rows / 8 columns).
// plane_floats: size of BOTH planes in floats.  Operands that many tiles re-read (the decoder states and the vocabulary
// matrix in the vocab-CE kernels) are split once; the GEMM then runs without landing ring and converter warps.
int64_t plane_floats(int R, int K);
bool single_acc_planes(int K);      // planes of K-deep operands use the single-accumulator convention (tc_planes.cuh)
int split_planes(const float* X, int64_t ld, int R, int K, float scale, void* planes, cudaStream_t st, bool force_dual = false);
int linear_planes(const void* a_planes, const void* b_planes, float* C, int64_t ldc, int M, int N, int K, const float* bias,
                  float beta, int act, float a_scale, float b_scale, const float* c_row_scale, bool c_zeroed, int max_splits,
                  cudaStream_t st, int b_kb0 = 0, int b_kbtot = 0, int max_ctas = 0, int a_kb0 = 0, int a_kbtot = 0,
                  const uint32_t* a_amax = nullptr, int a_amax_n = 1, const int* m_live = nullptr, const int* row_map = nullptr,
                  int live_k = 0);
// Weight-plane registry (api.cu): GEMMs whose B operand is a registered weight matrix (or a 128-row / 32-column aligned
// block of it) fetch B as pre-split planes by bulk copy; only A goes through the converter warps.
constexpr int kMaxPlaneEntries = 24;
struct PlaneTable {
  // ld: row stride of w (0 = C); amax: optional device bit patterns of max |w| (the planes then hold w * 2^(13 - floor(log2 amax)))
  struct Entry { const float* w; int R, C; void* planes; void* planes_t; int64_t ld; const uint32_t* amax; int amax_n; };
  Entry e[kMaxPlaneEntries];
  int n;
};
int weight_planes_launch(const PlaneTable& tab, cudaStream_t st);
struct PlaneHit { const void* planes; int tile0, kb0, kbtot; };
bool find_weight_planes(const float* B, int64_t ldb, int trans_b, int N, int K, PlaneHit* hit);
bool presplit_enabled();      // DVAE_VOCAB_PRESPLIT=0 disables
// h_planes / w_planes (both or neither): planes of h [N, H] and of the WHOLE w [V, H]
int ce_partials(const float* h, int64_t ldh, int N, int B, int H, int V, const float* w, const float* bias,
                const int64_t* targets, int64_t tgt_stride_b, const int64_t* lengths, int tiles_per_split, int nsplit,
                float* part, int* part_idx, const uint64_t* gumbel_seed, uint32_t gumbel_salt, const void* h_planes,
                const void* w_planes, const int* skip_flag, cudaStream_t st, const int* m_live = nullptr,
                const int* row_map = nullptr);
int softmax_grad(const float* h, int64_t ldh, int N, int B, int H, int V, int v0, int vc, const float* w, const float* bias,
                 const int64_t* targets, int64_t tgt_stride_b, const int64_t* lengths, const float* lse,
                 const float* grad_scale, float* P, int64_t ldp, const void* h_planes, const void* w_planes, float* zero_buf,
                 int64_t zero_n4, float* zero_buf2, int64_t zero2_n4, cudaStream_t st, void* p_planes_a = nullptr,
                 void* p_planes_t = nullptr, float* p_colsum = nullptr, float p_scale = 1.f, const int* m_live = nullptr,
                 const int* row_map = nullptr);

}  // namespace tc16
}  // namespace dvae
