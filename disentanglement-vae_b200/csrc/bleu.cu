// Corpus BLEU on token ids (see include/dvae_b200.h):
//   dvae_bleu_counts -- the n-gram statistics of vae/losses.py:128-134 (torchtext 0.6 bleu_score, max_n = 4) of one batch,
//                       ADDED into int64 counters so that a corpus can be accumulated over calls and ranks
//   dvae_bleu_counts_ex -- the same with a row-length bound read from device memory (rows padded beyond their batch's
//                       length, the engine's eval graph at every padded length)
//   dvae_bleu_score  -- the score from those counters, in float64, written to device memory (graph-capturable)
// One warp per row: both truncated rows are staged in shared memory, every lane takes candidate positions, and a position
// contributes min(count_cand, count_ref) of its n-gram only where that n-gram first occurs in the candidate.  O(4 T^2) per
// row.  Integer counts: the result is exact and does not depend on the order of rows or atomics.
#include "common.cuh"

namespace dvae {
namespace {

constexpr int kBleuWarps = 8;
constexpr int kBleuMaxN = 4;

// Length of a row after tensor2text's cut at the first EOS (inclusive; the whole row if there is none) and [1:-1].
__device__ __forceinline__ int bleu_cut_len(const int64_t* __restrict__ row, int T, int64_t eos, int lane) {
  int first = T;
  for (int t = lane; t < T; t += 32)
    if (row[t] == eos) { first = t; break; }
  first = __reduce_min_sync(0xffffffffu, (unsigned)first);
  const int cut = first < T ? first + 1 : T;
  return cut > 2 ? cut - 2 : 0;
}

__device__ __forceinline__ bool ngram_eq(const int64_t* a, int i, const int64_t* b, int j, int n) {
  for (int k = 0; k < n; ++k)
    if (a[i + k] != b[j + k]) return false;
  return true;
}

__global__ void __launch_bounds__(kBleuWarps * 32) bleu_counts_kernel(const int64_t* __restrict__ ref, int64_t ref_stride,
                                                                        int T_ref, const int64_t* __restrict__ cand,
                                                                        int64_t cand_stride, int T_cand, int B, int64_t eos,
                                                                        const int* __restrict__ t_max,
                                                                        unsigned long long* __restrict__ counts) {
  if (t_max != nullptr) {      // rows end at the batch's own padded length: EOS-less rows are cut there, not at the buffer's end
    const int t = max(*t_max, 0);
    T_ref = min(T_ref, t);
    T_cand = min(T_cand, t);
  }
  __shared__ int64_t s_ref[kBleuWarps][DVAE_BLEU_MAX_T];
  __shared__ int64_t s_cand[kBleuWarps][DVAE_BLEU_MAX_T];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int64_t* r = s_ref[w];
  int64_t* c = s_cand[w];
  // [0..3] clipped n-gram matches, [4..7] candidate n-grams, [8] candidate length, [9] reference length
  long long acc[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
  for (int b = blockIdx.x * kBleuWarps + w; b < B; b += gridDim.x * kBleuWarps) {
    const int64_t* rrow = ref + (int64_t)b * ref_stride;
    const int64_t* crow = cand + (int64_t)b * cand_stride;
    const int Lr = bleu_cut_len(rrow, T_ref, eos, lane);
    const int Lc = bleu_cut_len(crow, T_cand, eos, lane);
    for (int t = lane; t < Lr; t += 32) r[t] = rrow[1 + t];
    for (int t = lane; t < Lc; t += 32) c[t] = crow[1 + t];
    __syncwarp();
    if (lane == 0) {
      acc[8] += Lc;
      acc[9] += Lr;
      for (int n = 1; n <= kBleuMaxN; ++n) acc[4 + n - 1] += Lc >= n ? Lc - n + 1 : 0;
    }
#pragma unroll
    for (int n = 1; n <= kBleuMaxN; ++n) {
      for (int i = lane; i + n <= Lc; i += 32) {
        bool first = true;
        for (int j = 0; j < i && first; ++j) first = !ngram_eq(c, j, c, i, n);
        if (!first) continue;
        int cc = 1, rc = 0;
        for (int j = i + 1; j + n <= Lc; ++j) cc += ngram_eq(c, j, c, i, n);
        for (int j = 0; j + n <= Lr; ++j) rc += ngram_eq(r, j, c, i, n);
        acc[n - 1] += cc < rc ? cc : rc;
      }
    }
    __syncwarp();      // the next row overwrites this warp's staging rows
  }
#pragma unroll
  for (int k = 0; k < 10; ++k) {
    long long v = acc[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0 && v != 0) atomicAdd(counts + k, (unsigned long long)v);
  }
}

// torchtext 0.6: 0 if any clipped count is 0, else exp(min(1 - r/c, 0)) * exp(sum_n 0.25 log(clipped_n / total_n))
__global__ void bleu_score_kernel(const int64_t* __restrict__ counts, float* __restrict__ score) {
  double log_p = 0.0;
  for (int n = 0; n < kBleuMaxN; ++n) {
    if (counts[n] <= 0) {
      score[0] = 0.f;
      return;
    }
    log_p += 0.25 * log((double)counts[n] / (double)counts[kBleuMaxN + n]);
  }
  const double bp = exp(fmin(1.0 - (double)counts[9] / (double)counts[8], 0.0));
  score[0] = (float)(bp * exp(log_p));
}

}  // namespace
}  // namespace dvae

extern "C" int dvae_bleu_counts_ex(const int64_t* ref, int64_t ref_stride, int T_ref, const int64_t* cand,
                                   int64_t cand_stride, int T_cand, int B, int64_t eos, const int* t_max, int64_t* counts,
                                   void* stream) {
  DVAE_REQUIRE(ref && cand && counts && B > 0 && T_ref > 0 && T_cand > 0 && ref_stride >= T_ref && cand_stride >= T_cand,
               "dvae_bleu_counts: bad argument");
  DVAE_REQUIRE(T_ref <= DVAE_BLEU_MAX_T && T_cand <= DVAE_BLEU_MAX_T,
               "dvae_bleu_counts: T_ref = %d, T_cand = %d; at most %d tokens per row", T_ref, T_cand, DVAE_BLEU_MAX_T);
  const int grid = dvae::ceil_div(B, dvae::kBleuWarps) < 148 * 4 ? dvae::ceil_div(B, dvae::kBleuWarps) : 148 * 4;
  dvae::bleu_counts_kernel<<<grid, dvae::kBleuWarps * 32, 0, (cudaStream_t)stream>>>(
      ref, ref_stride, T_ref, cand, cand_stride, T_cand, B, eos, t_max, reinterpret_cast<unsigned long long*>(counts));
  DVAE_LAUNCH_CHECK();
  return DVAE_OK;
}

extern "C" int dvae_bleu_counts(const int64_t* ref, int64_t ref_stride, int T_ref, const int64_t* cand, int64_t cand_stride,
                                int T_cand, int B, int64_t eos, int64_t* counts, void* stream) {
  return dvae_bleu_counts_ex(ref, ref_stride, T_ref, cand, cand_stride, T_cand, B, eos, nullptr, counts, stream);
}

extern "C" int dvae_bleu_score(const int64_t* counts, float* score_out, void* stream) {
  DVAE_REQUIRE(counts && score_out, "dvae_bleu_score: bad argument");
  dvae::bleu_score_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(counts, score_out);
  DVAE_LAUNCH_CHECK();
  return DVAE_OK;
}
