// Tile-blocked fp16 (hi, lo) operand planes: the format the pre-split tensor-core GEMM paths read with plain bulk copies
// (tc_gemm16.cu), shared with the kernels that PRODUCE operands in that format (split_planes, the LSTM cell kernels).
//   X [R, K] -> tile (rb = r / 128, kb = k / 32) at byte (rb * KB + kb) * 16384, KB = ceil(K / 32): [hi plane 8 KB][lo plane 8 KB];
//   element (r, k) of a plane at ((r % 128) / 8) * 512 + ((k % 32) / 8) * 128 + (r % 8) * 16 + (k % 8) * 2
//   (UMMA no-swizzle K-major core matrices: 8 rows x 16 bytes, LBO 128 B along K, SBO 512 B along rows).
// Dual-accumulator convention: hi = fp16(x * s), lo = fp16((x * s - hi) * 2^11); the single-accumulator (A-stationary)
// kernels use s * 2^8 and an unscaled lo instead.
#pragma once
#include <cuda_fp16.h>

#include "common.cuh"

namespace dvae {
namespace tc16 {

constexpr int kPlaneRows = 128, kPlaneK = 32;
constexpr int kPlaneBytes = kPlaneRows * kPlaneK * 2, kPlaneTileBytes = 2 * kPlaneBytes;      // 8 KB per plane, 16 KB per [hi | lo] tile
constexpr float kPlaneLoScale = 2048.f;
constexpr float kSingleScale = 256.f;                    // operand scale of the single-accumulator planes

// (x0, x1) * s -> packed fp16 hi pair (returned) and lo pair; packed fp32 arithmetic (FMUL2 / FFMA2)
__device__ __forceinline__ uint32_t pack_hi_lo(float x0, float x1, float s, uint32_t& lo, float ls = kPlaneLoScale) {
  const float2 x = __fmul2_rn(make_float2(x0, x1), make_float2(s, s));
  const __half2 h = __float22half2_rn(x);
  const float2 hf = __half22float2(h);
  // (x - hi) * ls = x * ls - hi * ls (ls a power of two: both products exact); ls = 2^11, or 1 for single-accumulator planes
  const float2 r = __ffma2_rn(x, make_float2(ls, ls), __fmul2_rn(hf, make_float2(-ls, -ls)));
  const __half2 l = __float22half2_rn(r);
  lo = *reinterpret_cast<const uint32_t*>(&l);
  return *reinterpret_cast<const uint32_t*>(&h);
}

// byte offset of the 16-byte chunk holding k .. k+7 (k % 8 == 0) of row r inside the hi plane; the lo chunk is kPlaneBytes later
__host__ __device__ __forceinline__ int64_t plane_chunk_offset(int r, int k, int KB) {
  return ((int64_t)(r >> 7) * KB + (k >> 5)) * kPlaneTileBytes + ((r & 127) >> 3) * 512 + ((k & 31) >> 3) * 128 + (r & 7) * 16;
}

// eight consecutive k of one row -> the row's hi and lo chunks (two 16-byte stores)
__device__ __forceinline__ void store_plane_chunk(uint8_t* planes, int r, int k, int KB, const float (&v)[8], float s) {
  uint4 h, l;
  h.x = pack_hi_lo(v[0], v[1], s, l.x); h.y = pack_hi_lo(v[2], v[3], s, l.y);
  h.z = pack_hi_lo(v[4], v[5], s, l.z); h.w = pack_hi_lo(v[6], v[7], s, l.w);
  const int64_t off = plane_chunk_offset(r, k, KB);
  *reinterpret_cast<uint4*>(planes + off) = h;
  *reinterpret_cast<uint4*>(planes + off + kPlaneBytes) = l;
}

}  // namespace tc16
}  // namespace dvae
