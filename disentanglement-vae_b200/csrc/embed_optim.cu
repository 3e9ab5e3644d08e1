// Embedding lookup / dropout / scatter-add gradient and the fused clip + Adam + zero_grad tail
// (see include/dvae_b200.h).  All HBM-bound element-wise work: float4 accesses, grids sized in
// multiples of the SM count, counter-based Philox so no mask is ever stored.
#include "common.cuh"

namespace dvae {

constexpr int kSMs = 148;

// x[t][b][:] = emb[tok(t,b)][:] * keep_scale ; one warp-quad of float4 lanes per row
__global__ void embedding_fwd_kernel(const float* __restrict__ emb, int E, const int64_t* __restrict__ tokens,
                                     int64_t sb, int64_t st_, int T, int B, float p, const uint64_t* seed_dev,
                                     uint32_t salt, int64_t first_token, int t0, float* __restrict__ x) {
  const int64_t total4 = (int64_t)T * B * ((E + 3) / 4);
  const uint64_t seed = (p > 0.f && seed_dev) ? *seed_dev : 0;
  const float inv_keep = p > 0.f ? 1.f / (1.f - p) : 1.f;
  const int e4n = (E + 3) / 4;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total4; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = i / e4n + (int64_t)t0 * B;      // absolute (t, b) row: the dropout counters match the full-sequence call
    const int e0 = (int)(i % e4n) * 4;
    const int t = (int)(row / B), b = (int)(row % B);
    const int64_t tok = (t == 0 && first_token >= 0) ? first_token : tokens[b * sb + t * st_];
    const float* src = emb + tok * E + e0;
    float s[4] = {1.f, 1.f, 1.f, 1.f};
    if (p > 0.f && seed_dev) dropout_scale4(seed, salt, (uint64_t)(row * e4n + e0 / 4), p, inv_keep, s);
    float* dst = x + row * E + e0;
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (e0 + j < E) dst[j] = src[j] * s[j];
  }
}

__global__ void embedding_bwd_kernel(const float* __restrict__ d_x, int E, const int64_t* __restrict__ tokens,
                                     int64_t sb, int64_t st_, int T, int B, float p, const uint64_t* seed_dev,
                                     uint32_t salt, int64_t first_token, int t0, float* __restrict__ d_emb) {
  const int e4n = (E + 3) / 4;
  const int64_t total4 = (int64_t)T * B * e4n;
  const uint64_t seed = (p > 0.f && seed_dev) ? *seed_dev : 0;
  const float inv_keep = p > 0.f ? 1.f / (1.f - p) : 1.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total4; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = i / e4n + (int64_t)t0 * B;      // absolute (t, b) row: the dropout counters match the full-sequence call
    const int e0 = (int)(i % e4n) * 4;
    const int t = (int)(row / B), b = (int)(row % B);
    const int64_t tok = (t == 0 && first_token >= 0) ? first_token : tokens[b * sb + t * st_];
    float s[4] = {1.f, 1.f, 1.f, 1.f};
    if (p > 0.f && seed_dev) dropout_scale4(seed, salt, (uint64_t)(row * e4n + e0 / 4), p, inv_keep, s);
    const float* src = d_x + row * E + e0;
    float* dst = d_emb + tok * E + e0;
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (e0 + j < E) {
        float v = src[j] * s[j];
        if (v != 0.f) atomicAdd(dst + j, v);
      }
  }
}

// BOWEncoder (vae/model.py:42-49): ctx[b][e] = max_t emb[tok(b,t)][e] * keep_scale(t,b,e) over ALL T positions (padding
// tokens included, as the reference); argmax keeps the first position attaining the maximum (torch.max).  Same Philox
// counters as embedding_fwd_kernel, so the backward pass regenerates the mask of the winning position.
__global__ void bow_max_fwd_kernel(const float* __restrict__ emb, int E, const int64_t* __restrict__ tokens, int64_t sb,
                                   int64_t st_, int T, int B, float p, const uint64_t* seed_dev, uint32_t salt,
                                   float* __restrict__ ctx, int64_t ldctx, int32_t* __restrict__ argmax) {
  const int e4n = (E + 3) / 4;
  const int64_t total = (int64_t)B * e4n;
  const uint64_t seed = (p > 0.f && seed_dev) ? *seed_dev : 0;
  const float inv_keep = p > 0.f ? 1.f / (1.f - p) : 1.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int b = (int)(i / e4n), e0 = (int)(i % e4n) * 4;
    float best[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
    int arg[4] = {0, 0, 0, 0};
    for (int t = 0; t < T; ++t) {
      const int64_t tok = tokens[b * sb + t * st_];
      float s[4] = {1.f, 1.f, 1.f, 1.f};
      if (p > 0.f && seed_dev) dropout_scale4(seed, salt, (uint64_t)(((int64_t)t * B + b) * e4n + e0 / 4), p, inv_keep, s);
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (e0 + j < E) {
          const float v = emb[tok * E + e0 + j] * s[j];
          if (v > best[j]) { best[j] = v; arg[j] = t; }
        }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (e0 + j < E) {
        ctx[(int64_t)b * ldctx + e0 + j] = best[j];
        argmax[(int64_t)b * E + e0 + j] = arg[j];
      }
  }
}

__global__ void bow_max_bwd_kernel(const float* __restrict__ d_ctx, int64_t ldd, const int32_t* __restrict__ argmax, int E,
                                   const int64_t* __restrict__ tokens, int64_t sb, int64_t st_, int T, int B, float p,
                                   const uint64_t* seed_dev, uint32_t salt, float* __restrict__ d_emb) {
  const int e4n = (E + 3) / 4;
  const int64_t total = (int64_t)B * E;
  const uint64_t seed = (p > 0.f && seed_dev) ? *seed_dev : 0;
  const float inv_keep = p > 0.f ? 1.f / (1.f - p) : 1.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int b = (int)(i / E), e = (int)(i % E);
    const int t = argmax[i];
    float s[4] = {1.f, 1.f, 1.f, 1.f};
    if (p > 0.f && seed_dev) dropout_scale4(seed, salt, (uint64_t)(((int64_t)t * B + b) * e4n + e / 4), p, inv_keep, s);
    const float v = d_ctx[(int64_t)b * ldd + e] * s[e & 3];
    if (v != 0.f) atomicAdd(d_emb + tokens[b * sb + t * st_] * E + e, v);
  }
}

__global__ void dropout_kernel(const float* __restrict__ x, int64_t ldx, int64_t rows, int width, float p,
                               const uint64_t* seed_dev, uint32_t salt, float* __restrict__ y, int64_t ldy, int64_t row0) {
  // the recurrence that follows a layer's dropout is launched programmatically: it may start its prologue now and waits
  // for this grid to complete before it reads y
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const int w4n = (width + 3) / 4;
  const int64_t total4 = rows * w4n;
  const uint64_t seed = (p > 0.f && seed_dev) ? *seed_dev : 0;
  const float inv_keep = p > 0.f ? 1.f / (1.f - p) : 1.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total4; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = i / w4n + row0;
    const int c0 = (int)(i % w4n) * 4;
    float s[4] = {1.f, 1.f, 1.f, 1.f};
    if (p > 0.f && seed_dev) dropout_scale4(seed, salt, (uint64_t)(row * w4n + c0 / 4), p, inv_keep, s);
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (c0 + j < width) y[row * ldy + c0 + j] = x[row * ldx + c0 + j] * s[j];
  }
}

// out[i] ~ N(0,1): Box-Muller on Philox uniforms (4 normals per counter)
__global__ void randn_kernel(float* __restrict__ out, int64_t n, const uint64_t* seed_dev, uint32_t salt) {
  const uint64_t seed = *seed_dev;
  const int64_t n4 = (n + 3) / 4;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    uint32_t r[4];
    Philox::gen(seed, salt, (uint64_t)i, r);
    float u0 = ((float)r[0] + 1.f) * 2.3283064365386963e-10f, u1 = (float)r[1] * 2.3283064365386963e-10f;
    float u2 = ((float)r[2] + 1.f) * 2.3283064365386963e-10f, u3 = (float)r[3] * 2.3283064365386963e-10f;
    float a = sqrtf(-2.f * logf(u0)), b = sqrtf(-2.f * logf(u2));
    float s0, c0, s1, c1;
    sincospif(2.f * u1, &s0, &c0);
    sincospif(2.f * u3, &s1, &c1);
    float v[4] = {a * c0, a * s0, b * c1, b * s1};
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (i * 4 + j < n) out[i * 4 + j] = v[j];
  }
}

// ---- optimiser tail ---------------------------------------------------------------------------
constexpr int kRedBlocks = 1024;

__global__ void __launch_bounds__(256) sumsq_kernel(const float* __restrict__ g, int64_t n, float* __restrict__ sumsq,
                                                    float* __restrict__ ws) {
  __shared__ float red[8];
  __shared__ int is_last;
  float acc = 0.f;
  const int64_t n4 = n / 4;
  const float4* g4 = reinterpret_cast<const float4*>(g);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    float4 v = g4[i];
    acc = fmaf(v.x, v.x, acc); acc = fmaf(v.y, v.y, acc); acc = fmaf(v.z, v.z, acc); acc = fmaf(v.w, v.w, acc);
  }
  if (blockIdx.x == 0)
    for (int64_t i = n4 * 4 + threadIdx.x; i < n; i += blockDim.x) acc = fmaf(g[i], g[i], acc);
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int i = 0; i < 8; ++i) t += red[i];
    ws[blockIdx.x] = t;
    __threadfence();
    unsigned int* counter = reinterpret_cast<unsigned int*>(ws + kRedBlocks);
    is_last = atomicAdd(counter, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (is_last) {
    __threadfence();
    // fixed-order tree over the per-block partials (double accumulation)
    double t = 0.0;
    for (int i = threadIdx.x; i < (int)gridDim.x; i += blockDim.x) t += (double)((volatile float*)ws)[i];
    __shared__ double dred[256];
    dred[threadIdx.x] = t;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
      if ((int)threadIdx.x < o) dred[threadIdx.x] += dred[threadIdx.x + o];
      __syncthreads();
    }
    if (threadIdx.x == 0) {
      sumsq[0] = (float)dred[0];
      *reinterpret_cast<unsigned int*>(ws + kRedBlocks) = 0u;   // re-arm for the next call / graph replay
    }
  }
}

__global__ void __launch_bounds__(256) clip_adam_kernel(float* __restrict__ p, float* __restrict__ g,
                                                        float* __restrict__ m, float* __restrict__ v, int64_t n,
                                                        const float* __restrict__ sumsq, float max_norm,
                                                        float grad_scale, const float* __restrict__ hyper,
                                                        int zero_grad) {
  const float lr = hyper[0], b1 = hyper[1], b2 = hyper[2], eps = hyper[3], step = hyper[4];
  float coef = grad_scale;
  if (sumsq) {
    const float norm = sqrtf(sumsq[0]) * fabsf(grad_scale);
    coef *= fminf(1.f, max_norm / (norm + 1e-6f));
  }
  const float bc1 = 1.f - powf(b1, step), bc2 = 1.f - powf(b2, step);
  const float step_size = lr / bc1, inv_bc2_sqrt = 1.f / sqrtf(bc2);
  auto update = [&](float& pi, float& gi_io, float& mi_io, float& vi_io) {
    const float gi = gi_io * coef;
    const float mi = fmaf(b1, mi_io, (1.f - b1) * gi);
    const float vi = fmaf(b2, vi_io, (1.f - b2) * gi * gi);
    mi_io = mi; vi_io = vi;
    pi -= step_size * mi / (sqrtf(vi) * inv_bc2_sqrt + eps);
    gi_io = zero_grad ? 0.f : gi;
  };
  // 16-byte accesses, two vectors per thread and iteration in flight (HBM-bound: 32 B of traffic per parameter)
  const bool vec = (((uintptr_t)p | (uintptr_t)g | (uintptr_t)m | (uintptr_t)v) & 15) == 0;
  const int64_t n4 = vec ? n / 4 : 0;
  float4* p4 = reinterpret_cast<float4*>(p); float4* g4 = reinterpret_cast<float4*>(g);
  float4* m4 = reinterpret_cast<float4*>(m); float4* v4 = reinterpret_cast<float4*>(v);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += 2 * stride) {
    const int64_t j = i + stride;
    const bool two = j < n4;
    float4 pa = p4[i], ga = g4[i], ma = m4[i], va = v4[i];
    float4 pb, gb, mb, vb;
    if (two) { pb = p4[j]; gb = g4[j]; mb = m4[j]; vb = v4[j]; }
    update(pa.x, ga.x, ma.x, va.x); update(pa.y, ga.y, ma.y, va.y); update(pa.z, ga.z, ma.z, va.z); update(pa.w, ga.w, ma.w, va.w);
    p4[i] = pa; g4[i] = ga; m4[i] = ma; v4[i] = va;
    if (two) {
      update(pb.x, gb.x, mb.x, vb.x); update(pb.y, gb.y, mb.y, vb.y); update(pb.z, gb.z, mb.z, vb.z); update(pb.w, gb.w, mb.w, vb.w);
      p4[j] = pb; g4[j] = gb; m4[j] = mb; v4[j] = vb;
    }
  }
  for (int64_t i = n4 * 4 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) update(p[i], g[i], m[i], v[i]);
}

}  // namespace dvae

using namespace dvae;

static int ew_grid(int64_t work) {
  int64_t blocks = (work + 255) / 256;
  int64_t cap = (int64_t)kSMs * 8;
  return (int)(blocks < 1 ? 1 : (blocks > cap ? cap : blocks));
}

extern "C" int dvae_embedding_fwd(const float* emb, int E, const int64_t* tokens, int64_t sb, int64_t st_, int T,
                                  int B, float p, const uint64_t* seed_dev, uint32_t salt, int64_t first_token, int t0, float* x, void* stream) {
  DVAE_REQUIRE(emb && tokens && x && E > 0 && T > 0 && B > 0 && p >= 0.f && p < 1.f, "dvae_embedding_fwd: bad argument");
  embedding_fwd_kernel<<<ew_grid((int64_t)T * B * ((E + 3) / 4)), 256, 0, (cudaStream_t)stream>>>(emb, E, tokens, sb, st_, T, B, p, seed_dev, salt, first_token, t0, x);
  DVAE_LAUNCH_CHECK();
  return DVAE_OK;
}

extern "C" int dvae_embedding_bwd(const float* d_x, int E, const int64_t* tokens, int64_t sb, int64_t st_, int T,
                                  int B, float p, const uint64_t* seed_dev, uint32_t salt, int64_t first_token, int t0, float* d_emb, void* stream) {
  DVAE_REQUIRE(d_x && tokens && d_emb && E > 0 && T > 0 && B > 0 && p >= 0.f && p < 1.f, "dvae_embedding_bwd: bad argument");
  embedding_bwd_kernel<<<ew_grid((int64_t)T * B * ((E + 3) / 4)), 256, 0, (cudaStream_t)stream>>>(d_x, E, tokens, sb, st_, T, B, p, seed_dev, salt, first_token, t0, d_emb);
  DVAE_LAUNCH_CHECK();
  return DVAE_OK;
}

extern "C" int dvae_bow_encoder_fwd(const float* emb, int E, const int64_t* tokens, int64_t sb, int64_t st_, int T, int B, float p,
                                    const uint64_t* seed_dev, uint32_t salt, float* ctx, int64_t ldctx, int32_t* argmax, void* stream) {
  DVAE_REQUIRE(emb && tokens && ctx && argmax && E > 0 && T > 0 && B > 0 && p >= 0.f && p < 1.f, "dvae_bow_encoder_fwd: bad argument");
  bow_max_fwd_kernel<<<ew_grid((int64_t)B * ((E + 3) / 4)), 256, 0, (cudaStream_t)stream>>>(emb, E, tokens, sb, st_, T, B, p, seed_dev, salt, ctx, ldctx, argmax);
  DVAE_LAUNCH_CHECK();
  return DVAE_OK;
}

extern "C" int dvae_bow_encoder_bwd(const float* d_ctx, int64_t ldd, const int32_t* argmax, int E, const int64_t* tokens, int64_t sb,
                                    int64_t st_, int T, int B, float p, const uint64_t* seed_dev, uint32_t salt, float* d_emb, void* stream) {
  DVAE_REQUIRE(d_ctx && argmax && tokens && d_emb && E > 0 && T > 0 && B > 0 && p >= 0.f && p < 1.f, "dvae_bow_encoder_bwd: bad argument");
  bow_max_bwd_kernel<<<ew_grid((int64_t)B * E), 256, 0, (cudaStream_t)stream>>>(d_ctx, ldd, argmax, E, tokens, sb, st_, T, B, p, seed_dev, salt, d_emb);
  DVAE_LAUNCH_CHECK();
  return DVAE_OK;
}

extern "C" int dvae_dropout(const float* x, int64_t ldx, int64_t rows, int width, float p, const uint64_t* seed_dev,
                            uint32_t salt, float* y, int64_t ldy, int64_t row0, void* stream) {
  DVAE_REQUIRE(x && y && rows > 0 && width > 0 && p >= 0.f && p < 1.f, "dvae_dropout: bad argument");
  dropout_kernel<<<ew_grid(rows * ((width + 3) / 4)), 256, 0, (cudaStream_t)stream>>>(x, ldx, rows, width, p, seed_dev, salt, y, ldy, row0);
  DVAE_LAUNCH_CHECK();
  return DVAE_OK;
}

extern "C" int dvae_randn(float* out, int64_t n, const uint64_t* seed_dev, uint32_t salt, void* stream) {
  DVAE_REQUIRE(out && seed_dev && n > 0, "dvae_randn: bad argument");
  randn_kernel<<<ew_grid((n + 3) / 4), 256, 0, (cudaStream_t)stream>>>(out, n, seed_dev, salt);
  DVAE_LAUNCH_CHECK();
  return DVAE_OK;
}

extern "C" int dvae_grad_sumsq(const float* g, int64_t n, float* sumsq, float* ws, void* stream) {
  DVAE_REQUIRE(g && sumsq && ws && n > 0, "dvae_grad_sumsq: bad argument");
  DVAE_REQUIRE((reinterpret_cast<uintptr_t>(g) & 15) == 0, "dvae_grad_sumsq: gradient buffer must be 16-byte aligned");
  int blocks = ew_grid(n / 4 + 1);
  if (blocks > kRedBlocks) blocks = kRedBlocks;
  sumsq_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(g, n, sumsq, ws);
  DVAE_LAUNCH_CHECK();
  return DVAE_OK;
}

extern "C" int dvae_clip_adam(float* p, float* g, float* m, float* v, int64_t n, const float* sumsq, float max_norm,
                              float grad_scale, const float* hyper_dev, int zero_grad, void* stream) {
  DVAE_REQUIRE(p && g && m && v && hyper_dev && n > 0, "dvae_clip_adam: bad argument");
  clip_adam_kernel<<<ew_grid((n + 7) / 8), 256, 0, (cudaStream_t)stream>>>(p, g, m, v, n, sumsq, max_norm, grad_scale, hyper_dev, zero_grad);
  DVAE_LAUNCH_CHECK();
  return DVAE_OK;
}

// ---- length recount of sampled sentences (scripts/evaluation/consistency.py:186-190) ----------------------------
namespace dvae {
// lengths_out[b] = max(min_len, T - #{t : tokens[b,t] == eos or tokens[b,t] == pad}); one warp per row
__global__ void recount_lengths_kernel(const int64_t* __restrict__ tokens, int64_t sb, int64_t st_, int B, int T, int64_t eos,
                                       int64_t pad, int64_t min_len, int64_t* __restrict__ lengths_out) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= B) return;
  int n = 0;
  for (int t = lane; t < T; t += 32) {
    const int64_t tok = tokens[warp * sb + t * st_];
    n += (tok == eos || tok == pad) ? 1 : 0;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(0xffffffffu, n, o);
  if (lane == 0) {
    const int64_t len = (int64_t)T - n;
    lengths_out[warp] = len < min_len ? min_len : len;
  }
}
}  // namespace dvae

extern "C" int dvae_recount_lengths(const int64_t* tokens, int64_t tok_stride_b, int64_t tok_stride_t, int B, int T,
                                    int64_t eos, int64_t pad, int64_t min_len, int64_t* lengths_out, void* stream) {
  DVAE_REQUIRE(tokens && lengths_out && B > 0 && T > 0, "dvae_recount_lengths: bad argument");
  const int threads = 128, blocks = dvae::ceil_div((int64_t)B * 32, threads);
  dvae::recount_lengths_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(tokens, tok_stride_b, tok_stride_t, B, T, eos, pad,
                                                                            min_len, lengths_out);
  DVAE_LAUNCH_CHECK();
  return DVAE_OK;
}
