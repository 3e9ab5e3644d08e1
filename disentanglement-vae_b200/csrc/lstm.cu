// LSTM layer forward / backward-through-time (see include/dvae_b200.h, dvae_lstm_seq_fwd/bwd).
//
// General-shape path: the input projection for all T steps is one dense GEMM (dvae_linear), the
// recurrence is one launch per time step (both directions in the same grid) with the carried
// state ping-ponged in a small L2-resident buffer; the weight gradients are dense GEMMs over the
// saved gate gradients.  Exact fp32.  (lstm_persist.cu holds the SMEM-resident persistent-cluster
// variant for H <= 256.)
#include <stdlib.h>

#include <cstring>

#include "common.cuh"
#include "lstm_persist.cuh"
#include "tc_gemm16.cuh"

namespace dvae {

int linear_impl(const float* A, int64_t lda, int trans_a, const float* B, int64_t ldb, int trans_b, float* C,
                int64_t ldc, int M, int N, int K, const float* bias, const float* bias2, float beta, int act,
                cudaStream_t st);
int colsum_impl(const float* X, int64_t ldx, int M, int N, float* out, float beta, cudaStream_t st);

// ---- small utility kernels --------------------------------------------------------------------
// dst[d][b][0..H) (row stride ldd, direction stride dird) = src[d][b][..] or 0 when src == NULL
__global__ void copy_state_kernel(const float* __restrict__ src, int64_t lds, int64_t dirs, float* __restrict__ dst,
                                  int64_t ldd, int64_t dird, int D, int B, int H) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)D * B * H) return;
  int u = i % H, b = (i / H) % B, d = i / ((int64_t)H * B);
  dst[d * dird + b * ldd + u] = src ? src[d * dirs + b * lds + u] : 0.f;
}

// out [C,R] = in [R,C]^T
__global__ void transpose_kernel(const float* __restrict__ in, float* __restrict__ out, int R, int C) {
  __shared__ float tile[32][33];
  int c = blockIdx.x * 32 + threadIdx.x, r0 = blockIdx.y * 32;
  for (int j = threadIdx.y; j < 32; j += 8)
    if (r0 + j < R && c < C) tile[j][threadIdx.x] = in[(int64_t)(r0 + j) * C + c];
  __syncthreads();
  int r = r0 + threadIdx.x, c0 = blockIdx.x * 32;
  for (int j = threadIdx.y; j < 32; j += 8)
    if (c0 + j < C && r < R) out[(int64_t)(c0 + j) * R + r] = tile[threadIdx.x][j];
}

int transpose_launch(const float* in, float* out, int R, int C, cudaStream_t st) {
  transpose_kernel<<<dim3(ceil_div(C, 32), ceil_div(R, 32)), dim3(32, 8), 0, st>>>(in, out, R, C);
  DVAE_LAUNCH_CHECK();
  return DVAE_OK;
}
int copy_rows_launch(const float* src, int64_t lds, float* dst, int64_t ldd, int B, int H, cudaStream_t st) {
  copy_state_kernel<<<ceil_div((int64_t)B * H, 256), 256, 0, st>>>(src, lds, 0, dst, ldd, 0, 1, B, H);
  DVAE_LAUNCH_CHECK();
  return DVAE_OK;
}

// ---- per-step mini GEMM -----------------------------------------------------------------------
// acc[r][c] = sum_k A[row0 + rb*2 + r][k] * W[wrow(c)][k]   (both K-contiguous)
// 256 threads: rb = tid / 16 (16 row pairs -> 32 rows), tu = tid % 16; the caller maps (tu, c) to a
// W row.  K is consumed in chunks of KC through shared memory (rows padded to KC+4 floats so the
// float4 reads of 8 consecutive tu hit 8 distinct bank groups).
constexpr int kStepRows = 32, kStepKC = 64, kStepThreads = 256;

template <int NC>
struct StepGemm {
  static constexpr int WR = 16 * NC;  // W rows per tile
  static constexpr int LDS_ = kStepKC + 4;
  static constexpr int SMEM_FLOATS = (kStepRows + WR) * LDS_;

  template <class WRowFn>
  __device__ static __forceinline__ void run(const float* __restrict__ A, int64_t lda, int row0, int nrows,
                                             const float* __restrict__ W, int64_t ldw, WRowFn wrow, int K,
                                             float* smem, float (&acc)[2][NC]) {
    const int tid = threadIdx.x, rb = tid / 16, tu = tid % 16;
    float* As = smem;
    float* Ws = smem + kStepRows * LDS_;
    const bool a_vec = ((reinterpret_cast<uintptr_t>(A) & 15) == 0) && (lda % 4 == 0);
    const bool w_vec = ((reinterpret_cast<uintptr_t>(W) & 15) == 0) && (ldw % 4 == 0);
    for (int k0 = 0; k0 < K; k0 += kStepKC) {
      // A chunk: 32 rows x 64 k = 512 float4
      for (int v = tid; v < kStepRows * kStepKC / 4; v += kStepThreads) {
        int r = v / (kStepKC / 4), kq = v % (kStepKC / 4), gk = k0 + kq * 4, gr = row0 + r;
        float4 val = make_float4(0.f, 0.f, 0.f, 0.f);
        if (gr < nrows && gk < K) {
          const float* q = A + (int64_t)gr * lda + gk;
          if (a_vec && gk + 3 < K) val = *reinterpret_cast<const float4*>(q);
          else { val.x = q[0]; if (gk + 1 < K) val.y = q[1]; if (gk + 2 < K) val.z = q[2]; if (gk + 3 < K) val.w = q[3]; }
        }
        *reinterpret_cast<float4*>(&As[r * LDS_ + kq * 4]) = val;
      }
      for (int v = tid; v < WR * kStepKC / 4; v += kStepThreads) {
        int r = v / (kStepKC / 4), kq = v % (kStepKC / 4), gk = k0 + kq * 4;
        int64_t gr = wrow(r % 16, r / 16);  // < 0 when out of range
        float4 val = make_float4(0.f, 0.f, 0.f, 0.f);
        if (gr >= 0 && gk < K) {
          const float* q = W + gr * ldw + gk;
          if (w_vec && gk + 3 < K) val = *reinterpret_cast<const float4*>(q);
          else { val.x = q[0]; if (gk + 1 < K) val.y = q[1]; if (gk + 2 < K) val.z = q[2]; if (gk + 3 < K) val.w = q[3]; }
        }
        *reinterpret_cast<float4*>(&Ws[r * LDS_ + kq * 4]) = val;
      }
      __syncthreads();
#pragma unroll 4
      for (int kq = 0; kq < kStepKC / 4; ++kq) {
        float4 a0 = *reinterpret_cast<const float4*>(&As[(rb * 2 + 0) * LDS_ + kq * 4]);
        float4 a1 = *reinterpret_cast<const float4*>(&As[(rb * 2 + 1) * LDS_ + kq * 4]);
#pragma unroll
        for (int c = 0; c < NC; ++c) {
          float4 w = *reinterpret_cast<const float4*>(&Ws[(c * 16 + tu) * LDS_ + kq * 4]);
          acc[0][c] = fmaf(a0.x, w.x, acc[0][c]); acc[0][c] = fmaf(a0.y, w.y, acc[0][c]);
          acc[0][c] = fmaf(a0.z, w.z, acc[0][c]); acc[0][c] = fmaf(a0.w, w.w, acc[0][c]);
          acc[1][c] = fmaf(a1.x, w.x, acc[1][c]); acc[1][c] = fmaf(a1.y, w.y, acc[1][c]);
          acc[1][c] = fmaf(a1.z, w.z, acc[1][c]); acc[1][c] = fmaf(a1.w, w.w, acc[1][c]);
        }
      }
      __syncthreads();
    }
  }
};

// ---- forward step -----------------------------------------------------------------------------
struct FwdStepArgs {
  const float* w_hh[2];
  float* gates;            // [D,T,B,4H]
  float* cs;               // [D,T,B,H]
  const float* h_in;       // carried state, [D,B,H]
  const float* c_in;
  float* h_out;
  float* c_out;
  float* hs;               // [T,B,D*H]
  int64_t ldhs;
  const int64_t* lengths;
  int s, T, B, H;
};

// grid (ceil(H/16), ceil(B/32), D); tile = 32 rows x 16 units x 4 gates
__global__ void __launch_bounds__(kStepThreads) lstm_step_fwd_kernel(FwdStepArgs p) {
  __shared__ __align__(16) float smem[StepGemm<4>::SMEM_FLOATS];
  const int d = blockIdx.z, H = p.H, B = p.B;
  const int t = d == 0 ? p.s : p.T - 1 - p.s;
  const int u0 = blockIdx.x * 16, b0 = blockIdx.y * kStepRows;
  const int tid = threadIdx.x, rb = tid / 16, tu = tid % 16;
  const float* h_in = p.h_in + (int64_t)d * B * H;
  float acc[2][4] = {};
  auto wrow = [&](int u, int g) -> int64_t { return (u0 + u < H) ? (int64_t)g * H + u0 + u : -1; };
  StepGemm<4>::run(h_in, H, b0, B, p.w_hh[d], H, wrow, H, smem, acc);
  const int u = u0 + tu;
  if (u >= H) return;
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    const int b = b0 + rb * 2 + r;
    if (b >= B) continue;
    const int64_t sb = ((int64_t)d * B + b) * H + u;                       // carried-state index
    const int64_t gi = (((int64_t)d * p.T + t) * B + b) * 4 * H + u;       // gate slab index (gate 0)
    const int64_t ci = (((int64_t)d * p.T + t) * B + b) * H + u;
    const float c_prev = p.c_in[sb], h_prev = p.h_in[sb];
    const bool live = p.lengths == nullptr || t < p.lengths[b];
    float* hs = p.hs + ((int64_t)t * B + b) * p.ldhs + d * H + u;
    if (live) {
      const float ig = sigmoidf_(p.gates[gi] + acc[r][0]);
      const float fg = sigmoidf_(p.gates[gi + H] + acc[r][1]);
      const float gg = tanhf(p.gates[gi + 2 * H] + acc[r][2]);
      const float og = sigmoidf_(p.gates[gi + 3 * H] + acc[r][3]);
      const float c = fmaf(fg, c_prev, ig * gg);
      const float h = og * tanhf(c);
      p.gates[gi] = ig; p.gates[gi + H] = fg; p.gates[gi + 2 * H] = gg; p.gates[gi + 3 * H] = og;
      p.cs[ci] = c; p.c_out[sb] = c; p.h_out[sb] = h; *hs = h;
    } else {
      p.gates[gi] = 0.f; p.gates[gi + H] = 0.f; p.gates[gi + 2 * H] = 0.f; p.gates[gi + 3 * H] = 0.f;
      p.cs[ci] = c_prev; p.c_out[sb] = c_prev; p.h_out[sb] = h_prev; *hs = 0.f;
    }
  }
}

// ---- backward step ----------------------------------------------------------------------------
struct BwdStepArgs {
  const float* w_hh_t[2];  // [H,4H] (transposed recurrent weights)
  float* gates;            // [D,T,B,4H]: post-activation gates in, dG out
  const float* cs;         // [D,T,B,H]
  const float* c0;         // initial cell state [D][B] rows (ld0, dir0) or NULL
  int64_t ld0, dir0;
  const float* d_hs;       // [T,B,D*H] or NULL
  int64_t lddhs;
  const float* carry_in;   // [D,B,H] gradient carried by frozen rows / final-state gradient
  const float* dc_in;
  float* carry_out;
  float* dc_out;
  float* d_h0;             // final launch only: gradient w.r.t. the initial state
  float* d_c0;
  int64_t ldd0, dird0;
  const int64_t* lengths;
  int s, T, B, H, final_;
};

// grid (ceil(H/32), ceil(B/32), D); tile = 32 rows x 32 units
__global__ void __launch_bounds__(kStepThreads) lstm_step_bwd_kernel(BwdStepArgs p) {
  __shared__ __align__(16) float smem[StepGemm<2>::SMEM_FLOATS];
  const int d = blockIdx.z, H = p.H, B = p.B, T = p.T;
  // time index processed at this step and the one processed at the previous step
  const int t = d == 0 ? T - 1 - p.s : p.s;
  const int t_next = d == 0 ? t + 1 : t - 1;
  const int u0 = blockIdx.x * 32, b0 = blockIdx.y * kStepRows;
  const int tid = threadIdx.x, rb = tid / 16, tu = tid % 16;
  float acc[2][2] = {};
  if (p.s > 0) {
    const float* dg_next = p.gates + ((int64_t)d * T + t_next) * B * 4 * H;
    auto wrow = [&](int u, int c) -> int64_t { return (u0 + c * 16 + u < H) ? (int64_t)(u0 + c * 16 + u) : -1; };
    StepGemm<2>::run(dg_next, 4 * H, b0, B, p.w_hh_t[d], 4 * H, wrow, 4 * H, smem, acc);
  }
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    const int b = b0 + rb * 2 + r;
    if (b >= B) continue;
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      const int u = u0 + c * 16 + tu;
      if (u >= H) continue;
      const int64_t sb = ((int64_t)d * B + b) * H + u;
      const float dh_in = p.carry_in[sb] + acc[r][c];
      const float dc_in = p.dc_in[sb];
      if (p.final_) {
        if (p.d_h0) p.d_h0[d * p.dird0 + (int64_t)b * p.ldd0 + u] = dh_in;
        if (p.d_c0) p.d_c0[d * p.dird0 + (int64_t)b * p.ldd0 + u] = dc_in;
        continue;
      }
      const int64_t gi = (((int64_t)d * T + t) * B + b) * 4 * H + u;
      const bool live = p.lengths == nullptr || t < p.lengths[b];
      if (!live) {
        p.gates[gi] = 0.f; p.gates[gi + H] = 0.f; p.gates[gi + 2 * H] = 0.f; p.gates[gi + 3 * H] = 0.f;
        p.carry_out[sb] = dh_in; p.dc_out[sb] = dc_in;
        continue;
      }
      const int64_t ci = (((int64_t)d * T + t) * B + b) * H + u;
      const int t_prev = d == 0 ? t - 1 : t + 1;     // step that ran before t in the forward traversal
      float c_prev;
      if (t_prev >= 0 && t_prev < T) c_prev = p.cs[(((int64_t)d * T + t_prev) * B + b) * H + u];
      else c_prev = p.c0 ? p.c0[d * p.dir0 + (int64_t)b * p.ld0 + u] : 0.f;
      const float dh = dh_in + (p.d_hs ? p.d_hs[((int64_t)t * B + b) * p.lddhs + d * H + u] : 0.f);
      const float ig = p.gates[gi], fg = p.gates[gi + H], gg = p.gates[gi + 2 * H], og = p.gates[gi + 3 * H];
      const float tc = tanhf(p.cs[ci]);
      const float dc = fmaf(dh * og, 1.f - tc * tc, dc_in);
      p.gates[gi] = dc * gg * ig * (1.f - ig);
      p.gates[gi + H] = dc * c_prev * fg * (1.f - fg);
      p.gates[gi + 2 * H] = dc * ig * (1.f - gg * gg);
      p.gates[gi + 3 * H] = dh * tc * og * (1.f - og);
      p.carry_out[sb] = 0.f;
      p.dc_out[sb] = dc * fg;
    }
  }
}

// ---- host orchestration -----------------------------------------------------------------------
// DVAE_LSTM_IMPL=step forces the general per-step path (A/B tests of the persistent kernels)
static bool force_step_path() {
  const char* e = getenv("DVAE_LSTM_IMPL");
  return e && !strcmp(e, "step");
}
static int64_t state_floats(int B, int H, int D) { return 4LL * D * B * H; }
// state workspace (floats): [carried state 4*D*B*H][transposed W_hh 4*D*H*H][8 rotating max|dG| slot sets][operand planes]
static int64_t planes_ws_offset(int B, int H, int D) { return state_floats(B, H, D) + 4LL * D * H * H + 8LL * amax_slot_entries(B, D); }

// gates[d] [T*B, 4H] = x . W_ih[d]^T + b_ih[d] + b_hh[d]: the time-parallel half of the layer (one GEMM per direction)
int lstm_input_proj_impl(const float* x, int64_t ldx, int T, int B, int I, int H, int D, const float* const* w_ih,
                         const float* const* b_ih, const float* const* b_hh, float* gates, cudaStream_t st) {
  DVAE_REQUIRE(x && gates && w_ih, "dvae_lstm_input_proj: null pointer");
  DVAE_REQUIRE(T > 0 && B > 0 && I > 0 && H > 0 && (D == 1 || D == 2), "dvae_lstm_input_proj: bad shape T=%d B=%d I=%d H=%d D=%d", T, B, I, H, D);
  const int64_t slab = (int64_t)T * B * 4 * H;
  Fork fork(st);           // the two directions' input projections are independent
  GemmHints gh;
  gh.concurrency = D;      // they run at the same time: each sizes its grid for half of the SMs
  for (int d = 0; d < D; ++d) {
    int rc = linear_impl_ex(x, ldx, 0, w_ih[d], I, 0, gates + d * slab, 4 * H, T * B, 4 * H, I, b_ih ? b_ih[d] : nullptr,
                            b_hh ? b_hh[d] : nullptr, 0.f, 0, gh, d == 0 ? st : fork.side(0));
    if (rc) return rc;
  }
  return fork.join();
}

int lstm_seq_fwd_impl(const float* x, int64_t ldx, int T, int B, int I, int H, int D, const float* const* w_ih,
                      const float* const* w_hh, const float* const* b_ih, const float* const* b_hh,
                      const float* h0, const float* c0, int64_t ld0, int64_t dir0, const int64_t* lengths,
                      float* hs, int64_t ldhs, float* hn, float* cn, int64_t ldn, int64_t dirn, float* gates,
                      float* cs, float* ws, bool gates_ready, cudaStream_t st) {
  DVAE_REQUIRE(x && hs && gates && cs && ws && w_ih && w_hh, "dvae_lstm_seq_fwd: null pointer");
  DVAE_REQUIRE(T > 0 && B > 0 && I > 0 && H > 0 && (D == 1 || D == 2), "dvae_lstm_seq_fwd: bad shape T=%d B=%d I=%d H=%d D=%d", T, B, I, H, D);
  DVAE_REQUIRE(!(lengths && h0), "dvae_lstm_seq_fwd: length-masked layers start from the zero state");
  const int64_t sf = (int64_t)D * B * H;
  if (!gates_ready) {
    int rc = lstm_input_proj_impl(x, ldx, T, B, I, H, D, w_ih, b_ih, b_hh, gates, st);
    if (rc) return rc;
  }
  {
    const void* ptrs[] = {x, w_hh[0], w_hh[D - 1], h0, c0, hs, hn, cn, gates, cs, ws};
    const int64_t lds[] = {ld0, dir0, ldhs, ldn, dirn};
    if (!force_step_path() && persist_supported(B, H, D, ptrs, 11, lds, 5)) {
      PersistFwdArgs a;
      a.w_hh[0] = w_hh[0]; a.w_hh[1] = w_hh[D - 1];
      a.gates = gates; a.cs = cs; a.hs = hs; a.ldhs = ldhs; a.h0 = h0; a.c0 = c0; a.ld0 = ld0; a.dir0 = dir0;
      a.hstate = ws; a.hn = hn; a.cn = cn; a.ldn = ldn; a.dirn = dirn; a.lengths = lengths;
      a.T = T; a.B = B; a.D = D; a.n_slices = ceil_div(B, 16); a.d_off = 0;
      a.dbg = nullptr;
      if (const char* e = getenv("DVAE_LSTM_DBG")) a.dbg = reinterpret_cast<unsigned long long*>(strtoull(e, nullptr, 0));
      return persist_fwd(H, a, st);
    }
    // hidden sizes beyond the cluster-resident kernels (512, 1024, ...): per-step tensor-core GEMMs over operand planes
    if (!force_step_path() && planes_lstm_supported(B, H, D, ptrs, 11, lds, 5) && resident_lstm_supported(B, H))
      return resident_lstm_fwd(T, B, H, D, w_hh, h0, c0, ld0, dir0, lengths, hs, ldhs, hn, cn, ldn, dirn, gates, cs,
                               ws + planes_ws_offset(B, H, D), st);
    if (!force_step_path() && planes_lstm_supported(B, H, D, ptrs, 11, lds, 5))
      return planes_lstm_fwd(T, B, H, D, w_hh, h0, c0, ld0, dir0, lengths, hs, ldhs, hn, cn, ldn, dirn, gates, cs, ws,
                             ws + planes_ws_offset(B, H, D), st);
  }
  float* hbuf[2] = {ws, ws + 2 * sf};
  float* cbuf[2] = {ws + sf, ws + 3 * sf};
  const int nthr = 256, nblk = ceil_div(sf, nthr);
  copy_state_kernel<<<nblk, nthr, 0, st>>>(h0, ld0, dir0, hbuf[0], H, (int64_t)B * H, D, B, H);
  DVAE_LAUNCH_CHECK();
  copy_state_kernel<<<nblk, nthr, 0, st>>>(c0, ld0, dir0, cbuf[0], H, (int64_t)B * H, D, B, H);
  DVAE_LAUNCH_CHECK();
  FwdStepArgs a;
  for (int d = 0; d < 2; ++d) a.w_hh[d] = w_hh[d < D ? d : 0];
  a.gates = gates; a.cs = cs; a.hs = hs; a.ldhs = ldhs; a.lengths = lengths; a.T = T; a.B = B; a.H = H;
  dim3 grid(ceil_div(H, 16), ceil_div(B, kStepRows), D);
  for (int s = 0; s < T; ++s) {
    a.s = s;
    a.h_in = hbuf[s & 1]; a.c_in = cbuf[s & 1]; a.h_out = hbuf[(s + 1) & 1]; a.c_out = cbuf[(s + 1) & 1];
    lstm_step_fwd_kernel<<<grid, kStepThreads, 0, st>>>(a);
    DVAE_LAUNCH_CHECK();
  }
  if (hn) {
    copy_state_kernel<<<nblk, nthr, 0, st>>>(hbuf[T & 1], H, (int64_t)B * H, hn, ldn, dirn, D, B, H);
    DVAE_LAUNCH_CHECK();
  }
  if (cn) {
    copy_state_kernel<<<nblk, nthr, 0, st>>>(cbuf[T & 1], H, (int64_t)B * H, cn, ldn, dirn, D, B, H);
    DVAE_LAUNCH_CHECK();
  }
  return DVAE_OK;
}

// dvae_lstm_bwd_dx_stream: where the d_x GEMM of a unidirectional layer's backward runs (nullptr: the call's stream)
static thread_local cudaStream_t g_dx_stream = nullptr;

int lstm_seq_bwd_impl(const float* x, int64_t ldx, int T, int B, int I, int H, int D, const float* const* w_ih,
                      const float* const* w_hh, const float* h0, const float* c0, int64_t ld0, int64_t dir0,
                      const int64_t* lengths, const float* hs, int64_t ldhs, float* gates, const float* cs,
                      const float* d_hs, int64_t lddhs, const float* d_hn, const float* d_cn, int64_t ldn,
                      int64_t dirn, float* d_x, int64_t lddx, float* const* d_w_ih, float* const* d_w_hh,
                      float* const* d_b_ih, float* const* d_b_hh, float* d_h0, float* d_c0, int64_t ldd0,
                      int64_t dird0, float* ws, float* planes_ws, cudaStream_t st) {
  DVAE_REQUIRE(x && hs && gates && cs && ws && w_ih && w_hh, "dvae_lstm_seq_bwd: null pointer");
  DVAE_REQUIRE(T > 0 && B > 0 && I > 0 && H > 0 && (D == 1 || D == 2), "dvae_lstm_seq_bwd: bad shape");
  DVAE_REQUIRE(!(lengths && h0), "dvae_lstm_seq_bwd: length-masked layers start from the zero state");
  const int64_t slab = (int64_t)T * B * 4 * H, sf = (int64_t)D * B * H;
  bool persisted = false;
  uint32_t* amax = nullptr;
  int amax_n = 1;
  bool dx_zeroed = false;
  {
    const void* ptrs[] = {w_hh[0], w_hh[D - 1], c0, gates, cs, d_hs, d_hn, d_cn, d_h0, d_c0};
    const int64_t lds[] = {ld0, dir0, lddhs, ldn, dirn, ldd0, dird0};
    if (!force_step_path() && persist_supported(B, H, D, ptrs, 10, lds, 7)) {
      PersistBwdArgs a;
      a.w_hh[0] = w_hh[0]; a.w_hh[1] = w_hh[D - 1];
      a.gates = gates; a.cs = cs; a.c0 = c0; a.ld0 = ld0; a.dir0 = dir0; a.d_hs = d_hs; a.lddhs = lddhs;
      a.d_hn = d_hn; a.d_cn = d_cn; a.ldn = ldn; a.dirn = dirn; a.d_h0 = d_h0; a.d_c0 = d_c0; a.ldd0 = ldd0;
      a.dird0 = dird0; a.lengths = lengths; a.T = T; a.B = B; a.D = D; a.n_slices = ceil_div(B, 16); a.d_off = 0;
      a.amax_out = nullptr;
      a.zero_buf = nullptr; a.zero_n4 = 0;
      if (tc_lstm_supported(H)) {      // the tcgen05 kernel also reports max |dG|: the operand scale of the GEMMs below
        // 8 rotating slots: with deferred joins the previous layers' GEMMs may still be reading theirs
        static thread_local unsigned slot = 0;
        amax = reinterpret_cast<uint32_t*>(ws + state_floats(B, H, D) + 4LL * D * H * H) + amax_slot_entries(B, D) * (slot++ & 7);
        a.amax_out = amax;               // one entry per CTA of the recurrence kernel (<= amax_slot_entries), written, never accumulated
        amax_n = tc_lstm_bwd_ctas(B, D);
        if (d_x && lddx == I && (((uintptr_t)d_x) & 15) == 0 && ((int64_t)T * B * I) % 4 == 0 && d_x != d_hs) {
          a.zero_buf = d_x; a.zero_n4 = (int64_t)T * B * I / 4;
          dx_zeroed = true;
        }
      }
      int rc = persist_bwd(H, a, st);
      if (rc) return rc;
      persisted = true;
    } else {
      const void* ptrs2[] = {w_hh[0], w_hh[D - 1], c0, gates, cs, d_hs, d_hn, d_cn, d_h0, d_c0, ws};
      if (!force_step_path() && planes_lstm_supported(B, H, D, ptrs2, 11, lds, 7)) {
        static thread_local unsigned slot2 = 0;      // rotating: deferred weight-gradient GEMMs of earlier layers may still read theirs
        amax = reinterpret_cast<uint32_t*>(ws + state_floats(B, H, D) + 4LL * D * H * H) + amax_slot_entries(B, D) * (slot2++ & 7);
        amax_n = D;
        int rc = planes_lstm_bwd(T, B, H, D, w_hh, c0, ld0, dir0, lengths, gates, cs, d_hs, lddhs, d_hn, d_cn, ldn, dirn, d_h0,
                                 d_c0, ldd0, dird0, ws, ws + 4 * sf, ws + planes_ws_offset(B, H, D), amax, st);
        if (rc) return rc;
        persisted = true;
      }
    }
  }
  float* carry[2] = {ws, ws + 2 * sf};
  float* dcb[2] = {ws + sf, ws + 3 * sf};
  float* wt = ws + 4 * sf;  // [D][H,4H]
  for (int d = 0; d < D && !persisted; ++d) {
    transpose_kernel<<<dim3(ceil_div(H, 32), ceil_div(4 * H, 32)), dim3(32, 8), 0, st>>>(w_hh[d], wt + (int64_t)d * 4 * H * H, 4 * H, H);
    DVAE_LAUNCH_CHECK();
  }
  const int nthr = 256, nblk = ceil_div(sf, nthr);
  if (!persisted) {
    copy_state_kernel<<<nblk, nthr, 0, st>>>(d_hn, ldn, dirn, carry[0], H, (int64_t)B * H, D, B, H);
    DVAE_LAUNCH_CHECK();
    copy_state_kernel<<<nblk, nthr, 0, st>>>(d_cn, ldn, dirn, dcb[0], H, (int64_t)B * H, D, B, H);
    DVAE_LAUNCH_CHECK();
  }
  BwdStepArgs a;
  for (int d = 0; d < 2; ++d) a.w_hh_t[d] = wt + (int64_t)(d < D ? d : 0) * 4 * H * H;
  a.gates = gates; a.cs = cs; a.c0 = c0; a.ld0 = ld0; a.dir0 = dir0; a.d_hs = d_hs; a.lddhs = lddhs;
  a.d_h0 = d_h0; a.d_c0 = d_c0; a.ldd0 = ldd0; a.dird0 = dird0; a.lengths = lengths; a.T = T; a.B = B; a.H = H;
  dim3 grid(ceil_div(H, 32), ceil_div(B, kStepRows), D);
  const int nsteps = persisted ? 0 : T + ((d_h0 || d_c0) ? 1 : 0);
  for (int s = 0; s < nsteps; ++s) {
    a.s = s; a.final_ = (s == T);
    a.carry_in = carry[s & 1]; a.dc_in = dcb[s & 1]; a.carry_out = carry[(s + 1) & 1]; a.dc_out = dcb[(s + 1) & 1];
    if (a.final_) {
      // s == T: t_next must be the last processed index; reuse the formulas with s = T
      // (dir 0: t = -1 -> t_next = 0; dir 1: t = T -> t_next = T-1)
    }
    lstm_step_bwd_kernel<<<grid, kStepThreads, 0, st>>>(a);
    DVAE_LAUNCH_CHECK();
  }
  // dense gradients from the saved dG slabs (A operand = dG: a gradient, scaled by its measured amax when known)
  GemmHints gh;
  gh.a_wide = true;
  gh.a_amax_bits = amax;
  gh.a_amax_n = amax_n;
  // the weight-gradient GEMMs below run on side streams beside the NEXT layer's recurrence (deferred joins): sized to leave
  // that recurrence its SMs (64 at cfg 2).  Two machine-filling split-K grids (2 x 144 CTAs) kept the recurrence kernel
  // from being scheduled for 25-40 us at every layer boundary.  (Caps derived from the SMs the recurrence leaves, 42 per
  // GEMM or 28 with d_x beside them, measured slower at cfg 2: 1.064 against 1.042 ms per step.)
  GemmHints gh_bg = gh;
  {
    static const int cap = [] { const char* e = getenv("DVAE_DW_MAX_CTAS"); return e ? atoi(e) : 48; }();
    // Only where the neighbour is the cluster recurrence (H <= 256: a 64-CTA launch that must be placed at once).  At
    // H = 1024 the recurrences are per-step launches / a grid-resident kernel and the GEMMs are 100x larger: the cap cost
    // 2.3 % there (cfg 4: 25.70 ms capped, 25.10 ms uncapped).
    gh_bg.max_ctas = (defer_joins_enabled() && tc_lstm_supported(H)) ? cap : 0;
  }
  // a unidirectional layer's d_x on the caller-named stream (dvae_lstm_bwd_dx_stream), ordered after the recurrence: a
  // background GEMM there, sized like the weight gradients
  const bool dx_bg = d_x && D == 1 && g_dx_stream && g_dx_stream != st;
  // d_x accumulates over the directions (main stream, in order); the weight / bias gradients of each direction are
  // independent of it and of each other: parallel branches
  Fork fork(st);
  // d_x of a bidirectional layer = sum of the two directions' products.  When the recurrence kernel already cleared d_x, both
  // GEMMs add into it with atomics and run CONCURRENTLY (the reverse direction's on a side stream, marked so that only this
  // one launch is waited for before d_x is consumed) instead of back to back on the critical path
  const bool dx_pair = d_x && D == 2 && dx_zeroed && !force_simt_gemm() && tc_lstm_supported(H) &&
                       !(getenv("DVAE_DX_PAIR") && getenv("DVAE_DX_PAIR")[0] == '0');
  if (dx_pair) {
    GemmHints ghx = gh;
    ghx.c_zeroed = true; ghx.atomic_out = true; ghx.concurrency = 2;
    int rc = linear_impl_ex(gates + slab, 4 * H, 0, w_ih[1], I, 1, d_x, lddx, T * B, I, 4 * H, nullptr, nullptr, 1.f, 0, ghx, fork.side(2));
    if (rc) return rc;
    if ((rc = fork.mark(2))) return rc;
  }
  // Weight gradients dW_ih = dG^T x, dW_hh = dG^T h_prev contract over the T*B positions: both operands are read "transposed"
  // (MN-major), the converter path's slowest case (0.74 us per k-block, tensor pipe 9 %).  With a plane workspace the three
  // matrices are transposed ONCE into fp16 operand planes by one launch (dG scaled by its measured amax) and the GEMMs run
  // bulk-copy fed on both operands; time steps shift by whole k-blocks (B % 32 == 0) for the h_{t-1} pairing.
  const int TB = T * B, KBt = ceil_div(TB, 32);
  // Measured (A/B on one box, graph replay): 25.7 vs 28.0 ms per step at H = 1024 (cfg4), but 1.163 vs 1.142 ms at cfg2 and
  // 0.938 vs 0.929 at cfg3, where the GEMMs are a few k-blocks per CTA and the extra transposing launch sits in the step's
  // tail: the planes are used from 2^32 multiply-adds per GEMM upwards (DVAE_DW_PLANES=1 / 0 forces either way).
  const char* dwp_env = getenv("DVAE_DW_PLANES");
  const bool dwp_on = dwp_env ? dwp_env[0] != '0' : (int64_t)4 * H * (I > H ? I : H) * TB >= ((int64_t)1 << 32);
  const bool dw_planes = planes_ws && amax && !force_simt_gemm() && tc16::enabled() && TB >= 128 &&
                         (reinterpret_cast<uintptr_t>(planes_ws) & 15) == 0 && dwp_on;
  const bool hh_planes = dw_planes && T > 1 && B % 32 == 0;
  float *xT = planes_ws, *dGt[2] = {nullptr, nullptr}, *hsT[2] = {nullptr, nullptr};
  if (dw_planes) {
    float* q = xT + tc16::plane_floats(I, TB);
    for (int d = 0; d < D; ++d) { dGt[d] = q; q += tc16::plane_floats(4 * H, TB); }
    for (int d = 0; d < D; ++d) { hsT[d] = q; q += tc16::plane_floats(H, TB); }
    tc16::PlaneTable tab;
    tab.n = 0;
    if (d_w_ih) tab.e[tab.n++] = tc16::PlaneTable::Entry{x, TB, I, nullptr, xT, ldx, nullptr, 0};
    for (int d = 0; d < D; ++d) {
      tab.e[tab.n++] = tc16::PlaneTable::Entry{gates + d * slab, TB, 4 * H, nullptr, dGt[d], 4 * H, amax, amax_n};
      if (hh_planes && d_w_hh) tab.e[tab.n++] = tc16::PlaneTable::Entry{hs + d * H, TB, H, nullptr, hsT[d], ldhs, nullptr, 0};
    }
    int rc = tc16::weight_planes_launch(tab, fork.side(0));
    if (rc) return rc;
    if ((rc = fork.chain(0, 1))) return rc;
  }
  cudaStream_t dx_st = st;
  if (dx_bg) {
    static thread_local cudaEvent_t ev[64] = {};
    int dev = 0;
    DVAE_CUDA(cudaGetDevice(&dev));
    DVAE_REQUIRE(dev >= 0 && dev < 64, "dvae_lstm_seq_bwd: device %d", dev);
    if (!ev[dev]) DVAE_CUDA(cudaEventCreateWithFlags(&ev[dev], cudaEventDisableTiming));
    DVAE_CUDA(cudaEventRecord(ev[dev], st));
    DVAE_CUDA(cudaStreamWaitEvent(g_dx_stream, ev[dev], 0));
    dx_st = g_dx_stream;
  }
  for (int d = 0; d < D; ++d) {
    const float* dG = gates + d * slab;
    int rc;
    if (d_x && !(dx_pair && d == 1)) {
      GemmHints ghx = dx_st == st ? gh : gh_bg;
      ghx.c_zeroed = dx_zeroed;
      if (dx_pair) { ghx.atomic_out = true; ghx.concurrency = 2; }
      rc = linear_impl_ex(dG, 4 * H, 0, w_ih[d], I, 1, d_x, lddx, T * B, I, 4 * H, nullptr, nullptr, (d == 0 && !dx_pair) ? 0.f : 1.f, 0, ghx, dx_st);
      if (rc) return rc;
      if (dx_pair && (rc = fork.wait_mark())) return rc;
    }
    if (d_w_ih && d_w_ih[d]) {
      if (dw_planes)
        rc = tc16::linear_planes(dGt[d], xT, d_w_ih[d], I, 4 * H, I, TB, nullptr, 0.f, 0, 1.f, 1.f, nullptr, false, 16, fork.side(0), 0, 0,
                                 gh_bg.max_ctas, 0, 0, amax, amax_n);
      else
        rc = linear_impl_ex(dG, 4 * H, 1, x, ldx, 1, d_w_ih[d], I, 4 * H, I, T * B, nullptr, nullptr, 0.f, 0, gh_bg, fork.side(0));
      if (rc) return rc;
    }
    if (d_w_hh && d_w_hh[d]) {
      cudaStream_t s1 = fork.side(1);
      // h_prev[t] = hs at the previously traversed step (zero / h0 at the first one)
      bool wrote = false;
      if (T > 1) {
        const float* dGs = d == 0 ? dG + (int64_t)B * 4 * H : dG;
        const float* hp = d == 0 ? hs + d * H : hs + (int64_t)B * ldhs + d * H;
        if (hh_planes)      // forward direction: dG rows t >= 1 against h rows t <= T-2 (the reverse direction the other way round)
          rc = tc16::linear_planes(dGt[d], hsT[d], d_w_hh[d], H, 4 * H, H, (T - 1) * B, nullptr, 0.f, 0, 1.f, 1.f, nullptr, false, 16, s1,
                                   d == 0 ? 0 : B / 32, KBt, gh_bg.max_ctas, d == 0 ? B / 32 : 0, KBt, amax, amax_n);
        else
          rc = linear_impl_ex(dGs, 4 * H, 1, hp, ldhs, 1, d_w_hh[d], H, 4 * H, H, (T - 1) * B, nullptr, nullptr, 0.f, 0, gh_bg, s1);
        if (rc) return rc;
        wrote = true;
      }
      if (h0) {
        const float* dG0 = d == 0 ? dG : dG + (int64_t)(T - 1) * B * 4 * H;
        rc = linear_impl_ex(dG0, 4 * H, 1, h0 + d * dir0, ld0, 1, d_w_hh[d], H, 4 * H, H, B, nullptr, nullptr, wrote ? 1.f : 0.f, 0, gh_bg, s1);
        if (rc) return rc;
        wrote = true;
      }
      if (!wrote) DVAE_CUDA(cudaMemsetAsync(d_w_hh[d], 0, sizeof(float) * 4 * H * H, s1));
    }
    cudaStream_t s2 = fork.side(2);
    if (d_b_ih && d_b_ih[d]) {
      rc = colsum_impl(dG, 4 * H, T * B, 4 * H, d_b_ih[d], 0.f, s2);
      if (rc) return rc;
      if (d_b_hh && d_b_hh[d]) DVAE_CUDA(cudaMemcpyAsync(d_b_hh[d], d_b_ih[d], sizeof(float) * 4 * H, cudaMemcpyDeviceToDevice, s2));
    } else if (d_b_hh && d_b_hh[d]) {
      rc = colsum_impl(dG, 4 * H, T * B, 4 * H, d_b_hh[d], 0.f, s2);
      if (rc) return rc;
    }
  }
  {
    int rc = fork.join_or_defer();
    if (rc) return rc;
  }
  return DVAE_OK;
}

// gates_t [B,4H] pre-activations -> post-activation gates; c = f * c_prev + i * g; h = o * tanh(c).  One thread = 4 units.
__global__ void lstm_cell_step_kernel(float* __restrict__ gates_t, const float* __restrict__ c_prev, int64_t ldc, float* __restrict__ cs_t,
                                      float* __restrict__ hs_t, int B, int H) {
  const int HQ = H / 4, idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * HQ) return;
  const int b = idx / HQ, u0 = (idx % HQ) * 4;
  float* g = gates_t + (int64_t)b * 4 * H + u0;
  float4 gi = *reinterpret_cast<float4*>(g), gf = *reinterpret_cast<float4*>(g + H), gg = *reinterpret_cast<float4*>(g + 2 * H),
         go = *reinterpret_cast<float4*>(g + 3 * H);
  float4 c = c_prev ? *reinterpret_cast<const float4*>(c_prev + (int64_t)b * ldc + u0) : make_float4(0.f, 0.f, 0.f, 0.f), h;
#define DVAE_CELL(x)                                                                  \
  gi.x = sigmoidf_(gi.x); gf.x = sigmoidf_(gf.x); gg.x = tanhf(gg.x); go.x = sigmoidf_(go.x); \
  c.x = fmaf(gf.x, c.x, gi.x * gg.x); h.x = go.x * tanhf(c.x);
  DVAE_CELL(x) DVAE_CELL(y) DVAE_CELL(z) DVAE_CELL(w)
#undef DVAE_CELL
  *reinterpret_cast<float4*>(g) = gi; *reinterpret_cast<float4*>(g + H) = gf; *reinterpret_cast<float4*>(g + 2 * H) = gg;
  *reinterpret_cast<float4*>(g + 3 * H) = go;
  *reinterpret_cast<float4*>(cs_t + (int64_t)b * H + u0) = c;
  *reinterpret_cast<float4*>(hs_t + (int64_t)b * H + u0) = h;
}

// One time step of one (uni-directional) layer on the full-sequence buffers: used by sampled decoding, where step
// t+1's input token is only known after step t's vocabulary sample (vae/model.py:457-472).
int lstm_step_impl(const float* x, int64_t ldx, int t, int T, int B, int I, int H, const float* w_ih, const float* w_hh,
                   const float* b_ih, const float* b_hh, const float* h0, const float* c0, int64_t ld0, float* hs,
                   float* gates, float* cs, float* ws, cudaStream_t st) {
  DVAE_REQUIRE(x && w_ih && w_hh && hs && gates && cs && ws, "dvae_lstm_step: null pointer");
  DVAE_REQUIRE(t >= 0 && t < T && B > 0 && I > 0 && H > 0, "dvae_lstm_step: bad shape");
  int rc = linear_impl(x + (int64_t)t * B * ldx, ldx, 0, w_ih, I, 0, gates + (int64_t)t * B * 4 * H, 4 * H, B, 4 * H, I, b_ih, b_hh,
                       0.f, 0, st);
  if (rc) return rc;
  const int64_t sf = (int64_t)B * H;
  // Large batches (inference at B = 1024): the recurrent product is a dense contraction too -- gates[t] += h_{t-1} . W_hh^T on
  // the tensor cores (W_hh arrives as registered weight planes when the caller registered it), then an element-wise cell
  // kernel; the SIMT step kernel below took 32 us per layer and step at B = 1024, H = 256
  {
    const void* ptrs[] = {x, w_hh, h0, c0, hs, gates, cs};
    bool aligned = H % 4 == 0 && ld0 % 4 == 0;
    for (const void* q : ptrs) aligned = aligned && ((reinterpret_cast<uintptr_t>(q) & 15) == 0);
    const char* e = getenv("DVAE_LSTM_IMPL");
    if (aligned && B >= 256 && H >= 64 && !force_simt_gemm() && !(e && !strcmp(e, "step"))) {
      float* gates_t = gates + (int64_t)t * B * 4 * H;
      const float* h_prev = t == 0 ? h0 : hs + (int64_t)(t - 1) * sf;
      const float* c_prev = t == 0 ? c0 : cs + (int64_t)(t - 1) * sf;
      if (h_prev && (rc = linear_impl(h_prev, t == 0 ? ld0 : H, 0, w_hh, H, 0, gates_t, 4 * H, B, 4 * H, H, nullptr, nullptr, 1.f, 0, st)))
        return rc;
      lstm_cell_step_kernel<<<ceil_div((int64_t)B * (H / 4), 256), 256, 0, st>>>(gates_t, c_prev, t == 0 ? ld0 : H, cs + (int64_t)t * sf,
                                                                               hs + (int64_t)t * sf, B, H);
      DVAE_LAUNCH_CHECK();
      return DVAE_OK;
    }
  }
  const float *h_in, *c_in;
  if (t == 0) {
    const int nthr = 256, nblk = ceil_div(sf, nthr);
    copy_state_kernel<<<nblk, nthr, 0, st>>>(h0, ld0, 0, ws, H, sf, 1, B, H);
    DVAE_LAUNCH_CHECK();
    copy_state_kernel<<<nblk, nthr, 0, st>>>(c0, ld0, 0, ws + sf, H, sf, 1, B, H);
    DVAE_LAUNCH_CHECK();
    h_in = ws; c_in = ws + sf;
  } else {
    h_in = hs + (int64_t)(t - 1) * sf; c_in = cs + (int64_t)(t - 1) * sf;
  }
  FwdStepArgs a;
  a.w_hh[0] = w_hh; a.w_hh[1] = w_hh;
  a.gates = gates; a.cs = cs; a.hs = hs; a.ldhs = H; a.lengths = nullptr; a.T = T; a.B = B; a.H = H; a.s = t;
  a.h_in = h_in; a.c_in = c_in; a.h_out = ws + 2 * sf; a.c_out = ws + 3 * sf;
  lstm_step_fwd_kernel<<<dim3(ceil_div(H, 16), ceil_div(B, kStepRows), 1), kStepThreads, 0, st>>>(a);
  DVAE_LAUNCH_CHECK();
  return DVAE_OK;
}

}  // namespace dvae

extern "C" int dvae_lstm_step(const float* x, int64_t ldx, int t, int T, int B, int I, int H, const float* w_ih,
                              const float* w_hh, const float* b_ih, const float* b_hh, const float* h0, const float* c0,
                              int64_t ld0, float* hs, float* gates, float* cs, float* state_ws, void* stream) {
  return dvae::lstm_step_impl(x, ldx, t, T, B, I, H, w_ih, w_hh, b_ih, b_hh, h0, c0, ld0, hs, gates, cs, state_ws,
                              (cudaStream_t)stream);
}

extern "C" int64_t dvae_lstm_state_ws_floats(int B, int H, int D) {
  // + 8 rotating sets of per-CTA max |dG| slots + the operand planes of the large-H path (0 for H it does not take)
  return dvae::planes_ws_offset(B, H, D) + dvae::planes_lstm_ws_floats(B, H, D);
}

extern "C" int dvae_lstm_seq_fwd(const float* x, int64_t ldx, int T, int B, int I, int H, int D,
                                 const float* const* w_ih, const float* const* w_hh, const float* const* b_ih,
                                 const float* const* b_hh, const float* h0, const float* c0, int64_t ld0,
                                 int64_t dir0, const int64_t* lengths, float* hs, int64_t ldhs, float* hn,
                                 float* cn, int64_t ldn, int64_t dirn, float* gates, float* cs, float* state_ws,
                                 void* stream) {
  return dvae::lstm_seq_fwd_impl(x, ldx, T, B, I, H, D, w_ih, w_hh, b_ih, b_hh, h0, c0, ld0, dir0, lengths, hs,
                                 ldhs, hn, cn, ldn, dirn, gates, cs, state_ws, false, (cudaStream_t)stream);
}

// The two halves of dvae_lstm_seq_fwd separately, so that a caller can run a layer's input projection early, on another
// stream (the decoder's layer-0 projection under teacher forcing depends on the input tokens only, not on the encoder):
// dvae_lstm_input_proj fills `gates`; dvae_lstm_seq_fwd_ex with flags bit 0 set then runs the recurrence alone.
extern "C" int dvae_lstm_input_proj(const float* x, int64_t ldx, int T, int B, int I, int H, int D,
                                    const float* const* w_ih, const float* const* b_ih, const float* const* b_hh,
                                    float* gates, void* stream) {
  return dvae::lstm_input_proj_impl(x, ldx, T, B, I, H, D, w_ih, b_ih, b_hh, gates, (cudaStream_t)stream);
}

extern "C" int dvae_lstm_seq_fwd_ex(const float* x, int64_t ldx, int T, int B, int I, int H, int D,
                                    const float* const* w_ih, const float* const* w_hh, const float* const* b_ih,
                                    const float* const* b_hh, const float* h0, const float* c0, int64_t ld0,
                                    int64_t dir0, const int64_t* lengths, float* hs, int64_t ldhs, float* hn,
                                    float* cn, int64_t ldn, int64_t dirn, float* gates, float* cs, float* state_ws,
                                    int flags, void* stream) {
  return dvae::lstm_seq_fwd_impl(x, ldx, T, B, I, H, D, w_ih, w_hh, b_ih, b_hh, h0, c0, ld0, dir0, lengths, hs,
                                 ldhs, hn, cn, ldn, dirn, gates, cs, state_ws, (flags & 1) != 0, (cudaStream_t)stream);
}

extern "C" int dvae_lstm_seq_bwd(const float* x, int64_t ldx, int T, int B, int I, int H, int D,
                                 const float* const* w_ih, const float* const* w_hh, const float* h0,
                                 const float* c0, int64_t ld0, int64_t dir0, const int64_t* lengths,
                                 const float* hs, int64_t ldhs, float* gates, const float* cs, const float* d_hs,
                                 int64_t lddhs, const float* d_hn, const float* d_cn, int64_t ldn, int64_t dirn,
                                 float* d_x, int64_t lddx, float* const* d_w_ih, float* const* d_w_hh,
                                 float* const* d_b_ih, float* const* d_b_hh, float* d_h0, float* d_c0,
                                 int64_t ldd0, int64_t dird0, float* state_ws, void* stream) {
  return dvae::lstm_seq_bwd_impl(x, ldx, T, B, I, H, D, w_ih, w_hh, h0, c0, ld0, dir0, lengths, hs, ldhs, gates, cs,
                                 d_hs, lddhs, d_hn, d_cn, ldn, dirn, d_x, lddx, d_w_ih, d_w_hh, d_b_ih, d_b_hh,
                                 d_h0, d_c0, ldd0, dird0, state_ws, nullptr, (cudaStream_t)stream);
}

extern "C" int dvae_lstm_bwd_dx_stream(void* stream) {
  dvae::g_dx_stream = (cudaStream_t)stream;
  return DVAE_OK;
}

extern "C" int64_t dvae_lstm_bwd_planes_ws_floats(int T, int B, int I, int H, int D) {
  const int TB = T * B;
  return dvae::tc16::plane_floats(I, TB) + (int64_t)D * (dvae::tc16::plane_floats(4 * H, TB) + dvae::tc16::plane_floats(H, TB));
}

extern "C" int dvae_lstm_seq_bwd_ex(const float* x, int64_t ldx, int T, int B, int I, int H, int D,
                                    const float* const* w_ih, const float* const* w_hh, const float* h0,
                                    const float* c0, int64_t ld0, int64_t dir0, const int64_t* lengths,
                                    const float* hs, int64_t ldhs, float* gates, const float* cs, const float* d_hs,
                                    int64_t lddhs, const float* d_hn, const float* d_cn, int64_t ldn, int64_t dirn,
                                    float* d_x, int64_t lddx, float* const* d_w_ih, float* const* d_w_hh,
                                    float* const* d_b_ih, float* const* d_b_hh, float* d_h0, float* d_c0,
                                    int64_t ldd0, int64_t dird0, float* state_ws, float* planes_ws, void* stream) {
  return dvae::lstm_seq_bwd_impl(x, ldx, T, B, I, H, D, w_ih, w_hh, h0, c0, ld0, dir0, lengths, hs, ldhs, gates, cs,
                                 d_hs, lddhs, d_hn, d_cn, ldn, dirn, d_x, lddx, d_w_ih, d_w_hh, d_b_ih, d_b_hh,
                                 d_h0, d_c0, ldd0, dird0, state_ws, planes_ws, (cudaStream_t)stream);
}
