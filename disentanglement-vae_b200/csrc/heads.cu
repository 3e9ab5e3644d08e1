// Fused latent heads (see include/dvae_b200.h, dvae_latent_heads_fwd/bwd).
//
// Both directions run on clusters of 8 CTAs; a cluster owns R batch rows and splits the latents, the z2hidden columns
// and the context columns between its CTAs, so that every weight element is read by one CTA of the cluster.
//
// Forward, ONE kernel: CTA `rank` computes the (mu, raw) projections of its latents over the full context width,
// logvar = tanh(raw), the reparameterised sample z = mu + eps * exp(logvar) and the KL terms; z (and, for rank 0, the KL
// terms) is all-gathered over distributed shared memory; rank 0 computes the discriminator logits, BCE/CE loss and
// accuracy, and every CTA writes its 1/8 of the decoder-initial-state columns tanh(z . W_z2h^T + b).  Per-cluster
// partial sums are combined in cluster order by the last cluster to arrive, so the scalars are bit-reproducible.
//
// Backward, ONE kernel for the chain the encoder's backward waits for: d_pre = d_hid (1 - hid^2); d_z = d_pre W_z2h for
// the CTA's latents; the per-element step (discriminator gradient, KL, the optional upstream extras, d_raw =
// dlv (1 - lv^2)); an all-gather of dp over distributed shared memory; d_ctx = dp W_c2p for the CTA's 1/8 of the context
// columns (no atomics: deterministic).  d_pre, dp and dl go to the workspace, from where the weight and bias gradients
// run on side streams.
#include <cooperative_groups.h>
#include "common.cuh"

namespace cg = cooperative_groups;

namespace dvae {

int linear_impl(const float* A, int64_t lda, int trans_a, const float* B, int64_t ldb, int trans_b, float* C,
                int64_t ldc, int M, int N, int K, const float* bias, const float* bias2, float beta, int act,
                cudaStream_t st);
int colsum_impl(const float* X, int64_t ldx, int M, int N, float* out, float beta, cudaStream_t st);

constexpr int kCl = 8;                // CTAs per cluster
constexpr int kHT = 512;              // threads per CTA
constexpr int kHW = kHT / 32;
constexpr int kMaxDscOut = 64;
constexpr size_t kHeadsSmemTarget = 160 * 1024;     // R is halved until a CTA's shared memory fits this

struct HeadsMeta {
  int S, Z, OD;                       // spaces, total latent dim, total discriminator outputs
  int zdim[DVAE_MAX_SPACES];
  int zoff[DVAE_MAX_SPACES];          // column offset of the space inside [B,Z]
  int dout[DVAE_MAX_SPACES];          // discriminator output dim (0 = none)
  int doff[DVAE_MAX_SPACES];          // column offset inside dsc_logits / b_dsc
  int dwoff[DVAE_MAX_SPACES];         // float offset inside w_dsc
  int dlab[DVAE_MAX_SPACES];          // index of the label row ([n_dsc][B])
};

static int make_meta(int S, const int* space_dims, const int* dsc_out, HeadsMeta* m) {
  DVAE_REQUIRE(S > 0 && S <= DVAE_MAX_SPACES, "latent heads: S=%d out of range", S);
  m->S = S;
  int z = 0, od = 0, w = 0, nl = 0;
  for (int s = 0; s < S; ++s) {
    DVAE_REQUIRE(space_dims[s] > 0, "latent heads: space %d has dim %d", s, space_dims[s]);
    m->zdim[s] = space_dims[s]; m->zoff[s] = z; z += space_dims[s];
    int o = dsc_out ? dsc_out[s] : 0;
    m->dout[s] = o; m->doff[s] = od; m->dwoff[s] = w; m->dlab[s] = o > 0 ? nl : -1;
    if (o > 0) { od += o; w += o * space_dims[s]; ++nl; }
  }
  DVAE_REQUIRE(od <= kMaxDscOut, "latent heads: %d discriminator outputs > %d", od, kMaxDscOut);
  m->Z = z; m->OD = od;
  return DVAE_OK;
}


// The LSTM recurrence that follows on the stream (decoder layer 0 after the forward, encoder layer Le-1 after the backward)
// is launched programmatically: it may start its prologue (barriers, TMEM allocation, resident weights) now and waits for
// this grid to complete before it reads anything written here.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

static inline int round4(int n) { return (n + 3) & ~3; }

__device__ __forceinline__ int space_of(const HeadsMeta& m, int zi) {
  int s = 0;
  while (s + 1 < m.S && zi >= m.zoff[s + 1]) ++s;
  return s;
}

__device__ __forceinline__ int dsc_space_of(const HeadsMeta& m, int od) {
  int s = 0;
  while (!(m.dout[s] > 0 && od >= m.doff[s] && od < m.doff[s] + m.dout[s])) ++s;
  return s;
}

// The cluster's share of n items for CTA `rank`: [lo, lo + cnt), blocks of ceil(n / 8)
__device__ __forceinline__ void cl_range(int n, int rank, int& lo, int& cnt) {
  const int per = (n + kCl - 1) / kCl;
  lo = min(n, rank * per);
  cnt = min(n, lo + per) - lo;
}

// Warp-wide sums of N per-lane values (N a power of two <= 32) by halving exchanges: at offset O a lane keeps one half of
// its values, hands the other half to its partner and adds what it receives (N - 1 shuffles in all, against 5 N for N
// separate reductions).  Afterwards v[0] of lane l holds the total of value l >> (5 - log2 N).
template <int N, int O = 16>
__device__ __forceinline__ void warp_reduce_scatter(float* v, int lane) {
  if constexpr (N > 1) {
    const bool hi = (lane & O) != 0;
#pragma unroll
    for (int i = 0; i < N / 2; ++i) {
      const float send = hi ? v[i] : v[i + N / 2], keep = hi ? v[i + N / 2] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, O);
    }
  } else {
    v[0] += __shfl_xor_sync(0xffffffffu, v[0], O);
  }
  if constexpr (O > 1) warp_reduce_scatter<(N > 1 ? N / 2 : 1), O / 2>(v, lane);
}

// out(r, j, sum_k X[r][k] W[rows[j] * K + k]) for j < nj.  W rows are contiguous in k: one warp per (Q rows, k-slice),
// lanes stride k (16-byte loads when aligned) so that each row is read coalesced once; the k-slices' partials are added
// in a fixed order.  Q = 4 rows share each X load; 2 at R = 16, where 4 x 16 accumulators would spill.
// red: >= ceil(nj / Q) * Q * KS * R floats (host: red_floats()).
template <int R, class Out>
__device__ void row_dot(const float* X, int ldx, int K, const float* __restrict__ W, const int* rows, int nj, float* red,
                        Out out) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int Q = R >= 16 ? 2 : 4;
  const int nq = (nj + Q - 1) / Q, KS = nq >= kHW ? 1 : kHW / max(nq, 1);
  const bool vec = (K & 3) == 0 && (reinterpret_cast<uintptr_t>(W) & 15) == 0;
  for (int u = warp; u < nq * KS; u += kHW) {
    const int q0 = (u / KS) * Q, ks = u % KS;
    const float* w[Q];
#pragma unroll
    for (int q = 0; q < Q; ++q) w[q] = W + (int64_t)rows[min(q0 + q, nj - 1)] * K;
    float acc[Q][R];
#pragma unroll
    for (int q = 0; q < Q; ++q)
#pragma unroll
      for (int r = 0; r < R; ++r) acc[q][r] = 0.f;
    if (vec) {
#pragma unroll 2
      for (int k = (ks * 32 + lane) * 4; k < K; k += KS * 128) {
        float4 wv[Q];
#pragma unroll
        for (int q = 0; q < Q; ++q) wv[q] = __ldg(reinterpret_cast<const float4*>(w[q] + k));
#pragma unroll
        for (int r = 0; r < R; ++r) {
          const float4 c = *reinterpret_cast<const float4*>(X + r * ldx + k);
#pragma unroll
          for (int q = 0; q < Q; ++q) {
            acc[q][r] = fmaf(c.x, wv[q].x, acc[q][r]); acc[q][r] = fmaf(c.y, wv[q].y, acc[q][r]);
            acc[q][r] = fmaf(c.z, wv[q].z, acc[q][r]); acc[q][r] = fmaf(c.w, wv[q].w, acc[q][r]);
          }
        }
      }
    } else {
      for (int k = ks * 32 + lane; k < K; k += KS * 32) {
        float wv[Q];
#pragma unroll
        for (int q = 0; q < Q; ++q) wv[q] = __ldg(w[q] + k);
#pragma unroll
        for (int r = 0; r < R; ++r) {
          const float c = X[r * ldx + k];
#pragma unroll
          for (int q = 0; q < Q; ++q) acc[q][r] = fmaf(c, wv[q], acc[q][r]);
        }
      }
    }
    constexpr int N = Q * R, SH = N >= 32 ? 0 : N >= 16 ? 1 : N >= 8 ? 2 : N >= 4 ? 3 : N >= 2 ? 4 : 5;
    warp_reduce_scatter<N>(&acc[0][0], lane);
    if ((lane & ((1 << SH) - 1)) == 0) {
      const int i = lane >> SH;          // value q * R + r
      red[(ks * nq * Q + q0 + i / R) * R + i % R] = acc[0][0];
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < nj * R; i += kHT) {
    const int j = i / R, r = i % R;
    float s = 0.f;
    for (int ks = 0; ks < KS; ++ks) s += red[(ks * nq * Q + j) * R + r];
    out(r, j, s);
  }
  __syncthreads();
}

// out(r, c, sum_k X[r][k] W[(c0 + c) * cs + k * ks]) for c < nc, k < K, where X rows (ldx floats, 16-byte aligned) are
// zero-padded up to a multiple of 4.  Thread t owns column slot t % NCP (NCP = nc rounded up to a power of two, at most
// kHT) and the k-chunks of 4 values g, g + JG, ... with g = t / NCP, JG = kHT / NCP; neighbouring lanes own neighbouring
// columns, so W is read coalesced when cs == 1 and the X loads are broadcasts.  The partials are added over the lanes of
// a warp by shuffles and then over the warps in a fixed order.  red: >= kHT * R floats.
template <int R, class Out>
__device__ void col_dot(const float* X, int ldx, int K, const float* __restrict__ W, int64_t cs, int64_t ks, int c0, int nc,
                        float* red, Out out) {
  constexpr int U = R >= 16 ? 2 : 4;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int ncp = 1;
  while (ncp < nc && ncp < kHT) ncp <<= 1;
  const int JG = kHT / ncp, K4 = (K + 3) >> 2, GW = ncp >= 32 ? JG : kHW;
  const int slot = tid % ncp, g = tid / ncp;
  const bool vec = ks == 1 && (cs & 3) == 0 && ((reinterpret_cast<uintptr_t>(W) + 4 * c0 * cs) & 15) == 0;
  for (int cb = 0; cb < nc; cb += ncp) {
    const int c = cb + slot;
    float acc[R];
#pragma unroll
    for (int r = 0; r < R; ++r) acc[r] = 0.f;
    if (c < nc) {
      const float* w = W + (int64_t)(c0 + c) * cs;
      for (int kc0 = g; kc0 < K4; kc0 += U * JG) {      // the weights of U chunks in flight, then their products
        float wv[U][4];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int k = (kc0 + u * JG) * 4;
          if (vec && k + 3 < K) {         // a row contiguous in k: one 16-byte load per chunk
            const float4 v = __ldg(reinterpret_cast<const float4*>(w + k));
            wv[u][0] = v.x; wv[u][1] = v.y; wv[u][2] = v.z; wv[u][3] = v.w;
          } else {
#pragma unroll
            for (int q = 0; q < 4; ++q) wv[u][q] = kc0 + u * JG < K4 && k + q < K ? __ldg(w + (int64_t)(k + q) * ks) : 0.f;
          }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int kc = kc0 + u * JG;
          if (kc >= K4) break;
#pragma unroll
          for (int r = 0; r < R; ++r) {
            const float4 x = *reinterpret_cast<const float4*>(X + r * ldx + kc * 4);
            acc[r] = fmaf(x.x, wv[u][0], acc[r]); acc[r] = fmaf(x.y, wv[u][1], acc[r]);
            acc[r] = fmaf(x.z, wv[u][2], acc[r]); acc[r] = fmaf(x.w, wv[u][3], acc[r]);
          }
        }
      }
    }
    if (ncp < 32) {
#pragma unroll
      for (int r = 0; r < R; ++r)
        for (int o = ncp; o < 32; o <<= 1) acc[r] += __shfl_xor_sync(0xffffffffu, acc[r], o);
    }
    if (ncp >= 32 || lane < ncp) {
      const int gw = ncp >= 32 ? g : warp;
#pragma unroll
      for (int r = 0; r < R; ++r) red[(gw * R + r) * ncp + slot] = acc[r];
    }
    __syncthreads();
    for (int i = tid; i < R * ncp; i += kHT) {
      const int r = i / ncp, cc = i % ncp;
      if (cb + cc >= nc) continue;
      float s = 0.f;
      for (int q = 0; q < GW; ++q) s += red[(q * R + r) * ncp + cc];
      out(r, cb + cc, s);
    }
    __syncthreads();
  }
}

// shared-memory floats of row_dot / col_dot's partials
static int red_floats(int R, int nj) {
  const int Q = R >= 16 ? 2 : 4, nq = (nj + Q - 1) / Q, KS = nq >= kHW ? 1 : kHW / (nq > 0 ? nq : 1);
  const int rd = nq * Q * KS * R;
  return round4(rd > kHT * R ? rd : kHT * R);
}

struct HeadsFwdArgs {
  const float *ctx, *w_c2p, *b_c2p, *eps, *w_dsc, *b_dsc, *labels, *kl_w, *w_z2h, *b_z2h;
  float *z, *mu, *logvar, *hid, *dsc_logits, *scalars, *ws;
  int B, C, H2L, red;
};

static size_t heads_fwd_smem(int R, int C, const HeadsMeta& m) {
  const int zcm = (m.Z + kCl - 1) / kCl;
  return sizeof(float) * ((size_t)R * round4(C) + red_floats(R, 2 * zcm) + R * round4(m.Z) + R * m.Z + 4 * R * zcm +
                          R * (m.OD > 0 ? m.OD : 1)) + sizeof(int) * 2 * zcm;
}

template <int R>
__global__ void __cluster_dims__(kCl, 1, 1) __launch_bounds__(kHT, 1) heads_fwd_kernel(HeadsFwdArgs a, HeadsMeta m) {
  extern __shared__ __align__(16) float sm[];
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank();
  const int C = a.C, Z = m.Z, S = m.S, OD = m.OD, B = a.B, tid = threadIdx.x;
  const int cl = blockIdx.x / kCl, ncl = gridDim.x / kCl, b0 = cl * R;
  const int ldc = (C + 3) & ~3, ldz = (Z + 3) & ~3, zcm = (Z + kCl - 1) / kCl;
  int z0, zc;
  cl_range(Z, rank, z0, zc);
  float* ctx_s = sm;                        // [R][ldc] context rows
  float* red = ctx_s + R * ldc;             // [a.red] partial sums
  float* z_s = red + a.red;                 // [R][ldz] z of every latent (all-gathered)
  float* klt_s = z_s + R * ldz;             // [R][Z] KL terms of every latent (rank 0 gathers them)
  float* par_s = klt_s + R * Z;             // [R][2 zcm] this CTA's mu | raw
  float* zl_s = par_s + 2 * R * zcm;        // [R][zcm] this CTA's z
  float* kl_s = zl_s + R * zcm;             // [R][zcm] this CTA's KL terms
  float* lg_s = kl_s + R * zcm;             // [R][OD]
  int* rows_s = reinterpret_cast<int*>(lg_s + R * (OD > 0 ? OD : 1));     // [2 zc] W_c2p row of each local column
  pdl_launch_dependents();

  for (int j = tid; j < 2 * zc; j += kHT) {
    const int zi = z0 + j % zc, s = space_of(m, zi);
    rows_s[j] = 2 * m.zoff[s] + (j < zc ? 0 : m.zdim[s]) + zi - m.zoff[s];
  }
  if ((C & 3) == 0 && (reinterpret_cast<uintptr_t>(a.ctx) & 15) == 0) {
    for (int i = tid; i < R * C / 4; i += kHT) {
      const int r = i / (C / 4), k = (i % (C / 4)) * 4;
      *reinterpret_cast<float4*>(ctx_s + r * ldc + k) =
          b0 + r < B ? __ldg(reinterpret_cast<const float4*>(a.ctx + (int64_t)(b0 + r) * C + k)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  } else {
    for (int i = tid; i < R * C; i += kHT) {
      const int r = i / C, k = i % C;
      ctx_s[r * ldc + k] = b0 + r < B ? a.ctx[(int64_t)(b0 + r) * C + k] : 0.f;
    }
  }
  __syncthreads();
  // (mu, raw) of this CTA's latents over the full context width
  row_dot<R>(ctx_s, ldc, C, a.w_c2p, rows_s, 2 * zc, red,
             [&](int r, int j, float s) { par_s[r * 2 * zcm + j] = s + a.b_c2p[rows_s[j]]; });
  // reparameterisation + KL terms
  for (int i = tid; i < R * zc; i += kHT) {
    const int r = i / zc, j = i % zc, zi = z0 + j, b = b0 + r;
    const float mu = par_s[r * 2 * zcm + j];
    const float lv = tanhf(par_s[r * 2 * zcm + zc + j]);
    const float e = expf(lv);
    float zz = 0.f, kt = 0.f;
    if (b < B) {
      zz = fmaf(a.eps[(int64_t)b * Z + zi], e, mu);
      kt = 0.5f * (e + mu * mu - 1.f - lv);
      a.z[(int64_t)b * Z + zi] = zz;
      a.mu[(int64_t)b * Z + zi] = mu;
      a.logvar[(int64_t)b * Z + zi] = lv;
    }
    zl_s[r * zcm + j] = zz;
    kl_s[r * zcm + j] = kt;
  }
  // all-gather z (and the KL terms into rank 0) over distributed shared memory
  cluster.sync();
  for (int i = tid; i < R * ldz; i += kHT) {
    const int r = i / ldz, zi = i % ldz, p = zi / zcm, j = zi - p * zcm;
    float v = 0.f;
    if (zi < Z) {
      v = cluster.map_shared_rank(zl_s, p)[r * zcm + j];
      if (rank == 0) klt_s[r * Z + zi] = cluster.map_shared_rank(kl_s, p)[r * zcm + j];
    }
    z_s[i] = v;
  }
  cluster.sync();           // no CTA leaves or overwrites its z while a peer may still read it
  // discriminator logits, then this cluster's partial sums and its arrival (rank 0)
  unsigned int arrived = 0;
  if (rank == 0) {
    for (int i = tid; i < R * OD; i += kHT) {
      const int r = i / OD, od = i % OD, b = b0 + r, s = dsc_space_of(m, od), o = od - m.doff[s];
      const float* w = a.w_dsc + m.dwoff[s] + o * m.zdim[s];
      float acc = a.b_dsc[od];
      for (int d = 0; d < m.zdim[s]; ++d) acc = fmaf(z_s[r * ldz + m.zoff[s] + d], w[d], acc);
      lg_s[i] = acc;
      if (b < B) a.dsc_logits[(int64_t)b * OD + od] = acc;
    }
    __syncthreads();
    // warp s sums space s: KL terms strided over the lanes, one row per lane for the discriminator; fixed order
    const int warp = tid >> 5, lane = tid & 31, nr = min(R, B - b0);
    if (warp < S) {
      const int s = warp, zs = m.zdim[s];
      float kl = 0.f, dl = 0.f, da = 0.f;
      for (int i = lane; i < nr * zs; i += 32) kl += klt_s[(i / zs) * Z + m.zoff[s] + i % zs];
      if (m.dout[s] > 0 && a.labels && lane < nr) {
        const float y = a.labels[(int64_t)m.dlab[s] * B + b0 + lane];
        const float* l = lg_s + lane * OD + m.doff[s];
        if (m.dout[s] == 1) {
          const float x = l[0];
          dl = fmaxf(x, 0.f) - x * y + log1pf(expf(-fabsf(x)));
          da = ((x > 0.f ? 1.f : 0.f) == y) ? 1.f : 0.f;
        } else {
          float mx = l[0];
          int am = 0;
          for (int o = 1; o < m.dout[s]; ++o)
            if (l[o] > mx) { mx = l[o]; am = o; }
          float se = 0.f;
          for (int o = 0; o < m.dout[s]; ++o) se += expf(l[o] - mx);
          const int yi = (int)y;
          dl = mx + logf(se) - l[yi];
          da = (am == yi) ? 1.f : 0.f;
        }
      }
      kl = warp_sum(kl); dl = warp_sum(dl); da = warp_sum(da);
      if (lane == 0) {
        float* part = a.ws + 4 + (int64_t)cl * 3 * S;
        part[s] = kl; part[S + s] = dl; part[2 * S + s] = da;
      }
    }
    __threadfence();
    __syncthreads();
    // atomicInc wraps to 0 on the last arrival: the counter re-arms itself (no memset node in front of the kernel); the
    // caller zero-fills ws once before the first call.  Its result is first needed after z2hidden.
    if (tid == 0) arrived = atomicInc(reinterpret_cast<unsigned int*>(a.ws), ncl - 1);
  }
  // decoder initial state: this CTA's 1/8 of the columns of hid = tanh(z . W_z2h^T + b_z2h)
  int h0, hc;
  cl_range(a.H2L, rank, h0, hc);
  col_dot<R>(z_s, ldz, Z, a.w_z2h, Z, 1, h0, hc, red, [&](int r, int c, float s) {
    if (b0 + r < B) a.hid[(int64_t)(b0 + r) * a.H2L + h0 + c] = tanhf(s + a.b_z2h[h0 + c]);
  });
  if (rank != 0) return;
  // the last cluster to arrive combines the partials in cluster order
  __shared__ int is_last;
  if (tid == 0) is_last = arrived == (unsigned int)ncl - 1;
  __syncthreads();
  if (!is_last) return;
  // all threads fetch the partials into shared memory in parallel; thread 0 then adds them in cluster order
  const int n_part = ncl * 3 * S;
  const bool staged = n_part <= R * ldc;          // ctx_s is free by now
  __threadfence();
  if (staged)
    for (int i = tid; i < n_part; i += kHT) ctx_s[i] = __ldcg(a.ws + 4 + i);
  __syncthreads();
  if (tid == 0) {
    float wkl = 0.f, tkl = 0.f, tdl = 0.f;
    for (int s = 0; s < S; ++s) {
      float kl = 0.f, dl = 0.f, da = 0.f;
      for (int c = 0; c < ncl; ++c) {
        if (staged) {
          const float* part = ctx_s + c * 3 * S;
          kl += part[s]; dl += part[S + s]; da += part[2 * S + s];
        } else {
          const float* part = a.ws + 4 + (int64_t)c * 3 * S;
          kl += __ldcg(part + s); dl += __ldcg(part + S + s); da += __ldcg(part + 2 * S + s);
        }
      }
      kl /= (float)B;
      dl /= (float)B;
      da /= (float)B;
      a.scalars[3 + s] = kl;
      a.scalars[3 + S + s] = m.dout[s] > 0 ? dl : 0.f;
      a.scalars[3 + 2 * S + s] = m.dout[s] > 0 ? da : 0.f;
      wkl = fmaf(a.kl_w ? a.kl_w[s] : 0.f, kl, wkl);
      tkl += kl;
      if (m.dout[s] > 0) tdl += dl;
    }
    a.scalars[0] = wkl; a.scalars[1] = tkl; a.scalars[2] = tdl;
  }
}

// ---- backward ---------------------------------------------------------------------------------
struct HeadsBwdArgs {
  const float *w_c2p, *eps, *w_dsc, *labels, *kl_w, *w_z2h, *mu, *logvar, *hid, *dsc_logits, *d_hid;
  const float *d_z_extra, *d_mu_extra, *d_logvar_extra, *d_logits_extra;
  float *d_pre, *dp, *dl, *d_ctx;     // [B,H2L], [B,2Z], [B,OD], [B,C]
  int B, C, H2L, red;
};

static size_t heads_bwd_smem(int R, int H2L, const HeadsMeta& m) {
  const int zcm = (m.Z + kCl - 1) / kCl;
  return sizeof(float) * ((size_t)R * round4(H2L) + red_floats(R, 0) + R * round4(2 * m.Z) + 2 * R * zcm + R * (m.OD > 0 ? m.OD : 1));
}

template <int R>
__global__ void __cluster_dims__(kCl, 1, 1) __launch_bounds__(kHT, 1) heads_bwd_kernel(HeadsBwdArgs a, HeadsMeta m) {
  extern __shared__ __align__(16) float sm[];
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank();
  const int Z = m.Z, OD = m.OD, B = a.B, H2L = a.H2L, tid = threadIdx.x;
  const int b0 = (blockIdx.x / kCl) * R;
  const int ldh = (H2L + 3) & ~3, ldp = (2 * Z + 3) & ~3, zcm = (Z + kCl - 1) / kCl;
  int z0, zc, h0, hc;
  cl_range(Z, rank, z0, zc);
  cl_range(H2L, rank, h0, hc);
  float* dpre_s = sm;                       // [R][ldh] d_pre of the cluster's rows
  pdl_launch_dependents();
  float* red = dpre_s + R * ldh;            // [a.red]
  float* dp_s = red + a.red;                // [R][ldp] dp of every latent (all-gathered)
  float* dpl_s = dp_s + R * ldp;            // [R][2 zcm] this CTA's d_mu | d_raw
  float* g_s = dpl_s + 2 * R * zcm;         // [R][OD] discriminator logit gradients

  // d_pre = d_hid (1 - hid^2): every CTA keeps all columns of its rows, CTA `rank` stores its 1/8 of them
  if ((H2L & 3) == 0 && ((reinterpret_cast<uintptr_t>(a.hid) | reinterpret_cast<uintptr_t>(a.d_hid)) & 15) == 0) {
    const int n4 = H2L / 4;
    int q0, qc;               // this CTA's 1/8 of the 4-column chunks
    cl_range(n4, rank, q0, qc);
#pragma unroll 4
    for (int i = tid; i < R * n4; i += kHT) {
      const int r = i / n4, j = (i % n4) * 4, b = b0 + r;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (b < B) {
        const int64_t e = (int64_t)b * H2L + j;
        const float4 h = __ldg(reinterpret_cast<const float4*>(a.hid + e)), g = __ldg(reinterpret_cast<const float4*>(a.d_hid + e));
        v = make_float4(g.x * (1.f - h.x * h.x), g.y * (1.f - h.y * h.y), g.z * (1.f - h.z * h.z), g.w * (1.f - h.w * h.w));
        if (j / 4 >= q0 && j / 4 < q0 + qc) *reinterpret_cast<float4*>(a.d_pre + e) = v;
      }
      *reinterpret_cast<float4*>(dpre_s + r * ldh + j) = v;
    }
  } else {
    for (int i = tid; i < R * ldh; i += kHT) {
      const int r = i / ldh, j = i % ldh, b = b0 + r;
      float v = 0.f;
      if (b < B && j < H2L) {
        const int64_t e = (int64_t)b * H2L + j;
        const float h = a.hid[e];
        v = a.d_hid[e] * (1.f - h * h);
        if (j >= h0 && j < h0 + hc) a.d_pre[e] = v;
      }
      dpre_s[i] = v;
    }
  }
  // discriminator: d(loss)/d(logits) (+ the upstream extra); rank 0 stores them
  for (int i = tid; i < R * OD; i += kHT) {
    const int r = i / OD, od = i % OD, b = b0 + r;
    if (b >= B) { g_s[i] = 0.f; continue; }
    const int s = dsc_space_of(m, od), o = od - m.doff[s];
    const float* l = a.dsc_logits + (int64_t)b * OD + m.doff[s];
    float g = a.d_logits_extra ? a.d_logits_extra[(int64_t)b * OD + od] : 0.f;
    if (a.labels) {
      const float y = a.labels[(int64_t)m.dlab[s] * B + b];
      if (m.dout[s] == 1) {
        g += (sigmoidf_(l[0]) - y) / (float)B;
      } else {
        float mx = l[0];
        for (int q = 1; q < m.dout[s]; ++q) mx = fmaxf(mx, l[q]);
        float se = 0.f;
        for (int q = 0; q < m.dout[s]; ++q) se += expf(l[q] - mx);
        g += (expf(l[o] - mx) / se - (o == (int)y ? 1.f : 0.f)) / (float)B;
      }
    }
    g_s[i] = g;
    if (rank == 0) a.dl[(int64_t)b * OD + od] = g;
  }
  __syncthreads();
  // d_z = d_pre W_z2h for this CTA's latents, then the per-element step into d_mu | d_raw
  col_dot<R>(dpre_s, ldh, H2L, a.w_z2h, 1, Z, z0, zc, red, [&](int r, int c, float acc) {
    const int b = b0 + r, zi = z0 + c;
    float dmu = 0.f, draw = 0.f;
    if (b < B) {
      const int64_t i = (int64_t)b * Z + zi;
      const int s = space_of(m, zi), d = zi - m.zoff[s], zs = m.zdim[s];
      float dz = acc + (a.d_z_extra ? a.d_z_extra[i] : 0.f);
      if (m.dout[s] > 0) {
        const float* w = a.w_dsc + m.dwoff[s];
        for (int o = 0; o < m.dout[s]; ++o) dz = fmaf(g_s[r * OD + m.doff[s] + o], w[o * zs + d], dz);
      }
      const float w_kl = a.kl_w ? a.kl_w[s] : 0.f;
      const float mu = a.mu[i], lv = a.logvar[i], e = expf(lv);
      dmu = fmaf(w_kl / (float)B, mu, dz) + (a.d_mu_extra ? a.d_mu_extra[i] : 0.f);
      const float dlv = fmaf(dz * a.eps[i], e, w_kl * 0.5f * (e - 1.f) / (float)B) + (a.d_logvar_extra ? a.d_logvar_extra[i] : 0.f);
      draw = dlv * (1.f - lv * lv);
      a.dp[(int64_t)b * 2 * Z + 2 * m.zoff[s] + d] = dmu;
      a.dp[(int64_t)b * 2 * Z + 2 * m.zoff[s] + zs + d] = draw;
    }
    dpl_s[r * 2 * zcm + c] = dmu;
    dpl_s[r * 2 * zcm + zcm + c] = draw;
  });
  // all-gather dp (columns in W_c2p row order: per space mu then raw) over distributed shared memory
  cluster.sync();
  for (int i = tid; i < R * ldp; i += kHT) {
    const int r = i / ldp, col = i % ldp;
    float v = 0.f;
    if (col < 2 * Z) {
      int s = 0;
      while (col >= 2 * (m.zoff[s] + m.zdim[s])) ++s;
      const int e = col - 2 * m.zoff[s], raw = e >= m.zdim[s] ? 1 : 0, zi = m.zoff[s] + e - raw * m.zdim[s];
      const int p = zi / zcm;
      v = cluster.map_shared_rank(dpl_s, p)[r * 2 * zcm + raw * zcm + zi - p * zcm];
    }
    dp_s[i] = v;
  }
  cluster.sync();           // no CTA leaves while a peer may still read its dp
  // d_ctx = dp W_c2p for this CTA's 1/8 of the context columns
  int c0, cc;
  cl_range(a.C, rank, c0, cc);
  col_dot<R>(dp_s, ldp, 2 * Z, a.w_c2p, 1, a.C, c0, cc, red, [&](int r, int c, float s) {
    if (b0 + r < B) a.d_ctx[(int64_t)(b0 + r) * a.C + c0 + c] = s;
  });
}

// d_w_dsc[o][d] = sum_b dl[b][o] z[b][zoff+d]; d_b_dsc[o] = sum_b dl[b][o].  One warp per element.
__global__ void heads_bwd_dsc_kernel(const float* __restrict__ dl, const float* __restrict__ z, float* d_w_dsc,
                                     float* d_b_dsc, int B, HeadsMeta m, int n_w) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= n_w + m.OD) return;
  float acc = 0.f;
  if (warp < n_w) {
    int s = 0;
    while (!(m.dout[s] > 0 && warp >= m.dwoff[s] && warp < m.dwoff[s] + m.dout[s] * m.zdim[s])) ++s;
    int o = (warp - m.dwoff[s]) / m.zdim[s], d = (warp - m.dwoff[s]) % m.zdim[s];
    for (int b = lane; b < B; b += 32) acc = fmaf(dl[(int64_t)b * m.OD + m.doff[s] + o], z[(int64_t)b * m.Z + m.zoff[s] + d], acc);
    acc = warp_sum(acc);
    if (lane == 0) d_w_dsc[warp] = acc;
  } else {
    int od = warp - n_w;
    for (int b = lane; b < B; b += 32) acc += dl[(int64_t)b * m.OD + od];
    acc = warp_sum(acc);
    if (lane == 0) d_b_dsc[od] = acc;
  }
}

// Standalone discriminator loss (used when labels are not handed to the fused forward):
// out[s] = loss, out[S+s] = accuracy; d_logits optional.
__global__ void dsc_loss_kernel(const float* __restrict__ logits, const float* __restrict__ labels, int B, HeadsMeta m,
                                float* __restrict__ out, const float* __restrict__ d_out, float* __restrict__ d_logits) {
  const int s = blockIdx.x, OD = m.OD;
  if (m.dout[s] == 0) { if (out && threadIdx.x == 0) { out[s] = 0.f; out[m.S + s] = 0.f; } return; }
  __shared__ float red[2][8];
  float ls = 0.f, ac = 0.f;
  const float go = d_out ? d_out[s] / (float)B : 0.f;
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    const float* l = logits + (int64_t)b * OD + m.doff[s];
    const float y = labels[(int64_t)m.dlab[s] * B + b];
    if (m.dout[s] == 1) {
      float x = l[0];
      ls += fmaxf(x, 0.f) - x * y + log1pf(expf(-fabsf(x)));
      ac += ((x > 0.f ? 1.f : 0.f) == y) ? 1.f : 0.f;
      if (d_logits) d_logits[(int64_t)b * OD + m.doff[s]] = (sigmoidf_(x) - y) * go;
    } else {
      float mx = l[0];
      int am = 0;
      for (int o = 1; o < m.dout[s]; ++o)
        if (l[o] > mx) { mx = l[o]; am = o; }
      float se = 0.f;
      for (int o = 0; o < m.dout[s]; ++o) se += expf(l[o] - mx);
      const int yi = (int)y;
      ls += mx + logf(se) - l[yi];
      ac += (am == yi) ? 1.f : 0.f;
      if (d_logits)
        for (int o = 0; o < m.dout[s]; ++o) d_logits[(int64_t)b * OD + m.doff[s] + o] = (expf(l[o] - mx) / se - (o == yi ? 1.f : 0.f)) * go;
    }
  }
  ls = warp_sum(ls); ac = warp_sum(ac);
  if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = ls; red[1][threadIdx.x >> 5] = ac; }
  __syncthreads();
  if (threadIdx.x == 0 && out) {
    float a0 = 0.f, a1 = 0.f;
    for (int i = 0; i < 8; ++i) { a0 += red[0][i]; a1 += red[1][i]; }
    out[s] = a0 / (float)B; out[m.S + s] = a1 / (float)B;
  }
}

}  // namespace dvae

using namespace dvae;

extern "C" int dvae_dsc_loss(const float* dsc_logits, const float* labels, int B, int S, const int* space_dims,
                             const int* dsc_out, float* out, const float* d_out, float* d_logits, void* stream) {
  DVAE_REQUIRE(dsc_logits && labels && B > 0 && (out || d_logits), "dvae_dsc_loss: bad argument");
  HeadsMeta m;
  int rc = make_meta(S, space_dims, dsc_out, &m);
  if (rc) return rc;
  dsc_loss_kernel<<<S, 256, 0, (cudaStream_t)stream>>>(dsc_logits, labels, B, m, out, d_out, d_logits);
  DVAE_LAUNCH_CHECK();
  return DVAE_OK;
}

// arrival counter, then at most one partial row per batch row (R >= 1)
extern "C" int64_t dvae_heads_ws_floats(int B, int S) { return 4 + (int64_t)B * 3 * S; }

// Rows per cluster: 8 clusters at B = 64 and B = 128 (64 CTAs, which leaves room for the background weight-gradient
// GEMMs), 16 rows at larger batches; halved until a CTA's shared memory fits.
template <class SmemFor>
static int heads_rows(int B, SmemFor smem_for) {
  int R = B > 64 ? 16 : 8;
  while (R > 1 && smem_for(R) > kHeadsSmemTarget) R /= 2;
  return R;
}

#define DVAE_HEADS_DISPATCH(KERNEL, R, grid_rows, smem, st, a, m)                                                     \
  do {                                                                                                                \
    void (*k_)(decltype(a), HeadsMeta) = R == 16 ? KERNEL<16> : R == 8 ? KERNEL<8> : R == 4 ? KERNEL<4> : R == 2 ? KERNEL<2> : KERNEL<1>; \
    DVAE_CUDA(cudaFuncSetAttribute(k_, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(smem)));                    \
    k_<<<ceil_div(grid_rows, R) * kCl, kHT, smem, st>>>(a, m);                                                       \
    DVAE_LAUNCH_CHECK();                                                                                              \
  } while (0)

extern "C" int dvae_latent_heads_fwd(const float* ctx, int B, int C, int S, const int* space_dims,
                                     const int* dsc_out, const float* w_c2p, const float* b_c2p, const float* eps,
                                     const float* w_dsc, const float* b_dsc, const float* labels,
                                     const float* kl_w_dev, const float* w_z2h, const float* b_z2h, int H2L,
                                     float* z, float* mu, float* logvar, float* hid, float* dsc_logits,
                                     float* scalars, float* ws, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  DVAE_REQUIRE(ctx && space_dims && w_c2p && b_c2p && eps && w_z2h && b_z2h && z && mu && logvar && hid && scalars && ws,
               "dvae_latent_heads_fwd: null pointer");
  DVAE_REQUIRE(B > 0 && C > 0 && H2L > 0, "dvae_latent_heads_fwd: bad shape");
  HeadsMeta m;
  int rc = make_meta(S, space_dims, dsc_out, &m);
  if (rc) return rc;
  DVAE_REQUIRE(m.OD == 0 || (w_dsc && b_dsc && dsc_logits), "dvae_latent_heads_fwd: discriminator buffers missing");
  const int R = heads_rows(B, [&](int r) { return heads_fwd_smem(r, C, m); });
  const size_t smem = heads_fwd_smem(R, C, m);
  DVAE_REQUIRE(smem <= 227 * 1024, "dvae_latent_heads_fwd: context width %d / %d latents too large for shared memory", C, m.Z);
  HeadsFwdArgs a{ctx, w_c2p, b_c2p, eps, w_dsc, b_dsc, labels, kl_w_dev, w_z2h, b_z2h,
                 z, mu, logvar, hid, dsc_logits, scalars, ws, B, C, H2L, red_floats(R, 2 * ceil_div(m.Z, kCl))};
  DVAE_HEADS_DISPATCH(heads_fwd_kernel, R, B, smem, st, a, m);
  return DVAE_OK;
}

extern "C" int64_t dvae_heads_bwd_ws_floats(int B, int Z, int H2L) { return (int64_t)B * (H2L + 2 * Z + kMaxDscOut); }

extern "C" int dvae_latent_heads_bwd(const float* ctx, int B, int C, int S, const int* space_dims,
                                     const int* dsc_out, const float* w_c2p, const float* eps, const float* w_dsc,
                                     const float* labels, const float* kl_w_dev, const float* w_z2h, int H2L,
                                     const float* z, const float* mu, const float* logvar, const float* hid,
                                     const float* dsc_logits, const float* d_hid, const float* d_z_extra,
                                     const float* d_mu_extra, const float* d_logvar_extra,
                                     const float* d_logits_extra, float* d_w_c2p, float* d_b_c2p, float* d_w_dsc, float* d_b_dsc,
                                     float* d_w_z2h, float* d_b_z2h, float* d_ctx, float* ws, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  DVAE_REQUIRE(ctx && space_dims && w_c2p && eps && w_z2h && z && mu && logvar && hid && d_hid && d_w_c2p && d_b_c2p &&
                   d_w_z2h && d_b_z2h && d_ctx && ws, "dvae_latent_heads_bwd: null pointer");
  HeadsMeta m;
  int rc = make_meta(S, space_dims, dsc_out, &m);
  if (rc) return rc;
  DVAE_REQUIRE(m.OD == 0 || (w_dsc && dsc_logits && d_w_dsc && d_b_dsc), "dvae_latent_heads_bwd: discriminator buffers missing");
  const int Z = m.Z;
  float* d_pre = ws;                              // [B,H2L]
  float* dp = d_pre + (int64_t)B * H2L;           // [B,2Z]
  float* dl = dp + (int64_t)B * 2 * Z;            // [B,OD]
  const int R = heads_rows(B, [&](int r) { return heads_bwd_smem(r, H2L, m); });
  const size_t smem = heads_bwd_smem(R, H2L, m);
  DVAE_REQUIRE(smem <= 227 * 1024, "dvae_latent_heads_bwd: %d decoder-state columns too many for shared memory", H2L);
  HeadsBwdArgs a{w_c2p, eps, w_dsc, labels, kl_w_dev, w_z2h, mu, logvar, hid, dsc_logits, d_hid, d_z_extra, d_mu_extra,
                 d_logvar_extra, d_logits_extra, d_pre, dp, dl, d_ctx, B, C, H2L, red_floats(R, 0)};
  DVAE_HEADS_DISPATCH(heads_bwd_kernel, R, B, smem, st, a, m);
  // weight and bias gradients from the workspace, on side streams (the encoder's backward waits for d_ctx only)
  GemmHints grad_hints;            // A operands below are gradients of unknown magnitude
  grad_hints.a_wide = true;
  Fork fork(st);
  // z2hidden: d_w = d_pre^T z, d_b = colsum(d_pre)
  if ((rc = linear_impl_ex(d_pre, H2L, 1, z, Z, 1, d_w_z2h, Z, H2L, Z, B, nullptr, nullptr, 0.f, 0, grad_hints, fork.side(0)))) return rc;
  if ((rc = colsum_impl(d_pre, H2L, B, H2L, d_b_z2h, 0.f, fork.side(1)))) return rc;
  if (m.OD > 0) {
    int n_w = 0;
    for (int s = 0; s < S; ++s) n_w += m.dout[s] * m.zdim[s];
    heads_bwd_dsc_kernel<<<ceil_div((int64_t)(n_w + m.OD) * 32, 256), 256, 0, fork.side(2)>>>(dl, z, d_w_dsc, d_b_dsc, B, m, n_w);
    DVAE_LAUNCH_CHECK();
  }
  // context2params: d_w = dp^T ctx, d_b = colsum(dp)
  if ((rc = linear_impl_ex(dp, 2 * Z, 1, ctx, C, 1, d_w_c2p, C, 2 * Z, C, B, nullptr, nullptr, 0.f, 0, grad_hints, fork.side(2)))) return rc;
  if ((rc = colsum_impl(dp, 2 * Z, B, 2 * Z, d_b_c2p, 0.f, fork.side(2)))) return rc;
  return fork.join_or_defer();
}
