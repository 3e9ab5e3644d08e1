/*
 * dvae_b200.h -- C ABI of the B200-native disentangled sentence-VAE hot path.
 *
 * The reference (jvasilakes/disentanglement-vae) is pure Python and has no FFI: its de-facto
 * plugin boundary is `vae.model.build_vae()` (vae/model.py:515-559) plus the `vae.losses` free
 * functions (vae/losses.py:137-242).  The Python package `disentanglement-vae_b200/` mirrors that
 * surface and lowers every tensor op on the path to the entry points below, bound with ctypes
 * (see INTEGRATION.md for the stub).  Each entry point cites the reference code it replaces.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in `_host`;
 *   - all real data is float32, token ids / lengths are int64 (as in the reference);
 *   - matrices are row-major with an explicit row stride (`ld*`, in elements);
 *   - sequence buffers are TIME-MAJOR: [T][B][width];
 *   - no allocation, no ownership transfer, no synchronisation: kernels are enqueued on `stream`
 *     (a cudaStream_t) and the call returns; buffers (incl. workspaces) are caller-allocated;
 *   - per-step scalars that change between replays of a captured CUDA graph (dropout seed, KL
 *     weights, Adam step/lr) are read from device memory, never baked into launch arguments;
 *   - return value: 0 on success, negative `DVAE_E*` otherwise (`dvae_last_error_string()`
 *     describes the last failure on the calling thread).  There is no CPU fallback.
 */
#ifndef DVAE_B200_H_
#define DVAE_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DVAE_OK 0
#define DVAE_EINVAL (-1)   /* bad argument (null pointer, non-positive size, unsupported shape) */
#define DVAE_ECUDA (-2)    /* a CUDA runtime call or kernel launch failed                        */
#define DVAE_EWORKSPACE (-3) /* caller-provided workspace too small                              */

#define DVAE_MAX_SPACES 8  /* latent spaces per model (labels + "content")                        */

const char* dvae_last_error_string(void);
int dvae_version(void);
/* Number of kernels this library has launched in the calling process (for bench.py's
 * `gpu_launches`). */
int64_t dvae_launch_count(void);

/* ---------------------------------------------------------------------------------------------
 * Dense layer: C[M,N] = act(A . B^T + bias + bias2) + beta * C          (fp32 SIMT GEMM)
 * Replaces nn.Linear / torch.mm call sites on the path (vae/model.py:164,196,388,403 and the
 * input projections inside nn.LSTM, vae/model.py:95,158) and their autograd transposes.
 *   trans_a == 0: A is [M,K] row-major (row stride lda);  trans_a == 1: A is stored [K,M].
 *   trans_b == 0: B is [N,K] row-major (an nn.Linear weight); trans_b == 1: B is stored [K,N].
 *   bias, bias2: [N] or NULL.  act: 0 none, 1 tanh.  beta: 0 overwrites C, 1 accumulates.
 * ------------------------------------------------------------------------------------------- */
int dvae_linear(const float* A, int64_t lda, int trans_a, const float* B, int64_t ldb, int trans_b,
                float* C, int64_t ldc, int M, int N, int K, const float* bias, const float* bias2,
                float beta, int act, void* stream);

/* Same contract as dvae_linear, computed on the 5th-generation tensor cores (TMA-staged 128x128x32
 * tiles, tcgen05.mma.kind::tf32 into TMEM).  passes = 3: 3xTF32 split (hi*hi + hi*lo + lo*hi), fp32-grade
 * accuracy -- the forward path's setting; passes = 1: single TF32 pass with round-to-nearest operands.
 * Requires 16-byte aligned A, B and lda, ldb multiples of 4 (TMA). */
int dvae_tc_linear(const float* A, int64_t lda, int trans_a, const float* B, int64_t ldb, int trans_b,
                   float* C, int64_t ldc, int M, int N, int K, const float* bias, const float* bias2,
                   float beta, int act, int passes, void* stream);

/* Same contract again, second-generation tensor-core kernel (tc_gemm16.cu): the fp32 operands are split on the fly
 * into fp16 (hi, lo * 2^11) planes -- 22 mantissa bits each -- and multiplied by tcgen05.mma.kind::f16 into two TMEM
 * accumulators (hi*hi | hi*lo + lo*hi); three K=16 MMAs per 16 k instead of 3xTF32's six K=8 ones, and a third of the
 * shared-memory traffic.  fp16 has a narrow exponent range, so each operand is first multiplied by a power of two:
 * `a_scale` / `b_scale` (host constants, 1 = none) or, when `a_amax_bits` / `b_amax_bits` (device, may be NULL) is
 * given, 2^(13 - floor(log2 amax)) from the bit pattern of a device-side max |x|.  The product is unscaled in the
 * epilogue.  K-major operands need 16-byte alignment, ld % 4 == 0 and K % 4 == 0; returns DVAE_EINVAL otherwise. */
int dvae_tc16_linear(const float* A, int64_t lda, int trans_a, const float* B, int64_t ldb, int trans_b,
                     float* C, int64_t ldc, int M, int N, int K, const float* bias, const float* bias2,
                     float beta, int act, float a_scale, float b_scale, const uint32_t* a_amax_bits,
                     const uint32_t* b_amax_bits, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Auxiliary disentanglement objectives on the latent spaces (adversaries and CLUB mutual-information estimators;
 * vae/model.py:219-258,323-355, vae/losses.py:10-74,199-242).  Operands are [B, O] / [B, D] row-major matrices of a few
 * KB; each entry point is forward + backward: gradients are written when their output pointers are non-NULL,
 * multiplied by *g (device scalar, NULL = 1).
 *   dvae_entropy_loss: loss = mean_b sum_c p log p with p = clamp(sigmoid(x) if O == 1 else softmax(x), 1e-8, 1-1e-8)
 *                      -- AdversarialDiscriminator.compute_adversarial_loss (model.py:247-258).
 *   dvae_club_mi:      mi = mean_i sum_d [ -(mu_id - y_id)^2 + mean_j (y_jd - mu_id)^2 ] / (2 exp(logvar_id))
 *                      -- CLUB.forward (losses.py:53-67); gradients w.r.t. mu, logvar AND y; ws: 3*D floats.
 *   dvae_club_nll:     loss = mean_b sum_d [ (mu - y)^2 / exp(logvar) + logvar ] -- CLUB.learning_loss (losses.py:69-74).
 *   dvae_act_bwd:      d = g * (1 - y^2) (act 1, tanh) or g * [y > 0] (act 2, ReLU), y = the activation's OUTPUT.
 *   dvae_relu:         in-place ReLU.
 * ------------------------------------------------------------------------------------------- */
int dvae_entropy_loss(const float* logits, int B, int O, float* loss, const float* g_loss, float* d_logits,
                      void* stream);
int dvae_club_mi(const float* mu, const float* logvar, const float* y, int B, int D, float* mi,
                 const float* g_mi, float* d_mu, float* d_logvar, float* d_y, float* ws, void* stream);
int dvae_club_nll(const float* mu, const float* logvar, const float* y, int B, int D, float* loss,
                  const float* g_loss, float* d_mu, float* d_logvar, void* stream);
int dvae_act_bwd(const float* y, const float* g, float* d, int64_t n, int act, void* stream);
int dvae_relu(float* x, int64_t n, void* stream);

/* Weight planes.  The tensor-core GEMMs multiply fp16 (hi, lo) operand planes; for an fp32 operand those planes are
 * normally produced inside every CTA that reads it.  A caller that knows when a weight matrix changes (a training loop:
 * once per optimizer step) can instead register it with caller-allocated plane buffers
 *     planes   : dvae_weight_planes_floats(R, C, 0) floats -- W   [R, C] as a K-major B operand (x . W^T: the input projections)
 *     planes_t : dvae_weight_planes_floats(R, C, 1) floats -- W^T [C, R] (g . W: the dx / d_h GEMMs); either may be NULL
 * recompute the planes of ALL registered weights with one launch (dvae_weight_planes_refresh, e.g. first thing in a step)
 * and switch the registry on around its own calls (dvae_weight_planes_enable; host-side, per process, off by default).
 * While on, a GEMM inside any entry point whose B operand is a registered weight -- or a block of it starting on a
 * multiple of 128 rows / 32 columns -- fetches B as ready-made tiles by bulk copy.  The planes MUST be current whenever
 * such a GEMM runs; dvae_weight_planes_clear forgets every registration and switches the registry off.
 * Replaces nothing in the reference: it is operand staging for vae/model.py:95,158 (nn.LSTM input projections) and
 * their autograd transposes. */
int64_t dvae_weight_planes_floats(int R, int C, int transposed);
int dvae_weight_planes_register(const float* w, int R, int C, void* planes, void* planes_t);
int dvae_weight_planes_refresh(void* stream);
/* Only the entries [first, first + count) in registration order: lets a caller refresh the weights its first kernels
 * read on the main stream and the others (e.g. W_out^T, needed by the vocabulary backward only) on a side stream. */
int dvae_weight_planes_refresh_ex(int first, int count, void* stream);
int dvae_weight_planes_enable(int on);
int dvae_weight_planes_clear(void);

/* Independent kernels inside one call (e.g. the weight-gradient GEMMs of an LSTM layer) run on library-owned side
 * streams and are joined back into `stream` before the call returns.  dvae_defer_joins(1) lets the backward entry
 * points (dvae_lstm_seq_bwd, dvae_latent_heads_bwd) return with that side work still in flight, so that it overlaps
 * the next layer's recurrence; the caller must then call dvae_join_side_streams(stream) -- which also switches the
 * deferral off -- before anything consumes the weight / bias gradients (or before a graph capture ends).
 * Per host thread.  Replaces nothing in the reference: it is scheduling of run.py:254's backward() work. */
int dvae_defer_joins(int on);
int dvae_join_side_streams(void* stream);

/* Scheduling of the gradient exchange inside a data-parallel step captured as ONE CUDA graph:
 *   dvae_counter_increment   *counter += 1 (first node of the captured step): the step counter from which the exchange
 *                            kernels derive their barrier epochs, so that nothing is reset between replays
 *   dvae_fork_after          the library's signal stream, made to wait for everything enqueued so far on `stream` -- and,
 *                            include_sides != 0, the detached side-stream work (dvae_defer_joins) and `extra_stream` (or
 *                            NULL); what the caller enqueues on *forked_stream_out afterwards runs beside `stream` until
 *                            dvae_join_side_streams(stream)
 * Replaces nothing in the reference: it is the scheduling of DistributedDataParallel's bucketed gradient exchange. */
int dvae_counter_increment(uint32_t* counter, void* stream);
int dvae_fork_after(int include_sides, void* extra_stream, void* stream, void** forked_stream_out);

/* All-reduce (SUM, in place) of one gradient bucket over NVSwitch multicast memory, one kernel per rank (nvls.cu):
 * cross-rank barrier, multimem.ld_reduce of this rank's 1/world slice, multimem.st of the sums into every rank's buffer,
 * cross-rank barrier.  `mc_ptr` is the MULTICAST address of the bucket inside a symmetric allocation that every rank made
 * with the same size (torch.distributed._symmetric_memory: handle.multicast_ptr + byte offset), 16-byte aligned, n % 4 == 0.
 * `barrier_ptrs_host[r]`: peer-mapped address of rank r's barrier block (dvae_nvls_barrier_words() zeroed uint32 words in
 * a second symmetric allocation).  Every call on a barrier block must use a larger epoch = *counter_dev * epoch_mul +
 * epoch_add than the one before (>= 1), and all ranks must make the same sequence of calls with the same n and ctas.
 * ctas = 0: sized from the bucket (<= 128).  soft_timeout_ns > 0: a rank that waits longer sets *err_dev = 1 and returns
 * (start-up self-test); 0: trap after 60 s.  Replaces DistributedDataParallel's bucketed ncclAllReduce. */
/* dvae_p2p_all_reduce: the same kernel with plain loads / stores through peer-mapped addresses (peer_ptrs_host[r] = the
 * bucket inside rank r's buffer) instead of the switch: the owner adds the world copies in rank order and stores the sum
 * to every copy.  The better of the two on 2 GPUs (0.5x the bucket per direction instead of 1.5x). */
int64_t dvae_nvls_barrier_words(void);
int dvae_p2p_all_reduce(float* const* peer_ptrs_host, int64_t n, uint32_t* const* barrier_ptrs_host, int rank, int world,
                        const uint32_t* counter_dev, uint32_t epoch_mul, uint32_t epoch_add, int ctas,
                        uint64_t soft_timeout_ns, uint32_t* err_dev, void* stream);
int dvae_nvls_all_reduce(float* mc_ptr, int64_t n, uint32_t* const* barrier_ptrs_host, int rank, int world,
                         const uint32_t* counter_dev, uint32_t epoch_mul, uint32_t epoch_add, int ctas,
                         uint64_t soft_timeout_ns, uint32_t* err_dev, void* stream);

/* out[n] = sum_m X[m, n] (+ out[n] if beta == 1); X is [M,N] row-major with row stride ldx. */
int dvae_colsum(const float* X, int64_t ldx, int M, int N, float* out, float beta, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Embedding lookup + element-wise dropout (vae/model.py:90,153):
 *   x[t][b][:] = emb[tokens[b*tok_stride_b + t*tok_stride_t]][:] * mask(t,b,:) / (1-p)
 * mask is a counter-based Philox4x32-10 Bernoulli(1-p) keyed by (*seed_dev, salt, element index);
 * p == 0 (or seed_dev == NULL) disables it.  `dvae_dropout` applies the same kind of mask to a
 * dense [rows, width] activation (the nn.LSTM inter-layer dropout, vae/model.py:74-77,137-140).
 * `dvae_embedding_bwd` scatter-ADDS d_x (masked the same way) into d_emb [V, E].
 * first_token >= 0 replaces the token at t == 0 for every row (the decoder is always fed <SOS>
 * first, vae/model.py:445-447, then inputs[:, t] under teacher forcing, model.py:464-466).
 * t0 / row0: the call covers time steps [t0, t0+T) (rows [row0, row0+rows)) of buffers addressed by ABSOLUTE
 * step / row, so a single decode step uses the same dropout counters as the full-sequence call (and the
 * full-sequence backward regenerates the same masks).
 * `dvae_randn` fills out[n] with N(0,1) draws (Philox + Box-Muller): the reparameterisation
 * noise of vae/model.py:392-395 when the caller does not supply it.
 * ------------------------------------------------------------------------------------------- */
int dvae_randn(float* out, int64_t n, const uint64_t* seed_dev, uint32_t salt, void* stream);
int dvae_embedding_fwd(const float* emb, int E, const int64_t* tokens, int64_t tok_stride_b,
                       int64_t tok_stride_t, int T, int B, float p, const uint64_t* seed_dev,
                       uint32_t salt, int64_t first_token, int t0, float* x, void* stream);
int dvae_embedding_bwd(const float* d_x, int E, const int64_t* tokens, int64_t tok_stride_b,
                       int64_t tok_stride_t, int T, int B, float p, const uint64_t* seed_dev,
                       uint32_t salt, int64_t first_token, int t0, float* d_emb, void* stream);
/* Bag-of-words encoder (BOWEncoder.forward, vae/model.py:42-49): ctx[b, e] = max over all T positions of
 * emb[tokens[b, t], e] * dropout keep-scale; argmax [B, E] int32 records the winning position (first on ties) for the
 * backward pass, which scatter-adds d_ctx (masked like the forward) into d_emb. */
int dvae_bow_encoder_fwd(const float* emb, int E, const int64_t* tokens, int64_t tok_stride_b, int64_t tok_stride_t,
                         int T, int B, float p, const uint64_t* seed_dev, uint32_t salt, float* ctx, int64_t ldctx,
                         int32_t* argmax, void* stream);
int dvae_bow_encoder_bwd(const float* d_ctx, int64_t ldd, const int32_t* argmax, int E, const int64_t* tokens,
                         int64_t tok_stride_b, int64_t tok_stride_t, int T, int B, float p, const uint64_t* seed_dev,
                         uint32_t salt, float* d_emb, void* stream);
int dvae_dropout(const float* x, int64_t ldx, int64_t rows, int width, float p,
                 const uint64_t* seed_dev, uint32_t salt, float* y, int64_t ldy, int64_t row0,
                 void* stream);

/* ---------------------------------------------------------------------------------------------
 * One LSTM layer (1 or 2 directions) over a padded, time-major batch.  Replaces nn.LSTM inside
 * VariationalEncoder.forward (vae/model.py:88-101, incl. pack/pad = per-row length masking) and
 * the T-1 single-step calls of VariationalDecoder.forward (vae/model.py:152-165,457-460) when the
 * decoder inputs are known (teacher forcing).  Gate order i,f,g,o (PyTorch).
 *
 *   x        [T,B,I] (row stride ldx) -- already embedded / dropped out
 *   w_ih[d]  [4H,I], w_hh[d] [4H,H], b_ih[d], b_hh[d] [4H]   (d = 0 forward, 1 reverse)
 *   h0, c0   [D][B] rows of H with row stride ld0 and direction stride dir0, or NULL (zeros)
 *   lengths  [B] int64 or NULL (every row runs all T steps, as the decoder does, model.py:448)
 *   hs       [T,B,D*H] (row stride ldhs; direction d occupies columns [d*H,(d+1)*H)); rows with
 *            t >= lengths[b] are written as zeros (pad_packed_sequence)
 *   hn, cn   final state of each row's own traversal, [D][B] rows with stride ldn / dirn; NULL ok
 *   gates    [D,T,B,4H] post-activation gates, cs [D,T,B,H] cell states: saved for backward.
 *            `gates` doubles as the pre-activation workspace.
 *   state_ws scratch of dvae_lstm_state_ws_floats(B,H,D) floats (carried h/c ping-pong)
 * ------------------------------------------------------------------------------------------- */
int64_t dvae_lstm_state_ws_floats(int B, int H, int D);
int dvae_lstm_seq_fwd(const float* x, int64_t ldx, int T, int B, int I, int H, int D,
                      const float* const* w_ih_host, const float* const* w_hh_host,
                      const float* const* b_ih_host, const float* const* b_hh_host,
                      const float* h0, const float* c0, int64_t ld0, int64_t dir0,
                      const int64_t* lengths, float* hs, int64_t ldhs, float* hn, float* cn,
                      int64_t ldn, int64_t dirn, float* gates, float* cs, float* state_ws,
                      void* stream);

/* One time step t of one uni-directional layer, operating on the full-sequence buffers of dvae_lstm_seq_fwd
 * (x [T,B,I], hs [T,B,H], gates [1,T,B,4H], cs [1,T,B,H]).  Sampled decoding (teacher_forcing_prob < 1, sample();
 * vae/model.py:457-472,498-508) needs step t's vocabulary sample before step t+1's input exists, so the decoder
 * advances one step per call; the buffers end up exactly as after a whole-sequence call, so the backward pass
 * (dvae_lstm_seq_bwd) is shared.  h0/c0 (row stride ld0, NULL = zeros) are read at t == 0. */
int dvae_lstm_step(const float* x, int64_t ldx, int t, int T, int B, int I, int H, const float* w_ih,
                   const float* w_hh, const float* b_ih, const float* b_hh, const float* h0,
                   const float* c0, int64_t ld0, float* hs, float* gates, float* cs, float* state_ws,
                   void* stream);

/* The two halves of dvae_lstm_seq_fwd separately: dvae_lstm_input_proj fills `gates` with x.W_ih^T + b_ih + b_hh for all
 * time steps (one GEMM per direction); dvae_lstm_seq_fwd_ex with flags bit 0 set then runs the recurrence alone.  Lets a
 * caller run a layer's projection early on another stream (the decoder's layer 0 under teacher forcing depends on the
 * input tokens only).  flags = 0: identical to dvae_lstm_seq_fwd. */
int dvae_lstm_input_proj(const float* x, int64_t ldx, int T, int B, int I, int H, int D,
                         const float* const* w_ih, const float* const* b_ih, const float* const* b_hh,
                         float* gates, void* stream);
int dvae_lstm_seq_fwd_ex(const float* x, int64_t ldx, int T, int B, int I, int H, int D,
                         const float* const* w_ih, const float* const* w_hh, const float* const* b_ih,
                         const float* const* b_hh, const float* h0, const float* c0, int64_t ld0,
                         int64_t dir0, const int64_t* lengths, float* hs, int64_t ldhs, float* hn,
                         float* cn, int64_t ldn, int64_t dirn, float* gates, float* cs, float* state_ws,
                         int flags, void* stream);

/* Back-propagation through time for dvae_lstm_seq_fwd (the autograd of nn.LSTM).
 *   d_hs [T,B,D*H] (row stride lddhs) or NULL; d_hn, d_cn as hn/cn or NULL.
 *   gates is OVERWRITTEN with the pre-activation gradients dG [D,T,B,4H].
 *   Outputs (overwritten): d_x [T,B,I] (sum over directions; NULL to skip), d_w_ih[d], d_w_hh[d],
 *   d_b_ih[d], d_b_hh[d], d_h0/d_c0 (layout of h0/c0; NULL to skip). */
int dvae_lstm_seq_bwd(const float* x, int64_t ldx, int T, int B, int I, int H, int D,
                      const float* const* w_ih_host, const float* const* w_hh_host,
                      const float* h0, const float* c0, int64_t ld0, int64_t dir0,
                      const int64_t* lengths, const float* hs, int64_t ldhs, float* gates,
                      const float* cs, const float* d_hs, int64_t lddhs, const float* d_hn,
                      const float* d_cn, int64_t ldn, int64_t dirn, float* d_x, int64_t lddx,
                      float* const* d_w_ih_host, float* const* d_w_hh_host,
                      float* const* d_b_ih_host, float* const* d_b_hh_host, float* d_h0,
                      float* d_c0, int64_t ldd0, int64_t dird0, float* state_ws, void* stream);

/* The same with a plane workspace (dvae_lstm_bwd_planes_ws_floats(T, B, I, H, D) floats, 16-byte aligned, or NULL): the
 * weight gradients dW_ih = dG^T x and dW_hh = dG^T h_prev contract over the T*B positions, i.e. read both operands
 * transposed.  With the workspace x, dG and hs are transposed once into fp16 operand planes (one launch; dG scaled by the
 * max |dG| the recurrence kernel measured) and those GEMMs are bulk-copy fed on both operands. */
int64_t dvae_lstm_bwd_planes_ws_floats(int T, int B, int I, int H, int D);
/* Per host thread: the d_x GEMM of the following unidirectional (D = 1) dvae_lstm_seq_bwd / _ex calls runs on `stream`,
 * ordered after the call's recurrence, as background work beside what the caller's stream does next (NULL: the call's own
 * stream, the default).  The caller orders its reads of d_x after `stream`.  Scheduling only: d_x is the same. */
int dvae_lstm_bwd_dx_stream(void* stream);
int dvae_lstm_seq_bwd_ex(const float* x, int64_t ldx, int T, int B, int I, int H, int D,
                         const float* const* w_ih_host, const float* const* w_hh_host,
                         const float* h0, const float* c0, int64_t ld0, int64_t dir0,
                         const int64_t* lengths, const float* hs, int64_t ldhs, float* gates,
                         const float* cs, const float* d_hs, int64_t lddhs, const float* d_hn,
                         const float* d_cn, int64_t ldn, int64_t dirn, float* d_x, int64_t lddx,
                         float* const* d_w_ih_host, float* const* d_w_hh_host,
                         float* const* d_b_ih_host, float* const* d_b_hh_host, float* d_h0,
                         float* d_c0, int64_t ldd0, int64_t dird0, float* state_ws, float* planes_ws,
                         void* stream);

/* ---------------------------------------------------------------------------------------------
 * Fused latent heads.  Replaces compute_latent_params (vae/model.py:384-398), the
 * discriminators' forward / loss / accuracy (vae/model.py:195-216, vae/losses.py:180-196),
 * kl_divergence + compute_kl_divergence_losses (vae/losses.py:153-177) and compute_hidden
 * (vae/model.py:400-411) in ONE kernel.
 *
 *   ctx [B,C]; w_c2p [2Z,C] = the context2params weights concatenated in space order, each space
 *   contributing rows [mu(zs); raw(zs)]; b_c2p [2Z]; eps [B,Z] (N(0,1) draws, space-concatenated);
 *   space_dims_host[S]; w_dsc / b_dsc: discriminator weights concatenated over the spaces that
 *   have one (dsc_out_host[s] = output dim, 0 = none): rows [out_s, zs]; labels [ND_total? no: one
 *   float per (dsc, b)] laid out [n_dsc][B] (class index as float for multi-class heads), NULL in
 *   inference; kl_w_dev [S] KL weights (lambda or the cyclic value, vae/losses.py:143-150);
 *   w_z2h [2*H*Ld, Z], b_z2h.
 * Outputs: z, mu, logvar [B,Z]; hid [B,2*H*Ld] = tanh(z2hidden(z)) -- decoder layer l takes
 *   h0 = hid[:, l*H:(l+1)*H], c0 = hid[:, (Ld+l)*H:(Ld+l+1)*H] (row stride 2*H*Ld);
 *   dsc_logits [B, sum(out)]; scalars[ ] (device, DVAE_HEADS_NSCALARS floats):
 *   [0] total_weighted_kl, [1] total_kl, [2] total_dsc_loss, [3..3+S) kl per space,
 *   [3+S..3+2S) dsc loss per space (0 where none), [3+2S..3+3S) dsc accuracy per space.
 *   ws: dvae_heads_ws_floats(B,S) floats of scratch, zero-filled by the caller before the FIRST call (every call leaves
 *   its arrival counter re-armed).
 * ------------------------------------------------------------------------------------------- */
#define DVAE_HEADS_NSCALARS (3 + 3 * DVAE_MAX_SPACES)
int64_t dvae_heads_ws_floats(int B, int S);
int dvae_latent_heads_fwd(const float* ctx, int B, int C, int S, const int* space_dims_host,
                          const int* dsc_out_host, const float* w_c2p, const float* b_c2p,
                          const float* eps, const float* w_dsc, const float* b_dsc,
                          const float* labels, const float* kl_w_dev, const float* w_z2h,
                          const float* b_z2h, int H2L, float* z, float* mu, float* logvar,
                          float* hid, float* dsc_logits, float* scalars, float* ws, void* stream);

/* Backward of the fused heads w.r.t. total = weighted KL + dsc losses + (decoder path via d_hid).
 *   d_hid [B,H2L] gradient w.r.t. `hid`;  d_z_extra / d_mu_extra / d_logvar_extra [B,Z] and
 *   d_logits_extra [B,sum(out)]: optional upstream gradients on the returned tensors (NULL ok) --
 *   how the adversarial / MI objectives (vae/losses.py:199-242) and losses computed outside the
 *   fused kernel reach the encoder.
 *   Outputs (overwritten): d_w_c2p, d_b_c2p, d_w_dsc, d_b_dsc, d_w_z2h, d_b_z2h, d_ctx [B,C].
 *   ws: dvae_heads_bwd_ws_floats(B,Z,H2L) floats. */
int64_t dvae_heads_bwd_ws_floats(int B, int Z, int H2L);
int dvae_latent_heads_bwd(const float* ctx, int B, int C, int S, const int* space_dims_host,
                          const int* dsc_out_host, const float* w_c2p, const float* eps,
                          const float* w_dsc, const float* labels, const float* kl_w_dev,
                          const float* w_z2h, int H2L, const float* z, const float* mu,
                          const float* logvar, const float* hid, const float* dsc_logits,
                          const float* d_hid, const float* d_z_extra, const float* d_mu_extra,
                          const float* d_logvar_extra, const float* d_logits_extra, float* d_w_c2p,
                          float* d_b_c2p, float* d_w_dsc, float* d_b_dsc, float* d_w_z2h,
                          float* d_b_z2h, float* d_ctx, float* ws, void* stream);

/* Discriminator loss on its own (Discriminator.compute_loss / compute_accuracy,
 * vae/model.py:199-216; vae/losses.py:180-196) for callers that did not pass labels to the fused
 * forward: out[s] = loss, out[S+s] = accuracy (NULL to skip); when d_logits != NULL it receives
 * d_out[s] * d(loss_s)/d(logits). */
int dvae_dsc_loss(const float* dsc_logits, const float* labels, int B, int S,
                  const int* space_dims_host, const int* dsc_out_host, float* out,
                  const float* d_out, float* d_logits, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Fused vocabulary projection + online log-softmax + masked NLL.  Replaces the per-step
 * decoder.linear (vae/model.py:164,462), the [B,T,V] `out_logits` buffer (model.py:452-454) and
 * reconstruction_loss -> texar sequence_sparse_softmax_cross_entropy (vae/losses.py:137-140).
 * The logits are never written to memory.
 *
 *   h [N,H] time-major decoder outputs, N = T1*B, row n = (t-1)*B + b covers target position t
 *   (t = 1..T1); w [V,H], bias [V]; targets [B, *] int64 with strides (tgt_stride_b, 1);
 *   lengths [B] int64; sos = <SOS> id.
 * Outputs: lse [N]; nll [N] (unmasked); argmax [N] int32 (token-level reconstruction argmax);
 *   loss[0] = (1/B) * sum_b ( nll0_b + sum_{1<=t<len_b} nll[b,t] ) where nll0_b is the constant
 *   contribution of the one-hot pseudo-logit row at t = 0 (model.py:454):
 *   log(e + V - 1) - [targets[b,0] == sos].
 *   ws: dvae_vocab_ce_ws_floats(N, V, H) floats.
 * ------------------------------------------------------------------------------------------- */
int64_t dvae_vocab_ce_ws_floats(int N, int V, int H);
int dvae_vocab_ce_fwd(const float* h, int64_t ldh, int T1, int B, int H, int V, const float* w,
                      const float* bias, const int64_t* targets, int64_t tgt_stride_b,
                      const int64_t* lengths, int sos, float* lse, float* nll, int32_t* argmax,
                      float* loss, float* ws, void* stream);

/* The operand split of W_out as a call of its own (W_out does not depend on the step's activations): run it early, on
 * another stream, then pass flags bit 0 to dvae_vocab_ce_fwd_ex (same N = T1*B, V, H, w, ws).  Without the flag, or when
 * the split call was a no-op for the shape, the forward call splits W itself. */
int dvae_vocab_split_w(const float* w, int N, int V, int H, float* ws, void* stream);
int dvae_vocab_ce_fwd_ex(const float* h, int64_t ldh, int T1, int B, int H, int V, const float* w,
                         const float* bias, const int64_t* targets, int64_t tgt_stride_b,
                         const int64_t* lengths, int sos, float* lse, float* nll, int32_t* argmax,
                         float* loss, float* ws, int flags, void* stream);

/* The same over the LIVE rows only: positions with t < len_b (the ones the loss keeps), in ascending n.  Their count is
 * known on the device only -- the call builds the row list from `lengths` and sizes the GEMMs' work from it, with launch
 * grids for all N rows -- so one captured CUDA graph serves every length distribution.  lse / nll / argmax are written at
 * live positions only; the loss is that of dvae_vocab_ce_fwd.  ws (dvae_vocab_ce_ws_floats) keeps the row list at float
 * offset dvae_vocab_live_rows_at(N, V, H) (N int32 entries, then the live count) and the operand planes that
 * dvae_vocab_ce_bwd_live reads.  Shapes the pre-split tensor-core kernels do not take run over every row. */
int dvae_vocab_ce_fwd_live(const float* h, int64_t ldh, int T1, int B, int H, int V, const float* w,
                           const float* bias, const int64_t* targets, int64_t tgt_stride_b,
                           const int64_t* lengths, int sos, float* lse, float* nll, int32_t* argmax,
                           float* loss, float* ws, int flags, void* stream);
int64_t dvae_vocab_live_rows_at(int N, int V, int H);

/* Measurement entry (bench.py roofline, ncu): only the projection + online-softmax partials kernel of
 * dvae_vocab_ce_fwd (no operand split, no finalize).  ws must come from an earlier dvae_vocab_ce_fwd call with the same
 * arguments.  Not part of the reference-facing surface. */
int dvae_vocab_ce_partials(const float* h, int64_t ldh, int T1, int B, int H, int V, const float* w,
                           const float* bias, const int64_t* targets, int64_t tgt_stride_b,
                           const int64_t* lengths, int sos, float* ws, void* stream);

/* Sampled next token per row without materialising [B,V] logits or probabilities: replaces
 * decoder.linear + torch.softmax + torch.multinomial (vae/model.py:164,468-469,504-505).
 * tokens_out[b*tok_stride] = argmax_v( h[b].w[v] + bias[v] + g(b,v) ), g ~ Gumbel(0,1) from Philox keyed by
 * (*seed_dev, salt, b, v) -- the Gumbel-max trick: the arg-max is distributed as softmax(logits).
 *   ws: dvae_vocab_ce_ws_floats(B, V, H) floats. */
int dvae_vocab_sample_step(const float* h, int64_t ldh, int B, int H, int V, const float* w,
                           const float* bias, const uint64_t* seed_dev, uint32_t salt, int64_t* tokens_out,
                           int64_t tok_stride, float* ws, void* stream);

/* Same, decided on the DEVICE: when forced_flag_dev != NULL and *forced_flag_dev != 0 the call is a no-op and the token
 * already in tokens_out stays (the teacher-forced input of vae/model.py:464-466).  The coin of every decoding step lives in
 * device memory, so ONE captured CUDA graph serves every draw of the teacher-forcing coins. */
int dvae_vocab_sample_step_ex(const float* h, int64_t ldh, int B, int H, int V, const float* w,
                              const float* bias, const uint64_t* seed_dev, uint32_t salt, int64_t* tokens_out,
                              int64_t tok_stride, const int32_t* forced_flag_dev, float* ws, void* stream);

/* Decoding many steps against the same W_out: split it ONCE into the fp16 operand planes the vocabulary kernels read
 * (dvae_vocab_w_planes; planes: dvae_vocab_w_planes_floats(V, H) floats) and hand them to every step.  The step then
 * splits only its B x H decoder states and runs the bulk-copy-fed projection of the forward pass; shapes that kernel does
 * not take (B < 256, V < 1024, H % 32 != 0) fall back to dvae_vocab_sample_step_ex.  w_planes must be current with w. */
int64_t dvae_vocab_w_planes_floats(int V, int H);
int dvae_vocab_w_planes(const float* w, int V, int H, float* planes, void* stream);
int dvae_vocab_sample_step_planes(const float* h, int64_t ldh, int B, int H, int V, const float* w,
                                  const float* bias, const float* w_planes, const uint64_t* seed_dev, uint32_t salt,
                                  int64_t* tokens_out, int64_t tok_stride, const int32_t* forced_flag_dev, float* ws,
                                  void* stream);

/* Length recount of sampled sentences before they are re-encoded (scripts/evaluation/consistency.py:186-190):
 * lengths_out[b] = max(min_len, T - #{t : tokens[b,t] == eos or tokens[b,t] == pad}).  The reference computes this with
 * torch ops on the token tensor it built on the CPU; here it stays on the device between the sampled decode and the
 * re-encode.  min_len = 0 reproduces the reference exactly (which then fails inside pack_padded_sequence on an empty
 * row); the evaluation path passes 1. */
int dvae_recount_lengths(const int64_t* tokens, int64_t tok_stride_b, int64_t tok_stride_t, int B, int T,
                         int64_t eos, int64_t pad, int64_t min_len, int64_t* lengths_out, void* stream);

/* Corpus BLEU of predicted sentences against their inputs: `compute_bleu` (vae/losses.py:128-134), i.e. torchtext 0.6
 * `bleu_score` (max_n = 4, weights 0.25, one reference per candidate) over rows cut by `tensor2text` (vae/utils.py:225).
 * Each row of `ref` [B, T_ref] and `cand` [B, T_cand] (row strides in elements, tokens contiguous) is cut after its first
 * `eos` (the whole row if it has none) and then loses its first and last token ([1:-1]: SOS and EOS, or SOS and the last
 * token of a row without EOS).  Token ids are compared, not words: the same result as the reference's strings because
 * its idx2word is injective (the vocabulary is built from sorted unique tokens, run.py:491-504).
 *   dvae_bleu_counts: ADDS this batch's statistics into counts[10] = {clipped n-gram matches n = 1..4, candidate n-grams
 *                     n = 1..4, candidate length, reference length}, so a corpus accumulates over calls and ranks (zero the
 *                     counters first).  T_ref and T_cand may differ; each must be <= DVAE_BLEU_MAX_T (else DVAE_EINVAL).
 *   dvae_bleu_counts_ex: dvae_bleu_counts with t_max (device memory, one int32; NULL = no bound): each row ends at
 *                     min(T_ref, *t_max) resp. min(T_cand, *t_max) columns.  For rows padded beyond their batch's own
 *                     length: a row without EOS is cut at the batch's length, as the unpadded row would be, so one
 *                     captured call serves every padded length.
 *   dvae_bleu_score : score_out[0] = 0 if any clipped count is 0, else
 *                     exp(min(1 - ref_len / cand_len, 0)) * exp(sum_n 0.25 log(clipped_n / total_n)), in float64,
 *                     stored as float32 in device memory (one thread; capturable in a CUDA graph). */
#define DVAE_BLEU_MAX_T 256
int dvae_bleu_counts(const int64_t* ref, int64_t ref_stride, int T_ref, const int64_t* cand, int64_t cand_stride,
                     int T_cand, int B, int64_t eos, int64_t* counts, void* stream);
int dvae_bleu_counts_ex(const int64_t* ref, int64_t ref_stride, int T_ref, const int64_t* cand, int64_t cand_stride,
                        int T_cand, int B, int64_t eos, const int* t_max, int64_t* counts, void* stream);
int dvae_bleu_score(const int64_t* counts, float* score_out, void* stream);

/* Backward: d_h [N,H], d_w [V,H], d_bias [V] (all overwritten) for d(loss) = grad_scale_dev[0]
 * (NULL = 1).  Softmax tiles are recomputed from h, w and the saved lse.
 *   ws: dvae_vocab_ce_bwd_ws_floats(N, V, H) floats.
 *   fwd_ws: NULL, or the workspace of the dvae_vocab_ce_fwd call on the SAME h and w if it has not been touched since:
 *   its fp16 operand planes are reused instead of being rebuilt (two fewer kernels). */
int64_t dvae_vocab_ce_bwd_ws_floats(int N, int V, int H);
int dvae_vocab_ce_bwd(const float* h, int64_t ldh, int T1, int B, int H, int V, const float* w,
                      const float* bias, const int64_t* targets, int64_t tgt_stride_b,
                      const int64_t* lengths, const float* lse, const float* grad_scale_dev,
                      float* d_h, int64_t lddh, float* d_w, float* d_bias, const float* fwd_ws, float* ws,
                      void* stream);

/* Backward of dvae_vocab_ce_fwd_live: same arguments as dvae_vocab_ce_bwd, with fwd_ws (required) the workspace of the
 * dvae_vocab_ce_fwd_live call on the same h, w and lengths, untouched since.  Only live rows enter the GEMMs; the other
 * rows of d_h are zero, as they are in dvae_vocab_ce_bwd. */
int dvae_vocab_ce_bwd_live(const float* h, int64_t ldh, int T1, int B, int H, int V, const float* w,
                           const float* bias, const int64_t* targets, int64_t tgt_stride_b,
                           const int64_t* lengths, const float* lse, const float* grad_scale_dev,
                           float* d_h, int64_t lddh, float* d_w, float* d_bias, const float* fwd_ws, float* ws,
                           void* stream);

/* ---------------------------------------------------------------------------------------------
 * Train-step tail: clip_grad_norm_(5.0) + Adam + zero_grad (run.py:255,261-262) over ONE flat
 * parameter buffer.
 *   dvae_grad_sumsq: sumsq[0] = sum(g^2) (deterministic two-stage reduction; ws >= 1024 floats+1)
 *   dvae_clip_adam : coef = min(1, max_norm / (sqrt(sumsq) + 1e-6)); g *= coef * grad_scale;
 *                    torch.optim.Adam update with hyper[0]=lr, hyper[1]=beta1, hyper[2]=beta2,
 *                    hyper[3]=eps, hyper[4]=step (1-based, as float), all read from DEVICE memory;
 *                    g is zeroed afterwards when zero_grad != 0.
 * ------------------------------------------------------------------------------------------- */
int dvae_grad_sumsq(const float* g, int64_t n, float* sumsq, float* ws, void* stream);
int dvae_clip_adam(float* p, float* g, float* m, float* v, int64_t n, const float* sumsq,
                   float max_norm, float grad_scale, const float* hyper_dev, int zero_grad,
                   void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DVAE_B200_H_ */
