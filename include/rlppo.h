/*
 * rlppo.h -- C-ABI of librlppo_b200.so: the B200-native (sm_100a) learner hot path of rlgym-ppo.
 *
 * The reference (AechPro/rlgym-ppo v1.3.13) is pure Python and has no FFI; its boundary for this path is
 * its Python class surface (SURVEY.md 8b).  The Python classes in rlgym_ppo_b200/ keep that surface and
 * bind these entry points with ctypes (INTEGRATION.md shows the stub).  Each entry point cites the
 * reference code it replaces.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; no torch types.
 *   - Every pointer is a DEVICE pointer owned by the caller unless the name starts with `h_` (host).
 *   - No allocation, no host synchronisation, no stream creation inside; work is enqueued on `stream`
 *     (a cudaStream_t passed as void*; NULL = legacy default stream).  All calls are CUDA-graph capturable.
 *   - Return 0 on success, <0 on error; rlppo_last_error() gives the message (thread-local).
 *   - There is no CPU fallback: every compute entry point fails with RLPPO_ERR_DEVICE when the current
 *     device is not compute capability 10.x.
 *   - bf16 buffers are passed as uint16_t*.  "ld" = leading dimension (row stride) in elements.
 */
#ifndef RLPPO_H_
#define RLPPO_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RLPPO_OK 0
#define RLPPO_ERR_ARG (-1)
#define RLPPO_ERR_CUDA (-2)
#define RLPPO_ERR_DEVICE (-3)
#define RLPPO_ERR_WORKSPACE (-4)

/* ---- library ------------------------------------------------------------------------------------ */
/* 101: the layer-wise GEMM, policy-head and value-head entry points and rlppo_rows_to_bf16 have one form each, under the
 * plain name and with the argument list of the split-operand / standardising form it absorbed (those names are gone).
 * A binding written against 100 would pass the old, shorter argument lists to the same names without any error: check
 * this number before binding. */
int rlppo_version(void);
const char* rlppo_last_error(void);
/* 0 if the current CUDA device can run the sm_100a kernels; RLPPO_ERR_DEVICE otherwise. */
int rlppo_device_check(void);

/* ---- (b-2) GAE: rlgym_ppo/util/torch_functions.py:36-78 compute_gae --------------------------------
 * One-pass segmented reverse scan (decoupled look-back) over the flat rollout.
 *   delta_t = clip(r_t/std,-10,10) + gamma*V[t+1]*(1-done_t) - V[t]      (std = *ret_std, NULL: raw r)
 *   A_t = delta_t + gamma*lambda*(1-done_t)*(1-trunc_t)*A_{t+1};  R_t = r_t + gamma*(1-done_t)*(1-trunc_t)*R_{t+1}
 * Rounding points follow what NumPy>=2 executes in the reference (delta in f32, A and R carried in f64).
 *   trunc            f32[n] (trunc_is_f64=0) or f64[n] (=1; the dtype collect_timesteps produces,
 *                    batched_agent_manager.py:159-168)
 *   values           f32[n+1] (value net on [states ; next_states[-1]], learner.py:347-352)
 *   adv, vtarget, ret  f32[n] outputs (advantages, V[:-1]+A, returns)
 *   ret_head64       optional f64[n_head]: the first n_head returns un-rounded (fed to Welford,
 *                    learner.py:368-372)
 *   carry_in         optional f64[2] {A_n, R_n}: values just right of this chunk (sharded scan); NULL = 0
 *   ws               workspace of rlppo_gae_workspace_bytes(n) bytes (contents ignored; cleared inside)
 * Algorithmic traffic: 28 B/step (16 read + 12 written). */
size_t rlppo_gae_workspace_bytes(int64_t n);
int rlppo_gae_f32(const float* rew, const float* done, const void* trunc, int trunc_is_f64,
                  const float* values, int64_t n, double gamma, double lambda, const float* ret_std,
                  float* adv, float* vtarget, float* ret, double* ret_head64, int64_t n_head,
                  const double* carry_in, void* ws, size_t ws_bytes, void* stream);
/* Affine summary of a chunk for the sharded scan (SURVEY.md 8e): out f64[4] = {aA, bA, aR, bR} with
 * A_first = bA + aA*A_right, R_first = bR + aR*R_right. */
int rlppo_gae_chunk_summary(const float* rew, const float* done, const void* trunc, int trunc_is_f64,
                            const float* values, int64_t n, double gamma, double lambda,
                            const float* ret_std, double* out4, void* ws, size_t ws_bytes, void* stream);

/* Sharded scan, step 2 (SURVEY.md 8e): summaries f64[world,4] = every chunk's rlppo_gae_chunk_summary (chunk 0 = the start
 * of the rollout), gathered from the ranks.  carry2 f64[2] = {A, R} just right of chunk `rank`: the chunks to its right
 * composed onto 0, rightmost first.  Feed it to rlppo_gae_f32 as carry_in. */
int rlppo_gae_compose_carry(const double* summaries, int rank, int world, double* carry2, void* stream);

/* ---- (b-3) WelfordRunningStat: rlgym_ppo/util/running_stats.py:30-69 ------------------------------
 * Sequential Welford over n samples of width dim, bit-faithful to update() (:37-46): state mean/m2 f32[dim],
 * count i64[1]; f64 intermediates for f64 samples (NumPy>=2), f32 for f32 samples.  Afterwards writes
 * std_out[dim] (:60-69: ones if count<2, zero variance -> 1) and mean_out[dim] (:54-58) if non-NULL. */
int rlppo_welford_update(float* mean, float* m2, int64_t* count, const void* samples, int samples_are_f64,
                         int64_t n, int dim, float* std_out, float* mean_out, void* stream);

/* Merge of Welford states (running_stats.py:71-98, increment_from_serialized_other): folds n_others states into
 * (mean, m2, count) in order, bit for bit the host formula applied other after other: f32 round-to-nearest, no
 * contraction, counts converted to f32 as NumPy 2 converts a Python int (via double), mean (c*mu + c'*mu')/C and
 * m2 + m2' + ((delta^2*c)*c')/C; an other with count 0 is skipped.  Other i is the block at
 * others + i*other_stride_bytes laid out as [count i64 | mean f32[dim] | m2 f32[dim] | ...] (the device state of
 * WelfordRunningStat), so blocks all-gathered from data-parallel ranks merge in place; stride % 8 == 0.  Writes
 * std_out / mean_out as rlppo_welford_update does.  Any dim >= 1; one block, no host synchronisation, graph-capturable. */
int rlppo_welford_merge(float* mean, float* m2, int64_t* count, const void* others, int64_t other_stride_bytes,
                        int n_others, int dim, float* std_out, float* mean_out, void* stream);

/* ---- (c-1) ExperienceBuffer store: rlgym_ppo/ppo/experience_buffer.py:17-37,54-80 -----------------
 * The FIFO `_cat` as a ring: logical row i lives at physical row (start+i) % capacity.  The host keeps
 * (start,size); these kernels move rows.  rlppo_ring_append copies n_rows rows of `src` (row-major,
 * src_ld elements apart, element type f32, or f64 when src_is_f64 -> cast to f32 like torch.as_tensor)
 * to physical rows (phys_first + i) % capacity of `ring` (row width `width`, ld `ring_ld`).
 * If ring_bf16 != NULL the same rows are also written as bf16 (ld bf16_ld, zero padded to bf16_ld). */
int rlppo_ring_append(float* ring, int64_t ring_ld, uint16_t* ring_bf16, int64_t bf16_ld, int64_t capacity,
                      int64_t phys_first, const void* src, int src_is_f64, int64_t src_ld, int64_t n_rows,
                      int width, void* stream);

/* All fields of one submit_experience in ONE launch (nine rings, experience_buffer.py:68-80). */
typedef struct rlppo_append_field {
    float* ring;            /* f32 ring [capacity, ring_ld] */
    int64_t ring_ld;
    uint16_t* ring_bf16;    /* optional bf16 side copy (zero padded to bf16_ld), else NULL */
    int64_t bf16_ld;
    const void* src;        /* new rows, f32 or f64 */
    int64_t src_ld;
    int32_t src_is_f64;
    int32_t width;
} rlppo_append_field;
int rlppo_ring_append_fields(const rlppo_append_field* h_fields, int n_fields, int64_t capacity,
                             int64_t phys_first, int64_t n_rows, void* stream);
/* Same, with the ring position kept ON THE DEVICE: d_state = int64[2] {start, size} (logical row 0 lives at physical row
 * `start`, `size` valid rows).  Rows go to (start + size + i) % capacity and d_state is advanced afterwards exactly as
 * `_cat` would (experience_buffer.py:17-37: once full, the oldest rows fall out).  Nothing about the position is baked
 * into the launch, so a CUDA graph that contains this call keeps following the ring when it is replayed. */
int rlppo_ring_append_fields_dev(const rlppo_append_field* h_fields, int n_fields, int64_t capacity,
                                 int64_t* d_state, int64_t n_rows, void* stream);

/* ---- (c-2) minibatch gather: experience_buffer.py:82-102 _get_samples ------------------------------
 * idx: int64[B] LOGICAL indices (a slice of RandomState.permutation, generated on the host so the
 * stream is NumPy's own); physical row = (start + idx) % capacity.  Any output may be NULL.
 * d_start: optional device int64[1] overriding `start` (a captured CUDA graph then follows the ring as it wraps).
 *   out_actions/out_logp/out_values/out_adv  f32[B];  out_states f32[B,obs] (exact copy: the public
 *   get_all_batches_shuffled contract);  out_states_bf16 [B, bf16_ld] from the bf16 ring (GEMM operand). */
int rlppo_gather_batch(const float* actions, const float* logp, const float* values, const float* adv,
                       const float* states, int64_t states_ld, const uint16_t* states_bf16, int64_t bf16_ld,
                       int obs_dim, int64_t capacity, int64_t start, const int64_t* d_start, const int64_t* idx,
                       int64_t B, float* out_actions, float* out_logp, float* out_values, float* out_adv,
                       float* out_states, uint16_t* out_states_bf16, void* stream);
/* Host-side NumPy-legacy permutation (experience_buffer.py:98 `self.rng.permutation(total)`):
 * MT19937 + masked-rejection Fisher-Yates, bit-exact with np.random.RandomState.  h_key: uint32[624],
 * h_pos: int32[1] (both updated in place so the caller can set_state() the NumPy object back). */
int rlppo_host_permutation(uint32_t* h_key, int32_t* h_pos, int64_t n, int64_t* h_out);

/* ---- operand preparation ------------------------------------------------------------------------- */
/* f32 [n_rows, width] (ld src_ld) -> bf16 [n_rows, dst_ld], zero padded; used for the value-net input
 * [states ; next_states[-1]] (learner.py:347-349) and policy inference obs.
 *   mean, std f32[width] (both or neither): standardise first, clip((x-mean)/std, -clip, clip)
 *     (batched_agent_manager.py:303-315, clip = 5); NULL: the rows as they are.
 *   dst_f32 (optional, ld dst_f32_ld; needs mean): the standardised rows in f32 as well -- what the trajectory stores.
 *   Exactly one of mean / std NULL, or dst_f32 without mean: RLPPO_ERR_ARG. */
int rlppo_rows_to_bf16(const float* src, int64_t src_ld, int64_t n_rows, int width, const float* mean,
                       const float* std, float clip, uint16_t* dst, int64_t dst_ld, float* dst_f32,
                       int64_t dst_f32_ld, void* stream);
/* fp32 master weight W [out,in] (torch nn.Linear layout) -> bf16 W [out_pad, in_pad] (K-major operand of
 * the forward GEMM) and, if wt != NULL, bf16 W^T [in_pad, out_pad] (operand of the dgrad GEMM). */
int rlppo_weight_to_bf16(const float* w, int out_f, int in_f, uint16_t* wq, int64_t wq_ld, int out_pad,
                         uint16_t* wt, int64_t wt_ld, int in_pad, void* stream);

/* ---- precision mode "fp32": split bf16 operands on the same tcgen05 kernels ------------------------------
 * The reference computes its Linear layers in fp32 (torch CPU/GPU SGEMM, discrete_policy.py:22-31,
 * value_estimator.py:19-28).  With plain bf16 operands the forward pre-activations carry ~1e-3 relative error, which
 * flips ReLU masks of near-zero units and moves per-tensor gradients by several per cent -- outside the 1e-3 parity bar
 * (profiles/r02_precision_study.md).  In this mode every f32 matrix is stored as `parts` bf16 matrices side by side
 * in one buffer (value = part0 + part1 + part2; part q in columns [q*pstride, q*pstride + cols), pstride a multiple of
 * 64 columns, padding zero) and a GEMM accumulates the products part_i(A) x part_j(B) for i + j < order into the same
 * fp32 TMEM accumulator, smallest terms first:
 *   forward / heads: 3 x 3 parts, order 3 -> 6 products, ~2^-24 per product (fp32-equivalent pre-activations);
 *   dgrad / wgrad:   2 x 2 parts, order 2 -> 3 products, ~2^-16 (no branch points in the backward: linear errors only).
 * The GEMM and policy-head entry points below take the split descriptor `sp`: they run a longer k loop (a "k schedule"
 * of part pairs) and epilogues that write their f32 result as out_parts bf16 parts.  a = the row operand (x, dy, h),
 * b = the weight operand (w, wt; for wgrad: a = dy, b = x).  sp == NULL means plain bf16 operands. */
typedef struct rlppo_split {
    int32_t a_parts;        /* parts of the first (row) operand, 1..3 */
    int32_t b_parts;        /* parts of the second (weight) operand, 1..3 */
    int32_t order;          /* products kept: i + j < order */
    int32_t out_parts;      /* parts the result is written as, 1..3 */
    int64_t a_pstride;      /* column offset between parts of the first operand (elements) */
    int64_t b_pstride;      /* ... of the second operand */
    int64_t out_pstride;    /* ... of the output */
} rlppo_split;
/* f32 rows -> parts (optionally standardised first, as rlppo_rows_to_bf16; mean/std NULL: plain). */
int rlppo_rows_split_bf16(const float* src, int64_t src_ld, int64_t n_rows, int width, const float* mean,
                          const float* std, float clip, uint16_t* dst, int64_t dst_ld, int parts, int64_t pstride,
                          void* stream);
/* fp32 master weight W [out,in] -> split W [out_rows, q_parts*q_pstride] (forward operand) and/or split
 * W^T [in_rows, t_parts*t_pstride] (dgrad operand); either output may be NULL.  Padding rows/columns are zeroed. */
int rlppo_weight_split_bf16(const float* w, int out_f, int in_f, uint16_t* wq, int64_t wq_ld, int q_parts,
                            int64_t q_pstride, int out_rows, uint16_t* wt, int64_t wt_ld, int t_parts,
                            int64_t t_pstride, int in_rows, void* stream);

/* ---- (a-3, d-2) MLP on tcgen05 tensor cores: discrete_policy.py:22-42, value_estimator.py:19-36 ----
 * All GEMMs: bf16 operands staged by TMA (128B swizzle), fp32 accumulation in TMEM, one elected thread
 * issuing tcgen05.mma, epilogue warps reading TMEM with tcgen05.ld.  M = rows (timesteps).
 *
 * rlppo_linear_fwd:  Y[M,N] = act(X[M,K] * W[N,K]^T + bias)   (nn.Linear + ReLU), Y bf16.
 *   x ld = ldx (>= K, multiple of 8), w bf16 [>=N rows, ldw], bias f32[N] or NULL, relu 0/1.
 *   bias_n: entries of `bias` (0 = N): lets a Linear whose width is not a multiple of 8 (21 logits, 2n outputs) run with
 *   N padded to 8 without reading past its bias vector. */
int rlppo_linear_fwd(const uint16_t* x, int64_t ldx, const uint16_t* w, int64_t ldw, const float* bias, int bias_n,
                     uint16_t* y, int64_t ldy, int64_t M, int N, int K, int relu, const rlppo_split* sp, void* stream);
/* rlppo_linear_dgrad: dX[M,K] = (dY[M,N] * W[N,K]) (.) (Hprev > 0); wt = bf16 W^T [K, ldwt>=N].
 *   K >= 1 need not be a multiple of 8: dX is written over pad8(K) columns (lddx, ldh multiples of 8 covering
 *   pad8(K)); wt rows past K are read as zeros, so dX's padding columns come out zero.
 *   hprev = the ReLU output that was this layer's input (bf16 [M,ldh]) or NULL (no mask).
 *   db_below (optional f32[K]) += column sums of the stored dX over its K true columns (= the bias gradient of the
 *   layer that produced Hprev, ppo_learner.py:179-180 autograd): saves that layer's separate column-sum pass over dX.
 *   Split operands: the ReLU mask is read from part 0 of hprev (x > 0 <=> bf16(x) > 0); db_below sums the un-split f32
 *   values. */
int rlppo_linear_dgrad(const uint16_t* dy, int64_t lddy, const uint16_t* wt, int64_t ldwt, const uint16_t* hprev,
                       int64_t ldh, uint16_t* dx, int64_t lddx, float* db_below, int64_t M, int N, int K,
                       const rlppo_split* sp, void* stream);
/* rlppo_linear_wgrad: dW[N,K] += dY[M,N]^T * X[M,K]  (fp32, torch [out,in] layout with ld = lddw) and
 *   db[N] += column sums of dY (if db != NULL; over all parts of a split dY).  Split over M across the SMs; fp32
 *   atomics. */
int rlppo_linear_wgrad(const uint16_t* dy, int64_t lddy, const uint16_t* x, int64_t ldx, float* dw, int64_t lddw,
                       float* db, int64_t M, int N, int K, const rlppo_split* sp, void* stream);

/* All weight gradients of an optimiser step in ONE persistent launch (<= 8 layers): for every item
 * dW[N,K] += dY[M,N]^T * X[M,K] as rlppo_linear_wgrad, but dY is read once per 256 k (not once per 128), row
 * splits are balanced across layers by byte volume, and seven launches become one. */
typedef struct rlppo_wgrad_item {
    const uint16_t* dy;     /* bf16 [M, lddy] */
    int64_t lddy;
    const uint16_t* x;      /* bf16 [M, ldx] */
    int64_t ldx;
    float* dw;              /* f32 [N, lddw], accumulated */
    int64_t lddw;
    int64_t M;
    int32_t N, K;
    float* db;              /* optional f32 [N], accumulated: column sums of dy (the Linear's bias gradient) */
} rlppo_wgrad_item;
int rlppo_wgrad_multi(const rlppo_wgrad_item* h_items, int n_items, void* stream);

/* Policy head, sampling (DiscreteFF.get_action, discrete_policy.py:44-62): logits = H*W^T + b over
 * n_actions <= 256, softmax, clamp(1e-11,1), categorical sample by inverse CDF, log-prob of the sample.
 *   u_inject   optional f32[M] uniforms in [0,1) (tests); NULL -> Philox4x32-10(seed, offset + row)
 *   actions_out f32[M] (the manager casts actions to f32, batched_agent_manager.py:204) and/or
 *   actions_i64_out int64[M]; logp_out f32[M]; probs_out optional f32[M, n_actions] (get_output).
 *   deterministic != 0: per-row argmax, logp of it (the reference's deterministic branch returns one
 *   global argmax, discrete_policy.py:56-57; the per-row form is what its batch-of-1 use means).
 *   sp: split operands of the head GEMM, or NULL. */
int rlppo_policy_head_sample(const uint16_t* h, int64_t ldh, const uint16_t* w, int64_t ldw,
                             const float* bias, int64_t M, int n_actions, int K, const float* u_inject,
                             uint64_t seed, uint64_t offset, int deterministic, float* actions_out,
                             int64_t* actions_i64_out, float* logp_out, float* probs_out, const rlppo_split* sp,
                             void* stream);

/* Policy head, training (DiscreteFF.get_backprop_data discrete_policy.py:64-80 + ppo_learner.py:153-177
 * + the analytic backward of SURVEY.md A.3), fused into the head GEMM's epilogue:
 *   p = clamp(softmax(z),1e-11,1); logp = log p[a]; H = -sum p log p; ratio = exp(logp - old_logp);
 *   loss terms; dz[M, lddz] (bf16) = d(ppo_loss)/dz with weight inv_batch = 1/batch_size;
 *   metrics f32[8] accumulated with atomics: [0] sum entropy, [1] sum kl, [2] sum clipped-count,
 *   [3] sum min(ratio*A, clip(ratio)*A), [4] rows processed; [5..7] reserved.
 *   logp_out optional f32[M].
 *   sp: split operands, or NULL; d(logits) is then written as sp->out_parts parts of out_pstride columns each
 *   (lddz >= out_parts * out_pstride). */
int rlppo_policy_head_train(const uint16_t* h, int64_t ldh, const uint16_t* w, int64_t ldw,
                            const float* bias, int64_t M, int n_actions, int K, const float* actions,
                            const float* old_logp, const float* adv, float inv_batch, float clip,
                            float ent_coef, uint16_t* dz, int64_t lddz, float* logp_out, float* metrics,
                            const rlppo_split* sp, void* stream);

/* Value head (ValueEstimator last Linear(.,1), value_estimator.py:27; MSELoss ppo_learner.py:176),
 * fused SIMT pass over the last hidden activation H[M,K] (bf16), 1 <= K <= 28672:
 *   v = H*w + b  -> values_out f32[M] (if non-NULL).
 *   if targets != NULL: dv = 2*inv_batch*(v - target); dH[M,lddh] (bf16) = dv * w (.) (H > 0);
 *   dw[K] += sum_m dv*H;  db[1] += sum dv;  metrics[5] += sum (v-target)^2, metrics[6] += rows.
 *   H is given as h_parts split parts h_pstride columns apart and dH written as dh_parts parts dh_pstride apart
 *   (1..3 parts each, strides multiples of 8 covering pad8(K); plain bf16: 1, 0, 1, 0).  H and dH rows span pad8(K)
 *   columns (ldh, lddh multiples of 8 covering it): H's columns K..pad8(K)-1 must be zero, dH's are written as zeros;
 *   w and dw hold exactly K floats.  K > 2048 runs a second kernel form (w and the dw partials in shared memory). */
int rlppo_value_head(const uint16_t* h, int64_t ldh, const float* w, const float* bias, int64_t M, int K,
                     float* values_out, const float* targets, float inv_batch, uint16_t* dh, int64_t lddh,
                     float* dw, float* db, float* metrics, int h_parts, int64_t h_pstride, int dh_parts,
                     int64_t dh_pstride, void* stream);

/* ---- (f-4) the other two action heads: multi_discrete_policy.py:16-89, continuous_policy.py:23-120 ------------
 * Per-row tails over the output of the policy's last Linear (run it with rlppo_linear_fwd, relu = 0, out_parts = 3:
 * z = the logits as split bf16 parts, fp32-exact).  z view: z [M, ldz], z_parts parts z_pstride columns apart.
 *
 * MultiDiscrete (21 logits = 8 categoricals with bins 3,3,3,3,3,2,2,2; torch_functions.py:81-122): log-prob and entropy
 * are SUMMED over the 8 distributions, the entropy then averaged over the minibatch.
 *   _train: get_backprop_data (:74-89) + the PPO loss block (ppo_learner.py:153-177) + its backward into the logits:
 *     actions f32 [M, >= 8] (bin index per distribution, as stored by the buffer), dz written as dz_parts bf16 parts of
 *     dz_cols columns (columns past 21 zeroed), metrics as rlppo_policy_head_train ([0] = sum of row entropies).
 *   _sample: get_action (:44-72): inverse-CDF draw per distribution (u_inject f32 [M,8] or Philox(seed, offset + row)),
 *     deterministic != 0: per-distribution argmax; actions_out f32 [M, ld_aout >= 8], logp_out f32 [M]. */
int rlppo_head_multi_discrete_train(const uint16_t* z, int64_t ldz, int z_parts, int64_t z_pstride, int64_t M,
                                    const float* actions, int64_t ld_act, const float* old_logp, const float* adv,
                                    float inv_batch, float clip, float ent_coef, uint16_t* dz, int64_t lddz,
                                    int dz_parts, int64_t dz_pstride, int dz_cols, float* logp_out, float* metrics,
                                    void* stream);
int rlppo_head_multi_discrete_sample(const uint16_t* z, int64_t ldz, int z_parts, int64_t z_pstride, int64_t M,
                                     const float* u_inject, uint64_t seed, uint64_t offset, int deterministic,
                                     float* actions_out, int64_t ld_aout, float* logp_out, void* stream);
/* Continuous (2n outputs -> Tanh; mean = first n, std = second n mapped onto [var_min, var_max]; diagonal Gaussian):
 *   _train: the reference's four-term log-pdf summed over the n actions (continuous_policy.py:40-59, :112), entropy =
 *     mean of Normal.entropy() over all M*n elements (:117-118), PPO block, backward through the affine map and Tanh.
 *   _sample: action = clamp(mean + std * N(0,1), -1, 1) (:91-92) with Box-Muller normals from Philox (n_inject f32 [M,n]
 *     overrides them); deterministic != 0: action = mean, log-prob 0 (:87-89). */
int rlppo_head_continuous_train(const uint16_t* z, int64_t ldz, int z_parts, int64_t z_pstride, int64_t M, int n_act,
                                float var_min, float var_max, const float* actions, int64_t ld_act,
                                const float* old_logp, const float* adv, float inv_batch, float clip, float ent_coef,
                                uint16_t* dz, int64_t lddz, int dz_parts, int64_t dz_pstride, int dz_cols,
                                float* logp_out, float* metrics, void* stream);
int rlppo_head_continuous_sample(const uint16_t* z, int64_t ldz, int z_parts, int64_t z_pstride, int64_t M, int n_act,
                                 float var_min, float var_max, const float* n_inject, uint64_t seed, uint64_t offset,
                                 int deterministic, float* actions_out, int64_t ld_aout, float* logp_out, void* stream);

/* ---- backward entry points for torch autograd (the modules' get_output / get_backprop_data / forward) ------------
 * The training heads above differentiate the PPO loss only.  These take the gradient of each forward output as a
 * DEVICE pointer (every one optional, NULL = zero; the entropy gradient is f32[1], nothing is read on the host) and
 * write d(logits) in the layout the head's weight / data gradient GEMMs consume, as the _train forms do.
 *   rlppo_policy_head_backward: head GEMM + epilogue as rlppo_policy_head_train (sp and dz as there), minus the loss
 *     block.
 *     d_logp f32[M] (gathered log-prob of `actions`), d_ent f32[1] (mean entropy: each row gets d_ent / M),
 *     d_probs f32[M, n_actions] (get_output's unclamped softmax, added outside the clamp mask):
 *     g_j = [1e-11 <= s_j <= 1] (d_logp/p_a [j == a] - (d_ent/M)(log p_j + 1)) + d_probs_j;  dz = s (.) (g - sum g s)
 *     (oracle/ref_oracle.py:552-555 with the PPO factors replaced by the upstream gradients).
 *   rlppo_head_multi_discrete_backward: dz_i = d_logp (onehot_i - p_i) - (d_ent/M) p_i (log p_i + H_g)
 *     (ref_oracle.py:441-449).  get_output's gradient IS d(logits): stage it with rlppo_rows_to_bf16 / _split_bf16.
 *   rlppo_head_continuous_backward: d_logp, d_ent (mean over M*n elements, ref_oracle.py:473-478) and get_output's
 *     d_mean / d_std f32[M, n], back through the affine map of the std half and the Tanh.
 *   rlppo_value_head_backward: rlppo_value_head's training pass (split parts as there) with dv = d_values[row] loaded:
 *     dH = dv * w (.) (H > 0);  dw[K] += sum_m dv*H;  db[1] += sum dv.  d_values is the head's only upstream gradient
 *     and is required (NULL: RLPPO_ERR_ARG); db may be NULL. */
int rlppo_policy_head_backward(const uint16_t* h, int64_t ldh, const uint16_t* w, int64_t ldw, const float* bias,
                               int64_t M, int n_actions, int K, const float* actions, const float* d_logp,
                               const float* d_ent, const float* d_probs, uint16_t* dz, int64_t lddz,
                               const rlppo_split* sp, void* stream);
int rlppo_head_multi_discrete_backward(const uint16_t* z, int64_t ldz, int z_parts, int64_t z_pstride, int64_t M,
                                       const float* actions, int64_t ld_act, const float* d_logp, const float* d_ent,
                                       uint16_t* dz, int64_t lddz, int dz_parts, int64_t dz_pstride, int dz_cols,
                                       void* stream);
int rlppo_head_continuous_backward(const uint16_t* z, int64_t ldz, int z_parts, int64_t z_pstride, int64_t M, int n_act,
                                   float var_min, float var_max, const float* actions, int64_t ld_act,
                                   const float* d_logp, const float* d_ent, const float* d_mean, const float* d_std,
                                   uint16_t* dz, int64_t lddz, int dz_parts, int64_t dz_pstride, int dz_cols,
                                   void* stream);
int rlppo_value_head_backward(const uint16_t* h, int64_t ldh, const float* w, int64_t M, int K,
                              const float* d_values, uint16_t* dh, int64_t lddh, float* dw, float* db,
                              int h_parts, int64_t h_pstride, int dh_parts, int64_t dh_pstride, void* stream);

/* ---- whole-network fused kernels (hidden widths 64/128/192/256, <= 4 hidden layers, obs <= 256, <= 128 actions) ----
 * One persistent tcgen05 kernel runs a 128-row tile of samples through the WHOLE Linear/ReLU stack, the head and
 * (training) the backward data path without leaving the SM: hidden activations live in shared memory as the next
 * GEMM's A operand, ReLU masks as bit words in shared memory.  HBM sees x once, and (training) H_l, d(logits) and
 * dL/dH_l once each -- they are the operands of rlppo_wgrad_multi, which contracts over all rows and also forms the
 * bias gradients (column sums of the dL/dH_l tiles it stages; rlppo_wgrad_item.db).
 * Replaces the per-layer sequence rlppo_linear_fwd x L + head + rlppo_linear_dgrad x L for these shapes.
 * All pointers device; bf16 as uint16_t; l = 0..n_hidden-1 hidden Linear layers, index n_hidden = the head. */
typedef struct rlppo_fused_net {
    int n_hidden;               /* 1..4 */
    int in_dim;                 /* observation width (<= 256) */
    int64_t in_ld;              /* row stride of x in elements (multiple of 8) */
    int hidden[4];              /* hidden widths */
    const uint16_t* wq[5];      /* forward operands W_l bf16 [out_pad8, ld]; [n_hidden] = policy head (NULL for value).
                                   Columns past in_features are never read.  The head's rows n_actions .. out_pad8-1
                                   are read and must be finite; no output depends on their values */
    int64_t wq_ld[5];
    const uint16_t* wt[5];      /* unused (kept for layout): the backward data GEMMs read wq[l] as an MN-major operand */
    int64_t wt_ld[5];
    const float* bias[5];       /* f32 biases; [n_hidden] = head bias (policy: n_actions, value: 1) */
    float* gbias[5];            /* only [n_hidden] of the value net (its head's scalar bias gradient) is written here;
                                   every other bias gradient comes from rlppo_wgrad_multi (item.db) */
    uint16_t* h[4];             /* out (training): H_l bf16 [M, hidden_l], ld h_ld.  Except the value net's
                                   h[n_hidden-1]: that activation feeds only the in-kernel value head, so it is never
                                   written and may be NULL */
    int64_t h_ld[4];
    uint16_t* dh[4];            /* out (training): dL/dH_l (ReLU-masked) bf16 [M, hidden_l] */
    int64_t dh_ld[4];
    uint16_t* dz;               /* out (policy training): d(ppo_loss)/d(logits) bf16 [M, pad8(n_actions)] */
    int64_t dz_ld;
} rlppo_fused_net;

/* DiscreteFF.get_backprop_data + PPO loss + backward data path (discrete_policy.py:64-80, ppo_learner.py:153-180,
 * SURVEY.md A.3).  metrics as rlppo_policy_head_train.  Weight and bias gradients: rlppo_wgrad_multi on (dz, H_L),
 * (dh[l], H_{l-1}), (dh[0], x) with item.db set. */
int rlppo_policy_train_fused(const rlppo_fused_net* net, const uint16_t* x, int64_t M, int n_actions,
                             const float* actions, const float* old_logp, const float* adv, float inv_batch,
                             float clip, float ent_coef, float* logp_out, float* metrics, void* stream);
/* DiscreteFF.get_action (discrete_policy.py:44-62) for all rows: same sampler contract as rlppo_policy_head_sample.
 * d_offset (optional): device counter added to `offset` -- a captured CUDA graph (one per environment tick,
 * batched_agent_manager.py:180-221) then draws fresh numbers on every replay; advance it with rlppo_u64_add. */
int rlppo_policy_infer_fused(const rlppo_fused_net* net, const uint16_t* x, int64_t M, int n_actions,
                             const float* u_inject, uint64_t seed, uint64_t offset, const uint64_t* d_offset,
                             int deterministic, float* actions_out, int64_t* actions_i64_out, float* logp_out,
                             void* stream);
/* *d_counter += inc (one thread; graph-capturable). */
int rlppo_u64_add(uint64_t* d_counter, uint64_t inc, void* stream);
/* ValueEstimator forward + MSE loss + backward data path (value_estimator.py:30-36, ppo_learner.py:146,176).
 * w_head f32[hidden_last] (the last Linear's weight row), gw_head f32[hidden_last] accumulated; metrics[5,6] as
 * rlppo_value_head; values_out optional f32[M]. */
int rlppo_value_train_fused(const rlppo_fused_net* net, const uint16_t* x, int64_t M, const float* w_head,
                            const float* targets, float inv_batch, float* gw_head, float* values_out,
                            float* metrics, void* stream);
/* Both nets of a PPO batch in ONE persistent launch: the work items are (net, 128-row tile) -- (net, pair of tiles) for
 * the two-CTA cluster form -- policy tiles first, dealt out over one CTA per SM: 2 x ceil(M/128) items instead of two
 * launches that each end on a partly filled round of tiles.  Arguments as rlppo_policy_train_fused + rlppo_value_train_fused (both nets read the same x; `metrics`
 * is the shared 8-float block: policy sums in [0,5), value sums in [5,7)).  ppo_learner.py:146-180 for one minibatch. */
int rlppo_policy_value_train_fused(const rlppo_fused_net* policy_net, const rlppo_fused_net* value_net,
                                   const uint16_t* x, int64_t M, int n_actions, const float* actions,
                                   const float* old_logp, const float* adv, float inv_batch, float clip, float ent_coef,
                                   float* logp_out, const float* w_head, const float* targets, float* gw_head,
                                   float* values_out, float* metrics, void* stream);
/* ValueEstimator forward only (learner.py:352): values_out f32[M]. */
int rlppo_value_infer_fused(const rlppo_fused_net* net, const uint16_t* x, int64_t M, const float* w_head,
                            float* values_out, void* stream);

/* ---- (d-6) clip_grad_norm_ + Adam: ppo_learner.py:187-193, torch.optim.Adam ------------------------
 * Flat fp32 arenas; `seg` describes n_seg contiguous segments (policy params, value params): seg_off
 * int64[n_seg+1].  rlppo_grad_sqnorm writes per-segment sum of squares to sqnorm f32[n_seg] (zeroed
 * inside).  rlppo_clip_adam then applies, per segment s: c = min(1, max_norm/(sqrt(sqnorm[s])+1e-6));
 * g = c*grad; m = lerp(m,g,1-b1); v = b2*v+(1-b2)g*g; step = ++step_count[s] (device i64);
 * p -= lr[s]/(1-b1^step) * m / (sqrt(v)/sqrt(1-b2^step) + eps).  lr f32[n_seg] on device
 * (update_learning_rate, learner.py:205-216, rewrites it).  delta_sq (optional f32[n_seg]) accumulates
 * nothing here; see rlppo_sqdiff. */
int rlppo_grad_sqnorm(const float* grads, const int64_t* h_seg_off, int n_seg, float* sqnorm, void* stream);
/* h_views (optional, <= 16): weight matrices inside the arena whose bf16 GEMM operands (W and W^T, see
 * rlppo_weight_to_bf16) are rewritten by the same launch, so no separate refresh pass is needed after a step. */
typedef struct rlppo_bf16_view {
    int64_t offset;         /* element offset of W [out_f, in_f] in the parameter arena */
    int32_t out_f, in_f;
    uint16_t* wq;           /* bf16 W, ld wq_ld */
    int64_t wq_ld;
    uint16_t* wt;           /* bf16 W^T, ld wt_ld, or NULL */
    int64_t wt_ld;
} rlppo_bf16_view;
int rlppo_clip_adam(float* params, const float* grads, float* m, float* v, const int64_t* h_seg_off,
                    int n_seg, const float* sqnorm, const float* lr, int64_t* step_count, double max_norm,
                    double beta1, double beta2, double eps, const rlppo_bf16_view* h_views, int n_views,
                    void* stream);
/* The two calls above as ONE launch (grid barrier between norm and update) with a deterministic, fixed-order norm:
 * what PPOLearner uses.  sqnorm_out (optional f32[n_seg]) receives the norms.  ws: device workspace of
 * rlppo_norm_clip_adam_workspace_bytes() bytes, zeroed by the caller once when it is allocated (the kernel leaves its
 * counters zero again).  Same arithmetic as rlppo_clip_adam; only the summation order of the norm differs. */
size_t rlppo_norm_clip_adam_workspace_bytes(void);
int rlppo_norm_clip_adam(float* params, const float* grads, float* m, float* v, const int64_t* h_seg_off,
                         int n_seg, float* sqnorm_out, const float* lr, int64_t* step_count, double max_norm,
                         double beta1, double beta2, double eps, const rlppo_bf16_view* h_views, int n_views,
                         void* ws, size_t ws_bytes, void* stream);
/* Data-parallel form of rlppo_norm_clip_adam: the gradient all-reduce of the reference-equivalent accumulation
 * (ppo_learner.py:134-193 sums (mb/B)-scaled minibatch gradients before ONE clip + Adam step; here the minibatch slices
 * live on `world` GPUs of one box) is done INSIDE the launch over NVLink peer mappings -- no separate collective.
 * h_peer_grads[r] / h_peer_flags[r]: rank r's gradient arena (f32[total]) and flag block (rlppo_peer_flag_bytes() bytes,
 * zeroed once by its owner before the first launch) as mapped into THIS process (e.g. torch symmetric memory
 * buffer_ptrs); entry `rank` is the local one.  gsum: local f32[total] scratch that receives the summed gradient (rank
 * order 0..world-1 on every rank: replicas stay bit-identical).  Every rank must make the same sequence of calls; the
 * launch ends only after all peers have finished reading this rank's arena, so the caller may overwrite it right after.
 * A peer that never arrives traps the kernel after ~2 min instead of hanging.  world <= 8.  Other arguments as above. */
size_t rlppo_peer_flag_bytes(void);
int rlppo_norm_clip_adam_peers(float* params, const float* const* h_peer_grads, void* const* h_peer_flags, int rank,
                               int world, float* gsum, float* m, float* v, const int64_t* h_seg_off, int n_seg,
                               float* sqnorm_out, const float* lr, int64_t* step_count, double max_norm, double beta1,
                               double beta2, double eps, const rlppo_bf16_view* h_views, int n_views, void* ws,
                               size_t ws_bytes, void* stream);
/* Two-shot form of the call above (reduce-scatter + all-gather inside the launch: 2 * 4n bytes over NVLink per rank
 * instead of (world-1) * 4n; what PPOLearner picks for arenas too big for the one-shot form).  h_peer_red[r]: rank r's
 * f32[total] buffer for the reduced gradient in symmetric memory, as mapped here (entry `rank` receives the full sum).
 * Validated on 2 and 8 x B200 (tests/dp_check.py: equal to the NCCL all-reduce to rounding, same bits on every rank,
 * thousands of launches under random per-rank skew). */
int rlppo_norm_clip_adam_peers2(float* params, const float* const* h_peer_grads, void* const* h_peer_flags,
                                const float* const* h_peer_red, int rank, int world, float* m, float* v,
                                const int64_t* h_seg_off, int n_seg, float* sqnorm_out, const float* lr,
                                int64_t* step_count, double max_norm, double beta1, double beta2, double eps,
                                const rlppo_bf16_view* h_views, int n_views, void* ws, size_t ws_bytes, void* stream);
/* out f32[n_seg] = per-segment sum (a-b)^2 (update magnitudes, ppo_learner.py:212-220). */
int rlppo_sqdiff(const float* a, const float* b, const int64_t* h_seg_off, int n_seg, float* out,
                 void* stream);

/* ---- wide discrete head: DiscreteFF with 257 <= n_actions <= 4096 -------------------------------------------------
 * The fused epilogue of rlppo_policy_head_* holds a row's logits in one TMEM tile (<= 256 actions).  Wider softmax
 * policies run their last Linear as rlppo_linear_fwd (relu = 0, out_parts = 3: fp32-exact logits as split bf16
 * parts, as the (f-4) heads above) and these per-row kernels over it, one warp per row.  The z view is as for the (f-4)
 * heads and must allow 16-byte accesses: z 16-byte aligned, ldz and z_pstride multiples of 8, every part pad8(n_actions)
 * columns wide.  The arithmetic is that of the epilogue forms (p = clamp(softmax(z), 1e-11, 1)); only the order of the
 * row sums differs.  Every entry point checks 257 <= n_actions <= 4096.
 *   _sample (DiscreteFF.get_action / get_output, discrete_policy.py:35-62): as rlppo_policy_head_sample: inverse-CDF
 *     draw against u * (total clamped mass), u from u_inject f32[M] or Philox4x32-10(seed, offset + row), subsequence 0,
 *     u = (x >> 8) / 2^24; deterministic != 0: per-row argmax (first of ties), logp = log clamp(1/S).  Outputs (any may be
 *     NULL, not all): actions_out f32[M], actions_i64_out int64[M], logp_out f32[M], probs_out f32[M, n_actions] (the
 *     unclamped softmax).
 *   _train (get_backprop_data :64-80 + the PPO loss block ppo_learner.py:146-180): as rlppo_policy_head_train, with
 *     actions f32[M] (clamped to [0, n_actions-1]), d(logits) written as dz_parts bf16 parts of dz_cols columns
 *     (dz_cols a multiple of 8 >= pad8(n_actions), dz_pstride apart; columns past n_actions zeroed), metrics f32[8] as
 *     there ([0..4] accumulated), logp_out optional f32[M].
 *   _backward (autograd, discrete_policy.py:35-80): as rlppo_policy_head_backward: d_logp f32[M], d_ent f32[1] (of the
 *     mean entropy), d_probs f32[M, n_actions] (of get_output's unclamped softmax), each optional; dz as for _train. */
int rlppo_head_discrete_sample(const uint16_t* z, int64_t ldz, int z_parts, int64_t z_pstride, int64_t M, int n_actions,
                               const float* u_inject, uint64_t seed, uint64_t offset, int deterministic,
                               float* actions_out, int64_t* actions_i64_out, float* logp_out, float* probs_out,
                               void* stream);
int rlppo_head_discrete_train(const uint16_t* z, int64_t ldz, int z_parts, int64_t z_pstride, int64_t M, int n_actions,
                              const float* actions, const float* old_logp, const float* adv, float inv_batch, float clip,
                              float ent_coef, uint16_t* dz, int64_t lddz, int dz_parts, int64_t dz_pstride, int dz_cols,
                              float* logp_out, float* metrics, void* stream);
int rlppo_head_discrete_backward(const uint16_t* z, int64_t ldz, int z_parts, int64_t z_pstride, int64_t M,
                                 int n_actions, const float* actions, const float* d_logp, const float* d_ent,
                                 const float* d_probs, uint16_t* dz, int64_t lddz, int dz_parts, int64_t dz_pstride,
                                 int dz_cols, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RLPPO_H_ */
