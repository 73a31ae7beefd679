/*
 * morl_b200.h -- C-ABI of libmorl_b200.so: the B200 (sm_100a) update engine for the batched
 * multi-objective value-update hot path of LucasAlegre/morl-baselines (reference @ a8acdbb).
 *
 * The reference has NO plugin / FFI layer (SURVEY.md section 8(b)): its boundary is the Python class API.
 * Each entry point below therefore replaces an *inline tensor-op sequence* of the reference; the
 * file:line it replaces is cited per function (paths relative to the reference root).
 *
 * Conventions (all entry points):
 *   - every pointer is a DEVICE pointer owned by the caller (PyTorch); the library never allocates,
 *     frees or retains device memory; tensors are contiguous row-major, base pointers 16-byte aligned;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it; no host sync, no
 *     allocation => safe under CUDA-graph capture; re-entrant (no mutable global state);
 *   - return value: 0 = success; negative = MORL_ERR_* argument error; positive = cudaError_t of
 *     the launch.  morl_last_error() returns a thread-local message for the last non-zero return;
 *   - there is NO CPU fallback: without a CUDA device every compute entry point returns an error.
 *
 * Row-index maps.  Several per-row inputs of the reference are broadcast by `Tensor.repeat` (tile) or
 * `repeat_interleave` (block).  Instead of materialising them, an input X with x_rows < N rows is
 * addressed as
 *      MORL_MAP_TILE  : X[k % x_rows]            (reference: b_rewards.repeat(num_sample_w, 1), envelope.py:285-291)
 *      MORL_MAP_BLOCK : X[k / (N / x_rows)]      (reference: sampled_w.repeat_interleave(B, 0), envelope.py:284)
 *   x_rows == N is the identity under both maps.
 *
 * Scalarisation arithmetic (`dot_mode`).  s = w . q over D objectives, fp32:
 *      MORL_DOT_UNFUSED : ((w0*q0 + w1*q1) + w2*q2) + ...   every op rounded (IEEE, no contraction).  This is
 *                         bit-equal to the reference's th.einsum on CPU for small products (N_cols < 128),
 *                         e.g. the reference default num_sample_w=4 and every max_action / gpi_action call.
 *      MORL_DOT_PAIRFMA : fl(fma(w1,q1, fl(w0*q0)) + fl(w2*q2))   (D==3 only) -- bit-equal to what MKL's sgemm
 *                         produces for th.einsum("br,bwar->bwa") on the build container's AVX-512 CPU once
 *                         W*A >= 192 (probe in DESIGN.md); offered so golden vectors of the real reference at the
 *                         north-star shape can be matched bit-for-bit.
 *      MORL_DOT_FMA     : fma(w2,q2, fma(w1,q1, fl(w0*q0)))   the GPU-native chain (what cuBLAS would do).
 *   argmax / argmin are always FIRST-occurrence (th.max / th.argmax / th.argmin semantics).
 */
#ifndef MORL_B200_H_
#define MORL_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MORL_B200_VERSION 100 /* 0.1.0 */

#if defined(__GNUC__)
#define MORL_API __attribute__((visibility("default")))
#else
#define MORL_API
#endif

/* argument errors (negative); positive returns are cudaError_t values */
#define MORL_OK 0
#define MORL_ERR_NULL (-1)        /* required pointer is NULL */
#define MORL_ERR_SHAPE (-2)       /* non-positive / inconsistent dimension */
#define MORL_ERR_ALIGN (-3)       /* base pointer not 16-byte aligned */
#define MORL_ERR_UNSUPPORTED (-4) /* dimension outside the compiled range (D > 8, A > 64, ...) */
#define MORL_ERR_NO_DEVICE (-5)   /* no CUDA device / wrong architecture */

#define MORL_DOT_UNFUSED 0
#define MORL_DOT_FMA 1
#define MORL_DOT_PAIRFMA 2

#define MORL_MAP_TILE 0
#define MORL_MAP_BLOCK 1

#define MORL_ROWS_REFERENCE 0 /* effective-batch row k = i*B + b  (reference order, envelope.py:284-291) */
#define MORL_ROWS_BMAJOR 1    /* effective-batch row k = b*W + i  (coalesced order used by the fused update)  */

#define MORL_MAX_D 8
#define MORL_MAX_A 64

MORL_API int morl_version(void);
MORL_API const char* morl_last_error(void);
/* number of SMs of the current device (148 on B200), or a negative MORL_ERR_* */
MORL_API int morl_device_sm_count(void);

/* ------------------------------------------------------------------------------------------------
 * Fused envelope-max TD target.   Replaces Envelope.envelope_target (multi_policy/envelope/envelope.py:404-440)
 * + the vector Bellman line (envelope.py:298), evaluated on the B*W DISTINCT (s'_b, w_j) rows instead of the
 * reference's B*W^2 tiled rows (SURVEY.md headline 2).
 *   q_online, q_target : f32 [B, W, A, D]   Q(s'_b, w_j)[a, :] of the online / target net (row b*W + j)
 *   wset               : f32 [W, D]         sampled weight vectors
 *   reward             : f32 [B, D], done : f32 [B]
 * For every (i, b):  (j*, a*) = first argmax_{j,a} wset[i] . q_online[b, j, a, :]
 *                    target[k, :] = reward[b, :] + ((1 - done[b]) * gamma) * q_target[b, j*, a*, :]   (unfused)
 * with k = i*B + b (MORL_ROWS_REFERENCE) or b*W + i (MORL_ROWS_BMAJOR).
 *   target_out : f32 [W*B, D];  pref_out, act_out : int32 [W*B] or NULL  (reference keeps them as int64, :424-426)
 */
MORL_API int morl_envelope_td_f32(const float* q_online, const float* q_target, const float* wset, const float* reward,
                         const float* done, float gamma, int B, int W, int A, int D, int dot_mode, int row_order,
                         float* target_out, int32_t* pref_out, int32_t* act_out, void* stream);

/* Double-DQN target with a per-row weight.  Replaces Envelope.ddqn_target (envelope.py:442-463) + :298, and the
 * non-GPI branch of GPIPD._reset_priorities (multi_policy/gpi_pd/gpi_pd.py:648-656).
 *   q_select, q_eval : f32 [N, A, D];  w : f32 [w_rows, D];  reward : f32 [r_rows, D] or NULL;  done : f32 [r_rows]
 *   a* = first argmax_a w_k . q_select[k, a, :];   out[k] = q_eval[k, a*, :]  (then Bellman if reward != NULL)
 */
MORL_API int morl_greedy_td_f32(const float* q_select, const float* q_eval, const float* w, int w_rows, int w_map,
                       const float* reward, const float* done, int r_rows, int r_map, float gamma, int N, int A,
                       int D, int dot_mode, float* target_out, int32_t* act_out, void* stream);

/* GPI-PD / GPI-LS critic-min target.  Replaces GPIPD.update's target block (gpi_pd.py:445-463):
 *   q_nets : f32 [n_nets, N, A, D] target nets;  n*(k,a) = first argmin_n w_k . q_nets[n,k,a,:];
 *   Q~[k,a,:] = q_nets[n*,k,a,:];  a* = first argmax_a w_k . Q~[k,a,:];  out = reward + ((1-done)*gamma) * Q~[k,a*,:]
 */
MORL_API int morl_critic_min_td_f32(const float* q_nets, int n_nets, const float* w, int w_rows, int w_map,
                           const float* reward, const float* done, int r_rows, int r_map, float gamma, int N,
                           int A, int D, int dot_mode, float* target_out, int32_t* act_out, void* stream);

/* GPI envelope over a policy/weight-support set with per-row weights.  Replaces GPIPD._envelope_target
 * (gpi_pd.py:662-690), GPIPD.gpi_action (gpi_pd.py:564-582; n_nets = 1, reward = NULL), its batched twin in
 * _rollout_dynamics (gpi_pd.py:379-387) and the M x M GPI evaluation of GPIPDContinuousAction.eval
 * (multi_policy/gpi_pd/gpi_pd_continuous_action.py:464-478).
 *   q_nets : f32 [n_nets, B, P, A, D];  w : f32 [w_rows, D]
 *   per (b,p,a): critic-min over n as above (scalarised with w_b), then (p*, a*) = first joint argmax_{p,a}
 *   out[b,:] = Q~[b,p*,a*,:]  (Bellman applied iff reward != NULL);  policy_out / act_out : int32 [B] or NULL
 */
MORL_API int morl_gpi_envelope_f32(const float* q_nets, int n_nets, const float* w, int w_rows, int w_map,
                          const float* reward, const float* done, int r_rows, int r_map, float gamma, int B, int P,
                          int A, int D, int dot_mode, float* out, int32_t* policy_out, int32_t* act_out,
                          void* stream);

/* Actor-critic vector targets (continuous-action algorithms), three "min over critics" rules (SURVEY App. A.4):
 *   MORL_AC_ELEMENTWISE_MIN : CAPQL  (multi_policy/capql/capql.py:326-331)  min_n per objective, - alpha*logp, vector target
 *   MORL_AC_SCALAR_MIN      : MOSAC  (single_policy/ser/mosac_continuous_action.py:435-442) scalarise, min, - alpha*logp;
 *                             out is [N] and the reward is scalarised with w as well
 *   MORL_AC_ARGMIN_GATHER   : GPI-PD continuous / TD3 (gpi_pd_continuous_action.py:397-403) first argmin_n w.q_n, gather vector
 *   q_nets : f32 [n_nets, N, D];  logp : f32 [N] or NULL;  w : [w_rows, D] (unused for ELEMENTWISE_MIN)
 */
#define MORL_AC_ELEMENTWISE_MIN 0
#define MORL_AC_SCALAR_MIN 1
#define MORL_AC_ARGMIN_GATHER 2
MORL_API int morl_actor_critic_td_f32(const float* q_nets, int n_nets, const float* w, int w_rows, int w_map,
                             const float* reward, const float* done, const float* logp, float alpha, float gamma,
                             int N, int D, int variant, float* target_out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Fused TD loss + gradient seed + PER priority for Envelope.  Replaces envelope.py:301-313 (gather taken action,
 * MSE, homotopy auxiliary loss) and :329-331 (|w . td| priorities of the first B rows, i.e. weight index 0).
 *   q_values : f32 [W*B, A, D] online net output on the effective batch (row order `row_order`)
 *   action   : int32 [B];  target_q : f32 [W*B, D];  wset : f32 [W, D]
 *   homotopy_lambda_dev : optional device f32 [1]; when non-NULL the kernels read lambda from it instead of the by-value argument, so a
 *              captured CUDA graph stays valid while the homotopy schedule (envelope.py:351-358) changes lambda every update
 *   loss_out : f32 [1] = (1-lambda)*mean((q-t)^2) + lambda*mean((w.q - w.t)^2)
 *   grad_q   : f32 [W*B, A, D] = d loss / d q_values (dense; zero off the taken action), or NULL
 *   q_taken  : f32 [W*B, D] the gathered Q(s,a) (optional, NULL to skip)
 *   prio_out : f32 [B] = | wset[0] . (q - t) | for rows with i == 0, or NULL
 *   workspace: device scratch of morl_td_workspace_bytes(W*B) bytes (no initialisation required)
 */
MORL_API size_t morl_td_workspace_bytes(int n_rows);
MORL_API int morl_td_mse_priority_f32(const float* q_values, const int32_t* action, const float* target_q,
                             const float* wset, float homotopy_lambda, const float* homotopy_lambda_dev, int B, int W, int A,
                             int D, int row_order, float* loss_out, float* grad_q, float* q_taken, float* prio_out, void* workspace,
                             void* stream);

/* Huber-style TD loss of GPI-PD.  Replaces gpi_pd.py:469-487 per net and :507-520 (priority = | w . max_n |delta_n| |).
 *   q_values : f32 [n_nets, N, A, D];  action : int32 [a_rows] (tile map);  target_q : f32 [N, D]
 *   target_q_gpi : f32 [N, D] or NULL (gpi_pd=True -> priorities from the GPI envelope target)
 *   loss_out : f32 [1] = (1/n_nets) * sum_n mean( where(|d|<mp, 0.5 d^2, mp |d|) )   (common/networks.py:90-100)
 *   grad_q   : f32 [n_nets, N, A, D] or NULL;   prio_out : f32 [p_rows] (first p_rows rows), raw |w . err| before clip/pow
 */
MORL_API int morl_td_huber_priority_f32(const float* q_values, int n_nets, const int32_t* action, int a_rows,
                               const float* target_q, const float* target_q_gpi, const float* w, int w_rows,
                               int w_map, float min_priority, int N, int A, int D, int p_rows, float* loss_out,
                               float* grad_q, float* prio_out, void* workspace, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Host halves of the replay path (CPU code in the same library; no CUDA call, usable without a device).
 *
 * Prioritised replay sum tree, reference common/prioritized_buffer.py:12-82 (class SumTree).  `tree` is ONE float64 array of
 * 2^n_levels - 1 nodes: level l (2^l nodes, l = 0 the root, l = n_levels - 1 the leaves) starts at element 2^l - 1.
 *   morl_host_sumtree_walk      : SumTree.sample after the uniform draw (:35-49): descend for each query value -> leaf index.
 *   morl_host_sumtree_batch_set : SumTree.batch_set (:73-82): np.unique(index, return_index) then node += (new - old) on every
 *                                 level in array order -- the same float64 operations in the same order, so the tree (and the
 *                                 indices later sampled from it) is bit-identical to the reference's.
 * Minibatch packing, reference common/buffer.py:84-94 (fancy-index gathers before the host->device copies):
 *   morl_host_gather_rows       : dst[i, :] = src[index[i], :] for rows of row_bytes bytes (dst: pinned staging memory).
 *   morl_host_gather_u8_to_i32  : same for uint8 action rows, widened to int32 (the reference's callers call .long()). */
MORL_API int morl_host_sumtree_walk(const double* tree, int n_levels, const double* queries, int n, long long* out_index);
MORL_API int morl_host_sumtree_batch_set(double* tree, int n_levels, const long long* index, const double* priority, int n);
MORL_API int morl_host_gather_rows(const void* src, long long row_bytes, const long long* index, int n, void* dst);
MORL_API int morl_host_gather_u8_to_i32(const unsigned char* src, long long row_elems, const long long* index, int n, int* dst);

/* ------------------------------------------------------------------------------------------------
 * Device-resident replay: index gather.  Replaces the 5 fancy-index gathers + 6 host->device copies of
 * ReplayBuffer.sample (common/buffer.py:82-94) / PrioritizedReplayBuffer.sample (common/prioritized_buffer.py:160-166).
 *   stores: obs/next_obs f32 [cap, obs_dim], action u8|f32 [cap, act_dim], reward f32 [cap, rew_dim], done f32 [cap]
 *   idx : int64 [B];  outputs are [B, *];  discrete actions (act_is_u8 != 0) are widened to int32.
 */
MORL_API int morl_replay_gather(const float* obs_store, const float* next_obs_store, const void* act_store,
                       const float* rew_store, const float* done_store, const int64_t* idx, int B, int obs_dim,
                       int act_dim, int rew_dim, int act_is_u8, int64_t capacity, float* obs_out,
                       float* next_obs_out, void* act_out, float* rew_out, float* done_out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Pareto non-dominated mask (maximisation).  Replaces get_non_pareto_dominated_inds (common/pareto.py:34-57):
 *   keep[i] = 1 iff no OTHER value weakly dominates pts[i] (only exact copies are >= in every coordinate) and,
 *   when remove_duplicates != 0, i is the first index holding its value.  Comparisons are exact in the input dtype;
 *   a row containing NaN is never kept.  pts : [N, D] row-major; keep : uint8 [N].  D <= MORL_MAX_D.
 */
MORL_API int morl_pareto_mask_f32(const float* pts, int N, int D, int remove_duplicates, uint8_t* keep, void* stream);
MORL_API int morl_pareto_mask_f64(const double* pts, int N, int D, int remove_duplicates, uint8_t* keep, void* stream);

/* Fixed-shape records for the ONE all-gather of per-rank non-dominated fronts per evaluation round (BASELINE.json north_star; the
 * reference has no multi-GPU path -- the call it replaces is the single-process archive update of multi_policy/morld/morld.py:306-335).
 *   record (float64) = [ count | cap x d rows | n_extra extras ]
 * morl_front_pack_f64   : rows of pts [n, d] with keep[i] != 0 (keep NULL = all), in input order; count is NOT clipped to cap (overflow is
 *                         visible to every rank after the gather); unused rows are -inf (dominated by any real point).  One block.
 * morl_front_unpack_f64 : gathered [world][1 + cap*d + n_extra] -> pts_out [world*cap, d] (input of the global prune) and
 *                         meta_out [world][1 + n_extra] (every rank's count and extras, contiguous).
 * No host synchronisation, no allocation: the whole exchange is stream-ordered. */
MORL_API int morl_front_pack_f64(const double* pts, const uint8_t* keep, int n, int d, int cap, const double* extras, int n_extra, double* rec,
                                 void* stream);
MORL_API int morl_front_unpack_f64(const double* gathered, int world, int d, int cap, int n_extra, double* pts_out, double* meta_out, void* stream);

/* Exact hypervolume (maximisation) of the points with keep[i] != 0 (keep NULL = all) above the reference point `ref` [d], 1 <= d <= 3,
 * n <= 2048, float64, one launch, result in *out (device): replaces `hypervolume(ref_point, points)` of the reference
 * (common/performance_indicators.py:15-25; pymoo's exact HV) for fronts that already live on the device.  Points that do not exceed
 * `ref` in every objective contribute nothing; dominated points are harmless (the volume is that of the union of boxes). */
MORL_API int morl_hypervolume_f64(const double* pts, const uint8_t* keep, int n, int d, const double* ref, double* out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Multi-tensor target-network sync.  Replaces polyak_update (common/networks.py:121-139):
 *   tau == 1 : target <- param;  else target <- fma(tau, param, fl((1 - tau) * target))   (mul_ then ATen's fused add(alpha))
 *   params / targets : device arrays of n_tensors device pointers; sizes : device int64 [n_tensors]
 */
MORL_API int morl_polyak_f32(const float* const* params, float* const* targets, const int64_t* sizes, int n_tensors,
                    int64_t max_size, double tau, void* stream);


/* ------------------------------------------------------------------------------------------------
 * Device-resident prioritised-replay sum tree (SURVEY.md 8(f)1), bit-identical to the reference's numpy tree (common/prioritized_buffer.py:
 * 12-82): float64, level l (2^l nodes) at element 2^l - 1 of `tree`, root first -- the layout of morl_host_sumtree_*.
 *   morl_sumtree_walk_f64       : SumTree.sample without the RNG (:40-54): query_i = scale_by_root ? tree[0] * u[i] : u[i]  (the host draws
 *                                 u with np.random.random_sample, the same stream np.random.uniform(0, root) consumes), level walk with
 *                                 strict '>' going right; out_index int64 [n].
 *   morl_sumtree_batch_set_f64  : SumTree.batch_set (:66-82): np.unique first-occurrence semantics, diff = new - leaf, then the per-level
 *                                 additions of np.add.at in sorted-leaf order; n <= 2048 indices per call.  *err_flag (device int) is set
 *                                 to 1 if an index is out of range.
 *   morl_sumtree_set_f64        : SumTree.set (:56-64; replay_buffer.add): one leaf, scalar arguments; use_min_priority != 0 takes the new
 *                                 priority from the buffer's current min_priority (device float64: the reference's python float until the first ratchet) instead
 *                                 of `priority`.
 *   morl_per_priority_f32       : p = fl32(fl32(raw + fl32(min_p)) ** alpha) (envelope.py:333; gpi_pd.py:523-525 callers pass their own raw),
 *                                 prio64 = (double) p for the tree, optional float32 copy, then *min_priority = max(*min_priority, max p)
 *                                 (prioritized_buffer.py:194).
 * All of them are single stream-ordered launches without host synchronisation: sample -> gather -> update -> priorities -> tree is one CUDA graph. */
MORL_API int morl_sumtree_walk_f64(const double* tree, int n_levels, const double* u, int n, int scale_by_root, long long* out_index, void* stream);
MORL_API int morl_sumtree_batch_set_f64(double* tree, int n_levels, const long long* index, const double* priority, int n, int* err_flag,
                                        void* stream);
MORL_API int morl_sumtree_set_f64(double* tree, int n_levels, long long index, double priority, int use_min_priority, const double* min_priority,
                                  int* err_flag, void* stream);
MORL_API int morl_per_priority_f32(const float* raw, int n, float alpha, double* min_priority, double* prio64, float* prio32, void* stream);

/* ------------------------------------------------------------------------------------------------
 * FP32-accurate dense layers on the tcgen05 tensor cores.  Replace the fp32 GEMMs behind the reference's nn.Linear layers
 * (common/networks.py:10-48; called from envelope.py:59-77 / :300, :420, :429 on the 65,536-row effective batch).
 * Every fp32 operand is carried as P 16-bit planes [P][rows][ld] (`plane_stride` elements between planes) whose sum reproduces it;
 * a product is the sum of the significant plane-by-plane MMAs with fp32 accumulation in tensor memory (csrc/gemm_planes.cu):
 *   MORL_FMT_F16X2  : P = 2 fp16 planes of  scale * x  (scale: a power of two held in a DEVICE float, NULL = 1), 3 MMAs, exact to
 *                     2^-22; |scale * x| must stay below 65,504 -- beyond it the planes hold Inf/NaN (propagating to every output)
 *                     and morl_plane_overflow_count() becomes non-zero.  4 bytes / element.
 *   MORL_FMT_BF16X3 : P = 3 bf16 planes of x (fp32 exponent range, scale pointers normally NULL), 6 MMAs, exact to 2^-24.  6 bytes / element.
 * All scale arguments are device pointers so that a captured CUDA graph stays valid when the scales change.
 *
 * morl_amax_scale_f32 : *scale_out = 2^(target_exp - e) with max|src| < 2^e, i.e. scale * max|src| in [2^(target_exp-1), 2^target_exp)
 *                     (1 if src is all zero).  workspace: 8 bytes, ZERO before the first call (left zero again).
 * morl_split_planes : fp32 [rows, cols] (row stride ld_src; transposed read if `transpose`) -> planes [P][rows_pad][ldp] of scale * x,
 *                     zero padded.
 * morl_split_planes_multi : up to MORL_SPLIT_MAX_JOBS independent splits (all weight matrices of a network, plain and transposed) in
 *                     one launch; a job with auto_scale != 0 derives its scale from the largest magnitude of its own matrix
 *                     (scale * amax in [2^(target_exp-1), 2^target_exp)) and stores it in *scale.
 * morl_gemm_planes_f32 : C = act(A . B^T + bias),  A planes [P][M][K] (K-major), B planes [P][N_pad][K] (K-major weights);
 *                     K % 64 == 0 (f16x2) / K % 32 == 0 (bf16x3), N_pad % 32 == 0, N_pad <= 256.  The accumulator is multiplied by
 *                     1 / (a_scale * b_scale) before the bias.  Outputs: c_f32 [M, ldc] and/or c_planes [P][M][ldp] holding
 *                     c_scale * C (the operand format of the next layer).  relu != 0 applies max(x, 0); relu_mask_plane0 (plane 0 of
 *                     a forward activation, [M][ld_mask] 16-bit) zeroes the outputs where that activation was <= 0 (ReLU backward).
 *                     ReLU bit masks (the form the update uses; relu_mask_plane0 stays for callers that only hold planes):
 *                     relu_bits_out [M][8] uint32 receives bit j of word (c & 1) * 4 + (c >> 1) = (C[m, 32 c + j] > 0) -- 32 bytes per
 *                     row instead of the 512-byte activation row, words ordered so that the four chunks one epilogue thread owns
 *                     are one 16-byte load; relu_bits_in (same layout, written by the forward call of the layer or by
 *                     morl_pairs_relu_split_planes) zeroes the outputs whose bit is clear, i.e. relu'(x) = [x > 0] exactly as
 *                     torch's ReLU backward (reference networks.py:10-48 under autograd).  Both nullable, 16-byte aligned.
 *                     reverse_tiles != 0 walks the 128-row tiles from the last to the first: alternate it between the layers of
 *                     a chain so that a layer starts on the rows its producer wrote last (still in the 126 MB L2).
 *                     split_accumulators != 0: the leading products A0.B0 and the correction products accumulate in separate TMEM
 *                     buffers and are added once, correctly rounded, in the epilogue -- the tensor cores TRUNCATE their fp32
 *                     accumulation at every MMA, which costs ~2e-6 (f16x2) / ~4e-6 (bf16x3) of systematic relative shrinkage per
 *                     K = 256 layer in one accumulator and ~2.5x less in split mode (profiles/r02_gemm_error.txt); the price is that
 *                     the epilogue of a tile no longer overlaps the MMAs of the next one.
 */
#define MORL_FMT_BF16X3 0
#define MORL_FMT_F16X2 1
#define MORL_SPLIT_MAX_JOBS 16
typedef struct MorlSplitJob {
    const float* src;       /* fp32 [rows, cols], row stride ld_src */
    void* dst_planes;       /* 16-bit [P][rows_pad][ldp] */
    long long plane_stride; /* elements between planes */
    float* scale;           /* device float: read (auto_scale == 0; NULL = 1) or written first, then used (auto_scale != 0; must not be NULL) */
    int rows, cols, ld_src, transpose, rows_pad, ldp;
    int auto_scale, target_exp;
} MorlSplitJob;
MORL_API int morl_plane_overflow_count(int reset); /* >= 0: f16x2 range violations seen since the last reset (synchronises the device) */
MORL_API int morl_amax_scale_f32(const float* src, long long n, int target_exp, float* scale_out, void* workspace, void* stream);
MORL_API int morl_split_planes_multi(int fmt, const MorlSplitJob* jobs, int n_jobs, void* stream);
MORL_API int morl_split_planes(int fmt, const float* src, int rows, int cols, int ld_src, int transpose, void* dst_planes, int rows_pad,
                               int ldp, long long plane_stride, const float* scale, void* stream);
MORL_API int morl_gemm_planes_f32(int fmt, const void* a_planes, long long a_plane_stride, const float* a_scale, const void* b_planes,
                                  long long b_plane_stride, const float* b_scale, int M, int N, int N_pad, int K, const float* bias,
                                  int relu, const void* relu_mask_plane0, int ld_mask, float* c_f32, int ldc, void* c_planes, int ldp,
                                  long long c_plane_stride, const float* c_scale, int reverse_tiles, int split_accumulators,
                                  const void* relu_bits_in, void* relu_bits_out, void* stream);
/* Several 256-wide hidden layers (Linear + ReLU) of one or two networks in ONE persistent launch (csrc/gemm_planes.cu: gemm_chain_kernel):
 * job (c, l):  act[c][l+1] = f(act[c][l] . W[c][l]^T + bias[c][l]),  planes in / planes out at the scale `act_scale`; f = ReLU (relu != 0:
 * forward chains, optionally recording the ReLU bit masks) or the ReLU-backward mask relu_bits_in[job] (dX chains of the backward pass:
 * G_{l-1} = (G_l . W_l) * relu'(H_{l-1}), biases NULL) --
 * bit-identical to n_chains * n_layers calls of morl_gemm_planes_f32 (c_scale = a_scale) -- but a CTA pair takes each of its 256-row tiles
 * through all layers, so every intermediate activation is re-read from the L2 it was just written to instead of from HBM, and the launch
 * prologue / drain is paid once.  Replaces the per-layer launches behind the reference's hidden nn.Linear + ReLU stack (networks.py:10-48) in the
 * no-grad passes (both networks at once: n_chains = 2) and in the training pass (n_chains = 1, with ReLU bit masks).
 *   act_planes [n_chains * (n_layers + 1)] : plane tensors [P][M][256] (host array of device pointers; index c * (n_layers + 1) + l);
 *   w_planes / w_scales / biases / relu_bits_in / relu_bits_out [n_chains * n_layers] (index c * n_layers + l; all but w_planes nullable, also per entry).
 *   k_first (0 = K): reduction length of layer 0 -- its input act[c][0] may be a NARROWER dense tensor [P][M][k_first] with weights [P][256][k_first]
 *   (plane strides M * k_first and 256 * k_first): the dX product of the 24-wide output layer as the first job of the backward chain.
 * morl_gemm_chain_supported: K == 256 (square 256-wide layers), M >= 256. */
MORL_API int morl_gemm_chain_supported(int fmt, int M, int K);
MORL_API int morl_gemm_chain_f32(int fmt, int n_chains, int n_layers, const void* const* act_planes, long long act_plane_stride, const float* act_scale,
                                 const void* const* w_planes, long long w_plane_stride, const float* const* w_scales, const float* const* biases,
                                 int relu, const void* const* relu_bits_in, void* const* relu_bits_out, int M, int K, int k_first, void* stream);
/* Diagnostics (not part of the reference surface): per-role cycle counters of morl_gemm_planes_f32, summed over CTAs and launches
 * since the last reset; collected only when the environment variable MORL_GEMM_STATS=1 is set before the first GEMM call.
 * out8: [0] MMA thread waiting for TMA data, [1] waiting for the epilogue to free an accumulator, [2] MMA loop total,
 * [3] TMA thread waiting for a free stage, [4] epilogue waiting for an accumulator, [5] epilogue busy; [6], [7] reserved. */
MORL_API int morl_debug_gemm_stats(unsigned long long* out8, int reset);
/* GPI-PD Dyna planning (SURVEY 8(f)3): everything between the last layer of the probabilistic ensemble and the imagined transition in ONE
 * pass (reference common/model_based/probabilistic_ensemble.py:115-154, common/model_based/utils.py:162-170; csrc/dyna.cu).
 *   out [E, N, 2*O] : raw output of the last EnsembleLayer (mean | logvar);  max_logvar / min_logvar [O]: the soft clamps (:118-119);
 *   model_idx [N]   : the elite model drawn for every row (np.random.choice(self.elites, N), :143 -- drawn on the host: RNG parity);
 *   noise [E, N, O] : standard normal draws (th.randn(std.shape), :128) or NULL = deterministic;
 *   obs [N, O - rew_dim] or NULL: added to the state part of the sample (the model predicts deltas, utils.py:165);
 *   sample_out / var_out [N, O]: sample and variance of the drawn model;  uncertainty_out [N]: sum_o sqrt(var_ensemble + 1e-12) (:146-149). */
MORL_API int morl_ensemble_sample_f32(const float* out, const float* max_logvar, const float* min_logvar, const int32_t* model_idx, const float* noise,
                                      const float* obs, int rew_dim, int E, int N, int O, float* sample_out, float* var_out, float* uncertainty_out,
                                      void* stream);

/* Output layer of BOTH Q-networks + envelope operator + Bellman line as ONE kernel (csrc/qhead_envelope.cu): replaces, for the two no-grad
 * passes of Envelope.update (reference envelope.py:420, :429, :422-440, :298),
 *     morl_gemm_planes_f32 (online, N = A*D) + morl_gemm_planes_f32 (target) + morl_envelope_td_f32
 * -- the Q tensors live in tensor memory / shared memory only (SURVEY 8(f)2: "envelope operator folded into the last-layer epilogue").
 *   a_on_planes / a_tg_planes : last hidden activations of the online / target net on s', planes [2][B*W][K] (row b*W + j), f16x2;
 *   w_on_planes / w_tg_planes : output-layer weight planes [2][32][K] (rows >= A*D zero), scales as in morl_gemm_planes_f32;
 *   everything from `wset` on  : as morl_envelope_td_f32 (same arithmetic contract, row orders, first-occurrence ties, outputs);
 *   q_on_out / q_tg_out        : optional fp32 copies of the Q tiles [B*W, A*D] (validation; NULL in the update).
 * The accumulation order equals morl_gemm_planes_f32's, so targets / indices are bit-identical to the three-launch chain.
 * morl_qhead_envelope_supported: 1 if the configuration is inside the kernel (f16x2 planes, W <= 64 dividing 128, B*W % 128 == 0,
 * A*D <= 32, W*A % 16 == 0, W*A*D % 4 == 0, 2 <= D <= 4, K % 64 == 0, K <= 256), else 0 -- callers then use the three-launch chain. */
MORL_API int morl_qhead_envelope_supported(int fmt, int B, int W, int A, int D, int K);
/* The kernel above without its operator half: the output layer of ONE network, q_out [M, N] = A . W^T + bias as fp32 rows (N <= 32: a narrow
 * morl_gemm_planes_f32 with the weight planes resident in shared memory and a deep activation ring; same accumulation order, bit-identical).
 * Used for the training pass's output layer (reference envelope.py:300).  M % 128 == 0, f16x2 planes, K % 64 == 0, K <= 256. */
MORL_API int morl_qhead_gemm_supported(int fmt, int M, int N, int K);
MORL_API int morl_qhead_gemm_f32(int fmt, const void* a_planes, long long a_plane_stride, const float* a_scale, const void* w_planes,
                                 long long w_plane_stride, const float* w_scale, const float* bias, int M, int N, int K, int reverse_tiles,
                                 float* q_out, void* stream);
MORL_API int morl_qhead_envelope_td_f32(int fmt, const void* a_on_planes, const void* a_tg_planes, long long a_plane_stride,
                                        const float* a_scale_on, const float* a_scale_tg, const void* w_on_planes, const void* w_tg_planes,
                                        long long w_plane_stride, const float* w_scale_on, const float* w_scale_tg, const float* bias_on,
                                        const float* bias_tg, int K, const float* wset, const float* reward, const float* done, float gamma,
                                        int B, int W, int A, int D, int dot_mode, int row_order, int reverse_tiles, float* target_out,
                                        int32_t* pref_out, int32_t* act_out, float* q_on_out, float* q_tg_out, void* stream);
/* h[b*W + j, :] = relu(u[b, :] + v[j, :]) written directly as planes [P][B*W][H] of scale * h (separable first layer of the
 * weight-conditioned Q-network: W1 [s || w] + b1 = W1_s s + (W1_w w + b1); reference envelope.py:75 builds the concat). */
MORL_API int morl_pairs_relu_split_planes(int fmt, const float* u, const float* v, int B, int W, int H, void* dst_planes,
                                          long long plane_stride, const float* scale, void* relu_bits_out, void* stream);


/* Weight-gradient GEMM (reduction over the batch rows), split-K, deterministic:
 *   out[n, k] = sum_m G[m, n] * H[m, k]      G planes [P][M][ldg] (n < g_cols, scaled by *g_scale), H planes [P][M][ldh] (k < h_cols,
 *   scaled by *h_scale);  ldg, ldh multiples of 64, ldh <= 256;  transpose_out != 0 stores out[k, n] instead.  Replaces the
 *   dW = dY^T X products that torch autograd issues for the nn.Linear layers of the reference networks (loss.backward(), envelope.py:316).
 *   colsum_out (nullable, [g_cols]): out_b[n] = sum_m G[m, n], the bias gradient db = colsum(dY), evaluated in the same pass as
 *   G^T . ones on the tensor cores (replaces a separate sweep of the G planes).  Runs as a one-job launch of
 *   morl_gemm_planes_mn_multi_f32's kernel, then one reduction launch.
 *   workspace: morl_gemm_mn_workspace_bytes(M, g_cols, h_cols) bytes, 16-byte aligned (MORL_ERR_ALIGN otherwise). */
MORL_API size_t morl_gemm_mn_workspace_bytes(int M, int a_cols, int b_cols);
MORL_API int morl_gemm_planes_mn_f32(int fmt, const void* g_planes, long long g_plane_stride, int ldg, int g_cols, const float* g_scale,
                                     const void* h_planes, long long h_plane_stride, int ldh, int h_cols, const float* h_scale, int M,
                                     int transpose_out, float* out, int ld_out, float* colsum_out, void* workspace, void* stream);
/* Up to MORL_MN_MAX_JOBS weight-gradient products over the same M rows in ONE persistent launch plus ONE reduction launch: job j computes
 * out[n, k] (and colsum_out[n]) bit-identically to morl_gemm_planes_mn_f32 with transpose_out = 0 on that job alone (the same kernel; a job's
 * splits and summation order do not depend on the other jobs), but the operand stream does not stop between the products (the backward pass
 * of an update: the output layer and every hidden layer).  Per job: ldg, ldh multiples of
 * 64, ldh <= 256, h_cols % 4 == 0, ld_out % 4 == 0, out 16-byte aligned (others are refused with MORL_ERR_UNSUPPORTED); colsum_out nullable.
 *   workspace: morl_gemm_mn_multi_workspace_bytes(jobs, n_jobs, M) bytes, 16-byte aligned. */
#define MORL_MN_MAX_JOBS 4
typedef struct MorlMnJob {
    const void* g_planes;      /* [P][M][ldg], scaled by *g_scale (NULL = 1) */
    long long g_plane_stride;  /* elements between planes */
    const float* g_scale;
    const void* h_planes;      /* [P][M][ldh], scaled by *h_scale (NULL = 1) */
    long long h_plane_stride;
    const float* h_scale;
    float* out;                /* [g_cols][ld_out] */
    float* colsum_out;         /* [g_cols] or NULL */
    int ldg, g_cols, ldh, h_cols, ld_out;
} MorlMnJob;
MORL_API size_t morl_gemm_mn_multi_workspace_bytes(const MorlMnJob* jobs, int n_jobs, int M);
MORL_API int morl_gemm_planes_mn_multi_f32(int fmt, const MorlMnJob* jobs, int n_jobs, int M, void* workspace, void* stream);
/* out[n] = (1 / *scale) sum_m sum_p planes[p][m][n]  (bias gradients); workspace: 296 * N floats */
MORL_API int morl_colsum_planes(int fmt, const void* planes, long long plane_stride, const float* scale, int M, int ld, int N, float* out,
                                void* workspace, void* stream);
/* gradients of the separable first layer: dU[b,:] = sum_j G[b*W+j,:], dV[j,:] = sum_b G[b*W+j,:]  (G planes [P][B*W][H] scaled by
 * *scale, W <= 64 for the one-pass kernel); workspace: 296 * W * H floats */
MORL_API int morl_pairs_grad_reduce_planes(int fmt, const void* planes, long long plane_stride, const float* scale, int B, int W, int H,
                                           float* dU, float* dV, void* workspace, void* stream);

/* Separable first layer of the weight-conditioned Q-network on the pair batch (reference envelope.py:59-77 builds [s || w] rows for
 * nn.Linear; DESIGN.md section 2):  u[b, :] = W1[:, :F] feats[b],  v[j, :] = W1[:, F:] wset[j] + b1  in ONE launch (replaces two library
 * sgemms and their epilogue kernels).  W1 is the row-major nn.Linear weight [H, F + D]; u [B, H], v [W, H]. */
MORL_API int morl_pair_layer1_uv_f32(const float* feats, const float* wset, const float* W1, const float* b1, int B, int W, int F, int D, int H,
                                     float* u, float* v, void* stream);

/* Parameter gradients of the separable first layer (backward of morl_pair_layer1_uv_f32; autograd of nn.Linear at envelope.py:316 on the
 * effective batch, restricted to layer 1):  dW1 [H, F + D] = [dU^T feats | dV^T wset],  db1 [H] = colsum(dV), with dU [B, H] / dV [W, H]
 * from morl_pairs_grad_reduce_planes.  One launch, deterministic split reduction.  `workspace`: morl_pair_layer1_grad_workspace_bytes(F, D,
 * H) bytes that must be ZERO before the first call (the kernel leaves its arrival counters zeroed again). */
MORL_API size_t morl_pair_layer1_grad_workspace_bytes(int F, int D, int H);
MORL_API int morl_pair_layer1_grad_f32(const float* dU, const float* dV, const float* feats, const float* wset, int B, int W, int F,
                              int D, int H, float* dW1, float* db1, void* workspace, void* stream);


/* Fused gradient clipping + Adam step over a list of tensors (two launches).  Replaces th.nn.utils.clip_grad_norm_ +
 * optim.Adam.step (envelope.py:324-326; torch/optim/adam.py _single_tensor_adam arithmetic, amsgrad = False, weight_decay = 0).
 *   params/grads/exp_avg/exp_avg_sq/steps : device arrays of n_tensors device pointers (steps[t] -> float32 scalar, incremented here)
 *   max_grad_norm <= 0 disables clipping;  workspace: morl_adam_workspace_bytes(n_tensors, max_size) bytes */
MORL_API size_t morl_adam_workspace_bytes(int n_tensors, int64_t max_size);
MORL_API int morl_adam_clip_f32(float* const* params, const float* const* grads, float* const* exp_avg, float* const* exp_avg_sq,
                                float* const* steps, const int64_t* sizes, int n_tensors, int64_t max_size, float max_grad_norm,
                                float lr, float beta1, float beta2, float eps, void* workspace, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MORL_B200_H_ */
