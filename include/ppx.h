/* ppx.h -- C ABI of libppx.so: the B200 (sm_100a) learner hot path of BoogaQ/PPO-exploration.
 *
 * The reference is pure Python (no FFI of its own, SURVEY.md §8b); each entry point below names the
 * reference method (file:line under /root/reference) whose arithmetic it replaces.  The Python
 * package `ppo-exploration_b200` binds these with ctypes and mirrors the reference's class surface.
 *
 * Conventions
 *   - every function returns 0 (PPX_OK) or a negative PPX_ERR_*; ppx_last_error() gives the
 *     thread-local message.  Nothing is printed, no exception crosses the boundary.
 *   - all data pointers are DEVICE pointers borrowed for the duration of the call (never freed,
 *     never retained) unless the parameter name ends in `_host`.
 *   - `stream` is a cudaStream_t passed as void*; launches are asynchronous, the caller syncs.
 *   - rollout arrays are time-major [T,N,...] row-major exactly as buffer.py:153-161 allocates them;
 *     "flat index i" means the env-major flatten of buffer.py:49-52: (t, n) = (i % T, i / T).
 *   - weights of dense layers are stored IN-MAJOR: W[K_in][N_out] (transpose of torch's Linear.weight).
 */
#ifndef PPX_H_
#define PPX_H_
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PPX_OK 0
#define PPX_ERR_ARG (-1)
#define PPX_ERR_CUDA (-2)
#define PPX_ERR_CAPACITY (-3)
#define PPX_ERR_UNSUPPORTED (-4)

enum { PPX_ACT_NONE = 0, PPX_ACT_TANH = 1, PPX_ACT_LEAKY_RELU = 2, PPX_ACT_ELU = 3, PPX_ACT_RELU = 4 };

const char* ppx_last_error(void);
int ppx_version(void);
/* kernels launched by this library in this process (bench.py's gpu_launches) */
uint64_t ppx_launch_count(void);
int ppx_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ---------------------------------------------------------------- reverse scans ------------- */
/* RolloutStorage.compute_returns_and_advantages, buffer.py:203-230.
 * masks[t] is the `dones` stored by add() at step t (buffer.py:180); step t is cut by masks[t+1]
 * and the last step by last_done (buffer.py:221-226).  f64 carry, f32 store. */
int ppx_gae(const float* rewards, const float* values, const uint8_t* masks, const float* last_value,
            const uint8_t* last_done, double gamma, double lam, int T, int N, float* advantages,
            float* returns, void* stream);
/* IntrinsicStorage.compute_returns_and_advantages, buffer.py:321-362: the extrinsic head as above
 * plus the non-episodic intrinsic head (no terminal masking, its own gamma, same lambda). */
int ppx_gae_dual(const float* rewards, const float* values, const uint8_t* masks, const float* last_value,
                 const uint8_t* last_done, double gamma, double lam, const float* int_rewards,
                 const float* int_values, const float* last_int_value, double int_gamma, int T, int N,
                 float* advantages, float* returns, float* int_advantages, float* int_returns,
                 void* stream);
/* SilModule.discount_with_dones, sil_module.py:99-105: R_t = r_t + gamma*R_{t+1}*(1-done_t), per column. */
int ppx_discount(const double* rewards, const uint8_t* dones, double gamma, int T, int N, double* out,
                 void* stream);

/* ---------------------------------------------------------------- SimHash ------------------- */
/* bits of RolloutStorage.sim_hash, buffer.py:194: code bit b = (A[b,:] . obs[i,:] > 0), f64 dot.
 * A is [k,D] f64 row-major, k <= 64. */
int ppx_simhash_codes(const double* A, const float* obs, int k, int D, int64_t n, uint64_t* codes,
                      void* stream);

typedef struct ppx_count_table ppx_count_table;
/* the persistent count_table of buffer.py:136 as an open-addressing device table (linear probing,
 * 64-bit atomicCAS claim, 32-bit counts).  capacity is rounded up to a power of two. */
int ppx_count_table_create(uint64_t capacity, ppx_count_table** out);
int ppx_count_table_destroy(ppx_count_table* t);
int ppx_count_table_clear(ppx_count_table* t, void* stream);
/* buffer.py:197-198 on packed codes: counts_out[i] = count of codes[i] AFTER its own increment,
 * with the reference's sequential semantics (element i sees every j < i of this and earlier calls).
 * Returns PPX_ERR_CAPACITY (after syncing the stream) if the table filled up. */
int ppx_count_table_update(ppx_count_table* t, const uint64_t* codes, int64_t n, uint32_t* counts_out,
                           void* stream);
/* Sharded count table (SURVEY §8e row 2): W ranks each own the codes with hash(code) % W == rank.  Every rank passes the
 * SAME globally ordered code list (t-major, env-minor over all envs); it updates only the codes it owns and writes their
 * sequential-semantics counts, 0 for the others -- summing counts_out over the ranks (one all-reduce) gives every count
 * of the replicated update, at 1/W of the order-dependent work per rank.  The union of the ranks' tables is the
 * reference's dict. */
int ppx_count_table_update_owned(ppx_count_table* t, const uint64_t* codes, int64_t n, uint32_t* counts_out, int W, int rank,
                                 void* stream);
/* whole sim_hash(obs, rewards), buffer.py:188-200, fused: codes from obs, sequential count update,
 * rewards[i] += beta/sqrt(count_i) (bonus in f64, stored back in the dtype of `rewards`).
 * obs is [n,D]; pass n = T*N with a [T,N,D] rollout to apply the bonus post hoc in the reference's
 * t-major, env-minor order.  codes_out / counts_out may be NULL. */
int ppx_simhash_update(ppx_count_table* t, const double* A, const float* obs, int k, int D, int64_t n,
                       double beta, void* rewards_inout, int rewards_are_f64, uint64_t* codes_out,
                       uint32_t* counts_out, void* stream);
/* buffer.py:199 alone, from precomputed counts (multi-GPU path: counts come from gathered codes). */
int ppx_simhash_bonus(const uint32_t* counts, int64_t n, double beta, void* rewards_inout,
                      int rewards_are_f64, void* stream);
/* synchronous helpers (tests / checkpointing): number of distinct keys; dump of (key,count) pairs. */
int ppx_count_table_size(ppx_count_table* t, uint64_t* n_keys_host);
int ppx_count_table_dump(ppx_count_table* t, uint64_t* keys_dev, uint32_t* counts_dev, uint64_t max_out,
                         uint64_t* n_out_host);
/* checkpoint restore into an EMPTY table (PPX_ERR_ARG otherwise): grows it until n keys fit at <= 50 % load and inserts
 * the (key, count) pairs; afterwards updates, growth and ppx_count_table_size behave as on the table that was dumped.
 * Synchronous.  A duplicate key or a zero count returns PPX_ERR_ARG and leaves the table empty. */
int ppx_count_table_load(ppx_count_table* t, const uint64_t* keys_dev, const uint32_t* counts_dev, uint64_t n,
                         void* stream);
/* the table's current capacity (a power of two; the all-ones key lives in one extra slot) */
int ppx_count_table_capacity(ppx_count_table* t, uint64_t* capacity_host);

/* ---------------------------------------------------------------- shuffle-gather ------------ */
/* RolloutStorage._get_samples, buffer.py:256-267 / :384-394, without materialising the env-major
 * flatten: for each array a, dst_a[b,:] = src_a[(idx[b] % T) * N + idx[b] / T, :] (row_bytes[a] each).
 * Up to PPX_MAX_GATHER arrays per launch. */
#define PPX_MAX_GATHER 12
int ppx_gather_minibatch(const void* const* srcs_host, void* const* dsts_host, const int* row_bytes_host,
                         int n_arrays, const int64_t* idx, int64_t B, int T, int N, void* stream);
/* Same gather, and on the way {mean, unbiased std} (f64, device) of up to two gathered f32 [B] fields -- the
 * advantage normalisation statistics of algorithms.py:219 / :431-434 -- finished by the field's last CTA in a fixed
 * order: stat_outs_host[k] receives 2 doubles for array index stat_fields_host[k]. */
typedef struct {
  /* > 0: the arrays are all-gathered env shards [N / n_shard ranks][T][n_shard][...] and idx is a flat index over the
   * GLOBAL [T, N] rollout: row = ((n / n_shard) * T + t) * n_shard + n % n_shard with t = idx % T, n = idx / T */
  int n_shard;
  /* statistics range: the moments are taken over idx[stat_lo .. stat_lo + stat_n) (may start before this rank's slice:
   * a rank that holds the replicated rollout evaluates the moments of the WHOLE global minibatch itself, identically on
   * every rank); rows outside [0, B) are read, not stored.  stat_n == 0: the B rows of the call. */
  int64_t stat_lo, stat_n;
  /* optional device step cursor: idx += (row / n_mb) * epoch_stride + (row % n_mb) * mb_stride, row = *row_dev */
  const int64_t* row_dev;
  int64_t n_mb, epoch_stride, mb_stride;
  /* Sharded learner with per-rank shuffles (W >= 2; W <= 1: off): the statistics written to stat_outs are those of the
   * GLOBAL minibatch -- the block that finishes the local moments pushes its {n, mean, M2} record to every rank over
   * NVLink-mapped memory (value + sequence number per 8-byte store), polls the W records and merges them in rank order
   * (replaces ppx_moments_pack + an exchange + ppx_moments_merge).  peer_moments_host[p]: rank p's staging, 2 x 2 x W x 8
   * 8-byte words, zeroed once; seq_dev: TWO local device words (one per statistics slot), starting at 0. */
  int W, rank;
  void* const* peer_moments_host;
  unsigned int* seq_dev; unsigned int* status_dev;
} ppx_gather_opts;
int ppx_gather_minibatch_stats(const void* const* srcs_host, void* const* dsts_host, const int* row_bytes_host,
                               int n_arrays, const int64_t* idx, int64_t B, int T, int N, const int* stat_fields_host,
                               double* const* stat_outs_host, int n_stats, const ppx_gather_opts* opts_host /* optional */,
                               void* stream);
/* mean and unbiased std of a contiguous f32 vector, accumulated in f64 (advantages.mean()/.std(),
 * algorithms.py:219).  out[0]=mean, out[1]=std(ddof=1). */
int ppx_mean_std(const float* x, int64_t n, double* out2, void* stream);

/* Host-side (no GPU): bit-exact replay of numpy's legacy `np.random.permutation(n)` (the draw of
 * buffer.py:239) from numpy's own MT19937 state (np.random.get_state(): key[624], pos); the advanced
 * state is written back so the caller can np.random.set_state it. */
int ppx_np_permutation(uint32_t* key624_host, int* pos_host, int64_t n, int64_t* out_host);
/* Only the draws of the same stream, n <= 2^31 - 1, as an int32 Fisher-Yates partner list: _draws32 indexed by position
 * (j_out[i] = partner of position i, constant-mask scalar loop), _draws32_stream in acceptance order (acc[r] belongs to
 * position n-1-r; AVX-512 block rejection when available). */
int ppx_np_shuffle_draws32(uint32_t* key624_host, int* pos_host, int64_t n, int32_t* j_out_host);
int ppx_np_shuffle_draws32_stream(uint32_t* key624_host, int* pos_host, int64_t n, int32_t* acc_host);
/* The swaps applied ON THE DEVICE, in parallel and bit-exactly (shuffle_dev.cu): j_dev is the uploaded partner
 * list, either indexed by position (acceptance_order = 0: j_dev[i], i = 1 .. n-1, from ppx_np_shuffle_draws32) or in
 * acceptance order (1: entry r belongs to position n-1-r, from ppx_np_shuffle_draws32_stream);
 * out_dev [n] int64 is arange(n) after the swaps = np.random.permutation(n).  n < 2^31; workspace of
 * ppx_np_shuffle_apply_device_workspace(n) bytes (24 per index; -1 for an unsupported n); asynchronous on `stream`. */
int64_t ppx_np_shuffle_apply_device_workspace(int64_t n);
int ppx_np_shuffle_apply_device(const int32_t* j_dev, int64_t n, int acceptance_order, void* workspace, int64_t* out_dev,
                                void* stream);
/* One staging step of a permutation, callable from the host thread that drew it: H2D of the pinned partner list (acceptance
 * order) into j_dev, ppx_np_shuffle_apply_device into out_dev, and cudaEventRecord of `copied_event` (after the copy) and
 * `ready_event` (after the swaps) when given (cudaEvent_t; NULL = skip).  Makes the device owning j_dev current for the
 * calling thread.  1 <= n < 2^31. */
int ppx_np_shuffle_stage(const int32_t* j_host_pinned, int64_t n, int32_t* j_dev, void* workspace, int64_t* out_dev,
                         void* stream, void* copied_event, void* ready_event);


/* Sharded minibatches (SURVEY §8e): rec3 = {n, mean, M2} from the local {mean, std}; after an all-gather of the
 * W records, out2 = {mean, std(ddof 1)} of the global minibatch (merged in rank order). */
int ppx_moments_pack(const double* stats2, int64_t n, double* rec3, void* stream);
int ppx_moments_merge(const double* recs, int W, double* out2, void* stream);

/* ---------------------------------------------------------------- NVLink peer-memory exchanges ---- */
/* The three global points of the sharded PPO minibatch (SURVEY §8e) as ONE kernel each over symmetric peer memory
 * (p2p.cu): barrier (release store per peer + acquire polls) -> read the W peers' payloads in rank order -> consume.
 * peer_* are HOST arrays of W device pointers (rank r's payload / flag array of this channel, >= W uint32, zeroed
 * before first use); seq_dev / status_dev are local device words (sequence number; != 0 after a 4 s barrier timeout).
 * Slot-reuse rule: between two uses of the same payload slot every rank must pass two other barriers. */
int64_t ppx_p2p_max_params(void);
/* merged {mean, std(ddof 1)} per stream from the ranks' {n, mean, M2} records (ppx_moments_pack), nstreams in {1,2} */
int ppx_p2p_moments_merge(const void* const* peer_recs_host, void* const* peer_flags_host, int W, int rank, uint32_t* seq_dev,
                          uint32_t* status_dev, int nstreams, double* stats_out, void* stream);
/* sums_out[32] = sum over ranks of the loss partial sums written by ppx_ppo_loss_head; then ppx_ppo_loss_finalize */
int ppx_p2p_sums_allreduce(const void* const* peer_sums_host, void* const* peer_flags_host, int W, int rank, uint32_t* seq_dev,
                           uint32_t* status_dev, double* sums_out, void* stream);
/* gradient all-reduce + clip_grad_norm_ + Adam in one kernel (n <= ppx_p2p_max_params()): replaces the NCCL
 * all-reduce + ppx_clip_adam of algorithms.py:243-244 on replicated weights; every replica computes the identical sum. */
int ppx_p2p_clip_adam(float* params, const void* const* peer_grads_host, void* const* peer_flags_host, int W, int rank,
                      uint32_t* seq_dev, uint32_t* status_dev, float* exp_avg, float* exp_avg_sq, int64_t n, double max_norm,
                      int64_t n_clip, double lr, double beta1, double beta2, double eps, int64_t* step_dev, double* norm_out,
                      float* grad_sum_out, void* stream);

/* ---------------------------------------------------------------- dense layers (fp32) ------- */
/* Y[z] = act(X[z] @ W[z] + bias[z]) for z < batch.  X: [M,K] ld=ldx, W: [K,N] contiguous, Y ld=ldy.
 * Strides (in elements) step X/W/bias/Y per batch entry; batch=1 ignores them.
 * Replaces the nn.Linear+activation stacks of models.py:141-150, 220-234, 281-291. */
int ppx_linear_fwd(const float* X, int ldx, const float* W, const float* bias, int M, int K, int N, int act,
                   float* Y, int ldy, int batch, int64_t strideX, int64_t strideW, int64_t strideB,
                   int64_t strideY, void* stream);
/* dX[z] = (dY[z] @ W[z]^T) * act'(H[z]) where H is the post-activation output of the layer that
 * produced X (NULL / PPX_ACT_NONE: no derivative factor). */
int ppx_linear_bwd_data(const float* dY, int lddy, const float* W, int M, int K, int N, const float* H,
                        int ldh, int act, float* dX, int lddx, int batch, int64_t strideDY, int64_t strideW,
                        int64_t strideH, int64_t strideDX, void* stream);
/* dW[z] = X[z]^T @ dY[z] ([K,N]), dbias[z] = colsum(dY[z]).  Deterministic split-M reduction through
 * `workspace` (>= ppx_linear_bwd_weight_workspace(...) floats). */
int64_t ppx_linear_bwd_weight_workspace(int M, int K, int N, int batch);
int ppx_linear_bwd_weight(const float* X, int ldx, const float* dY, int lddy, int M, int K, int N, float* dW,
                          float* dbias, float* workspace, int batch, int64_t strideX, int64_t strideDY,
                          int64_t strideDW, int64_t strideDB, void* stream);

/* ---------------------------------------------------------------- fused policy MLPs ---------- */
/* G independent D -> H -> H -> o_g tanh MLPs over one minibatch (actor | critic | int_critic of
 * models.py:137-213), forward and backward each as ONE persistent kernel (mlp_fused.cu).
 * Parameter layout = the policy bank's: W1 [D, G*H], b1 [G*H], W2 [G,H,H] (in-major), b2 [G,H],
 * W3[g] [H,o_g], b3[g] [o_g].  H1/H2 [M, G*H] are the saved tanh activations.  `outs`, `W3`, `b3`,
 * `out`, `dOut`, `dW3`, `db3` are HOST arrays of G entries.  Supported: H in {64,128}, D <= 32,
 * o_g <= 32, G <= 4 (ppx_mlp3_supported); other shapes take the layer-by-layer ppx_linear_* path. */
int ppx_mlp3_supported(int D, int H, int G, const int* outs_host);
int ppx_mlp3_fwd(const float* X, int ldx, int M, int D, int H, int G, const int* outs_host, const float* W1,
                 const float* b1, const float* W2, const float* b2, const float* const* W3_host,
                 const float* const* b3_host, float* H1, float* H2, float* const* out_host, void* stream);
/* workspace size in floats (-1: unsupported shape) */
int64_t ppx_mlp3_bwd_workspace(int M, int D, int H, int G, const int* outs_host);
/* A value head (o_g = 1) may have its output gradient evaluated inside the backward kernel from the loss
 * inputs instead of being read from dOut[g]: d = scale * (w1*-2(R-v) + w2*-2(R-v_clip)*[|v-v_old|<=clip]) / B_total
 * with {w1,w2} = branch[0..1] written by ppx_ppo_loss_head_final (the max-of-means branch, algorithms.py:232). */
typedef struct {
  const float* values; const float* old_values; const float* returns;   /* [M]; values == NULL: read dOut[g] */
  const double* branch;                                                 /* device, 2 doubles */
  float scale;                                                          /* policy_weight*vf_coef or int_vf_coef */
} ppx_value_head;
/* Optional optimiser tail of the backward (algorithms.py:243-244 in the SAME launch sequence, no Adam kernel): the
 * blocks of the partial-sum reduce kernel (launched cooperatively) meet once, every block combines the per-block sums of
 * squares in the same fixed order (+ the gradients outside the MLP, `extra_grads`, e.g. action_log_std, which must live
 * inside `grads`) and applies clip_grad_norm_(max_norm) + Adam to the parameters whose gradients it has just reduced;
 * block 0 takes the extra parameters and bumps *step_dev.  params / grads / exp_avg / exp_avg_sq are the bank's flat
 * vectors (same offsets).  max_norm <= 0: no clipping.  `ticket` = two zeroed device words owned by the bank. */
typedef struct {
  float* params; const float* grads; float* exp_avg; float* exp_avg_sq; int64_t n;
  double max_norm, lr, beta1, beta2, eps;
  int64_t* step_dev; double* norm_out /* optional */;
  const float* extra_grads; int n_extra;
  unsigned int* ticket;
  /* Sharded learner (W >= 2; W <= 1: single GPU): the gradient all-reduce runs inside the same kernel over peer memory
   * (one process per GPU, NVLink-mapped symmetric buffers).  Each block pushes the 32 gradients it reduced into every
   * rank's staging area as {f32 value, u32 sequence} 8-byte words, polls its own W slots for this launch's sequence
   * number and sums them in rank order before the clip + Adam above -- replaces the NCCL all-reduce + optimiser launch
   * of a data-parallel step (algorithms.py:243-244 under DDP).
   * peer_xg_host[p]: rank p's staging area, 2 x W x n 8-byte words (sequence parity, source rank, parameter), zeroed once;
   * seq_dev: local device word (sequence number, starts at 0, same on all ranks); status_dev: local device word set to 1
   * when a peer did not arrive within 4 s. */
  int W, rank;
  void* const* peer_xg_host;
  unsigned int* seq_dev; unsigned int* status_dev;
} ppx_fused_adam;
/* number of blocks of the reduce kernel that carries the optimiser tail for this shape when they can all be resident at
 * once (the tail needs that); 0 = the tail is not available (the backward then falls back to a separate clip + Adam launch on
 * one GPU, and must not be given a sharded ppx_fused_adam). */
int ppx_mlp3_fused_adam_blocks(int D, int H, int G, const int* outs_host);
int ppx_mlp3_bwd(const float* X, int ldx, int M, int D, int H, int G, const int* outs_host, const float* W2,
                 const float* const* W3_host, const float* H1, const float* H2, const float* const* dOut_host,
                 const ppx_value_head* value_heads_host /* G entries or NULL */, float clip_range, int64_t B_total,
                 float* dW1, float* db1, float* dW2, float* db2, float* const* dW3_host, float* const* db3_host,
                 float* workspace, double* sumsq_partials /* optional, ppx_mlp3_sumsq_partials() doubles: per-block sums of
                 squares of the final MLP gradients for ppx_clip_adam_pre; step_dev is then bumped here */,
                 int64_t* step_dev, const ppx_fused_adam* adam_host /* optional; needs sumsq_partials; step_dev ignored */,
                 void* stream);
int ppx_mlp3_sumsq_partials(int D, int H, int G, const int* outs_host);

/* Tensor-core variant of the same pair for H = 64, D <= 32, o_g <= 4, G <= 4 (ppx_mlp3_tc_supported): the two
 * 64x64 GEMMs of each pass run as tcgen05.mma kind::tf32 in three hi/lo passes (fp32-equivalent), operands are
 * written by the elementwise threads straight into swizzled shared-memory images, accumulators live in TMEM.
 * Same arguments and results as ppx_mlp3_fwd / ppx_mlp3_bwd except that H1t / H2t are OPAQUE activation
 * workspaces of ppx_mlp3_tc_act_elems(M, H, G) floats each (tile-transposed layout private to this pair), and the
 * backward workspace size comes from ppx_mlp3_tc_bwd_workspace.  The gradient partial sums go through the same
 * fixed-order reduce as ppx_mlp3_bwd (deterministic; sumsq_partials has ppx_mlp3_sumsq_partials() entries). */
int ppx_mlp3_tc_supported(int D, int H, int G, const int* outs_host);
int64_t ppx_mlp3_tc_act_elems(int M, int H, int G);
int ppx_mlp3_tc_fwd(const float* X, int ldx, int M, int D, int H, int G, const int* outs_host, const float* W1,
                    const float* b1, const float* W2, const float* b2, const float* const* W3_host,
                    const float* const* b3_host, float* H1t, float* H2t, float* const* out_host, void* stream);
int64_t ppx_mlp3_tc_bwd_workspace(int M, int D, int H, int G, const int* outs_host);
int ppx_mlp3_tc_bwd(const float* X, int ldx, int M, int D, int H, int G, const int* outs_host, const float* W2,
                    const float* const* W3_host, const float* H1t, const float* H2t, const float* const* dOut_host,
                    const ppx_value_head* value_heads_host, float clip_range, int64_t B_total,
                    float* dW1, float* db1, float* dW2, float* db2, float* const* dW3_host, float* const* db3_host,
                    float* workspace, double* sumsq_partials, int64_t* step_dev, const ppx_fused_adam* adam_host, void* stream);
/* Measurement hook (bench.py's roofline): the NEXT ppx_mlp3_tc_bwd call records this cudaEvent_t on its stream between
 * the backward kernel and the partial-sum reduce kernel, so that the dominant kernel can be timed by itself with CUDA
 * events.  One-shot; NULL clears. */
int ppx_mlp3_tc_bwd_probe(void* cuda_event);

/* ---------------------------------------------------------------- dense layers (tcgen05) ---- */
/* Blackwell tensor-core path for the same layers: C[M,N] = epi(A[M,R] . B[N,R]^T) with tcgen05.mma
 * kind::tf32 and a 3-pass hi/lo split (fp32-equivalent, error ~2^-21), TMA-fed, TMEM accumulators.
 *   forward:  A = X [M,K],   B = W^T [N,K] (ppx_tc_split hiT/loT of the in-major W), epi = act(acc + bias)
 *   dgrad:    A = dY [M,N],  B = W   [K,N] (ppx_tc_split hi/lo),                     epi = acc * act'(H)
 * ppx_tc_supported says whether a shape/alignment can take this path (TMA needs 16-byte pitches). */
int ppx_tc_supported(int M, int R, int N, int lda, int ldb, const void* A, const void* B);
int ppx_tc_split(const float* src, int rows, int cols, float* hi, float* lo, float* hiT, float* loT, void* stream);
int ppx_tc_linear(const float* A, int lda, const float* Bhi, const float* Blo, int ldb, int M, int R, int N,
                  const float* bias, const float* H, int ldh, int act, int dgrad,
                  const double* a_mean, const double* a_istd, float a_clip /* optional (both or neither): A is replaced
                  by clip((A - a_mean[k]) * a_istd[k], +-a_clip) in f64 on the fly (normalize_obs fused into the
                  A-split stage;
 a_istd from ppx_obs_istd) */,
                  float* C, int ldc, void* stream);
/* Same with a split-K workspace: when the M x N tiles do not fill the SMs and the reduction is long (wide first layers at
 * minibatch size: 32 tiles, 882 k-blocks) the reduction is cut S ways across CTAs (S chosen inside: fewest waves per
 * split), raw partial sums go to `workspace` [S][M][round4(N)] and a finish pass adds them in split order and applies the
 * epilogue -- deterministic.  ppx_tc_linear_workspace() = floats needed (0: the shape is not split; workspace may be NULL). */
int64_t ppx_tc_linear_workspace(int M, int R, int N);
int ppx_tc_linear_ws(const float* A, int lda, const float* Bhi, const float* Blo, int ldb, int M, int R, int N,
                     const float* bias, const float* H, int ldh, int act, int dgrad, const double* a_mean,
                     const double* a_istd, float a_clip, float* C, int ldc, float* workspace, int64_t workspace_floats,
                     void* stream);
/* Weight gradient of a wide layer on the tensor cores: dW [K,N] = X^T . dY over M samples, dbias = colsum(dY)
 * (dbias may be NULL).  X is transposed and dY split/transposed into `workspace` (>= ppx_tc_wgrad_workspace floats),
 * then the 3xTF32 kernel runs with the samples as the reduction dimension.  M % 4 == 0, M >= 256, K >= 128, N >= 16. */
int64_t ppx_tc_wgrad_workspace(int M, int K, int N);
int ppx_tc_wgrad_supported(int M, int K, int N, const void* X, const void* dY);
int ppx_tc_wgrad(const float* X, int ldx, const float* dY, int lddy, int M, int K, int N, float* dW, float* dbias,
                 float* workspace, void* stream);
/* istd[d] = 1/sqrt(var[d] + 1e-10) in f64 (the scale of BaseAlgorithm.normalize_obs, algorithms.py:111-118) */
int ppx_obs_istd(const double* var, int dim, double* istd, void* stream);

/* ---------------------------------------------------------------- conv front-end ------------- */
/* Convolutional front-end of the Atari-shaped configs (SURVEY §8f.2; spec: the reference's dead draft
 * .ipynb_checkpoints/models-checkpoint.py:48-66, :93-121 -- no live reference arithmetic, parity is defined against
 * torch.nn.Conv2d in fp64).  A convolution (no padding, square stride) is lowered onto the dense layers above:
 *   cols [N*OH*OW, C*KH*KW] = im2col(x);  Y [N*OH*OW, Cout] = act(cols . Wm + b)  (ppx_tc_linear_ws / ppx_linear_fwd);
 *   dWm = cols^T dY (ppx_tc_wgrad / ppx_linear_bwd_weight);  dcols = dY Wm^T (ppx_linear_bwd_data);  dx = col2im(dcols).
 * nchw = 1: x is [N,C,H,W], patch entries ordered (c, kh, kw) = torch's weight.view(Cout, -1) column order (first layer);
 * nchw = 0: x is [N,H,W,C] (= the previous layer's output rows), patch entries ordered (kh, kw, c).
 * OH = (H - KH) / stride + 1, OW likewise.  col2im is a deterministic gather (no atomics); dx has x's layout. */
int ppx_im2col(const float* x, int nchw, int N, int C, int H, int W, int KH, int KW, int stride, float* cols, void* stream);
int ppx_col2im(const float* dcols, int nchw, int N, int C, int H, int W, int KH, int KW, int stride, float* dx, void* stream);
/* out[i] = d[i] * act'(h[i]) with the derivative expressed through the post-activation value h (out may alias d): the
 * step from a gradient w.r.t. a layer's activated output to the gradient w.r.t. its pre-activation. */
int ppx_act_bwd_mul(const float* d, const float* h, int64_t n, int act, float* out, void* stream);

/* ---------------------------------------------------------------- PPO loss ------------------ */
/* Fused clipped-surrogate / clipped-value / entropy loss, forward and backward, for one minibatch:
 * PPO.train algorithms.py:219-238, PPO_RND.train :431-460 (dual=1), PPO_ICM.train :670-692 (the
 * policy_weight factor).  Inputs are the network outputs for the minibatch and the gathered sample
 * fields; outputs are the gradients w.r.t. the network outputs and the loss scalars.
 *
 *   discrete = 0 (Box):  actor_out = pre-tanh means [B,A]; actions f64 [B,A]; old_log_probs [B,A];
 *                        log-prob / ratio / surrogate evaluated in f64 like the reference
 *                        (actions are f64, buffer.py:154).  d_log_std[A] is accumulated.
 *   discrete = 1:        actor_out = logits [B,A]; actions f64 [B] (class ids); old_log_probs [B].
 *   adv_stats / int_adv_stats: device {mean, std} from ppx_mean_std.
 *   value head(s): values/old_values/returns [B]; the max-of-means branch (algorithms.py:232) is
 *                  resolved on device; d_values is the gradient of the SELECTED branch * vf_coef.
 *   losses_out[8] (device, f64): total, policy, value, entropy, int_value, 0, 0, 0.
 * `workspace` needs ppx_ppo_loss_workspace(B, A) bytes. */
typedef struct {
  int64_t B;        /* minibatch rows held by this rank */
  int64_t B_total;  /* rows of the global minibatch (0 = B); means and gradient scales use this */
  int A;
  int discrete;
  int dual;
  float clip_range, ent_coef, vf_coef, int_vf_coef, policy_weight;
  /* optional device step cursor (one CUDA graph serves every minibatch of a train() call): the loss row written is
   * losses_out + 8 * (*row_dev); the finalising thread then increments *row_dev unless row_hold (a later
   * ppx_loss_row_commit does it).  ppx_gather_minibatch_stats reads the same counter to find its index slice. */
  int64_t* row_dev;
  int row_hold;
  /* Sharded learner, ppx_ppo_loss_head_final only (W >= 2; W <= 1: single GPU): before the finalising block evaluates the
   * losses and the max-of-means branch, it all-reduces the 32 partial sums with its peers over NVLink-mapped memory
   * (value + sequence number in one 8-byte store; no exchange kernel) -- B_total must then be the global row count.
   * peer_sums_host[p]: rank p's staging, 2 x W x 64 8-byte words, zeroed once; seq_dev / status_dev as in ppx_fused_adam. */
  int W, rank;
  void* const* peer_sums_host;
  unsigned int* seq_dev; unsigned int* status_dev;
} ppx_ppo_cfg;
/* losses[8 * row + col] = *value; losses[8 * row] += *value if add_to_total; then ++*row_dev (row = *row_dev before).
 * The ICM learner's second loss (algorithms.py:688-692) lands in the row its policy step left open (row_hold). */
int ppx_loss_row_commit(double* losses, int64_t* row_dev, const double* value, int col, int add_to_total, void* stream);
int64_t ppx_ppo_loss_workspace(int64_t B, int A);
int ppx_ppo_loss_fwd_bwd(const ppx_ppo_cfg* cfg_host, const float* actor_out, const float* log_std,
                         const double* actions, const float* old_log_probs, const float* advantages,
                         const double* adv_stats, const float* values, const float* old_values,
                         const float* returns, const float* int_advantages, const double* int_adv_stats,
                         const float* int_values, const float* old_int_values, const float* int_returns,
                         float* d_actor_out, float* d_log_std, float* d_values, float* d_int_values,
                         double* losses_out, void* workspace, void* stream);
/* Single-GPU fast path: head + fixed-order sum of the CTA partials + loss scalars / branch / d_log_std in ONE
 * launch (the last CTA to finish does the tail).  branch_out[4] = {w1, w2, int_w1, int_w2}; the value-head
 * gradients are then evaluated inside ppx_mlp3_bwd (ppx_value_head) or by ppx_ppo_loss_finish. */
int ppx_ppo_loss_head_final(const ppx_ppo_cfg* cfg_host, const float* actor_out, const float* log_std,
                            const double* actions, const float* old_log_probs, const float* advantages,
                            const double* adv_stats, const float* values, const float* old_values,
                            const float* returns, const float* int_advantages, const double* int_adv_stats,
                            const float* int_values, const float* old_int_values, const float* int_returns,
                            float* d_actor_out, float* d_log_std, double* losses_out, double* branch_out,
                            void* workspace, void* stream);
/* finalize only (no value-head gradients): loss scalars, branch weights and d_log_std from GLOBAL sums[32]. */
int ppx_ppo_loss_finalize(const ppx_ppo_cfg* cfg_host, const double* sums, const float* log_std, float* d_log_std,
                          double* losses_out, double* branch_out, void* stream);
/* The same computation split at its only global dependency, for sharded minibatches (SURVEY §8e):
 * head   -> per-sample work + sums_out[32] (f64 partial sums of this rank);
 *           all-reduce sums_out across ranks (one 256-byte message), then
 * finish -> loss scalars, max-of-means branch, d_log_std, d_values from the GLOBAL sums. */
int ppx_ppo_loss_head(const ppx_ppo_cfg* cfg_host, const float* actor_out, const float* log_std,
                      const double* actions, const float* old_log_probs, const float* advantages,
                      const double* adv_stats, const float* values, const float* old_values, const float* returns,
                      const float* int_advantages, const double* int_adv_stats, const float* int_values,
                      const float* old_int_values, const float* int_returns, float* d_actor_out, double* sums_out,
                      void* workspace, void* stream);
int ppx_ppo_loss_finish(const ppx_ppo_cfg* cfg_host, const double* sums, const float* log_std, const float* values,
                        const float* old_values, const float* returns, const float* int_values,
                        const float* old_int_values, const float* int_returns, float* d_log_std, float* d_values,
                        float* d_int_values, double* losses_out, void* workspace, void* stream);

/* MSE / cross-entropy pieces of the ICM and RND-predictor losses (algorithms.py:497, :686-688):
 * loss = scale * mean((a-b)^2) over n elements; d_a = +g, d_b = -g (either may be NULL);
 * the scalar is ADDED to *loss_accum (device f64). */
int ppx_mse_fwd_bwd(const float* a, const float* b, int64_t n, double scale, float* d_a, float* d_b,
                    double* loss_accum, void* stream);
/* loss = scale * mean_b( -log softmax(logits[b])[target[b]] ), d_logits out; targets f64 class ids with
 * element stride `target_stride` (util.py:61-78: nn.CrossEntropyLoss on the inverse model). */
int ppx_xent_fwd_bwd(const float* logits, const double* targets, int target_stride, int64_t B, int C,
                     double scale, float* d_logits, double* loss_accum, void* stream);

/* ---------------------------------------------------------------- optimiser ----------------- */
/* clip_grad_norm_(max_norm) + Adam step on a flat parameter vector (algorithms.py:243-244):
 * coef = min(1, max_norm/(||g||+1e-6)) (skipped when max_norm <= 0), torch.optim.Adam update
 * (no weight decay / amsgrad) with bias correction for `step` (1-based). */
int ppx_clip_adam(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n,
                  double max_norm, int64_t n_clip /* grads [0,n_clip) enter the norm and are clipped */,
                  double lr, double beta1, double beta2, double eps, int64_t step,
                  int64_t* step_dev /* NULL, or device counter of steps done: incremented, then used (graph replay) */,
                  double* norm_out, void* workspace /* >= 4096 doubles */, void* stream);
/* Same update when the sum of squares of (most of) the gradient was already produced by the kernel that wrote it
 * (ppx_mlp3_bwd): the clip norm is sqrt(sum(sumsq_partials) + sum(extra_grads^2)); the whole vector is clipped;
 * *step_dev must already hold the NEW step number. */
int ppx_clip_adam_pre(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n, double max_norm,
                      double lr, double beta1, double beta2, double eps, const int64_t* step_dev, double* norm_out,
                      const double* sumsq_partials, int n_partials, const float* extra_grads, int n_extra, void* stream);

/* ---------------------------------------------------------------- bonus-net epilogues ------- */
/* RunningMeanStd.update (util.py:20-44), f64 moments on device: state = {mean[dim], var[dim], count}.
 * x is [n, dim] with element type f32 (x_is_f64=0) or f64. */
int ppx_rms_update(const void* x, int x_is_f64, int64_t n, int dim, double* mean, double* var, double* count,
                   void* workspace, void* stream);
/* BaseAlgorithm.normalize_obs (algorithms.py:111-118): out = f32(clip((obs-mean)/sqrt(var+1e-10),-5,5)), f64 math */
int ppx_normalize_obs(const float* obs, int64_t n, int dim, const double* mean, const double* var, float* out,
                      void* stream);
/* RndNetwork.int_reward tail (models.py:265): r = (pred-target)^2 */
int ppx_rnd_sqerr(const float* pred, const float* target, int64_t n, float* r, void* stream);
/* algorithms.py:396-398 for a whole rollout: for t in 0..T-1: rms.update(r[t,:]); r[t,:] /= sqrt(var)+1e-8 */
int ppx_rnd_normalize_rollout(float* r, int T, int N, double* mean, double* var, double* count, void* stream);
/* ICM int_reward tail (models.py:319-320) + blend (algorithms.py:630):
 * ri = clamp(mean_f((pred-feat)^2), -5, 5); rewards = (1-eta)*rewards + eta*ri; ri_out optional */
int ppx_icm_bonus_tail(const float* pred_feat, const float* next_feat, int64_t n, int F, double eta,
                       float* rewards_inout, float* ri_out, void* stream);
/* rows of an embedding table (ICM action_encoder for Discrete, models.py:294): out[b,:] = table[id[b],:]
 * ids are f64 (stored actions) or i64; out has leading dimension ldo. */
int ppx_embedding_fwd(const float* table, int C, const void* ids, int ids_are_f64, int id_stride, int64_t B,
                      float* out, int ldo, void* stream);
int ppx_embedding_bwd(const float* d_out, int ldo, const void* ids, int ids_are_f64, int id_stride, int64_t B,
                      int C, float* d_table, void* stream);

/* VecNormalize on the device (SURVEY §8f.3; the reference wraps its envs in stable_baselines3's VecNormalize with
 * norm_reward=True, env.py:11).  obs: out = clip((obs - mean) / sqrt(var + eps), +-clip) from RunningMeanStd state
 * (ppx_rms_update).  reward: returns = returns * gamma + r; the return statistics {mean, var, count} absorb the batch of
 * returns (update_stats); out = clip(r / sqrt(ret_var + eps), +-clip); returns[done] = 0.  n <= any (one CTA). */
int ppx_vecnorm_obs(const float* obs, int64_t n, int dim, const double* mean, const double* var, double eps, double clip,
                    float* out, void* stream);
int ppx_vecnorm_reward(const float* rewards, const uint8_t* dones, double* returns_inout, int n, double gamma,
                       double* ret_mean, double* ret_var, double* ret_count, double eps, double clip, int update_stats,
                       float* rewards_out, void* stream);
/* Policy.act tail (models.py:30-50, 75-99; SURVEY §8f.1): sample one action per env from Normal(tanh(actor_out),
 * exp(log_std)) (Box: actions f64 [N,A], log-probs f32 [N,A]) or Categorical(softmax(actor_out)) (Discrete: action ids as
 * f64 [N], log-probs f32 [N]) and evaluate its log-probability as torch.distributions would.  Philox4x32-10 keyed by
 * `seed`, counter (env, draw): pass a new `draw` number per call. */
int ppx_policy_sample(const float* actor_out, const float* log_std, int64_t N, int A, int discrete, uint64_t seed,
                      uint64_t draw, double* actions_out, float* logp_out, void* stream);
/* Device-env rollout step, first half (replaces Policy.act's sampling and value clones, models.py:30-50 / 75-99, and the
 * obs / action / value / log-prob copies of RolloutStorage.add, buffer.py:165-186, IntrinsicStorage.add, :305-318): from the
 * policy forward's outputs (actor_out [N,A], value [N], int_value [N] or NULL, log_std [A]; Box only) and the observation the
 * policy acted on (obs f32 [N,D], contiguous), draw the actions exactly as ppx_policy_sample does for (seed, draw) and write
 * rollout step `pos`'s rows: obs_row [N,D], actions_row f64 [N,A], logp_row f32 [N,A], value_row [N], int_value_row [N]
 * (NULL: none).  env_actions receives a separate copy for the env (Box: f64 [N,A]; Discrete: int64 [N]).  One launch. */
int ppx_policy_act_record(const float* actor_out, const float* value, const float* int_value, const float* log_std,
                          const float* obs, int64_t N, int A, int D, int discrete, uint64_t seed, uint64_t draw,
                          float* obs_row, double* actions_row, float* logp_row, float* value_row, float* int_value_row,
                          void* env_actions, void* stream);
/* Device-env rollout step, second half (the reward / mask / int-reward copies of buffer.py:165-186, :305-318): rewards
 * (f32, or f64 if rewards_f64) [N] cast round-to-nearest into rewards_row; with rewards_f64 and rewards_f64_row non-NULL
 * they go to that f64 row instead (a SimHash bonus is added to them in f64 later).  dones (bool / uint8 [N]) copied byte for
 * byte into masks_row; their nonzero count added to *episodes.  int_rewards_row (NULL: none) receives int_rewards, or zeros
 * if int_rewards is NULL.  One launch. */
int ppx_rollout_record_step(const void* rewards, int rewards_f64, const uint8_t* dones, const float* int_rewards, int64_t N,
                            float* rewards_row, double* rewards_f64_row, uint8_t* masks_row, float* int_rewards_row,
                            int64_t* episodes, void* stream);

/* ---------------------------------------------------------------- policy evaluation --------- */
/* Env-facing actions of an evaluation step (evaluate.cu; DESIGN.md §3.17) from the policy forward's actor_out [N,A] (log_std
 * [A]: Box only): Box f64 [N,A], Discrete int64 [N] into env_actions.  deterministic: Box (double)tanhf(actor_out), the
 * sampled action of ppx_policy_sample at z = 0; Discrete the index of the largest logit, lowest on ties.  Otherwise one
 * draw with ppx_policy_sample's arithmetic, Philox counter (row_offset + n, draw): rows of a sharded call equal the same rows
 * of one call over all envs.  `draw` must have bit 63 set (the training stream counts up from 1).  One launch. */
int ppx_policy_act_eval(const float* actor_out, const float* log_std, int64_t N, int A, int discrete, int deterministic,
                        uint64_t seed, uint64_t draw, int64_t row_offset, void* env_actions, void* stream);
/* After env.step of evaluation step `step`: env n (global env g = env_offset + n of total_envs) records its first
 * (n_eval_episodes + g) / total_envs finished episodes (dones[n] != 0): ep_returns[n] (f64), ep_lengths[n] (int64) and
 * `step` go to row n, column counts[n] of the [N, kmax] tables (kmax >= ceil(n_eval_episodes / total_envs)), then
 * counts[n] += 1.  Later episodes are ignored.  state: int64 [3], zero before the first step; state[2] receives the number
 * of episodes this rank still misses (the other two words are re-armed scratch).  One launch. */
int ppx_eval_episode_step(const uint8_t* dones, const double* ep_returns, const int64_t* ep_lengths, int64_t N,
                          int64_t n_eval_episodes, int64_t env_offset, int64_t total_envs, int64_t step, int64_t* counts,
                          double* out_ret, int64_t* out_len, int64_t* out_end, int64_t kmax, int64_t* state, void* stream);

/* ---------------------------------------------------------------- classic control ----------- */
/* Gym 0.17 classic-control envs with TimeLimit, on the device (classic_control.cu; DESIGN.md §3.13).  env: 0 CartPole-v1,
 * 1 MountainCar-v0, 2 MountainCarContinuous-v0, 3 Pendulum-v0.  State f64 [S, N] (S = 4, 2, 2, 2), observations f32 [N, D]
 * (D = 4, 2, 2, 3).  Per env: elapsed steps, episode number, monitor accumulators (f64 return, length) and the return / length
 * of the last finished episode.  Reset draws: Philox4x32-10 under `seed`, counter (global env env_offset + n, episode number).
 * step: actions int64 [N] (Discrete) or f64 [N, 1] (Box); reward f32 (rounded once from f64) or f64 [N] (reward_f64); done
 * uint8 [N]; behavior (NULL: none) f64 [N, S] receives the pre-reset state; finished envs are reset in place.  reset: every
 * env starts its next episode.  One launch each. */
int ppx_classic_step(int env, int64_t N, int64_t env_offset, uint64_t seed, const void* actions, double* state, int64_t* elapsed,
                     int64_t* episode, double* mon_ret, int64_t* mon_len, double* ep_ret, int64_t* ep_len, float* obs, void* reward,
                     int reward_f64, uint8_t* done, double* behavior, void* stream);
int ppx_classic_reset(int env, int64_t N, int64_t env_offset, uint64_t seed, double* state, int64_t* elapsed, int64_t* episode,
                      double* mon_ret, int64_t* mon_len, float* obs, void* stream);
/* Episode monitor of any env on the device: acc_ret += reward (f32 or f64 [N], f64 sum), acc_len += 1; where dones[n] != 0
 * the sums go to ep_ret[n] / ep_len[n] and restart from 0.  One launch. */
int ppx_episode_monitor_step(const void* rewards, int rewards_f64, const uint8_t* dones, int64_t N, double* acc_ret, int64_t* acc_len,
                             double* ep_ret, int64_t* ep_len, void* stream);
/* Learner episode log.  record: where dones[n] != 0, ep_ret[n] / ep_len[n] -> log rows (one step, [N]).  tail: over the flat
 * t-major done flags [total] and the log, the newest min(K, #dones) finished episodes go to out_ret / out_len [K], newest
 * first, and their number to *out_count.  One launch each (tail: one block). */
int ppx_episode_log_record(const uint8_t* dones, const double* ep_ret, const int64_t* ep_len, int64_t N, double* log_ret_row,
                           int64_t* log_len_row, void* stream);
int ppx_episode_log_tail(const uint8_t* dones, const double* log_ret, const int64_t* log_len, int64_t total, int64_t K,
                         double* out_ret, int64_t* out_len, int64_t* out_count, void* stream);

/* ---------------------------------------------------------------- ES-NSRA ------------------- */
/* fill a shared noise table with N(0,1) f32 (Philox4x32-10 + Box-Muller); build-side design, the
 * reference draws fresh randn per member (evolution_strategies.py:172-182). */
int ppx_noise_fill(float* table, int64_t n, uint64_t seed, void* stream);
/* _get_weights_try for the whole population (evolution_strategies.py:137-145):
 * out[p,j] = theta[j] + sigma * eps[p,j], eps[p,:] = noise[offsets[p] : offsets[p]+D] (offsets NULL:
 * noise is dense [P,D]).  out is f64 (out_is_f64=1, reference dtype) or f32.
 * CONTRACT: when offsets != NULL and D % 4 == 0, every offset must be a multiple of 4 (16-byte aligned noise
 * rows; ppx_es_perturb and ppx_es_update read them as 16-byte vectors). */
int ppx_es_perturb(const double* theta, const float* noise, const int64_t* offsets, double sigma, int P, int D,
                   void* out, int out_is_f64, void* stream);
/* FeedForwardNetwork.predict (evolution_strategies.py:48-61) for the whole population at once (SURVEY §8f.4): member p
 * acts on obs[p, :] with weights theta + sigma*eps_p formed on the fly from the noise table (offsets) or the dense eps
 * rows (offsets == NULL) -- never materialised.  Bias-free MLP layer_sizes_host[0..n_layers] (D0, h1, ..., A), hidden
 * activation arctan; fp32 arithmetic on f64 inputs / outputs (1e-5 relative against the f64 reference; the FP64 pipe
 * made an f64 version 6x slower); squash_tanh = 1 applies continuous_action's tanh (:84-89), 0 leaves the logits
 * (Discrete: the categorical draw stays with the host RNG).  out is [P, A] f64. */
int ppx_es_forward(const double* theta, const float* noise, const int64_t* offsets, double sigma, int P,
                   const int* layer_sizes_host, int n_layers, const double* obs, int squash_tanh, double* out, void* stream);
/* Episode evaluation on an env that lives on the GPU (evaluate / get_action, evolution_strategies.py:75-95, 153-170), env m
 * running member m.  ppx_es_act: the population forward of ppx_es_forward (same per-member code, bit-identical logits) on
 * f32 observations obs [N, D0], for the members with alive[m] != 0 (alive NULL: all); a finished member reads no noise and
 * gets action 0.  actions: Box (discrete = 0) f64 [N, A] = tanh(logits); Discrete int64 [N] = numpy's RandomState.choice
 * over softmax(logits) -- p = exp(l) / sum(exp(l)) in f64, cdf = cumsum(p) / its last entry, the number of cdf entries
 * <= u -- with u = uniforms[m] (f64 [N], e.g. numpy's own draws) or, uniforms NULL, the 53-bit uniform of
 * Philox4x32-10 keyed by `seed` at counter (member_lo + m, step, *draw_dev) (draw_dev NULL: 0).  One launch. */
int ppx_es_act(const double* theta, const float* noise, const int64_t* offsets, double sigma, int N, const int* layer_sizes_host,
               int n_layers, const float* obs, const uint8_t* alive, int discrete, uint64_t seed, const int64_t* draw_dev,
               int64_t step, int64_t member_lo, const double* uniforms, void* actions, void* stream);
/* ppx_es_act_rows: the brains of EvolutionStrategy.run, env row m acting with its own parameter vector thetas[m] (f64 [M, D],
 * row-major) at sigma = 0 -- for every row the logits and action of ppx_es_act(theta = thetas[m], sigma = 0, table offset 0)
 * bit for bit, Discrete u from Philox4x32-10 keyed by `seed` at counter (m, step, *draw_dev).  noise: the table (row m reads
 * its first D floats, multiplied by 0); obs f32 [M, D0]; alive and actions as in ppx_es_act.  One launch, one CTA per row. */
int ppx_es_act_rows(const double* thetas, const float* noise, int M, const int* layer_sizes_host, int n_layers, const float* obs,
                    const uint8_t* alive, int discrete, uint64_t seed, const int64_t* draw_dev, int64_t step, void* actions,
                    void* stream);
/* ppx_es_episode_step, after env.step, for every member with alive[n] != 0: fitness[n] += reward (f32 or f64 rewards [N],
 * f64 sum), lengths[n] += 1; when dones[n] != 0 or last_step != 0 the behaviour row behavior[n, 0..k) (NULL: none) is copied
 * to behavior_out[n] and alive[n] = 0.  state: int64 [3], zero before the first step; state[2] receives the number of
 * members still running (the other two words are re-armed scratch).  One launch. */
int ppx_es_episode_step(const void* rewards, int rewards_f64, const uint8_t* dones, const double* behavior, int k, int64_t N,
                        int last_step, uint8_t* alive, double* fitness, int64_t* lengths, double* behavior_out, int64_t* state,
                        void* stream);
/* _update_weights (evolution_strategies.py:217-239): z-score rewards (ddof 0); skip entirely if std==0;
 * theta += lr/(P*sigma) * sum_p w_p eps_p with w_p = ((1-nw)*z_p + nw*novelty)/2 (use_novelty=1) or z_p;
 * then *lr_inout *= decay.  rank_mode=1 replaces the z-score by centred ranks (BASELINE north_star;
 * not in the reference).  All scalars state lives on device: lr_inout[1]; status_out[0]=1 if skipped. */
int64_t ppx_es_update_workspace(int P, int D);
int ppx_es_update(double* theta, const float* noise, const int64_t* offsets, const double* rewards, int P, int D,
                  double sigma, double novelty_param, double novelty, const double* novelty_dev /* overrides `novelty` when
                  non-NULL: the k-NN result stays on the device, no host round trip */, int use_novelty, int rank_mode,
                  double decay, double* lr_inout, int* status_out, void* workspace, void* stream);
/* The population of one ES iteration as noise-table offsets drawn ON THE DEVICE (build-side design: the reference draws
 * fresh randn per member, :172-182): Philox4x32-10 keyed by `seed`, counter = (member, draw_dev[0]); draw_dev[0] is bumped
 * (draw_dev[1] is a zeroed ticket word),
 * so the launch replays from a CUDA graph and ranks sharing (seed, draw number) draw the identical population.
 * offsets_out[p] is a multiple of 4 in [0, table_size - D]. */
int ppx_es_offsets(uint64_t seed, int64_t* draw_dev, int P, int64_t table_size, int D, int64_t* offsets_out, void* stream);
/* _update_weights with the population sharded over W ranks (SURVEY §8e row 6): every rank holds all P rewards (after the
 * fitness all-gather) and computes the identical z-scores, runs the GEMV over ITS members [p_lo, p_lo + p_n) only,
 * leaves the partial update in `dtheta_local` (its slot of a symmetric, peer-mapped allocation) and one kernel per rank
 * meets the others at a flag barrier, sums the W partial updates in rank order over NVLink and applies them -- theta and
 * lr stay bit-identical replicas; the noise is streamed once over all ranks together (strong scaling). */
int ppx_es_update_sharded(double* theta, const float* noise, const int64_t* offsets, const double* rewards, int P, int p_lo,
                          int p_n, int D, double sigma, double novelty_param, double novelty, const double* novelty_dev,
                          int use_novelty, double decay, double* lr_inout, int* status_out, void* workspace,
                          double* dtheta_local, const void* const* peer_dtheta_host, void* const* peer_flags_host, int W,
                          int rank, uint32_t* seq_dev, uint32_t* status_dev, void* stream);
/* centred ranks: rank_out[p] = #{q: r_q < r_p or (r_q == r_p and q < p)}, centred_out = rank/(P-1) - 0.5 */
int ppx_rank_center(const double* r, int P, int64_t* rank_out, double* centred_out, void* stream);
/* get_kNN + novelty (evolution_strategies.py:264-281, 318-325), batched over Q queries:
 * sum_out[q] = sum of the S=min(K,M) smallest Euclidean distances (ascending order, f64, no FMA);
 * novelty_out[q] = sum/S floored (<=1e-3 -> 5e-3).  K <= 32. */
int ppx_knn_novelty(const double* archive, int64_t M, const double* queries, int Q, int dim, int K,
                    double* sum_out, double* novelty_out, void* stream);

/* ppx_knn_novelty for a population of queries: the same sum_out / novelty_out as ppx_knn_novelty, bit for bit, for any
 * Q >= 1 (no grid limit, no scratch).  One thread per query keeps a top-K of squared distances; only the S = min(K, M)
 * winners take a square root (monotone under correct rounding, so the selection is the same).  dim 1..8, K 1..32.
 * One launch. */
int ppx_knn_novelty_many(const double* archive, int64_t M, const double* queries, int Q, int dim, int K,
                         double* sum_out, double* novelty_out, void* stream);
/* NSRA-ES update with a novelty per member (Conti et al. 2018, Alg. 3; not in the reference):
 * theta += sum_p c_p eps_p, c_p = lr/(P sigma) * ((1-w) F~_p + w N~_p) / 2 with w = novelty_param, F~ = shape(rewards),
 * N~ = shape(novelties), both over all P members: z-score (ddof 0; a vector whose std is 0 shapes to 0) or, rank_mode = 1,
 * ppx_rank_center's centred ranks.  z-score skips the update (theta and lr untouched, status_out[0] = 1) only when BOTH stds
 * are 0; otherwise, and always in rank mode, *lr_inout *= decay.  W == 1: p_lo = 0, p_n = P, peer arguments NULL, theta
 * updated in place.  W >= 2: the GEMV over this rank's members [p_lo, p_lo + p_n) and the rank-ordered peer-memory apply
 * of ppx_es_update_sharded.  Workspace: ppx_es_update_member_workspace(P, D) bytes. */
int64_t ppx_es_update_member_workspace(int P, int D);
int ppx_es_update_member(double* theta, const float* noise, const int64_t* offsets, const double* rewards, const double* novelties,
                         int P, int p_lo, int p_n, int D, double sigma, double novelty_param, int rank_mode, double decay,
                         double* lr_inout, int* status_out, void* workspace, double* dtheta_local,
                         const void* const* peer_dtheta_host, void* const* peer_flags_host, int W, int rank, uint32_t* seq_dev,
                         uint32_t* status_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PPX_H_ */
