/*
 * cql_b200.h -- C ABI of the B200-native CQL recommender hot path.
 *
 * This is the drop-in boundary (SURVEY.md section 8b).  The reference has NO
 * native interface for this path (it ships no native code at all, SURVEY.md
 * section 2.2) -- the functions below replace *Python* call sites, cited per
 * entry point as reference file:line where the call site is in the mounted
 * checkout, or as the upstream d3rlpy / RePlay-CQL location ([EXT], not in
 * the checkout) otherwise.  The Python host (replay_cql_b200/_lib.py) binds
 * them with ctypes; INTEGRATION.md shows the stub a RePlay maintainer adds.
 *
 * Conventions: plain pointers and sizes, no C++/torch types.  Every function
 * returns 0 on success, non-zero on error (cql_last_error() has the text):
 * 3 when an argument, the call sequence or the input data was rejected,
 * 1 or 2 for a CUDA or other failure.
 * "host" pointers are ordinary (ideally pinned) host memory, "dev" pointers
 * are device memory on the handle's GPU.  One handle per GPU; a handle is not
 * thread-safe.  `stream` is a cudaStream_t passed as void*.  NULL selects the
 * handle's own non-blocking stream; functions that take caller-owned DEVICE
 * pointers then synchronise that stream before returning (the caller must have
 * finished producing the inputs), so a NULL-stream call is always safe to follow
 * with work on any other stream.
 */
#ifndef CQL_B200_H
#define CQL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CQL_ABI_VERSION 2
#define CQL_HIDDEN 256          /* d3rlpy default encoder: [256, 256] */
#define CQL_OBS_DIM 2           /* (user_idx, item_idx) */
#define CQL_ACT_DIM 1           /* relevance */
#define CQL_MAX_CRITICS 4
#define CQL_MAX_TOPK 1024
#define CQL_MAX_N_STEPS 64      /* longest n-step TD horizon (cql_set_n_steps) */

/* precision of the 256x256 hidden-layer contraction */
enum { CQL_PREC_FP32 = 0,      /* CUDA-core FP32 (exact-order reference path on the GPU) */
       CQL_PREC_TF32X3 = 1,    /* tcgen05 kind::tf32, 3-term split, FP32-grade */
       CQL_PREC_BF16 = 2,      /* tcgen05 kind::f16 (bf16 operands, fp32 accumulate) */
       CQL_PREC_F16X3 = 3 };   /* tcgen05 kind::f16, fp16 hi/lo 3-term split with exact power-of-two row scales, FP32-grade */

enum { CQL_SQUASH_EPS = 0, CQL_SQUASH_SOFTPLUS = 1 };
enum { CQL_SCORE_Q = 0,        /* mean_i Q_i(x, tanh(mu(x)))  (d3rlpy predict_value(x, predict(x))) */
       CQL_SCORE_POLICY = 1 }; /* tanh(mu(x))                  (d3rlpy predict(x)) */

typedef struct cql_config {
  int32_t struct_size;          /* = sizeof(cql_config), ABI check */
  int32_t device;               /* CUDA ordinal */
  int32_t batch_size;           /* B (per GPU) */
  int32_t n_critics;            /* C, 1..CQL_MAX_CRITICS */
  int32_t n_action_samples;     /* n, 1..10 */
  int32_t precision;            /* CQL_PREC_* */
  int32_t squash;               /* CQL_SQUASH_* */
  int32_t rank, world_size;     /* data-parallel position (sampling streams only; no comms inside) */
  float gamma, tau;
  float actor_lr, critic_lr, temp_lr, alpha_lr;
  float initial_temperature, initial_alpha;
  float alpha_threshold, conservative_weight;
  float beta1, beta2, adam_eps;
  uint64_t seed;
} cql_config;

typedef struct cql_handle cql_handle;

/* ---- lifetime ---------------------------------------------------------- */
/* replaces: d3rlpy.algos.CQL(...).create_impl() [EXT d3rlpy/algos/cql.py]   */
int  cql_create(const cql_config* cfg, cql_handle** out);
void cql_destroy(cql_handle* h);
const char* cql_last_error(const cql_handle* h);   /* h may be NULL: error of the last failed cql_create */
int  cql_abi_version(void);

/* ---- flat state -------------------------------------------------------- */
/* Flat layout (floats), NET = 67136-float slot per network (see DESIGN.md):
 *   [actor | critic_0..C-1 | targ_actor | targ_critic_0..C-1 | scalars(64)]
 *   net slot: W1[H][in] b1[H] W2[H][H] b2[H] W3[out][H] b3[out]  (PyTorch (out,in) row-major)
 *   scalars : [0]=log_temp [1]=log_alpha
 * replaces: torch state_dict save/load in the wrapper's _save_model/_load_model
 *           (hook: replay/models/base_rec.py:280-284; caller replay/model_handler.py:38,90) */
int64_t cql_state_floats(const cql_handle* h);
int  cql_set_weights(cql_handle* h, const float* host_flat, int64_t n);
int  cql_get_weights(cql_handle* h, float* host_flat, int64_t n);
/* Adam moments (same flat layout, trainable part meaningful) + step counter: exact resume (SURVEY 8f-4) */
int  cql_set_optimizer(cql_handle* h, const float* host_m, const float* host_v, int64_t n, int64_t step);
int  cql_get_optimizer(cql_handle* h, float* host_m, float* host_v, int64_t n, int64_t* step);

/* ---- replay table (K1) ------------------------------------------------- */
/* Episode-ordered steps -> 32-byte transition rows resident in HBM.
 * replaces: d3rlpy MDPDataset(...) + Episode._to_transitions [EXT d3rlpy/dataset.pyx]
 * obs [n][2], act [n], rew [n], term [n]  (host).  next_obs = next row unless term. */
int  cql_load_transitions(cql_handle* h, const float* obs, const float* act,
                          const float* rew, const float* term, int64_t n);
int64_t cql_num_transitions(const cql_handle* h);
/* MDP builder on the GPU: interaction log columns (host, input order) -> replay table, one episode per user.
 * order (user, timestamp, input order); reward = 1 for the user's top_k rows by (relevance desc, timestamp desc);
 * terminal = user's last row (top_k <= 0 rewards nothing); action = (float)relevance + noise.  action_noise (host, per ORIGINAL row, already
 * scaled; may be NULL => seeded N(0,1)*noise_scale on the device).  Optional host outputs (all NULL or all set):
 * obs_out [n][2], act_out/rew_out/term_out [n] in episode order; order_out [n] = original row of each step.
 * timestamp holds int64 sort keys: float timestamps go through an order-preserving key on the host first
 * (replay_cql_b200/frames.py timestamps_to_int64).  A NaN or infinite relevance fails the call (no table is left).
 * replaces: MdpDatasetBuilder.build (two Spark window sorts + orderBy + toPandas) [EXT upstream RePlay CQL wrapper] */
int  cql_build_mdp(cql_handle* h, const int32_t* user_idx, const int32_t* item_idx, const int64_t* timestamp,
                   const double* relevance, const double* action_noise, int64_t n, int32_t top_k, float noise_scale,
                   float* obs_out, float* act_out, float* rew_out, float* term_out, int64_t* order_out);
/* The same builder fed in CHUNKS (SURVEY 8f-1: Arrow record batches / Parquet row groups / pandas columns, each in its
 * own dtype, no intermediate frame): cql_mdp_begin announces n rows; cql_mdp_append adds the next `count` values of
 * one column (col: 0 user_idx, 1 item_idx, 2 timestamp, 3 relevance, 4 action noise [optional]; dtype CQL_DT_*,
 * but only CQL_DT_I32 / CQL_DT_I64 keys for timestamps -- a float timestamp is rejected, not truncated; chunks
 * of a column arrive in row order, columns in any order -- timestamps first lets their sorts overlap the other
 * uploads).  Every chunk goes host -> pinned ring (up to four copy threads) -> device asynchronously.
 * cql_mdp_finish sorts, builds the replay table and ends the session (outputs as for cql_build_mdp).
 * replaces: `log.toPandas()` (pattern replay/models/neuromf.py:332) + MdpDatasetBuilder.build [EXT] */
enum { CQL_DT_I32 = 0, CQL_DT_I64 = 1, CQL_DT_F32 = 2, CQL_DT_F64 = 3 };
int  cql_mdp_begin(cql_handle* h, int64_t n_rows);
int  cql_mdp_append(cql_handle* h, int32_t col, int32_t dtype, const void* host_chunk, int64_t count);
int  cql_mdp_finish(cql_handle* h, int32_t top_k, float noise_scale,
                    float* obs_out, float* act_out, float* rew_out, float* term_out, int64_t* order_out);
/* Data parallel with the replay table SHARDED by user range (SURVEY 8e): this rank's table holds only its own users'
 * episodes, so on-device sampling walks this rank's own epoch permutation (position = step * B + j) instead of the
 * job-wide one ((step * world + rank) * B + j over a replicated table).  The Philox streams stay per rank. */
int  cql_set_table_sharded(cql_handle* h, int32_t sharded);
/* Synthetic replay table of a BASELINE.json shape generated IN PLACE on the device (measurement aid for the stress
 * configuration: 1e9 rows x 32 B = 32 GB): user-major episodes of fixed length ceil(n / n_users), Zipf-like items,
 * ML-like ratings + N(0, 1e-3) as actions, ~10 rewarded rows per episode, terminal on each episode's last row.
 * Row i depends only on (seed, i).  replaces: nothing in the reference -- stands in for SURVEY 8d's generator where
 * the log itself (24 GB of columns) is not worth moving through the host. */
int  cql_synth_table(cql_handle* h, int64_t n_rows, int64_t n_users, int64_t n_items, uint64_t seed);
/* n-step TD returns (d3rlpy's `n_steps`, DESIGN.md section 1), 1..CQL_MAX_N_STEPS, default 1.  With n_steps > 1 every
 * table built after the call (cql_build_mdp, cql_mdp_finish, cql_load_transitions, cql_synth_table) holds n-step rows:
 * for one-step row t with k = min(n_steps, steps from t to its episode's end, t included) -- an episode ends at a
 * terminal row or at the end of the table -- the row is (s_t, a_t, R | s'_{t+k-1}, term_{t+k-1}, discount) with
 * R = sum_{j<k} gamma^j r_{t+j} and discount = gamma^k, both accumulated in float64 and stored as float; the TD
 * target is then y = R + discount * min_i Q_targ_i(s', tanh(mu(s'))) * (1 - term).  The one-step expansion is an
 * out-of-place pass over the rows the builder writes (transiently twice the table's memory); the builders' optional
 * host outputs stay the one-step episode steps.  With n_steps = 1 the tables (slot 7 = 0) and the update are as they
 * always were.  A table already loaded is DROPPED when the value changes (it was built for the other horizon: rebuild
 * or reload it); captured update graphs are destroyed. */
int  cql_set_n_steps(cql_handle* h, int32_t n_steps);
/* Replay table uploaded verbatim from rows_host [n][8] in the table's own format (e.g. cql_sample_rows / a checkpoint
 * of this handle's table): no expansion, whatever n_steps is. */
int  cql_set_table_rows(cql_handle* h, const float* rows_host, int64_t n);
/* Column statistics of the loaded table (d3rlpy's scaler fit, DESIGN.md section 1): every table producer
 * (cql_build_mdp, cql_mdp_finish, cql_load_transitions, cql_synth_table, cql_set_table_rows) reduces the one-step rows
 * it builds -- before any n-step expansion -- to count, min, max, mean and M2 = sum (x - mean)^2 per column, in float64
 * and in a fixed order that depends only on the row count: the same steps give the same bits whichever producer built
 * them.  col[]: 0 obs.x (user), 1 obs.y (item), 2 act, 3 rew.  cql_set_table_rows with n_steps > 1 sees n-step
 * returns in the reward slot: rew_available = 0 there (and 0 when no table is loaded). */
typedef struct cql_column_stats { int64_t count; double min, max, mean, m2; } cql_column_stats;
typedef struct cql_table_stats {
  cql_column_stats col[4];
  int32_t rew_available;
  int32_t pad;
} cql_table_stats;
int  cql_get_table_stats(cql_handle* h, cql_table_stats* out);
/* d3rlpy's observation / action / reward scalers (scaler, action_scaler, reward_scaler; DESIGN.md section 1), applied
 * to every minibatch as the update gathers it (s and s', a, r; the table stays raw) and to the (user, item)
 * observations of the scorers; CQL_SCORE_POLICY returns the reverse action transform of tanh(mu(x')).  All float32,
 * each operation rounded separately:
 *   min_max (obs, rew): x' = (x - a) / (b - a)              a = minimum, b = maximum, (b - a) rounded once
 *   standard (obs, rew): x' = (x - a) / (b + 1e-3)          a = mean, b = std, (b + 1e-3) rounded once
 *   min_max (act): a' = ((a - min) / (max - min)) * 2 - 1;  reverse ((a' + 1) / 2) * (max - min) + min
 * Observation parameters are per dimension (user, item).  Kinds: obs and rew NONE / MIN_MAX / STANDARD, act NONE /
 * MIN_MAX; a min_max column needs max > min, a standard one std >= 0.  Captured update graphs are destroyed when the
 * parameters change.  A staged minibatch (cql_upload_batch) stays raw: phase 4 scales it on every run.  All kinds NONE (the default) leaves every kernel on its unscaled path. */
enum { CQL_SCALER_NONE = 0, CQL_SCALER_MIN_MAX = 1, CQL_SCALER_STANDARD = 2 };
typedef struct cql_preprocessing {
  int32_t obs_kind, act_kind, rew_kind, pad;
  float obs_a[2], obs_b[2];     /* per dimension: min_max (minimum, maximum), standard (mean, std) */
  float act_a, act_b;
  float rew_a, rew_b;
} cql_preprocessing;
int  cql_set_preprocessing(cql_handle* h, const cql_preprocessing* p);
int  cql_get_preprocessing(cql_handle* h, cql_preprocessing* out);
/* stand-alone gather for the K1 roofline sweep: out_dev [count][8] floats.
 * idx_dev NULL => the handle's epoch permutation starting at position `pos`. */
int  cql_sample_rows(cql_handle* h, const int64_t* idx_dev, int64_t pos, int64_t count,
                     float* out_dev, void* stream);

/* ---- update (K2-K4) ---------------------------------------------------- */
/* n_steps fused updates with on-device sampling and Philox noise.
 * metrics6 (host, may be NULL): temp_loss,temp,alpha_loss,alpha,critic_loss,actor_loss of the LAST step.
 * replaces: d3rlpy CQL._update per step of CQL.fit [EXT d3rlpy/algos/cql.py, algos/torch/cql_impl.py] */
int  cql_update(cql_handle* h, int64_t n_steps, float* metrics6, void* stream);

/* One update on a caller-supplied minibatch (host buffers, B rows) -- the parity
 * and end-to-end entry.  noise (host, may be NULL => Philox): packed
 * [temp_eps B | alpha_eps_t B*n | alpha_eps_t1 B*n | alpha_u B*n |
 *  critic_eps_t B*n | critic_eps_t1 B*n | critic_u B*n | actor_eps B].
 * grads_out (host, may be NULL): trainable gradients in flat layout
 * [actor | critics | scalars] = (1+C)*NET + 64 floats (averaged over the batch).
 * replaces: CQLImpl.update_temp/update_alpha/update_critic/update_actor/update_*_target [EXT] */
int  cql_update_batch(cql_handle* h, const float* obs, const float* act, const float* rew,
                      const float* next_obs, const float* term, const float* noise,
                      float* metrics6, float* grads_out, void* stream);
/* The same update on B table-format rows (host [B][8]: s.x s.y a r s'.x s'.y term discount), e.g. rows of an n-step
 * table; slot 7 is the row's TD discount when n_steps > 1 and is ignored otherwise.  cql_update_batch (and the
 * one-step batches of cql_update_batches / cql_upload_batch) stage discount = gamma when n_steps > 1. */
int  cql_update_batch_rows(cql_handle* h, const float* rows_host, const float* noise, float* metrics6, float* grads_out,
                           void* stream);

/* n_batches consecutive updates on caller-supplied minibatches (host buffers, n_batches x B rows each, Philox noise):
 * the host loop of an offline trainer that owns its batches.  Per step the minibatch goes host -> pinned ring -> device
 * and the six metrics come back; copies and steps are pipelined on `stream` (the host runs up to 8 steps ahead) and the
 * call returns after the last step.  metrics_out (host, may be NULL): [n_batches][6].
 * replaces: the per-step loop of d3rlpy LearnableBase.fit over TransitionMiniBatch objects [EXT d3rlpy/base.py] */
int  cql_update_batches(cql_handle* h, int64_t n_batches, const float* obs, const float* act, const float* rew,
                        const float* next_obs, const float* term, float* metrics_out, void* stream);

/* Data-parallel split of one update.  The host all-reduces (mean) the exposed
 * gradient buffer between phases; with world_size==1 the phases can be called
 * back to back (f16x3 at world_size==1: the critic and actor gradients are summed
 * by the Adam step, i.e. they are in the buffer after phase 2 and phase 3).
 *                phase 0: sample + forward passes + temp/alpha grads
 *                phase 1: temp/alpha Adam, critic backward  -> critic grads
 *                phase 2: critic Adam + Polyak, actor passes -> actor grads
 *                phase 3: actor Adam + Polyak, step counter
 *                phase 4: phase 0 on the minibatch staged by cql_upload_batch  */
int  cql_step_phase(cql_handle* h, int phase, void* stream);
/* Data-parallel end-to-end variant: stage a caller-supplied host minibatch (B rows), then run the phases with
 * phase 4 in place of phase 0 (same work, the uploaded batch instead of a sampled one). */
int  cql_upload_batch(cql_handle* h, const float* obs, const float* act, const float* rew,
                      const float* next_obs, const float* term, void* stream);
enum { CQL_BUF_SCALAR_GRADS = 0,   /* 64 floats: [0]=d log_temp [1]=d log_alpha */
       CQL_BUF_CRITIC_GRADS = 1,   /* C*NET floats */
       CQL_BUF_ACTOR_GRADS = 2,    /* NET floats */
       CQL_BUF_METRICS = 3,        /* 8 floats */
       CQL_BUF_PARAMS = 4,
       CQL_BUF_ALL_GRADS = 5 };    /* (1+C)*NET+64 floats: [actor | critics | scalars] */
int  cql_device_buffer(cql_handle* h, int which, void** dev_ptr, int64_t* n_floats);

/* Seen-items CSR of an interaction log, built on the device -- the structure the scorer's lazy seen filter searches
 * (replaces the host-side joins of `_filter_seen`, replay/models/base_rec.py:417-464, for the GPU path).
 * users_host / items_host [n] int32: the log's id columns in any order, duplicates allowed (host memory); rows with
 * a user outside [0, n_users_dim) or a negative item are dropped (no candidate id is negative: they filter nothing);
 * wanted_host [n_users_dim] uint8 or NULL: keep only rows of users whose flag is non-zero;
 * indptr_dev [n_users_dim + 1] int64 and seen_dev [>= n] int32: device buffers of the caller; on return user u's
 * de-duplicated items, ascending, are seen_dev[indptr_dev[u] .. indptr_dev[u + 1]); *n_seen_out = entries written.
 * Two column uploads, one radix sort over the significant key bits, one unique pass, one emit pass; synchronises. */
int  cql_seen_csr(cql_handle* h, const int32_t* users_host, const int32_t* items_host, int64_t n, int64_t n_users_dim,
                  const uint8_t* wanted_host, int64_t* indptr_dev, int32_t* seen_dev, int64_t* n_seen_out, void* stream);

/* Data-parallel gradient exchange over NVLink peer memory instead of a collective library call (SURVEY 8e).
 * cql_dp_attach: stage_ptrs[world] / signal_ptrs[world] are every rank's symmetric, zero-initialised staging buffer
 *   (buffer_floats floats: >= 2 x stage_floats, stage_floats >= the CQL_BUF_ALL_GRADS size; with another
 *   4 x world x stage_floats behind them the exchange is fused into the update kernels, see cql_dp_mode) and
 *   zero-initialised signal pad (>= world x 4 64-bit words), mapped into this process (e.g.
 *   torch.distributed._symmetric_memory handles); all ranks must attach before the first exchange and call the
 *   exchanges in the same order.
 * cql_dp_allreduce: mean over ranks of one gradient buffer (CQL_BUF_SCALAR_GRADS / _CRITIC_GRADS / _ACTOR_GRADS), in
 *   place, one kernel on `stream` (publish + one-shot reduce in rank order: bit-identical on every rank).  Replaces the
 *   torch.distributed.all_reduce between cql_step_phase calls.  cql_dp_error returns 1 after a wait timed out. */
int  cql_dp_attach(cql_handle* h, int32_t world, int32_t rank, const void* const* stage_ptrs,
                   const void* const* signal_ptrs, int64_t stage_floats, int64_t buffer_floats);
int  cql_dp_allreduce(cql_handle* h, int which, void* stream);
int  cql_dp_error(cql_handle* h, int32_t* flag_out);
/* *fused_out = 1 when, after cql_dp_attach, the gradient exchange happens INSIDE the update kernels (f16x3 path, staging
 *   buffers with room for the pushed packets): the kernel that produces a gradient group stores its sums of slice o
 *   straight into rank o's staging buffer over NVLink as {value, epoch tag} pairs; in the kernel that consumes the group
 *   (Adam + Polyak + pack) the owner of a slice polls its own buffer for the tags, sums in rank order and pushes the mean
 *   to every rank, and every thread polls the means it needs; the two scalar gradients travel inside the signal words --
 *   no exchange launch, no fence, and cql_update / cql_update_batches / cql_step_phase run data-parallel as they are
 *   (cql_dp_allreduce is then a no-op).
 *   0: call cql_dp_allreduce (or an NCCL all-reduce) between the phases. */
int  cql_dp_mode(cql_handle* h, int32_t* fused_out);

/* ---- scoring (K5) ------------------------------------------------------ */
/* For each user: relevance of every candidate item, minus the user's seen
 * items (CSR, sorted item ids per user; seen_indptr may be NULL = no filter),
 * top-k by (relevance desc, item asc).  Rows with fewer than k candidates are
 * padded with item -1 / score -inf.  A negative candidate id is skipped: it is
 * never returned and does not count as a candidate.
 * replaces: CQL._predict per-user loop [EXT; pattern replay/models/neuromf.py:394-438]
 *           + _filter_seen replay/models/base_rec.py:417-464
 *           + get_top_k_recs replay/utils.py:112-127
 * All pointers host; out_items [U][k] int32, out_scores [U][k] float. */
int  cql_score_topk(cql_handle* h, const int32_t* users, int64_t n_users,
                    const int32_t* items, int64_t n_items,
                    const int64_t* seen_indptr, const int32_t* seen_items,
                    int32_t k, int32_t mode,
                    int32_t* out_items, float* out_scores, void* stream);
/* same, every pointer already on the device (HBM-resident measurement) */
int  cql_score_topk_dev(cql_handle* h, const int32_t* users, int64_t n_users,
                        const int32_t* items, int64_t n_items,
                        const int64_t* seen_indptr, const int32_t* seen_items,
                        int32_t k, int32_t mode,
                        int32_t* out_items, float* out_scores, void* stream);
/* relevance of explicit (user,item) pairs (host pointers).
 * replaces: the generic _predict_pairs fallback replay/models/base_rec.py:784-823 */
int  cql_score_pairs(cql_handle* h, const int32_t* users, const int32_t* items, int64_t n,
                     int32_t mode, float* out_scores, void* stream);

/* Stand-alone HBM-bound top-k + seen filter over a materialised score matrix
 * scores_dev [U][I] (SURVEY 8d: the well-defined HBM denominator for scoring/top-k).
 * users_dev gives each row's user id for the seen CSR (NULL => row index). */
int  cql_topk_filter_dev(cql_handle* h, const float* scores_dev, int64_t n_users, int64_t n_items,
                         const int32_t* users_dev, const int32_t* items_dev,
                         const int64_t* seen_indptr, const int32_t* seen_items,
                         int32_t k, int32_t* out_items, float* out_scores, void* stream);

/* Ranking metrics of a U x k_rec recommendation table against the ground truth, on the GPU (host pointers).
 * replaces: Metric.__call__ -> get_enriched_recommendations + _get_metric_value_by_user,
 *           replay/metrics/base_metric.py:102-140,178-200 and ndcg.py:51-61, hitrate.py, map.py, mrr.py,
 *           precision.py, recall.py (the evaluation step of optimize(), replay/models/base_rec.py:150-274).
 * rec_items [U][k_rec]: best first, padded with -1; users [U]: user id of each row (the ground-truth users --
 * a user without recommendations is a row of -1 and scores 0); gt_indptr/gt_items: CSR over user id, items
 * sorted ascending per user; ks [n_ks] (n_ks <= 8, each <= k_rec is not required).
 * out_means [6][n_ks] in the order NDCG, HitRate, MAP, MRR, Precision, Recall (means over the U users). */
int  cql_rank_metrics(cql_handle* h, const int32_t* rec_items, int64_t n_users, int32_t k_rec,
                      const int32_t* users, const int64_t* gt_indptr, const int32_t* gt_items,
                      const int32_t* ks, int32_t n_ks, double* out_means, void* stream);

/* ---- offline evaluation ------------------------------------------------ */
/* d3rlpy's offline scorers (DESIGN.md section 1) over the loaded one-step replay table, as float64 SUMS and counts so
 * that the results of several table shards can be combined.  An episode ends at a terminal row or at the end of the
 * table; d3rlpy's 1024-transition windows restart the advantage recursion.  Per row, in float32 as the update forms them
 * (scalers applied: s and s' observation-scaled, a action-scaled into Q, r reward-scaled in the target; the greedy action
 * tanh(mu(x)) enters Q in network space): Q(s,a) = mean_i Q_i(s, a), V(x) = mean_i Q_i(x, tanh(mu(x))), sigma(x) =
 * population std of the Q_i(x, tanh(mu(x))).  return_threshold: episodes whose float64 sum of RAW rewards is >= it are
 * successes (soft OPC); NaN = no soft OPC (success sums 0).  Rejected (3) when no table is loaded or n_steps > 1.
 * Synchronises `stream`.
 * replaces: d3rlpy.metrics.scorer td_error_scorer, discounted_sum_of_advantage_scorer, average_value_estimation_scorer,
 *           value_estimation_std_scorer, initial_state_value_estimation_scorer, soft_opc_scorer,
 *           continuous_action_diff_scorer [EXT d3rlpy 1.x metrics/scorer.py] */
typedef struct cql_offline_sums {
  double td_error;              /* sum over rows of (Q(s,a) - y)^2, y = r' + gamma * V(s') * (1 - term) (one-step) */
  double discounted_advantage;  /* sum over rows of the windowed discounted advantage sum A_t (adv = Q(s,a) - V(s)) */
  double value;                 /* sum over rows of V(s) */
  double value_std;             /* sum over rows of sigma(s) */
  double initial_value;         /* sum over episodes of V(s_0) */
  double action_diff;           /* sum over rows of (a - reverse(tanh(mu(s))))^2, a raw */
  double success_q;             /* sum of Q(s,a) over the rows of successful episodes */
  double all_q;                 /* sum of Q(s,a) over all rows */
  int64_t n_rows, n_episodes, n_success_rows;
} cql_offline_sums;
int  cql_offline_eval(cql_handle* h, float return_threshold, cql_offline_sums* out, void* stream);

/* Measurement aid: runs ONE sampled update with CUDA events around the heavy launches and
 * returns their durations in milliseconds (synchronises).  out_ms[0] = critic forward (alpha +
 * critic + target rows), [1] = critic backward-1, [2] = critic backward-2 (dW2), [3] = whole
 * update, [4] = actor-step critic forward, [5] = actor backward (1+2), [6] = shared actor
 * forward, [7] = everything else.  The update is a real one (weights advance).  Programmatic dependent launch is
 * off for this step (events between overlapping kernels would not separate them), and the critic forward is launched
 * four times back to back between its two events (same inputs, same outputs; the repeats with programmatic dependent
 * launch, as in the step graph): [0] is that span / 4, the kernel's steady-state duration without the launch latency of
 * a lone launch; [3] counts it once. */
int  cql_timed_update(cql_handle* h, float* out_ms8, void* stream);

/* Self-test of the tensor-core building blocks (tcgen05.mma + TMEM + operand layout):
 * D[128][n] = A[128][k] * B[n][k]^T with `precision` = CQL_PREC_BF16 or CQL_PREC_TF32X3 (host pointers);
 * add 0x100 to `precision` to stage operand A in tensor memory (tcgen05.st, "TS" MMA) instead of shared memory. */
int  cql_selftest_umma(cql_handle* h, int precision, const float* A_host, const float* B_host,
                       int n, int k, float* D_host);

/* Measurement aid (DESIGN.md section 3): issue rate of back-to-back tcgen05.mma kind::f16 K=16 instructions.
 * mode bit 0: A operand in tensor memory (else shared memory); bit 1: N = 256 (else 128); bit 2: cta_group::2 on a
 * CTA pair, M = 256 (else one CTA, M = 128); bit 3: alternate operand addresses in the 3-term pattern.
 * out_clk2[0] = SM clocks to ISSUE `iters` MMAs, [1] = clocks until the last one has retired. */
int  cql_mma_bench(cql_handle* h, int mode, int iters, int64_t* out_clk2);

/* number of kernels this library has launched on the handle (bench "gpu_launches") */
int64_t cql_launch_count(const cql_handle* h);

#ifdef __cplusplus
}
#endif
#endif /* CQL_B200_H */
