/*
 * dqn_zoo_b200 — C ABI of the B200-native replay-sampler + learner-update hot path.
 *
 * The reference (google-deepmind/dqn_zoo) has no FFI layer: its extension point is the
 * duck-typed Python surface `parts.Agent` / `replay.*` (SURVEY.md §8(b)).  This header is
 * the boundary a maintainer would bind from Python (ctypes stub in INTEGRATION.md); each
 * entry point cites the reference code it replaces.  All citations are relative to the
 * reference repository root.
 *
 * Conventions
 *   - every function returns 0 on success, a negative DZ_E* code otherwise;
 *     dz_last_error() returns a thread-local message for the last failure.
 *   - all pointers named d_* are DEVICE pointers (the caller owns the memory — in the
 *     Python host they are torch.Tensor.data_ptr()); h_* are host pointers.
 *   - `stream` is a cudaStream_t passed as void*.  Nothing synchronises the device
 *     unless the comment says so.  Handles are not thread-safe; distinct handles on
 *     distinct streams may run concurrently.
 *   - no torch / C++ types cross this boundary.
 */
#ifndef DQN_ZOO_B200_H_
#define DQN_ZOO_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DZ_OK 0
#define DZ_EINVAL (-1)   /* bad argument (ValueError in the Python shim) */
#define DZ_ECUDA (-2)    /* CUDA runtime error */
#define DZ_ERANGE (-3)   /* index / target out of range (IndexError / ValueError) */
#define DZ_ESTATE (-4)   /* device-side sticky error flag was raised by a previous kernel */

const char* dz_last_error(void);
/* "dqn_zoo_b200 <version> sm_100a <build date>"; also proves the library loaded. */
const char* dz_build_info(void);
/* Number of kernels this library has launched in this process (bench.py `gpu_launches`). */
int64_t dz_launch_count(void);
/* Measurement aid (bench.py roofline): between begin and end every kernel launch is bracketed by
 * CUDA events on its own stream; end synchronises the device and writes a JSON object
 * {"<kernel or layer tag>": [launches, total_ms], ...} into `out`.  Never active in a timed run. */
int dz_profile_begin(void);
int dz_profile_end(char* out, int64_t cap);

/* ------------------------------------------------------------------------------------------
 * R1  Sum tree  (replaces replay.py:246-426, class SumTree)
 *
 * d_nodes is float64[2*first_leaf]; node i has children 2i, 2i+1; root = node 1; leaves at
 * [first_leaf, 2*first_leaf).  Internal nodes are always recomputed as fl(left+right)
 * (replay.py:284-290, :394-404), so every function below leaves the tree bit-identical to
 * the reference's after the same call.
 * ---------------------------------------------------------------------------------------- */

/* replay.py:394-404 (_set_values): leaves [n_valid, first_leaf) are zeroed, every internal
 * node resummed bottom-up, node 0 cleared. */
int dz_sumtree_rebuild(double* d_nodes, int64_t first_leaf, int64_t n_valid, void* stream);

/* replay.py:278-290 (set): d_nodes[first_leaf+idx[i]] = values[i] for i in order (duplicates:
 * last write wins), then the root paths are resummed.  Values must be finite and >= 0 and
 * indices in [0,size): violations raise the sticky flag bit DZ_FLAG_BAD_VALUE / _BAD_INDEX
 * in *d_flags (checked by the caller when it next synchronises) and the call is a no-op for
 * that element. */
int dz_sumtree_set(double* d_nodes, int64_t first_leaf, int64_t size, const int64_t* d_idx,
                   const double* d_values, int64_t n, int32_t* d_flags, void* stream);

/* replay.py:299-313,406-426 (query/_query_single): smallest leaf index whose inclusive prefix
 * sum exceeds the target; requires 0 <= target < root else DZ_FLAG_BAD_TARGET. */
int dz_sumtree_query(const double* d_nodes, int64_t first_leaf, const double* d_targets, int64_t n,
                     int64_t* d_out_idx, int32_t* d_flags, void* stream);

/* replay.py:271-276 (get). */
int dz_sumtree_get(const double* d_nodes, int64_t first_leaf, int64_t size, const int64_t* d_idx,
                   int64_t n, double* d_out, int32_t* d_flags, void* stream);

#define DZ_FLAG_BAD_VALUE 1
#define DZ_FLAG_BAD_INDEX 2
#define DZ_FLAG_BAD_TARGET 4
#define DZ_FLAG_ROOT_ZERO 8   /* fused PER step met root == 0 (reference would skip an RNG draw) */
#define DZ_FLAG_NONFINITE_WEIGHT 16
#define DZ_FLAG_FRAME_POOL_FULL 32   /* frame store: the ring slot an insert needed is still referenced by a live row */

/* ------------------------------------------------------------------------------------------
 * R5/R6  Replay storage in HBM (replaces the OrderedDict storage of replay.py:120-200 and
 * :654-768; transition-major layout, see DESIGN.md §3)
 * ---------------------------------------------------------------------------------------- */

/* Frame-deduplicated observation storage (DESIGN.md §3).  Observations are uint8 [H][W][S] stacks; each
 * distinct [H][W] plane is kept once in a ring of F frame slots and a row holds 2S slot numbers instead of
 * two stacks.  d_frames == NULL means the raw layout of dz_replay_view.d_obs.
 *
 * Insert rule (dz_replay_add): the 2S planes of s_tm1 | s_t are visited in that order; a plane reuses the
 * most recently appended candidate whose hash AND bytes are equal, among the zero frame (slot 0), the
 * frames appended by the last DZ_FRAME_WINDOW adds and the frames appended earlier in the same add;
 * otherwise it is appended at slot 1 + appends % F.  A frame appended by add j is therefore referenced only
 * by ids in [j, j + DZ_FRAME_WINDOW], and the ring slot at the head may be overwritten iff its last_ref is
 * below the oldest live id.  When it may not, DZ_FLAG_FRAME_POOL_FULL is raised and the row's slots are
 * set to -1 (its observations then read as zeros). */
#define DZ_FRAME_WINDOW 16
#define DZ_FRAME_MAX_STACK 8
#define DZ_FRAME_MAX_STAGE_BYTES (200 * 1024)   /* 2 * stack * frame_stride: the insert de-interleaves both stacks
                                                   into shared memory (84x84x4: 56,448 B) */
typedef struct dz_frame_store {
  uint8_t* d_frames;          /* [F + 1][frame_stride]; slot 0 is the all-zero frame                       */
  int32_t* d_row_frames;      /* [capacity][2S]: frame slot of each plane of s_tm1 | s_t (-1: invalid row) */
  uint64_t* d_frame_hash;     /* [F + 1] frame hash of each slot (slot 0: unused)                          */
  int64_t* d_frame_born;      /* [F + 1] id of the add that appended the frame                             */
  int64_t* d_frame_last_ref;  /* [F + 1] newest id whose row references the frame                          */
  int64_t* d_state;           /* [2 + DZ_FRAME_WINDOW * (1 + 2S)]: appends so far, reserved, then one
                                 window entry per add (id % DZ_FRAME_WINDOW): add id (-1: none) and the 2S
                                 slots it appended in append order (-1 padded)                           */
  uint8_t* d_add_stage;       /* [2][obs_stride]: the two stacks of the add in flight                      */
  uint8_t* d_batch_stage;     /* [2][batch_capacity][obs_stride]: stacks assembled for the fused learner   */
  int64_t num_frames;         /* F */
  int64_t frame_bytes;        /* H * W */
  int64_t frame_stride;       /* frame_bytes rounded up to 16 */
  int32_t stack;              /* S <= DZ_FRAME_MAX_STACK */
  int32_t batch_capacity;
} dz_frame_store;

typedef struct dz_replay_view {
  uint8_t* d_obs;        /* [capacity][2][obs_stride]: s_tm1 then s_t of each transition      */
  int32_t* d_action;     /* [capacity]  a_tm1                                                 */
  double* d_reward;      /* [capacity]  r_t   (float64: n-step returns are built in f64,
                                               replay.py:808-814; rounded to f32 at the learner) */
  double* d_discount;    /* [capacity]  discount_t                                            */
  int64_t capacity;
  int64_t obs_bytes;     /* bytes per observation (84*84*4 = 28224)                           */
  int64_t obs_stride;    /* obs_bytes rounded up to 16                                        */
  /* prioritized replay only (NULL / 0 for uniform) */
  double* d_tree;        /* float64[2*first_leaf]                                             */
  int64_t first_leaf;
  int64_t* d_live;       /* `_active_indices` (replay.py:459): dense list of tree indices     */
  int64_t* d_id_at;      /* `_index_to_id`   (replay.py:455): tree index -> id                */
  /* uniform replay only */
  int64_t* d_ids;        /* `UniformDistribution._ids` (replay.py:49): dense list of ids      */
  int32_t* d_flags;      /* sticky error flags (1 int32)                                      */
  dz_frame_store frames; /* frame-deduplicated storage; frames.d_frames == NULL: d_obs holds raw rows */
} dz_replay_view;

/* One `add` (replay.py:142-151 / :690-699) after the HOST has done the O(1) integer
 * bookkeeping: copies the two observations from host memory into row `slot`, writes the
 * scalars, applies up to 4 (position,value) patches to the dense id/index lists and, for
 * prioritized replay, sets leaf `tree_index` to `leaf_value` (= priority**alpha, evaluated on
 * the host in float64 as replay.py:507 does) and resums its root path.  `evict_index` >= 0
 * zeroes that leaf first (replay.py:533-534). */
typedef struct dz_add_record {
  int64_t slot;
  int32_t action;
  double reward, discount;
  int32_t n_patches;
  int64_t patch_pos[4];
  int64_t patch_val[4];
  int32_t patch_target[4];   /* 0 = d_live, 1 = d_id_at, 2 = d_ids */
  int64_t tree_index;        /* -1 for uniform replay */
  double leaf_value;
  int64_t evict_index;       /* -1 if nothing evicted */
  int64_t size_after;        /* sum-tree `size` for range checks */
  const float* d_priority;   /* optional: take the priority from this DEVICE float32 (the learner's
                                max_seen_priority, rainbow/agent.py:148-149) instead of leaf_value;
                                leaf = ((double)*d_priority) ** alpha in float64, exact for alpha 0.5 / 1 */
  double alpha;
  int64_t item_id;           /* frame store only: id of the transition being added            */
  int64_t oldest_live;       /* frame store only: oldest live id after this add's eviction    */
} dz_add_record;

/* s_tm1 / s_t sources may be HOST arrays or DEVICE buffers (cudaMemcpyDefault; NULL = leave the row's bytes). */
int dz_replay_add(const dz_replay_view* view, const dz_add_record* rec, const uint8_t* h_s_tm1,
                  const uint8_t* h_s_t, void* stream);

/* Bulk pre-fill for benchmarks/tests: rows [row0,row0+n) get deterministic pseudo-random
 * contents (splitmix64 counter hash; byte-identical to oracle/replay_oracle.py:synthetic_rows):
 * uint8 observations iid uniform, action uniform, reward in {-1,0,1} w.p. .05/.9/.05, discount_t =
 * `discount` w.p. .99 else 0 (SURVEY §8(d)). */
int dz_replay_fill_synthetic(const dz_replay_view* view, int64_t row0, int64_t n, uint64_t seed,
                             int32_t num_actions, double discount, void* stream);

/* Frame-store counterpart of dz_replay_fill_synthetic: brings an EMPTY frame store to the exact state that n
 * sequential adds (ids 0..n-1, rows 0..n-1) of 1-step transitions of synthetic episodes produce.  Episodes are
 * `episode_length` transitions long; every timestep shows a new iid frame (splitmix64 of seed and its append
 * index, byte-identical to oracle/frame_store_oracle.py:synthetic_frame); stacks are padded with trailing zero
 * planes at episode start (processors.py:497-504).  Scalars are those of dz_replay_fill_synthetic.  Needs
 * frame_bytes % 8 == 0 and F >= the frames appended (n + ceil(n / episode_length)). */
int dz_replay_fill_synthetic_frames(const dz_replay_view* view, int64_t n, int64_t episode_length, uint64_t seed,
                                    int32_t num_actions, double discount, void* stream);
/* The insert rule's 64-bit frame hash of n host bytes, evaluated on the HOST by the same source the kernels
 * compile; tests only.  hash = mix64(n ^ K0) + sum_k mix64(w_k ^ k * K1) mod 2^64 over the little-endian 8-byte
 * words w_k of the zero-padded bytes (mix64 = the splitmix64 finalizer; constants in csrc/dz_frames.cu). */
int dz_test_frame_hash(const uint8_t* h_bytes, int64_t n, uint64_t* out);

/* Per-step sampling inputs that live in device memory so that a captured CUDA graph can be
 * replayed: the three host RandomState draws of replay.py:551-567 plus the scalars that
 * change as items are added. */
typedef struct dz_sample_inputs {
  const int64_t* d_rand_pos;   /* [B] randint(size, size=B)            (replay.py:551-554 / :78) */
  const double* d_u_tree;      /* [B] uniform(size=B), scaled by root   (replay.py:559)          */
  const double* d_u_mix;       /* [B] uniform(size=B) < usp             (replay.py:563-567)      */
  const double* d_scalars;     /* [4]: size, beta (IS exponent), usp, normalize(0/1)            */
} dz_sample_inputs;

typedef struct dz_sample_outputs {
  int64_t* d_ids;        /* [B] sampled ids                        (replay.py:578-582)     */
  int64_t* d_indices;    /* [B] tree indices (PER) / list positions (uniform)              */
  int64_t* d_slots;      /* [B] storage rows                                               */
  double* d_probs;       /* [B] sampling probabilities (PER)       (replay.py:569-577)     */
  double* d_weights;     /* [B] importance weights, float64 (PER)  (replay.py:211-243)     */
} dz_sample_outputs;

/* replay.py:547-583 + :706-717 (PER) or :76-82 (uniform): indices, ids, probabilities and
 * importance-sampling weights for one batch.  Warp-cooperative sum-tree descent. */
int dz_replay_sample(const dz_replay_view* view, int32_t prioritized, const dz_sample_inputs* in,
                     const dz_sample_outputs* out, int32_t batch, void* stream);

/* replay.py:718-722 (`get` + np.stack): gather rows d_slots[0..B) into dense batch arrays
 * (uint8 [B][obs_bytes] x2, int64 a, float64 r, float64 discount — the dtypes np.stack
 * yields, SURVEY §8(a) R5). */
int dz_replay_gather(const dz_replay_view* view, const int64_t* d_slots, int32_t batch, uint8_t* d_s_tm1,
                     uint8_t* d_s_t, int64_t* d_a, double* d_r, double* d_disc, void* stream);

/* replay.py:725-730 -> :536-545 -> :203-208 (`update_priorities`, `_power` in FLOAT32 as the
 * priorities arrive as a float32 array, SURVEY §8(a) R3) -> SumTree.set.  d_indices are tree
 * indices (as returned in dz_sample_outputs.d_indices).  alpha == 0.5 uses sqrt.rn.f32. */
int dz_replay_update_priorities(const dz_replay_view* view, const int64_t* d_indices, const float* d_priorities,
                                int32_t n, double alpha, int64_t size, void* stream);

/* ------------------------------------------------------------------------------------------
 * Learner (replaces the jitted `update` closure and `_learn` glue of every agent:
 * dqn/agent.py:85-119,179-189; double_q/agent.py:85-123; prioritized/agent.py:86-129,187-206;
 * c51/agent.py:87-120; qrdqn/agent.py:88-122; rainbow/agent.py:85-123,181-198;
 * iqn/agent.py:178-226; networks: networks.py:58-363)
 * ---------------------------------------------------------------------------------------- */

enum dz_agent_kind { DZ_DQN = 0, DZ_DOUBLE_Q = 1, DZ_PRIORITIZED = 2, DZ_C51 = 3, DZ_QRDQN = 4, DZ_RAINBOW = 5, DZ_IQN = 6 };
enum dz_optimizer_kind { DZ_ADAM = 0, DZ_RMSPROP_CENTERED = 1 };

typedef struct dz_learner_config {
  int32_t kind;              /* dz_agent_kind */
  int32_t num_actions;
  int32_t num_atoms;         /* c51 / rainbow: 51 */
  int32_t num_quantiles;     /* qrdqn: 201 */
  int32_t latent_dim;        /* iqn: 64 */
  int32_t tau_samples_s_tm1, tau_samples_policy, tau_samples_s_t; /* iqn: N, K, N' */
  int32_t batch;             /* 32 */
  int32_t obs_h, obs_w, obs_c; /* 84,84,4 */
  float vmax;                /* c51 / rainbow support is linspace(-vmax, vmax, atoms) */
  float grad_error_bound;    /* dqn family: 1/32 (dqn/run_atari.py:79) */
  float huber_param;         /* qrdqn / iqn: 1.0 */
  int32_t optimizer;         /* dz_optimizer_kind */
  float learning_rate, opt_eps, rms_decay, adam_b1, adam_b2;
  float max_global_grad_norm; /* 0 = off (optax.clip_by_global_norm) */
} dz_learner_config;

typedef struct dz_learner_plan {
  int64_t param_count;       /* floats in one parameter blob */
  int32_t num_tensors;
  int64_t opt_state_floats;  /* 2*param_count (adam: mu,nu; rmsprop: mu,nu) */
  int64_t workspace_bytes;
  int64_t noise_floats;      /* rainbow: floats of factorised noise for ONE update (3 applies) */
  int64_t tau_floats;        /* iqn: batch*(N+K+N') */
} dz_learner_plan;

int dz_learner_plan_query(const dz_learner_config* cfg, dz_learner_plan* out);
/* Tensor i of the parameter blob: canonical name ("conv1/w", "adv1/sigma/b", ...), shape
 * (conv w = HWIO, linear w = (in,out); networks_test.py:44,53) and float offset. */
int dz_learner_tensor_info(const dz_learner_config* cfg, int32_t i, char* name64, int64_t* shape4,
                           int32_t* ndim, int64_t* offset);

typedef struct dz_learner_buffers {
  float* d_online;       /* [param_count] */
  float* d_target;       /* [param_count] */
  float* d_grads;        /* [param_count] */
  float* d_opt_state;    /* [opt_state_floats] */
  void* d_workspace;     /* [workspace_bytes] */
  int64_t* d_counters;   /* [4]: 0 = optimizer step count (adam `count`), 1 = rng counter, 2.. reserved */
} dz_learner_buffers;

typedef struct dz_learner dz_learner;
int dz_learner_create(const dz_learner_config* cfg, const dz_learner_buffers* buf, dz_learner** out);
void dz_learner_destroy(dz_learner* l);

/* One batch as device arrays (what `jit(update)` receives after the host->device transfer).
 * Observations are addressed through a pointer table so the fused path can read rows of the
 * replay store in place (gather fused into the conv1 operand load) while the explicit-batch
 * path points into dense arrays. */
typedef struct dz_batch {
  const uint8_t* const* d_s_tm1_rows;  /* [B] device pointers to obs rows */
  const uint8_t* const* d_s_t_rows;    /* [B] */
  const int32_t* d_a_tm1;              /* [B] */
  const float* d_r_t;                  /* [B] float32, as inside jit */
  const float* d_discount_t;           /* [B] */
  const float* d_weights;              /* [B] importance weights (float32) or NULL -> 1 */
  const float* d_taus;                 /* iqn: [B*N | B*K | B*N'] in U[0,1)  (iqn/agent.py:182-190) or NULL */
  const float* d_noise;                /* rainbow: 3 applies x 8 vectors in the order of networks.py:235-248 (adv1 in/out,
                                          adv2 in/out, val1 in/out, val2 in/out), each padded to a multiple of 4 floats; or NULL */
} dz_batch;

typedef struct dz_update_outputs {
  float* d_loss;         /* [1] scalar loss (mean of weighted per-example losses) */
  float* d_per_example;  /* [B] per-example losses (c51/rainbow/qr/iqn) or td errors (dqn family) */
  float* d_priorities;   /* [B] new priorities: rainbow clip(|loss|,0,100) (rainbow/agent.py:194),
                                prioritized |td| (prioritized/agent.py:201); else untouched; may be NULL */
  float* d_grad_norm;    /* [1] global gradient norm before clipping; may be NULL */
} dz_update_outputs;

/* jit(update): forward passes, loss, backward, clip, optimizer, parameter update.
 * `apply_update` = 0 stops after the gradients (d_grads holds dLoss/dparams) for parity tests. */
int dz_learner_update(dz_learner* l, const dz_batch* batch, const dz_update_outputs* out, int32_t apply_update,
                      void* stream);

/* The whole `_learn()` (rainbow/agent.py:181-198) in one enqueue: sample -> (rows addressed in
 * place; with a frame store, stacks assembled into replay->frames.d_batch_stage, DZ_EINVAL when the
 * batch exceeds its batch_capacity) -> update -> priority write-back.  `d_max_seen_priority` ([1] float32, device) is
 * updated as max(old, batch max) (rainbow/agent.py:196-197). */
typedef struct dz_learn_io {
  dz_sample_inputs sample_in;
  dz_sample_outputs sample_out;
  const float* d_taus;
  const float* d_noise;
  dz_update_outputs update_out;
  float* d_max_seen_priority;
  double priority_exponent;  /* alpha */
} dz_learn_io;
int dz_learner_learn(dz_learner* l, const dz_replay_view* replay, int32_t prioritized, const dz_learn_io* io,
                     void* stream);

/* Fills d_taus / d_noise for one update from a counter-based generator (Philox4x32-10 keyed by
 * `seed`, counter d_counters[1] which it advances): taus ~ U[0,1) (iqn/agent.py:45-50); noise =
 * sign(n)*sqrt(|n|), n ~ TruncNormal(-2,2) (networks.py:142-144).  NOT the JAX threefry stream. */
int dz_learner_generate_randomness(dz_learner* l, uint64_t seed, float* d_taus, float* d_noise, void* stream);
/* Same draws, enqueued on the learner's side stream: ordered after the work already on `stream` and before the next
 * dz_learner_learn / dz_learner_update / dz_learner_q_values on `stream` (they run beside the sampler instead of in
 * front of it).  Any other reader of d_taus / d_noise must synchronise the device first. */
int dz_learner_generate_randomness_async(dz_learner* l, uint64_t seed, float* d_taus, float* d_noise, void* stream);

/* select_action's network part (dqn/agent.py:121-131; rainbow/agent.py:125-133; iqn/agent.py:228-243):
 * online forward on ONE observation -> q_values[num_actions] on device.  The epsilon-greedy draw stays on the host. */
int dz_learner_q_values(dz_learner* l, const uint8_t* d_obs, const float* d_taus, const float* d_noise,
                        float* d_q_out, void* stream);

/* Batched acting for E <= batch independent environment streams (parts.py:342-411 run over many actors;
 * dqn/agent.py:121-131,169-177): online forward on E observations in one enqueue, q-values [E][num_actions] and the
 * epsilon-greedy choice on the device, so a tick costs ONE device-to-host copy of E int32 actions.
 *   d_obs      E contiguous uint8 observations (obs_h*obs_w*obs_c bytes each), device memory
 *   d_taus     iqn: [E][tau_samples_policy];  d_noise  rainbow: one noise apply, shared by the E streams of the tick
 *   d_explore  [2][E] float32 uniforms in [0,1) (device) or NULL for greedy acting:
 *              action = u0[e] < epsilon ? min(floor(u1[e] * num_actions), num_actions - 1) : first argmax of q[e] */
int dz_learner_act_batch(dz_learner* l, const uint8_t* d_obs, int32_t E, const float* d_taus, const float* d_noise,
                         const float* d_explore, float epsilon, float* d_q_out, int32_t* d_actions, void* stream);

/* target <- online (dqn/agent.py:155-156): device-to-device copy of the blob. */
int dz_learner_sync_target(dz_learner* l, void* stream);

/* Writes the device's uint8 -> float32/255 conversion of 0..255 (the conv1 operand load, networks.py:193)
 * into d_out256 so tests can check it is the correctly rounded quotient. */
int dz_test_u8_to_unit(float* d_out256, void* stream);


/* Self-test of the packed-operand tcgen05 GEMM (csrc/dz_tcp.cuh; the IQN 3136->512 layer's kernels): packs
 * A (a_rows x red) and B (b_rows x red) from plain fp32 matrices (x_red_contig = 1: element (row, r) at
 * x[row*ld + r]; 0: at x[r*ld + row]) into hi/lo TF32 tile images inside d_work (dz_test_tc_pgemm_work floats),
 * then D[i,j] = sum_r A(i,r) B(j,r).  a_ones_row = a_rows appends a row of ones to A (bias-gradient row), -1: none.
 * splits == 1: + d_bias[j] and ReLU are applied if given; otherwise raw partials at d_C + s*split_stride. */
/* ---- Atari frame preprocessing (SURVEY §8(f) #3) ---------------------------------------------------------------
 * Replaces the observation branch of processors.atari() — np.max over the pooled frame pair, rgb2y, PIL bilinear
 * resize, frame stack (dqn_zoo/processors.py:367-388, 482-501) — for n_env environment streams per launch.
 * One resampling axis of Pillow's bilinear filter (libImaging/Resample.c): window [first, first + count) and
 * fixed-point (22-bit) coefficients per output index; the tables are host-computed by the caller. */
typedef struct dz_resample_axis {
  const int32_t* d_bounds;   /* [out_size][2] = (first, count) */
  const int32_t* d_kk;       /* [out_size][ksize] */
  int32_t ksize, in_size, out_size;
} dz_resample_axis;
/* d_frame_a/b: [n_env] device pointers to uint8 [in_h][in_w][3] raw frames, 16-byte aligned, 3*in_w % 16 == 0
 * (NULL = zero padding, processors.py:54-66);
 * d_stacks[e]: device pointer to stream e's uint8 [out_h][out_w][stack]; d_counts[e] = frames already in stream e's stack
 * (< stack: the new frame goes to channel count; == stack: channels shift left, new frame last);
 * luma3 = {0.299, 0.587, 1 - (0.299 + 0.587)} (host doubles); max_band_rows = the largest number of input rows any
 * band of dz_atari_preprocess_band_rows() output rows touches (sizes the shared-memory staging). */
int dz_atari_preprocess(const uint8_t* const* d_frame_a, const uint8_t* const* d_frame_b, int32_t n_env,
                        const dz_resample_axis* horizontal, const dz_resample_axis* vertical,
                        uint8_t* const* d_stacks, const int32_t* d_counts, int32_t stack, const double* luma3,
                        int32_t max_band_rows, void* stream);
int32_t dz_atari_preprocess_band_rows(void);

/* ---- JAX-compatible uniform draws (SURVEY §8(f) #2) -----------------------------------------------------------
 * jax.random.uniform(key, (count,), float32) for up to 4 independent keys per launch, bit-identical to jax 0.3.10's
 * threefry2x32 path (iqn/agent.py:45-50 `_sample_tau`).  d_keys: DEVICE uint32 [nblocks][2] (so that a captured CUDA
 * graph can be replayed with fresh keys); counts: HOST int64 [nblocks]; block b is written at
 * d_out + sum(counts[:b]). */
int dz_jax_uniform(const uint32_t* d_keys, const int64_t* counts, int32_t nblocks, float* d_out, void* stream);
/* threefry2x32 (20 rounds) evaluated on the HOST by the same source the kernel compiles; tests only. */
int dz_test_threefry2x32(uint32_t k0, uint32_t k1, uint32_t c0, uint32_t c1, uint32_t* out2);

/* Device pointer + element count of an internal learner buffer of the last update (pass 0: "act1", "act2", "act3",
 * "h1", "h1_val", "dh1", "iqn_e0", "iqn_hi", "iqn_dhi");
 * tests/tools only. */
int dz_test_learner_buffer(dz_learner* l, const char* name, float** d_ptr, int64_t* count);
int dz_test_copy(void* d_dst, const void* d_src, int64_t bytes, void* stream);   /* device-to-device, tests only */
/* Debug: the tcgen05 launch named `tag` writes the clock stamps of its CTA 0 into d_trace (512 int64). */
int dz_test_learner_trace(dz_learner* l, const char* tag, long long* d_trace);
/* Debug: every kernel appends (globaltimer ns, gridDim.x << 32 | gridDim.y << 16 | blockDim.x) to d_buf right after its
 * dependencies completed; d_buf[0] (low 32 bits) counts the entries, entries start at d_buf[2].  d_buf: 2 + 2 * 4000
 * uint64, zeroed by the caller; nullptr switches the stamps off.  Works under CUDA-graph replay (tools/step_timeline.py). */
int dz_debug_timeline(unsigned long long* d_buf);
int64_t dz_test_tc_pgemm_work(int32_t a_rows, int32_t b_rows, int32_t red);
int dz_test_tc_pgemm(const float* d_A, int32_t a_rows, int32_t a_ld, int32_t a_red_contig, const float* d_B,
                     int32_t b_rows, int32_t b_ld, int32_t b_red_contig, int32_t red, int32_t a_ones_row,
                     float* d_work, float* d_C, int64_t sc_i, int64_t sc_j, int32_t splits, int64_t split_stride,
                     const float* d_bias, int32_t relu, void* stream);
/* Self-test of the TMA-fed tcgen05 GEMM family (csrc/dz_umma.cuh; conv / FC layers of the batch-32 step):
 * C[MI][NJ] = sum_r A(i,r) B(j,r), NJ <= 64.  x_mn_major = 0: the operand is stored [rows][R]; 1: [R][rows] (the
 * instruction descriptor transposes).  convert = 0: operands pre-split into tf32 hi/lo arrays (activation path);
 * 1: raw fp32 tiles split in shared memory by the converter warps (weight path), A optionally scaled by
 * d_scale_r[r].  epi_rows = 1: row epilogue (+ d_bias[j], relu; tf32 hi/lo copies in d_hi / d_lo).  Synchronizes. */
int dz_test_umma_gemm(const float* d_A, int32_t a_mn_major, const float* d_B, int32_t b_mn_major, int32_t MI, int32_t NJ,
                      int32_t R, int32_t convert, const float* d_scale_r, int32_t run_stages, int32_t epi_rows,
                      const float* d_bias, int32_t relu, float* d_C, float* d_hi, float* d_lo, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DQN_ZOO_B200_H_ */
