/*
 * bsuite_b200 -- C ABI of the batched bsuite environment engine (sm_100a).
 *
 * This header is the drop-in boundary for the one hot path this repo builds:
 * the per-environment step()/reset() dynamics of google-deepmind/bsuite
 * (reference: bsuite/environments/<name>.py, experiments/cartpole_swingup,
 * utils/wrappers.py::RewardNoise/RewardScale), executed for B independent
 * environment "lanes" in lock-step.
 *
 * The reference has no FFI layer (SURVEY.md 8b): its boundary is the Python
 * object contract of bsuite/environments/base.py:34-77.  Each entry point
 * below names the reference interface it replaces.  The Python binding a
 * maintainer would add is a ctypes stub (INTEGRATION.md); ours lives in
 * bsuite_b200/_lib.py.
 *
 * Conventions
 *   - plain C, no C++/torch types; every function returns a bsb_status.
 *   - buffers are CALLER-OWNED.  For a device environment every pointer in
 *     bsb_outputs / `actions` is a device pointer on that device and the work
 *     is enqueued on `stream` (a cudaStream_t passed as void*; NULL = legacy
 *     default stream).  For a host environment (device == BSB_DEVICE_HOST) the
 *     pointers are host pointers and the call is synchronous.
 *   - the library owns only lane state, RNG counters and config tables.
 *   - calls on one handle are not thread-safe; distinct handles are independent.
 *   - a lane whose previous timestep was LAST ignores its action and emits
 *     FIRST (base.py:59-65).  FIRST lanes carry reward = 0, discount = 0; the
 *     reference's `None` is recovered from step_type == BSB_FIRST.
 */
#ifndef BSUITE_B200_H_
#define BSUITE_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BSB_ABI_VERSION 8
#define BSB_DEVICE_HOST (-1)
#define BSB_MAX_INFO 4

typedef enum bsb_status {
  BSB_OK = 0,
  BSB_INVALID_ARGUMENT = 1,
  BSB_UNSUPPORTED = 2,
  BSB_CUDA_ERROR = 3,
  BSB_OUT_OF_MEMORY = 4,
  BSB_INTERNAL = 5
} bsb_status;

/* dm_env.StepType values (dm_env is the reference's L0 substrate). */
typedef enum bsb_step_type { BSB_FIRST = 0, BSB_MID = 1, BSB_LAST = 2 } bsb_step_type;

/* One entry per environment CLASS of the reference (SURVEY.md 8a a2..a11). */
typedef enum bsb_family {
  BSB_DEEP_SEA = 0,          /* environments/deep_sea.py:51-155            */
  BSB_CATCH = 1,             /* environments/catch.py:45-117               */
  BSB_CARTPOLE = 2,          /* environments/cartpole.py:37-181            */
  BSB_CARTPOLE_SWINGUP = 3,  /* experiments/cartpole_swingup/cartpole_swingup.py:41-155 */
  BSB_MOUNTAIN_CAR = 4,      /* environments/mountain_car.py:33-102        */
  BSB_MEMORY_CHAIN = 5,      /* environments/memory_chain.py:37-112        */
  BSB_BANDIT = 6,            /* environments/bandit.py:35-73               */
  BSB_UMBRELLA_CHAIN = 7,    /* environments/umbrella_chain.py:39-114      */
  BSB_DISCOUNTING_CHAIN = 8, /* environments/discounting_chain.py:40-105   */
  BSB_MNIST = 9,             /* environments/mnist.py:36-85                */
  BSB_NUM_FAMILIES = 10
} bsb_family;

/* utils/wrappers.py:250-373, fused into the transition kernel's epilogue. */
typedef enum bsb_wrapper {
  BSB_WRAP_NONE = 0,
  BSB_WRAP_REWARD_NOISE = 1, /* r + noise_scale * randn()   (wrappers.py:275-283) */
  BSB_WRAP_REWARD_SCALE = 2  /* r * reward_scale            (wrappers.py:338-346) */
} bsb_wrapper;

/* Which bit source feeds numpy's legacy RandomState algorithms per lane. */
typedef enum bsb_rng_kind {
  /* Philox4x64-10 (numpy.random.Philox layout): lane i of the batch consumes
   * exactly the stream of numpy.random.RandomState(numpy.random.Philox(
   * key=[seed, lane_offset+i])); the reward wrapper's private RandomState
   * (wrappers.py:267,330) is the same key with counter=[0,0,0,1].           */
  BSB_RNG_PHILOX = 0,
  /* MT19937 exactly as numpy.random.RandomState(seed + lane_offset + i): a
   * B=1 environment then reproduces the UNPATCHED reference for integer
   * seeds.  2.5 KB of generator state per lane; meant for small batches.    */
  BSB_RNG_MT19937 = 1
} bsb_rng_kind;

/*
 * Environment configuration: the keyword arguments of the reference
 * constructors, flattened into one POD.  Fields that do not apply to `family`
 * are ignored.  Tables are HOST pointers; bsb_create copies them.
 */
typedef struct bsb_config {
  int32_t family;        /* bsb_family */
  int32_t wrapper;       /* bsb_wrapper */
  int32_t rng_kind;      /* bsb_rng_kind */
  int32_t flags;         /* BSB_FLAG_* */

  /* deep_sea.py:51-57 */
  int32_t size;          /* N */
  int32_t deterministic; /* 1 = deterministic (default), 0 = 'windy' */
  /* catch.py:45-48 */
  int32_t rows, columns;
  /* memory_chain.py:37-40 */
  int32_t memory_length, num_bits;
  /* umbrella_chain.py:39-42 */
  int32_t chain_length, n_distractor;
  /* bandit.py:35 */
  int32_t num_actions;
  /* mountain_car.py:36-38 */
  int32_t max_steps;
  /* mnist.py:36 (num_data = int(fraction * len(labels)), 28x28 images) */
  int32_t num_data, image_rows, image_cols;
  /* bsb_experiment whose score summary the lanes keep (BSB_FLAG_SCORE_SUMMARY;
   * read only with that flag, so zeroed configs are unaffected) */
  int32_t score_experiment;

  double unscaled_move_cost;                         /* deep_sea.py:54 */
  double height_threshold, x_threshold, timescale,   /* cartpole.py:82-87 */
         max_time, init_range;
  double theta_dot_threshold, x_reward_threshold,    /* cartpole_swingup.py:51-60 */
         move_cost;
  double noise_scale;                                /* wrappers.py:253-256 */
  double reward_scale;                               /* wrappers.py:316-319 */

  /* Host tables, built by the caller with the SAME numpy calls the reference
   * constructors make, so they are equal by construction:
   *   deep_sea : uint8  [N*N]  action mapping  (deep_sea.py:79-85)
   *   bandit   : double [num_actions] rewards  (bandit.py:45-47)
   *   discounting_chain : double [5] rewards   (discounting_chain.py:55-56)
   *   mnist    : int8   [num_data*rows*cols] images (utils/datasets.py:52-56) */
  const void* table;
  int64_t table_bytes;
  /*   mnist    : uint8  [num_data] labels */
  const void* table2;
  int64_t table2_bytes;

  /* Log schedule of the reference's Logging wrapper (utils/wrappers.py:99-110,
   * 140-147): the ascending episode counts {1, 1.2, ..., 10} x 10^k up to
   * bsuite_num_episodes at which it writes a row.  When given (host int64
   * array; needs BSB_FLAG_TRACK_EPISODES) every lane records its own row --
   * the five Logging columns + bsuite_info() at that LAST timestep -- on the
   * device (bsb_read_log_rows).  NULL / 0: no rows are recorded.
   * BSB_FLAG_NO_LOG_ROWS keeps the schedule and the per-lane row count but no
   * row store; BSB_FLAG_SCORE_SUMMARY folds every row into a score summary. */
  const int64_t* log_schedule;
  int64_t log_schedule_len;
} bsb_config;

/* bsb_config.flags */
#define BSB_FLAG_TRACK_EPISODES 1u /* keep the Logging-wrapper accumulators
                                      (wrappers.py:85-110) per lane on device */
/* Keep, per lane, the score summary of experiment `score_experiment` (see
 * bsb_read_score_summary): what its scoring rule reads of the rows, folded in
 * as each row falls due.  Needs a log schedule that is a prefix of that
 * experiment's own schedule, BSB_FLAG_TRACK_EPISODES, and an experiment of the
 * environment's family. */
#define BSB_FLAG_SCORE_SUMMARY 2u
/* With a log schedule: count the rows per lane but keep no row store (a
 * summary-only environment does not pay for the rows). */
#define BSB_FLAG_NO_LOG_ROWS 4u

/*
 * Caller-allocated outputs of one lock-step transition.  For bsb_rollout each
 * array carries a leading T axis.  Any pointer except `observation` may be
 * NULL (that output is then not written).
 *   observation : float32 [B, obs_numel]   fresh dense tensor every step
 *   reward      : float32 [B]   (float32 rounding of the float64 reward)
 *   reward_f64  : float64 [B]   (the reference's double-precision reward)
 *   discount    : float32 [B]   1 (MID) / 0 (LAST) / 0 (FIRST = None)
 *   step_type   : int32   [B]   bsb_step_type
 */
typedef struct bsb_outputs {
  float* observation;
  float* reward;
  double* reward_f64;
  float* discount;
  int32_t* step_type;
} bsb_outputs;

typedef struct bsb_env bsb_env; /* opaque handle */

int32_t bsb_abi_version(void);

/* Thread-local description of the last failure on the calling thread. */
const char* bsb_last_error(void);

/*
 * Replaces bsuite.load(name, kwargs) -> env constructor (bsuite/bsuite.py:93-98
 * and the constructors listed at bsb_family).  Creates `batch` lanes of one
 * environment; lane i has global id lane_offset + i (RNG keys depend on the
 * GLOBAL id only, so results are invariant to how lanes are sharded over GPUs).
 * Every lane starts with _reset_next_step = True (base.py:51-52) and performs
 * the constructor's RNG draws (memory_chain.py:49-50, umbrella_chain.py:55).
 * device >= 0: CUDA device ordinal; BSB_DEVICE_HOST: explicit host path.
 */
int32_t bsb_create(const bsb_config* config, int64_t batch, int32_t device,
                   uint64_t seed, uint64_t lane_offset, bsb_env** out);

int32_t bsb_destroy(bsb_env* env);

/* observation_spec() / action_spec() (e.g. deep_sea.py:146-151). */
int32_t bsb_obs_numel(const bsb_env* env, int64_t* numel);
int32_t bsb_obs_shape(const bsb_env* env, int32_t* rows, int32_t* cols);
int32_t bsb_num_actions(const bsb_env* env, int32_t* num_actions);
int32_t bsb_batch(const bsb_env* env, int64_t* batch);

/* base.Environment.reset (base.py:54-57; cartpole.py:118-128): every lane
 * starts a new episode and emits FIRST. */
int32_t bsb_reset(bsb_env* env, const bsb_outputs* out, void* stream);

/* base.Environment.step (base.py:59-65) for all lanes; actions int32 [B]. */
int32_t bsb_step(bsb_env* env, const int32_t* actions, const bsb_outputs* out,
                 void* stream);

/*
 * T consecutive step() calls fused in one launch, lane state held in
 * registers (replaces the inner loop of baselines/experiment.py:45-57).
 * actions: int32 [T,B], or NULL to sample uniform random actions on device
 * (the workload of baselines/random/agent.py:35-37) from the action stream
 * (action_seed, global lane, global step index) -- bsb_random_actions is its
 * host mirror.  actions_out (nullable) int32 [T,B] receives the actions used.
 * Outputs carry a leading T axis.
 */
int32_t bsb_rollout(bsb_env* env, int64_t num_steps, const int32_t* actions,
                    uint64_t action_seed, const bsb_outputs* out,
                    int32_t* actions_out, void* stream);

/* Host mirror of the on-device action sampler: out int32 [T,B] (host). */
int32_t bsb_random_actions(uint64_t action_seed, uint64_t lane_offset,
                           int64_t batch, int64_t first_step, int64_t num_steps,
                           int32_t num_actions, int32_t* out);

/* Number of step()/reset() calls made so far (global step index). */
int32_t bsb_steps_done(const bsb_env* env, int64_t* steps);

/*
 * bsuite_info() (e.g. deep_sea.py:153-155): per-lane accumulators.
 * bsb_info_count / bsb_info_name enumerate the keys of the reference dict;
 * bsb_read_info copies field `index` as float64 [B] into dst (same memory
 * space as the environment).
 */
int32_t bsb_info_count(const bsb_env* env, int32_t* count);
const char* bsb_info_name(const bsb_env* env, int32_t index);
int32_t bsb_read_info(bsb_env* env, int32_t index, double* dst, void* stream);

/*
 * Logging-wrapper accumulators (utils/wrappers.py:85-110), kept per lane when
 * BSB_FLAG_TRACK_EPISODES is set: field 0 steps, 1 episode, 2 total_return,
 * 3 episode_len, 4 episode_return; float64 [B] each.  episode_len and
 * episode_return are zeroed when the NEXT episode starts, so from a LAST
 * timestep (when the reference writes its row, :99-101) until the lane steps
 * again they hold the finished episode's values.
 */
int32_t bsb_read_episode_stats(bsb_env* env, int32_t field, double* dst,
                               void* stream);

/*
 * CUDA graphs.  bsb_step / bsb_reset / bsb_rollout / bsb_read_* / bsb_sum_episode_stats may be called on a stream
 * that is being captured.  A graph freezes launch arguments, so the first captured launch moves the handle's step
 * counter (it indexes the on-device action stream and the Logging columns) and its chunk scheduler into device
 * memory, for good: replays and eager calls can then be mixed in any order, and bsb_steps_done / bsb_get_state
 * synchronise the device to read the counter back.  Consecutive captured steps keep their programmatic dependent
 * launch (it becomes a programmatic graph edge; BSB_GRAPH_PDL=0 turns that off).
 * bsb_step_host (internal stream, host-side wait) cannot be captured.
 */

/*
 * Device-side reduction of the same five columns over the lanes of this
 * environment: dst[5] (same memory space as the environment) receives the SUMS
 * of steps, episode, total_return, episode_len, episode_return -- one small
 * kernel, so a log point costs a 40-byte read (or a 40-byte all-gather across
 * ranks) instead of five per-lane arrays.
 */
int32_t bsb_sum_episode_stats(bsb_env* env, double* dst5, void* stream);

/* The same reduction for `count` environments of one device in ONE kernel launch:
 * dst receives [count][5].  A log point of a whole sweep (bsuite/sweep.py:134-150:
 * 23 experiments) is then one launch and one all-gather. */
int32_t bsb_sum_episode_stats_many(bsb_env* const* envs, int32_t count,
                                   double* dst, void* stream);

/*
 * Per-lane log rows (see bsb_config.log_schedule): row k of lane i holds the
 * reference wrapper's columns steps, episode, total_return, episode_len,
 * episode_return followed by the bsuite_info() fields (bsb_info_name order) at
 * the LAST timestep that completed episode log_schedule[k] of that lane.
 * bsb_log_layout reports [n_points, n_columns]; bsb_read_log_rows copies
 * rows float64 [n_points][n_columns][B] and counts int32 [B] (rows recorded so
 * far per lane) into caller buffers in the environment's memory space.
 */
int32_t bsb_log_layout(const bsb_env* env, int32_t* n_points, int32_t* n_columns);
int32_t bsb_read_log_rows(bsb_env* env, double* rows, int32_t* counts, void* stream);

/*
 * Per-lane score summary (BSB_FLAG_SCORE_SUMMARY): float64 [BSB_SCORE_SUMMARY_FIELDS][B], field f of lane i at
 * summary[f * B + i], and counts int32 [B] (rows folded in so far per lane), copied into caller buffers in the
 * environment's memory space.  The fields, over the rows of the lane so far:
 *   last_episode, last_value   episode and value column (bsb_score_source.col_value) of the latest row
 *   prev_episode, prev_value   the same of the row before it (NaN while there is none)
 *   best                       running max of best_episode (cartpole, cartpole_swingup; NaN elsewhere)
 *   first_solved               deep_sea(_stochastic): episode of the first row at or past the experiment's first
 *                              scored episode with value / episode below its threshold (NaN until one)
 * Every field is NaN in a lane without rows.  Because a lane's rows are always a prefix of the log schedule,
 * these six values determine everything the experiment's scoring rule reads (bsb_scorer_* give the same bits
 * from them as from the rows).
 */
#define BSB_SCORE_SUMMARY_FIELDS 6
int32_t bsb_read_score_summary(bsb_env* env, double* summary, int32_t* counts, void* stream);

/* Flat snapshot of all lane state (checkpoint/resume; absent in the reference). */
int32_t bsb_state_bytes(const bsb_env* env, int64_t* nbytes);
int32_t bsb_get_state(bsb_env* env, void* dst_host, int64_t nbytes, void* stream);
int32_t bsb_set_state(bsb_env* env, const void* src_host, int64_t nbytes,
                      void* stream);

/*
 * Host-buffer convenience for FFI callers without a device allocator: takes
 * `actions` (host, int32 [B]), steps, and delivers the requested outputs into
 * HOST buffers (`host_out`; NULL members are skipped, so an agent that consumes
 * observations on the device passes observation = NULL and supplies
 * `device_obs`, a device pointer that receives them).  Synchronous for the
 * host outputs: on return they have landed (for `device_obs` see
 * BSB_HOST_FENCE_CALLER).  This
 * is the call pattern of the reference's agent loop, one env.step(action) per
 * decision (baselines/experiment.py:45-57).
 *
 * When `actions` and the requested scalar outputs are PINNED host memory the
 * kernel accesses them in place over PCIe (zero-copy: no separate H2D / D2H
 * copies) and signals completion through a pinned mailbox word the host spins
 * on (no stream synchronise; BSB_HOST_SPIN=0 restores it); pageable buffers
 * take the staged-copy path.  Host actions are range-checked: an action outside
 * [0, num_actions) yields BSB_INVALID_ARGUMENT (the reference raises IndexError,
 * e.g. bandit.py:61).
 *
 * flags
 *   BSB_HOST_ORDER_AFTER_STREAM  work enqueued EARLIER on this handle through
 *       bsb_reset / bsb_step / bsb_rollout on `caller_stream` is waited for (on
 *       the device) before the step runs.  Without the flag the caller must
 *       have synchronised that stream: the step runs on a stream the handle owns.
 *   BSB_HOST_FENCE_CALLER  deep_sea from size 16 up (its observation is a function
 *       of the lane state and dwarfs the scalar traffic) runs host steps in two
 *       phases: the transitions of all lanes first (scalars staged on the device
 *       and shipped to the host by a few copier blocks), then the observation
 *       stream.  The call returns as soon as the scalars have landed -- the agent
 *       decides its next action while the observations are still being written.  With this flag `caller_stream`
 *       is fenced (on the device) behind the step, so work enqueued there
 *       afterwards sees complete observations; without it, order a consumer by
 *       the next call on this handle (every entry point waits for the step) or
 *       set BSB_HOST_EARLY=0 to make the call wait for the whole kernel.
 *   BSB_HOST_PRELAUNCH  (pinned buffers only) after ringing this step, the NEXT
 *       step's kernel is enqueued at once; it becomes resident as this one drains
 *       and polls the mailbox doorbell, so the next call costs neither a launch
 *       nor a wake-up -- for agents whose policy runs on the HOST.  While it
 *       waits it occupies the SMs: other GPU work of the process queues behind it
 *       until the next call, bsb_host_flush, or BSB_DOORBELL_TIMEOUT_MS (default
 *       200) without a ring, after which it stands down by itself.  Every other
 *       entry point of this handle stands it down first.
 *   BSB_HOST_NO_WAIT  (pinned buffers; otherwise the call is simply synchronous)
 *       the call returns once the step is enqueued; the host outputs are valid
 *       after bsb_host_wait(env).  One step per handle may be outstanding (any
 *       entry point of the handle collects it first).  The use: split the lanes
 *       over TWO handles (bsb_create's lane_offset keeps the lanes' random streams
 *       those of one big batch) and alternate -- while one half's scalars cross
 *       PCIe and its agent decides, the other half's kernel has the GPU, so each
 *       half remains the reference's strict loop (act on what the previous step
 *       returned) and the GPU is not left idle in between (two to four handles;
 *       three measured best on a B200).  Pass BSB_HOST_FENCE_CALLER with it: the
 *       loop measured 1.5x slower without the fence's event record between a
 *       handle's observation launch and its next launch.  Not with
 *       BSB_HOST_PRELAUNCH.
 */
#define BSB_HOST_ORDER_AFTER_STREAM 1u
#define BSB_HOST_PRELAUNCH 2u
#define BSB_HOST_FENCE_CALLER 4u
#define BSB_HOST_NO_WAIT 8u
int32_t bsb_step_host(bsb_env* env, const int32_t* actions,
                      const bsb_outputs* host_out, float* device_obs,
                      void* caller_stream, uint32_t flags);

/* Stands down a launch queued by BSB_HOST_PRELAUNCH (no-op otherwise). */
int32_t bsb_host_flush(bsb_env* env);

/* Completes a step issued with BSB_HOST_NO_WAIT: returns when its host outputs
 * have landed (no-op when nothing is outstanding).  Reports an out-of-range
 * action of that step as BSB_INVALID_ARGUMENT, like the synchronous call. */
int32_t bsb_host_wait(bsb_env* env);

/* Diagnostics (BSB_HOST_TIMING=1): %globaltimer stamps, in ns, the latest two-phase
 * host step left in the mailbox: [0] kernel past its dependency wait, [1] phase 1
 * complete, [2] scalars fenced, [3] latest block exit of the previous launch. */
int32_t bsb_host_timing(bsb_env* env, uint64_t* stamps8);

/*
 * Out-of-range actions.  Host-resident actions (host environments,
 * bsb_step_host) are validated before anything moves.  Device-resident action
 * tensors cannot be inspected without a synchronise: the kernels clamp such an
 * action into [0, num_actions) before it indexes a table or is packed into lane
 * state, and raise a flag.  *seen receives the flag (1 = some action since the
 * last call was out of range) and clears it; synchronise the stream first.
 */
int32_t bsb_invalid_actions(bsb_env* env, int32_t* seen);

/*
 * Multi-GPU log points without torch.distributed (SURVEY.md 8e: "one collective:
 * ncclAllGather of a per-rank stats block at log points only").  One process per
 * GPU; rank 0 calls bsb_comm_unique_id and shares the 128 bytes out of band (a
 * file, a socket, MPI, torch's store), every rank calls bsb_comm_create.  NCCL is
 * loaded at run time (BSB_NCCL_LIBRARY, else libnccl.so.2): single-GPU callers
 * never need it.
 *
 * bsb_log_point: the Logging sums of `count` environments of this rank are
 * reduced by ONE kernel on `stream` into local [count][5] and all-gathered into
 * gathered [world][count][5] on a side stream the communicator owns, fenced by
 * events -- `stream` is free to run the next steps at once (the reference writes
 * log rows at log-spaced episodes only: utils/wrappers.py:99-110).  local and
 * gathered are caller-owned device buffers that must stay valid until
 * bsb_comm_wait(comm, s), which makes stream `s` wait (on the device) for the
 * latest gather.  Replaces the process pool's result collection of
 * bsuite/baselines/utils/pool.py:28-54.
 */
#define BSB_COMM_ID_BYTES 128
typedef struct bsb_comm bsb_comm;
int32_t bsb_comm_unique_id(uint8_t* id /* [BSB_COMM_ID_BYTES] */);
int32_t bsb_comm_create(const uint8_t* id, int32_t rank, int32_t world,
                        int32_t device, bsb_comm** out);
int32_t bsb_comm_destroy(bsb_comm* comm);
int32_t bsb_comm_world(const bsb_comm* comm, int32_t* rank, int32_t* world);
int32_t bsb_log_point(bsb_comm* comm, bsb_env* const* envs, int32_t count,
                      double* local, double* gathered, void* stream);
int32_t bsb_comm_wait(bsb_comm* comm, void* stream);

/*
 * Scores (experiments/<name>/analysis.py::score, experiments/summary_analysis.py::bsuite_score and
 * ave_score_by_tag) computed from the per-lane log rows, without the rows leaving the device.
 *
 * Every lane is one run of the bsuite: lane j's score for an experiment is what the reference's score(df) returns
 * for the DataFrame holding lane j's rows of that experiment's ids (with the sweep metadata joined), i.e. what
 * csv_load.load_bsuite would read back from lane j's CSV files.  Only the ids given to the scorer count.  A lane
 * with no row of an experiment has that experiment "not scored": score NaN, finished 0.  A tag average is the
 * NaN-skipping mean over the experiments carrying the tag (NaN when there is none).
 *
 * bsb_experiment is the reference's registration order (bsuite/sweep.py); bsb_tag is the tag names sorted.
 */
typedef enum bsb_experiment {
  BSB_EXP_BANDIT = 0, BSB_EXP_BANDIT_NOISE = 1, BSB_EXP_BANDIT_SCALE = 2,
  BSB_EXP_CARTPOLE = 3, BSB_EXP_CARTPOLE_NOISE = 4, BSB_EXP_CARTPOLE_SCALE = 5, BSB_EXP_CARTPOLE_SWINGUP = 6,
  BSB_EXP_CATCH = 7, BSB_EXP_CATCH_NOISE = 8, BSB_EXP_CATCH_SCALE = 9,
  BSB_EXP_DEEP_SEA = 10, BSB_EXP_DEEP_SEA_STOCHASTIC = 11, BSB_EXP_DISCOUNTING_CHAIN = 12,
  BSB_EXP_MEMORY_LEN = 13, BSB_EXP_MEMORY_SIZE = 14,
  BSB_EXP_MNIST = 15, BSB_EXP_MNIST_NOISE = 16, BSB_EXP_MNIST_SCALE = 17,
  BSB_EXP_MOUNTAIN_CAR = 18, BSB_EXP_MOUNTAIN_CAR_NOISE = 19, BSB_EXP_MOUNTAIN_CAR_SCALE = 20,
  BSB_EXP_UMBRELLA_DISTRACT = 21, BSB_EXP_UMBRELLA_LENGTH = 22,
  BSB_NUM_EXPERIMENTS = 23
} bsb_experiment;

typedef enum bsb_tag {
  BSB_TAG_BASIC = 0, BSB_TAG_CREDIT_ASSIGNMENT = 1, BSB_TAG_EXPLORATION = 2, BSB_TAG_GENERALIZATION = 3,
  BSB_TAG_MEMORY = 4, BSB_TAG_NOISE = 5, BSB_TAG_SCALE = 6,
  BSB_NUM_TAGS = 7
} bsb_tag;

/* "bandit", "bandit_noise", ... / "basic", "credit_assignment", ...; NULL when out of range. */
const char* bsb_experiment_name(int32_t experiment);
const char* bsb_tag_name(int32_t tag);

/*
 * The rows of one bsuite_id, in the layout of bsb_read_log_rows: rows float64 [n_points][n_columns][batch] and
 * counts int32 [batch], in the memory space of `device`, ascending in episode within a lane.  Column indices name
 * what the experiment's rule reads: col_episode always; col_value the experiment's regret-like column
 * (total_regret for bandit / catch / mnist / umbrella, raw_return for cartpole / mountain_car, total_return for
 * cartpole_swingup / discounting_chain, total_bad_episodes for deep_sea, total_perfect for memory); col_best
 * best_episode for cartpole and cartpole_swingup (-1 elsewhere).  group_key is the sweep setting the rule groups
 * by: noise_scale / reward_scale (the _noise / _scale experiments), height_threshold (cartpole_swingup), size
 * (deep_sea), memory_length / num_bits (memory_len / memory_size), n_distractor / chain_length (umbrella_distract /
 * umbrella_length); ignored by the other experiments.
 *
 * layout BSB_SCORE_ROWS (0, the value of a zeroed struct) describes rows as above.  layout BSB_SCORE_SUMMARY
 * describes a score summary (bsb_read_score_summary, bsb_score_summarize): rows float64
 * [BSB_SCORE_SUMMARY_FIELDS][batch], counts the rows folded in per lane, n_columns BSB_SCORE_SUMMARY_FIELDS,
 * n_points the length of the log schedule; the col_* fields are not read.
 */
#define BSB_SCORE_ROWS 0
#define BSB_SCORE_SUMMARY 1
typedef struct bsb_score_source {
  int32_t experiment;    /* bsb_experiment */
  int32_t device;        /* BSB_DEVICE_HOST or CUDA ordinal */
  int64_t batch;
  int32_t n_points, n_columns;
  int32_t col_episode, col_value, col_best;
  int32_t layout;        /* BSB_SCORE_ROWS or BSB_SCORE_SUMMARY */
  double group_key;
  const double* rows;
  const int32_t* counts;
} bsb_score_source;

/* Fills `out` with the row store of a record-rows environment (created with a log schedule): no copy, the scorer
 * reads the environment's own rows, so the environment must outlive every scorer built from it.  An environment
 * that keeps a score summary and no rows gives a BSB_SCORE_SUMMARY source over its summary instead (`experiment`
 * must then be the one the summary is kept for).  Fails when the environment records neither, or its family does
 * not run `experiment`. */
int32_t bsb_score_source_from_env(const bsb_env* env, int32_t experiment, double group_key, bsb_score_source* out);

/* Host only: folds caller-owned host rows (a BSB_SCORE_ROWS source on BSB_DEVICE_HOST) into a score summary,
 * summary float64 [BSB_SCORE_SUMMARY_FIELDS][batch] and counts int32 [batch] (host buffers), with the fold the
 * engine applies as rows fall due.  Fails when a lane's episode column is not a prefix of the experiment's log
 * schedule (the summary is exact only for such rows). */
int32_t bsb_score_summarize(const bsb_score_source* rows_source, double* summary, int32_t* counts);

/*
 * A scorer is built once (the inputs are validated and a descriptor table is uploaded) and run many times.
 * Every source must have `batch` lanes on `device`; at most 128 sources per experiment, n_points <= 4096.
 * Sources of both layouts may be mixed; a summary scores exactly as the rows it was folded from.
 * bsb_scorer_run writes scores float64 [BSB_NUM_EXPERIMENTS][batch], finished int32 [BSB_NUM_EXPERIMENTS][batch]
 * (the reference's _is_finished) and tags float64 [BSB_NUM_TAGS][batch], all in the memory space of `device`.
 * On CUDA it is ONE kernel launch on `stream`, with no allocation and no synchronisation, so it may be captured
 * into a CUDA graph; it reads the rows as they are when the launch runs.  On BSB_DEVICE_HOST the same rules run
 * in a host loop.  Calls on one scorer are not thread-safe.
 */
typedef struct bsb_scorer bsb_scorer;
int32_t bsb_scorer_create(const bsb_score_source* sources, int32_t count, int64_t batch, int32_t device,
                          bsb_scorer** out);
int32_t bsb_scorer_run(bsb_scorer* scorer, double* scores, int32_t* finished, double* tags, void* stream);
int32_t bsb_scorer_destroy(bsb_scorer* scorer);

/* Number of kernels this library has launched in this process (bench evidence). */
int64_t bsb_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* BSUITE_B200_H_ */
