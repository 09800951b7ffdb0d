// Scorer objects of the C ABI (bsb_scorer_*, bsb_score_source_from_env) and the scoring kernel.
//
// The kernel runs a whole sweep in ONE launch: a CTA holds 32 consecutive lanes x BSB_NUM_EXPERIMENTS warps, warp
// e scores experiment e for its 32 lanes (so every row read is one coalesced 256-byte line across the warp), the
// scores meet in shared memory and the first BSB_NUM_TAGS warps average them by tag.  The rules are the
// __host__ __device__ functions of bsb_scoring.cuh, which the host path runs in a plain loop.
#include <algorithm>
#include <cstring>
#include <string>
#include <vector>

#include "bsb_env.h"
#include "bsb_scoring.cuh"

using namespace bsb;
using namespace bsb::scoring;

namespace {

constexpr int kLanesPerCta = 32;

const char* const kExperimentNames[BSB_NUM_EXPERIMENTS] = {
    "bandit", "bandit_noise", "bandit_scale", "cartpole", "cartpole_noise", "cartpole_scale", "cartpole_swingup",
    "catch", "catch_noise", "catch_scale", "deep_sea", "deep_sea_stochastic", "discounting_chain", "memory_len",
    "memory_size", "mnist", "mnist_noise", "mnist_scale", "mountain_car", "mountain_car_noise",
    "mountain_car_scale", "umbrella_distract", "umbrella_length"};
const char* const kTagNames[BSB_NUM_TAGS] = {"basic", "credit_assignment", "exploration", "generalization",
                                             "memory", "noise", "scale"};

// The family whose environments an experiment runs (bsb_score_source_from_env checks it).
int experiment_family(int e) {
  switch (exp_info(e).rule) {
    case kRegret: return e <= BSB_EXP_BANDIT_SCALE ? BSB_BANDIT : BSB_CATCH;
    case kCartpole: return BSB_CARTPOLE;
    case kSwingup: return BSB_CARTPOLE_SWINGUP;
    case kMountainCar: return BSB_MOUNTAIN_CAR;
    case kMnist: return BSB_MNIST;
    case kDeepSea: return BSB_DEEP_SEA;
    case kDiscounting: return BSB_DISCOUNTING_CHAIN;
    case kMemory: return BSB_MEMORY_CHAIN;
    case kUmbrella: return BSB_UMBRELLA_CHAIN;
  }
  return -1;
}

// The info column holding an experiment's col_value (nullptr: one of the five standard columns, see below).
const char* value_column(int e) {
  switch (exp_info(e).rule) {
    case kCartpole:
    case kMountainCar: return "raw_return";
    case kDeepSea: return "total_bad_episodes";
    case kMemory: return "total_perfect";
    case kSwingup:
    case kDiscounting: return nullptr;      // total_return
  }
  return "total_regret";
}

// The reference Logging wrapper's schedule (wrappers.py:140-147), as recording.log_schedule computes it: the
// episode counts in [1, NUM_EPISODES] equal to {1, 1.2, 1.4, 1.7, 2, 2.5, 3, 4, ..., 10} x 10^k.
std::vector<int64_t> experiment_schedule(int e) {
  static const double kRatios[] = {1., 1.2, 1.4, 1.7, 2., 2.5, 3., 4., 5., 6., 7., 8., 9., 10.};
  std::vector<int64_t> out;
  const int64_t n = (int64_t)exp_info(e).num_episodes;
  for (int64_t count = 1; count <= n; ++count) {
    const double scale = pow(10.0, floor(log10((double)count)));
    for (double r : kRatios)
      if ((double)count == scale * r) { out.push_back(count); break; }
  }
  return out;
}

__global__ void __launch_bounds__(kLanesPerCta * BSB_NUM_EXPERIMENTS)
score_kernel(const ScoreDesc* __restrict__ descs, const ScoreExp* __restrict__ exps, int64_t B,
             double* __restrict__ scores, int32_t* __restrict__ finished, double* __restrict__ tags) {
  __shared__ double s_score[BSB_NUM_EXPERIMENTS][kLanesPerCta];
  __shared__ int32_t s_present[BSB_NUM_EXPERIMENTS][kLanesPerCta];
  const int e = threadIdx.y, x = threadIdx.x;
  const int64_t lane = (int64_t)blockIdx.x * kLanesPerCta + x;
  if (lane < B) {
    const ScoreOut o = score_lane(descs, exps[e], e, lane, B);
    scores[(int64_t)e * B + lane] = o.score;
    finished[(int64_t)e * B + lane] = o.finished;
    s_score[e][x] = o.score;
    s_present[e][x] = o.present;
  }
  __syncthreads();
  if (e < BSB_NUM_TAGS && lane < B)
    tags[(int64_t)e * B + lane] = tag_average(e, &s_score[0][x], &s_present[0][x], kLanesPerCta);
}

}  // namespace

namespace bsb {

int check_score_summary(const bsb_config& c) {
  const int e = c.score_experiment;
  if (e < 0 || e >= BSB_NUM_EXPERIMENTS) return fail(BSB_INVALID_ARGUMENT, "unknown score_experiment " + std::to_string(e));
  if (c.family != experiment_family(e))
    return fail(BSB_INVALID_ARGUMENT, std::string("the environment's family does not run experiment ") + kExperimentNames[e]);
  const std::vector<int64_t> sched = experiment_schedule(e);
  if ((size_t)c.log_schedule_len > sched.size() || !std::equal(c.log_schedule, c.log_schedule + c.log_schedule_len, sched.begin()))
    return fail(BSB_INVALID_ARGUMENT, std::string("a score summary needs a log schedule that is a prefix of ") +
                                          kExperimentNames[e] + "'s (episodes up to " + std::to_string(sched.back()) + ")");
  return BSB_OK;
}

void score_summary_columns(int e, const InfoNames& names, int32_t* col_value, int32_t* col_best) {
  const char* want = value_column(e);
  *col_value = want ? -1 : 2;                              // total_return
  *col_best = -1;
  for (int k = 0; k < names.n; ++k) {
    if (want && strcmp(names.names[k], want) == 0) *col_value = 5 + k;
    if (rule_needs_best(exp_info(e).rule) && strcmp(names.names[k], "best_episode") == 0) *col_best = 5 + k;
  }
}

}  // namespace bsb

struct bsb_scorer {
  int device;
  int64_t batch;
  std::vector<ScoreDesc> descs;        // sorted by experiment (and group key where the rule groups)
  ScoreExp exps[BSB_NUM_EXPERIMENTS];
  void* table;                         // device copy: descs, then exps
};

namespace {

// The checks a source passes before it is folded or scored (`at` prefixes the message).
int check_source(const bsb_score_source& s, const std::string& at) {
  if (s.experiment < 0 || s.experiment >= BSB_NUM_EXPERIMENTS)
    return fail(BSB_INVALID_ARGUMENT, at + "unknown experiment " + std::to_string(s.experiment));
  const ExpInfo info = exp_info(s.experiment);
  if (s.layout != BSB_SCORE_ROWS && s.layout != BSB_SCORE_SUMMARY)
    return fail(BSB_INVALID_ARGUMENT, at + "unknown layout " + std::to_string(s.layout));
  if (s.batch <= 0) return fail(BSB_INVALID_ARGUMENT, at + "batch must be positive");
  if (!s.rows || !s.counts) return fail(BSB_INVALID_ARGUMENT, at + "null rows or counts");
  if (s.n_points < 1 || s.n_points > kMaxPoints) return fail(BSB_INVALID_ARGUMENT, at + "n_points must be in [1, 4096]");
  if (s.layout == BSB_SCORE_SUMMARY) {
    if (s.n_columns != BSB_SCORE_SUMMARY_FIELDS)
      return fail(BSB_INVALID_ARGUMENT, at + "a score summary has n_columns = " + std::to_string(BSB_SCORE_SUMMARY_FIELDS) + " fields, not " + std::to_string(s.n_columns));
  } else {
    if (s.n_columns < 1) return fail(BSB_INVALID_ARGUMENT, at + "n_columns must be positive");
    auto has = [&](int32_t c) { return c >= 0 && c < s.n_columns; };
    if (!has(s.col_episode)) return fail(BSB_INVALID_ARGUMENT, at + "missing column: episode");
    if (!has(s.col_value)) {
      const char* name = value_column(s.experiment);
      return fail(BSB_INVALID_ARGUMENT, at + "missing column: " + (name ? name : "total_return") + " (" + kExperimentNames[s.experiment] + ")");
    }
    if (rule_needs_best(info.rule) && !has(s.col_best))
      return fail(BSB_INVALID_ARGUMENT, at + "missing column: best_episode (" + kExperimentNames[s.experiment] + ")");
  }
  if (info.grouped && !(s.group_key == s.group_key))
    return fail(BSB_INVALID_ARGUMENT, at + "group_key is NaN (" + kExperimentNames[s.experiment] + " groups by it)");
  return BSB_OK;
}

}  // namespace

extern "C" {

const char* bsb_experiment_name(int32_t experiment) {
  return experiment >= 0 && experiment < BSB_NUM_EXPERIMENTS ? kExperimentNames[experiment] : nullptr;
}

const char* bsb_tag_name(int32_t tag) { return tag >= 0 && tag < BSB_NUM_TAGS ? kTagNames[tag] : nullptr; }

int32_t bsb_score_source_from_env(const bsb_env* env, int32_t experiment, double group_key, bsb_score_source* out) {
  if (!env || !out) return fail(BSB_INVALID_ARGUMENT, "null argument");
  if (experiment < 0 || experiment >= BSB_NUM_EXPERIMENTS)
    return fail(BSB_INVALID_ARGUMENT, "unknown experiment " + std::to_string(experiment));
  if (!env->p.log_next) return fail(BSB_INVALID_ARGUMENT, "environment was created without a log schedule (no rows to score)");
  if (!env->p.log_rows && !env->p.score_sum)
    return fail(BSB_INVALID_ARGUMENT, "environment keeps neither log rows nor a score summary (BSB_FLAG_NO_LOG_ROWS without BSB_FLAG_SCORE_SUMMARY)");
  if (env->p.family != experiment_family(experiment))
    return fail(BSB_INVALID_ARGUMENT, std::string("the environment's family does not run experiment ") + kExperimentNames[experiment]);
  bsb_score_source s;
  memset(&s, 0, sizeof(s));
  s.experiment = experiment; s.device = env->device; s.batch = env->p.batch;
  s.n_points = env->p.n_log_points;
  s.group_key = group_key;
  s.counts = env->p.log_next;
  if (!env->p.log_rows) {
    if (env->p.score_exp != experiment)
      return fail(BSB_INVALID_ARGUMENT, std::string("the environment keeps the score summary of ") + kExperimentNames[env->p.score_exp] +
                                            ", not of " + kExperimentNames[experiment]);
    s.layout = BSB_SCORE_SUMMARY; s.n_columns = BSB_SCORE_SUMMARY_FIELDS;
    s.col_episode = s.col_value = s.col_best = -1;
    s.rows = env->p.score_sum;
    *out = s;
    return BSB_OK;
  }
  s.layout = BSB_SCORE_ROWS; s.n_columns = 5 + env->names.n;
  s.col_episode = 1;
  score_summary_columns(experiment, env->names, &s.col_value, &s.col_best);
  s.rows = env->p.log_rows;
  *out = s;
  return BSB_OK;
}

int32_t bsb_score_summarize(const bsb_score_source* src, double* summary, int32_t* counts) {
  if (!src || !summary || !counts) return fail(BSB_INVALID_ARGUMENT, "null argument");
  const bsb_score_source& s = *src;
  if (s.layout != BSB_SCORE_ROWS) return fail(BSB_INVALID_ARGUMENT, "bsb_score_summarize folds a BSB_SCORE_ROWS source");
  if (s.device != BSB_DEVICE_HOST) return fail(BSB_INVALID_ARGUMENT, "bsb_score_summarize reads host rows (device BSB_DEVICE_HOST)");
  { int rc = check_source(s, ""); if (rc != BSB_OK) return rc; }
  const std::vector<int64_t> sched = experiment_schedule(s.experiment);
  const int64_t B = s.batch;
  const bool best = rule_needs_best(exp_info(s.experiment).rule);
  for (int64_t i = 0; i < (int64_t)BSB_SCORE_SUMMARY_FIELDS * B; ++i) summary[i] = NAN;
  for (int64_t lane = 0; lane < B; ++lane) {
    const int32_t c = s.counts[lane] < 0 ? 0 : (s.counts[lane] > s.n_points ? s.n_points : s.counts[lane]);
    auto at = [&](int32_t k, int32_t col) { return s.rows[((int64_t)k * s.n_columns + col) * B + lane]; };
    for (int32_t k = 0; k < c; ++k)
      if ((size_t)k >= sched.size() || at(k, s.col_episode) != (double)sched[(size_t)k])
        return fail(BSB_INVALID_ARGUMENT, "lane " + std::to_string(lane) + ": row " + std::to_string(k) +
                                              " is not at episode " + ((size_t)k < sched.size() ? std::to_string(sched[(size_t)k]) : std::string("<none>")) +
                                              " of " + kExperimentNames[s.experiment] + "'s log schedule (the rows must be a prefix of it)");
    for (int32_t k = 0; k < c; ++k)
      fold_row(summary, lane, B, s.experiment, k, at(k, s.col_episode), at(k, s.col_value), best ? at(k, s.col_best) : NAN);
    counts[lane] = c;
  }
  return BSB_OK;
}

int32_t bsb_scorer_create(const bsb_score_source* sources, int32_t count, int64_t batch, int32_t device,
                          bsb_scorer** out) {
  if (!out) return fail(BSB_INVALID_ARGUMENT, "null argument");
  *out = nullptr;
  if (!sources || count <= 0) return fail(BSB_INVALID_ARGUMENT, "a scorer needs at least one source");
  if (batch <= 0) return fail(BSB_INVALID_ARGUMENT, "batch must be positive");
  if (device < BSB_DEVICE_HOST) return fail(BSB_INVALID_ARGUMENT, "device must be >= 0 or BSB_DEVICE_HOST");
  int per_exp[BSB_NUM_EXPERIMENTS] = {0};
  for (int32_t i = 0; i < count; ++i) {
    const bsb_score_source& s = sources[i];
    const std::string at = "source " + std::to_string(i) + ": ";
    int rc = check_source(s, at);
    if (rc != BSB_OK) return rc;
    if (s.batch != batch) return fail(BSB_INVALID_ARGUMENT, at + "batch " + std::to_string(s.batch) + " differs from the scorer's " + std::to_string(batch));
    if (s.device != device) return fail(BSB_INVALID_ARGUMENT, at + "lives on another device than the scorer");
    if (++per_exp[s.experiment] > kMaxSourcesPerExperiment)
      return fail(BSB_INVALID_ARGUMENT, std::string("more than 128 sources for experiment ") + kExperimentNames[s.experiment]);
  }
  if (device >= 0) {
    int n_dev = 0;
    cudaError_t err = cudaGetDeviceCount(&n_dev);
    if (err != cudaSuccess || n_dev == 0)
      return fail(BSB_CUDA_ERROR, std::string("no CUDA device available (") + cudaGetErrorString(err) + ")");
    if (device >= n_dev) return fail(BSB_INVALID_ARGUMENT, "device ordinal out of range");
  }
  std::vector<int32_t> order(count);
  for (int32_t i = 0; i < count; ++i) order[i] = i;
  std::stable_sort(order.begin(), order.end(), [&](int32_t a, int32_t b) {
    const bsb_score_source &x = sources[a], &y = sources[b];
    if (x.experiment != y.experiment) return x.experiment < y.experiment;
    return exp_info(x.experiment).grouped && x.group_key < y.group_key;    // groupby sorts its keys
  });
  bsb_scorer* sc = new bsb_scorer();
  sc->device = device; sc->batch = batch; sc->table = nullptr;
  for (int e = 0; e < BSB_NUM_EXPERIMENTS; ++e) sc->exps[e] = ScoreExp{0, 0, kViewRows, 0};
  for (int32_t i : order) {
    const bsb_score_source& s = sources[i];
    ScoreDesc d;
    d.rows = s.rows; d.counts = s.counts; d.n_points = s.n_points; d.n_columns = s.n_columns;
    d.col_episode = s.col_episode; d.col_value = s.col_value; d.col_best = s.col_best; d.layout = s.layout;
    d.key = s.group_key;
    ScoreExp& ex = sc->exps[s.experiment];
    const int32_t view = s.layout == BSB_SCORE_SUMMARY ? kViewSummary : kViewRows;
    if (ex.count == 0) { ex.first = (int32_t)sc->descs.size(); ex.view = view; }
    else if (ex.view != view) ex.view = kViewMixed;
    ++ex.count;
    sc->descs.push_back(d);
  }
  if (device >= 0) {
    int prev = 0;
    cudaGetDevice(&prev);
    cudaSetDevice(device);
    const size_t desc_bytes = sc->descs.size() * sizeof(ScoreDesc), exp_bytes = sizeof(sc->exps);
    cudaError_t err = cudaMalloc(&sc->table, desc_bytes + exp_bytes);
    if (err == cudaSuccess) err = cudaMemcpy(sc->table, sc->descs.data(), desc_bytes, cudaMemcpyHostToDevice);
    if (err == cudaSuccess) err = cudaMemcpy(static_cast<char*>(sc->table) + desc_bytes, sc->exps, exp_bytes, cudaMemcpyHostToDevice);
    cudaSetDevice(prev);
    if (err != cudaSuccess) {
      if (sc->table) cudaFree(sc->table);
      delete sc;
      return fail(err == cudaErrorMemoryAllocation ? BSB_OUT_OF_MEMORY : BSB_CUDA_ERROR,
                  std::string("scorer descriptor upload: ") + cudaGetErrorString(err));
    }
  }
  *out = sc;
  return BSB_OK;
}

int32_t bsb_scorer_run(bsb_scorer* sc, double* scores, int32_t* finished, double* tags, void* stream) {
  if (!sc || !scores || !finished || !tags) return fail(BSB_INVALID_ARGUMENT, "null argument");
  const int64_t B = sc->batch;
  if (sc->device >= 0) {
    int prev = 0;
    cudaGetDevice(&prev);
    cudaSetDevice(sc->device);
    const ScoreDesc* descs = static_cast<const ScoreDesc*>(sc->table);
    const ScoreExp* exps = reinterpret_cast<const ScoreExp*>(descs + sc->descs.size());
    const unsigned blocks = (unsigned)((B + kLanesPerCta - 1) / kLanesPerCta);
    score_kernel<<<blocks, dim3(kLanesPerCta, BSB_NUM_EXPERIMENTS), 0, static_cast<cudaStream_t>(stream)>>>(
        descs, exps, B, scores, finished, tags);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    const cudaError_t err = cudaGetLastError();
    cudaSetDevice(prev);
    if (err != cudaSuccess) return fail(BSB_CUDA_ERROR, std::string("score kernel: ") + cudaGetErrorString(err));
    return BSB_OK;
  }
  double lane_scores[BSB_NUM_EXPERIMENTS];
  int32_t present[BSB_NUM_EXPERIMENTS];
  for (int64_t lane = 0; lane < B; ++lane) {
    for (int e = 0; e < BSB_NUM_EXPERIMENTS; ++e) {
      const ScoreOut o = score_lane(sc->descs.data(), sc->exps[e], e, lane, B);
      scores[(int64_t)e * B + lane] = o.score;
      finished[(int64_t)e * B + lane] = o.finished;
      lane_scores[e] = o.score;
      present[e] = o.present;
    }
    for (int t = 0; t < BSB_NUM_TAGS; ++t) tags[(int64_t)t * B + lane] = tag_average(t, lane_scores, present, 1);
  }
  return BSB_OK;
}

int32_t bsb_scorer_destroy(bsb_scorer* sc) {
  if (!sc) return BSB_OK;
  if (sc->table) {
    int prev = 0;
    cudaGetDevice(&prev);
    cudaSetDevice(sc->device);
    cudaFree(sc->table);
    cudaSetDevice(prev);
  }
  delete sc;
  return BSB_OK;
}

}  // extern "C"
