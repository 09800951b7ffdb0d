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

struct bsb_scorer {
  int device;
  int64_t batch;
  std::vector<ScoreDesc> descs;        // sorted by experiment (and group key where the rule groups)
  ScoreExp exps[BSB_NUM_EXPERIMENTS];
  void* table;                         // device copy: descs, then exps
};

extern "C" {

const char* bsb_experiment_name(int32_t experiment) {
  return experiment >= 0 && experiment < BSB_NUM_EXPERIMENTS ? kExperimentNames[experiment] : nullptr;
}

const char* bsb_tag_name(int32_t tag) { return tag >= 0 && tag < BSB_NUM_TAGS ? kTagNames[tag] : nullptr; }

int32_t bsb_score_source_from_env(const bsb_env* env, int32_t experiment, double group_key, bsb_score_source* out) {
  if (!env || !out) return fail(BSB_INVALID_ARGUMENT, "null argument");
  if (experiment < 0 || experiment >= BSB_NUM_EXPERIMENTS)
    return fail(BSB_INVALID_ARGUMENT, "unknown experiment " + std::to_string(experiment));
  if (!env->p.log_rows) return fail(BSB_INVALID_ARGUMENT, "environment was created without a log schedule (no rows to score)");
  if (env->p.family != experiment_family(experiment))
    return fail(BSB_INVALID_ARGUMENT, std::string("the environment's family does not run experiment ") + kExperimentNames[experiment]);
  bsb_score_source s;
  memset(&s, 0, sizeof(s));
  s.experiment = experiment; s.device = env->device; s.batch = env->p.batch;
  s.n_points = env->p.n_log_points; s.n_columns = 5 + env->names.n;
  s.col_episode = 1; s.col_value = -1; s.col_best = -1;
  const char* want = value_column(experiment);
  for (int k = 0; k < env->names.n; ++k) {
    if (want && strcmp(env->names.names[k], want) == 0) s.col_value = 5 + k;
    if (rule_needs_best(exp_info(experiment).rule) && strcmp(env->names.names[k], "best_episode") == 0) s.col_best = 5 + k;
  }
  if (!want) s.col_value = 2;                              // total_return
  s.group_key = group_key;
  s.rows = env->p.log_rows; s.counts = env->p.log_next;
  *out = s;
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
    if (s.experiment < 0 || s.experiment >= BSB_NUM_EXPERIMENTS)
      return fail(BSB_INVALID_ARGUMENT, at + "unknown experiment " + std::to_string(s.experiment));
    const ExpInfo info = exp_info(s.experiment);
    if (s.batch != batch) return fail(BSB_INVALID_ARGUMENT, at + "batch " + std::to_string(s.batch) + " differs from the scorer's " + std::to_string(batch));
    if (s.device != device) return fail(BSB_INVALID_ARGUMENT, at + "lives on another device than the scorer");
    if (!s.rows || !s.counts) return fail(BSB_INVALID_ARGUMENT, at + "null rows or counts");
    if (s.n_points < 1 || s.n_points > kMaxPoints) return fail(BSB_INVALID_ARGUMENT, at + "n_points must be in [1, 4096]");
    if (s.n_columns < 1) return fail(BSB_INVALID_ARGUMENT, at + "n_columns must be positive");
    auto has = [&](int32_t c) { return c >= 0 && c < s.n_columns; };
    if (!has(s.col_episode)) return fail(BSB_INVALID_ARGUMENT, at + "missing column: episode");
    if (!has(s.col_value)) {
      const char* name = value_column(s.experiment);
      return fail(BSB_INVALID_ARGUMENT, at + "missing column: " + (name ? name : "total_return") + " (" + kExperimentNames[s.experiment] + ")");
    }
    if (rule_needs_best(info.rule) && !has(s.col_best))
      return fail(BSB_INVALID_ARGUMENT, at + "missing column: best_episode (" + kExperimentNames[s.experiment] + ")");
    if (info.grouped && !(s.group_key == s.group_key))
      return fail(BSB_INVALID_ARGUMENT, at + "group_key is NaN (" + kExperimentNames[s.experiment] + " groups by it)");
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
  for (int e = 0; e < BSB_NUM_EXPERIMENTS; ++e) sc->exps[e] = ScoreExp{0, 0};
  for (int32_t i : order) {
    const bsb_score_source& s = sources[i];
    ScoreDesc d;
    d.rows = s.rows; d.counts = s.counts; d.n_points = s.n_points; d.n_columns = s.n_columns;
    d.col_episode = s.col_episode; d.col_value = s.col_value; d.col_best = s.col_best; d.reserved0 = 0;
    d.key = s.group_key;
    ScoreExp& ex = sc->exps[s.experiment];
    if (ex.count == 0) ex.first = (int32_t)sc->descs.size();
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
