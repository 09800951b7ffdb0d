// bsuite_b200 engine: handle management, kernel dispatch, explicit host path and
// the extern "C" surface declared in include/bsuite_b200.h.
//
// Build: nvcc -gencode arch=compute_100a,code=sm_100a --fmad=false -lineinfo ...
// (--fmad=false: CPython/numpy never contract a*b+c; the float-dynamics
// families must evaluate the reference's expressions operation by operation.)
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <cstring>
#include <atomic>
#include <chrono>
#if defined(__x86_64__)
#include <immintrin.h>
#endif

#include "bsb_env.h"

using namespace bsb;

namespace bsb {
std::atomic<int64_t> g_launches{0};
namespace { thread_local std::string g_last_error; }
int fail(int code, const std::string& msg) { g_last_error = msg; return code; }
const char* last_error_cstr() { return g_last_error.c_str(); }
}  // namespace bsb

namespace {

InfoNames info_names(int family) {
  switch (family) {
    case BSB_DEEP_SEA: return {2, {"total_bad_episodes", "denoised_return", nullptr, nullptr}};
    case BSB_CATCH: return {1, {"total_regret", nullptr, nullptr, nullptr}};
    case BSB_CARTPOLE: return {2, {"raw_return", "best_episode", nullptr, nullptr}};
    case BSB_CARTPOLE_SWINGUP: return {3, {"raw_return", "total_upright", "best_episode", nullptr}};
    case BSB_MOUNTAIN_CAR: return {1, {"raw_return", nullptr, nullptr, nullptr}};
    case BSB_MEMORY_CHAIN: return {2, {"total_perfect", "total_regret", nullptr, nullptr}};
    case BSB_BANDIT: return {1, {"total_regret", nullptr, nullptr, nullptr}};
    case BSB_UMBRELLA_CHAIN: return {1, {"total_regret", nullptr, nullptr, nullptr}};
    case BSB_DISCOUNTING_CHAIN: return {0, {nullptr, nullptr, nullptr, nullptr}};
    case BSB_MNIST: return {1, {"total_regret", nullptr, nullptr, nullptr}};
  }
  return {0, {nullptr, nullptr, nullptr, nullptr}};
}

}  // namespace

namespace {

struct DeviceGuard {
  int prev; bool on;
  explicit DeviceGuard(int dev) : prev(0), on(dev >= 0) { if (on) { cudaGetDevice(&prev); cudaSetDevice(dev); } }
  ~DeviceGuard() { if (on) cudaSetDevice(prev); }
};

int env_alloc(bsb_env* e, void** out, size_t bytes, bool snapshot) {
  if (bytes == 0) { *out = nullptr; return BSB_OK; }
  void* ptr = nullptr;
  if (e->device >= 0) {
    BSB_CUDA(cudaMalloc(&ptr, bytes));
    BSB_CUDA(cudaMemset(ptr, 0, bytes));
  } else {
    ptr = calloc(1, bytes);
    if (!ptr) return fail(BSB_OUT_OF_MEMORY, "calloc failed");
  }
  e->allocs.push_back(ptr);
  if (snapshot) e->state_blocks.push_back(std::make_pair(ptr, bytes));
  *out = ptr;
  return BSB_OK;
}

int env_upload(bsb_env* e, void* dst, const void* src, size_t bytes) {
  if (bytes == 0) return BSB_OK;
  if (e->device >= 0) { BSB_CUDA(cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice)); }
  else memcpy(dst, src, bytes);
  return BSB_OK;
}

template <class T> int env_alloc_t(bsb_env* e, T** out, size_t count, bool snapshot) {
  void* ptr = nullptr;
  int rc = env_alloc(e, &ptr, count * sizeof(T), snapshot);
  *out = static_cast<T*>(ptr);
  return rc;
}

int run(bsb_env* e, const LaunchArgs& args, cudaStream_t stream) {
  DeviceGuard guard(e->device);
  LaunchArgs a = args;
  if (e->device >= 0) {
    cudaStreamCaptureStatus capture = cudaStreamCaptureStatusNone;
    BSB_CUDA(cudaStreamIsCapturing(stream, &capture));
    if (capture != cudaStreamCaptureStatusNone) { e->graph_safe = true; a.no_pdl = e->graph_pdl ? 0 : 1; }
    if (e->graph_safe) a.clock = e->clock;      // a.step0 == e->steps_done, which no longer moves
  }
  switch (e->p.family) {
    case BSB_DEEP_SEA: return run_deep_sea(e, a, stream);
    case BSB_CATCH: return run_catch(e, a, stream);
    case BSB_CARTPOLE: return run_cartpole(e, a, stream);
    case BSB_CARTPOLE_SWINGUP: return run_cartpole_swingup(e, a, stream);
    case BSB_MOUNTAIN_CAR: return run_mountain_car(e, a, stream);
    case BSB_MEMORY_CHAIN: return run_memory_chain(e, a, stream);
    case BSB_BANDIT: return run_bandit(e, a, stream);
    case BSB_UMBRELLA_CHAIN: return run_umbrella_chain(e, a, stream);
    case BSB_DISCOUNTING_CHAIN: return run_discounting_chain(e, a, stream);
    case BSB_MNIST: return run_mnist(e, a, stream);
  }
  return fail(BSB_INVALID_ARGUMENT, "unknown family");
}

LaunchArgs make_args(const bsb_env* e, const bsb_outputs* out, const int32_t* actions, int64_t T, int mode) {
  LaunchArgs a;
  memset(&a, 0, sizeof(a));
  a.actions = actions;
  if (out) { a.obs = out->observation; a.reward = out->reward; a.reward_f64 = out->reward_f64; a.discount = out->discount; a.step_type = out->step_type; }
  a.T = T; a.step0 = e->steps_done; a.mode = mode;
  const size_t step_bytes = (size_t)e->p.batch * (size_t)e->p.obs_numel * sizeof(float);
  a.obs_vec_ok = (out && (reinterpret_cast<uintptr_t>(out->observation) % 16 == 0) && (T == 1 || step_bytes % 16 == 0)) ? 1 : 0;
  return a;
}

int validate(const bsb_config& c, int64_t batch, int* obs_rows, int* obs_cols, int* n_actions) {
  if (batch <= 0) return fail(BSB_INVALID_ARGUMENT, "batch must be positive");
  if (c.wrapper < 0 || c.wrapper > 2) return fail(BSB_INVALID_ARGUMENT, "unknown wrapper");
  if (c.rng_kind < 0 || c.rng_kind > 1) return fail(BSB_INVALID_ARGUMENT, "unknown rng_kind");
  switch (c.family) {
    case BSB_DEEP_SEA:
      if (c.size < 1 || c.size > 255) return fail(BSB_INVALID_ARGUMENT, "deep_sea size must be in [1, 255]");
      if (!c.table || c.table_bytes != (int64_t)c.size * c.size) return fail(BSB_INVALID_ARGUMENT, "deep_sea needs a uint8 [N*N] action mapping table");
      *obs_rows = c.size; *obs_cols = c.size; *n_actions = 2; break;
    case BSB_CATCH:
      if (c.rows < 2 || c.rows > 255 || c.columns < 1 || c.columns > 255) return fail(BSB_INVALID_ARGUMENT, "catch rows in [2,255], columns in [1,255]");
      *obs_rows = c.rows; *obs_cols = c.columns; *n_actions = 3; break;
    case BSB_CARTPOLE: *obs_rows = 1; *obs_cols = 6; *n_actions = 3; break;
    case BSB_CARTPOLE_SWINGUP: *obs_rows = 1; *obs_cols = 8; *n_actions = 3; break;
    case BSB_MOUNTAIN_CAR:
      if (c.max_steps < 1) return fail(BSB_INVALID_ARGUMENT, "mountain_car max_steps must be >= 1");
      *obs_rows = 1; *obs_cols = 3; *n_actions = 3; break;
    case BSB_MEMORY_CHAIN:
      if (c.num_bits < 1 || c.num_bits > 64) return fail(BSB_UNSUPPORTED, "memory_chain num_bits must be in [1, 64]");
      if (c.memory_length < 1 || c.memory_length >= (1 << 24)) return fail(BSB_INVALID_ARGUMENT, "memory_length must be in [1, 2^24)");
      *obs_rows = 1; *obs_cols = c.num_bits + 2; *n_actions = 2; break;
    case BSB_BANDIT:
      if (c.num_actions < 1) return fail(BSB_INVALID_ARGUMENT, "bandit num_actions must be >= 1");
      if (!c.table || c.table_bytes != (int64_t)c.num_actions * 8) return fail(BSB_INVALID_ARGUMENT, "bandit needs a float64 [num_actions] reward table");
      *obs_rows = 1; *obs_cols = 1; *n_actions = c.num_actions; break;
    case BSB_UMBRELLA_CHAIN:
      if (c.chain_length < 1 || c.chain_length >= (1 << 24)) return fail(BSB_INVALID_ARGUMENT, "chain_length must be in [1, 2^24)");
      if (c.n_distractor < 0 || c.n_distractor > 1533) return fail(BSB_UNSUPPORTED, "n_distractor must be in [0, 1533]");
      *obs_rows = 1; *obs_cols = 3 + c.n_distractor; *n_actions = 2; break;
    case BSB_DISCOUNTING_CHAIN:
      if (!c.table || c.table_bytes != 5 * 8) return fail(BSB_INVALID_ARGUMENT, "discounting_chain needs a float64 [5] reward table");
      *obs_rows = 1; *obs_cols = 2; *n_actions = 5; break;
    case BSB_MNIST:
      if (c.num_data < 1 || c.image_rows < 1 || c.image_cols < 1) return fail(BSB_INVALID_ARGUMENT, "mnist needs num_data, image_rows, image_cols");
      if (c.image_rows > 4096 || c.image_cols > 4096) return fail(BSB_UNSUPPORTED, "mnist image sides must be <= 4096");
      if (!c.table || c.table_bytes != (int64_t)c.num_data * c.image_rows * c.image_cols) return fail(BSB_INVALID_ARGUMENT, "mnist needs an int8 image table");
      if (!c.table2 || c.table2_bytes != c.num_data) return fail(BSB_INVALID_ARGUMENT, "mnist needs a uint8 label table");
      *obs_rows = c.image_rows; *obs_cols = c.image_cols; *n_actions = 10; break;
    default: return fail(BSB_INVALID_ARGUMENT, "unknown family");
  }
  if (c.log_schedule_len < 0 || c.log_schedule_len > 4096) return fail(BSB_INVALID_ARGUMENT, "log_schedule_len must be in [0, 4096]");
  if (c.log_schedule_len > 0) {
    if (!c.log_schedule) return fail(BSB_INVALID_ARGUMENT, "log_schedule_len > 0 needs a log_schedule");
    if (!(c.flags & BSB_FLAG_TRACK_EPISODES)) return fail(BSB_INVALID_ARGUMENT, "a log schedule needs BSB_FLAG_TRACK_EPISODES");
    for (int64_t k = 0; k < c.log_schedule_len; ++k)
      if (c.log_schedule[k] < 1 || (k > 0 && c.log_schedule[k] <= c.log_schedule[k - 1]))
        return fail(BSB_INVALID_ARGUMENT, "log_schedule must be positive and strictly ascending");
  }
  if ((c.flags & BSB_FLAG_NO_LOG_ROWS) && c.log_schedule_len == 0)
    return fail(BSB_INVALID_ARGUMENT, "BSB_FLAG_NO_LOG_ROWS needs a log schedule");
  if (c.flags & BSB_FLAG_SCORE_SUMMARY) {
    if (c.log_schedule_len == 0) return fail(BSB_INVALID_ARGUMENT, "BSB_FLAG_SCORE_SUMMARY needs a log schedule");
    int rc = check_score_summary(c);
    if (rc != BSB_OK) return rc;
  }
  return BSB_OK;
}

bool family_uses_env_rng(const bsb_config& c) {
  switch (c.family) {
    case BSB_DEEP_SEA: return !c.deterministic;
    case BSB_BANDIT: case BSB_DISCOUNTING_CHAIN: return false;
    default: return true;
  }
}
bool family_uses_env_gauss(const bsb_config& c) { return c.family == BSB_DEEP_SEA && !c.deterministic; }

// Device-side alias of a pinned (page-locked, mapped) host pointer, or nullptr for pageable memory.  Queried on
// every call (well under a microsecond): a cached answer could outlive the buffer it described.
void* mapped_device_pointer(bsb_env*, const void* host_ptr) {
  cudaPointerAttributes attr;
  if (cudaPointerGetAttributes(&attr, host_ptr) == cudaSuccess && attr.type == cudaMemoryTypeHost) return attr.devicePointer;
  cudaGetLastError();   // clear the error a pageable pointer may leave behind
  return nullptr;
}


// Host-supplied actions are validated before anything moves (the reference raises IndexError for an arm that does
// not exist: bandit.py:61; catch.py:84).  Device-resident actions cannot be inspected without a synchronise: the
// kernels clamp them and raise env->bad_action_host instead (bsb_invalid_actions).
int check_host_actions(const bsb_env* e, const int32_t* actions, int64_t count) {
  const uint32_t n = (uint32_t)e->p.num_actions;
  for (int64_t k = 0; k < count; ++k)
    if ((uint32_t)actions[k] >= n)
      return fail(BSB_INVALID_ARGUMENT, "action " + std::to_string(actions[k]) + " at index " + std::to_string(k) +
                                            " is outside [0, " + std::to_string(n) + ")");
  return BSB_OK;
}

inline void cpu_relax() {
#if defined(__x86_64__)
  _mm_pause();
#endif
}

// ---- host-driven steps: mailbox completion and pre-launched doorbell kernels --------------------------------
int mailbox_open(bsb_env* e) {
  if (e->mailbox) return BSB_OK;
  void* host = nullptr; void* dev = nullptr;
  BSB_CUDA(cudaHostAlloc(&host, sizeof(HostMailbox), cudaHostAllocMapped | cudaHostAllocPortable));
  memset(host, 0, sizeof(HostMailbox));
  BSB_CUDA(cudaHostGetDevicePointer(&dev, host, 0));
  BSB_CUDA(cudaMalloc(reinterpret_cast<void**>(&e->mail), sizeof(DeviceMail)));
  BSB_CUDA(cudaMemset(e->mail, 0, sizeof(DeviceMail)));
  e->mailbox = static_cast<HostMailbox*>(host);
  e->mailbox_dev = static_cast<HostMailbox*>(dev);
  return BSB_OK;
}

// Enqueues one single-step launch that signals `ticket` through the mailbox.  wait_doorbell: the launch takes its
// buffers from the mailbox once the host rings `ticket` (pre-launch); otherwise from `fields` right away.
// Two-phase host steps pay off where the observation stream is long next to the scalar traffic over PCIe (12 B per
// lane out, 4 B in): deep_sea from N = 16 up (>= 1 KB of observation per lane).  catch (200 B per lane) is bound
// by the 2 MB of scalars per step either way and keeps the single-phase kernel (measured: 86 vs 51 us per step).
bool family_obs_from_state(const bsb_env* e) {
  return (e->p.family == BSB_DEEP_SEA || e->p.family == BSB_CATCH) && (size_t)e->p.obs_numel * sizeof(float) >= 1024;
}

int mailbox_launch(bsb_env* e, unsigned long long ticket, int64_t step0, const MailFields* fields, bool wait_doorbell, bool split = false) {
  LaunchArgs a;
  memset(&a, 0, sizeof(a));
  if (fields) {
    a.actions = fields->actions; a.obs = fields->obs; a.reward = fields->reward; a.reward_f64 = fields->reward_f64;
    a.discount = fields->discount; a.step_type = fields->step_type; a.obs_vec_ok = fields->obs_vec_ok;
  }
  a.T = 1; a.step0 = step0; a.mode = MODE_STEP;
  a.mailbox = e->mailbox_dev; a.mail = e->mail; a.ticket = ticket; a.wait_doorbell = wait_doorbell ? 1 : 0;
  a.doorbell_timeout_ns = e->doorbell_timeout_ns;
  { static const int timing = getenv("BSB_HOST_TIMING") ? atoi(getenv("BSB_HOST_TIMING")) : 0; a.timing = timing; }
  a.early_scalars = (e->host_early && family_obs_from_state(e)) ? 1 : 0;      // device_launch turns it into the copier count
  if (a.early_scalars) {
    // device staging of the scalars: reward | discount | step_type in one block (as the staged-copy path keeps them)
    const size_t B = (size_t)e->p.batch;
    if (!e->d_reward) {
      BSB_CUDA(cudaMalloc(&e->d_reward, 3 * B * 4));
      e->d_discount = e->d_reward + B;
      e->d_step_type = reinterpret_cast<int32_t*>(e->d_reward + 2 * B);
    }
    if (!e->d_reward64) BSB_CUDA(cudaMalloc(&e->d_reward64, B * 8));
    a.stage.reward = e->d_reward; a.stage.reward_f64 = e->d_reward64; a.stage.discount = e->d_discount; a.stage.step_type = e->d_step_type;
    e->early_inflight = true;
    if (split && e->host_split && !wait_doorbell) {
      // BSB_HOST_NO_WAIT: the caller alternates between handles.  Two launches instead of one -- transitions + copiers
      // (no shared memory), then the observation stream -- so that THIS handle's transitions and PCIe traffic run
      // while the OTHER handle's observations have the SMs' shared memory and the HBM.
      LaunchArgs first = a, second = a;
      first.phase = 1;
      second.phase = 2; second.mailbox = nullptr; second.early_scalars = 0;
      int rc = run(e, first, e->copy_stream);
      return rc != BSB_OK ? rc : run(e, second, e->copy_stream);
    }
  }
  return run(e, a, e->copy_stream);
}

// Spins on the mailbox until `ticket` is done (the kernel's last CTA stores it after a system-scope fence).
int mailbox_wait(bsb_env* e, unsigned long long ticket, bool* cancelled) {
  const auto start = std::chrono::steady_clock::now();
  unsigned long long seen;
  uint32_t spins = 0;
  while (((seen = e->mailbox->done) & ~MAIL_CANCEL) < ticket) {
    cpu_relax();
    if ((++spins & 0xfffffu) == 0 && std::chrono::steady_clock::now() - start > std::chrono::seconds(20)) {
      cudaError_t err = cudaStreamSynchronize(e->copy_stream);      // a faulted kernel never signals: surface its error
      if (err != cudaSuccess) return fail(BSB_CUDA_ERROR, std::string("host step: ") + cudaGetErrorString(err));
      if ((e->mailbox->done & ~MAIL_CANCEL) >= ticket) { seen = e->mailbox->done; break; }
      return fail(BSB_INTERNAL, "host step: the kernel finished without signalling the mailbox");
    }
  }
  std::atomic_thread_fence(std::memory_order_acquire);
  *cancelled = (seen & MAIL_CANCEL) != 0;
  return BSB_OK;
}

// Collects a step issued with BSB_HOST_NO_WAIT: spins until its completion word is in and counts the step.
int finish_awaited(bsb_env* e) {
  if (!e || e->device < 0 || !e->awaiting_ticket) return BSB_OK;
  const unsigned long long ticket = e->awaiting_ticket;
  e->awaiting_ticket = 0;
  bool cancelled = false;
  int rc = mailbox_wait(e, ticket, &cancelled);
  if (rc != BSB_OK) return rc;
  e->steps_done += 1;
  return BSB_OK;
}

// Stands down the pre-launched launch, if any: rings its ticket with the cancel bit and waits for it to leave
// (and collects a BSB_HOST_NO_WAIT step nobody waited for).
// Every entry point that enqueues work for this handle or reads its state calls this first.
int flush_pending(bsb_env* e) {
  { int arc = finish_awaited(e); if (arc != BSB_OK) return arc; }
  if (!e || e->device < 0 || !e->pending_ticket) return BSB_OK;
  DeviceGuard guard(e->device);
  const unsigned long long ticket = e->pending_ticket;
  e->pending_ticket = 0;
  std::atomic_thread_fence(std::memory_order_release);
  e->mailbox->doorbell = ticket | MAIL_CANCEL;
  bool cancelled = false;
  return mailbox_wait(e, ticket, &cancelled);
}

// Two-phase host steps return when the scalars have landed; the observation stores of the latest one may still
// be in flight on the handle's stream.  Anything that leaves that stream (work on a caller's stream, state reads,
// destruction) waits for it here.
int drain_host_steps(bsb_env* e) {
  int rc = flush_pending(e);
  if (rc != BSB_OK) return rc;
  if (e && e->device >= 0 && e->early_inflight) {
    DeviceGuard guard(e->device);
    e->early_inflight = false;
    BSB_CUDA(cudaStreamSynchronize(e->copy_stream));
  }
  return BSB_OK;
}

void destroy_env(bsb_env* e) {
  drain_host_steps(e);
  DeviceGuard guard(e->device);
  for (size_t k = 0; k < e->allocs.size(); ++k) { if (e->device >= 0) cudaFree(e->allocs[k]); else free(e->allocs[k]); }
  if (e->device >= 0) {
    if (e->h2d_actions) cudaFree(e->h2d_actions);
    if (e->d_reward) cudaFree(e->d_reward);      // also owns d_discount / d_step_type
    if (e->d_reward64) cudaFree(e->d_reward64);
    if (e->d_obs) cudaFree(e->d_obs);
    if (e->copy_stream) cudaStreamDestroy(e->copy_stream);
    if (e->order_event) cudaEventDestroy(e->order_event);
    if (e->fence_event) cudaEventDestroy(e->fence_event);
    if (e->h2d_event) cudaEventDestroy(e->h2d_event);
    if (e->h2d_stream) cudaStreamDestroy(e->h2d_stream);
    if (e->bad_action_host) cudaFreeHost(e->bad_action_host);
    if (e->mailbox) cudaFreeHost(e->mailbox);
    if (e->mail) cudaFree(e->mail);
  }
  delete e;
}

}  // namespace

__global__ void episode_stat_kernel(const EnvParams p, int field, int64_t calls, const unsigned long long* clock, double* dst) {
  if (clock) calls += (int64_t)*clock;      // graph-safe mode: steps since the switch are counted on the device
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < p.batch) dst[i] = episode_stat(p, i, field, calls);
}

// Sums of the five Logging columns over the lanes.  Deterministic: a fixed grid (a function of the batch only) of
// block-strided partial sums lands in scratch[block][5]; the block that finishes last adds the partials in block
// order and re-arms the ticket.  (No floating-point atomics: the result must not depend on scheduling -- a graph
// replay and an eager call must agree to the bit.)
constexpr int kSumBlocks = 64, kSumThreads = 256;
__global__ void episode_sum_kernel(const EnvParams p, int64_t calls, const unsigned long long* clock,
                                   double* scratch, unsigned long long* ticket, double* dst5) {
  if (clock) calls += (int64_t)*clock;
  __shared__ double partial[5][kSumThreads / 32];
  __shared__ bool is_last;
  double v[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < p.batch; i += (int64_t)gridDim.x * blockDim.x)
#pragma unroll
    for (int f = 0; f < 5; ++f) v[f] += episode_stat(p, i, f, calls);
#pragma unroll
  for (int f = 0; f < 5; ++f)
    for (int o = 16; o > 0; o >>= 1) v[f] += __shfl_down_sync(0xffffffffu, v[f], o);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) for (int f = 0; f < 5; ++f) partial[f][warp] = v[f];
  __syncthreads();
  if (threadIdx.x < 5) {
    double s = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += partial[threadIdx.x][w];
    scratch[blockIdx.x * 5 + threadIdx.x] = s;
    __threadfence();
  }
  __syncthreads();
  if (threadIdx.x == 0) is_last = atomicAdd(ticket, 1ull) == (unsigned long long)gridDim.x - 1ull;
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  if (threadIdx.x < 5) {
    double s = 0.0;
    for (unsigned b = 0; b < gridDim.x; ++b) s += __ldcg(scratch + b * 5 + threadIdx.x);
    dst5[threadIdx.x] = s;
  }
  if (threadIdx.x == 0) *ticket = 0ull;
}

// The same reduction for up to kSumManyMax environments in ONE launch (blockIdx.y = environment): a log point of
// the 23-experiment sweep is one kernel instead of 23.  Each environment keeps its own scratch and ticket, and
// its sums are combined in block order, so the result equals episode_sum_kernel's bit for bit.
constexpr int kSumManyMax = 64;
struct SumJob { const double* ep; int64_t batch; int64_t calls; const unsigned long long* clock; double* scratch; };
struct SumJobs { SumJob job[kSumManyMax]; };
__global__ void episode_sum_many_kernel(const SumJobs jobs, double* dst) {
  const SumJob j = jobs.job[blockIdx.y];
  EnvParams p;
  p.ep = const_cast<double*>(j.ep); p.batch = j.batch;
  int64_t calls = j.calls;
  if (j.clock) calls += (int64_t)*j.clock;
  __shared__ double partial[5][kSumThreads / 32];
  __shared__ bool is_last;
  double v[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < p.batch; i += (int64_t)gridDim.x * blockDim.x)
#pragma unroll
    for (int f = 0; f < 5; ++f) v[f] += episode_stat(p, i, f, calls);
#pragma unroll
  for (int f = 0; f < 5; ++f)
    for (int o = 16; o > 0; o >>= 1) v[f] += __shfl_down_sync(0xffffffffu, v[f], o);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) for (int f = 0; f < 5; ++f) partial[f][warp] = v[f];
  __syncthreads();
  // blocks that own no lanes of this environment contribute exact zeros, so the block-order sum below equals the
  // one episode_sum_kernel forms over min(blocks, ceil(batch / threads)) blocks
  if (threadIdx.x < 5) {
    double s = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += partial[threadIdx.x][w];
    j.scratch[blockIdx.x * 5 + threadIdx.x] = s;
    __threadfence();
  }
  __syncthreads();
  unsigned long long* ticket = reinterpret_cast<unsigned long long*>(j.scratch + kSumBlocks * 5);
  if (threadIdx.x == 0) is_last = atomicAdd(ticket, 1ull) == (unsigned long long)gridDim.x - 1ull;
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  if (threadIdx.x < 5) {
    double s = 0.0;
    for (unsigned b = 0; b < gridDim.x; ++b) s += __ldcg(j.scratch + b * 5 + threadIdx.x);
    dst[blockIdx.y * 5 + threadIdx.x] = s;
  }
  if (threadIdx.x == 0) *ticket = 0ull;
}

// ============================ extern "C" ====================================
extern "C" {

int32_t bsb_abi_version(void) { return BSB_ABI_VERSION; }
const char* bsb_last_error(void) { return bsb::last_error_cstr(); }
int64_t bsb_launch_count(void) { return g_launches.load(); }

int32_t bsb_create(const bsb_config* config, int64_t batch, int32_t device, uint64_t seed, uint64_t lane_offset, bsb_env** out) {
  if (!config || !out) return fail(BSB_INVALID_ARGUMENT, "null argument");
  *out = nullptr;
  const bsb_config& c = *config;
  int obs_rows = 0, obs_cols = 0, n_actions = 0;
  int rc = validate(c, batch, &obs_rows, &obs_cols, &n_actions);
  if (rc != BSB_OK) return rc;
  if (device >= 0) {
    int count = 0;
    cudaError_t err = cudaGetDeviceCount(&count);
    if (err != cudaSuccess || count <= 0)
      return fail(BSB_CUDA_ERROR, std::string("no CUDA device available (") + cudaGetErrorString(err) +
                                      "); this engine has no implicit CPU fallback -- pass device=BSB_DEVICE_HOST explicitly for the host path");
    if (device >= count) return fail(BSB_INVALID_ARGUMENT, "device ordinal out of range");
  } else if (device != BSB_DEVICE_HOST) {
    return fail(BSB_INVALID_ARGUMENT, "device must be >= 0 or BSB_DEVICE_HOST");
  }

  bsb_env* e = new bsb_env();
  memset(&e->p, 0, sizeof(e->p));
  e->device = device; e->steps_done = 0; e->graph_safe = false; e->clock = nullptr; e->sum_scratch = nullptr; e->names = info_names(c.family);
  {  // tuning knobs (environment variables, read once per handle)
    auto flag = [](const char* name, int dflt) { const char* v = getenv(name); return v ? (atoi(v) != 0 ? 1 : 0) : dflt; };
    const char* bt = getenv("BSB_BLOCK_THREADS");
    e->block_threads = bt ? atoi(bt) : 64;
    if (e->block_threads != 32 && e->block_threads != 64 && e->block_threads != 128) e->block_threads = 64;
    e->emit_bulk = flag("BSB_EMIT_BULK", 1);
    e->deep_sea_bulk = flag("BSB_DEEP_SEA_BULK", 1);
    { const char* g = getenv("BSB_DEEP_SEA_GROUP"); e->deep_sea_group = g ? atoi(g) : 0;
      if (e->deep_sea_group < 0 || e->deep_sea_group > 32 || (e->deep_sea_group & (e->deep_sea_group - 1))) e->deep_sea_group = 0; }
    e->use_pdl = flag("BSB_PDL", 1);
    e->graph_pdl = flag("BSB_GRAPH_PDL", 1);
    e->deep_sea_persistent = flag("BSB_DEEP_SEA_PERSISTENT", 1);
    e->zero_copy = flag("BSB_ZERO_COPY", 1);
    e->lazy_fetch = flag("BSB_LAZY_FETCH", 1);
    { const char* v = getenv("BSB_L2_HINT"); e->l2_hint = v ? atoi(v) : 1; if (e->l2_hint < 0 || e->l2_hint > 2) e->l2_hint = 1; }
    { const char* v = getenv("BSB_IMAGE_STAGES"); e->image_stages = (v && atoi(v) == 2) ? 2 : 1; }
    { const char* v = getenv("BSB_IMAGE_GROUP"); const int g = v ? atoi(v) : 4; e->image_group = (g == 1 || g == 2) ? g : 4; }
    { const char* v = getenv("BSB_CHUNK_LANES"); e->chunk_lanes = v ? atoi(v) : 0;
      if (e->chunk_lanes != 8 && e->chunk_lanes != 16 && e->chunk_lanes != 32) e->chunk_lanes = 0; }
    e->work_counter = nullptr; e->work_base = 0;
    e->num_sms = 148;
    if (device >= 0) { int n = 0; if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, device) == cudaSuccess && n > 0) e->num_sms = n; }
  }
  e->order_event = nullptr; e->fence_event = nullptr; e->bad_action_host = nullptr; e->bad_action_dev = nullptr;
  e->mailbox = nullptr; e->mailbox_dev = nullptr; e->mail = nullptr; e->next_ticket = 0; e->pending_ticket = 0; e->awaiting_ticket = 0;
  { const char* v = getenv("BSB_DOORBELL_TIMEOUT_MS"); const long ms = v ? atol(v) : 200; e->doorbell_timeout_ns = (unsigned long long)(ms > 0 ? ms : 200) * 1000000ull; }
  { const char* v = getenv("BSB_HOST_SPIN"); e->host_spin = v ? (atoi(v) != 0) : 1; }
  { const char* v = getenv("BSB_HOST_EARLY"); e->host_early = v ? (atoi(v) != 0) : 1; }
  { const char* v = getenv("BSB_HOST_SPLIT"); e->host_split = v ? (atoi(v) != 0) : 1; }
  { const char* v = getenv("BSB_SPLIT_GROUP"); e->split_group = v ? atoi(v) : 0;
    if (e->split_group < 0 || e->split_group > 32 || (e->split_group & (e->split_group - 1))) e->split_group = 0; }
  { const char* v = getenv("BSB_SPLIT_CTAS_PER_SM"); e->split_ctas_per_sm = v ? atoi(v) : 0;
    if (e->split_ctas_per_sm < 0 || e->split_ctas_per_sm > 16) e->split_ctas_per_sm = 0; }
  { const char* v = getenv("BSB_HOST_STAGE_ACTIONS"); e->host_stage_actions = v ? (atoi(v) != 0) : 1; }
  e->h2d_stream = nullptr; e->h2d_event = nullptr;
  e->early_inflight = false;
  e->h2d_actions = nullptr; e->d_reward = nullptr; e->d_reward64 = nullptr; e->d_discount = nullptr; e->d_step_type = nullptr; e->d_obs = nullptr;
  e->copy_stream = nullptr;
  DeviceGuard guard(device);

  EnvParams& p = e->p;
  p.family = c.family; p.wrapper = c.wrapper; p.rng_kind = c.rng_kind; p.flags = c.flags;
  p.size = c.size; p.deterministic = c.deterministic; p.rows = c.rows; p.columns = c.columns;
  p.memory_length = c.memory_length; p.num_bits = c.num_bits; p.chain_length = c.chain_length; p.n_distractor = c.n_distractor;
  p.num_actions = n_actions; p.max_steps = c.max_steps; p.num_data = c.num_data; p.image_numel = c.family == BSB_MNIST ? c.image_rows * c.image_cols : 0;
  p.obs_rows = obs_rows; p.obs_cols = obs_cols; p.obs_numel = obs_rows * obs_cols; p.n_info = e->names.n;
  p.batch = batch; p.seed = seed; p.lane_offset = lane_offset;
  if (c.family == BSB_DEEP_SEA) { p.move_cost_step = c.unscaled_move_cost / (double)c.size; p.inv_size = 1.0 / (double)c.size; }
  p.height_threshold = c.height_threshold; p.x_threshold = c.x_threshold; p.timescale = c.timescale; p.max_time = c.max_time;
  p.init_range = c.init_range; p.theta_dot_threshold = c.theta_dot_threshold; p.x_reward_threshold = c.x_reward_threshold;
  p.move_cost = c.move_cost; p.noise_scale = c.noise_scale; p.reward_scale = c.reward_scale;
  {  // cartpole.py:106-112 and the locals of step_cartpole (:40-47)
    const double mass_cart = 1.0, mass_pole = 0.1, length = 0.5;
    p.cp_force_mag = 10.0; p.cp_gravity = 9.8; p.cp_length = length; p.cp_mass_pole = mass_pole;
    p.cp_pl = mass_pole * length; p.cp_mass_total = mass_cart + mass_pole;
    p.cp_four_thirds = 4.0 / 3.0; p.cp_two_pi = 2.0 * 3.141592653589793;
  }

#define BSB_TRY(expr) do { rc = (expr); if (rc != BSB_OK) { destroy_env(e); return rc; } } while (0)
  const size_t B = (size_t)batch;
  // tables
  if (c.family == BSB_DEEP_SEA) {
    const int cells = c.size * c.size;
    std::vector<uint32_t> bits((size_t)(cells + 31) / 32, 0u);
    const uint8_t* m = static_cast<const uint8_t*>(c.table);
    for (int k = 0; k < cells; ++k) if (m[k]) bits[(size_t)k >> 5] |= 1u << (k & 31);
    uint32_t* d = nullptr;
    BSB_TRY(env_alloc_t(e, &d, bits.size(), false));
    BSB_TRY(env_upload(e, d, bits.data(), bits.size() * 4));
    p.mapping_bits = d;
  } else if (c.family == BSB_BANDIT || c.family == BSB_DISCOUNTING_CHAIN) {
    double* d = nullptr;
    BSB_TRY(env_alloc_t(e, &d, (size_t)c.table_bytes / 8, false));
    BSB_TRY(env_upload(e, d, c.table, (size_t)c.table_bytes));
    p.reward_table = d;
  } else if (c.family == BSB_MNIST) {
    int8_t* d = nullptr; uint8_t* l = nullptr;
    BSB_TRY(env_alloc_t(e, &d, (size_t)c.table_bytes, false));
    BSB_TRY(env_upload(e, d, c.table, (size_t)c.table_bytes));
    BSB_TRY(env_alloc_t(e, &l, (size_t)c.table2_bytes, false));
    BSB_TRY(env_upload(e, l, c.table2, (size_t)c.table2_bytes));
    p.images = d; p.labels = l;
  }
  if (device >= 0) {
    BSB_TRY(env_alloc_t(e, &e->work_counter, 1, false));
    BSB_TRY(env_alloc_t(e, &e->clock, CLOCK_WORDS, false));
    BSB_TRY(env_alloc_t(e, &e->sum_scratch, kSumBlocks * 5 + 1, false));
    void* flag = nullptr; void* flag_dev = nullptr;
    if (cudaHostAlloc(&flag, sizeof(int32_t), cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess ||
        cudaHostGetDevicePointer(&flag_dev, flag, 0) != cudaSuccess) {
      destroy_env(e); return fail(BSB_OUT_OF_MEMORY, "pinned allocation for the invalid-action flag failed");
    }
    e->bad_action_host = static_cast<int32_t*>(flag); *e->bad_action_host = 0;
    e->bad_action_dev = static_cast<int32_t*>(flag_dev);
  }
  // lane state
  BSB_TRY(env_alloc_t(e, &p.st_word, B, true));
  if (c.family == BSB_MEMORY_CHAIN) BSB_TRY(env_alloc_t(e, &p.st_ctx, B, true));
  if (c.family == BSB_CARTPOLE || c.family == BSB_CARTPOLE_SWINGUP) BSB_TRY(env_alloc_t(e, &p.st_f64, 6 * B, true));
  if (c.family == BSB_MOUNTAIN_CAR) BSB_TRY(env_alloc_t(e, &p.st_f64, 2 * B, true));
  BSB_TRY(env_alloc_t(e, &p.info, (size_t)BSB_MAX_INFO * B, true));
  if (c.flags & BSB_FLAG_TRACK_EPISODES) BSB_TRY(env_alloc_t(e, &p.ep, 5 * B, true));
  if (c.log_schedule_len > 0) {      // per-lane rows at the Logging wrapper's log-spaced episodes (wrappers.py:140-147)
    int64_t* sched = nullptr;
    BSB_TRY(env_alloc_t(e, &sched, (size_t)c.log_schedule_len, false));
    BSB_TRY(env_upload(e, sched, c.log_schedule, (size_t)c.log_schedule_len * sizeof(int64_t)));
    p.log_sched = sched; p.n_log_points = (int32_t)c.log_schedule_len;
    if (!(c.flags & BSB_FLAG_NO_LOG_ROWS))
      BSB_TRY(env_alloc_t(e, &p.log_rows, (size_t)c.log_schedule_len * (size_t)(5 + e->names.n) * B, true));
    BSB_TRY(env_alloc_t(e, &p.log_next, B, true));
  }
  if (c.flags & BSB_FLAG_SCORE_SUMMARY) {      // per-lane score summary (bsb_scoring.cuh, fold_row); NaN until a row
    p.score_exp = c.score_experiment;
    score_summary_columns(c.score_experiment, e->names, &p.score_col_value, &p.score_col_best);
    BSB_TRY(env_alloc_t(e, &p.score_sum, (size_t)BSB_SCORE_SUMMARY_FIELDS * B, true));
    const std::vector<double> nans((size_t)BSB_SCORE_SUMMARY_FIELDS * B, NAN);
    BSB_TRY(env_upload(e, p.score_sum, nans.data(), nans.size() * sizeof(double)));
  }
  // RNG state
  const bool env_rng = family_uses_env_rng(c);
  const bool noise = c.wrapper == BSB_WRAP_REWARD_NOISE;
  if (env_rng) {
    BSB_TRY(env_alloc_t(e, &p.rng_pos, B, true));
    if (family_uses_env_gauss(c)) BSB_TRY(env_alloc_t(e, &p.rng_gauss, B, true));
  }
  if (noise) {
    BSB_TRY(env_alloc_t(e, &p.wrng_pos, B, true));
    BSB_TRY(env_alloc_t(e, &p.wrng_gauss, B, true));
  }
  if (c.rng_kind == BSB_RNG_MT19937 && (env_rng || noise)) {
    // numpy.random.RandomState(seed + global lane); the wrapper's RandomState is
    // seeded with the SAME integer as the environment's (wrappers.py:267).
    std::vector<uint32_t> keys(624 * B);
    std::vector<int32_t> idx(B, 624);
    for (size_t i = 0; i < B; ++i) mt19937_seed_host(keys.data() + i, (int64_t)B, (uint32_t)(seed + lane_offset + i));
    if (env_rng) {
      BSB_TRY(env_alloc_t(e, &p.mt_key, 624 * B, true)); BSB_TRY(env_upload(e, p.mt_key, keys.data(), keys.size() * 4));
      BSB_TRY(env_alloc_t(e, &p.mt_idx, B, true)); BSB_TRY(env_upload(e, p.mt_idx, idx.data(), B * 4));
    }
    if (noise) {
      BSB_TRY(env_alloc_t(e, &p.wmt_key, 624 * B, true)); BSB_TRY(env_upload(e, p.wmt_key, keys.data(), keys.size() * 4));
      BSB_TRY(env_alloc_t(e, &p.wmt_idx, B, true)); BSB_TRY(env_upload(e, p.wmt_idx, idx.data(), B * 4));
    }
  }
  // constructor: _reset_next_step = True and the constructor's RNG draws
  LaunchArgs a = make_args(e, nullptr, nullptr, 0, MODE_INIT);
  BSB_TRY(run(e, a, nullptr));
  if (device >= 0) {
    cudaError_t err = cudaDeviceSynchronize();
    if (err != cudaSuccess) { destroy_env(e); return fail(BSB_CUDA_ERROR, std::string("init kernel: ") + cudaGetErrorString(err)); }
  }
#undef BSB_TRY
  *out = e;
  return BSB_OK;
}

int32_t bsb_destroy(bsb_env* env) { if (env) destroy_env(env); return BSB_OK; }

int32_t bsb_obs_numel(const bsb_env* env, int64_t* numel) {
  if (!env || !numel) return fail(BSB_INVALID_ARGUMENT, "null argument");
  *numel = env->p.obs_numel; return BSB_OK;
}
int32_t bsb_obs_shape(const bsb_env* env, int32_t* rows, int32_t* cols) {
  if (!env || !rows || !cols) return fail(BSB_INVALID_ARGUMENT, "null argument");
  *rows = env->p.obs_rows; *cols = env->p.obs_cols; return BSB_OK;
}
int32_t bsb_num_actions(const bsb_env* env, int32_t* n) {
  if (!env || !n) return fail(BSB_INVALID_ARGUMENT, "null argument");
  *n = env->p.num_actions; return BSB_OK;
}
int32_t bsb_batch(const bsb_env* env, int64_t* batch) {
  if (!env || !batch) return fail(BSB_INVALID_ARGUMENT, "null argument");
  *batch = env->p.batch; return BSB_OK;
}
// Host view of the step counter.  In graph-safe mode the count lives on the device (graph replays advance it
// without the host seeing them): wait for the device and read it back.
static int current_steps(const bsb_env* env, int64_t* steps) {
  *steps = env->steps_done;
  if (env->graph_safe) {
    DeviceGuard guard(env->device);
    unsigned long long since = 0;
    BSB_CUDA(cudaDeviceSynchronize());
    BSB_CUDA(cudaMemcpy(&since, env->clock, sizeof(since), cudaMemcpyDeviceToHost));
    *steps += (int64_t)since;
  }
  return BSB_OK;
}
static void advance_steps(bsb_env* env, int64_t n) { if (!env->graph_safe) env->steps_done += n; }

int32_t bsb_steps_done(const bsb_env* env, int64_t* steps) {
  if (!env || !steps) return fail(BSB_INVALID_ARGUMENT, "null argument");
  int rc = current_steps(env, steps);     // a pre-launched host step (if any) has not been counted: it is for step steps_done
  if (rc == BSB_OK && env->awaiting_ticket) *steps += 1;      // a BSB_HOST_NO_WAIT step has been issued: it counts
  return rc;
}

int32_t bsb_reset(bsb_env* env, const bsb_outputs* out, void* stream) {
  if (!env || !out || !out->observation) return fail(BSB_INVALID_ARGUMENT, "bsb_reset needs outputs with an observation buffer");
  { int frc = drain_host_steps(env); if (frc != BSB_OK) return frc; }
  LaunchArgs a = make_args(env, out, nullptr, 1, MODE_RESET);
  int rc = run(env, a, static_cast<cudaStream_t>(stream));
  if (rc == BSB_OK) advance_steps(env, 1);
  return rc;
}

int32_t bsb_step(bsb_env* env, const int32_t* actions, const bsb_outputs* out, void* stream) {
  if (!env || !actions || !out || !out->observation) return fail(BSB_INVALID_ARGUMENT, "bsb_step needs actions and outputs with an observation buffer");
  { int frc = drain_host_steps(env); if (frc != BSB_OK) return frc; }
  if (env->device < 0) { int vrc = check_host_actions(env, actions, env->p.batch); if (vrc != BSB_OK) return vrc; }
  LaunchArgs a = make_args(env, out, actions, 1, MODE_STEP);
  int rc = run(env, a, static_cast<cudaStream_t>(stream));
  if (rc == BSB_OK) advance_steps(env, 1);
  return rc;
}

int32_t bsb_rollout(bsb_env* env, int64_t num_steps, const int32_t* actions, uint64_t action_seed,
                    const bsb_outputs* out, int32_t* actions_out, void* stream) {
  if (!env || !out || !out->observation) return fail(BSB_INVALID_ARGUMENT, "bsb_rollout needs outputs with an observation buffer");
  if (num_steps <= 0) return fail(BSB_INVALID_ARGUMENT, "num_steps must be positive");
  { int frc = drain_host_steps(env); if (frc != BSB_OK) return frc; }
  if (env->device < 0 && actions) { int vrc = check_host_actions(env, actions, num_steps * env->p.batch); if (vrc != BSB_OK) return vrc; }
  LaunchArgs a = make_args(env, out, actions, num_steps, MODE_STEP);
  a.action_seed = action_seed; a.actions_out = actions_out;
  int rc = run(env, a, static_cast<cudaStream_t>(stream));
  if (rc == BSB_OK) advance_steps(env, num_steps);
  return rc;
}

int32_t bsb_random_actions(uint64_t action_seed, uint64_t lane_offset, int64_t batch, int64_t first_step,
                           int64_t num_steps, int32_t num_actions, int32_t* out) {
  if (!out || batch <= 0 || num_steps <= 0 || num_actions <= 0) return fail(BSB_INVALID_ARGUMENT, "bad arguments");
  for (int64_t t = 0; t < num_steps; ++t)
    for (int64_t i = 0; i < batch; ++i)
      out[t * batch + i] = sample_action(action_seed, lane_offset + (uint64_t)i, (uint64_t)(first_step + t), num_actions);
  return BSB_OK;
}

int32_t bsb_info_count(const bsb_env* env, int32_t* count) {
  if (!env || !count) return fail(BSB_INVALID_ARGUMENT, "null argument");
  *count = env->names.n; return BSB_OK;
}
const char* bsb_info_name(const bsb_env* env, int32_t index) {
  if (!env || index < 0 || index >= env->names.n) return nullptr;
  return env->names.names[index];
}

static int copy_field(bsb_env* env, const double* src, double* dst, void* stream) {
  const size_t bytes = (size_t)env->p.batch * sizeof(double);
  if (env->device >= 0) {
    DeviceGuard guard(env->device);
    BSB_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream)));
  } else {
    memcpy(dst, src, bytes);
  }
  return BSB_OK;
}

int32_t bsb_read_info(bsb_env* env, int32_t index, double* dst, void* stream) {
  if (!env || !dst) return fail(BSB_INVALID_ARGUMENT, "null argument");
  if (index < 0 || index >= env->names.n) return fail(BSB_INVALID_ARGUMENT, "info index out of range");
  { int frc = drain_host_steps(env); if (frc != BSB_OK) return frc; }
  return copy_field(env, env->p.info + (size_t)index * (size_t)env->p.batch, dst, stream);
}

int32_t bsb_read_episode_stats(bsb_env* env, int32_t field, double* dst, void* stream) {
  if (!env || !dst) return fail(BSB_INVALID_ARGUMENT, "null argument");
  if (!env->p.ep) return fail(BSB_INVALID_ARGUMENT, "environment was created without BSB_FLAG_TRACK_EPISODES");
  if (field < 0 || field >= 5) return fail(BSB_INVALID_ARGUMENT, "episode-stat field out of range");
  { int frc = drain_host_steps(env); if (frc != BSB_OK) return frc; }
  const int64_t B = env->p.batch;
  if (env->device >= 0) {
    DeviceGuard guard(env->device);
    episode_stat_kernel<<<(unsigned)((B + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(env->p, field, env->steps_done, env->graph_safe ? env->clock : nullptr, dst);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    BSB_CUDA(cudaGetLastError());
  } else {
    for (int64_t i = 0; i < B; ++i) dst[i] = episode_stat(env->p, i, field, env->steps_done);
  }
  return BSB_OK;
}

int32_t bsb_sum_episode_stats(bsb_env* env, double* dst5, void* stream) {
  if (!env || !dst5) return fail(BSB_INVALID_ARGUMENT, "null argument");
  if (!env->p.ep) return fail(BSB_INVALID_ARGUMENT, "environment was created without BSB_FLAG_TRACK_EPISODES");
  { int frc = drain_host_steps(env); if (frc != BSB_OK) return frc; }
  const int64_t B = env->p.batch;
  if (env->device >= 0) {
    DeviceGuard guard(env->device);
    int64_t blocks = (B + kSumThreads - 1) / kSumThreads;
    if (blocks > kSumBlocks) blocks = kSumBlocks;
    episode_sum_kernel<<<(unsigned)blocks, kSumThreads, 0, static_cast<cudaStream_t>(stream)>>>(
        env->p, env->steps_done, env->graph_safe ? env->clock : nullptr, env->sum_scratch,
        reinterpret_cast<unsigned long long*>(env->sum_scratch + kSumBlocks * 5), dst5);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    BSB_CUDA(cudaGetLastError());
  } else {
    for (int f = 0; f < 5; ++f) {
      double s = 0.0;
      for (int64_t i = 0; i < B; ++i) s += episode_stat(env->p, i, f, env->steps_done);
      dst5[f] = s;
    }
  }
  return BSB_OK;
}

int32_t bsb_sum_episode_stats_many(bsb_env* const* envs, int32_t count, double* dst, void* stream) {
  if (!envs || !dst || count <= 0) return fail(BSB_INVALID_ARGUMENT, "bad arguments");
  for (int32_t k = 0; k < count; ++k) {
    if (!envs[k]) return fail(BSB_INVALID_ARGUMENT, "null environment");
    if (!envs[k]->p.ep) return fail(BSB_INVALID_ARGUMENT, "environment was created without BSB_FLAG_TRACK_EPISODES");
    if (envs[k]->device != envs[0]->device) return fail(BSB_INVALID_ARGUMENT, "environments live on different devices");
  }
  if (envs[0]->device < 0 || count > kSumManyMax) {       // host path / oversized lists: one environment at a time
    for (int32_t k = 0; k < count; ++k) { int rc = bsb_sum_episode_stats(envs[k], dst + 5 * k, stream); if (rc != BSB_OK) return rc; }
    return BSB_OK;
  }
  DeviceGuard guard(envs[0]->device);
  SumJobs jobs;
  memset(&jobs, 0, sizeof(jobs));
  for (int32_t k = 0; k < count; ++k) {
    { int frc = drain_host_steps(envs[k]); if (frc != BSB_OK) return frc; }
    jobs.job[k].ep = envs[k]->p.ep; jobs.job[k].batch = envs[k]->p.batch; jobs.job[k].calls = envs[k]->steps_done;
    jobs.job[k].clock = envs[k]->graph_safe ? envs[k]->clock : nullptr; jobs.job[k].scratch = envs[k]->sum_scratch;
  }
  episode_sum_many_kernel<<<dim3(kSumBlocks, (unsigned)count), kSumThreads, 0, static_cast<cudaStream_t>(stream)>>>(jobs, dst);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  BSB_CUDA(cudaGetLastError());
  return BSB_OK;
}

int32_t bsb_log_layout(const bsb_env* env, int32_t* n_points, int32_t* n_columns) {
  if (!env || !n_points || !n_columns) return fail(BSB_INVALID_ARGUMENT, "null argument");
  *n_points = env->p.n_log_points; *n_columns = env->p.log_rows ? 5 + env->names.n : 0;
  return BSB_OK;
}

int32_t bsb_read_log_rows(bsb_env* env, double* rows, int32_t* counts, void* stream) {
  if (!env || !rows || !counts) return fail(BSB_INVALID_ARGUMENT, "null argument");
  if (env->p.log_next && !env->p.log_rows) return fail(BSB_INVALID_ARGUMENT, "environment keeps no log rows (BSB_FLAG_NO_LOG_ROWS)");
  if (!env->p.log_rows) return fail(BSB_INVALID_ARGUMENT, "environment was created without a log schedule");
  { int frc = drain_host_steps(env); if (frc != BSB_OK) return frc; }
  const size_t B = (size_t)env->p.batch;
  const size_t row_bytes = (size_t)env->p.n_log_points * (size_t)(5 + env->names.n) * B * sizeof(double);
  if (env->device >= 0) {
    DeviceGuard guard(env->device);
    BSB_CUDA(cudaMemcpyAsync(rows, env->p.log_rows, row_bytes, cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream)));
    BSB_CUDA(cudaMemcpyAsync(counts, env->p.log_next, B * sizeof(int32_t), cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream)));
  } else {
    memcpy(rows, env->p.log_rows, row_bytes);
    memcpy(counts, env->p.log_next, B * sizeof(int32_t));
  }
  return BSB_OK;
}

int32_t bsb_read_score_summary(bsb_env* env, double* summary, int32_t* counts, void* stream) {
  if (!env || !summary || !counts) return fail(BSB_INVALID_ARGUMENT, "null argument");
  if (!env->p.score_sum) return fail(BSB_INVALID_ARGUMENT, "environment was created without BSB_FLAG_SCORE_SUMMARY");
  { int frc = drain_host_steps(env); if (frc != BSB_OK) return frc; }
  const size_t B = (size_t)env->p.batch;
  const size_t bytes = (size_t)BSB_SCORE_SUMMARY_FIELDS * B * sizeof(double);
  if (env->device >= 0) {
    DeviceGuard guard(env->device);
    BSB_CUDA(cudaMemcpyAsync(summary, env->p.score_sum, bytes, cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream)));
    BSB_CUDA(cudaMemcpyAsync(counts, env->p.log_next, B * sizeof(int32_t), cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream)));
  } else {
    memcpy(summary, env->p.score_sum, bytes);
    memcpy(counts, env->p.log_next, B * sizeof(int32_t));
  }
  return BSB_OK;
}

int32_t bsb_state_bytes(const bsb_env* env, int64_t* nbytes) {
  if (!env || !nbytes) return fail(BSB_INVALID_ARGUMENT, "null argument");
  size_t total = sizeof(int64_t);
  for (size_t k = 0; k < env->state_blocks.size(); ++k) total += env->state_blocks[k].second;
  *nbytes = (int64_t)total; return BSB_OK;
}

int32_t bsb_get_state(bsb_env* env, void* dst_host, int64_t nbytes, void* stream) {
  int64_t need = 0;
  if (!env || !dst_host) return fail(BSB_INVALID_ARGUMENT, "null argument");
  bsb_state_bytes(env, &need);
  if (nbytes != need) return fail(BSB_INVALID_ARGUMENT, "state buffer has the wrong size");
  { int frc = drain_host_steps(env); if (frc != BSB_OK) return frc; }
  DeviceGuard guard(env->device);
  char* dst = static_cast<char*>(dst_host);
  if (env->device >= 0) BSB_CUDA(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
  int64_t steps = 0;
  { int rc = current_steps(env, &steps); if (rc != BSB_OK) return rc; }
  memcpy(dst, &steps, sizeof(int64_t)); dst += sizeof(int64_t);
  for (size_t k = 0; k < env->state_blocks.size(); ++k) {
    if (env->device >= 0) BSB_CUDA(cudaMemcpy(dst, env->state_blocks[k].first, env->state_blocks[k].second, cudaMemcpyDeviceToHost));
    else memcpy(dst, env->state_blocks[k].first, env->state_blocks[k].second);
    dst += env->state_blocks[k].second;
  }
  return BSB_OK;
}

int32_t bsb_set_state(bsb_env* env, const void* src_host, int64_t nbytes, void* stream) {
  int64_t need = 0;
  if (!env || !src_host) return fail(BSB_INVALID_ARGUMENT, "null argument");
  bsb_state_bytes(env, &need);
  if (nbytes != need) return fail(BSB_INVALID_ARGUMENT, "state buffer has the wrong size");
  { int frc = drain_host_steps(env); if (frc != BSB_OK) return frc; }
  DeviceGuard guard(env->device);
  const char* src = static_cast<const char*>(src_host);
  if (env->device >= 0) BSB_CUDA(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
  int64_t restored = 0;
  memcpy(&restored, src, sizeof(int64_t)); src += sizeof(int64_t);
  if (env->graph_safe) {
    // steps_done is baked into the captured launches as their base: it must not move.  The restored count goes
    // into the device clock as an offset from that base (two's complement, so it may be "negative").
    const unsigned long long since = (unsigned long long)restored - (unsigned long long)env->steps_done;
    BSB_CUDA(cudaDeviceSynchronize());
    unsigned long long replicas[CLOCK_GROUPS];
    for (int r = 0; r < CLOCK_GROUPS; ++r) replicas[r] = since;
    BSB_CUDA(cudaMemcpy2D(env->clock, 16 * sizeof(unsigned long long), replicas, sizeof(unsigned long long),
                          sizeof(unsigned long long), CLOCK_GROUPS, cudaMemcpyHostToDevice));
  } else {
    env->steps_done = restored;
  }
  for (size_t k = 0; k < env->state_blocks.size(); ++k) {
    if (env->device >= 0) BSB_CUDA(cudaMemcpy(env->state_blocks[k].first, src, env->state_blocks[k].second, cudaMemcpyHostToDevice));
    else memcpy(env->state_blocks[k].first, src, env->state_blocks[k].second);
    src += env->state_blocks[k].second;
  }
  return BSB_OK;
}

int32_t bsb_invalid_actions(bsb_env* env, int32_t* seen) {
  if (!env || !seen) return fail(BSB_INVALID_ARGUMENT, "null argument");
  *seen = 0;
  if (env->bad_action_host) { *seen = *env->bad_action_host; *env->bad_action_host = 0; }
  return BSB_OK;
}

int32_t bsb_host_timing(bsb_env* env, uint64_t* stamps8) {
  if (!env || !stamps8) return fail(BSB_INVALID_ARGUMENT, "null argument");
  if (!env->mailbox) return fail(BSB_INVALID_ARGUMENT, "no host-driven step has run on this handle");
  for (int k = 0; k < 8; ++k) stamps8[k] = env->mailbox->stamp[k];
  return BSB_OK;
}

int32_t bsb_host_flush(bsb_env* env) {
  if (!env) return fail(BSB_INVALID_ARGUMENT, "null argument");
  return flush_pending(env);
}

// Reports (and clears) an out-of-range action seen by the kernels of a synchronous host step.
static int report_bad_actions(bsb_env* env) {
  if (env->bad_action_host && *env->bad_action_host) {
    *env->bad_action_host = 0;
    return fail(BSB_INVALID_ARGUMENT, "an action was outside [0, " + std::to_string(env->p.num_actions) +
                                          "): the step was taken with that action clamped into range");
  }
  return BSB_OK;
}

int32_t bsb_step_host(bsb_env* env, const int32_t* actions, const bsb_outputs* host_out, float* device_obs,
                      void* caller_stream, uint32_t flags) {
  if (!env || !actions || !host_out) return fail(BSB_INVALID_ARGUMENT, "null argument");
  if (env->device < 0) {
    if (!host_out->observation) return fail(BSB_INVALID_ARGUMENT, "a host environment writes observations to host_out->observation");
    return bsb_step(env, actions, host_out, nullptr);
  }
  if (!host_out->observation && !device_obs) return fail(BSB_INVALID_ARGUMENT, "need host_out->observation or device_obs");
  if ((flags & BSB_HOST_NO_WAIT) && (flags & BSB_HOST_PRELAUNCH)) return fail(BSB_INVALID_ARGUMENT, "BSB_HOST_NO_WAIT and BSB_HOST_PRELAUNCH exclude each other");
  DeviceGuard guard(env->device);
  { int arc = finish_awaited(env); if (arc != BSB_OK) return arc; }      // one step in flight per handle
  const size_t B = (size_t)env->p.batch, K = (size_t)env->p.obs_numel;
  if (!env->copy_stream) BSB_CUDA(cudaStreamCreateWithFlags(&env->copy_stream, cudaStreamNonBlocking));
  if (flags & BSB_HOST_ORDER_AFTER_STREAM) {
    // Work the caller enqueued earlier on ITS stream (bsb_reset / bsb_step / bsb_rollout of this handle) must have
    // finished with the lane state before this step touches it: fence the handle's stream behind it.
    { int frc = drain_host_steps(env); if (frc != BSB_OK) return frc; }
    if (!env->order_event) BSB_CUDA(cudaEventCreateWithFlags(&env->order_event, cudaEventDisableTiming));
    BSB_CUDA(cudaEventRecord(env->order_event, static_cast<cudaStream_t>(caller_stream)));
    BSB_CUDA(cudaStreamWaitEvent(env->copy_stream, env->order_event, 0));
  }

  // Zero-copy path: when the caller's action and scalar buffers are PINNED host memory (device-addressable under
  // unified addressing), the transition kernel reads the actions from and writes reward / discount / step_type to
  // host memory directly over PCIe -- 1 MB per step, overlapped with the observation stream -- instead of three
  // separate copies with their launch and DMA latencies before and after the kernel.
  if (env->zero_copy) {
    void* d_actions = mapped_device_pointer(env, actions);
    void* d_reward = host_out->reward ? mapped_device_pointer(env, host_out->reward) : nullptr;
    void* d_reward64 = host_out->reward_f64 ? mapped_device_pointer(env, host_out->reward_f64) : nullptr;
    void *d_discount = nullptr, *d_step_type = nullptr;
    const bool packed_scalars = d_reward && host_out->discount == host_out->reward + B &&
                                reinterpret_cast<char*>(host_out->step_type) == reinterpret_cast<char*>(host_out->reward + 2 * B);
    if (packed_scalars) {       // reward | discount | step_type back to back in one pinned block: one query covers all
      d_discount = static_cast<float*>(d_reward) + B;
      d_step_type = static_cast<float*>(d_reward) + 2 * B;
    } else {
      d_discount = host_out->discount ? mapped_device_pointer(env, host_out->discount) : nullptr;
      d_step_type = host_out->step_type ? mapped_device_pointer(env, host_out->step_type) : nullptr;
    }
    const bool all_mapped = d_actions && (!host_out->reward || d_reward) && (!host_out->reward_f64 || d_reward64) &&
                            (!host_out->discount || d_discount) && (!host_out->step_type || d_step_type);
    if (all_mapped) {
      if (!device_obs && !env->d_obs) BSB_CUDA(cudaMalloc(&env->d_obs, B * K * 4));
      MailFields f;
      memset(&f, 0, sizeof(f));
      f.actions = static_cast<const int32_t*>(d_actions);
      f.obs = device_obs ? device_obs : env->d_obs;
      f.reward = static_cast<float*>(d_reward);
      f.reward_f64 = static_cast<double*>(d_reward64);
      f.discount = static_cast<float*>(d_discount);
      f.step_type = static_cast<int32_t*>(d_step_type);
      f.obs_vec_ok = (reinterpret_cast<uintptr_t>(f.obs) % 16 == 0) ? 1 : 0;
      cudaStream_t zs = env->copy_stream;
      // Completion through the mailbox (BSB_HOST_SPIN=0 turns it off): the kernel's last CTA stores the ticket into
      // pinned host memory after a system-scope fence and the host spins on that word -- a stream synchronise costs
      // a wake-up of ~10 us per step.  Observations copied to the host, graph-safe handles and unaligned
      // observation buffers keep the synchronise.
      const bool spin = env->host_spin && !env->graph_safe && !host_out->observation && f.obs_vec_ok;
      if (!spin) {
        { int frc = drain_host_steps(env); if (frc != BSB_OK) return frc; }
        bsb_outputs dev;
        dev.observation = f.obs; dev.reward = f.reward; dev.reward_f64 = f.reward_f64; dev.discount = f.discount; dev.step_type = f.step_type;
        int zrc = bsb_step(env, f.actions, &dev, zs);
        if (zrc != BSB_OK) return zrc;
        if (host_out->observation) BSB_CUDA(cudaMemcpyAsync(host_out->observation, dev.observation, B * K * 4, cudaMemcpyDeviceToHost, zs));
        BSB_CUDA(cudaStreamSynchronize(zs));
        return report_bad_actions(env);
      }
      { int mrc = mailbox_open(env); if (mrc != BSB_OK) return mrc; }
      const bool prelaunch = (flags & BSB_HOST_PRELAUNCH) != 0;
      for (int attempt = 0; attempt < 2; ++attempt) {
        unsigned long long ticket;
        if (env->pending_ticket) {
          // The kernel of this step is already resident and polling: hand it the buffers and ring.
          ticket = env->pending_ticket;
          env->pending_ticket = 0;
          env->mailbox->in = f;
          std::atomic_thread_fence(std::memory_order_release);
          env->mailbox->doorbell = ticket;
        } else {
          ticket = ++env->next_ticket;
          if (env->host_stage_actions && env->host_early && family_obs_from_state(env)) {
            // Two-phase step: phase 1 (the transitions of every lane) is all that stands between this launch and the
            // observation stream, and reading 4 B per lane over PCIe from inside the kernel is most of it.  The DMA
            // engine brings the actions over NOW, on a side stream, while the previous step's kernel is still
            // streaming observations; the launch waits for that copy on the device.  (The previous kernel read its
            // actions in phase 1, which ended before its completion word was seen: the buffer is free.)
            if (!env->h2d_actions) BSB_CUDA(cudaMalloc(&env->h2d_actions, B * 4));
            if (!env->h2d_stream) {
              BSB_CUDA(cudaStreamCreateWithFlags(&env->h2d_stream, cudaStreamNonBlocking));
              BSB_CUDA(cudaEventCreateWithFlags(&env->h2d_event, cudaEventDisableTiming));
            }
            BSB_CUDA(cudaMemcpyAsync(env->h2d_actions, actions, B * 4, cudaMemcpyHostToDevice, env->h2d_stream));
            BSB_CUDA(cudaEventRecord(env->h2d_event, env->h2d_stream));
            BSB_CUDA(cudaStreamWaitEvent(zs, env->h2d_event, 0));
            f.actions = env->h2d_actions;
          }
          int lrc = mailbox_launch(env, ticket, env->steps_done, &f, false, (flags & BSB_HOST_NO_WAIT) != 0);
          if (lrc != BSB_OK) return lrc;
        }
        if ((flags & BSB_HOST_FENCE_CALLER) && env->early_inflight) {
          // Two-phase step: the observation stores outlive this call.  Fence the caller's stream behind the kernel
          // (the event is recorded BEFORE the next step's kernel is queued, so it stands for this step only):
          // whatever the caller enqueues there afterwards sees complete observations.
          if (!env->fence_event) BSB_CUDA(cudaEventCreateWithFlags(&env->fence_event, cudaEventDisableTiming));
          BSB_CUDA(cudaEventRecord(env->fence_event, zs));
          BSB_CUDA(cudaStreamWaitEvent(static_cast<cudaStream_t>(caller_stream), env->fence_event, 0));
        }
        if (flags & BSB_HOST_NO_WAIT) {
          // Split call: the completion word is collected by bsb_host_wait (or by whichever entry point of this handle
          // runs next), so the caller can drive ANOTHER handle while this step's scalars cross PCIe.
          env->awaiting_ticket = ticket;
          return BSB_OK;
        }
        if (prelaunch) {
          // Queue the NEXT step's kernel now: it becomes resident as this one drains and waits for its doorbell,
          // so the next call pays neither a launch nor a wake-up.  It stands down by itself after
          // BSB_DOORBELL_TIMEOUT_MS without a ring.
          const unsigned long long next = ++env->next_ticket;
          int lrc = mailbox_launch(env, next, env->steps_done + 1, nullptr, true);
          if (lrc != BSB_OK) return lrc;
          env->pending_ticket = next;
        }
        bool cancelled = false;
        { int wrc = mailbox_wait(env, ticket, &cancelled); if (wrc != BSB_OK) return wrc; }
        if (!cancelled) { env->steps_done += 1; return report_bad_actions(env); }
        // The pre-launched kernel had given up waiting before the ring arrived: nothing was stepped.  The launch
        // queued behind it carries the wrong step index now; stand it down and take the step again, launched now.
        { int frc = flush_pending(env); if (frc != BSB_OK) return frc; }
      }
      return fail(BSB_INTERNAL, "host step: a freshly launched kernel reported a cancelled doorbell");
    }
  }
  { int frc = drain_host_steps(env); if (frc != BSB_OK) return frc; }
  if (!env->h2d_actions) BSB_CUDA(cudaMalloc(&env->h2d_actions, B * 4));
  // reward | discount | step_type live in ONE device block so that a caller who keeps its three host arrays
  // back to back (BatchedEnvironment.make_host_buffers does) gets them with a single D2H copy.
  if (!env->d_reward) {
    BSB_CUDA(cudaMalloc(&env->d_reward, 3 * B * 4));
    env->d_discount = env->d_reward + B;
    env->d_step_type = reinterpret_cast<int32_t*>(env->d_reward + 2 * B);
  }
  if (host_out->reward_f64 && !env->d_reward64) BSB_CUDA(cudaMalloc(&env->d_reward64, B * 8));
  if (!device_obs && !env->d_obs) BSB_CUDA(cudaMalloc(&env->d_obs, B * K * 4));
  { int vrc = check_host_actions(env, actions, (int64_t)B); if (vrc != BSB_OK) return vrc; }
  cudaStream_t s = env->copy_stream;
  BSB_CUDA(cudaMemcpyAsync(env->h2d_actions, actions, B * 4, cudaMemcpyHostToDevice, s));
  bsb_outputs dev;
  dev.observation = device_obs ? device_obs : env->d_obs;
  dev.reward = host_out->reward ? env->d_reward : nullptr;
  dev.reward_f64 = host_out->reward_f64 ? env->d_reward64 : nullptr;
  dev.discount = host_out->discount ? env->d_discount : nullptr;
  dev.step_type = host_out->step_type ? env->d_step_type : nullptr;
  int rc = bsb_step(env, env->h2d_actions, &dev, s);
  if (rc != BSB_OK) return rc;
  const bool packed = host_out->reward && host_out->discount && host_out->step_type &&
                      host_out->discount == host_out->reward + B &&
                      reinterpret_cast<char*>(host_out->step_type) == reinterpret_cast<char*>(host_out->reward + 2 * B);
  if (packed) {
    BSB_CUDA(cudaMemcpyAsync(host_out->reward, env->d_reward, 3 * B * 4, cudaMemcpyDeviceToHost, s));
  } else {
    if (host_out->reward) BSB_CUDA(cudaMemcpyAsync(host_out->reward, dev.reward, B * 4, cudaMemcpyDeviceToHost, s));
    if (host_out->discount) BSB_CUDA(cudaMemcpyAsync(host_out->discount, dev.discount, B * 4, cudaMemcpyDeviceToHost, s));
    if (host_out->step_type) BSB_CUDA(cudaMemcpyAsync(host_out->step_type, dev.step_type, B * 4, cudaMemcpyDeviceToHost, s));
  }
  if (host_out->reward_f64) BSB_CUDA(cudaMemcpyAsync(host_out->reward_f64, dev.reward_f64, B * 8, cudaMemcpyDeviceToHost, s));
  if (host_out->observation) BSB_CUDA(cudaMemcpyAsync(host_out->observation, dev.observation, B * K * 4, cudaMemcpyDeviceToHost, s));
  BSB_CUDA(cudaStreamSynchronize(s));
  return BSB_OK;
}


int32_t bsb_host_wait(bsb_env* env) {
  if (!env) return fail(BSB_INVALID_ARGUMENT, "null argument");
  if (env->device < 0 || !env->awaiting_ticket) return BSB_OK;
  DeviceGuard guard(env->device);
  { int rc = finish_awaited(env); if (rc != BSB_OK) return rc; }
  return report_bad_actions(env);
}

}  // extern "C"
