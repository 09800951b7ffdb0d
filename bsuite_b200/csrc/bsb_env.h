// Internal declarations shared by the engine and the per-family translation units.
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <string>
#include <utility>
#include <vector>

#include "../../include/bsuite_b200.h"
#include "bsb_kernels.cuh"

namespace bsb {

struct InfoNames { int n; const char* names[BSB_MAX_INFO]; };

int fail(int code, const std::string& msg);           // records the thread-local error string
const char* last_error_cstr();
extern std::atomic<int64_t> g_launches;                // kernels launched by this library

// BSB_FLAG_SCORE_SUMMARY (bsb_scoring.cu): check_score_summary validates a configuration (experiment of the
// family, log schedule a prefix of the experiment's); score_summary_columns finds the row columns the fold reads
// (value column, best_episode or -1) among the five Logging columns and the family's info fields.
int check_score_summary(const bsb_config& c);
void score_summary_columns(int experiment, const InfoNames& names, int32_t* col_value, int32_t* col_best);

#define BSB_CUDA(expr)                                                                   \
  do {                                                                                   \
    cudaError_t e__ = (expr);                                                            \
    if (e__ != cudaSuccess)                                                              \
      return ::bsb::fail(e__ == cudaErrorMemoryAllocation ? BSB_OUT_OF_MEMORY : BSB_CUDA_ERROR, \
                         std::string(#expr) + ": " + cudaGetErrorString(e__));           \
  } while (0)

}  // namespace bsb

struct bsb_env {
  bsb::EnvParams p;
  int device;             // BSB_DEVICE_HOST or CUDA ordinal
  int64_t steps_done;     // step() calls so far (host counter; frozen at the switch to graph-safe mode)
  // Graph-safe mode: entered for good when a launch of this handle is first captured into a CUDA graph.  From
  // then on the device clock counts the steps (kernel comment in bsb_kernels.cuh) and steps = steps_done + clock[0].
  bool graph_safe;
  unsigned long long* clock;         // device, CLOCK_WORDS words: step count (replicated), chunk counter, finished-CTA counters
  double* sum_scratch;               // device: bsb_sum_episode_stats partials [64][5] + the ticket
  // tuning knobs (environment variables, read once per handle)
  int block_threads;      // CTA size of the transition kernel (32 / 64 / 128)
  int emit_bulk;          // TMA bulk stores for the row / board emitters
  int deep_sea_bulk;      // TMA bulk stores for deep_sea tiles (else 16-byte streaming stores)
  int deep_sea_group;     // lanes per deep_sea bulk store (0 = automatic)
  int deep_sea_persistent; // persistent grid + dynamic chunk dealing for the deep_sea bulk path
  unsigned long long* work_counter;  // device counter of the dynamic chunk scheduler
  unsigned long long work_base;      // its value when the next launch starts
  int use_pdl;            // programmatic dependent launch between consecutive steps
  int graph_pdl;          // ... also between launches captured into a CUDA graph (programmatic graph edges)
  int zero_copy;          // bsb_step_host: kernel reads/writes pinned host buffers directly
  int lazy_fetch;         // persistent kernel: fetch the next chunk lazily (default) or one chunk ahead
  int l2_hint;            // L2 eviction hint of the observation bulk stores (0 none, 1 evict_first, 2 evict_last)
  int image_stages;       // mnist TMA path: staging buffers per warp (1 or 2)
  int image_group;        // mnist TMA path: tiles per staged store (1, 2 or 4)
  int chunk_lanes;        // lanes per chunk: 0 = automatic (32; 16 / 8 for small mnist batches), BSB_CHUNK_LANES forces
  int num_sms;
  bsb::InfoNames names;
  std::vector<void*> allocs;
  std::vector<std::pair<void*, size_t> > state_blocks;  // snapshot layout
  // bsb_step_host scratch (device)
  int32_t* h2d_actions; float* d_reward; double* d_reward64; float* d_discount; int32_t* d_step_type; float* d_obs;
  cudaStream_t copy_stream;
  cudaEvent_t order_event;            // BSB_HOST_ORDER_AFTER_STREAM: fences copy_stream behind the caller's stream
  cudaEvent_t fence_event;            // BSB_HOST_FENCE_CALLER: fences the caller's stream behind a two-phase host step
  // Out-of-range actions (ADVICE r01): the kernels clamp them before any table index or state packing and raise
  // this pinned flag; bsb_step_host / bsb_invalid_actions report it.
  int32_t* bad_action_host; int32_t* bad_action_dev;
  // Host-driven steps without a stream synchronise (bsb_step_host on pinned buffers): the kernel signals completion
  // through a pinned mailbox the host spins on; with BSB_HOST_PRELAUNCH the next step's kernel is already queued
  // and waits for the mailbox doorbell (bsb_kernels.cuh, HostMailbox).
  bsb::HostMailbox* mailbox; bsb::HostMailbox* mailbox_dev; bsb::DeviceMail* mail;
  unsigned long long next_ticket;     // last ticket handed out
  unsigned long long awaiting_ticket; // a BSB_HOST_NO_WAIT step whose completion word has not been collected yet (0 = none)
  unsigned long long pending_ticket;  // pre-launched launch waiting for its doorbell (0 = none); it is for step steps_done
  unsigned long long doorbell_timeout_ns;
  int host_spin;                      // BSB_HOST_SPIN (default 1): completion through the mailbox instead of a synchronise
  int host_split;                     // BSB_HOST_SPLIT (default 1): BSB_HOST_NO_WAIT two-phase steps run as two launches (transitions, observations)
  int split_group;                    // BSB_SPLIT_GROUP (default 0 = as ordinary steps): lanes per bulk store of the observation-only launch of a split step
  int split_ctas_per_sm;              // BSB_SPLIT_CTAS_PER_SM (default 0 = no cap): persistent CTAs per SM of that launch, so that the
                                      // observation streams of two handles can be co-resident (shared memory) instead of taking turns
  int host_early;                     // BSB_HOST_EARLY (default 1): two-phase host steps (scalars first) where the family allows
  bool early_inflight;                // a two-phase host step may still be streaming observations on copy_stream
  int host_stage_actions;             // BSB_HOST_STAGE_ACTIONS (default 1): two-phase steps get their actions by DMA on a side stream instead of reading them in place
  cudaStream_t h2d_stream; cudaEvent_t h2d_event;
};

namespace bsb {
// One entry per family, each defined in its own translation unit (fam_<name>.cu).
int run_deep_sea(bsb_env*, const LaunchArgs&, cudaStream_t);
int run_catch(bsb_env*, const LaunchArgs&, cudaStream_t);
int run_cartpole(bsb_env*, const LaunchArgs&, cudaStream_t);
int run_cartpole_swingup(bsb_env*, const LaunchArgs&, cudaStream_t);
int run_mountain_car(bsb_env*, const LaunchArgs&, cudaStream_t);
int run_memory_chain(bsb_env*, const LaunchArgs&, cudaStream_t);
int run_bandit(bsb_env*, const LaunchArgs&, cudaStream_t);
int run_umbrella_chain(bsb_env*, const LaunchArgs&, cudaStream_t);
int run_discounting_chain(bsb_env*, const LaunchArgs&, cudaStream_t);
int run_mnist(bsb_env*, const LaunchArgs&, cudaStream_t);
}  // namespace bsb
