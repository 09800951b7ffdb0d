// Host path and kernel launch, instantiated once per family (fam_<name>.cu).
#pragma once
#include "bsb_env.h"

namespace bsb {

// --------------------------- host path --------------------------------------
template <class F> struct HostEmit {
  template <class R> static void run(const EnvParams& p, const typename F::Lane& L, R&, float* dst) { F::row(p, L, dst, 1); }
};
template <> struct HostEmit<UmbrellaChain> {
  template <class R> static void run(const EnvParams& p, const UmbrellaChain::Lane& L, R& r, float* dst) { UmbrellaChain::row(p, L, r, dst, 1); }
};
template <> struct HostEmit<DeepSea> {
  template <class R> static void run(const EnvParams& p, const DeepSea::Lane& L, R&, float* dst) {
    for (int e = 0; e < p.obs_numel; ++e) dst[e] = 0.f;
    if (L.hot >= 0) dst[L.hot] = 1.f;
  }
};
template <> struct HostEmit<Catch> {
  template <class R> static void run(const EnvParams& p, const Catch::Lane& L, R&, float* dst) {
    for (int e = 0; e < p.obs_numel; ++e) dst[e] = 0.f;
    dst[L.hot_a] = 1.f; dst[L.hot_b] = 1.f;
  }
};
template <> struct HostEmit<Mnist> {
  template <class R> static void run(const EnvParams& p, const Mnist::Lane& L, R&, float* dst) {
    if (L.image < 0) { for (int e = 0; e < p.obs_numel; ++e) dst[e] = 0.f; return; }
    const int8_t* src = p.images + (int64_t)L.image * p.obs_numel;
    for (int e = 0; e < p.obs_numel; ++e) dst[e] = Mnist::pixel(src[e]);
  }
};

template <class F, int RK>
void host_run(const EnvParams& p, const LaunchArgs& a) {
  typedef typename RngOf<RK>::type R;
  const int64_t B = p.batch;
  const int K = p.obs_numel;
  const bool noise = p.wrapper == BSB_WRAP_REWARD_NOISE;
  const bool has_rng = p.rng_pos != nullptr;
  const bool track = p.ep != nullptr;
  for (int64_t lane = 0; lane < B; ++lane) {
    typename F::Lane L;
    R rng, wrng;
    EpisodeStats ep;
    ActionStream action_stream;
    action_stream.open();
    if (a.mode == MODE_INIT) F::init(p, L); else F::load(p, lane, L);
    if (has_rng) rng_open(rng, p, lane, false);
    if (noise) rng_open(wrng, p, lane, true);
    if (track) ep.load(p, lane);
    if (a.mode == MODE_INIT) {
      F::ctor_draws(p, L, rng);
      F::store(p, lane, L);
      if (has_rng) rng_close(rng, p, lane, false);
      continue;
    }
    for (int64_t t = 0; t < a.T; ++t) {
      const int64_t off = t * B + lane;
      int32_t action = 0;
      if (a.mode == MODE_STEP) {
        action = a.actions ? a.actions[off]
                           : action_stream.sample(a.action_seed, p.lane_offset + (uint64_t)lane, (uint64_t)(a.step0 + t), p.num_actions);
        if (a.actions_out) a.actions_out[off] = action;
      }
      const bool after_last = L.nr != 0;
      const StepOut o = lane_transition<F, R, R>(p, lane, L, rng, wrng, action, a.mode, noise);
      if (track) {
        ep.track(p, lane, o, a.step0 + t, after_last);
        if (p.log_next && o.step_type == LAST && log_row_due(p, lane)) {
          F::store(p, lane, L); ep.store(p, lane);
          log_point_record(p, lane, a.step0 + t + 1);
        }
      }
      if (a.reward) a.reward[off] = (float)o.reward;
      if (a.reward_f64) a.reward_f64[off] = o.reward;
      if (a.discount) a.discount[off] = o.discount;
      if (a.step_type) a.step_type[off] = o.step_type;
      HostEmit<F>::run(p, L, rng, a.obs + off * (int64_t)K);
    }
    F::store(p, lane, L);
    if (has_rng) rng_close(rng, p, lane, false);
    if (noise) rng_close(wrng, p, lane, true);
    if (track) ep.store(p, lane);
  }
}

// --------------------------- device dispatch --------------------------------
template <class F, int RK, bool kNoise, bool kTrack>
int device_launch(bsb_env* e, LaunchArgs a, cudaStream_t stream) {
  const int K = e->p.obs_numel;
  const bool is_onehot = EmitKind<F>::value == EMIT_ONEHOT;
  const bool is_image = EmitKind<F>::value == EMIT_IMAGE;
  const int64_t B = e->p.batch;
  a.emit_bulk = is_onehot ? e->deep_sea_bulk : e->emit_bulk;
  a.group_lanes = 1;
  a.work_counter = nullptr;
  a.work_base = 0;
  a.lazy_fetch = e->lazy_fetch;
  a.l2_hint = e->l2_hint;
  // Row / board stages per warp: two (the next row block is rendered while the TMA unit still reads the previous
  // one) unless that costs resident warps -- 16 warps per SM fit the register budget, so a warp can afford
  // ~14 KB of shared memory.  umbrella_distract (103-float rows, 13 KB per stage) ran 7 warps per SM with two
  // stages (profiles/r02a_family_ncu_metrics.csv) and is bound by integer-multiply latency, not by the store.
  a.stage_rows = ((size_t)2 * 32 * (size_t)K * sizeof(float) <= 14 * 1024) ? 2 : 1;
  // A single-step launch gives every warp exactly one row block to emit: the second stage would only be zeroed
  // (catch) and hold shared memory that another CTA could use.
  if (a.T == 1 && (EmitKind<F>::value == EMIT_ROWS || EmitKind<F>::value == EMIT_TWOHOT)) a.stage_rows = 1;
  a.cta_extra_floats = 0;
  a.bad_action = e->bad_action_dev;
  // Lanes per chunk.  The image emitter walks the chunk's lanes a few 3 KB tiles at a time, so it is bound by how
  // many warps share the batch: keep >= 4 warps per SM by halving the chunk (down to 8 lanes) when 32-lane chunks
  // would not.  Measured at 4 096 lanes (rollout us/step, 32-lane vs 8-lane chunks): mnist 14.8 -> 4.2; the deep_sea
  // bulk path gets WORSE (N = 32: 2.4 -> 3.5, N = 50: 5.6 -> 6.0 -- fewer, larger TMA stores win), so it keeps 32.
  int chunk = 32;
  if (is_image)
    while (chunk > 8 && (B + chunk - 1) / chunk < 4 * (int64_t)e->num_sms) chunk >>= 1;
  if (e->chunk_lanes > 0) chunk = e->chunk_lanes;
  a.chunk_lanes = chunk;
  const int64_t n_chunks = (B + chunk - 1) / chunk;
  int threads = e->block_threads;
  bool persistent = false;
  const size_t tile = (size_t)K * 4;
  if (is_onehot && a.emit_bulk) {
    // Lanes per bulk store: the largest power of two <= 16 with one store <= 40 KB (BSB_DEEP_SEA_GROUP overrides).
    // Measured on B200 (tools/bench_variants.py): N = 32 -> 8 lanes (32 KB stores), N = 50 -> 4 lanes (40 KB).
    int m = 1;
    while (m < 16 && (size_t)(2 * m) * tile <= 40 * 1024) m <<= 1;
    if (e->deep_sea_group > 0) m = e->deep_sea_group;
    if (a.phase == 2 && e->split_group > 0) m = e->split_group;      // observation-only launch of a split host step
    if (m > chunk) m = chunk;               // a group never spans chunks
    if (((size_t)m * tile) % 16 != 0 || (size_t)TILE_STAGES * m * tile > 100 * 1024) {
      a.emit_bulk = 0;                      // tiles too large (or misaligned) for the staged path: vector stores
    } else {
      a.group_lanes = m; threads = 32; persistent = e->deep_sea_persistent != 0;
    }
  }
  if (is_image && a.emit_bulk) {
    // mnist through the TMA unit: groups of m tiles staged in shared memory + mz all-zero tiles per CTA for the LAST
    // frames.  16-byte image loads need K % 16 == 0 (28 x 28 = 784 is).  Defaults (BSB_IMAGE_STAGES, BSB_IMAGE_GROUP):
    // ONE staging buffer of m = 2 tiles per warp (6 KB) in 128-thread CTAs with mz = 8 zero tiles (25 KB, shared by
    // the CTA's warps): 50 KB per CTA -> 4 CTAs = 16 warps per SM, the register limit.  The pixel conversion is
    // issue-bound, so resident warps matter more than overlapping a warp's own fill with its own store (other
    // warps fill that gap) or than the size of the staged stores; the zero frames still leave in 25 KB stores.
    const int stages = e->image_stages;
    int m = e->image_group;
    while (m > 1 && (size_t)stages * m * tile > 28 * 1024) m >>= 1;
    if (m > chunk) m = chunk;
    int mz = 8;
    while (mz > 1 && ((size_t)mz * tile > 28 * 1024 || mz > chunk)) mz >>= 1;
    if (mz < m) mz = m;
    if ((K & 15) != 0 || (size_t)stages * m * tile > 64 * 1024) {
      a.emit_bulk = 0;
    } else {
      a.group_lanes = m; a.stage_rows = stages; threads = 128; a.cta_extra_floats = mz * K; persistent = e->deep_sea_persistent != 0;
      if (n_chunks < 2 * (int64_t)e->num_sms) threads = 64;      // small batches: more, smaller CTAs
    }
  }
  a.use_pdl = (e->use_pdl && !a.no_pdl && a.mode == MODE_STEP && a.T == 1) ? 1 : 0;
  if (a.phase == 1) {
    // transitions-only launch of a split host step: no emitter, no shared memory (so that it is co-resident with the
    // observation stream of ANOTHER handle), one chunk per warp
    a.emit_bulk = 0; a.stage_rows = 0; a.cta_extra_floats = 0; a.group_lanes = 1; threads = 128; persistent = false;
  }
  size_t per_warp = smem_floats_per_warp<F>(K, a.emit_bulk != 0, a.group_lanes, a.stage_rows) * sizeof(float);
  if ((EmitKind<F>::value == EMIT_ROWS || EmitKind<F>::value == EMIT_TWOHOT) && per_warp > 96 * 1024) {
    // rows / boards too long for a per-warp stage (catch boards beyond ~19 x 20 cells, umbrella_chain with more than
    // ~380 distractors): boards fall back to shuffle-rendered vector stores, rows are rendered in place
    a.emit_bulk = 0; a.stage_rows = 0; per_warp = 0;
  }
  const size_t cta_extra = (size_t)a.cta_extra_floats * sizeof(float);
  size_t smem = per_warp * (size_t)(threads / 32) + cta_extra;
  while (smem > 96 * 1024 && threads > 32) { threads >>= 1; smem = per_warp * (size_t)(threads / 32) + cta_extra; }
  if (smem > 200 * 1024) return fail(BSB_UNSUPPORTED, "observation too large for the staged emitter");
  auto kernel = transition_kernel<F, RK, kNoise, kTrack>;
  if (smem > 48 * 1024) BSB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int64_t grid = (n_chunks + threads / 32 - 1) / (threads / 32);
  // Two-phase host step: the first blocks are COPIERS (they ship the staged scalars to the host, then join phase 2):
  // enough of them for ~512 threads, i.e. ~64 KB of 16-byte loads in flight.
  const bool two_phase = a.early_scalars != 0 && a.mailbox != nullptr;
  const int copiers = two_phase ? (512 / threads > 1 ? 512 / threads : 1) : 0;
  a.early_scalars = copiers;
  grid += copiers;
  if (persistent) {
    // As many CTAs as are co-resident (shared-memory bound; 1 KB per CTA is reserved by the driver); their warps
    // draw chunks from the environment's global counter.
    int64_t per_sm = (int64_t)((227 * 1024) / (smem + 1024));
    per_sm = per_sm < 1 ? 1 : (per_sm > 16 ? 16 : per_sm);
    // observation-only launch of a split host step: leave room for ANOTHER handle's observation stream on every SM
    if (a.phase == 2 && e->split_ctas_per_sm > 0 && per_sm > e->split_ctas_per_sm) per_sm = e->split_ctas_per_sm;
    const int64_t resident = (int64_t)e->num_sms * per_sm;
    if (grid > resident) {
      grid = resident;
      a.work_counter = a.clock ? a.clock + CLOCK_CHUNK : e->work_counter;
      a.work_base = a.clock ? 0ull : e->work_base;
    } else {
      persistent = false;      // everything is resident anyway: one chunk per warp
    }
  }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3((unsigned)threads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  if (a.use_pdl) {
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
  }
  BSB_CUDA(cudaLaunchKernelEx(&cfg, kernel, e->p, a));
  // chunks [warps, n_chunks) are fetched once each and every warp makes exactly one failing fetch
  // (graph-safe mode: the last CTA zeroes the counter instead)
  if (a.work_counter && !a.clock) e->work_base += (unsigned long long)n_chunks + (unsigned long long)(copiers * (threads / 32));
  g_launches.fetch_add(1, std::memory_order_relaxed);
  return BSB_OK;
}

template <class F, int RK>
int device_launch_flags(bsb_env* e, const LaunchArgs& a, cudaStream_t stream) {
  const bool noise = e->p.wrapper == BSB_WRAP_REWARD_NOISE && a.mode != MODE_INIT;
  const bool track = e->p.ep != nullptr && a.mode != MODE_INIT;
  if (noise) return track ? device_launch<F, RK, true, true>(e, a, stream) : device_launch<F, RK, true, false>(e, a, stream);
  return track ? device_launch<F, RK, false, true>(e, a, stream) : device_launch<F, RK, false, false>(e, a, stream);
}

template <class F>
int run_family(bsb_env* e, const LaunchArgs& a, cudaStream_t stream) {
  const bool mt = e->p.rng_kind == BSB_RNG_MT19937;
  if (e->device < 0) {
    if (mt) host_run<F, 1>(e->p, a); else host_run<F, 0>(e->p, a);
    return BSB_OK;
  }
  return mt ? device_launch_flags<F, 1>(e, a, stream) : device_launch_flags<F, 0>(e, a, stream);
}

}  // namespace bsb
