// Fused transition kernels: one per environment family (template F), specialised
// on the bit source (Philox / MT19937), on whether the RewardNoise wrapper stream
// is live, and on whether the Logging accumulators are tracked.
//
// Thread = lane for the scalar transition (state word(s), action, reward,
// discount, step_type are coalesced 4/8-byte accesses).  Observations are dense
// float32 tensors that must be written fresh every step (the reference allocates
// a new array per step: deep_sea.py:104, catch.py:114); they are the HBM traffic
// that bounds the kernel and are emitted WARP-COOPERATIVELY:
//
//   * row families ((1,k) vectors): each thread renders its row into a per-warp
//     shared-memory stage (double buffered); the warp's [32, k] block is
//     contiguous in global memory, so one elected lane sends it with a single TMA
//     bulk store (cp.async.bulk shared::cta -> global).
//   * catch: the same stage holds the warp's 32 boards and stays ZERO between
//     steps; each thread only un-pokes its two old cells and pokes its two new
//     ones before the elected lane issues the bulk store of all 32 boards.
//   * deep_sea (N x N one-hot tile per lane, 4 KB at N = 32): per warp two staging buffers of m zeroed tiles
//     (m = 8 at N = 32); the threads of a group poke their lanes' hot cells (un-poking what they poked into that
//     buffer two stores ago) and the elected lane issues ONE bulk store of the m contiguous tiles (32 KB).
//     Large stores matter: the TMA unit costs ~70 ns + bytes / 64 GB/s per SM, so 4 KB stores cap the chip at
//     ~4.6 TB/s while 32 KB stores reach the HBM write ceiling.  Unaligned tiles (odd N) use 16-byte streaming
//     stores instead: the warp walks its lanes, every thread writes part of each lane's tile, the hot cell
//     chosen per float4 from a descriptor broadcast by __shfl_sync.
//   * mnist: groups of 4 gathered int8 images -> float32 tiles in shared memory -> one bulk store; the all-zero
//     LAST frames of a group leave as one bulk store from zero tiles the CTA's warps share.
//
// A launch covers T consecutive steps with lane state held in registers (T = 1
// for bsb_step); actions come from the caller or from the on-device Philox
// action stream.  Host-driven steps (bsb_step_host) signal completion through a
// pinned mailbox and, for deep_sea, run in two phases (all transitions first, the
// scalars shipped to the host by a few copier blocks, then the observations).  With use_pdl the kernel is launched with programmatic stream
// serialization: everything before griddepcontrol.wait (index math, zeroing the
// shared-memory stages) overlaps the tail of the previous step's kernel.
#pragma once
#include "bsb_families.cuh"

namespace bsb {

// Caller-owned buffers of one step (launch arguments, or the fields of the host mailbox below).
struct MailFields {
  const int32_t* actions; float* obs; float* reward; double* reward_f64; float* discount; int32_t* step_type;
  int32_t obs_vec_ok, pad;
};

struct LaunchArgs {
  const int32_t* actions;   // [T,B] or null (sample on device)
  int32_t* actions_out;     // [T,B] or null
  float* obs;               // [T,B,K]
  float* reward;            // [T,B] or null
  double* reward_f64;       // [T,B] or null
  float* discount;          // [T,B] or null
  int32_t* step_type;       // [T,B] or null
  int64_t T;
  int64_t step0;            // global index of the first step of this launch
  uint64_t action_seed;
  int32_t mode;             // 0 = step, 1 = reset every lane, 2 = constructor init
  int32_t obs_vec_ok;       // obs base and per-step stride are 16-byte aligned
  int32_t emit_bulk;        // use TMA bulk stores where the emitter supports them
  int32_t use_pdl;          // launched with programmatic stream serialization
  int32_t group_lanes;      // deep_sea bulk path: lanes per bulk store (power of two, 1..32)
  int32_t lazy_fetch;       // persistent launches: 1 = fetch the next chunk only when the current one is issued
  int32_t l2_hint;          // L2 policy of the observation bulk stores: 0 none, 1 evict_first (default), 2 evict_last
  unsigned long long* work_counter;  // persistent launches: monotonically increasing chunk counter (device)
  unsigned long long work_base;      // value of *work_counter at which this launch's chunk 0 starts
  // Device clock (graph-safe mode, see the kernel): {steps advanced in this mode, chunk counter, finished CTAs}.
  // Null in the default mode, where `step0` / `work_base` arrive as launch arguments from the host's counters.
  unsigned long long* clock;
  int32_t no_pdl;           // set while the stream is being captured
  int32_t chunk_lanes;      // lanes per chunk (= per warp pass): 32, or 16 / 8 when the batch would under-fill the SMs
  int32_t stage_rows;       // row / board emitters: number of [32, K] shared-memory stages per warp (2: double buffered;
                            // 1: long rows, where a second stage would cost resident warps; 0: straight to global memory)
  int32_t cta_extra_floats; // shared memory after the per-warp stages (mnist bulk path: the CTA's all-zero tiles)
  // Host-driven steps (bsb_step_host, pinned buffers): completion is signalled through a pinned mailbox; with
  // BSB_HOST_PRELAUNCH the launch is even enqueued BEFORE its inputs exist and waits for the host to ring
  // `ticket`, taking pointers and actions from the mailbox.
  struct HostMailbox* mailbox;       // pinned host memory, device alias (null: ordinary launch).  The last CTA to
                                     // finish stores `done = ticket` there: the host spins on it instead of
                                     // paying a stream synchronise.
  struct DeviceMail* mail;           // device memory: doorbell relay + finished-CTA counter
  unsigned long long ticket;
  int32_t early_scalars;             // > 0: two-phase host step; the value is the number of COPIER blocks (blocks
                                     // [0, n) own no chunks at first: they ship the scalars to the host, see below)
  MailFields stage;                  // two-phase: device staging of reward / reward_f64 / discount / step_type
  int32_t timing;                    // BSB_HOST_TIMING: leave %globaltimer stamps in the mailbox
  int32_t wait_doorbell;             // 1: pre-launched -- poll the doorbell for `ticket`, then take the buffers from the mailbox
  unsigned long long doorbell_timeout_ns;
  int32_t* bad_action;      // pinned host flag (device alias): set to 1 when an action is outside [0, num_actions)
  int32_t phase;            // two-phase host step split over TWO launches (BSB_HOST_NO_WAIT): 1 = transitions + copiers
                            // only (no shared memory: co-resident with another handle's observation stream),
                            // 2 = observations only (waits for mail->phase1 == ticket, not for launch 1 to END); 0 = one launch
};

// Host <-> device mailbox of the doorbell mode.  The host fills `in` and then stores `doorbell = ticket` (release
// order); block 0 of the waiting launch polls it over PCIe, copies `in` to device memory and relays the ticket to the
// other blocks through L2.  The last block to finish stores `done = ticket` after a system-scope fence, so every
// output written to host memory (reward / discount / step_type, zero-copy) is visible when the host sees it.
static const unsigned long long MAIL_CANCEL = 1ull << 63;      // doorbell: skip the step; done: the step was skipped
struct HostMailbox {
  volatile unsigned long long doorbell;   // host -> device, word 0 of the line the device polls
  MailFields in;                          // words 1..7 of the same 64-byte line
  unsigned long long pad0[8];
  volatile unsigned long long done;     unsigned long long pad1[7];     // device -> host, a line of its own
  // BSB_HOST_TIMING=1 (tools/e2e_timeline.py): %globaltimer stamps of the latest two-phase launch, written by its
  // signaller before `done`: [0] block 0 past the dependency wait, [1] phase 1 complete on every block, [2] just
  // before `done`, [3] the latest exit of any block of the PREVIOUS launch
  volatile unsigned long long stamp[8];
};
static_assert(sizeof(MailFields) == 56, "doorbell + fields must fill exactly one 64-byte line");
struct DeviceMail {
  volatile unsigned long long relay;      // ticket (| MAIL_CANCEL) most recently taken from the host doorbell
  unsigned long long last_exit;           // BSB_HOST_TIMING: max %globaltimer at which a block of the latest launch left
  unsigned long long finished;            // blocks of the current launch that have finished (phase 1, if two-phase)
  volatile unsigned long long phase1;     // ticket of the latest two-phase launch whose phase 1 is complete
  unsigned long long copied;              // copier blocks of the current two-phase launch that have shipped their share
  MailFields in;                          // the host's fields, copied once per launch by block 0
};

enum { MODE_STEP = 0, MODE_RESET = 1, MODE_INIT = 2 };

// ----- RNG plumbing ---------------------------------------------------------
template <int RK> struct RngOf;
template <> struct RngOf<0> { typedef LegacyRng<PhiloxSrc> type; };
template <> struct RngOf<1> { typedef LegacyRng<MtSrc> type; };

BSB_HD void rng_open(LegacyRng<PhiloxSrc>& r, const EnvParams& p, int64_t i, bool wrapper) {
  const uint64_t packed = wrapper ? p.wrng_pos[i] : p.rng_pos[i];
  r.src.open(p.seed, p.lane_offset + (uint64_t)i, wrapper ? STREAM_WRAPPER : STREAM_ENV, packed);
  r.g.has = (packed & RNG_HASGAUSS) ? 1 : 0;
  const double* gz = wrapper ? p.wrng_gauss : p.rng_gauss;
  r.g.value = (r.g.has && gz) ? gz[i] : 0.0;
}
BSB_HD void rng_close(const LegacyRng<PhiloxSrc>& r, const EnvParams& p, int64_t i, bool wrapper) {
  const uint64_t packed = r.src.packed() | (r.g.has ? RNG_HASGAUSS : 0ull);
  if (wrapper) p.wrng_pos[i] = packed; else p.rng_pos[i] = packed;
  double* gz = wrapper ? p.wrng_gauss : p.rng_gauss;
  if (gz && r.g.has) gz[i] = r.g.value;
}
BSB_HD void rng_open(LegacyRng<MtSrc>& r, const EnvParams& p, int64_t i, bool wrapper) {
  const int64_t stride = (p.batch > 0) ? p.batch : 1;
  r.src.open((wrapper ? p.wmt_key : p.mt_key) + i, stride, (wrapper ? p.wmt_idx : p.mt_idx)[i]);
  const uint64_t packed = wrapper ? p.wrng_pos[i] : p.rng_pos[i];
  r.g.has = (packed & RNG_HASGAUSS) ? 1 : 0;
  const double* gz = wrapper ? p.wrng_gauss : p.rng_gauss;
  r.g.value = (r.g.has && gz) ? gz[i] : 0.0;
}
BSB_HD void rng_close(const LegacyRng<MtSrc>& r, const EnvParams& p, int64_t i, bool wrapper) {
  (wrapper ? p.wmt_idx : p.mt_idx)[i] = r.src.idx;
  const uint64_t packed = r.g.has ? RNG_HASGAUSS : 0ull;
  if (wrapper) p.wrng_pos[i] = packed; else p.rng_pos[i] = packed;
  double* gz = wrapper ? p.wrng_gauss : p.rng_gauss;
  if (gz && r.g.has) gz[i] = r.g.value;
}

// ----- the per-lane call sequence of base.Environment.step (base.py:59-65) --
// followed by the reward wrappers (utils/wrappers.py:275-283, 338-346), which
// act on every non-FIRST timestep; bsuite_info() stays un-noised / un-scaled.
template <class F, class R, class WR>
BSB_HD StepOut lane_transition(const EnvParams& p, int64_t i, typename F::Lane& L, R& rng, WR& wrng,
                               int32_t action, int32_t mode, bool noise) {
  StepOut o;
  if (mode == MODE_RESET || L.nr) {        // `if self._reset_next_step: return self.reset()`
    o = F::reset(p, i, L, rng);
    L.nr = 0;
  } else {
    o = F::step(p, i, L, action, rng);
    L.nr = (o.step_type == LAST) ? 1u : 0u;
    if (noise) { o.reward = o.reward + p.noise_scale * wrng.randn(); }
    else if (p.wrapper == 2) { o.reward = o.reward * p.reward_scale; }
  }
  return o;
}

// Observation emitter of each family.
static const int EMIT_ROWS = 0, EMIT_ONEHOT = 1, EMIT_TWOHOT = 2, EMIT_IMAGE = 3;
// Families whose observation is a pure function of the STORED lane state (F::describe after F::load): their
// host-driven steps can deliver the scalars before the observation is streamed (two-phase host step).
template <class F> struct ObsFromState { static const bool value = false; };
template <> struct ObsFromState<DeepSea> { static const bool value = true; };
template <> struct ObsFromState<Catch> { static const bool value = true; };
template <class F> struct EmitKind { static const int value = EMIT_ROWS; };
template <> struct EmitKind<DeepSea> { static const int value = EMIT_ONEHOT; };
template <> struct EmitKind<Catch> { static const int value = EMIT_TWOHOT; };
template <> struct EmitKind<Mnist> { static const int value = EMIT_IMAGE; };
static const int ROW_STAGES = 2;      // at most: double-buffered [32, K] stage per warp (LaunchArgs::stage_rows)
static const int TILE_STAGES = 2;     // deep_sea bulk path: double-buffered groups of `group_lanes` tiles per warp

// Dynamic shared memory per warp, in floats.
template <class F> inline
#if defined(__CUDACC__)
__host__ __device__
#endif
size_t smem_floats_per_warp(int K, bool emit_bulk, int group_lanes, int row_stages) {
  if (EmitKind<F>::value == EMIT_ROWS || EmitKind<F>::value == EMIT_TWOHOT) return (size_t)row_stages * 32 * (size_t)K;
  if (EmitKind<F>::value == EMIT_ONEHOT && emit_bulk) return (size_t)TILE_STAGES * (size_t)group_lanes * (size_t)K;
  if (EmitKind<F>::value == EMIT_IMAGE)                    // int8 pixel -> float32 table (+ two staging buffers of m tiles)
    return 256 + (emit_bulk ? (size_t)row_stages * (size_t)group_lanes * (size_t)K : 0);
  return 0;
}

#if defined(__CUDACC__)

__device__ __forceinline__ void st_stream(float4* dst, float4 v) { __stcs(dst, v); }
__device__ __forceinline__ void st_stream(float* dst, float v) { __stcs(dst, v); }

// ----- TMA bulk store (shared::cta -> global) and PDL primitives --------------
__device__ __forceinline__ void bulk_store_s2g(void* gdst, const void* ssrc, uint32_t bytes) {
  const uint32_t s = (uint32_t)__cvta_generic_to_shared(ssrc);
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(s), "r"(bytes) : "memory");
}
// Same store with an L2 eviction-priority hint (policy from createpolicy.fractional.L2::evict_first / evict_last).
__device__ __forceinline__ void bulk_store_s2g_hint(void* gdst, const void* ssrc, uint32_t bytes, uint64_t policy) {
  const uint32_t s = (uint32_t)__cvta_generic_to_shared(ssrc);
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;" ::"l"(gdst), "r"(s), "r"(bytes), "l"(policy) : "memory");
}
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t p; asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p)); return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
  uint64_t p; asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p)); return p;
}
// Bulk store with the launch's L2 policy: observations are written once and never re-read by this kernel, so they
// are marked evict_first (default) -- measured 43.9 -> 40.8 us/step on the headline kernel (evict_last: 44.8).
__device__ __forceinline__ void bulk_store_obs(void* gdst, const void* ssrc, uint32_t bytes, int l2_hint) {
  if (l2_hint == 1) bulk_store_s2g_hint(gdst, ssrc, bytes, l2_policy_evict_first());
  else if (l2_hint == 2) bulk_store_s2g_hint(gdst, ssrc, bytes, l2_policy_evict_last());
  else bulk_store_s2g(gdst, ssrc, bytes);
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ----- vector-store emitters ---------------------------------------------------
// One-hot tiles: `hot` is the flat index of the single 1.0 (or -1: all zeros).
__device__ __forceinline__ void emit_onehot_vec(float* obs_t, int64_t warp_base, int n_lanes, int K, int hot, bool vec) {
  const int tid = threadIdx.x & 31;
  if (vec) {
    const int K4 = K >> 2;
    for (int j = 0; j < n_lanes; ++j) {
      const int h = __shfl_sync(0xffffffffu, hot, j);
      const int hq = h >> 2, hc = h & 3;
      float4* dst = reinterpret_cast<float4*>(obs_t + (warp_base + j) * (int64_t)K);
#pragma unroll 8
      for (int q = tid; q < K4; q += 32) {
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (q == hq) { if (hc == 0) v.x = 1.f; else if (hc == 1) v.y = 1.f; else if (hc == 2) v.z = 1.f; else v.w = 1.f; }
        st_stream(dst + q, v);
      }
    }
  } else {
    for (int j = 0; j < n_lanes; ++j) {
      const int h = __shfl_sync(0xffffffffu, hot, j);
      float* dst = obs_t + (warp_base + j) * (int64_t)K;
      for (int e = tid; e < K; e += 32) st_stream(dst + e, e == h ? 1.f : 0.f);
    }
  }
}

// Boards with up to two hot cells; the warp's boards form one contiguous span.
__device__ __forceinline__ void emit_twohot_vec(float* obs_t, int64_t warp_base, int n_lanes, int K, int hot_a, int hot_b, bool vec) {
  const int tid = threadIdx.x & 31;
  const int total = n_lanes * K;
  float* dst = obs_t + warp_base * (int64_t)K;
  if (vec && (total & 3) == 0) {
    const int total4 = total >> 2;
    for (int q0 = 0; q0 < total4; q0 += 32) {
      const int q = q0 + tid;
      const int e0 = (q < total4 ? q : 0) << 2;
      int j = e0 / K, c = e0 - j * K;
      float v[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int jj = j < 32 ? j : 31;
        const int a = __shfl_sync(0xffffffffu, hot_a, jj);
        const int b = __shfl_sync(0xffffffffu, hot_b, jj);
        v[k] = (c == a || c == b) ? 1.f : 0.f;
        if (++c >= K) { c = 0; ++j; }
      }
      if (q < total4) st_stream(reinterpret_cast<float4*>(dst) + q, make_float4(v[0], v[1], v[2], v[3]));
    }
  } else {
    for (int e0 = 0; e0 < total; e0 += 32) {
      const int e = e0 + tid;
      const int ee = e < total ? e : 0;
      const int j = ee / K, c = ee - j * K;
      const int a = __shfl_sync(0xffffffffu, hot_a, j);
      const int b = __shfl_sync(0xffffffffu, hot_b, j);
      if (e < total) st_stream(dst + e, (c == a || c == b) ? 1.f : 0.f);
    }
  }
}

// Image tiles gathered from the int8 dataset (`image` < 0: zeros).  `lut` is the warp's 256-entry table of
// (float)(int8)i / 255 in shared memory: IEEE float division costs ~10 instructions and takes a slow path for zero
// numerators (most MNIST pixels), a table lookup costs one LDS.  The gather is latency-bound if each load ->
// convert -> store chain runs serially, so all loads of a pass (8 x 32 char4 = 1 024 pixels) are issued first.
__device__ __forceinline__ void emit_image(const EnvParams& p, const float* lut, float* obs_t, int64_t warp_base, int n_lanes, int K, int image, bool vec) {
  const int tid = threadIdx.x & 31;
  constexpr int U = 8;
  for (int j = 0; j < n_lanes; ++j) {
    const int img = __shfl_sync(0xffffffffu, image, j);
    float* dst = obs_t + (warp_base + j) * (int64_t)K;
    const int8_t* src = p.images + (int64_t)(img < 0 ? 0 : img) * K;
    if (vec) {
      const int K4 = K >> 2;
      const uchar4* src4 = reinterpret_cast<const uchar4*>(src);
      float4* dst4 = reinterpret_cast<float4*>(dst);
      if (img < 0) {
        for (int q = tid; q < K4; q += 32) st_stream(dst4 + q, make_float4(0.f, 0.f, 0.f, 0.f));
        continue;
      }
      for (int q0 = 0; q0 < K4; q0 += 32 * U) {
        uchar4 c[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int q = q0 + u * 32 + tid;
          c[u] = make_uchar4(0, 0, 0, 0);
          if (q < K4) c[u] = __ldg(src4 + q);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int q = q0 + u * 32 + tid;
          if (q < K4) st_stream(dst4 + q, make_float4(lut[c[u].x], lut[c[u].y], lut[c[u].z], lut[c[u].w]));
        }
      }
    } else {
      for (int e = tid; e < K; e += 32) st_stream(dst + e, img >= 0 ? lut[(uint8_t)src[e]] : 0.f);
    }
  }
}

// image.astype(float32) / 255 (mnist.py:64) without a table, an IEEE division or an int->float conversion (I2F runs
// on the quarter-rate XU pipe): per pixel one PRMT (sign-extended byte: the reference parses images as INT8,
// utils/datasets.py:55-56), one IADD + one FADD (v as float through the 1.5 * 2^23 magic number, exact for
// |v| <= 128), then the quotient as fma(v, hi, v * lo) with hi + lo = 1/255 split into two floats.  That is the
// correctly rounded v / 255 for every int8 v: checked exhaustively against numpy on the device
// (tests/test_round2_features.py) -- 256 inputs, no reasoning about rounding needed.
__device__ __forceinline__ float pixel_div255(uint32_t word, int byte) {
  // prmt.b32: bit 3 of a selector nibble replicates the sign of the selected byte (the __byte_perm intrinsic masks
  // that bit off): byte `byte` in the low byte, its sign in the three bytes above = the sign-extended int8
  const uint32_t sel = (uint32_t)byte | ((8u | (uint32_t)byte) << 4) | ((8u | (uint32_t)byte) << 8) | ((8u | (uint32_t)byte) << 12);
  int v;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(v) : "r"(word), "r"(0u), "r"(sel));
  const float x = __fadd_rn(__int_as_float(0x4B400000 + v), -12582912.0f);
  const float hi = 0.003921568859368563f, lo = -2.319175823606301e-10f;      // float(1/255), float(1/255 - hi)
  return __fmaf_rn(x, hi, __fmul_rn(x, lo));
}
__device__ __forceinline__ float4 pixels4(uint32_t w) {
  return make_float4(pixel_div255(w, 0), pixel_div255(w, 1), pixel_div255(w, 2), pixel_div255(w, 3));
}

// Image tiles through shared memory and the TMA unit (K % 16 == 0, e.g. 28 x 28).  The chunk's lanes are walked in
// blocks of `mz` consecutive lanes (= mz contiguous tiles in global memory):
//   * a block whose lanes all show the all-zero LAST frame (mnist.py:74; every other step of every lane) is ONE
//     bulk store of mz tiles (25 KB at mz = 8) from the CTA's zero tiles -- nothing is staged, nothing waited for;
//   * otherwise the block goes in groups of `m` (<= 4) lanes: all 16-byte loads of the group's int8 images (49 per
//     28 x 28 tile) are issued before the first conversion, the float32 tiles land in a staging buffer and leave
//     as one bulk store of m * 4K bytes.
// stage = [256 floats: table of the vector path][stages x m x K floats]; `emitted` counts staged stores (buffer
// parity).  Small staging buffers (m = 2, one stage: 6 KB per warp) keep 16 warps per SM resident -- the conversion
// is issue-bound (ncu: 266 warp instructions per tile, 40 % issue utilisation at 8 warps per SM) -- while the
// zero frames, which are pure bandwidth, still leave in 25 KB stores.
__device__ __forceinline__ void emit_image_bulk(const EnvParams& p, float* stage, const float* cta_zero, float* obs_t,
                                                int64_t warp_base, int n_lanes, int K, int image, int m, int mz,
                                                int l2_hint, int stages, unsigned& emitted) {
  constexpr int MAXM = 4;
  const int tid = threadIdx.x & 31;
  float* tiles = stage + 256;
  const int K16 = K >> 4;
  const unsigned showing = __ballot_sync(0xffffffffu, image >= 0);
  for (int z0 = 0; z0 < n_lanes; z0 += mz) {
    const int in_block = (n_lanes - z0) < mz ? (n_lanes - z0) : mz;
    const unsigned block_mask = (in_block >= 32 ? 0xffffffffu : ((1u << in_block) - 1u));
    if (((showing >> z0) & block_mask) == 0u) {
      if (tid == 0) {
        bulk_store_obs(obs_t + (warp_base + z0) * (int64_t)K, cta_zero, (uint32_t)in_block * (uint32_t)K * 4u, l2_hint);
        bulk_commit();
      }
      continue;
    }
    for (int g0 = z0; g0 < z0 + in_block; g0 += m) {
      const int in_group = (z0 + in_block - g0) < m ? (z0 + in_block - g0) : m;
      float* dst = obs_t + (warp_base + g0) * (int64_t)K;
      const uint32_t bytes = (uint32_t)in_group * (uint32_t)K * 4u;
      float* buf = tiles + (size_t)(stages == 2 ? (emitted & 1u) : 0u) * m * K;
      // two staging buffers: at most the newest store may still be reading, never this buffer; one: none may
      if (tid == 0) { if (stages == 2) bulk_wait_read<1>(); else bulk_wait_read<0>(); }
      __syncwarp();
      int img[MAXM];
#pragma unroll
      for (int j = 0; j < MAXM; ++j) img[j] = __shfl_sync(0xffffffffu, image, (g0 + j) & 31);
      for (int q0 = 0; q0 < K16; q0 += 64) {
        uint4 c[MAXM][2];
#pragma unroll
        for (int j = 0; j < MAXM; ++j)
#pragma unroll
          for (int r = 0; r < 2; ++r) {
            const int q = q0 + r * 32 + tid;
            c[j][r] = make_uint4(0u, 0u, 0u, 0u);
            if (j < in_group && img[j] >= 0 && q < K16)
              c[j][r] = __ldg(reinterpret_cast<const uint4*>(p.images + (int64_t)img[j] * K) + q);
          }
#pragma unroll
        for (int j = 0; j < MAXM; ++j)
#pragma unroll
          for (int r = 0; r < 2; ++r) {
            const int q = q0 + r * 32 + tid;
            if (j < in_group && q < K16) {
              float4* out = reinterpret_cast<float4*>(buf + (size_t)j * K) + 4 * q;
              out[0] = pixels4(c[j][r].x); out[1] = pixels4(c[j][r].y);
              out[2] = pixels4(c[j][r].z); out[3] = pixels4(c[j][r].w);
            }
          }
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (tid == 0) { bulk_store_obs(dst, buf, bytes, l2_hint); bulk_commit(); }
      ++emitted;
    }
  }
}

// Stream the warp's staged [n_lanes, K] block with ordinary stores (ragged tail warps, unaligned buffers).
__device__ __forceinline__ void flush_rows_vec(const float* stage, float* obs_t, int64_t warp_base, int n_lanes, int K, bool vec) {
  const int tid = threadIdx.x & 31;
  const int total = n_lanes * K;
  float* dst = obs_t + warp_base * (int64_t)K;
  if (vec && (total & 3) == 0) {
    const float4* s4 = reinterpret_cast<const float4*>(stage);
    for (int q = tid; q < (total >> 2); q += 32) st_stream(reinterpret_cast<float4*>(dst) + q, s4[q]);
  } else {
    for (int e = tid; e < total; e += 32) st_stream(dst + e, stage[e]);
  }
}

// ----- per-family glue ------------------------------------------------------------
template <class F, class R> struct RowRenderer {
  static __device__ __forceinline__ void run(const EnvParams& p, const typename F::Lane& L, R&, float* dst) { F::row(p, L, dst, 1); }
};
template <class R> struct RowRenderer<UmbrellaChain, R> {   // the observation itself draws from the stream
  static __device__ __forceinline__ void run(const EnvParams& p, const UmbrellaChain::Lane& L, R& r, float* dst) { UmbrellaChain::row(p, L, r, dst, 1); }
};
template <class R> struct RowRenderer<DeepSea, R> { static __device__ __forceinline__ void run(const EnvParams&, const DeepSea::Lane&, R&, float*) {} };
template <class R> struct RowRenderer<Catch, R> { static __device__ __forceinline__ void run(const EnvParams&, const Catch::Lane&, R&, float*) {} };
template <class R> struct RowRenderer<Mnist, R> { static __device__ __forceinline__ void run(const EnvParams&, const Mnist::Lane&, R&, float*) {} };

template <class F> struct Descriptor {
  static __device__ __forceinline__ int a(const typename F::Lane&) { return -1; }
  static __device__ __forceinline__ int b(const typename F::Lane&) { return -1; }
};
template <> struct Descriptor<DeepSea> {
  static __device__ __forceinline__ int a(const DeepSea::Lane& L) { return L.hot; }
  static __device__ __forceinline__ int b(const DeepSea::Lane&) { return -1; }
};
template <> struct Descriptor<Catch> {
  static __device__ __forceinline__ int a(const Catch::Lane& L) { return L.hot_a; }
  static __device__ __forceinline__ int b(const Catch::Lane& L) { return L.hot_b; }
};
template <> struct Descriptor<Mnist> {
  static __device__ __forceinline__ int a(const Mnist::Lane& L) { return L.image; }
  static __device__ __forceinline__ int b(const Mnist::Lane&) { return -1; }
};

// ----- the fused transition kernel ----------------------------------------------
// Work unit: a CHUNK of 32 consecutive lanes, processed by one warp (thread = lane).  When the batch is too small
// to give every SM a few warps that way and the emitter walks the chunk's lanes serially (mnist images), the host
// shrinks chunks to 16 or 8 lanes (a.chunk_lanes): the transition then idles some threads, which costs nothing
// next to spreading 4 096 lanes x 3 KB over 512 warps instead of 128.
//   * default launch: one chunk per warp, ceil(B / 32) warps; small CTAs (64 threads) keep the per-SM share of
//     the 2048 chunks of a 65 536-lane batch within ~1% of even on 148 SMs and let the hardware CTA scheduler
//     balance SMs dynamically.
//   * deep_sea bulk path: a PERSISTENT grid (as many warps as fit the SMs' shared memory: 3 per SM at N = 32)
//     whose warps pull chunk indices from a global counter (atomicAdd by the elected lane).  SMs drain HBM at
//     slightly different rates (L2 slice / die distance), so dynamic dealing matters -- and so does not reserving
//     work early: measured on one box, static equal split 48.0 us/step, two fetches ahead 48.0, one ahead 45.5,
//     LAZY (fetch only after the current chunk's stores are issued; the default) 43.9.  The TMA unit keeps
//     draining the warp's last two stores while it fetches and loads the next chunk's state.  Every warp's
//     first chunk is its own index (no atomic on the start-up path); the counter deals the rest and is never
//     reset: a launch with C chunks and W warps performs exactly C atomicAdds (C - W successful fetches plus one
//     failing fetch per warp), so launch k starts at work_base_k = work_base_(k-1) + C.
// Graph-safe mode (a.clock != null; the handle switches to it for good the first time one of its launches is
// captured into a CUDA graph): launch arguments are frozen in a graph, so everything that changes from launch to
// launch lives in device memory instead (layout: CLOCK_* below): the steps this handle has advanced since the
// switch (step index = a.step0 + that count: the on-device action stream and the Logging columns depend on it), the
// chunk counter, and the count of finished CTAs.  The CTA that finishes last advances the step count by T and
// zeroes the other two; every CTA reads the step count before it counts itself finished, so the update cannot
// overtake a reader.
// Register budget per family (second __launch_bounds__ argument, counted in 128-thread blocks per SM).  The
// generic kernel is register-hungry (two Philox streams, action stream, accumulators); left alone ptxas takes
// 160-220 registers and 64-thread CTAs then run at 8 warps/SM, which starves the latency-bound small families.
// Measured on B200 (rollout us/step at 128 vs ~220 registers): cartpole 5.3 vs 8.1, mountain_car 2.6 vs 4.2,
// umbrella_length 12.7 vs 19.7, memory_len 5.0 vs 7.2; bandit / discounting_chain gain again at <= 64.
template <class F> struct MinBlocksPerSM { static const int value = 4; };        // <= 128 registers
template <> struct MinBlocksPerSM<MemoryChain> { static const int value = 6; };   // <= 80
template <> struct MinBlocksPerSM<Bandit> { static const int value = 8; };        // <= 64
template <> struct MinBlocksPerSM<DiscountingChain> { static const int value = 8; };
#ifdef BSB_MIN_BLOCKS_PER_SM   // build-time override for tuning experiments
#define BSB_LAUNCH_MIN_BLOCKS(F) BSB_MIN_BLOCKS_PER_SM
#else
#define BSB_LAUNCH_MIN_BLOCKS(F) MinBlocksPerSM<F>::value
#endif
// System-scope accesses to the pinned mailbox (host memory over PCIe) and volatile accesses to its L2 relay.
__device__ __forceinline__ unsigned long long ld_sys_u64(const volatile unsigned long long* ptr) {
  unsigned long long v; asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(ptr) : "memory"); return v;
}
__device__ __forceinline__ void st_sys_u64(volatile unsigned long long* ptr, unsigned long long v) {
  asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(ptr), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long global_timer_ns() {
  unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t;
}
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// Graph-safe mode keeps the step count, the chunk counter and the finished-CTA count in device memory.  Every
// word that many CTAs touch is spread over CLOCK_GROUPS 128-byte lines, because same-line traffic serialises in
// one L2 slice (~2 ns per access): a 16 384-CTA launch reads the step count once per warp and counts itself out
// once per CTA.
//   clock[16 r]                 r < 32: the step count, REPLICATED (CTA b reads replica b % 32; the last CTA of
//                               a launch rewrites all 32); the host reads / writes replica 0 .. 31
//   clock[CLOCK_CHUNK]          chunk counter of the persistent grids (a line of its own)
//   clock[CLOCK_TOP]            groups that have finished
//   clock[CLOCK_SUB0 + 16 g]    CTAs of group g (= blockIdx % 32) that have finished
static const int CLOCK_GROUPS = 32, CLOCK_CHUNK = 16 * CLOCK_GROUPS, CLOCK_TOP = CLOCK_CHUNK + 16,
                 CLOCK_SUB0 = CLOCK_TOP + 16, CLOCK_WORDS = CLOCK_SUB0 + 16 * CLOCK_GROUPS;

template <class F, int RK, bool kNoise, bool kTrack>
__global__ void __launch_bounds__(128, BSB_LAUNCH_MIN_BLOCKS(F)) transition_kernel(const EnvParams p, const LaunchArgs a) {
  typedef typename RngOf<RK>::type R;
  constexpr int kEmit = EmitKind<F>::value;
  extern __shared__ float4 smem_raw[];
  __shared__ MailFields mail_in;
  __shared__ int mail_cancel;
  const int tid = threadIdx.x & 31, warp = threadIdx.x >> 5, warps_per_cta = blockDim.x >> 5;
  const int64_t B = p.batch;
  const int K = p.obs_numel;
  const size_t stage_floats = smem_floats_per_warp<F>(K, a.emit_bulk != 0, a.group_lanes, a.stage_rows);
  const unsigned row_mask = a.stage_rows == 2 ? 1u : 0u;      // row / board stage of store number n: n & row_mask
  float* stage = reinterpret_cast<float*>(smem_raw) + (size_t)warp * stage_floats;
  // mnist bulk path: all-zero tiles shared by the CTA's warps (source of the LAST-frame stores), after the stages
  float* cta_zero = reinterpret_cast<float*>(smem_raw) + (size_t)warps_per_cta * stage_floats;

  // Stages that rely on staying zero between steps are cleared once, before the dependency wait.
  if (kEmit == EMIT_TWOHOT || (kEmit == EMIT_ONEHOT && a.emit_bulk)) {
    float4* s4 = reinterpret_cast<float4*>(stage);
    const int total4 = (int)(stage_floats >> 2);
    for (int q = tid; q < total4; q += 32) s4[q] = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int e = (total4 << 2) + tid; e < (int)stage_floats; e += 32) stage[e] = 0.f;
    __syncwarp();
  }
  if (kEmit == EMIT_IMAGE) {      // pixel table: image.astype(float32) / 255 for every int8 value (mnist.py:64)
    for (int i = tid; i < 256; i += 32) stage[i] = Mnist::pixel((int8_t)(uint8_t)i);
    for (int i = threadIdx.x; i < a.cta_extra_floats; i += blockDim.x) cta_zero[i] = 0.f;
    fence_proxy_async_smem();
    __syncthreads();
  }
  // Wait for the previous step's kernel (it wrote the lane state read below), THEN allow the next step's kernel
  // to become resident: its CTAs park at their own wait, so at most one dependent grid is ever pending.
  // (The observation-only launch of a split host step must not wait for its predecessor -- the transitions launch,
  // whose copiers are still shipping scalars over PCIe -- to END: it waits for that launch's phase-1 flag below.)
  if (a.use_pdl) { if (a.phase != 2) pdl_wait(); pdl_launch_dependents(); }
  int64_t step0 = a.step0;
  if (a.clock) step0 += (int64_t)*reinterpret_cast<volatile unsigned long long*>(a.clock + 16 * (blockIdx.x % CLOCK_GROUPS));

  // Caller-owned buffers: launch arguments, or -- doorbell mode -- whatever the host wrote into the mailbox
  // before it rang this launch's ticket.
  MailFields io;
  io.actions = a.actions; io.obs = a.obs; io.reward = a.reward; io.reward_f64 = a.reward_f64;
  io.discount = a.discount; io.step_type = a.step_type; io.obs_vec_ok = a.obs_vec_ok; io.pad = 0;
  bool cancelled = false;
  if (a.mailbox && a.wait_doorbell) {
    if (blockIdx.x == 0 && warp == 0) {
      // The one poller of host memory: lanes 0..7 read the mailbox's first 64-byte line (doorbell + fields) with ONE
      // coalesced request per poll; when the ring shows, the line is read once more (the host wrote the fields
      // before the doorbell, so this second read cannot be stale), parked in device memory, and the ticket is
      // relayed to the other blocks through L2.
      const volatile unsigned long long* line = &a.mailbox->doorbell;
      const unsigned long long deadline = global_timer_ns() + a.doorbell_timeout_ns;
      unsigned long long word = 0, seen;
      do {
        if (tid < 8) word = ld_sys_u64(line + tid);
        seen = __shfl_sync(0xffffffffu, word, 0);
      } while ((seen & ~MAIL_CANCEL) < a.ticket && global_timer_ns() < deadline);
      if ((seen & ~MAIL_CANCEL) < a.ticket) seen = a.ticket | MAIL_CANCEL;        // nobody rang: stand down
      __threadfence_system();
      if (tid < 8) word = ld_sys_u64(line + tid);
      if (tid >= 1 && tid < 8) reinterpret_cast<unsigned long long*>(&a.mail->in)[tid - 1] = word;
      __threadfence();
      __syncwarp();
      if (tid == 0) a.mail->relay = seen;
    }
    if (threadIdx.x == 0) {
      unsigned long long seen;
      do { seen = a.mail->relay; } while ((seen & ~MAIL_CANCEL) < a.ticket);
      __threadfence();
      mail_cancel = (seen & MAIL_CANCEL) ? 1 : 0;
      const volatile unsigned long long* src = reinterpret_cast<const volatile unsigned long long*>(&a.mail->in);
      unsigned long long* dst = reinterpret_cast<unsigned long long*>(&mail_in);
      for (int k = 0; k < (int)(sizeof(MailFields) / 8); ++k) dst[k] = src[k];
    }
    __syncthreads();
    io = mail_in;
    cancelled = mail_cancel != 0;
  }
  const bool vec = io.obs_vec_ok != 0;

  const int cl = a.chunk_lanes;
  const int64_t n_chunks = (B + cl - 1) / cl;
  const bool dynamic = a.work_counter != nullptr;
  const bool lazy = a.lazy_fetch != 0;
  // The elected lane draws chunk indices [total_warps, n_chunks) from the global counter and broadcasts them
  // with a shuffle; chunk (global warp index) is taken without asking.
  // Two-phase host steps set the first blocks aside as COPIERS (see below): they own no chunks at first.
  const bool two_phase = ObsFromState<F>::value && a.early_scalars > 0 && a.mailbox && !cancelled;
  const unsigned copier_blocks = two_phase ? (unsigned)a.early_scalars : 0u;
  const unsigned worker_blocks = gridDim.x - copier_blocks;
  const unsigned worker_block = blockIdx.x - copier_blocks;
  const int64_t total_warps = (int64_t)worker_blocks * warps_per_cta;
  auto fetch_chunk = [&]() -> int64_t {
    unsigned long long v = 0;
    if (tid == 0) v = atomicAdd(a.work_counter, 1ull) - a.work_base;      // graph-safe mode: clock + 1, base 0
    return total_warps + (int64_t)__shfl_sync(0xffffffffu, v, 0);
  };
  int64_t cur_chunk = (int64_t)worker_block * warps_per_cta + warp;
  if (cancelled) {
    // A stood-down launch still owes the chunk counter its share: a launch over C chunks advances it by exactly C.
    // (a two-phase launch also owes one failing fetch per copier warp, which the host's arithmetic counts too)
    if (dynamic && blockIdx.x == 0 && threadIdx.x == 0)
      atomicAdd(a.work_counter, (unsigned long long)n_chunks + (unsigned long long)(a.early_scalars > 0 ? a.early_scalars * warps_per_cta : 0));
    cur_chunk = n_chunks;
  }

  const bool has_rng = p.rng_pos != nullptr;
  // catch: cells this thread poked into stage buffer 0 / 1 (cleared when that buffer is reused)
  int poked_a0 = -1, poked_b0 = -1, poked_a1 = -1, poked_b1 = -1;
  // deep_sea bulk path: offset of the cell this thread poked into group buffer 0 / 1 (cleared on reuse)
  int tile_poked0 = -1, tile_poked1 = -1;
  unsigned emitted = 0;          // bulk stores issued by this warp so far (double-buffer parity)
  bool any_bulk = false;

  // Observation emitter of this warp for one chunk and step (shared by the ordinary loop and by the two-phase
  // host-step path below); the staging state above persists across calls.
  auto emit_obs = [&](const typename F::Lane& L, R& rng, float* obs_t, int64_t warp_base, int n_lanes, int64_t lane,
                      bool active, bool bulk) {
    if (kEmit == EMIT_ONEHOT) {
      const int hot = Descriptor<F>::a(L);
      if (bulk) {
        // Groups of m consecutive lanes share one staging buffer (m tiles, contiguous in global memory too) and
        // leave as ONE bulk store of up to m * 4K bytes: large stores amortise the per-operation cost of the
        // TMA unit (measured: ~70 ns + bytes / 64 GB/s per SM).
        const int m = a.group_lanes;
        for (int g0 = 0; g0 < n_lanes; g0 += m) {
          const int in_group = (n_lanes - g0) < m ? (n_lanes - g0) : m;
          const int s = (int)(emitted & 1u);
          float* group = stage + (size_t)s * m * K;
          if (tid == 0) bulk_wait_read<TILE_STAGES - 1>();    // the store two back, last reader of `group`, is done
          __syncwarp();
          if (s == 0) { if (tile_poked0 >= 0) { group[tile_poked0] = 0.f; tile_poked0 = -1; } }
          else        { if (tile_poked1 >= 0) { group[tile_poked1] = 0.f; tile_poked1 = -1; } }
          __syncwarp();     // a thread of an earlier group may clear the very cell another thread sets now
          if (tid >= g0 && tid < g0 + in_group && hot >= 0) {
            const int cell = (tid - g0) * K + hot;
            group[cell] = 1.f;
            if (s == 0) tile_poked0 = cell; else tile_poked1 = cell;
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (tid == 0) {
            float* tile_dst = obs_t + (warp_base + g0) * (int64_t)K;
            const uint32_t tile_bytes = (uint32_t)in_group * (uint32_t)K * 4u;
            bulk_store_obs(tile_dst, group, tile_bytes, a.l2_hint);
            bulk_commit();
          }
          ++emitted;
        }
      } else {
        emit_onehot_vec(obs_t, warp_base, n_lanes, K, hot, vec && (K & 3) == 0);
      }
    } else if (kEmit == EMIT_TWOHOT) {
      const int hot_a = Descriptor<F>::a(L), hot_b = Descriptor<F>::b(L);
      if (bulk) {
        const int buf = (int)(emitted & row_mask);
        float* boards = stage + (size_t)buf * 32 * K;
        if (tid == 0) { if (row_mask) bulk_wait_read<1>(); else bulk_wait_read<0>(); }   // the store that last read `boards` is done with it
        __syncwarp();
        float* mine = boards + tid * K;
        const int old_a = buf ? poked_a1 : poked_a0, old_b = buf ? poked_b1 : poked_b0;
        if (old_a >= 0) mine[old_a] = 0.f;
        if (old_b >= 0) mine[old_b] = 0.f;
        int new_a = -1, new_b = -1;
        if (active) { mine[hot_a] = 1.f; mine[hot_b] = 1.f; new_a = hot_a; new_b = hot_b; }
        if (buf) { poked_a1 = new_a; poked_b1 = new_b; } else { poked_a0 = new_a; poked_b0 = new_b; }
        fence_proxy_async_smem();
        __syncwarp();
        if (tid == 0) { bulk_store_obs(obs_t + warp_base * (int64_t)K, boards, (uint32_t)n_lanes * (uint32_t)K * 4u, a.l2_hint); bulk_commit(); }
        ++emitted;
      } else {
        emit_twohot_vec(obs_t, warp_base, n_lanes, K, hot_a, hot_b, vec);
      }
    } else if (kEmit == EMIT_IMAGE) {
      const int image = Descriptor<F>::a(L);
      if (bulk) emit_image_bulk(p, stage, cta_zero, obs_t, warp_base, n_lanes, K, active ? image : -1, a.group_lanes,
                                a.cta_extra_floats / K, a.l2_hint, a.stage_rows, emitted);
      else emit_image(p, stage, obs_t, warp_base, n_lanes, K, image, vec && (K & 3) == 0);
    } else if (!a.stage_rows) {
      // observation rows too long for a shared-memory stage: every thread renders its row in place
      if (active) RowRenderer<F, R>::run(p, L, rng, obs_t + lane * (int64_t)K);
    } else {
      float* rows = stage + (size_t)(emitted & row_mask) * 32 * K;
      if (bulk) { if (tid == 0) { if (row_mask) bulk_wait_read<1>(); else bulk_wait_read<0>(); } }
      __syncwarp();
      if (active) RowRenderer<F, R>::run(p, L, rng, rows + tid * K);
      if (bulk) {
        fence_proxy_async_smem();
        __syncwarp();
        if (tid == 0) { bulk_store_obs(obs_t + warp_base * (int64_t)K, rows, (uint32_t)n_lanes * (uint32_t)K * 4u, a.l2_hint); bulk_commit(); }
      } else {
        __syncwarp();
        flush_rows_vec(rows, obs_t, warp_base, n_lanes, K, vec);
      }
      ++emitted;
    }
  };
  // Which chunks leave through the TMA unit (16-byte aligned spans); warp-uniform per chunk.
  auto chunk_is_bulk = [&](int n_lanes) -> bool {
    bool bulk = a.emit_bulk && vec;
    if (kEmit == EMIT_ROWS) bulk = bulk && K >= 3 && ((n_lanes * K) & 3) == 0;
    if (kEmit == EMIT_TWOHOT) bulk = bulk && ((n_lanes * K) & 3) == 0;
    if (kEmit == EMIT_ONEHOT) bulk = bulk && ((K & 3) == 0 || ((n_lanes % a.group_lanes) == 0 && ((a.group_lanes * K) & 3) == 0));
    if (kEmit == EMIT_IMAGE) bulk = bulk && (K & 3) == 0;
    return bulk;
  };

  // ---- two-phase host step (a.early_scalars; families whose observation is a function of the stored state) ----
  // A host-driven step (bsb_step_host) returns when reward / discount / step_type are in host memory; the
  // observation stays on the device.  So the transitions of ALL chunks run first (phase 1: statically dealt; the
  // actions of a warp's chunks are fetched over PCIe in one round trip), and the observations are streamed
  // afterwards (phase 2, dynamically dealt as usual) while the host already decides the next action.  Phase 2
  // re-reads the lane state phase 1 stored (L2-resident) and renders from it; a warp's first chunk stays in
  // registers.
  // Who ships the scalars to the host?  Not the workers: 768 KB of posted PCIe writes per step back-pressure the
  // warps that issue them (GPU timeline, profiles/r02_e2e_timeline.txt: a phase 1 that wrote to host memory took
  // 13 us instead of ~3, and 25 us when it also read its actions over PCIe), and they have 268 MB of observations
  // to issue.  The workers write reward / discount / step_type to a DEVICE staging block, fence at GPU scope and
  // count themselves out.  The first `early_scalars` blocks, the COPIERS, own no chunks at first: they wait for
  // that count, copy the staging block to the host's pinned buffers with 16-byte stores (16 per thread in flight:
  // ~128 KB across the copiers, enough for the link), issue the system fence, and the last one stores the completion
  // word; then they join phase 2 through the chunk counter like everybody else.
  // (PTX memory model: workers release / copiers acquire at gpu scope; the copiers' own stores, fence.sc.sys and the
  // completion word are program-ordered; the host's acquire load of the word therefore sees every scalar.)
  if constexpr (ObsFromState<F>::value) {
    if (two_phase && blockIdx.x < copier_blocks) {
      if (threadIdx.x == 0) {
        const unsigned long long t_start = a.timing ? global_timer_ns() : 0ull;
        while (*reinterpret_cast<volatile unsigned long long*>(&a.mail->finished) < (unsigned long long)worker_blocks) {}
        if (blockIdx.x == 0) {
          a.mail->phase1 = a.ticket;         // every chunk's state is stored: phase 2 may read any lane's state
          if (a.timing) {
            st_sys_u64(&a.mailbox->stamp[0], t_start);
            st_sys_u64(&a.mailbox->stamp[1], global_timer_ns());
            st_sys_u64(&a.mailbox->stamp[3], a.mail->last_exit);
          }
        }
      }
      __syncthreads();
      __threadfence();                       // acquire: the staging block is read below
      const int64_t n_thr = (int64_t)copier_blocks * blockDim.x, me = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
      auto ship = [&](const void* from, void* to, int64_t bytes) {
        if (!from || !to) return;
        if ((reinterpret_cast<uintptr_t>(from) | reinterpret_cast<uintptr_t>(to)) & 15) {      // odd batch sizes: words
          const uint32_t* s32 = reinterpret_cast<const uint32_t*>(from);
          uint32_t* d32 = reinterpret_cast<uint32_t*>(to);
          for (int64_t i = me; i < (bytes >> 2); i += n_thr) d32[i] = __ldcg(s32 + i);
          return;
        }
        const uint4* src = reinterpret_cast<const uint4*>(from);
        uint4* dst = reinterpret_cast<uint4*>(to);
        const int64_t n16 = bytes >> 4;
        constexpr int U = 16;     // 16 x 16 B per thread in flight: ~128 KB across the copiers, enough for the PCIe link
        for (int64_t i0 = me; i0 < n16; i0 += U * n_thr) {
          uint4 v[U];
#pragma unroll
          for (int u = 0; u < U; ++u) { const int64_t i = i0 + u * n_thr; if (i < n16) v[u] = __ldcg(src + i); }
#pragma unroll
          for (int u = 0; u < U; ++u) { const int64_t i = i0 + u * n_thr; if (i < n16) dst[i] = v[u]; }
        }
        const char* tail_src = reinterpret_cast<const char*>(from) + (n16 << 4);
        char* tail_dst = reinterpret_cast<char*>(to) + (n16 << 4);
        for (int64_t i = me; i < (bytes & 15); i += n_thr) tail_dst[i] = tail_src[i];
      };
      ship(a.stage.reward, io.reward, B * 4);
      ship(a.stage.reward_f64, io.reward_f64, B * 8);
      ship(a.stage.discount, io.discount, B * 4);
      ship(a.stage.step_type, io.step_type, B * 4);
      __threadfence_system();
      __syncthreads();
      if (threadIdx.x == 0 && atomicAdd(&a.mail->copied, 1ull) == (unsigned long long)copier_blocks - 1ull) {
        a.mail->finished = 0ull;             // every copier is past its wait: re-arm both counts for the next launch
        a.mail->copied = 0ull;
        __threadfence_system();
        if (a.timing) st_sys_u64(&a.mailbox->stamp[2], global_timer_ns());
        st_sys_u64(&a.mailbox->done, a.ticket);      // the host may read its scalars
      }
      // join phase 2: the copiers own no chunk of their own, the counter deals them the rest
      cur_chunk = n_chunks;
      if (dynamic) {
        typename F::Lane L;
        int64_t c = fetch_chunk();
        while (c < n_chunks) {
          const int64_t warp_base = c * cl;
          const int n_lanes = (B - warp_base) < cl ? (int)(B - warp_base) : cl;
          const int64_t lane = warp_base + tid;
          const bool active = tid < n_lanes;
          F::init(p, L);
          if (active) { F::load(p, lane, L); F::describe(p, L); }
          const bool bulk = chunk_is_bulk(n_lanes);
          any_bulk = any_bulk || bulk;
          R unused_rng;
          emit_obs(L, unused_rng, io.obs, warp_base, n_lanes, lane, active, bulk);
          c = fetch_chunk();
        }
      }
    } else if (two_phase) {
      const int64_t own = cur_chunk;
      typename F::Lane keep;
      F::init(p, keep);
      constexpr int kAhead = 4;              // chunks whose loads (action, lane state, accumulators) are in flight together
      for (int64_t c0 = own; c0 < n_chunks; c0 += kAhead * total_warps) {
        // every independent load of up to kAhead chunks first: one round trip to L2 (or over PCIe, when the actions
        // were not staged on the device) instead of one per chunk -- a warp owns 4-5 chunks of a 65 536-lane batch
        int32_t fetched[kAhead];
        typename F::Lane lanes[kAhead];
        EpisodeStats eps[kAhead];
#pragma unroll
        for (int k = 0; k < kAhead; ++k) {
          const int64_t c = c0 + k * total_warps;
          const int64_t lane = c * cl + tid;
          const bool live = c < n_chunks && tid < cl && lane < B;
          fetched[k] = 0;
          F::init(p, lanes[k]);
          if (live) {
            fetched[k] = __ldcv(io.actions + lane);
            F::load(p, lane, lanes[k]);
            if (kTrack) eps[k].load(p, lane);
          }
        }
#pragma unroll
        for (int k = 0; k < kAhead; ++k) {
          const int64_t c = c0 + k * total_warps;
          if (c >= n_chunks) break;
          const int64_t lane = c * cl + tid;
          typename F::Lane& L = lanes[k];
          if (tid < cl && lane < B) {
            R rng, wrng;
            if (has_rng) rng_open(rng, p, lane, false);
            if (kNoise) rng_open(wrng, p, lane, true);
            int32_t action = fetched[k];
            if ((uint32_t)action >= (uint32_t)p.num_actions) {
              if (a.bad_action) *a.bad_action = 1;
              action = action < 0 ? 0 : p.num_actions - 1;
            }
            const bool after_last = L.nr != 0;
            const StepOut o = lane_transition<F, R, R>(p, lane, L, rng, wrng, action, MODE_STEP, kNoise);
            F::store(p, lane, L);
            if (has_rng) rng_close(rng, p, lane, false);
            if (kNoise) rng_close(wrng, p, lane, true);
            if (kTrack) {
              eps[k].track(p, lane, o, step0, after_last);
              eps[k].store(p, lane);
              if (p.log_next && o.step_type == LAST && log_row_due(p, lane)) log_point_record(p, lane, step0 + 1);
            }
            if (a.stage.reward) a.stage.reward[lane] = (float)o.reward;
            if (a.stage.reward_f64) a.stage.reward_f64[lane] = o.reward;
            if (a.stage.discount) a.stage.discount[lane] = o.discount;
            if (a.stage.step_type) a.stage.step_type[lane] = o.step_type;
          }
          if (c == own) keep = L;
        }
      }
      __threadfence();                       // gpu scope (device memory only): the copiers do the system-scope one
      __syncthreads();
      if (threadIdx.x == 0) atomicAdd(&a.mail->finished, 1ull);
      bool mine = true;
      int64_t c = a.phase == 1 ? n_chunks : own;      // split step: the observations are the next launch's
      while (c < n_chunks) {
        const int64_t warp_base = c * cl;
        const int n_lanes = (B - warp_base) < cl ? (int)(B - warp_base) : cl;
        const int64_t lane = warp_base + tid;
        const bool active = tid < n_lanes;
        typename F::Lane L = keep;
        if (!mine) {
          // a dynamically dealt chunk: some other warp ran its phase 1 -- long ago in practice, but wait for it
          if (tid == 0) while (a.mail->phase1 != a.ticket) {}
          __syncwarp();
          __threadfence();                   // acquire: the loads below must not be served from a stale L1 line
          F::init(p, L);
          if (active) { F::load(p, lane, L); F::describe(p, L); }
        }
        const bool bulk = chunk_is_bulk(n_lanes);
        any_bulk = any_bulk || bulk;
        R unused_rng;
        emit_obs(L, unused_rng, io.obs, warp_base, n_lanes, lane, active, bulk);
        mine = false;
        c = dynamic ? fetch_chunk() : n_chunks;
      }
      cur_chunk = n_chunks;                  // nothing left for the ordinary loop
    } else if (a.phase == 2) {
      // Observation-only launch of a split host step: the transitions launch ahead of it in the stream stored every
      // lane's state and raised mail->phase1; render from the stored state, chunks dealt as usual.
      if (tid == 0) while (a.mail->phase1 != a.ticket) {}
      __syncwarp();
      __threadfence();                       // acquire
      int64_t c = cur_chunk;
      while (c < n_chunks) {
        const int64_t warp_base = c * cl;
        const int n_lanes = (B - warp_base) < cl ? (int)(B - warp_base) : cl;
        const int64_t lane = warp_base + tid;
        const bool active = tid < n_lanes;
        typename F::Lane L;
        F::init(p, L);
        if (active) { F::load(p, lane, L); F::describe(p, L); }
        const bool bulk = chunk_is_bulk(n_lanes);
        any_bulk = any_bulk || bulk;
        R unused_rng;
        emit_obs(L, unused_rng, io.obs, warp_base, n_lanes, lane, active, bulk);
        c = dynamic ? fetch_chunk() : n_chunks;
      }
      cur_chunk = n_chunks;
    }
  }

  while (cur_chunk < n_chunks) {
    const int64_t warp_base = cur_chunk * cl;
    // eager policy: reserve the next chunk now; lazy (default): only after this chunk's stores are issued
    cur_chunk = (dynamic && !lazy) ? fetch_chunk() : n_chunks;
    const int n_lanes = (B - warp_base) < cl ? (int)(B - warp_base) : cl;
    const int64_t lane = warp_base + tid;
    const bool active = tid < n_lanes;
    const bool bulk = chunk_is_bulk(n_lanes);
    any_bulk = any_bulk || bulk;

    typename F::Lane L;
    R rng, wrng;
    EpisodeStats ep;
    ActionStream action_stream;
    action_stream.open();
    if (active) {
      if (a.mode == MODE_INIT) F::init(p, L); else F::load(p, lane, L);
      if (has_rng) rng_open(rng, p, lane, false);
      if (kNoise) rng_open(wrng, p, lane, true);
      if (kTrack) ep.load(p, lane);
    } else {
      F::init(p, L);
    }

    if (a.mode == MODE_INIT) {
      if (active) {
        F::ctor_draws(p, L, rng);
        F::store(p, lane, L);
        if (has_rng) rng_close(rng, p, lane, false);
      }
      if (dynamic && lazy) cur_chunk = fetch_chunk();
      continue;
    }

    for (int64_t t = 0; t < a.T; ++t) {
      const int64_t off = t * B + lane;
      if (active) {
        int32_t action = 0;
        if (a.mode == MODE_STEP) {
          if (io.actions) {
            // doorbell mode reads host memory the launch may have cached before the host wrote it: ld.cv
            action = a.mailbox ? __ldcv(io.actions + off) : io.actions[off];
            if ((uint32_t)action >= (uint32_t)p.num_actions) {      // never index a table or pack state with it
              if (a.bad_action) *a.bad_action = 1;
              action = action < 0 ? 0 : p.num_actions - 1;
            }
          } else {
            action = action_stream.sample(a.action_seed, p.lane_offset + (uint64_t)lane, (uint64_t)(step0 + t), p.num_actions);
          }
          if (a.actions_out) a.actions_out[off] = action;
        }
        const bool after_last = L.nr != 0;
        const StepOut o = lane_transition<F, R, R>(p, lane, L, rng, wrng, action, a.mode, kNoise);
        if (kTrack) {
          ep.track(p, lane, o, step0 + t, after_last);
          if (p.log_next && o.step_type == LAST && log_row_due(p, lane)) {      // <= 49 times per 10 000 episodes
            F::store(p, lane, L); ep.store(p, lane);
            log_point_record(p, lane, step0 + t + 1);
          }
        }
        if (io.reward) io.reward[off] = (float)o.reward;
        if (io.reward_f64) io.reward_f64[off] = o.reward;
        if (io.discount) io.discount[off] = o.discount;
        if (io.step_type) io.step_type[off] = o.step_type;
      }
      float* obs_t = io.obs + t * B * (int64_t)K;

      emit_obs(L, rng, obs_t, warp_base, n_lanes, lane, active, bulk);
    }

    if (active) {
      F::store(p, lane, L);
      if (has_rng) rng_close(rng, p, lane, false);
      if (kNoise) rng_close(wrng, p, lane, true);
      if (kTrack) ep.store(p, lane);
    }
    if (dynamic && lazy) cur_chunk = fetch_chunk();        // lazy: nothing was reserved while working
  }
  if (any_bulk && tid == 0) {
    // shared memory must outlive the last bulk read; in doorbell mode the host takes `done` to mean that the
    // observations are in device memory, so there the stores themselves must have completed
    if (a.mailbox && !a.early_scalars) bulk_wait_all(); else bulk_wait_read<0>();
  }
  if (a.timing && a.mail && threadIdx.x == 0) atomicMax(&a.mail->last_exit, global_timer_ns());
  if (a.mailbox && !two_phase) {
    __threadfence_system();                  // every thread: its zero-copy outputs are visible to the host ...
    __syncthreads();                         // ... before the CTA counts itself finished
    if (threadIdx.x == 0) {
      if (atomicAdd(&a.mail->finished, 1ull) == (unsigned long long)gridDim.x - 1ull) {
        a.mail->finished = 0ull;
        __threadfence_system();
        st_sys_u64(&a.mailbox->done, a.ticket | (cancelled ? MAIL_CANCEL : 0ull));
      }
    }
  }
  if (a.clock) {
    __syncthreads();
    if (threadIdx.x == 0) {
      const unsigned groups = gridDim.x < (unsigned)CLOCK_GROUPS ? gridDim.x : (unsigned)CLOCK_GROUPS;
      const unsigned g = blockIdx.x % groups;
      const unsigned members = gridDim.x / groups + (g < gridDim.x % groups ? 1u : 0u);
      unsigned long long* sub = a.clock + CLOCK_SUB0 + 16 * g;
      // No fence: the count only says "this CTA has READ the step count and drawn its chunks" -- both happened
      // (their values were consumed) long before; the state it wrote reaches the next launch through the kernel
      // boundary.  A membar here kept every CTA alive ~1 us longer: +2..7 us per launch on multi-wave grids.
      if (atomicAdd(sub, 1ull) == (unsigned long long)members - 1ull) {
        *sub = 0ull;                          // re-armed for the next launch (which starts after this one ends)
        if (atomicAdd(a.clock + CLOCK_TOP, 1ull) == (unsigned long long)groups - 1ull) {
          const unsigned long long steps = (unsigned long long)(step0 - a.step0) + (a.mode == MODE_INIT ? 0ull : (unsigned long long)a.T);
          for (int r = 0; r < CLOCK_GROUPS; ++r) a.clock[16 * r] = steps;
          a.clock[CLOCK_CHUNK] = 0ull;
          a.clock[CLOCK_TOP] = 0ull;
        }
      }
    }
  }
}

#endif  // __CUDACC__

}  // namespace bsb
