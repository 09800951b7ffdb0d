// Per-family lane transitions, written once as __host__ __device__ functions:
// the CUDA kernels (bsb_kernels.cuh) and the explicit host path both call them.
//
// Every function cites the reference lines whose behaviour it reproduces.
// Nothing here allocates or touches observations of other lanes; observation
// rendering is described by small per-lane descriptors so that the kernels can
// emit dense tensors warp-cooperatively.
#pragma once
#include "bsb_rng.cuh"
#include "bsb_scoring.cuh"

namespace bsb {

enum { FIRST = 0, MID = 1, LAST = 2 };

struct StepOut {
  double reward;     // float64, as the reference computes it
  float discount;    // 1 MID, 0 LAST, 0 FIRST (reference: None)
  int32_t step_type;
};

BSB_HD StepOut make_first() { StepOut o; o.reward = 0.0; o.discount = 0.0f; o.step_type = FIRST; return o; }
BSB_HD StepOut make_mid(double r) { StepOut o; o.reward = r; o.discount = 1.0f; o.step_type = MID; return o; }
BSB_HD StepOut make_last(double r) { StepOut o; o.reward = r; o.discount = 0.0f; o.step_type = LAST; return o; }

// Device-resident (or host-resident) description of one environment batch.
// Passed BY VALUE to kernels.
struct EnvParams {
  int32_t family, wrapper, rng_kind, flags;
  int32_t size, deterministic, rows, columns, memory_length, num_bits;
  int32_t chain_length, n_distractor, num_actions, max_steps, num_data, image_numel;
  int32_t obs_numel, obs_rows, obs_cols, n_info;
  int64_t batch;
  uint64_t seed, lane_offset;

  double move_cost_step;   // unscaled_move_cost / size       (deep_sea.py:132)
  double inv_size;         // 1 / size                        (deep_sea.py:130)
  double height_threshold, x_threshold, timescale, max_time, init_range;
  double theta_dot_threshold, x_reward_threshold, move_cost;
  double noise_scale, reward_scale;
  // cartpole.py:106-112 config, derived exactly as step_cartpole derives them
  double cp_force_mag, cp_pl, cp_length, cp_mass_pole, cp_mass_total, cp_gravity, cp_four_thirds, cp_two_pi;

  // tables
  const uint32_t* mapping_bits;  // deep_sea: bit (row*N+col) of the action mapping
  const double* reward_table;    // bandit / discounting_chain
  const int8_t* images;          // mnist
  const uint8_t* labels;         // mnist

  // lane state, structure-of-arrays over the batch
  uint32_t* st_word;   // [B]   packed small integers; bit 31 = _reset_next_step
  uint64_t* st_ctx;    // [B]   memory_chain context bits
  double* st_f64;      // [6][B] float64 dynamics state (+ episode_return)
  double* info;        // [BSB_MAX_INFO][B] bsuite_info() accumulators
  double* ep;          // [5][B] Logging accumulators, or null
  // Log-spaced rows of the Logging wrapper (wrappers.py:99-110, 140-147), recorded per lane on the device:
  // row k of lane i = the wrapper's columns at the LAST timestep that made episode == log_sched[k].
  double* log_rows;          // [n_log_points][5 + n_info][B], or null
  const int64_t* log_sched;  // [n_log_points] ascending episode counts at which the reference writes a row
  int32_t* log_next;         // [B] rows due so far (= index of the next schedule entry), or null without a schedule
  int32_t n_log_points, score_exp;
  // Score summary of experiment score_exp (bsb_scoring.cuh, fold_row), folded from the row columns
  // score_col_value / score_col_best (-1: none) as each row falls due.
  double* score_sum;         // [kSummaryFields][B], or null
  int32_t score_col_value, score_col_best;
  // RNG state: env stream and reward-wrapper stream
  uint64_t* rng_pos;  double* rng_gauss;
  uint64_t* wrng_pos; double* wrng_gauss;
  uint32_t* mt_key;  int32_t* mt_idx;   // [624][B], [B]  (rng_kind == MT19937)
  uint32_t* wmt_key; int32_t* wmt_idx;
};

static const uint32_t NEEDS_RESET = 0x80000000u;

BSB_HD double clampd(double v, double lo, double hi) { return fmin(fmax(v, lo), hi); }

// numpy.remainder for float64: fmod, then shifted into the divisor's sign.
BSB_HD double np_remainder(double a, double b) {
  double m = fmod(a, b);
  if (m != 0.0) { if ((b < 0.0) != (m < 0.0)) m += b; }
  else { m = copysign(0.0, b); }
  return m;
}

// x ** 2 as CPython / numpy scalars evaluate it: libm pow().  glibc's pow is not
// always equal to the correctly rounded x*x (about 1e-3 of inputs differ by one
// ulp), so the host path calls pow to stay bit-identical with the reference
// while the device uses the exact product (CUDA pow is looser than either).
BSB_HD double square_like_reference(double x) {
#if defined(__CUDA_ARCH__)
  return x * x;
#else
  return pow(x, 2.0);
#endif
}

// ===========================================================================
// deep_sea  (environments/deep_sea.py)
// ===========================================================================
struct DeepSea {
  static const bool kIsDeepSea = true;
  struct Lane { uint32_t row, col, bad, nr; int32_t hot; };
  enum { kInfo = 2 };  // total_bad_episodes, denoised_return  (deep_sea.py:153-155)

  static BSB_HD void load(const EnvParams& p, int64_t i, Lane& L) {
    const uint32_t w = p.st_word[i];
    L.row = w & 0xffu; L.col = (w >> 8) & 0xffu; L.bad = (w >> 16) & 1u; L.nr = w >> 31; L.hot = -1;
  }
  static BSB_HD void store(const EnvParams& p, int64_t i, const Lane& L) {
    p.st_word[i] = L.row | (L.col << 8) | (L.bad << 16) | (L.nr << 31);
  }
  static BSB_HD void init(const EnvParams&, Lane& L) { L.row = L.col = L.bad = 0; L.nr = 1; L.hot = -1; }
  template <class R> static BSB_HD void ctor_draws(const EnvParams&, Lane&, R&) {}

  static BSB_HD void describe(const EnvParams& p, Lane& L) {  // deep_sea.py:103-108
    L.hot = (L.row >= (uint32_t)p.size) ? -1 : (int32_t)(L.row * (uint32_t)p.size + L.col);
  }
  template <class R> static BSB_HD StepOut reset(const EnvParams& p, int64_t, Lane& L, R&) {
    L.row = 0; L.col = 0; L.bad = 0;  // deep_sea.py:110-114
    describe(p, L);
    return make_first();
  }
  template <class R> static BSB_HD StepOut step(const EnvParams& p, int64_t i, Lane& L, int32_t action, R& rng) {
    const uint32_t n = (uint32_t)p.size;
    const uint32_t cell = L.row * n + L.col;
    const int32_t mapped = (int32_t)((p.mapping_bits[cell >> 5] >> (cell & 31u)) & 1u);
    const bool right = (action == mapped);                 // deep_sea.py:118
    double reward = 0.0;
    if (L.col == n - 1 && right) {                          // :121-123
      reward += 1.0;
      p.info[1 * p.batch + i] += 1.0;                       // denoised_return
    }
    if (!p.deterministic) {                                 // :124-126
      if (L.row == n - 1 && (L.col == 0 || L.col == n - 1)) reward += rng.randn();
    }
    if (right) {                                            // :129-132
      // rand() is drawn before `or deterministic`; in the deterministic
      // environment nothing else reads the stream, so the draw is elided.
      bool moves = true;
      if (!p.deterministic) moves = rng.rand() > p.inv_size;
      if (moves) L.col = (L.col + 1 < n) ? L.col + 1 : n - 1;
      reward -= p.move_cost_step;
    } else {                                                // :133-136
      if (L.row == L.col) L.bad = 1;
      L.col = (L.col > 0) ? L.col - 1 : 0;
    }
    L.row += 1;                                             // :137
    describe(p, L);
    if (L.row == n) {                                       // :140-143
      if (L.bad) p.info[0 * p.batch + i] += 1.0;            // total_bad_episodes
      return make_last(reward);
    }
    return make_mid(reward);
  }
};

// ===========================================================================
// catch  (environments/catch.py)
// ===========================================================================
struct Catch {
  static const bool kIsDeepSea = false;
  struct Lane { uint32_t ball_x, ball_y, paddle_x, nr; int32_t hot_a, hot_b; };
  enum { kInfo = 1 };  // total_regret (catch.py:116-117)

  static BSB_HD void load(const EnvParams& p, int64_t i, Lane& L) {
    const uint32_t w = p.st_word[i];
    L.ball_x = w & 0xffu; L.ball_y = (w >> 8) & 0xffu; L.paddle_x = (w >> 16) & 0xffu; L.nr = w >> 31;
    L.hot_a = L.hot_b = -1;
  }
  static BSB_HD void store(const EnvParams& p, int64_t i, const Lane& L) {
    p.st_word[i] = L.ball_x | (L.ball_y << 8) | (L.paddle_x << 16) | (L.nr << 31);
  }
  static BSB_HD void init(const EnvParams&, Lane& L) { L.ball_x = L.ball_y = L.paddle_x = 0; L.nr = 1; L.hot_a = L.hot_b = -1; }
  template <class R> static BSB_HD void ctor_draws(const EnvParams&, Lane&, R&) {}

  static BSB_HD void describe(const EnvParams& p, Lane& L) {  // catch.py:109-114
    L.hot_a = (int32_t)(L.ball_y * (uint32_t)p.columns + L.ball_x);
    L.hot_b = (int32_t)((uint32_t)(p.rows - 1) * (uint32_t)p.columns + L.paddle_x);
  }
  template <class R> static BSB_HD StepOut reset(const EnvParams& p, int64_t, Lane& L, R& rng) {
    L.ball_x = rng.randint((uint32_t)p.columns);           // catch.py:71
    L.ball_y = 0;
    L.paddle_x = (uint32_t)(p.columns / 2);                // :73
    describe(p, L);
    return make_first();
  }
  template <class R> static BSB_HD StepOut step(const EnvParams& p, int64_t i, Lane& L, int32_t action, R&) {
    int32_t px = (int32_t)L.paddle_x + (action - 1);       // catch.py:84-85, _ACTIONS = (-1, 0, 1)
    px = px < 0 ? 0 : (px > p.columns - 1 ? p.columns - 1 : px);
    L.paddle_x = (uint32_t)px;
    L.ball_y += 1;                                          // :88
    describe(p, L);
    if (L.ball_y == (uint32_t)(p.rows - 1)) {               // :91-95
      const double reward = (L.paddle_x == L.ball_x) ? 1.0 : -1.0;
      p.info[i] += (1.0 - reward);
      return make_last(reward);
    }
    return make_mid(0.0);                                   // :97
  }
};

// ===========================================================================
// cartpole and cartpole_swingup
//   (environments/cartpole.py, experiments/cartpole_swingup/cartpole_swingup.py)
// ===========================================================================
struct PoleState { double x, x_dot, theta, theta_dot, t; };

// cartpole.py:37-65 (step_cartpole): explicit Euler from the OLD state; the
// operation order below is the reference's expression order, and this file is
// compiled with FMA contraction off.
//
// cos(theta) / sin(theta) of the CURRENT state are passed in: the reference evaluates them four times per step
// (cartpole.py:44-45 for the dynamics, :141 for the reward, :172-173 for the observation) on two distinct angles;
// the lane keeps the pair for its current angle (SinCos below), so each step computes them once.
struct SinCos { double sn, cs; };
BSB_HD SinCos sincos_of(double theta) {
  SinCos r;
#if defined(__CUDA_ARCH__)
  sincos(theta, &r.sn, &r.cs);
#else
  r.sn = sin(theta); r.cs = cos(theta);       // the host path calls libm exactly like numpy does
#endif
  return r;
}

BSB_HD PoleState advance_pole(const EnvParams& p, const PoleState& s, const SinCos& trig, int32_t action) {
  const double force = (double)(action - 1) * p.cp_force_mag;
  const double c = trig.cs, sn = trig.sn;
  const double temp = (force + p.cp_pl * square_like_reference(s.theta_dot) * sn) / p.cp_mass_total;
  const double theta_acc = (p.cp_gravity * sn - c * temp) /
      (p.cp_length * (p.cp_four_thirds - p.cp_mass_pole * square_like_reference(c) / p.cp_mass_total));
  const double x_acc = temp - p.cp_pl * theta_acc * c / p.cp_mass_total;
  PoleState n;
  n.x = s.x + p.timescale * s.x_dot;
  n.x_dot = s.x_dot + p.timescale * x_acc;
  n.theta = np_remainder(s.theta + p.timescale * s.theta_dot, p.cp_two_pi);
  n.theta_dot = s.theta_dot + p.timescale * theta_acc;
  n.t = s.t + p.timescale;
  return n;
}

template <bool kSwingup>
struct CartpoleT {
  static const bool kIsDeepSea = false;
  // obs: 6 (cartpole.py:167-177) or 8 (cartpole_swingup.py:137-150) floats
  enum { kObs = kSwingup ? 8 : 6, kInfo = kSwingup ? 3 : 2 };
  struct Lane { PoleState s; SinCos trig; double episode_return, raw_return; uint32_t nr; };

  static BSB_HD void load(const EnvParams& p, int64_t i, Lane& L) {
    const int64_t B = p.batch;
    L.s.x = p.st_f64[0 * B + i]; L.s.x_dot = p.st_f64[1 * B + i]; L.s.theta = p.st_f64[2 * B + i];
    L.s.theta_dot = p.st_f64[3 * B + i]; L.s.t = p.st_f64[4 * B + i];
    L.episode_return = p.st_f64[5 * B + i];
    L.raw_return = p.info[i];
    L.nr = p.st_word[i] >> 31;
    L.trig = sincos_of(L.s.theta);
  }
  static BSB_HD void store(const EnvParams& p, int64_t i, const Lane& L) {
    const int64_t B = p.batch;
    p.st_f64[0 * B + i] = L.s.x; p.st_f64[1 * B + i] = L.s.x_dot; p.st_f64[2 * B + i] = L.s.theta;
    p.st_f64[3 * B + i] = L.s.theta_dot; p.st_f64[4 * B + i] = L.s.t;
    p.st_f64[5 * B + i] = L.episode_return;
    p.info[i] = L.raw_return;
    p.st_word[i] = L.nr << 31;
  }
  static BSB_HD void init(const EnvParams&, Lane& L) {
    L.s.x = L.s.x_dot = L.s.theta = L.s.theta_dot = L.s.t = 0.0;   // cartpole.py:89
    L.trig.sn = 0.0; L.trig.cs = 1.0;
    L.episode_return = 0.0; L.raw_return = 0.0; L.nr = 1;
  }
  template <class R> static BSB_HD void ctor_draws(const EnvParams&, Lane&, R&) {}

  template <class R> static BSB_HD StepOut reset(const EnvParams& p, int64_t, Lane& L, R& rng) {
    // cartpole.py:118-128 / cartpole_swingup.py:81-91: four uniform draws in order.
    L.s.x = rng.uniform(-p.init_range, p.init_range);
    L.s.x_dot = rng.uniform(-p.init_range, p.init_range);
    const double th = rng.uniform(-p.init_range, p.init_range);
    L.s.theta = kSwingup ? (3.141592653589793 + th) : th;
    L.s.theta_dot = rng.uniform(-p.init_range, p.init_range);
    L.s.t = 0.0;
    L.trig = sincos_of(L.s.theta);
    L.episode_return = 0.0;
    return make_first();
  }
  template <class R> static BSB_HD StepOut step(const EnvParams& p, int64_t i, Lane& L, int32_t action, R&) {
    L.s = advance_pole(p, L.s, L.trig, action);
    L.trig = sincos_of(L.s.theta);
    double reward; bool done;
    if (!kSwingup) {                                       // cartpole.py:140-153
      const bool ok = L.trig.cs > p.height_threshold && fabs(L.s.x) < p.x_threshold;
      reward = ok ? 1.0 : 0.0;
      done = (L.s.t > p.max_time) || !ok;
    } else {                                               // cartpole_swingup.py:104-123
      const bool upright = L.trig.cs > p.height_threshold &&
                           fabs(L.s.theta_dot) < p.theta_dot_threshold &&
                           fabs(L.s.x) < p.x_reward_threshold;
      const int32_t moved = action - 1 < 0 ? 1 - action : action - 1;
      reward = -1.0 * (double)moved * p.move_cost;         // -0.0 when action == 1
      if (upright) { reward += 1.0; p.info[1 * p.batch + i] += 1.0; }  // total_upright
      done = (L.s.t > p.max_time) || (fabs(L.s.x) > p.x_threshold);
    }
    L.raw_return += reward;
    L.episode_return += reward;
    if (done) {
      double* best = &p.info[(kSwingup ? 2 : 1) * p.batch + i];
      if (L.episode_return > *best) *best = L.episode_return;  // max(episode_return, best_episode)
      return make_last(reward);
    }
    return make_mid(reward);
  }
  // Observation row; dst[k * stride].
  static BSB_HD void row(const EnvParams& p, const Lane& L, float* dst, int64_t stride) {
    dst[0 * stride] = (float)(L.s.x / p.x_threshold);
    dst[1 * stride] = (float)(L.s.x_dot / p.x_threshold);
    dst[2 * stride] = (float)L.trig.sn;
    dst[3 * stride] = (float)L.trig.cs;
    dst[4 * stride] = (float)L.s.theta_dot;
    dst[5 * stride] = (float)(L.s.t / p.max_time);
    if (kSwingup) {
      dst[6 * stride] = fabs(L.s.x) < p.x_reward_threshold ? 1.0f : -1.0f;
      dst[7 * stride] = fabs(L.s.theta_dot) < p.theta_dot_threshold ? 1.0f : -1.0f;
    }
  }
};
typedef CartpoleT<false> Cartpole;
typedef CartpoleT<true> CartpoleSwingup;

// ===========================================================================
// mountain_car  (environments/mountain_car.py)
// ===========================================================================
struct MountainCar {
  static const bool kIsDeepSea = false;
  enum { kObs = 3, kInfo = 1 };  // raw_return (mountain_car.py:101-102)
  struct Lane { double pos, vel, raw_return; uint32_t t, nr; };

  static BSB_HD void load(const EnvParams& p, int64_t i, Lane& L) {
    L.pos = p.st_f64[i]; L.vel = p.st_f64[p.batch + i]; L.raw_return = p.info[i];
    const uint32_t w = p.st_word[i]; L.t = w & 0x7fffffffu; L.nr = w >> 31;
  }
  static BSB_HD void store(const EnvParams& p, int64_t i, const Lane& L) {
    p.st_f64[i] = L.pos; p.st_f64[p.batch + i] = L.vel; p.info[i] = L.raw_return;
    p.st_word[i] = L.t | (L.nr << 31);
  }
  static BSB_HD void init(const EnvParams&, Lane& L) { L.pos = L.vel = L.raw_return = 0.0; L.t = 0; L.nr = 1; }
  template <class R> static BSB_HD void ctor_draws(const EnvParams&, Lane&, R&) {}

  template <class R> static BSB_HD StepOut reset(const EnvParams&, int64_t, Lane& L, R& rng) {
    L.t = 0; L.pos = rng.uniform(-0.6, -0.4); L.vel = 0.0;  // mountain_car.py:66-71
    return make_first();
  }
  template <class R> static BSB_HD StepOut step(const EnvParams& p, int64_t, Lane& L, int32_t action, R&) {
    L.t += 1;                                               // mountain_car.py:74
    const double reward = -1.0;
    L.raw_return += reward;
    // :79-85 with _force=0.001, _gravity=0.0025, speed 0.07, pos in [-1.2, 0.6]
    L.vel += (double)(action - 1) * 0.001 + cos(3.0 * L.pos) * -0.0025;
    L.vel = clampd(L.vel, -0.07, 0.07);
    L.pos += L.vel;
    L.pos = clampd(L.pos, -1.2, 0.6);
    if (L.pos == -1.2) L.vel = clampd(L.vel, 0.0, 0.07);
    if (L.pos >= 0.5 || L.t >= (uint32_t)p.max_steps) return make_last(reward);  // :88-90
    return make_mid(reward);
  }
  static BSB_HD void row(const EnvParams& p, const Lane& L, float* dst, int64_t stride) {
    dst[0] = (float)L.pos; dst[stride] = (float)L.vel;       // mountain_car.py:62-64
    dst[2 * stride] = (float)((double)L.t / (double)p.max_steps);
  }
};

// ===========================================================================
// memory_chain  (environments/memory_chain.py)
// ===========================================================================
struct MemoryChain {
  static const bool kIsDeepSea = false;
  enum { kInfo = 2 };  // total_perfect, total_regret (memory_chain.py:108-111)
  struct Lane { uint32_t t, query, nr, obs_t; uint64_t ctx; };

  static BSB_HD void load(const EnvParams& p, int64_t i, Lane& L) {
    const uint32_t w = p.st_word[i];
    L.t = w & 0xffffffu; L.query = (w >> 24) & 0x7fu; L.nr = w >> 31; L.ctx = p.st_ctx[i]; L.obs_t = L.t;
  }
  static BSB_HD void store(const EnvParams& p, int64_t i, const Lane& L) {
    p.st_word[i] = L.t | (L.query << 24) | (L.nr << 31); p.st_ctx[i] = L.ctx;
  }
  static BSB_HD void init(const EnvParams&, Lane& L) { L.t = 0; L.query = 0; L.nr = 1; L.ctx = 0; L.obs_t = 0; }

  template <class R> static BSB_HD void draw_context(const EnvParams& p, Lane& L, R& rng) {
    uint64_t c = 0;                                          // binomial(1, .5, num_bits), row-major
    c = rng.binomial_half_bits(p.num_bits);
    L.ctx = c;
    L.query = rng.randint((uint32_t)p.num_bits);
  }
  // The constructor draws a context and a query that are never shown
  // (memory_chain.py:49-50): two consumptions before the first reset.
  template <class R> static BSB_HD void ctor_draws(const EnvParams& p, Lane& L, R& rng) { draw_context(p, L, rng); }

  template <class R> static BSB_HD StepOut reset(const EnvParams& p, int64_t, Lane& L, R& rng) {
    L.t = 0; draw_context(p, L, rng); L.obs_t = 0;          // memory_chain.py:91-97
    return make_first();
  }
  template <class R> static BSB_HD StepOut step(const EnvParams& p, int64_t i, Lane& L, int32_t action, R&) {
    L.obs_t = L.t;                                           // observation BEFORE t += 1 (:74-75)
    L.t += 1;
    if (L.t - 1 < (uint32_t)p.memory_length) return make_mid(0.0);       // :77-79
    const int32_t want = (int32_t)((L.ctx >> L.query) & 1ull);            // :83-88
    if (action == want) { p.info[i] += 1.0; return make_last(1.0); }
    p.info[p.batch + i] += 2.0;
    return make_last(-1.0);
  }
  static BSB_HD void row(const EnvParams& p, const Lane& L, float* dst, int64_t stride) {  // :60-71
    dst[0] = (float)(1.0 - (double)L.obs_t / (double)p.memory_length);
    dst[stride] = (L.obs_t == (uint32_t)(p.memory_length - 1)) ? (float)L.query : 0.0f;
    for (int b = 0; b < p.num_bits; ++b)
      dst[(2 + b) * stride] = (L.obs_t == 0) ? (float)(2 * (int32_t)((L.ctx >> b) & 1ull) - 1) : 0.0f;
  }
};

// ===========================================================================
// bandit  (environments/bandit.py)
// ===========================================================================
struct Bandit {
  static const bool kIsDeepSea = false;
  enum { kObs = 1, kInfo = 1 };  // total_regret
  struct Lane { uint32_t nr; };
  static BSB_HD void load(const EnvParams& p, int64_t i, Lane& L) { L.nr = p.st_word[i] >> 31; }
  static BSB_HD void store(const EnvParams& p, int64_t i, const Lane& L) { p.st_word[i] = L.nr << 31; }
  static BSB_HD void init(const EnvParams&, Lane& L) { L.nr = 1; }
  template <class R> static BSB_HD void ctor_draws(const EnvParams&, Lane&, R&) {}
  template <class R> static BSB_HD StepOut reset(const EnvParams&, int64_t, Lane&, R&) { return make_first(); }
  template <class R> static BSB_HD StepOut step(const EnvParams& p, int64_t i, Lane&, int32_t action, R&) {
    const double reward = p.reward_table[action];            // bandit.py:60-64
    p.info[i] += 1.0 - reward;                               // _optimal_return = 1.
    return make_last(reward);
  }
  static BSB_HD void row(const EnvParams&, const Lane&, float* dst, int64_t) { dst[0] = 1.0f; }  // bandit.py:53-54
};

// ===========================================================================
// umbrella_chain  (environments/umbrella_chain.py)
// ===========================================================================
struct UmbrellaChain {
  static const bool kIsDeepSea = false;
  enum { kInfo = 1 };  // total_regret
  struct Lane { uint32_t t, need, has, nr; };
  static BSB_HD void load(const EnvParams& p, int64_t i, Lane& L) {
    const uint32_t w = p.st_word[i];
    L.t = w & 0xffffffu; L.need = (w >> 24) & 1u; L.has = (w >> 25) & 1u; L.nr = w >> 31;
  }
  static BSB_HD void store(const EnvParams& p, int64_t i, const Lane& L) {
    p.st_word[i] = L.t | (L.need << 24) | (L.has << 25) | (L.nr << 31);
  }
  static BSB_HD void init(const EnvParams&, Lane& L) { L.t = 0; L.need = 0; L.has = 0; L.nr = 1; }
  template <class R> static BSB_HD void ctor_draws(const EnvParams&, Lane& L, R& rng) { L.need = (uint32_t)rng.binomial_half(); }  // :55

  template <class R> static BSB_HD StepOut reset(const EnvParams&, int64_t, Lane& L, R& rng) {
    L.t = 0; L.need = (uint32_t)rng.binomial_half(); L.has = (uint32_t)rng.binomial_half();  // :87-92
    return make_first();
  }
  template <class R> static BSB_HD StepOut step(const EnvParams& p, int64_t i, Lane& L, int32_t action, R& rng) {
    L.t += 1;                                                // :69
    if (L.t == 1) L.has = (uint32_t)(action != 0);          // :71-72 (action_spec: {0, 1})
    if (L.t == (uint32_t)p.chain_length) {                   // :74-81
      if (L.has == L.need) return make_last(1.0);
      p.info[i] += 2.0;
      return make_last(-1.0);
    }
    const double reward = 2.0 * (double)rng.binomial_half() - 1.0;  // :83, drawn BEFORE the distractors
    return make_mid(reward);
  }
  // The observation draws n_distractor fresh Bernoullis on EVERY call (:60-66).
  template <class R> static BSB_HD void row(const EnvParams& p, const Lane& L, R& rng, float* dst, int64_t stride) {
    dst[0] = (float)L.need; dst[stride] = (float)L.has;
    dst[2 * stride] = (float)(1.0 - (double)L.t / (double)p.chain_length);
    for (int k0 = 0; k0 < p.n_distractor; k0 += 64) {
      const int n = (p.n_distractor - k0) < 64 ? (p.n_distractor - k0) : 64;
      const uint64_t bits = rng.binomial_half_bits(n);
      for (int k = 0; k < n; ++k) dst[(3 + k0 + k) * stride] = (float)((bits >> k) & 1ull);
    }
  }
};

// ===========================================================================
// discounting_chain  (environments/discounting_chain.py)
// ===========================================================================
struct DiscountingChain {
  static const bool kIsDeepSea = false;
  enum { kObs = 2, kInfo = 0 };  // bsuite_info() == {}
  struct Lane { uint32_t t, nr; int32_t context; };
  static BSB_HD void load(const EnvParams& p, int64_t i, Lane& L) {
    const uint32_t w = p.st_word[i];
    L.t = w & 0xffu; L.context = (int32_t)((w >> 8) & 0xffu) - 1; L.nr = w >> 31;
  }
  static BSB_HD void store(const EnvParams& p, int64_t i, const Lane& L) {
    p.st_word[i] = L.t | ((uint32_t)(L.context + 1) << 8) | (L.nr << 31);
  }
  static BSB_HD void init(const EnvParams&, Lane& L) { L.t = 0; L.context = -1; L.nr = 1; }
  template <class R> static BSB_HD void ctor_draws(const EnvParams&, Lane&, R&) {}
  template <class R> static BSB_HD StepOut reset(const EnvParams&, int64_t, Lane& L, R&) {
    L.t = 0; L.context = -1; return make_first();            // :69-73
  }
  static BSB_HD uint32_t reward_step(int32_t c) {           // _reward_timestep = [1, 3, 10, 30, 100]
    return c == 0 ? 1u : c == 1 ? 3u : c == 2 ? 10u : c == 3 ? 30u : 100u;
  }
  template <class R> static BSB_HD StepOut step(const EnvParams& p, int64_t, Lane& L, int32_t action, R&) {
    if (L.t == 0) L.context = action;                        // :76-77
    L.t += 1;
    const double reward = (L.t == reward_step(L.context)) ? p.reward_table[L.context] : 0.0;  // :80-83
    if (L.t == 100u) return make_last(reward);               // _episode_len = 100
    return make_mid(reward);
  }
  static BSB_HD void row(const EnvParams&, const Lane& L, float* dst, int64_t stride) {  // :63-67
    dst[0] = (float)L.context; dst[stride] = (float)((double)L.t / 100.0);
  }
};

// ===========================================================================
// mnist  (environments/mnist.py)
// ===========================================================================
struct Mnist {
  static const bool kIsDeepSea = false;
  enum { kInfo = 1 };  // total_regret
  struct Lane { uint32_t label, nr; int32_t image; };
  static BSB_HD void load(const EnvParams& p, int64_t i, Lane& L) {
    const uint32_t w = p.st_word[i]; L.label = w & 0xffu; L.nr = w >> 31; L.image = -1;
  }
  static BSB_HD void store(const EnvParams& p, int64_t i, const Lane& L) { p.st_word[i] = L.label | (L.nr << 31); }
  static BSB_HD void init(const EnvParams&, Lane& L) { L.label = 0; L.nr = 1; L.image = -1; }
  template <class R> static BSB_HD void ctor_draws(const EnvParams&, Lane&, R&) {}
  template <class R> static BSB_HD StepOut reset(const EnvParams& p, int64_t, Lane& L, R& rng) {
    L.image = (int32_t)rng.randint((uint32_t)p.num_data);    // mnist.py:63
    L.label = p.labels[L.image];                             // :65
    return make_first();
  }
  template <class R> static BSB_HD StepOut step(const EnvParams& p, int64_t i, Lane& L, int32_t action, R&) {
    const double reward = (action == (int32_t)L.label) ? 1.0 : -1.0;  // :71-72
    p.info[i] += 1.0 - reward;
    L.image = -1;                                            // zeros observation (:74)
    return make_last(reward);
  }
  // image.astype(float32) / 255 (mnist.py:64); images are parsed as INT8 by the
  // reference (utils/datasets.py:55-56), so pixels >= 128 come out negative.
  static BSB_HD float pixel(int8_t v) { return (float)v / 255.0f; }
};

// Logging-wrapper bookkeeping (utils/wrappers.py:85-110) on the wrapped reward.  The reference keeps five columns
// (steps, episode, total_return, episode_len, episode_return); only the two float sums change on every step, so
// only they are carried densely (16 B read + 16 B written per lane-step).  The integer columns follow from three
// values that change at episode boundaries only, because all lanes step in lock-step:
//   ep[0] total_return     dense      ep[1] episode         += 1 at LAST
//   ep[2] episode_return   dense      ep[3] first_count     += 1 at FIRST
//                                     ep[4] start_call      = global call index of the FIRST that followed the
//                                                             latest LAST, + 1 per further FIRST since
//   steps       = calls - first_count              (every call that did not return FIRST is a transition)
//   episode_len = calls - 1 - start_call           (transitions since the latest LAST; 0 before any call)
// The reference zeroes episode_len / episode_return right after logging a LAST timestep (:105-107) and NOT at a
// FIRST: an explicit reset() in the middle of an episode leaves both running.  Here they restart at the first
// call after a LAST (`after_last`: the lane's _reset_next_step flag before the call), so from a LAST timestep --
// the moment the reference writes its row (:99-101) -- until the lane steps again they hold the finished episode's
// values, and a mid-episode reset() only discounts its own non-transition call.
struct EpisodeStats {
  double total_return, episode_return;
  BSB_HD void load(const EnvParams& p, int64_t i) { total_return = p.ep[i]; episode_return = p.ep[2 * p.batch + i]; }
  BSB_HD void store(const EnvParams& p, int64_t i) const { p.ep[i] = total_return; p.ep[2 * p.batch + i] = episode_return; }
  BSB_HD void track(const EnvParams& p, int64_t i, const StepOut& o, int64_t call_index, bool after_last) {
    if (o.step_type == FIRST) {
      p.ep[3 * p.batch + i] += 1.0;
      if (after_last) { episode_return = 0.0; p.ep[4 * p.batch + i] = (double)call_index; }
      else p.ep[4 * p.batch + i] += 1.0;
      return;
    }
    episode_return += o.reward; total_return += o.reward;
    if (o.step_type == LAST) p.ep[p.batch + i] += 1.0;
  }
};

// Column `field` (0 steps, 1 episode, 2 total_return, 3 episode_len, 4 episode_return) of lane i after `calls` calls.
BSB_HD double episode_stat(const EnvParams& p, int64_t i, int field, int64_t calls);

// Does the LAST timestep lane i has just produced fall on the log schedule?  (`episode` already counts it.)
BSB_HD bool log_row_due(const EnvParams& p, int64_t i) {
  const int32_t k = p.log_next[i];
  return k < p.n_log_points && (int64_t)p.ep[p.batch + i] == p.log_sched[k];
}
// Column `col` of the row lane i would record now: the five Logging columns, then bsuite_info().
BSB_HD double row_column(const EnvParams& p, int64_t i, int col, int64_t calls) {
  return col < 5 ? episode_stat(p, i, col, calls) : p.info[(int64_t)(col - 5) * p.batch + i];
}
// Records row k: the five Logging columns and bsuite_info() exactly as the reference's `_log_bsuite_data`
// (wrappers.py:113-125) reads them right after the LAST timestep.
BSB_HD void log_row_write(const EnvParams& p, int64_t i, int32_t k, int64_t calls) {
  const int64_t cols = 5 + p.n_info;
  double* row = p.log_rows + ((int64_t)k * cols) * p.batch + i;
  for (int f = 0; f < 5; ++f) row[(int64_t)f * p.batch] = episode_stat(p, i, f, calls);
  for (int f = 0; f < p.n_info; ++f) row[(int64_t)(5 + f) * p.batch] = p.info[(int64_t)f * p.batch + i];
}
// A row has fallen due (log_row_due): store it if there is a row store, fold it into the score summary if there is
// one, and advance the cursor.  The lane's state, accumulators and info fields must have been stored to memory
// (F::store, EpisodeStats::store) before the call.
BSB_HD void log_point_record(const EnvParams& p, int64_t i, int64_t calls) {
  const int32_t k = p.log_next[i];
  if (p.log_rows) log_row_write(p, i, k, calls);
  if (p.score_sum)
    scoring::fold_row(p.score_sum, i, p.batch, p.score_exp, k, episode_stat(p, i, 1, calls),
                      row_column(p, i, p.score_col_value, calls),
                      p.score_col_best >= 0 ? row_column(p, i, p.score_col_best, calls) : NAN);
  p.log_next[i] = k + 1;
}

BSB_HD double episode_stat(const EnvParams& p, int64_t i, int field, int64_t calls) {
  const int64_t B = p.batch;
  switch (field) {
    case 0: return (double)calls - p.ep[3 * B + i];
    case 1: return p.ep[B + i];
    case 2: return p.ep[i];
    case 3: return p.ep[3 * B + i] == 0.0 ? 0.0 : (double)(calls - 1) - p.ep[4 * B + i];
    default: return p.ep[2 * B + i];
  }
}

}  // namespace bsb
