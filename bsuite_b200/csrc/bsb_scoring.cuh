// Scoring rules of the reference's analysis (experiments/<name>/analysis.py::score, utils/plotting.py:57-77,
// experiments/summary_analysis.py:103-173), restated over one lane's log rows.  One code path: the CUDA kernel and
// the host loop of bsb_scoring.cu call the same __host__ __device__ functions, and every sum is taken in the same
// fixed order (numpy's pairwise order, NpSum), so both give the same bits (the build uses --fmad=false and
// -ffp-contract=off).
//
// A lane's DataFrame for one experiment is its rows of the experiment's ids, one id after the other, each id's rows
// ascending in episode -- what csv_load builds from the lane's CSV files.  The functions below never materialise
// it: they read `counts`, the rows a rule selects (mostly the last row of each id), and nothing else.
#pragma once
#include <math.h>
#include <stdint.h>

#include "../../include/bsuite_b200.h"

#if defined(__CUDACC__)
#define BSB_SC_HD __host__ __device__ inline
#else
#define BSB_SC_HD inline
#endif

namespace bsb {
namespace scoring {

constexpr int kMaxSourcesPerExperiment = 128;   // NpSum restates numpy's pairwise sum for n <= 128 terms
constexpr int kMaxPoints = 4096;

// One bsuite_id's rows or score summary (bsb_score_source, as uploaded).  Within an experiment the descriptors of a
// grouping rule are sorted by group key (stable), so a group is a contiguous run.
struct ScoreDesc {
  const double* rows;      // [n_points][n_columns][B] (BSB_SCORE_ROWS) or [kSummaryFields][B] (BSB_SCORE_SUMMARY)
  const int32_t* counts;   // [B]
  int32_t n_points, n_columns, col_episode, col_value, col_best, layout;
  double key;
};

// Descriptor range of one experiment, and the layouts among them: kViewRows, kViewSummary or kViewMixed.
struct ScoreExp { int32_t first, count, view, pad; };
enum View : int32_t { kViewRows, kViewSummary, kViewMixed };

enum Rule : int32_t {
  kRegret,          // bandit, catch (+ _noise / _scale): ave_regret_score on total_regret
  kCartpole,        // cartpole_preprocess + 50% regret, 50% best_episode > 500
  kSwingup,         // cp_swingup_preprocess, per height_threshold: 50% regret, 50% best_episode > 100
  kMountainCar,     // mountain_car_preprocess + ave_regret_score
  kMnist,           // 50% regret, 50% final accuracy (episodes > 0.9 NUM_EPISODES)
  kDeepSea,         // find_solution: solved and below 2^size + 100
  kDiscounting,     // 1 - 10 (1.1 - average return), clipped
  kMemory,          // per memory_length / num_bits: regret ratio < 0.75
  kUmbrella,        // per chain_length / n_distractor: regret < 0.5
};

struct ExpInfo {
  int32_t rule;
  int32_t scaling;         // score_by_scaling over the group key (the _noise / _scale experiments)
  int32_t grouped;         // the group key is read (scaling, swingup, deep_sea, memory, umbrella)
  int32_t min_episode;     // deep_sea_stochastic drops episodes < 100 first
  double base;             // BASE_REGRET, or the threshold of deep_sea / memory / umbrella
  double num_episodes;     // NUM_EPISODES of the experiment's sweep.py
  uint32_t tags;           // bit t = bsb_tag t
};

#define BSB_T(t) (1u << BSB_TAG_##t)
BSB_SC_HD ExpInfo exp_info(int e) {
  switch (e) {
    case BSB_EXP_BANDIT: return {kRegret, 0, 0, 0, 0.5, 10000., BSB_T(BASIC)};
    case BSB_EXP_BANDIT_NOISE: return {kRegret, 1, 1, 0, 0.5, 10000., BSB_T(NOISE)};
    case BSB_EXP_BANDIT_SCALE: return {kRegret, 1, 1, 0, 0.5, 10000., BSB_T(SCALE)};
    case BSB_EXP_CARTPOLE: return {kCartpole, 0, 0, 0, 1000., 1000., BSB_T(BASIC) | BSB_T(CREDIT_ASSIGNMENT) | BSB_T(GENERALIZATION)};
    case BSB_EXP_CARTPOLE_NOISE: return {kCartpole, 1, 1, 0, 1000., 1000., BSB_T(NOISE) | BSB_T(GENERALIZATION)};
    case BSB_EXP_CARTPOLE_SCALE: return {kCartpole, 1, 1, 0, 1000., 1000., BSB_T(SCALE) | BSB_T(GENERALIZATION)};
    case BSB_EXP_CARTPOLE_SWINGUP: return {kSwingup, 0, 1, 0, 700., 1000., BSB_T(EXPLORATION) | BSB_T(GENERALIZATION)};
    case BSB_EXP_CATCH: return {kRegret, 0, 0, 0, 1.6, 10000., BSB_T(BASIC) | BSB_T(CREDIT_ASSIGNMENT)};
    case BSB_EXP_CATCH_NOISE: return {kRegret, 1, 1, 0, 1.6, 10000., BSB_T(NOISE) | BSB_T(CREDIT_ASSIGNMENT)};
    case BSB_EXP_CATCH_SCALE: return {kRegret, 1, 1, 0, 1.6, 10000., BSB_T(SCALE) | BSB_T(CREDIT_ASSIGNMENT)};
    case BSB_EXP_DEEP_SEA: return {kDeepSea, 0, 1, 0, 0.9, 10000., BSB_T(EXPLORATION)};
    case BSB_EXP_DEEP_SEA_STOCHASTIC: return {kDeepSea, 0, 1, 100, 0.8, 10000., BSB_T(EXPLORATION) | BSB_T(NOISE)};
    case BSB_EXP_DISCOUNTING_CHAIN: return {kDiscounting, 0, 0, 0, 0., 1000., BSB_T(CREDIT_ASSIGNMENT)};
    case BSB_EXP_MEMORY_LEN: return {kMemory, 0, 1, 0, 0.75, 10000., BSB_T(MEMORY)};
    case BSB_EXP_MEMORY_SIZE: return {kMemory, 0, 1, 0, 0.75, 10000., BSB_T(MEMORY)};
    case BSB_EXP_MNIST: return {kMnist, 0, 0, 0, 1.8, 10000., BSB_T(BASIC) | BSB_T(GENERALIZATION)};
    case BSB_EXP_MNIST_NOISE: return {kMnist, 1, 1, 0, 1.8, 10000., BSB_T(NOISE) | BSB_T(GENERALIZATION)};
    case BSB_EXP_MNIST_SCALE: return {kMnist, 1, 1, 0, 1.8, 10000., BSB_T(SCALE) | BSB_T(GENERALIZATION)};
    case BSB_EXP_MOUNTAIN_CAR: return {kMountainCar, 0, 0, 0, 1000., 1000., BSB_T(BASIC) | BSB_T(GENERALIZATION)};
    case BSB_EXP_MOUNTAIN_CAR_NOISE: return {kMountainCar, 1, 1, 0, 1000., 1000., BSB_T(NOISE) | BSB_T(GENERALIZATION)};
    case BSB_EXP_MOUNTAIN_CAR_SCALE: return {kMountainCar, 1, 1, 0, 1000., 1000., BSB_T(SCALE) | BSB_T(GENERALIZATION)};
    case BSB_EXP_UMBRELLA_DISTRACT: return {kUmbrella, 0, 1, 0, 0.5, 10000., BSB_T(CREDIT_ASSIGNMENT) | BSB_T(NOISE)};
    case BSB_EXP_UMBRELLA_LENGTH: return {kUmbrella, 0, 1, 0, 0.5, 10000., BSB_T(CREDIT_ASSIGNMENT) | BSB_T(NOISE)};
  }
  return {-1, 0, 0, 0, 0., 0., 0u};
}
#undef BSB_T

BSB_SC_HD bool rule_needs_best(int rule) { return rule == kCartpole || rule == kSwingup; }
// cartpole, cartpole_swingup and deep_sea keep only episode <= NUM_EPISODES (their preprocessors / find_solution)
BSB_SC_HD bool rule_caps_episodes(int rule) { return rule == kCartpole || rule == kSwingup || rule == kDeepSea; }

// Score summary of one id and lane (bsb_read_score_summary), field f at summary[f * B + lane].
enum SummaryField { kLastEpisode, kLastValue, kPrevEpisode, kPrevValue, kBest, kFirstSolved, kSummaryFields };
static_assert(kSummaryFields == BSB_SCORE_SUMMARY_FIELDS, "summary layout");

// Folds row k (k rows came before it) of one lane into its summary.  The rows of an id are a prefix of the log
// schedule, so the rules need only what is folded here (Lane<SummaryView> below): the latest row (the row at
// n_eps of mean_regret_at_last, _is_finished, the last episode of deep_sea), the row before it (mnist's diff()
// term: 10 000 is the only schedule point past 0.9 NUM_EPISODES), the running max of best_episode in the scan's
// own comparison order (solved_fraction), and deep_sea's first solved episode among the rows range() keeps.
// episode, value and best are the row's columns col_episode, col_value and col_best, the doubles the row store
// holds; `best` is not read where the rule has no best_episode.
BSB_SC_HD void fold_row(double* summary, int64_t lane, int64_t B, int experiment, int32_t k, double episode,
                        double value, double best) {
  const ExpInfo info = exp_info(experiment);
  double* s = summary + lane;
  if (k == 0) {
    s[kPrevEpisode * B] = NAN; s[kPrevValue * B] = NAN; s[kBest * B] = NAN; s[kFirstSolved * B] = NAN;
  } else {
    s[kPrevEpisode * B] = s[kLastEpisode * B]; s[kPrevValue * B] = s[kLastValue * B];
  }
  s[kLastEpisode * B] = episode; s[kLastValue * B] = value;
  if (rule_needs_best(info.rule) && (k == 0 || best > s[kBest * B])) s[kBest * B] = best;
  if (info.rule == kDeepSea && !(s[kFirstSolved * B] == s[kFirstSolved * B]) &&
      !(episode < (double)info.min_episode) && !(episode > info.num_episodes) && value / episode < info.base)
    s[kFirstSolved * B] = episode;
}

// numpy's pairwise summation (the order of np.sum / np.mean and of pandas' Series.mean) for n <= 128 terms, fed
// one term at a time: below 8 terms a running sum; otherwise 8 interleaved partial sums, combined as
// ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)), then the n % 8 trailing terms one by one.
struct NpSum {
  double r[8];
  double res;
  int i, n, blocked;
  BSB_SC_HD explicit NpSum(int count) : res(0.0), i(0), n(count), blocked(count - count % 8) {
    for (int j = 0; j < 8; ++j) r[j] = 0.0;
  }
  BSB_SC_HD double tree() const { return ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7])); }
  BSB_SC_HD void add(double x) {
    if (n < 8) res += x;
    else if (i < 8) r[i] = x;
    else if (i < blocked) r[i & 7] += x;
    else { if (i == blocked) res = tree(); res += x; }
    ++i;
  }
  BSB_SC_HD double sum() const { return (n >= 8 && blocked == n) ? tree() : res; }
};

BSB_SC_HD double clip01(double x) { return x < 0.0 ? 0.0 : (x > 1.0 ? 1.0 : x); }   // np.clip keeps NaN

// What the rules read of one id's rows, over the row store (RowView: the scans) or a score summary (SummaryView:
// the folded fields).  Row indices are those of the row store; a summary holds the last two rows of an id only,
// which is every row the rules index (see fold_row), and reads NaN elsewhere.
struct RowView {
  const ScoreDesc* d;      // the experiment's descriptors
  int64_t lane, B;
  ExpInfo info;

  BSB_SC_HD double at(int s, int k, int col) const {
    return d[s].rows[((int64_t)k * d[s].n_columns + col) * B + lane];
  }
  BSB_SC_HD double ep(int s, int k) const { return at(s, k, d[s].col_episode); }
  BSB_SC_HD double value(int s, int k) const { return at(s, k, d[s].col_value); }
  BSB_SC_HD int count(int s) const {
    int c = d[s].counts[lane];
    return c < 0 ? 0 : (c > d[s].n_points ? d[s].n_points : c);
  }
  // Rows [lo, hi) of id s that the rule keeps (episodes ascending, so the filters cut a prefix and a suffix).
  BSB_SC_HD void range(int s, int* lo, int* hi) const {
    int h = count(s), l = 0;
    if (rule_caps_episodes(info.rule))
      while (h > 0 && ep(s, h - 1) > info.num_episodes) --h;
    if (info.min_episode > 0)
      while (l < h && ep(s, l) < (double)info.min_episode) ++l;
    *lo = l; *hi = h;
  }
  // Row of id s with episode == e inside [lo, hi), or -1 (at most one: episodes are distinct within an id).
  BSB_SC_HD int row_at_episode(int s, int lo, int hi, double e) const {
    int k = hi - 1;
    while (k >= lo && ep(s, k) > e) --k;
    return (k >= lo && ep(s, k) == e) ? k : -1;
  }
  // max of best_episode over rows [lo, hi) (hi > lo), in the order of np.max's scan.
  BSB_SC_HD double best(int s, int lo, int hi) const {
    double best = at(s, lo, d[s].col_best);
    for (int k = lo + 1; k < hi; ++k) { const double b = at(s, k, d[s].col_best); if (b > best) best = b; }
    return best;
  }
  // Episode of the first row in [lo, hi) with value / episode < threshold (deep_sea's find_solution).
  BSB_SC_HD bool first_solved(int s, int lo, int hi, double* first) const {
    for (int k = lo; k < hi; ++k) {
      const double e = ep(s, k);
      if (value(s, k) / e < info.base) { *first = e; return true; }
    }
    return false;
  }
};

struct SummaryView {
  const ScoreDesc* d;
  int64_t lane, B;
  ExpInfo info;

  BSB_SC_HD double field(int s, int f) const { return d[s].rows[(int64_t)f * B + lane]; }
  BSB_SC_HD double ep(int s, int k) const {
    const int c = count(s);
    return k == c - 1 ? field(s, kLastEpisode) : (k == c - 2 ? field(s, kPrevEpisode) : NAN);
  }
  BSB_SC_HD double value(int s, int k) const {
    const int c = count(s);
    return k == c - 1 ? field(s, kLastValue) : (k == c - 2 ? field(s, kPrevValue) : NAN);
  }
  BSB_SC_HD int count(int s) const {
    int c = d[s].counts[lane];
    return c < 0 ? 0 : (c > d[s].n_points ? d[s].n_points : c);
  }
  // Every row of a schedule prefix is <= NUM_EPISODES (no cap), and the rows below min_episode are a prefix of
  // them: the rule keeps rows iff the last one is kept.  lo is only handed back to the queries below.
  BSB_SC_HD void range(int s, int* lo, int* hi) const {
    const int h = count(s);
    *hi = h;
    *lo = (h > 0 && info.min_episode > 0 && field(s, kLastEpisode) < (double)info.min_episode) ? h : 0;
  }
  // e is a schedule point whenever the rules ask (an id's last episode, or a first solved one), so the kept rows
  // hold it iff min_episode <= e <= last.  Only the last row is ever read back; an earlier one is reported as lo.
  BSB_SC_HD int row_at_episode(int s, int lo, int hi, double e) const {
    if (hi <= lo) return -1;
    const double last = field(s, kLastEpisode);
    if (e == last) return hi - 1;
    return (e < last && !(e < (double)info.min_episode)) ? lo : -1;
  }
  BSB_SC_HD double best(int s, int, int) const { return field(s, kBest); }
  BSB_SC_HD bool first_solved(int s, int, int, double* first) const {
    const double f = field(s, kFirstSolved);
    if (!(f == f)) return false;
    *first = f;
    return true;
  }
};

// Sources of both layouts within one experiment: each id is read through its own descriptor's view.
struct MixedView {
  RowView r;
  SummaryView m;
  BSB_SC_HD bool sm(int s) const { return r.d[s].layout == BSB_SCORE_SUMMARY; }
  BSB_SC_HD double ep(int s, int k) const { return sm(s) ? m.ep(s, k) : r.ep(s, k); }
  BSB_SC_HD double value(int s, int k) const { return sm(s) ? m.value(s, k) : r.value(s, k); }
  BSB_SC_HD int count(int s) const { return sm(s) ? m.count(s) : r.count(s); }
  BSB_SC_HD void range(int s, int* lo, int* hi) const { if (sm(s)) m.range(s, lo, hi); else r.range(s, lo, hi); }
  BSB_SC_HD int row_at_episode(int s, int lo, int hi, double e) const {
    return sm(s) ? m.row_at_episode(s, lo, hi, e) : r.row_at_episode(s, lo, hi, e);
  }
  BSB_SC_HD double best(int s, int lo, int hi) const { return sm(s) ? m.best(s, lo, hi) : r.best(s, lo, hi); }
  BSB_SC_HD bool first_solved(int s, int lo, int hi, double* first) const {
    return sm(s) ? m.first_solved(s, lo, hi, first) : r.first_solved(s, lo, hi, first);
  }
};

// One lane of one experiment, read through view V.
template <class V>
struct Lane {
  V v;
  const ScoreDesc* d;      // the experiment's descriptors
  ExpInfo info;

  BSB_SC_HD double ep(int s, int k) const { return v.ep(s, k); }
  BSB_SC_HD double value(int s, int k) const { return v.value(s, k); }
  BSB_SC_HD int count(int s) const { return v.count(s); }
  BSB_SC_HD void range(int s, int* lo, int* hi) const { v.range(s, lo, hi); }
  BSB_SC_HD int row_at_episode(int s, int lo, int hi, double e) const { return v.row_at_episode(s, lo, hi, e); }
  // The column ave_regret_score averages, as the preprocessors derive it.
  BSB_SC_HD double regret(int s, int k) const {
    const double e = ep(s, k), v = value(s, k);
    switch (info.rule) {
      case kCartpole: return 1000.0 * e - v;        // BASE_REGRET * episode - raw_return
      case kSwingup: return e * 700.0 - v;          // episode * BASE_REGRET - total_return
      case kMountainCar: return -100.0 * e - v;     // _SOLVED_STEPS * -1 * episode - raw_return
      case kMemory: return (e - v) / 0.5;           // (episode - total_perfect) / base_rate
      default: return v;
    }
  }
  BSB_SC_HD bool any_rows(int s0, int s1) const {
    for (int s = s0; s < s1; ++s) { int lo, hi; range(s, &lo, &hi); if (hi > lo) return true; }
    return false;
  }

  // mean of the regret column over the rows at episode n_eps = min(max episode, NUM_EPISODES) of ids [s0, s1),
  // divided by n_eps (plotting.ave_regret_score before its normalisation; memory / umbrella score_by_group).
  BSB_SC_HD double mean_regret_at_last(int s0, int s1) const {
    double max_ep = 0.0;
    bool any = false;
    for (int s = s0; s < s1; ++s) {
      int lo, hi; range(s, &lo, &hi);
      if (hi > lo) { const double e = ep(s, hi - 1); if (!any || e > max_ep) max_ep = e; any = true; }
    }
    const double n_eps = max_ep < info.num_episodes ? max_ep : info.num_episodes;
    int n = 0;
    for (int s = s0; s < s1; ++s) { int lo, hi; range(s, &lo, &hi); n += row_at_episode(s, lo, hi, n_eps) >= 0; }
    NpSum sum(n);
    for (int s = s0; s < s1; ++s) {
      int lo, hi; range(s, &lo, &hi);
      const int k = row_at_episode(s, lo, hi, n_eps);
      if (k >= 0) sum.add(regret(s, k));
    }
    return (sum.sum() / (double)n) / n_eps;
  }
  BSB_SC_HD double ave_regret_score(int s0, int s1) const {
    const double mean_regret = mean_regret_at_last(s0, s1);
    return clip01((info.base - mean_regret) / info.base);
  }
  // np.mean(groupby('bsuite_id').best_episode.max() > good) over the ids with rows.
  BSB_SC_HD double solved_fraction(int s0, int s1, double good) const {
    int ids = 0, hits = 0;
    for (int s = s0; s < s1; ++s) {
      int lo, hi; range(s, &lo, &hi);
      if (hi <= lo) continue;
      const double best = v.best(s, lo, hi);
      ++ids; hits += best > good;
    }
    return (double)hits / (double)ids;
  }
  // mnist's final-accuracy term: np.mean(1 - diff(total_regret) / diff(episode) + 1) * 0.5 over the rows with
  // episode > 0.9 NUM_EPISODES; diff() is against the previous row of the frame (the same id's, except for an
  // id's first row, whose predecessor is the previous id's last row; the frame's first row has none: NaN, skipped).
  BSB_SC_HD double mnist_accuracy(int s0, int s1) const {
    const double cut = 0.9 * info.num_episodes;
    int n = 0;
    for (int s = s0; s < s1; ++s) {
      int k = count(s);
      while (k > 0 && ep(s, k - 1) > cut) { --k; ++n; }
    }
    NpSum sum(n);
    int valid = 0, prev_s = -1;
    for (int s = s0; s < s1; ++s) {
      const int c = count(s);
      if (c == 0) continue;
      int k0 = c;
      while (k0 > 0 && ep(s, k0 - 1) > cut) --k0;
      for (int k = k0; k < c; ++k) {
        double r_prev = NAN, e_prev = NAN;
        if (k > 0) { r_prev = value(s, k - 1); e_prev = ep(s, k - 1); }
        else if (prev_s >= 0) { const int pc = count(prev_s); r_prev = value(prev_s, pc - 1); e_prev = ep(prev_s, pc - 1); }
        const double ave_return = 1.0 - ((value(s, k) - r_prev) / (ep(s, k) - e_prev));
        const double term = ave_return + 1.0;
        if (term == term) { sum.add(term); ++valid; } else sum.add(0.0);
      }
      prev_s = s;
    }
    return (sum.sum() / (double)valid) * 0.5;
  }

  // The score of one group of ids for the rules that score_by_scaling applies per noise / reward scale.
  BSB_SC_HD double base_score(int s0, int s1) const {
    switch (info.rule) {
      case kRegret:
      case kMountainCar: return ave_regret_score(s0, s1);
      case kCartpole: return 0.5 * (ave_regret_score(s0, s1) + solved_fraction(s0, s1, 500.0));
      case kMnist: return 0.5 * (ave_regret_score(s0, s1) + mnist_accuracy(s0, s1));
    }
    return NAN;
  }

  BSB_SC_HD int next_group(int s, int end) const {
    int t = s + 1;
    while (t < end && d[t].key == d[s].key) ++t;
    return t;
  }

  // plotting.score_by_scaling: 0.5 (clip(mean) + clip(mean - std)) over the groups' scores (population std).
  BSB_SC_HD double scaling_score(int end) const {
    int m = 0;
    for (int s = 0; s < end; s = next_group(s, end)) m += any_rows(s, next_group(s, end));
    NpSum total(m);
    for (int s = 0; s < end; s = next_group(s, end)) {
      const int t = next_group(s, end);
      if (any_rows(s, t)) total.add(base_score(s, t));
    }
    const double mean = total.sum() / (double)m;
    NpSum squares(m);
    for (int s = 0; s < end; s = next_group(s, end)) {
      const int t = next_group(s, end);
      if (any_rows(s, t)) { const double x = base_score(s, t) - mean; squares.add(x * x); }
    }
    const double std = sqrt(squares.sum() / (double)m);
    return 0.5 * (clip01(mean) + clip01(mean - std));
  }

  // cartpole_swingup: mean over height_threshold groups of 0.5 (regret score + fraction with best_episode > 100).
  BSB_SC_HD double swingup_score(int end) const {
    int m = 0;
    for (int s = 0; s < end; s = next_group(s, end)) m += any_rows(s, next_group(s, end));
    NpSum total(m);
    for (int s = 0; s < end; s = next_group(s, end)) {
      const int t = next_group(s, end);
      if (any_rows(s, t)) total.add(0.5 * (ave_regret_score(s, t) + solved_fraction(s, t, 100.0)));
    }
    return total.sum() / (double)m;
  }

  // memory_len / memory_size / umbrella_*: fraction of groups whose mean regret at their last episode is < base.
  BSB_SC_HD double threshold_score(int end) const {
    int m = 0, hits = 0;
    for (int s = 0; s < end; s = next_group(s, end)) {
      const int t = next_group(s, end);
      if (!any_rows(s, t)) continue;
      ++m; hits += mean_regret_at_last(s, t) < info.base;
    }
    return (double)hits / (double)m;
  }

  // deep_sea(_stochastic).find_solution + score: per size, the first episode with total_bad_episodes / episode
  // < thresh (else the last episode, unsolved); merged back onto the rows at that (size, episode), and the score
  // is the fraction of those rows that are solved before 2^size + 100.
  BSB_SC_HD double deep_sea_score(int end) const {
    int rows = 0, hits = 0;
    for (int s = 0; s < end; s = next_group(s, end)) {
      const int t = next_group(s, end);
      bool solved = false, any = false;
      double first = 0.0, last = 0.0;
      for (int u = s; u < t; ++u) {
        int lo, hi; range(u, &lo, &hi);
        if (hi <= lo) continue;
        const double e_last = ep(u, hi - 1);
        if (!any || e_last > last) last = e_last;
        any = true;
        double e;
        if (v.first_solved(u, lo, hi, &e)) {
          if (!solved || e < first) first = e;
          solved = true;
        }
      }
      if (!any) continue;
      const double e = solved ? first : last;
      const bool beat = solved && e < pow(2.0, d[s].key) + 100.0;
      for (int u = s; u < t; ++u) {
        int lo, hi; range(u, &lo, &hi);
        if (row_at_episode(u, lo, hi, e) >= 0) { ++rows; hits += beat; }
      }
    }
    return (double)hits / (double)rows;
  }

  // discounting_chain: 1 - 10 (1.1 - mean total_return at the last episode / n_eps), clipped.
  BSB_SC_HD double discounting_score(int end) const {
    const double ave_return = mean_regret_at_last(0, end);      // regret() is total_return for this rule
    return clip01(1. - 10. * (1.1 - ave_return));
  }
};

struct ScoreOut { double score; int32_t finished; int32_t present; };

template <class V>
BSB_SC_HD ScoreOut score_lane_as(const Lane<V>& L, int n) {
  ScoreOut out = {NAN, 0, 0};
  // _is_finished: every id with rows has reached NUM_EPISODES (on the unfiltered rows)
  double min_last = 0.0;
  bool any = false;
  for (int s = 0; s < n; ++s) {
    const int c = L.count(s);
    if (c == 0) continue;
    const double e_last = L.ep(s, c - 1);
    if (!any || e_last < min_last) min_last = e_last;
    any = true;
  }
  if (!any) return out;                       // not scored: the experiment is absent from the lane's frame
  out.present = 1;
  out.finished = min_last >= L.info.num_episodes;
  if (L.info.scaling) { out.score = L.scaling_score(n); return out; }
  switch (L.info.rule) {
    case kSwingup: out.score = L.swingup_score(n); break;
    case kDeepSea: out.score = L.deep_sea_score(n); break;
    case kDiscounting: out.score = L.discounting_score(n); break;
    case kMemory:
    case kUmbrella: out.score = L.threshold_score(n); break;
    default: out.score = L.base_score(0, n); break;
  }
  return out;
}

BSB_SC_HD ScoreOut score_lane(const ScoreDesc* descs, ScoreExp ex, int e, int64_t lane, int64_t B) {
  if (ex.count <= 0) return ScoreOut{NAN, 0, 0};
  const ScoreDesc* d = descs + ex.first;
  const ExpInfo info = exp_info(e);
  const RowView rows{d, lane, B, info};
  const SummaryView summary{d, lane, B, info};
  switch (ex.view) {
    case kViewSummary: return score_lane_as(Lane<SummaryView>{summary, d, info}, ex.count);
    case kViewMixed: return score_lane_as(Lane<MixedView>{MixedView{rows, summary}, d, info}, ex.count);
  }
  return score_lane_as(Lane<RowView>{rows, d, info}, ex.count);
}

// ave_score_by_tag for one lane: pandas' NaN-skipping mean over the scored experiments carrying the tag (NaN
// scores count as 0 in the pairwise sum and are left out of the count, as pandas does).
BSB_SC_HD double tag_average(int tag, const double* score, const int32_t* present, int stride) {
  int n = 0;
  for (int e = 0; e < BSB_NUM_EXPERIMENTS; ++e) n += present[e * stride] && (exp_info(e).tags >> tag & 1u);
  NpSum sum(n);
  int valid = 0;
  for (int e = 0; e < BSB_NUM_EXPERIMENTS; ++e) {
    if (!present[e * stride] || !(exp_info(e).tags >> tag & 1u)) continue;
    const double x = score[e * stride];
    if (x == x) { sum.add(x); ++valid; } else sum.add(0.0);
  }
  return sum.sum() / (double)valid;
}

}  // namespace scoring
}  // namespace bsb
