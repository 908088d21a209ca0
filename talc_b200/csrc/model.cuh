// model.cuh -- count prediction intervals and successor tagging (SURVEY rows a11, a23).
//
// Decisions are made in IEEE double with separate multiply/add (the reference's x86-64 build has
// no FMA: SURVEY F7), so this file must be compiled with -fmad=false; std::pow(x,2) is x*x.
#pragma once
#include <math.h>

#include "defs.cuh"

namespace talc {

enum Tag : u8 { kExpected = 0, kUnexpected = 1, kBreakpoint = 2 };

// Explorer.cpp:1185-1198.  upper==true is the reference's `classe == UNEXPECTED` branch (noise upper
// bound), upper==false the `EXPECTED` branch (lower bound).  sqrt of a negative value is NaN and
// makes the comparison false (cc = 0 lower bound).
TALC_HDN bool expected_by_model(u32 nextc, u32 cc, double alpha, bool upper) {
  if (cc <= 3) {
    if (upper) return ((double)nextc <= ((double)(cc + 0.5) + alpha * sqrt((double)(cc + 0.5))));
    return ((double)nextc >= ((double)(cc - 0.5) + (1 - alpha) * sqrt((double)(cc - 0.5))));
  }
  if (upper) {
    const double x = (alpha / 2 + sqrt((double)(cc + 0.96)));
    return ((double)nextc <= x * x);
  }
  const double y = (alpha / 2 - sqrt((double)(cc + 0.02)));
  return ((double)nextc >= y * y);
}

// Explorer.cpp:1200-1217
TALC_HDN bool expected_by_last_node(u32 nextc, u32 cc, double alpha) {
  return expected_by_model(nextc, cc, alpha, true) & expected_by_model(nextc, cc, alpha, false);
}

// The two interval bounds a step needs, each evaluated once instead of once per successor: the lower
// bound of the "expected" interval around the current count (Explorer.cpp:1191,1196) and the upper
// bound of the noise interval around lambda = (int)(count * SR_ERROR_RATE) (Explorer.cpp:1190,1195).
// Same expressions, same operation order as expected_by_model, so the comparisons are bit-identical.
TALC_HD double model_lower_bound(u32 cc, double alpha) {
  if (cc <= 3) return ((double)(cc - 0.5) + (1 - alpha) * sqrt((double)(cc - 0.5)));  // NaN for cc = 0
  const double y = (alpha / 2 - sqrt((double)(cc + 0.02)));
  return y * y;
}
TALC_HD double model_upper_bound(u32 cc, double alpha) {
  if (cc <= 3) return ((double)(cc + 0.5) + alpha * sqrt((double)(cc + 0.5)));
  const double x = (alpha / 2 + sqrt((double)(cc + 0.96)));
  return x * x;
}

// Per-step constants of the tagging rules: they depend on the current count only, so the caller can
// evaluate them while the four table probes are still in flight.
struct StepBounds {
  double lower;       // lower bound of the "expected" interval around count
  double upperNoise;  // upper bound of the noise interval around lambda (valid iff noiseModel)
  double sq;          // sqrt(count), the denominator of dist = |count - next| / sqrt(count)  (Explorer.cpp:1247)
  u32 lambda;         // (int)(count * SR_ERROR_RATE)
  bool noiseModel;    // lambda >= MIN_COUNT
};
TALC_HDN StepBounds step_bounds(u32 count, const Params& P) {
  StepBounds b;
  b.lambda = (u32)(i32)((double)count * P.sr_error);
  b.noiseModel = b.lambda >= P.min_count;
  b.lower = model_lower_bound(count, P.alpha);
  b.upperNoise = b.noiseModel ? model_upper_bound(b.lambda, P.alpha) : 0.0;
  b.sq = sqrt((double)count);
  return b;
}
// The same constants from per-context lookup tables (filled on the device by model_tabs_kernel with the very
// functions above, so the values are bit-identical); counts beyond the table are computed.
struct ModelTabs {
  const double* lower;  // model_lower_bound(c, alpha)
  const double* upper;  // model_upper_bound(c, alpha)
  const double* sq;     // sqrt((double)c)
  u32 n;
};
static const u32 kModelTabN = 16384;  // counts with tabulated bounds on the device
// Indexing M.upper[lambda] below relies on lambda <= count, i.e. on 0 <= sr_error <= 1: talc_ctx_create refuses any
// rate outside [0, 0.5].
TALC_HD StepBounds step_bounds_tab(u32 count, const Params& P, const ModelTabs& M) {
  if (count >= M.n) return step_bounds(count, P);
  StepBounds b;
  b.lambda = (u32)(i32)((double)count * P.sr_error);
  b.noiseModel = b.lambda >= P.min_count;
  b.lower = M.lower[count];
  b.upperNoise = b.noiseModel ? M.upper[b.lambda] : 0.0;  // lambda <= count < n
  b.sq = M.sq[count];
  return b;
}
TALC_HD double step_dist(u32 count, u32 nextc, const StepBounds& b) {
  return fabs((double)count - (double)nextc) / b.sq;
}

// Explorer.cpp:1226-1298.  Returns the number of tags (0 on a dead end, else 4).  The distance of a
// successor is step_dist(); the reference only ever reads it for successors that are not UNEXPECTED.
TALC_HDN int tag_next_nodes(const u32 cnt[4], const u32 col[4], const StepBounds& B, const Params& P, bool complex_,
                           u8 tag[4]) {
  int counter = 0;
  u32 nbExpected = 0, nbBreakpoints = 0, nbUnexpected = 0;
  for (int i = 0; i < 4; ++i)
    if (cnt[i] >= P.min_count) counter++;
  if (counter == 0) return 0;
  for (int b = 0; b < 4; ++b) {
    const u32 nextc = cnt[b];
    if (nextc >= P.min_count) {
      if (((double)nextc >= B.lower) || (counter == 1)) {
        tag[b] = kExpected;
        ++nbExpected;
      } else if (B.noiseModel) {
        if (!((double)nextc <= B.upperNoise) || (col[b] > 0)) {
          tag[b] = kBreakpoint;
          ++nbBreakpoints;
        } else {
          tag[b] = kUnexpected;
          ++nbUnexpected;
        }
      } else {
        tag[b] = kBreakpoint;
        ++nbBreakpoints;
      }
    } else
      tag[b] = kUnexpected;  // not counted in nbUnexpected (:1275)
  }
  if ((nbExpected == 0) & (nbBreakpoints == 1)) {
    for (int t = 0; t < 4; ++t)
      if (tag[t] == kBreakpoint) tag[t] = kExpected;
  }
  if ((nbExpected == 1) & (nbUnexpected > 0) & !complex_) {
    int sum = 0;
    u32 index = 0;
    for (u32 i = 0; i < 4; ++i) {
      if (tag[i] == kUnexpected) {
        if (sum == 0) index = i;
        sum += (int)cnt[i];
        if (cnt[index] < cnt[i]) index = i;
      }
    }
    // nbUnexpected > 0 implies the noise model is active, so upperNoise is valid
    if (!((double)(u32)sum <= B.upperNoise)) tag[index] = kBreakpoint;
  }
  return 4;
}

// The prediction intervals of expected_by_model / expected_by_last_node from the per-context tables (Explorer.cpp:
// 1185-1217, bit for bit: the tables hold model_lower_bound / model_upper_bound themselves); counts beyond them are
// computed.
TALC_HD bool expected_upper_tab(u32 nextc, u32 cc, const Params& P, const ModelTabs& M) {
  if (cc < M.n) return (double)nextc <= M.upper[cc];
  return expected_by_model(nextc, cc, P.alpha, true);
}
TALC_HD bool expected_last_node_tab(u32 nextc, u32 cc, const Params& P, const ModelTabs& M) {
  if (cc < M.n) return ((double)nextc <= M.upper[cc]) & ((double)nextc >= M.lower[cc]);
  return expected_by_last_node(nextc, cc, P.alpha);
}

// The child of a fast-walk step (Corrector::fast_walk, walk_kernel): a bucket with more than one successor in the
// graph goes through the exact tagger (complex_ = false, as the walk is never in a complex region when it takes the
// fast path); -1 unless exactly one successor is admissible.  Rare on the fast path, kept out of line.
TALC_HDN int pick_single_child(const u32 c4[4], u32 cm, u32 count, const Params& P, const ModelTabs& tabs) {
  u32 col4[4];
  TALC_ROLLED
  for (int i = 0; i < 4; ++i) col4[i] = (cm >> i) & 1u;
  const StepBounds sb = step_bounds_tab(count, P, tabs);
  u8 tag[4];
  tag_next_nodes(c4, col4, sb, P, false, tag);
  int child = -1, n = 0;
  TALC_ROLLED
  for (int i = 0; i < 4; ++i)
    if (tag[i] != kUnexpected) { child = i; ++n; }
  return n == 1 ? child : -1;
}
// The only successor in the graph is EXPECTED by the counter == 1 rule and needs no tagging; none is a dead end (-1).
TALC_HD int fast_step_child(const u32 c4[4], u32 cm, u32 count, const Params& P, const ModelTabs& tabs) {
  const u32 minCount = P.min_count;
  const u32 m = (u32)(c4[0] >= minCount) | ((u32)(c4[1] >= minCount) << 1) | ((u32)(c4[2] >= minCount) << 2) |
                ((u32)(c4[3] >= minCount) << 3);
  if (m != 0 && (m & (m - 1)) == 0) {
#if defined(__CUDA_ARCH__)
    return __ffs((int)m) - 1;
#else
    return __builtin_ctz(m);
#endif
  }
  if (m != 0) return pick_single_child(c4, cm, count, P, tabs);
  return -1;
}

// One query of talc_test_model (include/talc_b200.h) on the functions above, for the device self-test and the host
// emulation alike.  a[8]: ops 0-2 {count, c4[4], colmask, complex, -}, ops 3-4 {nextc, cc, ...}; out[9] (doubles as
// their bits): op 0 {lower, upperNoise, sq, lambda, noiseModel}; op 1 {tags, tag[4], step_dist[4]}; op 2 {child as
// int64}; ops 3-4 {0 / 1}.
TALC_HD u64 double_bits(double d) {
  u64 u;
  memcpy(&u, &d, 8);
  return u;
}
TALC_HDN void selftest_model_op(int op, const u32 a[8], const Params& P, const ModelTabs& M, u64 out[9]) {
  for (int q = 0; q < 9; ++q) out[q] = 0;
  const u32 c4[4] = {a[1], a[2], a[3], a[4]};
  if (op == 0) {
    const StepBounds b = step_bounds_tab(a[0], P, M);
    out[0] = double_bits(b.lower);
    out[1] = double_bits(b.upperNoise);
    out[2] = double_bits(b.sq);
    out[3] = b.lambda;
    out[4] = b.noiseModel ? 1 : 0;
  } else if (op == 1) {
    u32 col4[4];
    for (int i = 0; i < 4; ++i) col4[i] = (a[5] >> i) & 1u;
    const StepBounds sb = step_bounds_tab(a[0], P, M);
    u8 tag[4] = {kUnexpected, kUnexpected, kUnexpected, kUnexpected};
    const int n = tag_next_nodes(c4, col4, sb, P, a[6] != 0, tag);
    out[0] = (u64)n;
    for (int i = 0; i < n; ++i) {
      out[1 + i] = tag[i];
      out[5 + i] = double_bits(step_dist(a[0], c4[i], sb));
    }
  } else if (op == 2) {
    out[0] = (u64)(i64)fast_step_child(c4, a[5], a[0], P, M);
  } else if (op == 3) {
    out[0] = expected_upper_tab(a[0], a[1], P, M) ? 1 : 0;
  } else if (op == 4) {
    out[0] = expected_last_node_tab(a[0], a[1], P, M) ? 1 : 0;
  }
}

}  // namespace talc
