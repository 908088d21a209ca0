// correct.cuh -- per-read segmentation, anchor selection, bounded de Bruijn graph search and
// path scoring (SURVEY rows a4-a24).  One WARP owns one read: the gaps of a read form a dependency chain
// (SURVEY F5) and a frontier holds 1-3 trails for most steps, so the parallelism is across reads; inside a
// read the 32 lanes run the control code on identical data (no divergence) and split every primitive --
// trails of the frontier (fast_walk), windows of the cycle test, blocks / columns / diagonals of the scoring
// routines (align.cuh, xdrop.cuh), k-mers of a ballot (find_in_regions).  On the host (tests/hostemu) a
// "warp" is one lane and the same TALC_HD code runs scalar.
//
// The kernel is bound by instruction delivery (DESIGN.md section 5): loops of the control code stay rolled
// (TALC_ROLLED), rare paths sit out of line, and one routine serves where several would be faster apart.
//
// Reference files restated here (all under /root/reference/src):
//   Read.cpp:174-386,440-600   Explorer.cpp:155-297,402-1118   Trail.cpp:48-131,193-216,273-338
//   Trajectory.cpp:43-48,89-243,282-334,482-528
// The quirks listed in SURVEY A.7 (Q1-Q23) are reproduced on purpose; each is tagged where it occurs.
#pragma once
#include "align.cuh"
#include "defs.cuh"
#include "model.cuh"
#include "stdsort.cuh"
#include "table.cuh"

// the bodies of the general steps: real calls (TALC_HDN) or inlined into their one caller per kernel (TALC_HD)
#ifndef TALC_STEPFN
#define TALC_STEPFN TALC_HDN
#endif

namespace talc {

struct Counters {
  u64 lookups_seg, lookups_deg, lookups_walk;
  u64 steps_inner, steps_border, frontier_sum;
  u64 cells_nw, cells_lcs, cells_ovl, cells_xdrop;
  u64 gaps, gaps_bridged, gap_attempts, borders, borders_corrected;
  u64 ev_gardening, ev_bridge, ev_edge, ev_cycle;
  u64 bases_out, reads_ok, reads_overflow;
};
static const int kNumCounters = sizeof(Counters) / sizeof(u64);

struct Region {
  u32 start, end;  // k-mer coordinates, inclusive
};

struct AnchorRec {  // anchorTuple (kmer, position, count)
  u64 kmer;
  u32 pos;
  u32 count;
};

struct Trail {  // Trail.hpp:95-107 minus the sequence, which lives in a packed slot
  u64 kmer;     // last k-mer
  double dist;  // m_distance
  u32 count;    // last count
  i32 score;    // m_lastScore (always integral)
  u16 slot;
  u8 failures;  // m_nbFailuresInARow
  u8 pad;
};

struct GardenRank {
  u32 idx, r1, r2, sum;
};
struct GardenKey {
  u32 idx;
  i32 score;
  double dist;
};

// one corrected piece of the read, as ASCII in the persistent arena; len < 0 means "raw slice kept"
struct Piece {
  u32 off;
  i32 len;
};

// a candidate correction of a border (Trajectory after trim/reshape/cutAnchors), kept only while it
// is the running best of its list (findBestBORDER is a left fold: Trajectory.cpp:306-334, Q21)
struct EdgeBest {
  bool have;
  double score;     // NW score of the final extension
  double idscore;   // LCS / longer
  double md;        // mean distance (Q22)
  u32 path_keep;    // walk-order prefix of the trail that is kept (before anchor removal)
  u32 ref_from;     // then the raw border from this walk index on (only when `shorter`), else == ref.len
  u32 anchor_pos;   // whichStart of the anchor that produced it
  i32 ref_start;    // RefView of that anchor
  u32 ref_len;
  u64* seq;         // packed copy of the kept prefix
};

struct ReadJob {
  ReadView rd;
  const u32* cov;   // coverage counts of this read, C = len-K+1 entries
  u8* arena;        // per-thread scratch slice
  u32 arena_bytes;
  bool wide;        // second tier: worst-case buffer sizing
};

struct ReadOut {
  u8 status;
  u32 out_len;
};

class Corrector {
 public:
  TableView T;
  CtxView CR, CL;  // successor tables for RIGHT- and LEFT-ward questions (device only)
  Params P;
  ModelTabs tabs;  // n == 0: no tables (host emulation)
  ReadView rd;
  const u64* rdw;  // the read packed (keep arena): 2 bits per base, or 4 when it holds an N
  u32 rdlg;        // 5 or 4
  const u32* cov;
  u32 C;  // number of k-mers
  Arena keep;     // persistent per-read data: regions, pieces
  Arena scratch;  // per-attempt data
  bool wide;
  Counters* ctr;  // per-read tallies (may be null); the caller adds them to the batch totals
  DpStats dps;

  // --- structure
  Region* regs;
  u32 nregs;
  Piece* gapPiece;  // nregs-1 entries
  Piece headPiece, tailPiece;
  bool headPresent, tailPresent;
  double noise;  // m_priorLambda_noise

  // --- explorer state
  Region L, R;
  int location;  // 0 HEAD, 1 INNER, 2 TAIL
  bool dirRight;
  bool complexRegion;  // Q12: sticky for the rest of the read
  AnchorRec* ancL;
  u32 nAncL;
  AnchorRec* ancR;
  u32 nAncR;
  u32 weakLen;

  // --- search state
  u32 slotWords, nSlots, nFree;
  u64* slotPool;
  u16* freeList;
  Trail* cur;
  Trail* nxt;
  u32 nCur, nNxt, maxT;

  // --- resumable control flow.  The per-read program (run -> search_bridge / search_edge) is a state machine whose
  // loop variables live in these frames, so a read can be suspended where a long walk starts -- the walk then runs in
  // its own kernel (walk.cuh), one trail per lane next to the trails of other reads -- and resumed afterwards from
  // its context in HBM.  Without splitWalk (host emulation, tuning builds) nothing ever yields.
  enum : u8 { kStepFalse = 0, kStepTrue = 1, kStepYield = 2 };
  struct WalkReq {  // what the walk kernel needs besides cur[] / the slots, and what it hands back (step)
    const AnchorRec* aims;
    u32 nAims, step, pathMax, border;
  };
  struct RunFrame {
    u32 pc, reg;
    int attempt;
    bool success;
  };
  struct BridgeFrame {
    u32 pc, s, limit, mk0, whichStart, gapLen, pathMax, step;
    u32 maxBridges, maxKeep, nBr, nBrSeq;
    RefView ref;
    void* br;      // BridgeRec[maxBridges]
    u64* brSeq;
    i32 runScore;
    double runMd;
    bool runHave, found;
  };
  struct EdgeFrame {
    u32 pc, s, limit, mk0, whichStart, pathMax, step;
    int xdrop;
    RefView ref;
    EdgeBest bestLong, bestShort;
  };
  // A suspended read also gives its warp back when it has run for pauseBudget SM cycles since it was resumed (host
  // emulation: general steps): the control kernel works in rounds, and one read with a 500-base border would
  // otherwise hold a whole round for as long as its X-drop extensions take.  wq.border == 2 marks such a pause: the
  // walk kernel passes the context straight on.
  long long tResume;
  u32 pauseBudget, pauseCount;
  u32 inlineInner, inlineBorder;  // ordinary steps a warp still takes by itself before it hands the frontier over
  WalkReq wq;
  RunFrame fr;
  BridgeFrame fb;
  EdgeFrame fe;
  ReadJob job_;
  u32 splitWalk;  // 1: hand long walks to the walk kernel (yield), 0: walk inline

  TALC_HD u32 K() const { return P.K; }

  // ------------------------------------------------------------------ prediction intervals from the per-context tables
  TALC_HD bool expected_upper_tab(u32 nextc, u32 cc) { return talc::expected_upper_tab(nextc, cc, P, tabs); }
  TALC_HD bool expected_last_node_tab(u32 nextc, u32 cc) { return talc::expected_last_node_tab(nextc, cc, P, tabs); }

  // ------------------------------------------------------------------ table access with counters
  // a k-mer holding N: its successors x[1..]+b may or may not hold N; look each one up by bases (rare, out of line)
  TALC_HDN int out_degree_with_n(u32 pos, bool right) {
    int d = 0;
    for (u32 b = 0; b < 4; ++b) {
      bool ok2 = true;
      u64 v = 0;
      for (u32 j = 0; j < K(); ++j) {
        u32 c;
        if (right) c = (j + 1 < K()) ? rd.code(pos + j + 1) : b;
        else c = (j == 0) ? b : rd.code(pos + j - 1);
        if (c > 3) { ok2 = false; break; }
        v = (v << 2) | c;
      }
      if (ok2) {
        u32 cn, cl;
        table_lookup(T, v, cn, cl);
        d += (cn >= P.min_count) ? 1 : 0;
      }
    }
    return d;
  }
  TALC_HDN int out_degree(u32 pos, bool right) {
    if (ctr) ctr->lookups_deg += 4;
    bool ok = true;
    const u64 km = (rdlg == 5u) ? path_kmer_fwd(rdw, pos, K()) : rd.kmer_at(pos, K(), ok);
    if (!ok) return out_degree_with_n(pos, right);
#if defined(__CUDA_ARCH__)
    {  // one bucket of the successor table holds all four counts
      u32 c4[4], cm;
      ctx_lookup(right ? CR : CL, ctx_of(km, right, K()), c4, cm);
      return (int)(c4[0] >= P.min_count) + (int)(c4[1] >= P.min_count) + (int)(c4[2] >= P.min_count) + (int)(c4[3] >= P.min_count);
    }
#else
    return table_out_degree(T, km, right, K(), P.min_count);
#endif
  }
  // the four successor counts / junction flags of a k-mer in the search direction (getNextCountsFromDBG)
  TALC_HD void next_counts(u64 kmer, u32 cnt[4], u32 col[4]) {
#if defined(__CUDA_ARCH__)
    u32 cm;
    ctx_lookup(dirRight ? CR : CL, ctx_of(kmer, dirRight, K()), cnt, cm);
#pragma unroll
    for (int i = 0; i < 4; ++i) col[i] = (cm >> i) & 1u;  // only "colour > 0" is ever tested (Explorer.cpp:1258)
#else
    table_next_counts(T, kmer, dirRight, K(), cnt, col);
#endif
  }

  // ------------------------------------------------------------------ Read.cpp:493-518
  // robust mean over the [15%,90%) slice of the sorted in-counts, computed without sorting: the sum
  // of the r smallest values is exact in integers (and in double below 2^53), so order is irrelevant
  TALC_HDN u64 sum_of_smallest(u32 r, u32 maxv) {  // sum of the r smallest values among counts >= MIN
    if (r == 0) return 0;
    int top = 7;
    while (top > 0 && ((maxv >> (4 * top)) & 15u) == 0) --top;  // leading zero nibbles of the maximum
    u32 prefix = 0, remaining = r;
    u64 sumBelow = 0;
    const u32 lane = lane_id(), nl = lane_count();
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int nib = top; nib >= 0; --nib) {  // radix select, most significant nibble first
      u32 hist[16];
      u64 hsum[16];
      TALC_ROLLED
      for (int i = 0; i < 16; ++i) { hist[i] = 0; hsum[i] = 0; }
      const u32 shift = 4 * nib;
      const u32 himask = (nib == 7) ? 0u : (~0u << (shift + 4));
      TALC_ROLLED
      for (u32 i = lane; i < C; i += nl) {  // each lane bins every nl-th count
        const u32 v = cov[i];
        if (v < P.min_count) continue;
        if ((v & himask) != (prefix & himask)) continue;
        const u32 d = (v >> shift) & 15u;
        hist[d] += 1u;
        hsum[d] += (u64)v;
      }
      u32 d = 15;
      bool found = false;
      TALC_ROLLED
      for (int q = 0; q < 16; ++q) {
        const u32 h = warp_sum(hist[q]);
        const u64 hs = warp_sum64(hsum[q]);
        if (!found) {
          if (h >= remaining || q == 15) { d = (u32)q; found = true; }
          else { remaining -= h; sumBelow += hs; }
        }
      }
      prefix |= d << shift;
    }
    // `remaining` copies of value `prefix` complete the r smallest
    return sumBelow + (u64)remaining * prefix;
  }

  TALC_HDN double seq_error_threshold() {
    u32 n = 0, maxv = 0;
    TALC_ROLLED
    for (u32 i = lane_id(); i < C; i += lane_count()) {
      n += (cov[i] >= P.min_count) ? 1 : 0;
      maxv = cov[i] > maxv ? cov[i] : maxv;
    }
    n = warp_sum(n);
    maxv = warp_max(maxv);
    u32 first, last;
    if (n > 10) {
      first = (u32)(0.15 * (double)n);
      last = (u32)(0.90 * (double)n);
    } else {
      first = 0;
      last = n;
    }
    double robMean = (double)P.min_count;  // Q2
    const u64 s = sum_of_smallest(last, maxv) - sum_of_smallest(first, maxv);
    robMean += (double)s;
    robMean /= (double)(last - first);
    return robMean * P.sr_error;
  }

  // ------------------------------------------------------------------ Read.cpp:440-489
  TALC_HDN bool find_in_regions() {
#if defined(__CUDA_ARCH__)
    // 32 k-mers per ballot: a run starts where a set bit follows a clear one (carry = last bit of the previous
    // word) and ends where a clear bit follows a set one; C <= 1 yields no region (Read.cpp:446)
    const u32 lane = threadIdx.x & 31u;
    TALC_ROLLED
    for (int pass = 0; pass < 2; ++pass) {
      u32 n = 0, cs = 0, carry = 0;
      if (C > 1) {
        TALC_ROLLED
        for (u32 base = 0; base < C; base += 32) {
          const u32 pos = base + lane;
          const u32 m = __ballot_sync(0xffffffffu, pos < C && cov[pos] >= P.min_count);
          const u32 prev = (m << 1) | carry;
          u32 starts = m & ~prev, ends = ~m & prev;  // bit i: k-mer base+i opens / is the first one after a run
          carry = m >> 31;
          while (starts | ends) {
            const u32 fs = starts ? (u32)__ffs((int)starts) - 1 : 32u, fe = ends ? (u32)__ffs((int)ends) - 1 : 32u;
            if (fs < fe) {
              cs = base + fs;
              starts &= starts - 1;
            } else {
              if (pass) { regs[n].start = cs; regs[n].end = base + fe - 1; }
              ++n;
              ends &= ends - 1;
            }
          }
        }
        if (carry) {  // the last run reaches the end of the read
          if (pass) { regs[n].start = cs; regs[n].end = C - 1; }
          ++n;
        }
      }
      if (!pass) {
        nregs = n;
        regs = (Region*)keep.alloc((n ? n : 1) * sizeof(Region));
        if (!regs) return false;
      }
    }
    __syncwarp();
    return nregs > 0;
#else
    // first pass counts, second pass fills
    u32 n = 0;
    bool state = false;
    if (C > 1) {
      TALC_ROLLED
      for (u32 pos = 0; pos < C; ++pos) {
        const bool in = cov[pos] >= P.min_count;
        if (in & !state) state = true;
        else if (!in & state) { ++n; state = false; }
      }
      if (state) ++n;
    }
    nregs = n;
    regs = (Region*)keep.alloc((n ? n : 1) * sizeof(Region));
    if (!regs) return false;
    u32 k = 0, cs = 0;
    state = false;
    if (C > 1) {
      TALC_ROLLED
      for (u32 pos = 0; pos < C; ++pos) {
        const bool in = cov[pos] >= P.min_count;
        if (in & !state) { cs = pos; state = true; }
        else if (!in & state) { regs[k].start = cs; regs[k].end = pos - 1; ++k; state = false; }
      }
      if (state) { regs[k].start = cs; regs[k].end = C - 1; ++k; }
    }
    return n > 0;
#endif
  }

  // ------------------------------------------------------------------ Read.cpp:524-600
  TALC_HDN void analyze_in_regions(double thr) {
    // kept regions overwrite the front of a second array; the input list is mutated in place (Q5)
    Region* kept = (Region*)keep.alloc((nregs ? nregs : 1) * sizeof(Region));
    if (!kept) return;
    u32 nk = 0;
    TALC_ROLLED
    for (u32 reg = 0; reg < nregs; ++reg) {
      int span = 0;
      bool OK = true;
      u32 ns = regs[reg].start;
      const bool lastAndNone = ((nregs == reg + 1) & (nk == 0));
      const int degL = out_degree(ns, false);
      if (!lastAndNone & (degL == 0) & (ns != 0)) {
        OK = false;
        while ((ns < regs[reg].end) & !OK) {
          ++ns;
          if (out_degree(ns, false) > 1) OK = true;  // Q3
        }
      }
      u32 ne = regs[reg].end;
      if (OK & !lastAndNone) {
        const int degR = out_degree(ne, true);
        if ((degR == 0) & (ne != C - 1)) {
          OK = false;
          while ((ne > regs[reg].start) & !OK) {  // Q4
            --ne;
            if (out_degree(ne, true) > 1) OK = true;
          }
        }
      }
      if (OK) {
        if (reg + 1 < nregs) span = ((int)regs[reg + 1].start - (int)(ne + K()));
        if (span < 0) {
          if ((int)regs[reg + 1].end + span >= (int)regs[reg + 1].start) regs[reg + 1].start -= span;
          else {
            regs[reg + 1].start = ns;
            OK = false;
          }
        }
        if (OK) {
          u32 c = 0;
          TALC_ROLLED
          for (u32 i = ns; i <= ne; ++i) c = c < cov[i] ? cov[i] : c;
          if (!expected_upper_tab(c, (u32)thr)) {
            kept[nk].start = ns;
            kept[nk].end = ne;
            ++nk;
          }
        }
      }
    }
    if (nk > 0) {
      TALC_ROLLED
      for (u32 i = 0; i < nk; ++i) regs[i] = kept[i];
      nregs = nk;
    }
  }

  // ------------------------------------------------------------------ Read.cpp:214-258
  TALC_HDN bool initial_structure() {
    const u32 Lr = rd.len;
    u64 len = 0;
    headPresent = tailPresent = false;
    if (regs[0].start > 0) { headPresent = true; len += regs[0].start; }
    if (regs[nregs - 1].end + 1 < C) { tailPresent = true; len += Lr - (regs[nregs - 1].end + K()); }
    TALC_ROLLED
    for (u32 i = 0; i + 1 < nregs; ++i) {
      if (regs[i].end + K() < regs[i].start) return false;  // undefined in the reference; cannot sum to L
      len += regs[i].end + K() - regs[i].start;
      if (regs[i + 1].start > regs[i].end + K()) len += regs[i + 1].start - (regs[i].end + K());
    }
    if (regs[nregs - 1].end + K() < regs[nregs - 1].start) return false;
    len += regs[nregs - 1].end + K() - regs[nregs - 1].start;
    return len == Lr;
  }

  // ------------------------------------------------------------------ Explorer.cpp:402-411
  TALC_HDN void sort_anchors(AnchorRec* a, u32 n) {
    if (n < 2) return;
    const int cc = (int)(noise / P.sr_error);
    const u32 mk = scratch.mark();
    SortKey* keys = (SortKey*)scratch.alloc(n * sizeof(SortKey));
    AnchorRec* tmp = (AnchorRec*)scratch.alloc(n * sizeof(AnchorRec));
    if (!keys || !tmp) return;
    TALC_ROLLED
    for (u32 i = 0; i < n; ++i) {
      int d = cc - (int)a[i].count;
      keys[i].key = d < 0 ? -(i64)d : (i64)d;
      keys[i].idx = i;
      tmp[i] = a[i];
    }
    std_sort_keys(keys, n);
    TALC_ROLLED
    for (u32 i = 0; i < n; ++i) a[i] = tmp[keys[i].idx];
    scratch.release(mk);
  }

  TALC_HD u64 read_kmer(u32 pos) {  // anchors sit on k-mers with count >= MIN, hence without N
    if (rdlg == 5u) return path_kmer_fwd(rdw, pos, K());
    bool ok;
    return rd.kmer_at(pos, K(), ok);
  }

  // Explorer.cpp:413-478 (LEFT region: scan from its last k-mer down) and :480-543 (RIGHT region:
  // scan from its first k-mer up).  `left` selects which.
  TALC_HDN bool build_anchors(bool left) {
    const Region& rg = left ? L : R;
    const u32 nbKmers = rg.end - rg.start + 1;
    const u32 pivot = left ? rg.end : rg.start;
    const u32 limit = left ? rg.start : rg.end;
    const u32 want = kMinStartAnchors < nbKmers ? (u32)kMinStartAnchors : nbKmers;
    // anchorPos has at most nbKmers entries; anchors at most that plus the top-up
    u32* anchorPos = (u32*)scratch.alloc(nbKmers * 4);
    AnchorRec* out = (AnchorRec*)scratch.alloc((nbKmers + 4) * sizeof(AnchorRec));
    if (!anchorPos || !out) return false;
    u32 nPos = 0, nOut = 0;
    bool goFurther = true;
    double current_count = (double)cov[pivot];
    double next_count = 0;
    u32 j = pivot;
    anchorPos[nPos++] = pivot;
    while (goFurther & (left ? (j >= limit + 1) : ((j + 1) <= limit))) {
      const u32 q = left ? j - 1 : j + 1;
      next_count = (double)cov[q];
      if ((next_count >= P.min_count) & (next_count < kMaxInCount))
        goFurther = expected_last_node_tab((u32)next_count, (u32)current_count);
      else goFurther = false;
      if (!goFurther & (current_count >= P.min_count) & (next_count >= P.min_count) & (next_count < kMaxInCount)) {
        anchorPos[nPos++] = q;
        goFurther = true;
        current_count = next_count;
      }
      if (left) --j; else ++j;
    }
    TALC_ROLLED
    for (u32 anc = 0; anc < nPos; ++anc) {
      const int degree = out_degree(anchorPos[anc], left);  // LEFT region looks RIGHT, and vice versa
      if ((anc == 0) || ((anc != 0) & (degree > 1))) {
        out[nOut].kmer = read_kmer(anchorPos[anc]);
        out[nOut].pos = anchorPos[anc];
        out[nOut].count = cov[anc];  // Q6: coverage index is the loop index, not the position
        ++nOut;
      }
    }
    if (nOut < want) {
      j = pivot;
      goFurther = true;
      while ((left ? (j >= limit + 1) : ((j + 1) <= limit)) & (nOut < want)) {
        const u32 q = left ? j - 1 : j + 1;
        if (nOut > 0) goFurther &= (out[0].pos != q);  // Q7: only index 0 is ever examined
        if (!goFurther) break;  // sticky: the reference spins on without any effect (Q8)
        {
          const int degree = out_degree(q, left);
          if (degree > 1) {
            out[nOut].kmer = read_kmer(q);
            out[nOut].pos = q;
            out[nOut].count = cov[q];
            ++nOut;
          }
        }
        --j;  // Q8: the RIGHT-hand variant also decrements; j wraps below zero and the loop ends
      }
    }
    sort_anchors(out, nOut);
    if (left) { ancL = out; nAncL = nOut; }
    else { ancR = out; nAncR = nOut; }
    return true;
  }

  // ------------------------------------------------------------------ trail slots
  TALC_HDN bool setup_search(u32 pathMax) {
    slotWords = (K() + pathMax + 2 + 31) / 32 + 1;
    // frontier bound: <= 50 trails between steps (Explorer.cpp:940,1055), x4 children, plus the Q16 duplicates
    // (the MAX_NB_BRANCHES best by distance are pushed before the whole list is pushed again)
    maxT = 4u * kMaxInnerPaths + P.max_branches + 1u;
    cur = (Trail*)scratch.alloc(maxT * sizeof(Trail));
    nxt = (Trail*)scratch.alloc(maxT * sizeof(Trail));
    if (!cur || !nxt) return false;
    // slots: as many as fit, up to one per possible trail (cur + nxt) plus a few spares
    const u32 wantSlots = 2 * maxT + 8;
    u32 avail = scratch.cap - scratch.top;
    // leave room for DP scratch (horizontal deltas, X-drop diagonals, bridge copies)
    avail -= avail / 2;
    u32 n = avail / (slotWords * 8 + 2);
    if (n > wantSlots) n = wantSlots;
    if (n < 6) { scratch.overflow = 1; return false; }
    nSlots = n;
    freeList = (u16*)scratch.alloc(n * 2);
    slotPool = (u64*)scratch.alloc(n * slotWords * 8);
    if (!freeList || !slotPool) return false;
    nFree = n;
    TALC_ROLLED
    for (u32 i = lane_id(); i < n; i += lane_count()) freeList[i] = (u16)(n - 1 - i);
    warp_sync();
    nCur = nNxt = 0;
    return true;
  }
  TALC_HD u64* slot_ptr(u32 s) { return slotPool + (u64)s * slotWords; }
  TALC_HD int slot_alloc() {
    if (nFree == 0) { scratch.overflow = 1; return -1; }
    return (int)freeList[--nFree];
  }
  TALC_HD void slot_free(u32 s) { freeList[nFree++] = (u16)s; }
  TALC_HD void slot_copy(u32 dst, u32 src, u32 nbases) {
    const u32 nw = (nbases + 31) / 32;
    u64* d = slot_ptr(dst);
    const u64* s = slot_ptr(src);
    TALC_ROLLED
    for (u32 i = lane_id(); i < nw; i += lane_count()) d[i] = s[i];  // the warp's lanes share the copy
    warp_sync();
  }

  // root trail: the anchor k-mer in walk order (Trail.cpp:57-65)
  TALC_HDN bool push_root(const AnchorRec& a) {
    const int s = slot_alloc();
    if (s < 0) return false;
    u64* w = slot_ptr((u32)s);
    TALC_ROLLED
    for (u32 i = 0; i < slotWords; ++i) w[i] = 0;
    TALC_ROLLED
    for (u32 i = 0; i < K(); ++i) {
      // walk order: RIGHT = k-mer as is, LEFT = k-mer reversed
      const u32 src = dirRight ? i : (K() - 1 - i);
      const u32 c = (u32)((a.kmer >> (2 * (K() - 1 - src))) & 3ull);
      path_set(w, i, c);
    }
    Trail t;
    t.kmer = a.kmer;
    t.dist = 0;
    t.count = cov[a.pos];
    t.score = 0;
    t.slot = (u16)s;
    t.failures = 0;
    t.pad = 0;
    cur[0] = t;
    nCur = 1;
    return true;
  }

  // Trail.cpp:289-302 + SeqAn Finder/Pattern<Horspool>: does the child's last k-mer already occur in
  // the parent's sequence, first occurrence at a position > 0 (Q17)?  parent sequence = slot, plen bases.
  TALC_HDN bool already_got_there(u64 needle, const u64* w, u32 plen) {
    const u32 k = K();
    if (!(plen > k)) return false;
    const u32 stride = (P.cycle_mode == 0) ? k : 1u;
#if defined(__CUDA_ARCH__)
    {  // one window per lane; the first occurrence is the lowest lane of the first batch that matches
      u64 nd = needle;
      if (!dirRight) {
        nd = 0;
        TALC_ROLLED
        for (u32 i = 0; i < k; ++i) nd |= ((needle >> (2 * i)) & 3ull) << (2 * (k - 1 - i));
      }
      const u32 lane = threadIdx.x & 31u;
      TALC_ROLLED
      for (u32 base = 0; (u64)base * stride + k <= plen; base += 32) {
        const u32 p = (base + lane) * stride;
        bool match = false;
        if (p + k <= plen) match = path_kmer_fwd(w, dirRight ? p : (plen - k - p), k) == nd;
        const u32 mm = __ballot_sync(0xffffffffu, match);
        if (mm) return ((base + (u32)__ffs((int)mm) - 1) * stride) > 0;
      }
      return false;
    }
#endif
    if (dirRight) {
      TALC_ROLLED
      for (u32 p = 0; p + k <= plen; p += stride)
        if (path_kmer_fwd(w, p, k) == needle) return p > 0;
      return false;
    }
    // LEFT: actual sequence is the reversed walk; actual window p <-> walk window plen-k-p, reversed
    u64 rev = 0;
    TALC_ROLLED
    for (u32 i = 0; i < k; ++i) rev |= ((needle >> (2 * i)) & 3ull) << (2 * (k - 1 - i));
    TALC_ROLLED
    for (u32 p = 0; p + k <= plen; p += stride)
      if (path_kmer_fwd(w, plen - k - p, k) == rev) return p > 0;
    return false;
  }


  TALC_HD bool should_pause() {
    if (!splitWalk || !pauseBudget) return false;
#if defined(__CUDA_ARCH__)
    const int mine = (clock64() - tResume) > (long long)pauseBudget ? 1 : 0;
    return __shfl_sync(0xffffffffu, mine, 0) != 0;  // one decision per warp
#else
    return (++pauseCount % pauseBudget) == 0;
#endif
  }
  TALC_HD void mark_resumed() {
#if defined(__CUDA_ARCH__)
    tResume = clock64();
#endif
  }
  // a frontier the fast path (and the walk kernel, walk.cuh) can take: every trail in its own lane of a group
  TALC_HD bool walk_eligible(u32 nAims) const { return !(nCur == 0 || nCur > 7 || nCur > P.max_branches || nAims > 32); }

  // ------------------------------------------------------------------ single-trail fast path
  // The frontier holds one trail for ~96% of all steps (oracle counters).  While it does, and the step
  // is an ordinary one -- exactly one admissible successor, no aim reached, no cycle, no pruning point --
  // the step only touches registers, the table and the trail's packed sequence.  Anything else ends the
  // run *before* the step, and the general code below redoes that step in full; the two are therefore
  // interchangeable step by step and the result cannot depend on which one ran.
  // border == false: oneMoreStep (Explorer.cpp:546-612); border == true: oneMoreStepInTheDark (:615-687).
  // maxSteps bounds the run; returns true when the run ended on that bound (the trail was still walking)
  TALC_HDN bool fast_walk_scalar(u32& step, u32 pathMax, const AnchorRec* aims, u32 nAims, bool border, u32 maxSteps) {
    if (nCur != 1) return false;
    bool capped = false;
    const u32 k = P.K;
    const bool right = dirRight;
    Trail tr = cur[0];
    u64* w = slot_ptr(tr.slot);
    u64 kmer = tr.kmer;
    u32 count = tr.count;
    double dsum = tr.dist;
    u32 st = step;
    u32 nSteps = 0;
    const u32 stride = (P.cycle_mode == 0) ? k : 1u;
    const u64 kmask = kmer_mask(k);
    u64 rkmer = 0;  // the last k-mer with its bases in reverse order
    TALC_ROLLED
    for (u32 i = 0; i < k; ++i) rkmer |= ((kmer >> (2 * i)) & 3ull) << (2 * (k - 1 - i));
    // the word of the packed sequence that is being filled lives in a register
    u32 cwIdx = (k + st) >> 5;
    u64 cw = w[cwIdx];
    while (st < pathMax) {
      if (border && ((st + 1) % kCheckInterval == 0)) break;  // scoreEdges is due after this step
      if (nSteps >= maxSteps) { capped = true; break; }
      const u32 plen = k + st;
      u32 cnt[4], col[4];
      NextProbe probe;
      table_next_issue(T, kmer, right, k, probe);          // 8 loads in flight ...
      const StepBounds sb = step_bounds_tab(count, P, tabs);  // ... while the interval bounds are looked up
      table_next_resolve(T, probe, cnt, col);
      u8 tag[4];
      const int nt = tag_next_nodes(cnt, col, sb, P, false, tag);
      if (nt == 0) break;  // dead end
      int child = -1, nChildren = 0;
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (tag[i] != kUnexpected) { child = i; ++nChildren; }
      if (nChildren != 1) break;
      const u64 ck = kmer_next(kmer, (u32)child, right, k);
      if (!border) {
        bool aim = false;
        TALC_ROLLED
        for (u32 a = 0; a < nAims; ++a) aim |= (aims[a].kmer == ck);
        if (aim) break;
      }
      // cycle test against the parent's sequence (plen bases), current word taken from the register
      if (plen > k) {
        bool hit = false, cyc = false;
        // LEFT walks compare in walk order, i.e. against the reversed k-mer, which is maintained incrementally
        const u64 needle = right ? ck : (((rkmer << 2) | (u64)child) & kmask);
        TALC_ROLLED
        for (u32 p = 0; p + k <= plen && !hit; p += stride) {
          const u32 wi0 = right ? p : (plen - k - p);
          const u32 wi = wi0 >> 5, off = 2 * (wi0 & 31);
          const u64 a0 = (wi == cwIdx) ? cw : w[wi];
          u64 hi = a0 << off;
          if (off && (off + 2 * k > 64)) {
            const u64 a1 = (wi + 1 == cwIdx) ? cw : w[wi + 1];
            hi |= a1 >> (64 - off);
          }
          if ((hi >> (64 - 2 * k)) == needle) { hit = true; cyc = p > 0; }
        }
        if (cyc) break;
      }
      // commit the step
      {
        const u32 idx = plen >> 5;
        if (idx != cwIdx) { w[cwIdx] = cw; cwIdx = idx; cw = w[idx]; }
        const u32 sh = 62 - 2 * (plen & 31);
        cw = (cw & ~(3ull << sh)) | ((u64)child << sh);
        w[cwIdx] = cw;
      }
      dsum = dsum + step_dist(count, cnt[child], sb);
      if (!right) rkmer = ((rkmer << 2) | (u64)child) & kmask;  // reverse(b + x[..K-2]) = reverse(x)[1..] + b
      kmer = ck;
      count = cnt[child];
      ++st;
      ++nSteps;
    }
    if (nSteps) {
      w[cwIdx] = cw;
      tr.kmer = kmer;
      tr.count = count;
      tr.dist = dsum;
      cur[0] = tr;
      step = st;
      if (ctr) {
        if (border) ctr->steps_border += nSteps;
        else ctr->steps_inner += nSteps;
        ctr->frontier_sum += nSteps;
        ctr->lookups_walk += 4ull * nSteps;
      }
    }
    return capped;
  }


#if defined(__CUDA_ARCH__)
  static __device__ __noinline__ double sqrt_cold(u32 c) { return sqrt((double)c); }  // counts beyond the table: rare
  // The fast path on the device, for a frontier of 1..7 trails (two or three trails walking side by side
  // through a variant or an isoform bubble is the common multi-trail case: ~30% of all inner steps).
  // Lane l serves trail l/4 and successor base l%4: all successors of all trails are probed side by side, a
  // ballot per group of four lanes picks the branch, the aim k-mers are split over the four lanes of a group,
  // and the cycle test of each trail runs one window per lane.  A step is taken here only if EVERY trail has
  // exactly one admissible successor, reaches no aim and closes no cycle -- then the frontier keeps its size and
  // order (child t of trail t), nothing is scored or pruned (frontier <= MAX_NB_COMPETING_PATHS and <= 7, so
  // `complex` is false and gardening cannot trigger), and the step only appends one base per trail.  Any other
  // kind of step ends the run *before* the step; the general code then takes that step in full.
  __device__ __noinline__ bool fast_walk(u32& step, u32 pathMax, const AnchorRec* aims, u32 nAims, bool border, u32 maxSteps) {
    const u32 nT = nCur;
    if (!walk_eligible(nAims)) return false;
    bool capped = false;
    const u32 lane = threadIdx.x & 31u;
    const u64 myAim = (!border && lane < nAims) ? aims[lane].kmer : ~0ull;  // ~0 is not a k-mer (<= 60 bits)
    const bool act = lane < nT;  // lane t owns trail t: ONE bucket of the successor table answers its whole step
    const u32 k = P.K;
    const bool right = dirRight;
    const CtxView cv = right ? CR : CL;
    const u64 kmask = kmer_mask(k), cmask = kmer_mask(k - 1);
    const u32 stride = (P.cycle_mode == 0) ? k : 1u;
    const Trail tr = cur[act ? lane : 0];
    u64* const w = slot_ptr(tr.slot);
    u64 kmer = tr.kmer;
    u32 count = tr.count;
    double dsum = tr.dist;
    u64 rkmer = 0;  // the last k-mer with its bases in reverse order (LEFT walks compare in walk order)
    TALC_ROLLED
    for (u32 i = 0; i < k; ++i) rkmer |= ((kmer >> (2 * i)) & 3ull) << (2 * (k - 1 - i));
    u32 st = step, nSteps = 0;
    const u32 topShift = 2 * (k - 1);
    u32 untilCheck = border ? (kCheckInterval - 1u - (st % kCheckInterval)) : ~0u;  // steps before scoreEdges is due
#pragma unroll 1
    while (st < pathMax) {
      if (untilCheck == 0) break;  // border: (st + 1) % kCheckInterval == 0, scoreEdges is due after this step
      if (nSteps >= maxSteps) { capped = true; break; }
      const u32 plen = k + st;
      // ---- the four successors of every trail: one sector per trail
      int child = -1;
      u32 childCnt = 0;
      if (act) {
        u32 c4[4], cm;
        ctx_lookup(cv, right ? (kmer & cmask) : (kmer >> 2), c4, cm);
        child = fast_step_child(c4, cm, count, P, tabs);
        const u32 ch = (u32)(child < 0 ? 0 : child);
        childCnt = ch == 0 ? c4[0] : ch == 1 ? c4[1] : ch == 2 ? c4[2] : c4[3];
      }
      if (__ballot_sync(0xffffffffu, act && child < 0)) break;  // dead end or branching somewhere: general step
      const u32 ch = (u32)(child < 0 ? 0 : child);
      const u64 ck = right ? (((kmer << 2) | (u64)ch) & kmask) : ((kmer >> 2) | ((u64)ch << topShift));
      if (!border) {  // aim reached by any trail: the general step records the bridge (one aim k-mer per lane)
        bool aim = false;
#pragma unroll 1
        for (u32 q = 0; q < nT; ++q) aim |= (myAim == __shfl_sync(0xffffffffu, ck, q));
        if (__ballot_sync(0xffffffffu, aim)) break;
      }
      // ---- cycle test of every trail against its own sequence, one window per lane
      if (plen > k) {
        const u64 myNeedle = right ? ck : (((rkmer << 2) | (u64)ch) & kmask);
        bool cyc = false;
        TALC_ROLLED
        for (u32 q = 0; q < nT && !cyc; ++q) {
          const u64 needle = __shfl_sync(0xffffffffu, myNeedle, q);
          const u64* wq = (const u64*)__shfl_sync(0xffffffffu, (unsigned long long)w, q);
          TALC_ROLLED
          for (u32 base = 0; (u64)base * stride + k <= plen; base += 32) {
            const u32 p = (base + lane) * stride;
            bool match = false;
            if (p + k <= plen) match = path_kmer_fwd(wq, right ? p : (plen - k - p), k) == needle;
            const u32 mm = __ballot_sync(0xffffffffu, match);
            if (mm) {  // first occurrence = lowest lane of the first batch that matches
              cyc = ((base + (u32)__ffs((int)mm) - 1) * stride) > 0;
              break;
            }
          }
        }
        if (cyc) break;
      }
      // ---- commit the step: one base per trail
      if (act) {
        path_set(w, plen, ch);
        if (count != childCnt) {  // a zero numerator adds +0.0 (and would take the slow path of the double division)
          const double sq = (count < tabs.n) ? tabs.sq[count] : sqrt_cold(count);
          dsum = dsum + fabs((double)count - (double)childCnt) / sq;
        }
      }
      __syncwarp();
      if (!right) rkmer = ((rkmer << 2) | (u64)ch) & kmask;
      kmer = ck;
      count = childCnt;
      ++st;
      ++nSteps;
      --untilCheck;
    }
    __syncwarp();
    if (nSteps) {
      if (act) {
        cur[lane].kmer = kmer;
        cur[lane].count = count;
        cur[lane].dist = dsum;
      }
      __syncwarp();
      step = st;
      if (ctr) {
        if (border) ctr->steps_border += nSteps;
        else ctr->steps_inner += nSteps;
        ctr->frontier_sum += (u64)nSteps * nT;
        ctr->lookups_walk += 4ull * nSteps * nT;
      }
    }
    return capped;
  }
#else
  inline bool fast_walk(u32& step, u32 pathMax, const AnchorRec* aims, u32 nAims, bool border, u32 maxSteps) {
    return fast_walk_scalar(step, pathMax, aims, nAims, border, maxSteps);
  }
#endif

  // ------------------------------------------------------------------ gardening, Explorer.cpp:773-865
  // kept[] receives indices into nxt (duplicates possible, Q16); returns isComplex
  TALC_HDN bool gardening(u32* kept, u32& nKept) {
    if (ctr) ctr->ev_gardening++;
    const u32 n = nNxt;
    const u32 MAXP = P.max_branches;
    nKept = 0;
    const u32 mk = scratch.mark();
    SortKey* sk = (SortKey*)scratch.alloc((n + 1) * sizeof(SortKey));
    GardenRank* rankings = (GardenRank*)scratch.alloc(n * sizeof(GardenRank));
    GardenRank* newr = (GardenRank*)scratch.alloc((n + 1) * sizeof(GardenRank));
    GardenRank* tmpr = (GardenRank*)scratch.alloc((n + 1) * sizeof(GardenRank));
    if (!sk || !rankings || !newr || !tmpr) return false;
    u32 nNew = 0;
    bool isComplex = false;
    u32 nb = n < MAXP ? n : MAXP;
    TALC_ROLLED
    for (u32 t = 0; t < n; ++t) {
      rankings[t].idx = t; rankings[t].r1 = 0; rankings[t].r2 = 0; rankings[t].sum = 0;
      sk[t].key = -(i64)nxt[t].score;  // sortByScore: descending score
      sk[t].idx = t;
    }
    std_sort_keys(sk, n);
    {
      u32 rk = 0;
      rankings[sk[0].idx].r1 = 0;
      TALC_ROLLED
      for (u32 t = 1; t < n; ++t) {
        if (!(sk[t].key == sk[t - 1].key)) rk++;
        rankings[sk[t].idx].r1 = rk;
      }
    }
    TALC_ROLLED
    for (u32 t = 0; t < n; ++t) {
      sk[t].key = sort_key_of_nonneg_double(nxt[t].dist);  // sortByLikelihood: ascending distance
      sk[t].idx = t;
    }
    std_sort_keys(sk, n);
    {
      u32 rk = 0;
      rankings[sk[0].idx].r2 = 0;
      TALC_ROLLED
      for (u32 t = 1; t < n; ++t) {
        if (!(sk[t].key == sk[t - 1].key)) rk++;
        rankings[sk[t].idx].r2 = rk;
      }
    }
    TALC_ROLLED
    for (u32 t = 0; t < n; ++t) {
      rankings[t].sum = rankings[t].r1 + rankings[t].r2;
      if ((rankings[t].sum == 0) || (n <= MAXP)) newr[nNew++] = rankings[t];
    }
    if (nNew == 0) {
      TALC_ROLLED
      for (u32 t = 0; t < n; ++t) { sk[t].key = (i64)rankings[t].r1; sk[t].idx = t; tmpr[t] = rankings[t]; }
      std_sort_keys(sk, n);  // sortByMaxScore
      TALC_ROLLED
      for (u32 t = 0; t < n; ++t) rankings[t] = tmpr[sk[t].idx];
      u32 s = 0;
      bool ties = false;
      do {
        if ((s <= nb) || ties) newr[nNew++] = rankings[s];
        if (s < n - 1) ties = (rankings[s + 1].r1 == rankings[s].r1);
        ++s;
      } while (((s <= nb) || ties) & (s < n));
      if (nNew > MAXP) {
        const GardenRank atMax = newr[MAXP];
        if (newr[0].r1 != atMax.r1) {
          --nNew;
          ties = true;
          while ((nNew >= MAXP) & ties) {
            ties = (newr[nNew - 1].r1 == newr[nNew - 2].r1);
            ties |= (nNew >= MAXP);
            if (ties) --nNew;
          }
        }
        if ((nNew > MAXP) & (newr[0].r1 == atMax.r1)) {  // Q16
          isComplex = true;
          TALC_ROLLED
          for (u32 t = 0; t < nNew; ++t) { sk[t].key = (i64)newr[t].r2; sk[t].idx = t; tmpr[t] = newr[t]; }
          std_sort_keys(sk, nNew);  // sortByMinDist
          TALC_ROLLED
          for (u32 t = 0; t < nNew; ++t) newr[t] = tmpr[sk[t].idx];
          TALC_ROLLED
          for (u32 t = 0; t < MAXP; ++t) kept[nKept++] = newr[t].idx;
        }
      }
      TALC_ROLLED
      for (u32 t = 0; t < nNew; ++t) kept[nKept++] = newr[t].idx;
    } else {
      TALC_ROLLED
      for (u32 t = 0; t < nNew; ++t) kept[nKept++] = newr[t].idx;
    }
    scratch.release(mk);
    return isComplex;
  }

  // replace cur by nxt[kept[..]]; trails not kept release their slots, duplicates get copies
  TALC_HDN bool adopt_kept(const u32* kept, u32 nKept, u32 plen) {
    if (nKept > maxT) { scratch.overflow = 1; return false; }
    const u32 mk = scratch.mark();
    u8* used = (u8*)scratch.alloc(nNxt ? nNxt : 1);
    if (!used) return false;
    TALC_ROLLED
    for (u32 i = 0; i < nNxt; ++i) used[i] = 0;
    TALC_ROLLED
    for (u32 i = 0; i < nKept; ++i) used[kept[i]] = 1;
    TALC_ROLLED
    for (u32 i = 0; i < nNxt; ++i)
      if (!used[i]) slot_free(nxt[i].slot);
    TALC_ROLLED
    for (u32 i = 0; i < nNxt; ++i) used[i] = 0;
    TALC_ROLLED
    for (u32 i = 0; i < nKept; ++i) {
      Trail t = nxt[kept[i]];
      if (used[kept[i]]) {  // duplicate of an already adopted trail: private copy of the sequence
        const int s = slot_alloc();
        if (s < 0) { scratch.release(mk); return false; }
        slot_copy((u32)s, t.slot, plen);
        t.slot = (u16)s;
      }
      used[kept[i]] = 1;
      cur[i] = t;
    }
    nCur = nKept;
    scratch.release(mk);
    return true;
  }
  TALC_HD void adopt_all() {
    Trail* t = cur; cur = nxt; nxt = t;
    nCur = nNxt;
  }

  // ------------------------------------------------------------------ inner search, Explorer.cpp:868-989
  struct BridgeRec {
    i32 score;       // -editDistance (Trajectory.cpp:241)
    double idscore;  // LCS / max(len)  (:242)
    double md;       // Q22
    u32 leftAnchor, rightAnchor;
    u32 cutLen;      // sequence length after cutAnchors
    u32 fullLen;
    i32 seqSlot;     // index of the retained packed copy, -1 if not retained
    bool ok;
  };

  // fold of findBestBridge (Trajectory.cpp:282-303) over a prefix; also usable incrementally
  TALC_HD static bool fold_better(i32 score, double md, i32 bscore, double bmd) {
    if (score > bscore) return true;
    if (score == bscore && md > bmd) return true;  // Q21: later entry with larger mean distance wins
    return false;
  }

  // One call runs the search until it ends (kStepTrue: weakOut holds the accepted bridge, kStepFalse: none / scratch
  // overflow, see the arenas) or until a long walk is handed over (kStepYield: call again after the walk).
  // fb.pc == 0 starts a new search.
  TALC_HDN u8 search_bridge(Piece& weakOut) {
    const u32 k = K();
    const AnchorRec* anchors = dirRight ? ancL : ancR;
    const u32 nAnch = dirRight ? nAncL : nAncR;
    const AnchorRec* aims = dirRight ? ancR : ancL;
    const u32 nAims = dirRight ? nAncR : nAncL;
    for (;;) {
      switch (fb.pc) {
        case 0: {
          fb.limit = nAnch < kMaxStartAnchors ? nAnch : (u32)kMaxStartAnchors;
          fb.found = false;
          fb.mk0 = scratch.mark();
          fb.s = 0;
          fb.pc = 1;
          break;
        }
        case 1: {  // next start anchor (Explorer.cpp:905: at most 5, until one is accepted)
          if (!(fb.s < fb.limit && !fb.found)) {
            scratch.release(fb.mk0);
            fb.pc = 0;
            return fb.found ? kStepTrue : kStepFalse;
          }
          scratch.release(fb.mk0);
          if (ctr) ctr->gap_attempts++;
          const u32 whichStart = anchors[fb.s].pos;
          u32 gapLen = 0;
          if (dirRight & (whichStart + k < R.start)) gapLen = R.start - (whichStart + k);
          else if (!dirRight & (L.end + k < whichStart)) gapLen = whichStart - (L.end + k);
          fb.whichStart = whichStart;
          fb.gapLen = gapLen;
          fb.pathMax = (u32)(i32)(1.2 * (double)gapLen + (double)(3 * k));
          RefView ref;
          ref.w = rdw;
          ref.lg = rdlg;
          if (dirRight) { ref.start = (i32)whichStart; ref.step = 1; ref.len = R.end + k - whichStart; }
          else { ref.start = (i32)(whichStart + k - 1); ref.step = -1; ref.len = whichStart + k - L.start; }
          fb.ref = ref;
          if (!setup_search(fb.pathMax)) { fb.pc = 0; return kStepFalse; }
          if (!push_root(anchors[fb.s])) { fb.pc = 0; return kStepFalse; }
          // bridges: metadata for all, sequences only for running-best record setters
          // the reference puts no cap on recorded bridges: the caps grow with the arena (second tier: ~50 000 bridges)
          const u32 capShare = (scratch.cap - scratch.top) / 16u;
          u32 maxBridges = capShare / (u32)sizeof(BridgeRec);
          if (maxBridges < 1024u) maxBridges = 1024u;
          u32 maxKeep = capShare / (slotWords * 8u);
          if (maxKeep < 32u) maxKeep = 32u;
          if (maxKeep > maxBridges) maxKeep = maxBridges;
          fb.maxBridges = maxBridges;
          fb.maxKeep = maxKeep;
          fb.br = scratch.alloc(maxBridges * sizeof(BridgeRec));
          fb.brSeq = (u64*)scratch.alloc(maxKeep * slotWords * 8);
          if (!fb.br || !fb.brSeq) { fb.pc = 0; return kStepFalse; }
          fb.nBr = fb.nBrSeq = 0;
          fb.runScore = 0;
          fb.runMd = 0;
          fb.runHave = false;
          fb.step = 0;
          fb.pc = 2;
          break;
        }
        case 2: {  // loop head of Explorer.cpp:940
          if (!((nCur > 0) & (nCur <= kMaxInnerPaths) & (fb.step < fb.pathMax))) { fb.pc = 4; break; }
          const bool capped = fast_walk(fb.step, fb.pathMax, aims, nAims, false, splitWalk ? inlineInner : ~0u);
          fb.pc = 3;
          if (capped && splitWalk) {  // still walking: the walk kernel carries on from cur[] and hands fb.step back in wq
            wq.aims = aims;
            wq.nAims = nAims;
            wq.step = fb.step;
            wq.pathMax = fb.pathMax;
            wq.border = 0;
            return kStepYield;
          }
          break;
        }
        case 3: {
          if (!(fb.step < fb.pathMax)) { fb.pc = 4; break; }
          if (!bridge_general_step(aims, nAims)) { fb.pc = 0; return kStepFalse; }
          fb.pc = 2;
          if (should_pause()) {
            wq.step = fb.step;
            wq.border = 2;
            return kStepYield;
          }
          break;
        }
        default: {  // case 4: the attempt is over
          finish_bridge_attempt(weakOut);
          if (scratch.overflow || keep.overflow) { fb.pc = 0; return kStepFalse; }
          ++fb.s;
          fb.pc = 1;
          break;
        }
      }
    }
  }

  // ---- oneMoreStep, Explorer.cpp:546-612 (one synchronous expansion of the frontier, then pruning if due)
  TALC_STEPFN bool bridge_general_step(const AnchorRec* aims, u32 nAims) {
    const u32 k = K();
    const RefView ref = fb.ref;
    const SeqView refv = view_of(ref);
    BridgeRec* br = (BridgeRec*)fb.br;
    u64* brSeq = fb.brSeq;
    const u32 whichStart = fb.whichStart;
    u32 step = fb.step;
    {
        const u32 plen = k + step;  // every trail of the frontier has this length
        if (ctr) { ctr->steps_inner++; ctr->frontier_sum += nCur; }
        nNxt = 0;
        const bool complex_ = (nCur > P.max_branches);
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
        for (u32 t = 0; t < nCur; ++t) {
          const Trail par = cur[t];
          u32 cnt[4], col[4];
          next_counts(par.kmer, cnt, col);
          if (ctr) ctr->lookups_walk += 4;
          u8 tag[4];
          const StepBounds sb = step_bounds_tab(par.count, P, tabs);
          const int nt = tag_next_nodes(cnt, col, sb, P, complex_, tag);
          u32 nChildren = 0;
          TALC_ROLLED
          for (int i = 0; i < nt; ++i) nChildren += (tag[i] != kUnexpected) ? 1 : 0;
          bool parentSlotTaken = false;
#if defined(__CUDA_ARCH__)
#pragma unroll 1  // the body is large: unrolled four times it floods the instruction cache (see DESIGN.md section 5)
#endif
          for (int i = 0; i < nt; ++i) {
            if (tag[i] == kUnexpected) continue;
            Trail ch;
            ch.kmer = kmer_next(par.kmer, (u32)i, dirRight, k);
            ch.count = cnt[i];
            ch.score = par.score;
            ch.failures = par.failures;
            ch.dist = par.dist + step_dist(par.count, cnt[i], sb);
            ch.pad = 0;
            // sequence: a single child extends the parent's slot in place, siblings copy it
            if (nChildren == 1) {
              ch.slot = par.slot;
              parentSlotTaken = true;
            } else {
              const int sl = slot_alloc();
              if (sl < 0) return false;
              slot_copy((u32)sl, par.slot, plen);
              ch.slot = (u16)sl;
            }
            // cycle test looks at the parent's sequence only, so it may run before the append
            bool aim = false;
            u32 aimPos = 0;
            TALC_ROLLED
            for (u32 a = 0; a < nAims; ++a) {  // Trail.cpp:273-285, first match in sorted aim order
              if (aims[a].kmer == ch.kmer) { aim = true; aimPos = aims[a].pos; break; }
            }
            bool drop = false;
            if (!aim) {
              if (already_got_there(ch.kmer, slot_ptr(par.slot), plen)) {
                if (ctr) ctr->ev_cycle++;
                drop = true;
              }
            }
            path_set(slot_ptr(ch.slot), plen, (u32)i);
            if (aim) {
              // recordBridge (:1097) + scoreSequence + cutAnchors evaluated now; inputs are final
              if (ctr) ctr->ev_bridge++;
              if (fb.nBr >= fb.maxBridges) { scratch.overflow = 1; return false; }
              BridgeRec b;
              const u32 clen = plen + 1;
              b.fullLen = clen;
              b.md = ch.dist / ((double)clen + 0.01);
              b.leftAnchor = dirRight ? whichStart : aimPos;
              b.rightAnchor = dirRight ? aimPos : whichStart;
              const SeqView pv = view_of_path(slot_ptr(ch.slot), clen);
              int lcs = 0;
              b.score = -nw_lcs_fused(refv, ref.len, pv, clen, scratch, &dps, lcs, 3);
              b.idscore = (double)lcs / (double)(ref.len > clen ? ref.len : clen);
              // cutAnchors INNER (Trajectory.cpp:176-197), limit = RIGHT.end
              b.ok = true;
              b.cutLen = 0;
              if (clen >= 2 * k) b.cutLen = clen - 2 * k;
              else if ((clen < 2 * k) & (clen > k)) {
                if (b.rightAnchor + 2 * k - clen <= R.end) b.rightAnchor = b.rightAnchor + 2 * k - clen;
                else b.ok = false;
              } else b.ok = false;
              b.seqSlot = -1;
              if (!fb.runHave || fold_better(b.score, b.md, fb.runScore, fb.runMd)) {
                fb.runHave = true;
                fb.runScore = b.score;
                fb.runMd = b.md;
                if (fb.nBrSeq >= fb.maxKeep) { scratch.overflow = 1; return false; }
                u64* dst = brSeq + (u64)fb.nBrSeq * slotWords;
                const u64* src = slot_ptr(ch.slot);
                TALC_ROLLED
                for (u32 wi = 0; wi < (clen + 31) / 32; ++wi) dst[wi] = src[wi];
                b.seqSlot = (i32)fb.nBrSeq++;
              }
              br[fb.nBr++] = b;
              if (clen > ref.len) drop = true;  // Q10: otherwise the trail keeps exploring
            }
            if (drop) {
              if (ch.slot != par.slot) slot_free(ch.slot);
              else parentSlotTaken = false;
            } else {
              if (nNxt >= maxT) { scratch.overflow = 1; return false; }
              nxt[nNxt++] = ch;
            }
          }
          if (!parentSlotTaken) slot_free(par.slot);
        }
        ++step;
        fb.step = step;
        if ((nNxt > P.max_branches) & (step % kCheckInterval == 0)) {
          // scoreBridges, Explorer.cpp:689-706: reference truncated to K+step+WINDOW (walk order)
          u32 bound = k + step + P.window;
          const u32 rn = (bound >= ref.len) ? ref.len : bound;
          if (P.q11_zero) {
#if defined(__CUDA_ARCH__)
            if (!overlap_score_frontier(refv, rn, k + step, nNxt, [&](u32 j) { return (const u64*)slot_ptr(nxt[j].slot); },
                                        [&](u32 j, int s) { nxt[j].score = s; }, scratch, &dps))
              return false;
#else
            TALC_ROLLED
            for (u32 j = 0; j < nNxt; ++j) {
              const SeqView pv = view_of_path(slot_ptr(nxt[j].slot), k + step);
              nxt[j].score = overlap_score(refv, rn, pv, k + step, scratch, &dps);
            }
#endif
          }
          const u32 mkg = scratch.mark();
          u32* kept = (u32*)scratch.alloc((nNxt + P.max_branches + 1) * 4);
          if (!kept) return false;
          u32 nKept = 0;
          complexRegion |= gardening(kept, nKept);
          if (scratch.overflow) return false;
          if (!adopt_kept(kept, nKept, k + step)) return false;
          scratch.release(mkg);
        } else {
          adopt_all();
        }
        if (scratch.overflow) return false;
    }
    return true;
  }

  // Explorer.cpp:945-982: best recorded bridge of the attempt, acceptance test, corrected weak sequence
  TALC_STEPFN void finish_bridge_attempt(Piece& weakOut) {
    const u32 k = K();
    BridgeRec* br = (BridgeRec*)fb.br;
    const u64* brSeq = fb.brSeq;
    const u32 nBr = fb.nBr;
      if (nBr > 0) {
        // Q9: if cutAnchors rejected some bridges the survivors are the FIRST nOk entries
        u32 nOk = 0;
        TALC_ROLLED
        for (u32 t = 0; t < nBr; ++t) nOk += br[t].ok ? 1 : 0;
        const u32 nUse = nOk;  // == nBr when nothing was rejected
        if (nUse > 0) {
          u32 best = 0;
          TALC_ROLLED
          for (u32 i = 1; i < nUse; ++i)
            if (br[i].score > br[best].score) best = i;
          TALC_ROLLED
          for (u32 i = best + 1; i < nUse; ++i)
            if (br[i].score == br[best].score && br[i].md > br[best].md) best = i;  // sequential update == Q21
          const BridgeRec& B = br[best];
          // a rejected bridge inside the surviving prefix has had its sequence emptied (Trajectory.cpp:208)
          const u32 bestLen = B.ok ? B.cutLen : 0;
          const double diff = (double)weakLen - (double)bestLen;
          if ((diff < weakLen * 0.05 || ((weakLen < 6) & (bestLen < 6))) & (B.idscore >= P.min_inner)) {  // Q13
            L.end = B.leftAnchor;
            R.start = B.rightAnchor;
            // corrected weak sequence = path without its two anchors, in read orientation
            u8* dst = (u8*)keep.alloc(bestLen ? bestLen : 1);
            if (!dst) return;
            if (bestLen > 0) {
              if (B.seqSlot < 0) { scratch.overflow = 1; return; }  // cannot happen: see fold argument
              const u64* w = brSeq + (u64)B.seqSlot * slotWords;
              PathView pv; pv.w = w; pv.len = B.fullLen;
              TALC_ROLLED
              for (u32 i = 0; i < bestLen; ++i) {
                const u32 wi = dirRight ? (k + i) : (B.fullLen - k - 1 - i);
                dst[i] = code_char(pv.code(wi));
              }
            }
            weakOut.off = (u32)(dst - keep.base);
            weakOut.len = (i32)bestLen;
            fb.found = true;
          }
        }
      }
  }

  // ------------------------------------------------------------------ border search
  // Trail::seedAndExtend, Trail.cpp:193-216 (reference string vs this trail)
  TALC_HDN bool trail_seed_extend(Trail& t, u32 tlen, const SeqView& refv, int xdrop) {
    const SeqView pv = view_of_path(slot_ptr(t.slot), tlen);
    const SeedExt e = seed_and_extension(refv, pv, xdrop, dirRight, K(), scratch, wide, &dps);
    bool ok = (e.cand_ext == tlen);
    if (!ok) t.failures++;
    else t.failures = 0;
    t.score = e.score;
    ok = (t.failures <= kMaxBorderFailures);
    ok &= !e.stop;
    return ok;
  }

  // Trajectory.cpp:482-503
  TALC_HDN SeedExt find_stop_position(const SeqView& refArg, const SeqView& candArg, int xdrop) {
    int xdrop1 = xdrop;
    bool goFurther = true;
    SeedExt ext, next;
    next = seed_and_extension(refArg, candArg, xdrop1, dirRight, K(), scratch, wide, &dps);
    do {
      --xdrop1;
      ext = next;
      next = seed_and_extension(refArg, candArg, xdrop1, dirRight, K(), scratch, wide, &dps);  // Q20
      if (next.cand_ext < ext.cand_ext) goFurther = false;
    } while (goFurther & (xdrop1 > 0));
    return ext;
  }

  // Explorer::recordEdge, Explorer.cpp:1103-1118, folded straight into the running best of its list
  TALC_HDN bool record_edge(const Trail& t, u32 tlen, const RefView& ref, u32 whichStart, EdgeBest& bestLong,
                           EdgeBest& bestShort) {
    if (ctr) ctr->ev_edge++;
    const u32 k = K();
    // trim (Trajectory.cpp:89-112): drop failures*6 bases from the walking end
    u32 len = tlen;
    const u32 nbBases = (u32)t.failures * kCheckInterval;
    if (len >= nbBases + k) len -= nbBases;
    const bool shorter = (len <= ref.len);
    const SeqView pv = view_of_path(slot_ptr(t.slot), len);
    const SeqView refv = view_of(ref);
    const int xdrop1 = (int)t.score * (-1);
    SeedExt er;
    u32 pathKeep, refFrom;
    if (!shorter) {  // reshape, Trajectory.cpp:128-133: the path plays the reference role
      er = find_stop_position(pv, refv, xdrop1);
      pathKeep = er.ref_ext;
      refFrom = ref.len;
    } else {
      er = find_stop_position(refv, pv, xdrop1);
      pathKeep = len;
      refFrom = er.ref_ext;
    }
    if (scratch.overflow) return false;
    // computePercentID (Trajectory.cpp:505-528) on the two extensions
    const SeqView& ea = shorter ? refv : pv;   // "refExtension" argument order of getSeedAndExtension
    const SeqView& eb = shorter ? pv : refv;
    const u32 la = er.ref_ext, lb = er.cand_ext;
    double id;
    {
      const int l = (la > 0 && lb > 0) ? lcs_length(ea, la, eb, lb, scratch, &dps) : 0;
      const double longer = (lb <= la) ? (double)la : (double)lb;
      id = (double)l / longer;
    }
    const double score = (double)er.score;
    const u32 newLen = pathKeep + (ref.len - refFrom);
    // cutAnchors HEAD/TAIL (Trajectory.cpp:168-175) never rejects; it only empties short sequences
    EdgeBest& dst = shorter ? bestShort : bestLong;
    const double md = t.dist / ((double)tlen + 0.01);
    bool better;
    if (!dst.have) better = true;
    else if (score > dst.score) better = true;
    else better = (score == dst.score && md > dst.md);
    if (better) {
      dst.have = true;
      dst.score = score;
      dst.idscore = id;
      dst.md = md;
      dst.path_keep = pathKeep;
      dst.ref_from = refFrom;
      dst.anchor_pos = whichStart;
      dst.ref_start = ref.start;
      dst.ref_len = ref.len;
      const u64* src = slot_ptr(t.slot);
      TALC_ROLLED
      for (u32 wi = 0; wi < (pathKeep + 31) / 32; ++wi) dst.seq[wi] = src[wi];
    }
    (void)newLen;
    return true;
  }

  // Explorer::scoreEdges, Explorer.cpp:709-740 (operates on nxt)
  TALC_HDN bool score_edges(int& xdrop, u32 tlen, const RefView& ref, u32 whichStart, EdgeBest& bestLong,
                           EdgeBest& bestShort) {
    if (nNxt == 0) return true;
    const SeqView refv = view_of(ref);
    xdrop += 2;
    int new_xdrop = 0;
    const u32 mk = scratch.mark();
    u8* okf = (u8*)scratch.alloc(nNxt);
    if (!okf) return false;
    u32 nSel = 0;
    TALC_ROLLED
    for (u32 t = 0; t < nNxt; ++t) {
      const bool ok = trail_seed_extend(nxt[t], tlen, refv, xdrop);
      if (scratch.overflow) return false;
      okf[t] = ok ? 1 : 0;
      if (ok) {
        ++nSel;
        const int current = (int)nxt[t].score * (-1);
        if ((new_xdrop > current) || (new_xdrop == 0)) new_xdrop = current;  // Q14
      }
    }
    xdrop = new_xdrop;
    if (nSel == 0) {
      TALC_ROLLED
      for (u32 t = 0; t < nNxt; ++t) {
        if (!record_edge(nxt[t], tlen, ref, whichStart, bestLong, bestShort)) return false;
        slot_free(nxt[t].slot);
      }
      nNxt = 0;
    } else {
      u32 w = 0;
      TALC_ROLLED
      for (u32 t = 0; t < nNxt; ++t) {
        if (okf[t]) nxt[w++] = nxt[t];
        else slot_free(nxt[t].slot);
      }
      nNxt = w;
    }
    scratch.release(mk);
    return true;
  }

  // Explorer::searchEdge, Explorer.cpp:992-1081.  Resumable like search_bridge (fe.pc == 0 starts a new search).
  TALC_HDN u8 search_edge(Piece& weakOut) {
    const u32 k = K();
    const AnchorRec* anchors = dirRight ? ancL : ancR;
    const u32 nAnch = dirRight ? nAncL : nAncR;
    for (;;) {
      switch (fe.pc) {
        case 0: {
          fe.limit = nAnch < kMaxStartAnchors ? nAnch : (u32)kMaxStartAnchors;
          // running bests of m_longPaths / m_shortPaths across all anchors
          u32 maxGap = 0;
          TALC_ROLLED
          for (u32 s = 0; s < fe.limit; ++s) {
            const u32 g = (location == 0) ? anchors[s].pos : (rd.len - (anchors[s].pos + k));
            maxGap = g > maxGap ? g : maxGap;
          }
          const u32 maxPath = (u32)(i32)(1.2 * (double)maxGap + (double)(2 * k));
          const u32 bestWords = (k + maxPath + 2 + 31) / 32 + 1;
          fe.bestLong.have = fe.bestShort.have = false;
          fe.bestLong.seq = (u64*)scratch.alloc(bestWords * 8);
          fe.bestShort.seq = (u64*)scratch.alloc(bestWords * 8);
          if (!fe.bestLong.seq || !fe.bestShort.seq) return kStepFalse;
          fe.mk0 = scratch.mark();
          fe.s = 0;
          fe.pc = 1;
          break;
        }
        case 1: {  // next start anchor: EVERY anchor is searched (Explorer.cpp:1028)
          if (!(fe.s < fe.limit)) {
            fe.pc = 0;
            return finish_edge_search(weakOut) ? kStepTrue : kStepFalse;
          }
          scratch.release(fe.mk0);
          fe.xdrop = (int)((int)kCheckInterval * 0.3 + 1);  // Q15: 2
          const u32 whichStart = anchors[fe.s].pos;
          const u32 gapLen = (location == 0) ? whichStart : (rd.len - (whichStart + k));
          fe.whichStart = whichStart;
          fe.pathMax = (u32)(i32)(1.2 * (double)gapLen + (double)(2 * k));
          RefView ref;
          ref.w = rdw;
          ref.lg = rdlg;
          if (dirRight) { ref.start = (i32)whichStart; ref.step = 1; ref.len = rd.len - whichStart; }
          else { ref.start = (i32)(whichStart + k - 1); ref.step = -1; ref.len = whichStart + k; }
          fe.ref = ref;
          if (!setup_search(fe.pathMax)) { fe.pc = 0; return kStepFalse; }
          if (!push_root(anchors[fe.s])) { fe.pc = 0; return kStepFalse; }
          fe.step = 0;
          fe.pc = 2;
          break;
        }
        case 2: {  // loop head of Explorer.cpp:1055
          if (!((nCur > 0) & (nCur <= kMaxInnerPaths) & (fe.step < fe.pathMax))) { ++fe.s; fe.pc = 1; break; }
          const bool capped = fast_walk(fe.step, fe.pathMax, nullptr, 0, true, splitWalk ? inlineBorder : ~0u);
          fe.pc = 3;
          if (capped && splitWalk) {
            wq.aims = nullptr;
            wq.nAims = 0;
            wq.step = fe.step;
            wq.pathMax = fe.pathMax;
            wq.border = 1;
            return kStepYield;
          }
          break;
        }
        default: {  // case 3
          if (!(fe.step < fe.pathMax)) { ++fe.s; fe.pc = 1; break; }
          if (!edge_general_step()) { fe.pc = 0; return kStepFalse; }
          fe.pc = 2;
          if (should_pause()) {
            wq.step = fe.step;
            wq.border = 2;
            return kStepYield;
          }
          break;
        }
      }
    }
  }

  // ---- oneMoreStepInTheDark, Explorer.cpp:615-687
  TALC_STEPFN bool edge_general_step() {
    const u32 k = K();
    const RefView ref = fe.ref;
    const SeqView refv = view_of(ref);
    const u32 whichStart = fe.whichStart, pathMax = fe.pathMax;
    EdgeBest& bestLong = fe.bestLong;
    EdgeBest& bestShort = fe.bestShort;
    int xdrop = fe.xdrop;
    u32 step = fe.step;
    {
        const u32 plen = k + step;
        if (ctr) { ctr->steps_border++; ctr->frontier_sum += nCur; }
        nNxt = 0;
        const bool complex_ = (nCur > 7);
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
        for (u32 t = 0; t < nCur; ++t) {
          Trail par = cur[t];
          u32 cnt[4], col[4];
          next_counts(par.kmer, cnt, col);
          if (ctr) ctr->lookups_walk += 4;
          u8 tag[4];
          const StepBounds sb = step_bounds_tab(par.count, P, tabs);
          const int nt = tag_next_nodes(cnt, col, sb, P, complex_, tag);
          u32 nChildren = 0;
          TALC_ROLLED
          for (int i = 0; i < nt; ++i) nChildren += (tag[i] != kUnexpected) ? 1 : 0;
          bool parentSlotTaken = false;
#if defined(__CUDA_ARCH__)
#pragma unroll 1  // the body is large: unrolled four times it floods the instruction cache (see DESIGN.md section 5)
#endif
          for (int i = 0; i < nt; ++i) {
            if (tag[i] == kUnexpected) continue;
            Trail ch;
            ch.kmer = kmer_next(par.kmer, (u32)i, dirRight, k);
            ch.count = cnt[i];
            ch.score = par.score;
            ch.failures = par.failures;
            ch.dist = par.dist + step_dist(par.count, cnt[i], sb);
            ch.pad = 0;
            if (nChildren == 1) {
              ch.slot = par.slot;
              parentSlotTaken = true;
            } else {
              const int sl = slot_alloc();
              if (sl < 0) return false;
              slot_copy((u32)sl, par.slot, plen);
              ch.slot = (u16)sl;
            }
            const bool cycle = already_got_there(ch.kmer, slot_ptr(par.slot), plen);
            path_set(slot_ptr(ch.slot), plen, (u32)i);
            if (cycle || (step + 1 > pathMax)) {
              if (cycle && ctr) ctr->ev_cycle++;
              trail_seed_extend(ch, plen + 1, refv, xdrop);
              if (scratch.overflow) return false;
              if (!record_edge(ch, plen + 1, ref, whichStart, bestLong, bestShort)) return false;
              if (ch.slot != par.slot) slot_free(ch.slot);
              else parentSlotTaken = false;
            } else {
              if (nNxt >= maxT) { scratch.overflow = 1; return false; }
              nxt[nNxt++] = ch;
            }
          }
          if (nChildren == 0) {  // dead end: the trail itself becomes a candidate
            trail_seed_extend(par, plen, refv, xdrop);
            if (scratch.overflow) return false;
            if (!record_edge(par, plen, ref, whichStart, bestLong, bestShort)) return false;
          }
          if (!parentSlotTaken) slot_free(par.slot);
        }
        ++step;
        fe.step = step;
        if ((step % kCheckInterval == 0) || (nNxt >= kMaxBorderPaths)) {
          if (!score_edges(xdrop, k + step, ref, whichStart, bestLong, bestShort)) return false;
          fe.xdrop = xdrop;
          if (nNxt > 5) {
            const u32 mkg = scratch.mark();
            u32* kept = (u32*)scratch.alloc((nNxt + P.max_branches + 1) * 4);
            if (!kept) return false;
            u32 nKept = 0;
            complexRegion |= gardening(kept, nKept);
            if (scratch.overflow) return false;
            if (!adopt_kept(kept, nKept, k + step)) return false;
            scratch.release(mkg);
          } else
            adopt_all();
        } else
          adopt_all();
        if (scratch.overflow) return false;
    }
    return true;
  }

  // sortOutBestBorder (Explorer.cpp:310-329) + the acceptance test of :1063-1076
  TALC_STEPFN bool finish_edge_search(Piece& weakOut) {
    const u32 k = K();
    const EdgeBest& bestLong = fe.bestLong;
    const EdgeBest& bestShort = fe.bestShort;
    bool found = false;
    if (bestLong.have || bestShort.have) {
      const EdgeBest& W = bestLong.have ? bestLong : bestShort;  // sortOutBestBorder, :310-329
      const u32 newLen = W.path_keep + (W.ref_len - W.ref_from);
      const u32 wlen = (newLen > k) ? (newLen - k) : 0;  // cutAnchors HEAD/TAIL
      const double diff = (double)weakLen - (double)wlen;
      double minScore;
      if ((weakLen >= 300) || complexRegion) minScore = (0.75 > P.min_border) ? 0.75 : P.min_border;
      else minScore = P.min_border;
      if ((diff < weakLen * 0.05 || ((weakLen < 6) & (wlen < 6))) & (W.idscore >= minScore)) {
        found = true;
        if (location == 2) L.end = W.anchor_pos;
        else R.start = W.anchor_pos;
        u8* dst = (u8*)keep.alloc(wlen ? wlen : 1);
        if (!dst) return false;
        // walk-order sequence: trail prefix, then raw border; minus the first K (the anchor);
        // TAIL is already in read orientation, HEAD is reversed
        PathView pv; pv.w = W.seq; pv.len = W.path_keep;
        TALC_ROLLED
        for (u32 i = 0; i < wlen; ++i) {
          const u32 wi = k + i;  // walk index
          u8 ch;
          if (wi < W.path_keep) ch = code_char(pv.code(wi));
          else {
            const u32 ri = W.ref_from + (wi - W.path_keep);
            const i32 step = dirRight ? 1 : -1;
            ch = code_char(base_code(rd.s[W.ref_start + (i32)ri * step]));
          }
          dst[dirRight ? i : (wlen - 1 - i)] = ch;
        }
        weakOut.off = (u32)(dst - keep.base);
        weakOut.len = (i32)wlen;
      }
    }
    return found;
  }

  // ------------------------------------------------------------------ straight-line drivers (monolithic kernel, host)
  // The same searches without the suspend points: plain loops around the same step functions.  The monolithic kernel
  // (and the host emulation's default path) run these; the state machines above exist for reads that are suspended.
  TALC_HDN bool search_bridge_mono(Piece& weakOut) {
    const u32 k = K();
    const AnchorRec* anchors = dirRight ? ancL : ancR;
    const u32 nAnch = dirRight ? nAncL : nAncR;
    const AnchorRec* aims = dirRight ? ancR : ancL;
    const u32 nAims = dirRight ? nAncR : nAncL;
    const u32 limit = nAnch < kMaxStartAnchors ? nAnch : (u32)kMaxStartAnchors;
    fb.found = false;
    const u32 mk0 = scratch.mark();
#if defined(__CUDA_ARCH__)
#pragma unroll 1  // at most 5 start anchors: unrolled, the whole search would be in the binary five times
#endif
    for (u32 s = 0; s < limit && !fb.found; ++s) {
      scratch.release(mk0);
      if (ctr) ctr->gap_attempts++;
      const u32 whichStart = anchors[s].pos;
      u32 gapLen = 0;
      if (dirRight & (whichStart + k < R.start)) gapLen = R.start - (whichStart + k);
      else if (!dirRight & (L.end + k < whichStart)) gapLen = whichStart - (L.end + k);
      const u32 pathMax = (u32)(i32)(1.2 * (double)gapLen + (double)(3 * k));
      fb.whichStart = whichStart;
      fb.gapLen = gapLen;
      fb.pathMax = pathMax;
      RefView ref;
      ref.w = rdw;
      ref.lg = rdlg;
      if (dirRight) { ref.start = (i32)whichStart; ref.step = 1; ref.len = R.end + k - whichStart; }
      else { ref.start = (i32)(whichStart + k - 1); ref.step = -1; ref.len = whichStart + k - L.start; }
      fb.ref = ref;
      if (!setup_search(pathMax)) return false;
      if (!push_root(anchors[s])) return false;
      const u32 capShare = (scratch.cap - scratch.top) / 16u;
      u32 maxBridges = capShare / (u32)sizeof(BridgeRec);
      if (maxBridges < 1024u) maxBridges = 1024u;
      u32 maxKeep = capShare / (slotWords * 8u);
      if (maxKeep < 32u) maxKeep = 32u;
      if (maxKeep > maxBridges) maxKeep = maxBridges;
      fb.maxBridges = maxBridges;
      fb.maxKeep = maxKeep;
      fb.br = scratch.alloc(maxBridges * sizeof(BridgeRec));
      fb.brSeq = (u64*)scratch.alloc(maxKeep * slotWords * 8);
      if (!fb.br || !fb.brSeq) return false;
      fb.nBr = fb.nBrSeq = 0;
      fb.runScore = 0;
      fb.runMd = 0;
      fb.runHave = false;
      fb.step = 0;
      while ((nCur > 0) & (nCur <= kMaxInnerPaths) & (fb.step < pathMax)) {
        fast_walk(fb.step, pathMax, aims, nAims, false, ~0u);
        if (!(fb.step < pathMax)) break;
        if (!bridge_general_step(aims, nAims)) return false;
      }
      finish_bridge_attempt(weakOut);
      if (scratch.overflow || keep.overflow) return false;
    }
    scratch.release(mk0);
    return fb.found;
  }

  TALC_HDN bool search_edge_mono(Piece& weakOut) {
    const u32 k = K();
    const AnchorRec* anchors = dirRight ? ancL : ancR;
    const u32 nAnch = dirRight ? nAncL : nAncR;
    const u32 limit = nAnch < kMaxStartAnchors ? nAnch : (u32)kMaxStartAnchors;
    u32 maxGap = 0;
    TALC_ROLLED
    for (u32 s = 0; s < limit; ++s) {
      const u32 g = (location == 0) ? anchors[s].pos : (rd.len - (anchors[s].pos + k));
      maxGap = g > maxGap ? g : maxGap;
    }
    const u32 maxPath = (u32)(i32)(1.2 * (double)maxGap + (double)(2 * k));
    const u32 bestWords = (k + maxPath + 2 + 31) / 32 + 1;
    fe.bestLong.have = fe.bestShort.have = false;
    fe.bestLong.seq = (u64*)scratch.alloc(bestWords * 8);
    fe.bestShort.seq = (u64*)scratch.alloc(bestWords * 8);
    if (!fe.bestLong.seq || !fe.bestShort.seq) return false;
    const u32 mk0 = scratch.mark();
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (u32 s = 0; s < limit; ++s) {
      scratch.release(mk0);
      fe.xdrop = (int)((int)kCheckInterval * 0.3 + 1);  // Q15: 2
      const u32 whichStart = anchors[s].pos;
      const u32 gapLen = (location == 0) ? whichStart : (rd.len - (whichStart + k));
      const u32 pathMax = (u32)(i32)(1.2 * (double)gapLen + (double)(2 * k));
      fe.whichStart = whichStart;
      fe.pathMax = pathMax;
      RefView ref;
      ref.w = rdw;
      ref.lg = rdlg;
      if (dirRight) { ref.start = (i32)whichStart; ref.step = 1; ref.len = rd.len - whichStart; }
      else { ref.start = (i32)(whichStart + k - 1); ref.step = -1; ref.len = whichStart + k; }
      fe.ref = ref;
      if (!setup_search(pathMax)) return false;
      if (!push_root(anchors[s])) return false;
      fe.step = 0;
      while ((nCur > 0) & (nCur <= kMaxInnerPaths) & (fe.step < pathMax)) {
        fast_walk(fe.step, pathMax, nullptr, 0, true, ~0u);
        if (!(fe.step < pathMax)) break;
        if (!edge_general_step()) return false;
      }
    }
    return finish_edge_search(weakOut);
  }

  // Read::correct2 (Read.cpp:336-386) as plain loops
  TALC_HDN u8 run_mono(const ReadJob& job) {
    job_ = job;
    splitWalk = 0;
    pauseBudget = 0;
    const u32 k = K();
    {
      const u8 st = prepare_read();
      if (st != kReadOk) return st;
    }
    TALC_ROLLED
    for (u32 reg = 0; reg + 1 < nregs; ++reg) {
      if (ctr) ctr->gaps++;
      bool success = false;
      TALC_ROLLED
      for (int attempt = 0; attempt < 2 && !success; ++attempt) {
        scratch.release(0);  // initializeINNER (Explorer.cpp:228-243)
        location = 1;
        dirRight = (attempt == 0);
        L = regs[reg];
        R = regs[reg + 1];
        weakLen = R.start - (L.end + k);
        if (!build_anchors(true) || !build_anchors(false)) return kReadOverflow;
        Piece w;
        success = search_bridge_mono(w);
        if (scratch.overflow || keep.overflow) return kReadOverflow;
        if (success) gapPiece[reg] = w;
      }
      if (success && ctr) ctr->gaps_bridged++;
      regs[reg] = L;  // updateINNER (Read.cpp:294-303)
      regs[reg + 1] = R;
    }
    if (headPresent && headRaw <= kBorderMaxLen) {
      if (ctr) ctr->borders++;
      scratch.release(0);
      location = 0;
      dirRight = false;
      L.start = L.end = 0;
      R = regs[0];
      weakLen = R.start;
      nAncL = 0;
      if (!build_anchors(false)) return kReadOverflow;
      Piece w;
      const bool ok = search_edge_mono(w);
      if (scratch.overflow || keep.overflow) return kReadOverflow;
      if (ok) {
        if (ctr) ctr->borders_corrected++;
        regs[0] = R;  // updateHEAD (Read.cpp:305-311)
        headPiece = w;
      }
    }
    if (tailPresent && tailRaw <= kBorderMaxLen) {
      if (ctr) ctr->borders++;
      scratch.release(0);
      location = 2;
      dirRight = true;
      R.start = R.end = 0;
      L = regs[nregs - 1];
      weakLen = rd.len - (L.end + k);
      nAncR = 0;
      if (!build_anchors(true)) return kReadOverflow;
      Piece w;
      const bool ok = search_edge_mono(w);
      if (scratch.overflow || keep.overflow) return kReadOverflow;
      if (ok) {
        if (ctr) ctr->borders_corrected++;
        regs[nregs - 1] = L;  // updateTAIL (Read.cpp:313-318)
        tailPiece = w;
      }
    }
    return kReadOk;
  }

  // ------------------------------------------------------------------ per-read driver (main.cpp:258-296)
  // start() sets the read up and runs it; resume() continues after a yield (the walk kernel has advanced cur[] and
  // wq.step).  Both return a ReadStatus, or kReadYield when the read waits for the walk kernel.  On kReadOk the
  // pieces describe the corrected read.
  TALC_HDN u8 start(const ReadJob& job) {
    job_ = job;
    pauseCount = 0;
    mark_resumed();
    fr.pc = 0;
    fb.pc = 0;
    fe.pc = 0;
    return resume();
  }
  TALC_HDN u8 run(const ReadJob& job) {  // never yields: the walk is taken inline (host emulation, tuning builds)
    splitWalk = 0;
    pauseBudget = 0;
    return start(job);
  }
  // what the walk kernel (or its host stand-in) reports back
  TALC_HD void walk_done(u32 step) {
    if (location == 1) fb.step = step;
    else fe.step = step;
  }
  TALC_HDN u8 resume() {
    const u32 k = K();
    for (;;) {
      switch (fr.pc) {
        case 0: {
          const u8 st = prepare_read();
          if (st != kReadOk) return st;
          fr.reg = 0;
          fr.pc = 1;
          break;
        }
        case 1: {  // Read::correct2 (Read.cpp:336-386): the gaps in order
          if (!(fr.reg + 1 < nregs)) { fr.pc = 5; break; }
          if (ctr) ctr->gaps++;
          fr.success = false;
          fr.attempt = 0;
          fr.pc = 2;
          break;
        }
        case 2: {  // RIGHT-ward attempt, then LEFT-ward on failure (Read.cpp:350-355)
          if (!(fr.attempt < 2 && !fr.success)) { fr.pc = 4; break; }
          // initializeINNER (Explorer.cpp:228-243)
          scratch.release(0);
          location = 1;
          dirRight = (fr.attempt == 0);
          L = regs[fr.reg];
          R = regs[fr.reg + 1];
          weakLen = R.start - (L.end + k);
          if (!build_anchors(true) || !build_anchors(false)) return kReadOverflow;
          fb.pc = 0;
          fr.pc = 3;
          break;
        }
        case 3: {
          Piece w;
          const u8 r = search_bridge(w);
          if (r == kStepYield) return kReadYield;
          fr.success = (r == kStepTrue);
          if (scratch.overflow || keep.overflow) return kReadOverflow;
          if (fr.success) gapPiece[fr.reg] = w;
          ++fr.attempt;
          fr.pc = 2;
          break;
        }
        case 4: {
          if (fr.success && ctr) ctr->gaps_bridged++;
          regs[fr.reg] = L;  // updateINNER (Read.cpp:294-303)
          regs[fr.reg + 1] = R;
          ++fr.reg;
          fr.pc = 1;
          break;
        }
        case 5: {  // HEAD (Read.cpp:361-367); region 0's start is untouched by the inner gaps
          const u32 headLen = headRaw;
          if (!(headPresent && headLen <= kBorderMaxLen)) { fr.pc = 7; break; }
          if (ctr) ctr->borders++;
          scratch.release(0);
          location = 0;
          dirRight = false;
          L.start = L.end = 0;
          R = regs[0];
          weakLen = R.start;
          nAncL = 0;
          if (!build_anchors(false)) return kReadOverflow;
          fe.pc = 0;
          fr.pc = 6;
          break;
        }
        case 6: {
          Piece w;
          const u8 r = search_edge(w);
          if (r == kStepYield) return kReadYield;
          if (scratch.overflow || keep.overflow) return kReadOverflow;
          if (r == kStepTrue) {
            if (ctr) ctr->borders_corrected++;
            regs[0] = R;  // updateHEAD (Read.cpp:305-311)
            headPiece = w;
          }
          fr.pc = 7;
          break;
        }
        case 7: {  // TAIL (Read.cpp:368-374)
          const u32 tailLen = tailRaw;
          if (!(tailPresent && tailLen <= kBorderMaxLen)) return kReadOk;
          if (ctr) ctr->borders++;
          scratch.release(0);
          location = 2;
          dirRight = true;
          R.start = R.end = 0;
          L = regs[nregs - 1];
          weakLen = rd.len - (L.end + k);
          nAncR = 0;
          if (!build_anchors(true)) return kReadOverflow;
          fe.pc = 0;
          fr.pc = 8;
          break;
        }
        default: {  // case 8
          Piece w;
          const u8 r = search_edge(w);
          if (r == kStepYield) return kReadYield;
          if (scratch.overflow || keep.overflow) return kReadOverflow;
          if (r == kStepTrue) {
            if (ctr) ctr->borders_corrected++;
            regs[nregs - 1] = L;  // updateTAIL (Read.cpp:313-318)
            tailPiece = w;
          }
          return kReadOk;
        }
      }
    }
  }

  // everything of main.cpp:258-296 that precedes correct2: packing, the reCoverage gate, defineStructure2
  TALC_HDN u8 prepare_read() {
    const ReadJob& job = job_;
    rd = job.rd;
    cov = job.cov;
    wide = job.wide;
    dps.cells_nw = dps.cells_lcs = dps.cells_ovl = dps.cells_xdrop = 0;
    const u32 k = K();
    if (!((i32)rd.len > (i32)k)) return kReadShort;
    C = rd.len - k + 1;
    if (ctr) ctr->lookups_seg += C;
    const u32 keepBytes = job.arena_bytes / 4;
    keep.init(job.arena, keepBytes & ~7u);
    scratch.init(job.arena + (keepBytes & ~7u), job.arena_bytes - (keepBytes & ~7u));
    {  // packed copy of the read for the scoring loops: 2 bits per base, 4 when the read holds an N
      u64* pw = (u64*)keep.alloc(packed_read_alloc(rd.len) * 8);
      if (!pw) return kReadOverflow;
      bool hasN = false;
      TALC_ROLLED
      for (u32 i = lane_id(); i < rd.len; i += lane_count()) hasN |= rd.code(i) > 3;
      hasN = warp_any(hasN);
      const u32 nw = packed_read_words(rd.len, hasN);
      TALC_ROLLED
      for (u32 wi = lane_id(); wi < nw; wi += lane_count()) pw[wi] = packed_read_word(rd, wi, hasN);
      warp_sync();
      rdw = pw;
      rdlg = hasN ? 4u : 5u;
    }
    // Read::reCoverage gate (Read.cpp:190, Q1: strictly greater)
    u32 nbIn = 0;
    TALC_ROLLED
    for (u32 i = lane_id(); i < C; i += lane_count()) nbIn += (cov[i] > P.min_count) ? 1 : 0;
    nbIn = warp_sum(nbIn);
    if (nbIn == 0) return kReadNoSolid;
    // Read::defineStructure2 (Read.cpp:260-276)
    bool checok = find_in_regions();
    if (keep.overflow) return kReadOverflow;
    noise = seq_error_threshold();
    analyze_in_regions(noise);
    if (keep.overflow) return kReadOverflow;
    if (nregs > 0) checok &= initial_structure();
    if (!checok) return kReadNoStructure;
    headRaw = headPresent ? regs[0].start : 0;
    tailRaw = tailPresent ? rd.len - (regs[nregs - 1].end + k) : 0;
    gapPiece = (Piece*)keep.alloc((nregs ? nregs : 1) * sizeof(Piece));
    if (!gapPiece) return kReadOverflow;
    TALC_ROLLED
    for (u32 i = 0; i + 1 < nregs; ++i) gapPiece[i].len = -1;
    headPiece.len = tailPiece.len = -1;
    complexRegion = false;
    return kReadOk;
  }

  // length of the corrected read (Read::updateCorrSeq, Read.cpp:320-326)
  TALC_HDN u32 corrected_length() const {
    const u32 k = P.K;
    u32 n = 0;
    n += (headPiece.len >= 0) ? (u32)headPiece.len : (headPresent ? headRaw : 0);
    TALC_ROLLED
    for (u32 i = 0; i < nregs; ++i) {
      n += regs[i].end + k - regs[i].start;
      if (i + 1 < nregs) n += (gapPiece[i].len >= 0) ? (u32)gapPiece[i].len : gapRawLen(i);
    }
    n += (tailPiece.len >= 0) ? (u32)tailPiece.len : (tailPresent ? tailRaw : 0);
    return n;
  }
  u32 headRaw, tailRaw;  // lengths of the raw head / tail as first defined
  TALC_HD u32 gapRawLen(u32 i) const {
    const u32 a = regs[i].end + P.K, b = regs[i + 1].start;
    return b > a ? b - a : 0;
  }
  // write the corrected read as upper-case ASCII; the `nl` cooperating lanes each write every nl-th byte
  TALC_HDN void emit(u8* out, u32 lane, u32 nl) const {
    const u32 k = P.K;
    u32 o = 0;
    if (headPiece.len >= 0) {
      TALC_ROLLED
      for (u32 i = lane; i < (u32)headPiece.len; i += nl) out[o + i] = keep.base[headPiece.off + i];
      o += (u32)headPiece.len;
    } else if (headPresent) {
      TALC_ROLLED
      for (u32 i = lane; i < headRaw; i += nl) out[o + i] = code_char(rd.code(i));
      o += headRaw;
    }
    TALC_ROLLED
    for (u32 r = 0; r < nregs; ++r) {
      const u32 a = regs[r].start, n = regs[r].end + k - regs[r].start;
      TALC_ROLLED
      for (u32 i = lane; i < n; i += nl) out[o + i] = code_char(rd.code(a + i));
      o += n;
      if (r + 1 < nregs) {
        if (gapPiece[r].len >= 0) {
          TALC_ROLLED
          for (u32 i = lane; i < (u32)gapPiece[r].len; i += nl) out[o + i] = keep.base[gapPiece[r].off + i];
          o += (u32)gapPiece[r].len;
        } else {
          const u32 g0 = regs[r].end + k, gn = gapRawLen(r);
          TALC_ROLLED
          for (u32 i = lane; i < gn; i += nl) out[o + i] = code_char(rd.code(g0 + i));
          o += gn;
        }
      }
    }
    if (tailPiece.len >= 0) {
      TALC_ROLLED
      for (u32 i = lane; i < (u32)tailPiece.len; i += nl) out[o + i] = keep.base[tailPiece.off + i];
    } else if (tailPresent) {
      TALC_ROLLED
      for (u32 i = lane; i < tailRaw; i += nl) out[o + i] = code_char(rd.code(rd.len - tailRaw + i));
    }
  }
};

}  // namespace talc
