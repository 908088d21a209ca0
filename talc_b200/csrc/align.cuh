// align.cuh -- integer alignment scores used by path scoring (SURVEY A.6, rows a15/a17/a21/a22).
//
// The reference only ever reads the *score* of its SeqAn alignments (never the traceback), so:
//   NW(0,-1,-1)  Trajectory.cpp:413, Trail.cpp:422   -> Myers/Hyyro bit-parallel edit distance
//   SW(1,0,0)    Trajectory.cpp:368,525              -> bit-parallel LCS length
//   (4,-3,-2) with free leading gaps  Trail.cpp:166-172 -> two-row integer DP (rare: pruning only)
//   extendSeed(.., GappedXDrop) Trail.cpp:373,391    -> the anti-diagonal X-drop, restated exactly,
//                                                       because its *end position* is algorithm-defined
// All sequences are addressed in walk order (see defs.cuh); a LEFT-ward search is the RIGHT-ward
// algorithm on reversed strings (global/LCS scores are reversal-invariant, EXTEND_LEFT consumes the
// prefixes back to front, and AlignConfig<false,false,true,true> on reversed strings is
// AlignConfig<true,true,false,false>).
// Host form (tests/hostemu): one thread runs one alignment, 64 DP rows per machine word, rows > 64 in stripes
// with the horizontal deltas of the stripe boundary parked in the scratch arena.  Device forms: the warp that
// owns the read runs one alignment with the blocks / columns / diagonals spread over its lanes.
#pragma once
#include "defs.cuh"

namespace talc {

// a slice of the packed read in walk order, or a packed trail: element i is base (start + i*step) of w,
// 2 bits per base (lg = 5) or 4 bits per base (lg = 4, reads that hold an N)
struct SeqView {
  const u64* w;
  i32 start;
  i32 step;
  u32 len;
  u32 lg;
  TALC_HD u32 code(u32 i) const { return packed_code(w, (u32)(start + (i32)i * step), lg); }
};
TALC_HD SeqView view_of(const RefView& r) { SeqView v; v.w = r.w; v.start = r.start; v.step = r.step; v.len = r.len; v.lg = r.lg; return v; }
TALC_HD SeqView view_of(const PathView& p) { SeqView v; v.w = p.w; v.start = 0; v.step = 1; v.len = p.len; v.lg = 5; return v; }
TALC_HD SeqView view_of_path(const u64* w, u32 len) { SeqView v; v.w = w; v.start = 0; v.step = 1; v.len = len; v.lg = 5; return v; }
// packs ASCII into the 4-bit layout (test entry points): dst needs (n + 15) / 16 + 1 words
TALC_HD SeqView pack_ascii4(const u8* s, u32 n, u64* dst) {
  const u32 nw = (n + 15) / 16 + 1;
  for (u32 i = 0; i < nw; ++i) dst[i] = 0;
  for (u32 i = 0; i < n; ++i) dst[i >> 4] |= (u64)base_code(s[i]) << (60 - 4 * (i & 15));
  SeqView v; v.w = dst; v.start = 0; v.step = 1; v.len = n; v.lg = 4;
  return v;
}

struct DpStats {  // algorithmic DP cell updates (SURVEY 8d "integer work")
  u64 cells_nw, cells_lcs, cells_ovl, cells_xdrop;
};

// ---- match masks from 2-bit packed sequences without a per-row loop
// even-position bits of x (0, 2, .., 62) gathered into the low 32 bits
TALC_HD u32 compress_even(u64 x) {
  x &= 0x5555555555555555ull;
  x = (x | (x >> 1)) & 0x3333333333333333ull;
  x = (x | (x >> 2)) & 0x0f0f0f0f0f0f0f0full;
  x = (x | (x >> 4)) & 0x00ff00ff00ff00ffull;
  x = (x | (x >> 8)) & 0x0000ffff0000ffffull;
  x = (x | (x >> 16));
  return (u32)x;
}
TALC_HD u64 bit_reverse64(u64 x) {
#if defined(__CUDA_ARCH__)
  return __brevll(x);
#else
  x = ((x >> 1) & 0x5555555555555555ull) | ((x & 0x5555555555555555ull) << 1);
  x = ((x >> 2) & 0x3333333333333333ull) | ((x & 0x3333333333333333ull) << 2);
  x = ((x >> 4) & 0x0f0f0f0f0f0f0f0full) | ((x & 0x0f0f0f0f0f0f0f0full) << 4);
  return __builtin_bswap64(x);
#endif
}
// 32 packed bases starting at base index i, first base most significant; words beyond lastWord are not touched
TALC_HD u64 packed_chunk32(const u64* w, u32 i, u32 lastWord) {
  const u32 wi = i >> 5, off = 2 * (i & 31);
  if (wi > lastWord) return 0;
  u64 v = w[wi] << off;
  if (off && wi + 1 <= lastWord) v |= w[wi + 1] >> (64 - off);
  return v;
}

// match masks of pattern rows [64*block, 64*block+64) for the five symbols (N matches N)
TALC_HDN void build_peq(const SeqView& pat, u32 pn, u32 block, u64 peq[5]) {
  peq[0] = peq[1] = peq[2] = peq[3] = peq[4] = 0;
  const u32 r0 = block * 64;
  const u32 r1 = (pn - r0 < 64u) ? pn : r0 + 64;
  if (pat.lg == 5) {
    // the n rows are n consecutive packed bases, ascending (step +1) or descending (step -1): split the low and
    // the high bit of every base into two n-bit masks, then the four symbols are the four AND combinations
    const u32 n = r1 - r0;
    const u32 first = (u32)(pat.start + (i32)r0 * pat.step), last = (u32)(pat.start + (i32)(r1 - 1) * pat.step);
    const u32 lowIdx = first < last ? first : last, highIdx = first < last ? last : first;
    const u32 lastWord = highIdx >> 5;
    const u64 c0 = packed_chunk32(pat.w, lowIdx, lastWord);
    const u64 c1 = (n > 32) ? packed_chunk32(pat.w, lowIdx + 32, lastWord) : 0ull;
    // bit 63-j of lo/hi <-> base lowIdx + j
    u64 lo = ((u64)compress_even(c0) << 32) | (u64)compress_even(c1);
    u64 hi = ((u64)compress_even(c0 >> 1) << 32) | (u64)compress_even(c1 >> 1);
    if (pat.step > 0) {  // row r0+j <-> base lowIdx+j
      lo = bit_reverse64(lo);
      hi = bit_reverse64(hi);
    } else {             // row r0+t <-> base lowIdx + (n-1-t)
      lo >>= (64 - n);
      hi >>= (64 - n);
    }
    const u64 rowmask = (n == 64) ? ~0ull : ((1ull << n) - 1ull);
    peq[0] = ~hi & ~lo & rowmask;
    peq[1] = ~hi & lo & rowmask;
    peq[2] = hi & ~lo & rowmask;
    peq[3] = hi & lo & rowmask;
    return;
  }
  for (u32 r = r0; r < r1; ++r) peq[pat.code(r)] |= 1ull << (r - r0);
}

// unit-cost edit distance between a[0..an) and b[0..bn) (either may be empty)
TALC_HDN int nw_distance_scalar(const SeqView& a, u32 an, const SeqView& b, u32 bn, Arena& ar, DpStats* st) {
  // pattern (rows, bit-parallel) = the shorter one, text (columns) = the longer one
  const bool a_is_pat = an <= bn;
  const SeqView pat = a_is_pat ? a : b;
  const SeqView txt = a_is_pat ? b : a;
  const u32 pn = a_is_pat ? an : bn;
  const u32 tn = a_is_pat ? bn : an;
  if (pn == 0) return (int)tn;  // no block: the text is inserted whole
  if (st) st->cells_nw += (u64)an * bn;
  const u32 nblocks = (pn + 63) / 64;
  const u32 mk = ar.mark();
  signed char* h = nullptr;
  if (nblocks > 1) {
    h = (signed char*)ar.alloc(tn);
    if (!h) return 0;
  }
  int score = (int)pn;
  for (u32 blk = 0; blk < nblocks; ++blk) {
    u64 peq[5];
    build_peq(pat, pn, blk, peq);
    const bool last = (blk + 1 == nblocks);
    const u32 top = last ? (pn - blk * 64 - 1) : 63;
    u64 Pv = ~0ull, Mv = 0;
    for (u32 j = 0; j < tn; ++j) {
      u64 Eq = peq[txt.code(j)];
      const int hin = (blk == 0) ? 1 : (int)h[j];
      const u64 hneg = (hin < 0) ? 1ull : 0ull;
      const u64 Xv = Eq | Mv;
      Eq |= hneg;
      const u64 Xh = (((Eq & Pv) + Pv) ^ Pv) | Eq;
      u64 Ph = Mv | ~(Xh | Pv);
      u64 Mh = Pv & Xh;
      const int hout = (int)((Ph >> top) & 1ull) - (int)((Mh >> top) & 1ull);
      Ph <<= 1;
      Mh <<= 1;
      Mh |= hneg;
      Ph |= (hin > 0) ? 1ull : 0ull;
      Pv = Mh | ~(Xv | Ph);
      Mv = Ph & Xv;
      if (last) score += hout;
      else h[j] = (signed char)hout;
    }
  }
  ar.release(mk);
  return score;
}

// length of the longest common subsequence of a[0..an) and b[0..bn) (either may be empty)
TALC_HDN int lcs_length_scalar(const SeqView& a, u32 an, const SeqView& b, u32 bn, Arena& ar, DpStats* st) {
  const bool a_is_pat = an <= bn;
  const SeqView pat = a_is_pat ? a : b;
  const SeqView txt = a_is_pat ? b : a;
  const u32 pn = a_is_pat ? an : bn;
  const u32 tn = a_is_pat ? bn : an;
  if (st) st->cells_lcs += (u64)an * bn;
  const u32 nblocks = (pn + 63) / 64;
  const u32 mk = ar.mark();
  u8* carry = nullptr;
  if (nblocks > 1) {
    carry = (u8*)ar.alloc(tn);
    if (!carry) return 0;
  }
  int lcs = 0;
  for (u32 blk = 0; blk < nblocks; ++blk) {
    u64 peq[5];
    build_peq(pat, pn, blk, peq);
    const bool last = (blk + 1 == nblocks);
    const u32 rows = last ? (pn - blk * 64) : 64;
    u64 V = ~0ull;
    for (u32 j = 0; j < tn; ++j) {
      const u64 M = peq[txt.code(j)];
      const u64 U = V & M;
      const u64 cin = (blk == 0) ? 0ull : (u64)carry[j];
      const u64 t = V + U;
      const u64 sum = t + cin;
      const u64 cout = (u64)(t < V) | (u64)(sum < t);
      V = sum | (V & ~M);
      if (!last) carry[j] = (u8)cout;
    }
    const u64 zeros = ~V & ((rows == 64) ? ~0ull : ((1ull << rows) - 1ull));
#if defined(__CUDA_ARCH__)
    lcs += __popcll(zeros);
#else
    lcs += __builtin_popcountll(zeros);
#endif
  }
  ar.release(mk);
  return lcs;
}

#if defined(__CUDA_ARCH__)
// Edit distance and LCS length of the same pair in ONE systolic pass (Trajectory::scoreSequence computes both,
// Trajectory.cpp:239-243): the text stream, the match masks and the pipeline are shared, the two recurrences are
// independent dependency chains that fill each other's issue slots, and the two hand-over values travel in one
// shuffle.  Falls back to the two separate routines when a stripe of 32 blocks does not hold the longer sequence.
// `what`: 1 = the caller wants the distance, 2 = the LCS length, 3 = both (only decides which cells are tallied;
// ONE routine serves all three so that the scoring code the warps compete for in the instruction cache stays small).
__device__ __noinline__ int nw_lcs_fused(const SeqView& a, u32 an, const SeqView& b, u32 bn, Arena& ar, DpStats* st, int& lcsOut,
                                         int what) {
  const u32 longer = an >= bn ? an : bn;
  if (an == 0 || bn == 0) {  // the pipeline below needs a text character and a block
    lcsOut = 0;
    return (int)longer;
  }
  if (longer > 2048) {  // more than one stripe of 32 blocks: the striped scalar forms (rare)
    const int d = (what & 1) ? nw_distance_scalar(a, an, b, bn, ar, st) : 0;
    lcsOut = (what & 2) ? lcs_length_scalar(a, an, b, bn, ar, st) : 0;
    return d;
  }
  // rows (bit-parallel, 64 per lane) = the LONGER sequence: the pipeline runs for shorter + blocks steps
  const bool a_is_pat = an >= bn;
  const u32 pn = a_is_pat ? an : bn;
  const SeqView pat = a_is_pat ? a : b;  // by value: the fields stay in registers
  const SeqView txt = a_is_pat ? b : a;
  const u32 tn = a_is_pat ? bn : an;
  if (st) {
    if (what & 1) st->cells_nw += (u64)an * bn;
    if (what & 2) st->cells_lcs += (u64)an * bn;
  }
  const u32 lane = threadIdx.x & 31u;
  const u32 nblocks = (pn + 63) / 64;  // <= 32
  const bool haveBlk = lane < nblocks;
  u64 peq[5] = {0, 0, 0, 0, 0};
  if (haveBlk) build_peq(pat, pn, lane, peq);
  const bool last = haveBlk && (lane + 1 == nblocks);
  const u32 rows = last ? (pn - lane * 64) : 64;
  const u32 top = rows - 1;
  u64 Pv = ~0ull, Mv = 0, V = ~0ull;
  u32 outPrev = 1u | (4u << 4);  // what this lane hands to the next: (hout + 1) | (cout << 2) | (text character << 4)
  u32 chunk = 4u;                // the next 32 text characters, one per lane, reloaded every 32 steps
  int acc = 0;
  __syncwarp();
#pragma unroll 1
  for (u32 t = 0; t < tn + nblocks - 1; ++t) {
    const u32 ph = t & 31u;
    if (ph == 0) chunk = (t + lane < tn) ? txt.code(t + lane) : 4u;
    u32 in = __shfl_up_sync(0xffffffffu, outPrev, 1);
    const u32 c0 = __shfl_sync(0xffffffffu, chunk, ph);
    if (lane == 0) in = 2u | (c0 << 4);  // hin = +1 (first row of the distance matrix), no carry
    const u32 c = in >> 4;
    const bool valid = haveBlk && (t >= lane) && (t - lane < tn);
    u32 hand = 1u;
    if (valid) {
      const u64 M = peq[c];
      const int hin = (int)(in & 3u) - 1;
      // Myers / Hyyro
      u64 Eq = M;
      const u64 hneg = (hin < 0) ? 1ull : 0ull;
      const u64 Xv = Eq | Mv;
      Eq |= hneg;
      const u64 Xh = (((Eq & Pv) + Pv) ^ Pv) | Eq;
      u64 Ph = Mv | ~(Xh | Pv);
      u64 Mh = Pv & Xh;
      const int hout = (int)((Ph >> top) & 1ull) - (int)((Mh >> top) & 1ull);
      Ph <<= 1;
      Mh <<= 1;
      Mh |= hneg;
      Ph |= (hin > 0) ? 1ull : 0ull;
      Pv = Mh | ~(Xv | Ph);
      Mv = Ph & Xv;
      if (last) acc += hout;
      // bit-parallel LCS
      const u64 U = V & M;
      const u64 tt = V + U;
      const u64 sum = tt + (u64)((in >> 2) & 1u);
      const u32 cout = (u32)(tt < V) | (u32)(sum < tt);
      V = sum | (V & ~M);
      hand = (u32)(hout + 1) | (cout << 2);
    }
    outPrev = hand | (c << 4);
  }
  const int score = (int)pn + __shfl_sync(0xffffffffu, acc, nblocks - 1);
  int z = 0;
  if (haveBlk) z = __popcll(~V & ((rows == 64) ? ~0ull : ((1ull << rows) - 1ull)));
  lcsOut = (int)__reduce_add_sync(0xffffffffu, (unsigned)z);
  __syncwarp();
  return score;
}
__device__ __forceinline__ int nw_distance(const SeqView& a, u32 an, const SeqView& b, u32 bn, Arena& ar, DpStats* st) {
  int l;
  return nw_lcs_fused(a, an, b, bn, ar, st, l, 1);
}
__device__ __forceinline__ int lcs_length(const SeqView& a, u32 an, const SeqView& b, u32 bn, Arena& ar, DpStats* st) {
  int l;
  nw_lcs_fused(a, an, b, bn, ar, st, l, 2);
  return l;
}
#else
inline int nw_distance(const SeqView& a, u32 an, const SeqView& b, u32 bn, Arena& ar, DpStats* st) {
  return nw_distance_scalar(a, an, b, bn, ar, st);
}
inline int lcs_length(const SeqView& a, u32 an, const SeqView& b, u32 bn, Arena& ar, DpStats* st) {
  return lcs_length_scalar(a, an, b, bn, ar, st);
}
inline int nw_lcs_fused(const SeqView& a, u32 an, const SeqView& b, u32 bn, Arena& ar, DpStats* st, int& lcsOut, int what) {
  const int d = (what & 1) ? nw_distance_scalar(a, an, b, bn, ar, st) : 0;
  lcsOut = (what & 2) ? lcs_length_scalar(a, an, b, bn, ar, st) : 0;
  return d;
}
#endif

// Trail::Overlapscore in walk order: match 4 / mismatch -3 / gap -2, leading gaps of both
// sequences free, trailing gaps charged; score = bottom-right cell.
TALC_HDN int overlap_score_scalar(const SeqView& ref, u32 rn, const SeqView& cand, u32 cn, Arena& ar, DpStats* st) {
  if (st) st->cells_ovl += (u64)rn * cn;
  const u32 mk = ar.mark();
  i32* row = (i32*)ar.alloc((cn + 1) * 4);
  if (!row) return 0;
  for (u32 j = 0; j <= cn; ++j) row[j] = 0;
  for (u32 i = 0; i < rn; ++i) {
    const u32 rc = ref.code(i);
    i32 diag = row[0];  // S[i][0] = 0
    row[0] = 0;
    for (u32 j = 1; j <= cn; ++j) {
      const i32 up = row[j];
      i32 v = diag + ((rc == cand.code(j - 1)) ? 4 : -3);
      const i32 g1 = up - 2;
      const i32 g2 = row[j - 1] - 2;
      v = v > g1 ? v : g1;
      v = v > g2 ? v : g2;
      diag = up;
      row[j] = v;
    }
  }
  const int res = row[cn];
  ar.release(mk);
  return res;
}

#if defined(__CUDA_ARCH__)
// Device form: a skewed wavefront over stripes of 32 x kOvlCols columns.  Lane l owns kOvlCols adjacent columns
// of the stripe and works on row t-l at time t: the cell left of its first column (lane l-1, same row) was
// computed one step earlier and arrives by one shuffle together with the row's reference character; the diagonal
// term of the first column is the left value of the step before; inside the lane the columns chain through
// registers.  The last column of a stripe is parked in the arena (one value per row) and feeds lane 0 of the next
// stripe 32 rows at a time; lane 0 runs 31 rows ahead of lane 31, so the same buffer is read and overwritten in
// place.  Same integer recurrence as the scalar form; shuffles, loop control and the row feed are paid once per
// kOvlCols cells.  (Gardening scores EVERY trail of the frontier against the reference: with junction colours or
// at 15 % error this is the largest DP of a read -- 0.9 M and 4.5 M cells per read on configs 3 and 5.)
#define kOvlCols 4
// `bufs` (optional): one parked boundary column of rn+1 values per stripe, kept by the caller across calls.  The
// trails of a frontier share long prefixes (they branched from common ancestors) and are scored against the same
// reference in one scoreBridges round: a call may `skip` the leading stripes that lie inside the prefix the
// candidate shares with the candidate of the previous call -- their boundary columns are still valid.
__device__ __noinline__ int overlap_score_stripes(const SeqView& refArg, u32 rn, const SeqView& candArg, u32 cn, i32* bufs,
                                                  u32 skip, DpStats* st) {
  if (st) st->cells_ovl += (u64)rn * cn;
  const u32 W = 32u * kOvlCols;  // stripe width
  const SeqView ref = refArg, cand = candArg;  // by value: fields in registers
  const u32 lane = threadIdx.x & 31u;
  int result = 0;
  for (u32 j0 = 1 + skip * W; j0 <= cn; j0 += W) {
    const u32 sIdx = (j0 - 1) / W;
    const i32* colIn = sIdx ? bufs + (size_t)(sIdx - 1) * (rn + 1) : nullptr;  // S[i][j0-1]; column 0 is all zeros
    i32* colOut = bufs + (size_t)sIdx * (rn + 1);
    const u32 jf = j0 + kOvlCols * lane;  // this lane's first column
    const u32 ncols = cn - j0 + 1 < W ? cn - j0 + 1 : W;
    const u32 nl = (ncols + kOvlCols - 1) / kOvlCols;   // lanes that own a column of this stripe
    const bool park = (j0 + W <= cn) && (lane == 31);    // a further stripe follows
    u32 cc[kOvlCols];
    i32 up[kOvlCols];
#pragma unroll
    for (int c = 0; c < kOvlCols; ++c) {
      cc[c] = (jf + c <= cn) ? cand.code(jf + c - 1) : 9u;  // 9 never matches: columns beyond cn only ever feed
      up[c] = 0;                                            // columns further right, which do not exist either
    }
    i32 diag = 0;     // S[i-1][jf-1]
    i32 outPrev = 8;  // what this lane hands to the next: (value of its last column << 3) | reference character
    i32 chunk = 8;    // the same for lane 0, 32 rows at a time: (S[i][j0-1] << 3) | reference character
#pragma unroll 1
    for (u32 t = 1; t <= rn + nl - 1; ++t) {
      const u32 ph = (t - 1) & 31u;
      if (ph == 0) {
        const u32 r = t - 1 + lane;  // row r + 1
        chunk = (r < rn) ? (i32)(((u32)(colIn ? colIn[r + 1] : 0) << 3) | ref.code(r)) : 8;
      }
      i32 in = __shfl_up_sync(0xffffffffu, outPrev, 1);
      const i32 in0 = __shfl_sync(0xffffffffu, chunk, ph);
      if (lane == 0) in = in0;
      const u32 rc = (u32)in & 7u;
      const i32 leftIn = in >> 3;  // arithmetic shift: the value keeps its sign
      const u32 i = t - lane;      // wraps for t < lane: fails the range test below
      i32 v = 0;
      if (lane < nl && i >= 1 && i <= rn) {
        i32 left = leftIn, dg = diag;
#pragma unroll
        for (int c = 0; c < kOvlCols; ++c) {
          const i32 d = dg + ((rc == cc[c]) ? 4 : -3);
          const i32 g = (up[c] > left ? up[c] : left) - 2;
          v = d > g ? d : g;
          dg = up[c];   // S[i-1][col] is the diagonal term of the next column
          up[c] = v;
          left = v;
        }
        diag = leftIn;
        if (park) colOut[i] = v;
      }
      outPrev = (i32)(((u32)v << 3) | rc);
    }
    if (j0 + W > cn) {  // the last stripe holds column cn: lane (cn - j0) / kOvlCols, its column (cn - j0) % kOvlCols
      const u32 c = (cn - j0) % kOvlCols;
      i32 x = up[0];
#pragma unroll
      for (int q = 1; q < kOvlCols; ++q) x = (c == (u32)q) ? up[q] : x;
      result = __shfl_sync(0xffffffffu, x, (cn - j0) / kOvlCols);
    }
    __syncwarp();
  }
  return result;
}
// one pair on its own
__device__ __forceinline__ int overlap_score(const SeqView& ref, u32 rn, const SeqView& cand, u32 cn, Arena& ar, DpStats* st) {
  const u32 mk = ar.mark();
  const u32 ns = (cn + 32u * kOvlCols - 1) / (32u * kOvlCols);
  i32* bufs = (i32*)ar.alloc((ns ? ns : 1) * (rn + 1) * 4);
  if (!bufs) return 0;
  const int r = overlap_score_stripes(ref, rn, cand, cn, bufs, 0, st);
  ar.release(mk);
  return r;
}
// length of the common prefix (in bases, at most n) of two packed trails
__device__ __forceinline__ u32 packed_lcp(const u64* a, const u64* b, u32 n) {
  const u32 lane = threadIdx.x & 31u, nw = (n + 31) / 32;
  for (u32 base = 0; base < nw; base += 32) {
    const u32 wi = base + lane;
    const u64 x = (wi < nw) ? (a[wi] ^ b[wi]) : 0ull;
    const u32 m = __ballot_sync(0xffffffffu, x != 0ull);
    if (m) {
      const u32 l = (u32)__ffs((int)m) - 1;
      const u64 xl = __shfl_sync(0xffffffffu, x, l);
      const u32 p = (base + l) * 32 + (u32)__clzll((long long)xl) / 2;
      return p < n ? p : n;
    }
  }
  return n;
}
// Gardening (scoreBridges, Explorer.cpp:689-706): the n trails of a frontier, each cn bases long in a 2-bit slot
// (trail(j) -> words; bases past cn are stale), against the same reference.  The stripes of the DP that lie inside
// the prefix a trail shares with its predecessor in the list (siblings are neighbours) are not recomputed: their
// boundary columns are still parked from an earlier trail.  store(j, score) receives each result; false when the
// arena cannot hold the parked columns.
template <class TrailWords, class Store>
__device__ __forceinline__ bool overlap_score_frontier(const SeqView& ref, u32 rn, u32 cn, u32 n, TrailWords trail,
                                                       Store store, Arena& ar, DpStats* st) {
  const u32 W = 32u * kOvlCols, ns = (cn + W - 1) / W;
  const u32 mk = ar.mark();
  i32* bufs = (i32*)ar.alloc(ns * (rn + 1) * 4);
  if (!bufs) return false;
  TALC_ROLLED
  for (u32 j = 0; j < n; ++j) {
    u32 skip = 0;
    if (j) {
      skip = packed_lcp(trail(j), trail(j - 1), cn) / W;
      if (skip > ns - 1) skip = ns - 1;  // the last stripe carries the result
    }
    store(j, overlap_score_stripes(ref, rn, view_of_path(trail(j), cn), cn, bufs, skip, st));
  }
  ar.release(mk);
  return true;
}
#else
inline int overlap_score(const SeqView& ref, u32 rn, const SeqView& cand, u32 cn, Arena& ar, DpStats* st) {
  return overlap_score_scalar(ref, rn, cand, cn, ar, st);
}
#endif

// SeqAn 2.x _extendSeedGappedXDropOneDirection for Score(0,-1,-1) on query[qoff..qoff+qlen) (V, columns)
// and database[doff..doff+dlen) (H, rows), both in walk order.  Outputs how far the seed moved along
// the database (ext_rows) and the query (ext_cols).  `wide` sizes the three anti-diagonals for the
// worst case instead of the X-drop band (second-tier launch).
TALC_HDN void xdrop_extend_scalar(const SeqView& query, u32 qoff, u32 qlen, const SeqView& database, u32 doff, u32 dlen,
                          int scoreDropOff, u32& ext_rows, u32& ext_cols, i32& end_score, Arena& ar, bool wide, DpStats* st) {
  ext_rows = 0;
  ext_cols = 0;
  end_score = 0;
  const i64 cols = (i64)qlen + 1;
  const i64 rows = (i64)dlen + 1;
  if (rows == 1 || cols == 1) return;
  const int gapCost = -1;                 // max(scoreGap, INT_MIN / len) with scoreGap = -1
  const int undefined = INT32_MIN + 1;    // INT_MIN - gapCost
  // anti-diagonal storage: at most (maxCol - minCol) + 2 live entries each
  i64 capW = cols + 1;
  if (!wide) {
    const i64 band = (i64)(scoreDropOff > 0 ? scoreDropOff : 0) + 16;
    if (band < capW) capW = band;
  }
  const u32 mk = ar.mark();
  i32* buf = (i32*)ar.alloc((u32)(3 * capW * 4));
  if (!buf) return;
  i32* antiDiag1 = buf;
  i32* antiDiag2 = buf + capW;
  i32* antiDiag3 = buf + 2 * capW;
  i64 len1 = 0, len2 = 1, len3 = 2;

  i64 minCol = 1, maxCol = 2;
  i64 offset1 = 0, offset2 = 0, offset3 = 0;
  antiDiag2[0] = 0;
  if (-gapCost > scoreDropOff) {
    antiDiag3[0] = undefined;
    antiDiag3[1] = undefined;
  } else {
    antiDiag3[0] = gapCost;
    antiDiag3[1] = gapCost;
  }
  i64 antiDiagNo = 1;
  int best = 0;
  u64 cells = 0;

  while (minCol < maxCol) {
    ++antiDiagNo;
    {  // _swapAntiDiags
      i32* t = antiDiag1;
      antiDiag1 = antiDiag2;
      antiDiag2 = antiDiag3;
      antiDiag3 = t;
      len1 = len2;
      len2 = len3;
    }
    offset1 = offset2;
    offset2 = offset3;
    offset3 = minCol - 1;
    len3 = maxCol + 1 - offset3;
    if (len3 > capW) {  // band assumption violated: ask for the wide tier
      ar.overflow = 1;
      ar.release(mk);
      return;
    }
    {  // _initAntiDiag3
      const int minScore = best - scoreDropOff;
      antiDiag3[0] = undefined;
      antiDiag3[maxCol - offset3] = undefined;
      if ((int)antiDiagNo * gapCost > minScore) {
        if (offset3 == 0) antiDiag3[0] = (int)antiDiagNo * gapCost;
        if (antiDiagNo - maxCol == 0) antiDiag3[maxCol - offset3] = (int)antiDiagNo * gapCost;
      }
    }
    int antiDiagBest = (int)antiDiagNo * gapCost;
    for (i64 col = minCol; col < maxCol; ++col) {
      const i64 i3 = col - offset3, i2 = col - offset2, i1 = col - offset1;
      const u32 queryPos = (u32)(col - 1);
      const u32 dbPos = (u32)(antiDiagNo - col - 1);
      const int d2a = antiDiag2[i2 - 1], d2b = antiDiag2[i2];
      int tmp = (d2a > d2b ? d2a : d2b) + gapCost;
      const int sub = antiDiag1[i1 - 1] + ((query.code(qoff + queryPos) == database.code(doff + dbPos)) ? 0 : -1);
      tmp = tmp > sub ? tmp : sub;
      if (tmp < best - scoreDropOff) {
        antiDiag3[i3] = undefined;
      } else {
        antiDiag3[i3] = tmp;
        antiDiagBest = antiDiagBest > tmp ? antiDiagBest : tmp;
      }
    }
    cells += (u64)(maxCol - minCol);
    best = best > antiDiagBest ? best : antiDiagBest;

    while (minCol - offset3 < len3 && antiDiag3[minCol - offset3] == undefined && minCol - offset2 - 1 < len2 &&
           antiDiag2[minCol - offset2 - 1] == undefined) {
      ++minCol;
    }
    while (maxCol - offset3 > 0 && (antiDiag3[maxCol - offset3 - 1] == undefined) &&
           (antiDiag2[maxCol - offset2 - 1] == undefined)) {
      --maxCol;
    }
    ++maxCol;
    {
      const i64 lo = antiDiagNo + 2 - rows;  // end of databaseSeg reached?
      if (lo > minCol) minCol = lo;
      if (cols < maxCol) maxCol = cols;      // end of querySeg reached?
    }
  }
  if (st) st->cells_xdrop += cells;

  i64 longestExtensionCol = len3 + offset3 - 2;
  i64 longestExtensionRow = antiDiagNo - longestExtensionCol;
  int longestExtensionScore = antiDiag3[longestExtensionCol - offset3];
  if (longestExtensionScore == undefined) {
    if (antiDiag2[len2 - 2] != undefined) {  // reached end of query segment
      longestExtensionCol = len2 + offset2 - 2;
      longestExtensionRow = antiDiagNo - 1 - longestExtensionCol;
      longestExtensionScore = antiDiag2[longestExtensionCol - offset2];
    } else if (len2 > 2 && antiDiag2[len2 - 3] != undefined) {  // reached end of database segment
      longestExtensionCol = len2 + offset2 - 3;
      longestExtensionRow = antiDiagNo - 1 - longestExtensionCol;
      longestExtensionScore = antiDiag2[longestExtensionCol - offset2];
    }
  }
  if (longestExtensionScore == undefined) {  // general case: first strictly greatest on antiDiag1
    for (i64 i = 0; i < len1; ++i) {
      if (antiDiag1[i] > longestExtensionScore) {
        longestExtensionScore = antiDiag1[i];
        longestExtensionCol = i + offset1;
        longestExtensionRow = antiDiagNo - 2 - longestExtensionCol;
      }
    }
  }
  if (longestExtensionScore != undefined) {
    ext_rows = (u32)longestExtensionRow;
    ext_cols = (u32)longestExtensionCol;
    end_score = longestExtensionScore;
  }
  ar.release(mk);
}


}  // namespace talc
#include "xdrop.cuh"
namespace talc {

#if defined(__CUDA_ARCH__)
// Device form: the anti-diagonals live in registers (xdrop.cuh) while the band |diagonal| <= X fits 32*S
// diagonals (S = 1, 2, 4, 8; the slow tail of a batch are reads with long borders and large drop-offs, so S = 4 pays); beyond that (never seen on the benchmark workloads) every lane runs the scalar routine on the
// warp's arena.  Must be called by all 32 lanes with identical arguments.
__device__ __forceinline__ void xdrop_extend(const SeqView& query, u32 qoff, u32 qlen, const SeqView& database, u32 doff,
                                             u32 dlen, int scoreDropOff, u32& ext_rows, u32& ext_cols, i32& end_score,
                                             Arena& ar, bool wide, DpStats* st) {
  if (scoreDropOff <= 31) xdrop_extend_reg<1>(query, qoff, qlen, database, doff, dlen, scoreDropOff, ext_rows, ext_cols, end_score, st);
  else if (scoreDropOff <= 63) xdrop_extend_reg<2>(query, qoff, qlen, database, doff, dlen, scoreDropOff, ext_rows, ext_cols, end_score, st);
  else if (scoreDropOff <= 127) xdrop_extend_reg<4>(query, qoff, qlen, database, doff, dlen, scoreDropOff, ext_rows, ext_cols, end_score, st);
  else if (scoreDropOff <= 255) xdrop_extend_reg<8>(query, qoff, qlen, database, doff, dlen, scoreDropOff, ext_rows, ext_cols, end_score, st);
  else xdrop_extend_scalar(query, qoff, qlen, database, doff, dlen, scoreDropOff, ext_rows, ext_cols, end_score, ar, true, st);
}
#else
inline void xdrop_extend(const SeqView& query, u32 qoff, u32 qlen, const SeqView& database, u32 doff, u32 dlen,
                         int scoreDropOff, u32& ext_rows, u32& ext_cols, i32& end_score, Arena& ar, bool wide, DpStats* st) {
  xdrop_extend_scalar(query, qoff, qlen, database, doff, dlen, scoreDropOff, ext_rows, ext_cols, end_score, ar, wide, st);
}
#endif

// Trail.cpp:341-437 getSeedAndExtension in walk order.  refArg / candArg are the two arguments in the
// reference's order; `right` is the search direction.  Extensions are returned as walk-order prefix
// lengths of refArg and candArg.
struct SeedExt {
  u32 ref_ext;   // |refExtension|
  u32 cand_ext;  // |histExtension|
  i32 score;     // NW score of the two extensions (<= 0), or -xdrop when the seed could not extend
  bool stop;
};
TALC_HDN SeedExt seed_and_extension(const SeqView& refArg, const SeqView& candArg, int xdrop, bool right, u32 K,
                                   Arena& ar, bool wide, DpStats* st) {
  SeedExt r;
  const bool state = !(refArg.len < candArg.len);
  const SeqView& seq1 = state ? refArg : candArg;   // H / database (the longer one)
  const SeqView& seq2 = state ? candArg : refArg;   // V / query
  const u32 s = right ? (K - 1) : K;                // Q18: seed (0,0,K-1,K-1) vs (l1-K,l2-K,..)
  u32 er = 0, ec = 0;
  i32 endScore = 0;
  xdrop_extend(seq2, s, seq2.len - s, seq1, s, seq1.len - s, xdrop, er, ec, endScore, ar, wide, st);
  const u32 e1 = s + er, e2 = s + ec;
  r.ref_ext = state ? e1 : e2;
  r.cand_ext = state ? e2 : e1;
  const u32 mx = r.ref_ext > r.cand_ext ? r.ref_ext : r.cand_ext;
  if (mx >= K) {
    // Trail.cpp:422 runs a global alignment (0,-1,-1) of the two extended prefixes.  Its score is already known:
    // the cell the X-drop stopped in holds the exact edit distance of the two extensions (a cell survives only
    // with its true score, see xdrop.cuh), and the s leading bases are the anchor k-mer in both strings -- a common
    // prefix does not change an edit distance.  The reference's DP cells are still tallied.
#if defined(TALC_CHECK_SEED_SCORE)
    if (endScore != -nw_distance(refArg, r.ref_ext, candArg, r.cand_ext, ar, nullptr)) ar.overflow = 2;
#endif
    if (st) st->cells_nw += (u64)r.ref_ext * r.cand_ext;
    r.score = endScore;
    r.stop = false;
  } else {  // Q19
    r.score = -xdrop;
    r.stop = true;
  }
  return r;
}

// ---- self-tests of the scoring primitives (talc_test_align*, and the host emulation in tests/hostemu)
// One side of a pair as the pipeline hands it over: with step +1 / -1, `len` bases of `rd` from `start` in walk order,
// the read packed as the Corrector packs it (2 bits per base, 4 when the read holds an N); with step 0, the bases
// rd[start, start + len) (A, C, G, T only) as a 2-bit trail slot whose bits past `len` are stale (seeded by `salt`).
// Must be called by all lanes of the warp with identical arguments; nullptr words when the arena is exhausted.
TALC_HD SeqView selftest_view(const ReadView& rd, i32 start, i32 step, u32 len, u64 salt, Arena& ar) {
  SeqView v;
  v.start = start;
  v.step = step;
  v.len = len;
  v.lg = 5;
  if (step != 0) {
    u64* w = (u64*)ar.alloc(packed_read_alloc(rd.len) * 8);
    v.w = w;
    if (!w) return v;
    bool hasN = false;
    for (u32 i = lane_id(); i < rd.len; i += lane_count()) hasN |= rd.code(i) > 3;
    hasN = warp_any(hasN);
    for (u32 wi = lane_id(); wi < packed_read_words(rd.len, hasN); wi += lane_count()) w[wi] = packed_read_word(rd, wi, hasN);
    v.lg = hasN ? 4u : 5u;
  } else {
    const u32 nw = (len + 31) / 32 + 1;
    u64* w = (u64*)ar.alloc(nw * 8);
    v.w = w;
    v.start = 0;
    v.step = 1;
    if (!w) return v;
    for (u32 wi = lane_id(); wi < nw; wi += lane_count()) {
      u64 x = (salt << 20) + wi + 1;  // splitmix64
      x = (x ^ (x >> 30)) * 0xbf58476d1ce4e5b9ull;
      x = (x ^ (x >> 27)) * 0x94d049bb133111ebull;
      x ^= x >> 31;
      for (u32 j = 0; j < 32 && 32 * wi + j < len; ++j) {
        const u32 sh = 62 - 2 * j;
        x = (x & ~(3ull << sh)) | ((u64)(rd.code((u32)start + 32 * wi + j) & 3u) << sh);
      }
      w[wi] = x;
    }
  }
  warp_sync();
  return v;
}
// op 0: -edit distance, 1: LCS length, 2: overlap score (a = reference, b = candidate) -> r[0];
// 3: seed_and_extension(a, b, X = aux, right = aux2) -> {ref_ext, cand_ext, score, stop};
// 4: X-drop of query a against database b from the origin, X = aux -> {ext_rows, ext_cols, cells, end score};
// 5: distance and LCS of one fused pass -> {-distance, LCS length}.  r[0] = INT32_MIN when the arena overflowed.
TALC_HDN void selftest_align_op(int op, const SeqView& va, const SeqView& vb, int aux, int aux2, u32 K, Arena& ar, i32 r[4]) {
  r[0] = r[1] = r[2] = r[3] = 0;
  if (op == 0) r[0] = -nw_distance(va, va.len, vb, vb.len, ar, nullptr);
  else if (op == 1) r[0] = lcs_length(va, va.len, vb, vb.len, ar, nullptr);
  else if (op == 2) r[0] = overlap_score(va, va.len, vb, vb.len, ar, nullptr);
  else if (op == 5) {
    int l = 0;
    r[0] = -nw_lcs_fused(va, va.len, vb, vb.len, ar, nullptr, l, 3);
    r[1] = l;
  } else if (op == 4) {
    DpStats ds;
    ds.cells_xdrop = 0;
    u32 er = 0, ec = 0;
    i32 es = 0;
    xdrop_extend(va, 0, va.len, vb, 0, vb.len, aux, er, ec, es, ar, true, &ds);
    r[0] = (i32)er;
    r[1] = (i32)ec;
    r[2] = (i32)ds.cells_xdrop;
    r[3] = es;
  } else {
    const SeedExt e = seed_and_extension(va, vb, aux, aux2 != 0, K, ar, true, nullptr);
    r[0] = (i32)e.ref_ext;
    r[1] = (i32)e.cand_ext;
    r[2] = e.score;
    r[3] = e.stop ? 1 : 0;
  }
  if (ar.overflow) r[0] = INT32_MIN;
}

}  // namespace talc
