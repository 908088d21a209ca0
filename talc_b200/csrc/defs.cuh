// defs.cuh -- shared definitions for the TALC correction path on B200.
//
// Everything marked TALC_HD is plain C++ without warp intrinsics so that the same
// source compiles (a) with nvcc for sm_100a, where it is the product, and (b) with
// g++ inside tests/hostemu, where it is only a debugging aid that lets the logic be
// diffed against the oracle without a GPU.  The shipped library has no CPU path.
#pragma once
#include <stdint.h>
#include <string.h>

// TALC_HD: small helpers, always inlined.  TALC_HDN: the big routines; they stay real calls on the device
// (forcing the whole per-read pipeline into one function body makes the NVVM optimiser run for an hour).
// Loops of the per-read control code stay rolled on the device: the correction kernel is bound by instruction
// delivery (DESIGN.md section 5), and unrolled copies of rarely-hot loop bodies only evict the hot loops.
#if defined(__CUDACC__)
#define TALC_ROLLED _Pragma("unroll 1")
#else
#define TALC_ROLLED
#endif
#if defined(__CUDACC__)
#define TALC_HD __host__ __device__ __forceinline__
#define TALC_HDN __host__ __device__ __noinline__
#else
#define TALC_HD inline
#define TALC_HDN inline
#endif

// launch shape of the correction kernel: 4 warps (= 4 reads in flight) per 128-thread block
#define TALC_WARPS_PER_BLOCK 4

namespace talc {

typedef uint8_t u8;
typedef uint16_t u16;
typedef uint32_t u32;
typedef uint64_t u64;
typedef int32_t i32;
typedef int64_t i64;

// Tunables of the reference: Settings.cpp:33-69 (CLI-settable) and the file-static
// constants of Explorer.cpp:85-102 / Jellyfish.cpp:64 / Read.cpp:361,368.
struct Params {
  u32 K;
  u32 min_count;        // gp_MIN_COUNT
  u32 window;           // gp_WINDOW_SIZE
  u32 max_branches;     // gp_MAX_NB_COMPETING_PATHS
  double alpha;         // gp_ALPHA
  double sr_error;      // gp_SR_ERROR_RATE
  double min_inner;     // gp_MIN_INNER_SCORE
  double min_border;    // gp_MIN_BORDER_SCORE
  i32 cycle_mode;       // 0: SeqAn2 Horspool over mixed alphabets (stride-K windows); 1: exact first occurrence
  i32 q11_zero;         // Explorer.cpp:705 UB loop counter modelled as j = 0
};

enum : u32 {
  kMinStartAnchors = 3,      // Explorer.cpp:85
  kMaxStartAnchors = 5,      // :86
  kMaxInCount = 100000,      // :88
  kMaxBorderPaths = 75,      // :90
  kMaxInnerPaths = 50,       // :91
  kCheckInterval = 6,        // :93
  kMaxBorderFailures = 3,    // :97
  kBorderMaxLen = 500,       // Read.cpp:361,368
  kColouredCountThr = 10000  // Jellyfish.cpp:64
};

// per-read outcome (main.cpp:262-296)
enum ReadStatus : u8 {
  kReadOk = 0,
  kReadNoSolid = 1,      // "No solid kmer could be found."
  kReadNoStructure = 2,  // "Unable to define convenient structure."
  kReadShort = 3,        // len <= K : untouched, not logged
  kReadResource = 4,     // not in the reference: the read exhausted even the last scratch tier and passes through uncorrected
  kReadOverflow = 250,   // internal: scratch arena too small, re-run with a larger arena
  kReadYield = 251       // internal: the read waits for the walk kernel (its context stays in HBM)
};

// Dna5 code of an input character (SeqAn char -> Dna5): ACGT either case, U -> T, else N(4).
// Branch-free: bits 1-2 of the ASCII code separate A,C,G,T/U; five compares validate the letter.
TALC_HD u32 base_code(u8 c) {
  const u32 idx = ((u32)c | 0x20u) - 0x61u;  // a..u -> 0..20
  const u32 x = (((u32)c >> 1) & 3u) ^ (((u32)c >> 2) & 1u);
  const bool ok = (idx < 21u) & (((0x180045u >> (idx & 31u)) & 1u) != 0u);  // bit set for a, c, g, t, u
  return ok ? x : 4u;
}

// The 32 lanes of the warp that owns a read cooperate on the linear scans; on the host (tests/hostemu)
// a "warp" is one lane and the reductions are identities.
#if defined(__CUDA_ARCH__)
TALC_HD u32 lane_id() { return threadIdx.x & 31u; }
TALC_HD u32 lane_count() { return 32u; }
TALC_HD u32 warp_sum(u32 v) { return __reduce_add_sync(0xffffffffu, v); }
TALC_HD u32 warp_max(u32 v) { return __reduce_max_sync(0xffffffffu, v); }
TALC_HD void warp_sync() { __syncwarp(); }
TALC_HD bool warp_any(bool v) { return __any_sync(0xffffffffu, v) != 0; }
TALC_HD u64 warp_sum64(u64 v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
#else
inline u32 lane_id() { return 0; }
inline u32 lane_count() { return 1; }
inline u32 warp_sum(u32 v) { return v; }
inline u32 warp_max(u32 v) { return v; }
inline u64 warp_sum64(u64 v) { return v; }
inline void warp_sync() {}
inline bool warp_any(bool v) { return v; }
#endif
TALC_HD u8 code_char(u32 code) { return (u8)("ACGTN"[code]); }

// Dna5 conversion followed by SeqAn's reverseComplement, one base: ACGT in either case -> complement, anything else -> N
TALC_HD u8 dna5_complement(u8 c) {
  switch (c) {
    case 'A': case 'a': return 'T';
    case 'C': case 'c': return 'G';
    case 'G': case 'g': return 'C';
    case 'T': case 't': return 'A';
    default: return 'N';
  }
}

TALC_HD u64 kmer_mask(u32 K) { return (K >= 32) ? ~0ull : ((1ull << (2 * K)) - 1ull); }

// The reverse complement of a rolled k-mer, rolled alongside it: push base code c (0..3) of the read.  After K pushes
// it is the reverse complement of the last K bases, whatever it held before.
TALC_HD u64 kmer_roll_rc(u64 rc, u32 c, u32 K) { return (rc >> 2) | ((u64)(3u - (c & 3u)) << (2 * (K - 1))); }
TALC_HD u64 kmer_revcomp(u64 k, u32 K) {
  u64 r = 0;
  for (u32 i = 0; i < K; ++i) {
    r = (r << 2) | (3 - (k & 3));
    k >>= 2;
  }
  return r;
}

// --strand auto.  A read's k-mers and the k-mers of its reverse complement (dna5_complement, read backwards) rolled
// together, one byte per base, K <= 31.  After base p + K - 1 has been pushed, `fwd` is the window of the read at p and
// `rc` the window of the reverse complement at len - K - p, i.e. the reverse complement of `fwd`; a window holds no N
// when the matching run counter is >= K.  The two runs differ only on 'U', which base_code reads as T and
// dna5_complement turns into N.
struct StrandRoll {
  u64 fwd, rc;
  u32 runF, runR;  // bases since the last N of the read / of its reverse complement
};
TALC_HD StrandRoll strand_roll_start() { return StrandRoll{0ull, 0ull, 0u, 0u}; }
TALC_HD void strand_roll_push(StrandRoll& s, u8 ch, u32 K) {
  const u32 c = base_code(ch);
  const bool nR = (c > 3u) | (((u32)ch | 0x20u) == (u32)'u');
  s.runF = (c > 3u) ? 0u : s.runF + 1u;
  s.runR = nR ? 0u : s.runR + 1u;
  s.fwd = ((s.fwd << 2) | (u64)(c & 3u)) & kmer_mask(K);
  s.rc = kmer_roll_rc(s.rc, c, K);
}
// found_fwd / found_rc: windows without N found in the table on either strand.  Antisense (1) only on a strict
// majority: ties -- reads shorter than K, all-N reads, reverse palindromes -- stay forward (0).
TALC_HD u32 strand_decide(u32 found_fwd, u32 found_rc) { return found_rc > found_fwd ? 1u : 0u; }

// k-mers are 2-bit packed with the first base in the most significant position.
// Successors (utils.cpp:370-387): RIGHT x[1..]+b ; LEFT b+x[..K-2]
TALC_HD u64 kmer_next(u64 kmer, u32 b, bool right, u32 K) {
  return right ? (((kmer << 2) | (u64)b) & kmer_mask(K)) : ((kmer >> 2) | ((u64)b << (2 * (K - 1))));
}

// ---- bump arena over a per-thread slice of global scratch --------------------
struct Arena {
  u8* base;
  u32 cap;
  u32 top;
  u32 overflow;
  TALC_HD void init(u8* b, u32 c) { base = b; cap = c; top = 0; overflow = 0; }
  TALC_HD u32 mark() const { return top; }
  TALC_HD void release(u32 m) { top = m; }
  // returns nullptr (and latches overflow) when the slice is exhausted
  TALC_HD void* alloc(u32 bytes) {
    u32 t = (top + 7u) & ~7u;
    if (bytes > cap || t > cap - bytes) { overflow = 1; return nullptr; }
    top = t + bytes;
    return base + t;
  }
};

// ---- a read as the kernels see it: ASCII bytes in HBM --------------------------
struct ReadView {
  const u8* s;  // ASCII
  u32 len;
  TALC_HD u32 code(u32 i) const { return base_code(s[i]); }
  // packed k-mer starting at base i; ok=false if it contains N
  TALC_HD u64 kmer_at(u32 i, u32 K, bool& ok) const {
    u64 v = 0;
    ok = true;
    for (u32 j = 0; j < K; ++j) {
      u32 c = code(i + j);
      if (c > 3) { ok = false; c = 0; }
      v = (v << 2) | c;
    }
    return v;
  }
};

// The reference string of a search in *walk order*: element i is read[start + i] for a
// RIGHT-ward walk and read[start - i] for a LEFT-ward walk.  Every reference string the
// reference builds (anchor+gap+target, target+gap+anchor, anchor+border, border+anchor:
// Explorer.cpp:925-938,1042-1053) is a contiguous slice of the raw read, so no copy is made.
// The scoring loops never see ASCII: the read is packed once per read (Corrector::run), 2 bits per base when it
// holds no N (lg = 5: 32 bases per word, the same layout as a trail), else 4 bits per base (lg = 4, N = 4).
// One access path for both: word idx >> lg, field of 64 >> lg bits, first base most significant.
TALC_HD u32 packed_code(const u64* w, u32 idx, u32 lg) {
  // field width 64 >> lg = 1 << (6 - lg); base j of a word sits (per - 1 - j) fields above bit 0
  const u32 sh = (~idx & ((1u << lg) - 1u)) << (6u - lg);
  return (u32)(w[idx >> lg] >> sh) & (lg == 5u ? 3u : 15u);
}
// The packed read: words [0, packed_read_words(len, hasN)) are filled, one more than the bases need, with zeros past
// the read's end; a buffer of packed_read_alloc(len) words holds either layout.
TALC_HD u32 packed_read_alloc(u32 len) { return (len + 15) / 16 + 2; }
TALC_HD u32 packed_read_words(u32 len, bool hasN) { return hasN ? (len + 15) / 16 + 1 : (len + 31) / 32 + 1; }
TALC_HD u64 packed_read_word(const ReadView& rd, u32 wi, bool hasN) {
  const u32 per = hasN ? 16u : 32u, bits = hasN ? 4u : 2u;
  u64 x = 0;
  TALC_ROLLED
  for (u32 j = 0; j < per; ++j) {
    const u32 idx = wi * per + j;
    x = (x << bits) | (u64)((idx < rd.len) ? rd.code(idx) : 0u);
  }
  return x;
}
struct RefView {
  const u64* w;  // packed read
  i32 start;
  i32 step;  // +1 or -1
  u32 len;
  u32 lg;
  TALC_HD u32 code(u32 i) const { return packed_code(w, (u32)(start + (i32)i * step), lg); }
};

// A trail's sequence in walk order, 2-bit packed (32 bases per u64, first base most significant).
// Paths only ever contain A,C,G,T (anchors come from the table, successors from kDict).
struct PathView {
  const u64* w;
  u32 len;
  TALC_HD u32 code(u32 i) const { return (u32)((w[i >> 5] >> (62 - 2 * (i & 31))) & 3ull); }
};
TALC_HD void path_set(u64* w, u32 i, u32 c) {
  const u32 sh = 62 - 2 * (i & 31);
  w[i >> 5] = (w[i >> 5] & ~(3ull << sh)) | ((u64)c << sh);
}
// k-mer (first base most significant) whose first base is walk index i
TALC_HD u64 path_kmer_fwd(const u64* w, u32 i, u32 K) {
  const u32 wi = i >> 5, off = 2 * (i & 31);
  u64 hi = w[wi] << off;
  if (off && (off + 2 * K > 64)) hi |= w[wi + 1] >> (64 - off);
  return hi >> (64 - 2 * K);
}

}  // namespace talc
