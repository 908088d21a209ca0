// talc_b200.cu -- sm_100a kernels and the C ABI (include/talc_b200.h) of the TALC correction path.
//
// Kernels (all HBM / integer bound; nothing here is a dense contraction, so no tensor cores):
//   table_insert_kernel / table_finalize_kernel / table_colour_kernel   k-mer table build in HBM
//   ctx_fill_empty_kernel / ctx_build_kernel                            successor tables derived from the k-mer table
//   kmer_count_kernel + coverage_kernel                                 Read::reCoverage, batched
//   cost_key_kernel (+ cub radix sort)                                  processing order: estimated cost, descending
//   correct_kernel                                                      segmentation + graph search + scoring
//   gather_kernel                                                       corrected reads back into input order
//   revcomp_reads_kernel                                                --reverse: every read reverse-complemented first
// Grid sizes are multiples of the SM count; per-thread scratch lives in HBM (180 GB makes that cheap).
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <sys/stat.h>

#include <algorithm>
#include <chrono>
#include <cub/cub.cuh>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "../../include/talc_b200.h"
#include "correct.cuh"
#include "walk.cuh"
#include "count_gpu.cuh"
#include "dump_gpu.cuh"
#include "dump_parse.hpp"

using namespace talc;

// =====================================================================================
// table build
// =====================================================================================
// Entry i of the dump (file order) claims a slot with CAS, then the (line index, count) pair with the
// smallest line index wins through a 64-bit atomicMin: that is map::insert's "first line wins"
// (Jellyfish.cpp:262) independent of the order in which threads arrive (SURVEY E2).
// `line0` is the dump-line index of entry 0 (the GPU parser inserts a dump piece by piece); a table without a free
// slot ends the probe after one lap and raises *fail instead of spinning.
__global__ void table_insert_kernel(Slot* slots, u64 mask, const u64* keys, const u32* counts, u64 n, u64 line0, u32* fail) {
  const u64 stride = (u64)gridDim.x * blockDim.x;
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const u64 key = keys[i];
    if (key == kEmptyKey) continue;  // the GPU parser marks filtered / malformed lines this way
    u64 b = hash_kmer(key) & mask & ~1ull;
    Slot* hit = nullptr;
    for (u64 lap = 0; !hit && lap <= mask; lap += 2) {
      for (int j = 0; j < 2 && !hit; ++j) {
        Slot* s = slots + b + j;
        unsigned long long prev = *(volatile unsigned long long*)&s->key;
        if (prev == kEmptyKey) prev = atomicCAS((unsigned long long*)&s->key, (unsigned long long)kEmptyKey, (unsigned long long)key);
        if (prev == kEmptyKey || prev == key) hit = s;
      }
      b = (b + 2) & mask;
    }
    if (!hit) { atomicExch(fail, 1u); continue; }
    const unsigned long long v = ((unsigned long long)(line0 + i) << 32) | (unsigned long long)counts[i];
    atomicMin((unsigned long long*)&hit->count, v);  // {count, colour} viewed as one u64: colour half carries the line index
  }
}
// strip the line index: colour := 0 for every occupied slot, count stays
__global__ void table_finalize_kernel(Slot* slots, u64 capacity, unsigned long long* n_entries) {
  const u64 stride = (u64)gridDim.x * blockDim.x;
  unsigned long long mine = 0;
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < capacity; i += stride) {
    if (slots[i].key != kEmptyKey) {
      slots[i].colour = 0;
      ++mine;
    } else {
      slots[i].count = 0;
      slots[i].colour = 0;
    }
  }
  if (mine) atomicAdd(n_entries, mine);
}
__global__ void table_fill_empty_kernel(Slot* slots, u64 capacity) {
  const u64 stride = (u64)gridDim.x * blockDim.x;
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < capacity; i += stride) {
    slots[i].key = kEmptyKey;
    slots[i].count = 0xFFFFFFFFu;
    slots[i].colour = 0xFFFFFFFFu;
  }
}
// junction colours: the host has already reduced the junction dump to one final value per k-mer
// ("last line wins, forward before reverse complement": Jellyfish.cpp:284-286); only existing keys change
__global__ void table_colour_kernel(Slot* slots, u64 mask, const u64* keys, const u32* colours, u64 n) {
  const u64 stride = (u64)gridDim.x * blockDim.x;
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const u64 key = keys[i];
    u64 b = hash_kmer(key) & mask & ~1ull;
    for (u64 lap = 0; lap <= mask; lap += 2) {
      bool done = false;
      for (int j = 0; j < 2; ++j) {
        Slot* s = slots + b + j;
        if (s->key == key) { s->colour = colours[i]; done = true; break; }
        if (s->key == kEmptyKey) { done = true; break; }
      }
      if (done) break;
      b = (b + 2) & mask;
    }
  }
}
// successor tables (table.cuh): every occupied slot of the k-mer table enters its RIGHT context bucket (key
// without its last base) and its LEFT context bucket (key without its first base); a bucket is claimed with CAS
// on the context, each of its four count fields has exactly one writer
__global__ void ctx_fill_empty_kernel(CtxBucket* b, u64 capacity) {
  const u64 stride = (u64)gridDim.x * blockDim.x;
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < capacity; i += stride) {
    b[i].ctx = kEmptyKey;
    b[i].cnt[0] = b[i].cnt[1] = b[i].cnt[2] = b[i].cnt[3] = 0;
    b[i].colmask = 0;
    b[i].pad = 0;
  }
}
__device__ __forceinline__ void ctx_insert(CtxBucket* tb, u64 mask, u64 ctx, u32 b, u32 count, u32 colour, u32* fail) {
  u64 i = hash_ctx(ctx) & mask;
  for (u64 lap = 0; lap <= mask; ++lap) {
    unsigned long long prev = *(volatile unsigned long long*)&tb[i].ctx;
    if (prev == kEmptyKey) prev = atomicCAS((unsigned long long*)&tb[i].ctx, (unsigned long long)kEmptyKey, (unsigned long long)ctx);
    if (prev == kEmptyKey || prev == ctx) {
      tb[i].cnt[b] = count;
      if (colour) atomicOr(&tb[i].colmask, 1u << b);
      return;
    }
    i = (i + 1) & mask;
  }
  atomicExch(fail, 1u);  // no free bucket (cannot happen with the load <= 1/3 sizing from a recounted table)
}
__global__ void table_count_kernel(const Slot* slots, u64 capacity, unsigned long long* n_entries) {
  const u64 stride = (u64)gridDim.x * blockDim.x;
  unsigned long long mine = 0;
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < capacity; i += stride) mine += slots[i].key != kEmptyKey ? 1 : 0;
  mine = __reduce_add_sync(0xffffffffu, (u32)mine);  // <= 32 * (capacity / stride + 1) per warp: fits 32 bits
  if ((threadIdx.x & 31) == 0 && mine) atomicAdd(n_entries, mine);
}
__global__ void ctx_build_kernel(const Slot* slots, u64 capacity, CtxBucket* right, CtxBucket* left, u64 mask, u32 K, u32* fail) {
  const u64 stride = (u64)gridDim.x * blockDim.x;
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < capacity; i += stride) {
    const Slot s = slots[i];
    if (s.key == kEmptyKey) continue;
    ctx_insert(right, mask, s.key >> 2, (u32)(s.key & 3ull), s.count, s.colour, fail);
    ctx_insert(left, mask, s.key & kmer_mask(K - 1), (u32)(s.key >> (2 * (K - 1))), s.count, s.colour, fail);
  }
}

__global__ void table_lookup_kernel(TableView tv, const u64* keys, u64 n, u32* counts, u32* colours, u8* found) {
  const u64 stride = (u64)gridDim.x * blockDim.x;
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    u32 c, col;
    found[i] = table_lookup(tv, keys[i], c, col) ? 1 : 0;
    counts[i] = c;
    colours[i] = col;
  }
}

// =====================================================================================
// coverage (Read::reCoverage / getLRCountsInSRFromDBG, Read.cpp:174-195, Jellyfish.cpp:485-496)
// =====================================================================================
__global__ void kmer_count_kernel(const u64* offs, u32 n, u32 K, u64* nk, u32* sortKey, u32* sortVal) {
  const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const u64 len = offs[i + 1] - offs[i];
  nk[i] = len >= K ? len - K + 1 : 0;
  sortKey[i] = 0xFFFFFFFFu - (u32)len;  // ascending key = descending length
  sortVal[i] = i;
}
// Scheduling key of a read (results do not depend on it): reads are handed to the warps most expensive first.
// Cost grows with the length and, much faster, with the length of a correctable head / tail (<= 500 bases:
// Read.cpp:361,368): a border search re-scores every trail from its seed every 6 steps (Explorer.cpp:709-740),
// quadratic in the border length (profiles/r01_slow_reads.log).  One warp per read scans its coverage for the
// first and the last solid k-mer.
__global__ void cost_key_kernel(const u32* __restrict__ cov, const u64* __restrict__ kmerOff, const u64* __restrict__ offs, u32 n,
                                u32 minCount, u32* sortKey, u32* sortVal) {
  const u32 lane = threadIdx.x & 31;
  const u32 warpsPerBlock = blockDim.x >> 5;
  for (u32 r = blockIdx.x * warpsPerBlock + (threadIdx.x >> 5); r < n; r += gridDim.x * warpsPerBlock) {
    const u32 C = (u32)(kmerOff[r + 1] - kmerOff[r]);
    const u32* cv = cov + kmerOff[r];
    u32 first = C, last = 0;
    bool any = false;
    for (u32 base = 0; base < C && !any; base += 32) {
      const u32 m = __ballot_sync(0xffffffffu, base + lane < C && cv[base + lane] >= minCount);
      if (m) { first = base + (u32)__ffs((int)m) - 1; any = true; }
    }
    if (any) {
      for (u32 top = C; top > 0; top -= (top < 32 ? top : 32)) {
        const u32 base = top < 32 ? 0 : top - 32;
        const u32 m = __ballot_sync(0xffffffffu, base + lane < top && cv[base + lane] >= minCount);
        if (m) { last = base + 31 - (u32)__clz((int)m); break; }
      }
    }
    if (lane == 0) {
      const u64 len = offs[r + 1] - offs[r];
      u64 est = 0;
      if (any) {
        const u64 h = first <= kBorderMaxLen ? first : 0, t = (C - 1 - last) <= kBorderMaxLen ? (C - 1 - last) : 0;
        est = len + (h * h + t * t) / 5;
      }
      sortKey[r] = 0xFFFFFFFFu - (u32)(est > 0xFFFFFFFEull ? 0xFFFFFFFEull : est);  // ascending key = descending cost
      sortVal[r] = r;
    }
  }
}
// One warp per read; each lane rolls a 2-bit k-mer over 4 consecutive positions (K+3 byte loads for 4
// probes), probes the table (one 32-byte sector per probe), and the warp writes 512 contiguous bytes.
__global__ void __launch_bounds__(256) coverage_kernel(TableView tv, u32 K, const u8* __restrict__ bases,
                                                       const u64* __restrict__ offs, const u64* __restrict__ kmerOff,
                                                       u32 n, u32* __restrict__ cov) {
  const u32 lane = threadIdx.x & 31;
  const u32 warpsPerBlock = blockDim.x >> 5;
  const u64 kmask = kmer_mask(K);
  for (u32 r = blockIdx.x * warpsPerBlock + (threadIdx.x >> 5); r < n; r += gridDim.x * warpsPerBlock) {
    const u64 o = offs[r];
    const u32 len = (u32)(offs[r + 1] - o);
    if (len < K) continue;
    const u32 C = len - K + 1;
    const u8* s = bases + o;
    u32* out = cov + kmerOff[r];
    for (u32 base = 0; base < C; base += 128) {
      const u32 p0 = base + lane * 4;
      if (p0 >= C) continue;
      u64 km = 0;
      u32 bad = 0;  // number of bases since the last N, saturating at K
      for (u32 j = 0; j < K; ++j) {
        const u32 c = base_code(__ldg(s + p0 + j));
        bad = (c > 3) ? 0 : (bad + 1);
        km = ((km << 2) | (c & 3)) & kmask;
      }
      u32 cnt[4] = {0, 0, 0, 0};
      u64 kms[4];
      u32 okm = 0;
      kms[0] = km;
      okm |= (bad >= K) ? 1u : 0u;
#pragma unroll
      for (u32 q = 1; q < 4; ++q) {
        if (p0 + q < C) {
          const u32 c = base_code(__ldg(s + p0 + q + K - 1));
          bad = (c > 3) ? 0 : (bad + 1);
          km = ((km << 2) | (c & 3)) & kmask;
          okm |= (bad >= K) ? (1u << q) : 0u;
        }
        kms[q] = km;
      }
      // issue the four home-sector fetches together
      Slot s0[4], s1[4];
      u64 b[4];
#pragma unroll
      for (u32 q = 0; q < 4; ++q) {
        b[q] = hash_kmer(kms[q]) & tv.mask & ~1ull;
        if ((okm >> q) & 1u) load_sector(tv.slots + b[q], s0[q], s1[q]);
      }
#pragma unroll
      for (u32 q = 0; q < 4; ++q) {
        if ((okm >> q) & 1u) {
          u32 col;
          const int rr = sector_resolve(s0[q], s1[q], kms[q], cnt[q], col);
          if (rr < 0) table_probe_from(tv, b[q], kms[q], cnt[q], col);
        }
      }
      if (p0 + 3 < C && ((((size_t)(out + p0)) & 15) == 0)) {
        *reinterpret_cast<uint4*>(out + p0) = make_uint4(cnt[0], cnt[1], cnt[2], cnt[3]);
      } else {
        for (u32 q = 0; q < 4 && p0 + q < C; ++q) out[p0 + q] = cnt[q];
      }
    }
  }
}

// =====================================================================================
// correction: one warp per read, warps pull reads one at a time from a cost-sorted queue
// =====================================================================================
struct CorrectArgs {
  TableView tv;
  Params P;
  ModelTabs tabs;
  const u8* bases;
  const u64* offs;
  const u64* kmerOff;
  const u32* cov;
  const u32* order;   // read indices, longest first
  u32 nOrder;
  u8* arenas;
  u32 arenaBytes;
  u8* outArena;       // corrected reads, allocation order
  u64 outCap;
  unsigned long long* outCursor;
  u64* outPos;
  u32* outLen;
  u8* status;
  unsigned long long* counters;  // kNumCounters
  u32* workCounter;
  u32* overflowList;
  u32* nOverflow;
  u32* outFull;
  u32* readKcycles;  // optional: per-read elapsed SM cycles / 1024 (tuning aid)
  u32* readStats;    // optional: per read {span of the final solid regions in k-mers, number of regions} (Read.cpp:418-433)
  CtxView cright, cleft;  // successor tables
  u32 wide;      // worst-case sizing of the X-drop anti-diagonals (align.cuh)
  u32 inlineInner, inlineBorder;  // split mode: ordinary steps taken inside control_kernel before a frontier is handed over
  u32 pauseCycles;  // split mode: SM cycles a read may run per round before it gives its warp back (0 = no limit)
  u32 lastTier;  // no larger arena follows: a read that overflows passes through uncorrected (kReadResource)
};

// One warp owns one read.  All 32 lanes run the per-read control flow on the same data, so the warp
// never diverges (a thread-per-read mapping serialises: the threads of a warp drift onto different code
// paths and each one then pays its own chain of HBM latencies alone).  Lanes share the warp's scratch
// slice; identical stores to identical addresses are benign; side effects on global state are lane 0's.
// Residency: the per-read pipeline is ~0.5 MB of SASS and every warp sits in a different part of it, so beyond
// two warps per SM sub-partition the instruction caches thrash and throughput stops scaling (profiles/r01_icache_*).
#ifndef TALC_MIN_BLOCKS
#define TALC_MIN_BLOCKS 2
#endif
__global__ void __launch_bounds__(128, TALC_MIN_BLOCKS) correct_kernel(CorrectArgs A) {
  // One copy of the per-read state per warp, in shared memory: with 32 lanes holding identical state, keeping
  // it in (per-lane) local memory multiplies its cache footprint by 32 and the L1 thrashes.
  __shared__ Corrector cxs[TALC_WARPS_PER_BLOCK];
  __shared__ Counters mines[TALC_WARPS_PER_BLOCK];
  const u32 lane = threadIdx.x & 31;
  const u32 wib = (threadIdx.x >> 5) % TALC_WARPS_PER_BLOCK;
  Corrector& cx = cxs[wib];
  Counters& mine = mines[wib];
  const u64 gwarp = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  u8* myArena = A.arenas + gwarp * (u64)A.arenaBytes;
  for (;;) {
    u32 qi = 0;
    if (lane == 0) qi = atomicAdd(A.workCounter, 1u);
    qi = __shfl_sync(0xffffffffu, qi, 0);
    if (qi >= A.nOrder) break;
    const u32 r = A.order[qi];
    __syncwarp();
    cx.T = A.tv;
    cx.CR = A.cright;
    cx.CL = A.cleft;
    cx.P = A.P;
    cx.tabs = A.tabs;
    for (int i = 0; i < kNumCounters; ++i) ((u64*)&mine)[i] = 0;
    cx.ctr = &mine;
    ReadJob job;
    job.rd.s = A.bases + A.offs[r];
    job.rd.len = (u32)(A.offs[r + 1] - A.offs[r]);
    job.cov = A.cov + A.kmerOff[r];
    job.arena = myArena;
    job.arena_bytes = A.arenaBytes;
    job.wide = A.wide != 0;
    __syncwarp();
    const long long t0 = clock64();
    u8 st = cx.run_mono(job);
    __syncwarp();
    if (st == kReadOverflow && A.lastTier) {
      st = kReadResource;
      if (lane == 0) mine.reads_overflow += 1;
    }
    if (A.readKcycles && lane == 0) A.readKcycles[r] = (u32)((clock64() - t0) >> 10);
    if (A.readStats && lane == 0 && st != kReadOverflow) {
      // outputBasicReadStats (Read.cpp:418-433) reads m_InKmersPositions as correct2 / defineStructure2 left them
      u32 span = 0, nr = 0;
      if (st == kReadOk || st == kReadNoStructure || st == kReadResource) {
        nr = cx.nregs;
        for (u32 i = 0; i < nr; ++i) span += cx.regs[i].end - cx.regs[i].start + 1;
      }
      A.readStats[2 * r] = span;
      A.readStats[2 * r + 1] = nr;
    }
    if (st == kReadOverflow) {
      if (lane == 0) {
        A.status[r] = st;
        const u32 slot = atomicAdd(A.nOverflow, 1u);
        A.overflowList[slot] = r;
      }
    } else {
      const u32 olen = (st == kReadOk) ? cx.corrected_length() : job.rd.len;
      unsigned long long pos = 0;
      if (lane == 0) pos = atomicAdd(A.outCursor, (unsigned long long)olen);
      pos = __shfl_sync(0xffffffffu, pos, 0);
      if (pos + olen <= A.outCap) {
        u8* dst = A.outArena + pos;
        if (st == kReadOk) cx.emit(dst, lane, 32);
        else
          for (u32 i = lane; i < job.rd.len; i += 32) dst[i] = code_char(job.rd.code(i));
      } else if (lane == 0) {
        atomicExch(A.outFull, 1u);
      }
      if (lane == 0) {
        A.outPos[r] = pos;
        A.outLen[r] = olen;
        A.status[r] = st;
        mine.cells_nw += cx.dps.cells_nw;
        mine.cells_lcs += cx.dps.cells_lcs;
        mine.cells_ovl += cx.dps.cells_ovl;
        mine.cells_xdrop += cx.dps.cells_xdrop;
        mine.bases_out += olen;
        if (st == kReadOk) mine.reads_ok += 1;
        for (int i = 0; i < kNumCounters; ++i) {
          const u64 v = ((const u64*)&mine)[i];
          if (v) atomicAdd(A.counters + i, (unsigned long long)v);
        }
      }
    }
    __syncwarp();
  }
}

// ---- the same per-read program, suspendable: read contexts live in HBM, a round of control_kernel runs every ready
// context until its read is done (the context then takes the next read of the queue) or until it yields a long walk
// to walk_kernel (walk.cuh); walk_kernel advances the frontiers and hands the contexts back.  Rounds alternate until
// every read of the batch is done (host loop in run_split_rounds).
struct RoundArgs {
  CorrectArgs A;
  ReadCtx* ctxs;
  const u32* readyList;
  const u32* nReady;
  u32* walkList;
  u32* nWalk;
  u32* taskCursor;
  u32* finished;  // reads of this pass that are done (corrected, failed, or deferred to the next tier)
};

__global__ void __launch_bounds__(128, TALC_MIN_BLOCKS) control_kernel(RoundArgs R) {
  __shared__ Corrector cxs[TALC_WARPS_PER_BLOCK];
  __shared__ Counters mines[TALC_WARPS_PER_BLOCK];
  const CorrectArgs& A = R.A;
  const u32 lane = threadIdx.x & 31;
  const u32 wib = (threadIdx.x >> 5) % TALC_WARPS_PER_BLOCK;
  Corrector& cx = cxs[wib];
  Counters& mine = mines[wib];
  const u32 nReady = *R.nReady;
  for (;;) {
    u32 qi = 0;
    if (lane == 0) qi = atomicAdd(R.taskCursor, 1u);
    qi = __shfl_sync(0xffffffffu, qi, 0);
    if (qi >= nReady) break;
    const u32 id = R.readyList[qi];
    ReadCtx* rc = R.ctxs + id;
    u8* const myArena = A.arenas + (u64)id * (u64)A.arenaBytes;
    __syncwarp();
    u32 r = rc->read;
    u8 st = kReadYield;
    bool have = false;
    if (r != kCtxFree) {  // resume a suspended read from its context
      {
        const u32* src = (const u32*)&rc->cx;
        u32* dst = (u32*)&cx;
        for (u32 i = lane; i < sizeof(Corrector) / 4; i += 32) dst[i] = src[i];
        const u32* s2 = (const u32*)&rc->ctr;
        u32* d2 = (u32*)&mine;
        for (u32 i = lane; i < sizeof(Counters) / 4; i += 32) d2[i] = s2[i];
      }
      __syncwarp();
      cx.ctr = &mine;
      cx.walk_done(cx.wq.step);
      cx.mark_resumed();
      __syncwarp();
      st = cx.resume();
      __syncwarp();
      have = true;
    }
    for (;;) {
      if (have) {
        if (st == kReadYield) {  // suspend: context back to HBM, frontier to the walk kernel
          __syncwarp();
          {
            const u32* src = (const u32*)&cx;
            u32* dst = (u32*)&rc->cx;
            for (u32 i = lane; i < sizeof(Corrector) / 4; i += 32) dst[i] = src[i];
            const u32* s2 = (const u32*)&mine;
            u32* d2 = (u32*)&rc->ctr;
            for (u32 i = lane; i < sizeof(Counters) / 4; i += 32) d2[i] = s2[i];
          }
          if (lane == 0) {
            rc->read = r;
            const u32 pos = atomicAdd(R.nWalk, 1u);
            R.walkList[pos] = id;
          }
          __syncwarp();
          break;
        }
        // ---- the read is done: same epilogue as correct_kernel
        if (st == kReadOverflow && A.lastTier) {
          st = kReadResource;
          if (lane == 0) mine.reads_overflow += 1;
        }
        if (A.readStats && lane == 0 && st != kReadOverflow) {
          u32 span = 0, nr = 0;
          if (st == kReadOk || st == kReadNoStructure || st == kReadResource) {
            nr = cx.nregs;
            for (u32 i = 0; i < nr; ++i) span += cx.regs[i].end - cx.regs[i].start + 1;
          }
          A.readStats[2 * r] = span;
          A.readStats[2 * r + 1] = nr;
        }
        if (st == kReadOverflow) {
          if (lane == 0) {
            A.status[r] = st;
            const u32 slot = atomicAdd(A.nOverflow, 1u);
            A.overflowList[slot] = r;
          }
        } else {
          const u32 rlen = (u32)(A.offs[r + 1] - A.offs[r]);
          const u32 olen = (st == kReadOk) ? cx.corrected_length() : rlen;
          unsigned long long pos = 0;
          if (lane == 0) pos = atomicAdd(A.outCursor, (unsigned long long)olen);
          pos = __shfl_sync(0xffffffffu, pos, 0);
          if (pos + olen <= A.outCap) {
            u8* dst = A.outArena + pos;
            if (st == kReadOk) cx.emit(dst, lane, 32);
            else {
              const u8* src = A.bases + A.offs[r];
              for (u32 i = lane; i < rlen; i += 32) dst[i] = code_char(base_code(src[i]));
            }
          } else if (lane == 0) {
            atomicExch(A.outFull, 1u);
          }
          if (lane == 0) {
            A.outPos[r] = pos;
            A.outLen[r] = olen;
            A.status[r] = st;
            mine.cells_nw += cx.dps.cells_nw;
            mine.cells_lcs += cx.dps.cells_lcs;
            mine.cells_ovl += cx.dps.cells_ovl;
            mine.cells_xdrop += cx.dps.cells_xdrop;
            mine.bases_out += olen;
            if (st == kReadOk) mine.reads_ok += 1;
            for (int i = 0; i < kNumCounters; ++i) {
              const u64 v = ((const u64*)&mine)[i];
              if (v) atomicAdd(A.counters + i, (unsigned long long)v);
            }
          }
        }
        if (lane == 0) atomicAdd(R.finished, 1u);
        __syncwarp();
      }
      // ---- this context takes the next read of the queue (most expensive first)
      u32 wi = 0;
      if (lane == 0) wi = atomicAdd(A.workCounter, 1u);
      wi = __shfl_sync(0xffffffffu, wi, 0);
      if (wi >= A.nOrder) {
        if (lane == 0) rc->read = kCtxFree;
        __syncwarp();
        break;
      }
      r = A.order[wi];
      __syncwarp();
      cx.T = A.tv;
      cx.CR = A.cright;
      cx.CL = A.cleft;
      cx.P = A.P;
      cx.tabs = A.tabs;
      cx.splitWalk = 1;
      cx.pauseBudget = A.pauseCycles;
      cx.inlineInner = A.inlineInner;
      cx.inlineBorder = A.inlineBorder;
      for (int i = 0; i < kNumCounters; ++i) ((u64*)&mine)[i] = 0;
      cx.ctr = &mine;
      ReadJob job;
      job.rd.s = A.bases + A.offs[r];
      job.rd.len = (u32)(A.offs[r + 1] - A.offs[r]);
      job.cov = A.cov + A.kmerOff[r];
      job.arena = myArena;
      job.arena_bytes = A.arenaBytes;
      job.wide = A.wide != 0;
      __syncwarp();
      st = cx.start(job);
      __syncwarp();
      have = true;
    }
  }
}
__global__ void ctx_init_kernel(ReadCtx* ctxs, u32 nCtx, u32* readyList, u32* nReady) {
  const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nCtx) {
    ctxs[i].read = kCtxFree;
    readyList[i] = i;
  }
  if (i == 0) *nReady = nCtx;
}

// Dna5 conversion followed by SeqAn's reverseComplement, one base: ACGT in either case -> complement, anything else -> N
__device__ __forceinline__ u8 dna5_complement(u8 c) {
  switch (c) {
    case 'A': case 'a': return 'T';
    case 'C': case 'c': return 'G';
    case 'G': case 'g': return 'C';
    case 'T': case 't': return 'A';
    default: return 'N';
  }
}

// --reverse (main.cpp:253): every read reverse-complemented before anything else; one warp per read, same offsets
__global__ void revcomp_reads_kernel(const u8* __restrict__ in, const u64* __restrict__ offs, u32 n, u8* __restrict__ out) {
  const u32 lane = threadIdx.x & 31;
  const u32 warpsPerBlock = blockDim.x >> 5;
  for (u32 r = blockIdx.x * warpsPerBlock + (threadIdx.x >> 5); r < n; r += gridDim.x * warpsPerBlock) {
    const u64 off = offs[r];
    const u64 L = offs[r + 1] - off;
    const u8* src = in + off + L - 1;
    u8* dst = out + off;
    for (u64 i = lane; i < L; i += 32) dst[i] = dna5_complement(src[-(i64)i]);
  }
}

// corrected reads from allocation order into input order; one warp per read.  reverse (uniform per launch): a read
// that was corrected goes back to the input's strand (main.cpp:285-286); every other read leaves as its reverse-
// complemented input (Q24)
__global__ void gather_kernel(const u8* __restrict__ arena, const u64* __restrict__ pos, const u32* __restrict__ len,
                              const u64* __restrict__ outOff, u32 n, u8* __restrict__ out, const u8* __restrict__ status,
                              u32 reverse) {
  const u32 lane = threadIdx.x & 31;
  const u32 warpsPerBlock = blockDim.x >> 5;
  for (u32 r = blockIdx.x * warpsPerBlock + (threadIdx.x >> 5); r < n; r += gridDim.x * warpsPerBlock) {
    const u8* src = arena + pos[r];
    u8* dst = out + outOff[r];
    const u32 L = len[r];
    if (reverse && status[r] == TALC_READ_OK)
      for (u32 i = lane; i < L; i += 32) dst[i] = dna5_complement(src[L - 1 - i]);
    else
      for (u32 i = lane; i < L; i += 32) dst[i] = src[i];
  }
}
__global__ void len_to_u64_kernel(const u32* len, u32 n, u64* out) {
  const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = len[i];
}

__global__ void model_tabs_kernel(double alpha, u32 n, double* lower, double* upper, double* sq) {
  const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  lower[i] = model_lower_bound(i, alpha);
  upper[i] = model_upper_bound(i, alpha);
  sq[i] = sqrt((double)i);
}

// =====================================================================================
// random-sector peak (SURVEY 8d): the roofline of the hash probes is not the streaming HBM bandwidth but what the
// memory system delivers for uniformly random 32-byte sectors.  mode 0: `ILP` independent 256-bit loads in flight
// per thread (the coverage kernel's pattern); mode 1: one dependent chain per thread -- the next address is a hash
// of the loaded sector (the walk's pattern: the successor bucket decides the next k-mer).
// =====================================================================================
template <int ILP>
__global__ void __launch_bounds__(256) random_sector_kernel(const ulonglong4* __restrict__ buf, u64 sectorMask, u32 iters, int dependent,
                                                            unsigned long long* sink) {
  u64 x[ILP];
#pragma unroll
  for (int j = 0; j < ILP; ++j) x[j] = hash_kmer(((u64)blockIdx.x * blockDim.x + threadIdx.x) * ILP + j + 1);
  u64 acc = 0;
  for (u32 it = 0; it < iters; ++it) {
    u64 v[ILP];
#pragma unroll
    for (int j = 0; j < ILP; ++j) {
      u64 a0, a1, a2, a3;
      asm volatile("ld.global.nc.v4.u64 {%0,%1,%2,%3}, [%4];" : "=l"(a0), "=l"(a1), "=l"(a2), "=l"(a3) : "l"(buf + (x[j] & sectorMask)));
      v[j] = a0 ^ a1 ^ a2 ^ a3;
    }
#pragma unroll
    for (int j = 0; j < ILP; ++j) {
      acc += v[j];
      x[j] = x[j] * 0x9E3779B97F4A7C15ull + (dependent ? v[j] : 0ull) + 0x632BE59BD9B4E019ull;
      x[j] ^= x[j] >> 29;
    }
  }
  if (acc == 0x1234567ull) *sink = acc;
}

// =====================================================================================
// device self-tests of the primitives
// =====================================================================================
__global__ void test_align_kernel(int op, const u8* a, const u64* aoff, const u8* b, const u64* boff, u32 n, int aux,
                                  int aux2, u32 K, u8* arenas, u32 arenaBytes, i32* result) {
  // one warp per pair, all lanes with identical data (the scoring routines are warp-cooperative)
  const u32 i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const u32 lane = threadIdx.x & 31;
  if (i >= n) return;
  Arena ar;
  ar.init(arenas + (u64)i * arenaBytes, arenaBytes);
  // the sequences reach the scoring routines packed, as in the pipeline: 4 bits per base in general, and the
  // second string also as a 2-bit trail when it holds no N
  const u32 an = (u32)(aoff[i + 1] - aoff[i]), bn = (u32)(boff[i + 1] - boff[i]);
  u64* pa = (u64*)ar.alloc(((an + 15) / 16 + 2) * 8);
  u64* pb = (u64*)ar.alloc(((bn + 15) / 16 + 2) * 8);
  u64* packed = (u64*)ar.alloc(((bn + 31) / 32 + 2) * 8);
  if (!pa || !pb || !packed) return;
  SeqView va = pack_ascii4(a + aoff[i], an, pa);
  SeqView vb = pack_ascii4(b + boff[i], bn, pb);
  bool pure = true;
  for (u32 j = 0; j < vb.len && pure; ++j) pure = vb.code(j) < 4;
  if (pure) {
    for (u32 j = 0; j < (vb.len + 31) / 32 + 2; ++j) packed[j] = 0;
    for (u32 j = 0; j < vb.len; ++j) path_set(packed, j, vb.code(j));
    vb = view_of_path(packed, vb.len);
  }
  __syncwarp();
  i32 r0 = 0, r1 = 0, r2 = 0, r3 = 0;
  if (op == 0) r0 = -nw_distance(va, va.len, vb, vb.len, ar, nullptr);
  else if (op == 1) r0 = lcs_length(va, va.len, vb, vb.len, ar, nullptr);
  else if (op == 2) r0 = overlap_score(va, va.len, vb, vb.len, ar, nullptr);
  else if (op == 5) {  // fused distance + LCS
    int l = 0;
    r0 = -nw_lcs_fused(va, va.len, vb, vb.len, ar, nullptr, l, 3);
    r1 = l;
  } else if (op == 4) {  // raw X-drop: a = query segment, b = database segment, aux = score drop-off
    DpStats ds;
    ds.cells_xdrop = 0;
    u32 er = 0, ec = 0;
    i32 es = 0;
    xdrop_extend(va, 0, va.len, vb, 0, vb.len, aux, er, ec, es, ar, true, &ds);
    r0 = (i32)er;
    r1 = (i32)ec;
    r2 = (i32)ds.cells_xdrop;
    r3 = es;
  } else {
    const SeedExt e = seed_and_extension(va, vb, aux, aux2 != 0, K, ar, true, nullptr);
    r0 = (i32)e.ref_ext;
    r1 = (i32)e.cand_ext;
    r2 = e.score;
    r3 = e.stop ? 1 : 0;
  }
  if (ar.overflow) r0 = INT32_MIN;
  if (lane == 0) {
    if (op >= 3) {
      result[4 * i + 0] = r0;
      result[4 * i + 1] = r1;
      result[4 * i + 2] = r2;
      result[4 * i + 3] = r3;
    } else
      result[i] = r0;
  }
}
__global__ void test_sort_kernel(const i64* keys, u32 n, u32* perm, void* scratchKeys) {
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  SortKey* sk = (SortKey*)scratchKeys;
  for (u32 i = 0; i < n; ++i) { sk[i].key = keys[i]; sk[i].idx = i; }
  std_sort_keys(sk, n);
  for (u32 i = 0; i < n; ++i) perm[i] = sk[i].idx;
}

// =====================================================================================
// host side
// =====================================================================================
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
};

struct talc_ctx {
  talc_params params;
  Params P;
  int device = 0;
  int sms = 0;
  std::string err;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev[8];
  // table
  Slot* slots = nullptr;
  u64 capacity = 0;
  u64 nEntries = 0;
  bool tableOwned = true;
  bool tableReady = false;
  talc_ctx* parent = nullptr;  // a lane (talc_ctx_create_lane): tables and settings are the parent's, scratch and stream its own
  // where the table came from (recorded in the binary cache so that a cache of other inputs is not reused silently)
  u32 provJunctions = 0;
  u64 provDumpSize = 0, provDumpMtime = 0, provJuncSize = 0, provJuncMtime = 0;
  CtxBucket* ctxRight = nullptr;  // successor tables, derived from the k-mer table when it is sealed
  CtxBucket* ctxLeft = nullptr;
  u64 ctxCap = 0;
  // scratch sizing
  u32 tier1Bytes = 1u << 20;    // per warp (= per read in flight)
  u32 tier2Bytes = 64u << 20;
  u32 tier2Warps = 128;
  u32 blocksPerSm = TALC_MIN_BLOCKS;
  u32 splitWalk = 0;       // 1: suspendable reads + walk kernel (rounds), 0: one monolithic correct_kernel launch
  u32 nCtxTier1 = 16384;   // read contexts in flight (each with a tier-1 arena)
  u32 walkStepCap = 48;    // steps a frontier may take per round of the walk kernel (bounds the round's tail)
  u32 pauseCycles = 200000;  // SM cycles (~100 us) a read may run per round of the control kernel
  u32 inlineInner = 6, inlineBorder = 6;
  u32 reverse = 0;  // talc_ctx_set_reverse: the long reads are corrected on the opposite strand (rcBases)
  u64 lastRounds = 0;
  double* modelTabs = nullptr;  // 3 x kModelTabN doubles
  // cached device buffers
  DevBuf bases, offs, kmerOff, nk, cov, order, sortKey, sortKeyOut, sortVal, cubTmp, arenas, outArena, outPos, outLen,
      outLen64, status, outOffs, out, misc, overflowList, readCtxs, roundLists, rcBases;
};

static const u32 kModelTabN = 16384;
static void free_ctx_tables(talc_ctx* c) {
  if (c->ctxRight) cudaFree(c->ctxRight);
  if (c->ctxLeft) cudaFree(c->ctxLeft);
  c->ctxRight = c->ctxLeft = nullptr;
  c->ctxCap = 0;
}
static thread_local std::string g_createError;

#define CUDA_TRY(ctx, call)                                                                             \
  do {                                                                                                  \
    cudaError_t e__ = (call);                                                                           \
    if (e__ != cudaSuccess) {                                                                           \
      (ctx)->err = std::string(#call) + ": " + cudaGetErrorString(e__);                                 \
      return TALC_ERR_CUDA;                                                                             \
    }                                                                                                   \
  } while (0)

static Params to_device_params(const talc_params& q) {
  Params p;
  p.K = q.K;
  p.min_count = q.min_count;
  p.window = q.window_size;
  p.max_branches = q.max_nb_branches;
  p.alpha = q.alpha;
  p.sr_error = q.sr_error_rate;
  p.min_inner = q.min_inner_score;
  p.min_border = q.min_border_score;
  p.cycle_mode = q.cycle_mode;
  p.q11_zero = q.q11_zero_init;
  return p;
}

extern "C" {

void talc_params_default(talc_params* p, uint32_t K) {
  p->K = K;
  p->min_count = 2;
  p->window_size = 9;
  p->max_nb_branches = 7;
  p->alpha = 2.57;
  p->sr_error_rate = 0.025;
  p->min_inner_score = 0.7;
  p->min_border_score = 0.7;
  p->cycle_mode = 0;
  p->q11_zero_init = 1;
}

#ifndef TALC_SOURCE_HASH
#define TALC_SOURCE_HASH "unknown"
#endif
const char* talc_build_source_hash(void) { return TALC_SOURCE_HASH; }

const char* talc_last_error(talc_ctx* ctx) { return ctx ? ctx->err.c_str() : g_createError.c_str(); }

int talc_ctx_create(const talc_params* p, int cuda_device, talc_ctx** out) {
  if (!p || !out) return TALC_ERR_ARG;
  *out = nullptr;
  if (p->K < 2 || p->K > 31 || p->min_count < 1 || p->max_nb_branches < 1) {
    g_createError = "invalid parameters (K must be in [2,31])";
    return TALC_ERR_ARG;
  }
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    g_createError = std::string("no CUDA device: this library has no CPU path (") + cudaGetErrorString(e) + ")";
    return TALC_ERR_CUDA;
  }
  if (cuda_device < 0 || cuda_device >= ndev) {
    g_createError = "cuda_device out of range";
    return TALC_ERR_ARG;
  }
  if ((e = cudaSetDevice(cuda_device)) != cudaSuccess) {
    g_createError = std::string("cudaSetDevice: ") + cudaGetErrorString(e);
    return TALC_ERR_CUDA;
  }
  talc_ctx* c = new talc_ctx;
  c->params = *p;
  c->P = to_device_params(*p);
  c->device = cuda_device;
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, cuda_device);
  c->sms = prop.multiProcessorCount;
  if ((e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking)) != cudaSuccess) {
    g_createError = std::string("cudaStreamCreate: ") + cudaGetErrorString(e);
    delete c;
    return TALC_ERR_CUDA;
  }
  for (int i = 0; i < 8; ++i) cudaEventCreate(&c->ev[i]);
  if (cudaMalloc((void**)&c->modelTabs, (size_t)3 * kModelTabN * sizeof(double)) != cudaSuccess) {
    g_createError = "cudaMalloc(model tables) failed";
    delete c;
    return TALC_ERR_CUDA;
  }
  model_tabs_kernel<<<(kModelTabN + 255) / 256, 256, 0, c->stream>>>(p->alpha, kModelTabN, c->modelTabs, c->modelTabs + kModelTabN,
                                                                  c->modelTabs + 2 * kModelTabN);
  cudaStreamSynchronize(c->stream);
  if (const char* e2 = getenv("TALC_BLOCKS_PER_SM")) c->blocksPerSm = (u32)std::max(1, atoi(e2));
  if (const char* e2 = getenv("TALC_SPLIT")) c->splitWalk = atoi(e2) != 0;
  if (const char* e2 = getenv("TALC_CTX")) c->nCtxTier1 = (u32)std::max(4, atoi(e2));
  if (const char* e2 = getenv("TALC_WALK_CAP")) c->walkStepCap = (u32)std::max(1, atoi(e2));
  if (const char* e2 = getenv("TALC_PAUSE_CYCLES")) c->pauseCycles = (u32)std::max(0, atoi(e2));
  if (const char* e2 = getenv("TALC_INLINE_INNER")) c->inlineInner = (u32)std::max(0, atoi(e2));
  if (const char* e2 = getenv("TALC_INLINE_BORDER")) c->inlineBorder = (u32)std::max(0, atoi(e2));
  *out = c;
  return TALC_OK;
}

void talc_ctx_destroy(talc_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  if (c->parent) {  // a lane borrows its tables
    c->slots = nullptr;
    c->ctxRight = c->ctxLeft = nullptr;
  }
  if (c->slots && c->tableOwned) cudaFree(c->slots);
  free_ctx_tables(c);
  if (c->modelTabs) cudaFree(c->modelTabs);
  DevBuf* bufs[] = {&c->bases, &c->offs, &c->kmerOff, &c->nk, &c->cov, &c->order, &c->sortKey, &c->sortKeyOut, &c->sortVal,
                    &c->cubTmp, &c->arenas, &c->outArena, &c->outPos, &c->outLen, &c->outLen64, &c->status, &c->outOffs,
                    &c->out, &c->misc, &c->overflowList, &c->readCtxs, &c->roundLists, &c->rcBases};
  for (DevBuf* b : bufs) b->release();
  for (int i = 0; i < 8; ++i) cudaEventDestroy(c->ev[i]);
  cudaStreamDestroy(c->stream);
  delete c;
}

// A lane: a second context of the same device that borrows the tables and follows the settings of `parent` but has its
// own stream and scratch.  Batches corrected through a context and its lane from two host threads overlap on the
// device: the blocks of one batch start on the SMs that the last, longest reads of the other no longer fill (the
// per-read program is one warp per read, so every batch ends with a tail of a few long reads).  talc_stream uses one
// internally.  Destroy the lane (talc_ctx_destroy) before its parent.
static void lane_follow(talc_ctx* sh) {
  const talc_ctx* c = sh->parent;
  sh->params = c->params;
  sh->P = c->P;
  sh->slots = c->slots;
  sh->capacity = c->capacity;
  sh->nEntries = c->nEntries;
  sh->tableOwned = false;
  sh->tableReady = c->tableReady;
  sh->ctxRight = c->ctxRight;
  sh->ctxLeft = c->ctxLeft;
  sh->ctxCap = c->ctxCap;
  sh->tier1Bytes = c->tier1Bytes;
  sh->tier2Bytes = c->tier2Bytes;
  sh->tier2Warps = c->tier2Warps;
  sh->blocksPerSm = c->blocksPerSm;
  sh->splitWalk = c->splitWalk;
  sh->nCtxTier1 = c->nCtxTier1;
  sh->walkStepCap = c->walkStepCap;
  sh->pauseCycles = c->pauseCycles;
  sh->inlineInner = c->inlineInner;
  sh->inlineBorder = c->inlineBorder;
  sh->reverse = c->reverse;
}
int talc_ctx_create_lane(talc_ctx* parent, talc_ctx** out) {
  if (!parent || !out || parent->parent) return TALC_ERR_ARG;
  const int rc = talc_ctx_create(&parent->params, parent->device, out);
  if (rc != TALC_OK) { parent->err = std::string("talc_ctx_create_lane: ") + g_createError; return rc; }
  (*out)->parent = parent;
  lane_follow(*out);
  return TALC_OK;
}

int talc_ctx_set_scratch(talc_ctx* c, uint32_t tier1_bytes, uint32_t tier2_bytes, uint32_t tier2_threads) {
  if (!c) return TALC_ERR_ARG;
  if (tier1_bytes) c->tier1Bytes = (tier1_bytes + 255u) & ~255u;
  if (tier2_bytes) c->tier2Bytes = (tier2_bytes + 255u) & ~255u;
  if (tier2_threads) c->tier2Warps = (tier2_threads + 3u) & ~3u;
  return TALC_OK;
}

// execution shape of the correction (0 keeps a value): split_walk 1 = suspendable reads + walk kernel, 2 = one
// monolithic kernel (the round-1 shape, kept for A/B measurements); read_contexts in flight; steps per walk round
int talc_ctx_set_exec(talc_ctx* c, uint32_t split_walk, uint32_t read_contexts, uint32_t walk_step_cap) {
  if (!c) return TALC_ERR_ARG;
  if (split_walk) c->splitWalk = split_walk == 1 ? 1u : 0u;
  if (read_contexts) c->nCtxTier1 = read_contexts < 4 ? 4 : read_contexts;
  if (walk_step_cap) c->walkStepCap = walk_step_cap;
  return TALC_OK;
}

// --reverse (main.cpp:253,285-286).  A lane follows its parent; the stream's lanes read it at the start of each batch.
int talc_ctx_set_reverse(talc_ctx* c, int reverse) {
  if (!c) return TALC_ERR_ARG;
  if (c->parent) { c->err = "a lane follows the strand setting of the context it was made from"; return TALC_ERR_ARG; }
  c->reverse = reverse != 0;
  return TALC_OK;
}

// ---------------------------------------------------------------------------------- table
int talc_table_alloc(talc_ctx* c, uint64_t capacity_slots) {
  if (!c || capacity_slots < 2 || (capacity_slots & (capacity_slots - 1))) return TALC_ERR_ARG;
  if (c->parent) { c->err = "a lane has no table of its own: load it into the context the lane was made from"; return TALC_ERR_ARG; }
  CUDA_TRY(c, cudaSetDevice(c->device));
  if (c->slots && c->tableOwned) cudaFree(c->slots);
  free_ctx_tables(c);
  c->slots = nullptr;
  c->tableReady = false;
  CUDA_TRY(c, cudaMalloc((void**)&c->slots, capacity_slots * sizeof(Slot)));
  c->capacity = capacity_slots;
  c->tableOwned = true;
  const int blocks = c->sms * 8;
  table_fill_empty_kernel<<<blocks, 256, 0, c->stream>>>(c->slots, c->capacity);
  CUDA_TRY(c, cudaGetLastError());
  CUDA_TRY(c, cudaStreamSynchronize(c->stream));
  return TALC_OK;
}
int talc_table_device_ptr(talc_ctx* c, void** p) {
  if (!c || !p || !c->slots) return TALC_ERR_ARG;
  *p = c->slots;
  return TALC_OK;
}
// Recounts the occupied slots on the device (the caller's n_entries is a claim, not a fact), refuses a table without
// room to end a probe (load > 0.5), sizes the successor tables from the recount and derives them.
static int build_ctx_tables(talc_ctx* c) {
  CUDA_TRY(c, cudaSetDevice(c->device));
  free_ctx_tables(c);
  const int blocks = c->sms * 8;
  unsigned long long* dN = nullptr;
  CUDA_TRY(c, cudaMalloc((void**)&dN, 16));
  CUDA_TRY(c, cudaMemsetAsync(dN, 0, 16, c->stream));
  table_count_kernel<<<blocks, 256, 0, c->stream>>>(c->slots, c->capacity, dN);
  CUDA_TRY(c, cudaGetLastError());
  unsigned long long hN[2] = {0, 0};
  CUDA_TRY(c, cudaMemcpyAsync(hN, dN, 8, cudaMemcpyDeviceToHost, c->stream));
  CUDA_TRY(c, cudaStreamSynchronize(c->stream));
  if (2 * hN[0] > c->capacity) {
    cudaFree(dN);
    c->err = "k-mer table is more than half full (corrupt cache or wrong capacity): refused";
    return TALC_ERR_ARG;
  }
  c->nEntries = hN[0];
  u64 cap = 4;
  while (cap < 3 * c->nEntries + 4) cap <<= 1;  // load <= 1/3: a look-up rarely leaves its home pair of buckets
  CUDA_TRY(c, cudaMalloc((void**)&c->ctxRight, cap * sizeof(CtxBucket)));
  CUDA_TRY(c, cudaMalloc((void**)&c->ctxLeft, cap * sizeof(CtxBucket)));
  c->ctxCap = cap;
  ctx_fill_empty_kernel<<<blocks, 256, 0, c->stream>>>(c->ctxRight, cap);
  ctx_fill_empty_kernel<<<blocks, 256, 0, c->stream>>>(c->ctxLeft, cap);
  ctx_build_kernel<<<blocks, 256, 0, c->stream>>>(c->slots, c->capacity, c->ctxRight, c->ctxLeft, cap - 1, c->P.K, (u32*)(dN + 1));
  CUDA_TRY(c, cudaGetLastError());
  CUDA_TRY(c, cudaMemcpyAsync(hN + 1, dN + 1, 8, cudaMemcpyDeviceToHost, c->stream));
  CUDA_TRY(c, cudaStreamSynchronize(c->stream));
  cudaFree(dN);
  if (hN[1]) { c->err = "successor tables overflowed"; return TALC_ERR_ARG; }
  return TALC_OK;
}
// n_entries is informational: the occupied slots are recounted on the device
int talc_table_seal(talc_ctx* c, uint64_t n_entries) {
  if (!c || !c->slots) return TALC_ERR_ARG;
  (void)n_entries;
  const int rc = build_ctx_tables(c);
  if (rc) return rc;
  c->tableReady = true;
  return TALC_OK;
}
int talc_table_info(talc_ctx* c, uint64_t* cap, uint64_t* bytes, uint64_t* n) {
  if (!c) return TALC_ERR_ARG;
  if (cap) *cap = c->capacity;
  if (bytes) *bytes = c->capacity * sizeof(Slot);
  if (n) *n = c->nEntries;
  return c->tableReady ? TALC_OK : TALC_ERR_NO_TABLE;
}

extern "C" int talc_table_export_device(talc_ctx* c, void* dst, uint64_t bytes) {
  if (!c || !dst || !c->tableReady || bytes < c->capacity * sizeof(Slot)) return TALC_ERR_ARG;
  CUDA_TRY(c, cudaSetDevice(c->device));
  CUDA_TRY(c, cudaMemcpyAsync(dst, c->slots, c->capacity * sizeof(Slot), cudaMemcpyDeviceToDevice, c->stream));
  CUDA_TRY(c, cudaStreamSynchronize(c->stream));
  return TALC_OK;
}
extern "C" int talc_table_import_device(talc_ctx* c, const void* src, uint64_t capacity, uint64_t n_entries) {
  if (!c || !src) return TALC_ERR_ARG;
  int rc = talc_table_alloc(c, capacity);
  if (rc) return rc;
  CUDA_TRY(c, cudaMemcpyAsync(c->slots, src, capacity * sizeof(Slot), cudaMemcpyDeviceToDevice, c->stream));
  CUDA_TRY(c, cudaStreamSynchronize(c->stream));
  return talc_table_seal(c, n_entries);
}
extern "C" int talc_table_copy(talc_ctx* dst, talc_ctx* src) {
  if (!dst || !src || !src->tableReady) return TALC_ERR_ARG;
  int rc = talc_table_alloc(dst, src->capacity);
  if (rc) return rc;
  CUDA_TRY(dst, cudaMemcpyPeer(dst->slots, dst->device, src->slots, src->device, src->capacity * sizeof(Slot)));
  dst->provJunctions = src->provJunctions;
  dst->provDumpSize = src->provDumpSize; dst->provDumpMtime = src->provDumpMtime;
  dst->provJuncSize = src->provJuncSize; dst->provJuncMtime = src->provJuncMtime;
  return talc_table_seal(dst, src->nEntries);
}

// ---- binary table cache (include/talc_b200.h): header + raw slot array, streamed in 64 MiB pieces
struct TableCacheHeader {
  char magic[8];  // "TALCTBL2"
  u32 K, min_count;
  u64 capacity, entries;
  u32 junctions, pad;                                // junction colours baked in?
  u64 dumpSize, dumpMtime, juncSize, juncMtime;      // identity of the text inputs (0 = built from packed arrays)
};
static void file_identity(const char* path, u64& size, u64& mtime) {
  struct stat st;
  size = mtime = 0;
  if (path && stat(path, &st) == 0) { size = (u64)st.st_size; mtime = (u64)st.st_mtime; }
}
extern "C" int talc_table_save(talc_ctx* c, const char* path) {
  if (!c || !path || !c->tableReady) return TALC_ERR_ARG;
  CUDA_TRY(c, cudaSetDevice(c->device));
  FILE* f = fopen(path, "wb");
  if (!f) { c->err = std::string("cannot write ") + path; return TALC_ERR_IO; }
  TableCacheHeader h;
  memset(&h, 0, sizeof(h));
  memcpy(h.magic, "TALCTBL2", 8);
  h.K = c->P.K; h.min_count = c->P.min_count; h.capacity = c->capacity; h.entries = c->nEntries;
  h.junctions = c->provJunctions;
  h.dumpSize = c->provDumpSize; h.dumpMtime = c->provDumpMtime; h.juncSize = c->provJuncSize; h.juncMtime = c->provJuncMtime;
  bool ok = fwrite(&h, sizeof(h), 1, f) == 1;
  const size_t total = (size_t)c->capacity * sizeof(Slot), piece = 64u << 20;
  std::vector<char> buf(std::min(total, piece));
  for (size_t o = 0; o < total && ok; o += piece) {
    const size_t nb = std::min(piece, total - o);
    if (cudaMemcpy(buf.data(), (const char*)c->slots + o, nb, cudaMemcpyDeviceToHost) != cudaSuccess) ok = false;
    else ok = fwrite(buf.data(), 1, nb, f) == nb;
  }
  ok = (fclose(f) == 0) && ok;
  if (!ok) { c->err = std::string("error while writing ") + path; return TALC_ERR_IO; }
  return TALC_OK;
}
// check_inputs: the cache must have been made from exactly these text files (size + mtime) and junction setting
static int load_cache(talc_ctx* c, const char* path, bool check_inputs, const char* dump_path, const char* junction_path,
                      uint64_t* n_entries) {
  if (!c || !path) return TALC_ERR_ARG;
  FILE* f = fopen(path, "rb");
  if (!f) { c->err = std::string("cannot read ") + path; return TALC_ERR_IO; }
  TableCacheHeader h;
  struct stat st;
  if (fread(&h, sizeof(h), 1, f) != 1 || memcmp(h.magic, "TALCTBL2", 8) != 0 || h.capacity < 2 ||
      (h.capacity & (h.capacity - 1)) || fstat(fileno(f), &st) != 0 ||
      (u64)st.st_size != sizeof(h) + h.capacity * sizeof(Slot) || 2 * h.entries > h.capacity) {
    fclose(f);
    c->err = std::string(path) + " is not a table cache (or is truncated)";
    return TALC_ERR_IO;
  }
  if (h.K != c->P.K || h.min_count != c->P.min_count) {
    fclose(f);
    c->err = "table cache was built with another k-mer size or MIN_COUNT";
    return TALC_ERR_STALE;
  }
  if (check_inputs) {
    u64 ds, dm, js, jm;
    file_identity(dump_path, ds, dm);
    file_identity(junction_path, js, jm);
    if (h.junctions != (junction_path ? 1u : 0u) || h.dumpSize != ds || h.dumpMtime != dm || h.juncSize != js || h.juncMtime != jm) {
      fclose(f);
      c->err = "table cache was built from other --SRCounts / --junctions inputs";
      return TALC_ERR_STALE;
    }
  }
  int rc = talc_table_alloc(c, h.capacity);
  if (rc) { fclose(f); return rc; }
  const size_t total = (size_t)h.capacity * sizeof(Slot), piece = 64u << 20;
  std::vector<char> buf(std::min(total, piece));
  bool ok = true;
  for (size_t o = 0; o < total && ok; o += piece) {
    const size_t nb = std::min(piece, total - o);
    ok = fread(buf.data(), 1, nb, f) == nb &&
         cudaMemcpy((char*)c->slots + o, buf.data(), nb, cudaMemcpyHostToDevice) == cudaSuccess;
  }
  fclose(f);
  if (!ok) { c->err = std::string("truncated table cache ") + path; return TALC_ERR_IO; }
  c->provJunctions = h.junctions;
  c->provDumpSize = h.dumpSize; c->provDumpMtime = h.dumpMtime; c->provJuncSize = h.juncSize; c->provJuncMtime = h.juncMtime;
  rc = talc_table_seal(c, h.entries);
  if (rc) return rc;
  if (c->nEntries != h.entries) {
    c->tableReady = false;
    c->err = "table cache is corrupt: occupied slots differ from the header";
    return TALC_ERR_IO;
  }
  if (n_entries) *n_entries = c->nEntries;
  return TALC_OK;
}
extern "C" int talc_table_load_cache(talc_ctx* c, const char* path, uint64_t* n_entries) {
  return load_cache(c, path, false, nullptr, nullptr, n_entries);
}
extern "C" int talc_table_load_cache_for(talc_ctx* c, const char* path, const char* dump_path, const char* junction_path,
                                         uint64_t* n_entries) {
  if (!dump_path) return TALC_ERR_ARG;
  return load_cache(c, path, true, dump_path, junction_path, n_entries);
}

// common tail of every build: strip the line indices, apply the reduced junction colours + homopolymer resets, check
// the overflow flag at dN[1], derive the successor tables
static int finish_table(talc_ctx* c, unsigned long long* dN, const std::vector<u64>& ckeys, const std::vector<u32>& ccols,
                        uint64_t* n_kept) {
  const int blocks = c->sms * 8;
  const u64 cap = c->capacity;
  table_finalize_kernel<<<blocks, 256, 0, c->stream>>>(c->slots, cap, dN);
  CUDA_TRY(c, cudaGetLastError());
  if (!ckeys.empty()) {
    u64* dCk = nullptr;
    u32* dCc = nullptr;
    CUDA_TRY(c, cudaMalloc((void**)&dCk, ckeys.size() * 8));
    CUDA_TRY(c, cudaMalloc((void**)&dCc, ckeys.size() * 4));
    CUDA_TRY(c, cudaMemcpyAsync(dCk, ckeys.data(), ckeys.size() * 8, cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(c, cudaMemcpyAsync(dCc, ccols.data(), ckeys.size() * 4, cudaMemcpyHostToDevice, c->stream));
    table_colour_kernel<<<blocks, 256, 0, c->stream>>>(c->slots, cap - 1, dCk, dCc, ckeys.size());
    CUDA_TRY(c, cudaGetLastError());
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    cudaFree(dCk);
    cudaFree(dCc);
  }
  unsigned long long hN[2] = {0, 0};
  CUDA_TRY(c, cudaMemcpyAsync(hN, dN, 16, cudaMemcpyDeviceToHost, c->stream));
  CUDA_TRY(c, cudaStreamSynchronize(c->stream));
  if (hN[1]) { c->err = "k-mer table overflowed during the build"; return TALC_ERR_ARG; }
  c->nEntries = hN[0];
  const int rc = build_ctx_tables(c);
  if (rc) return rc;
  c->tableReady = true;
  if (n_kept) *n_kept = c->nEntries;
  return TALC_OK;
}
// entries on the device in dump-line order (kEmptyKey = no entry on that line); nKept of the nArr slots are occupied.
// ckeys / ccols: the junction colours already reduced to one final value per k-mer (host arrays)
static int build_table_device(talc_ctx* c, const u64* dKeys, const u32* dCounts, u64 nArr, u64 nKept, const std::vector<u64>& ckeys,
                              const std::vector<u32>& ccols, uint64_t* n_kept) {
  u64 cap = 2;
  while (cap < 2 * nKept + 2) cap <<= 1;
  int rc = talc_table_alloc(c, cap);
  if (rc) return rc;
  const int blocks = c->sms * 8;
  unsigned long long* dN = nullptr;
  CUDA_TRY(c, cudaMalloc((void**)&dN, 16));
  CUDA_TRY(c, cudaMemsetAsync(dN, 0, 16, c->stream));
  if (nArr) {
    table_insert_kernel<<<blocks, 256, 0, c->stream>>>(c->slots, cap - 1, dKeys, dCounts, nArr, 0, (u32*)(dN + 1));
    CUDA_TRY(c, cudaGetLastError());
  }
  const int rc2 = finish_table(c, dN, ckeys, ccols, n_kept);
  cudaFree(dN);
  return rc2;
}
// the same from host arrays: dump order, already filtered to count >= MIN and valid ACGT k-mers of length K
static int build_table(talc_ctx* c, const std::vector<u64>& keys, const std::vector<u32>& counts,
                       const std::vector<u64>& ckeys, const std::vector<u32>& ccols, uint64_t* n_kept) {
  const u64 n = keys.size();
  u64* dKeys = nullptr;
  u32* dCounts = nullptr;
  CUDA_TRY(c, cudaSetDevice(c->device));
  if (n) {
    CUDA_TRY(c, cudaMalloc((void**)&dKeys, n * 8));
    CUDA_TRY(c, cudaMalloc((void**)&dCounts, n * 4));
    CUDA_TRY(c, cudaMemcpyAsync(dKeys, keys.data(), n * 8, cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(c, cudaMemcpyAsync(dCounts, counts.data(), n * 4, cudaMemcpyHostToDevice, c->stream));
  }
  const int rc = build_table_device(c, dKeys, dCounts, n, n, ckeys, ccols, n_kept);
  if (dKeys) cudaFree(dKeys);
  if (dCounts) cudaFree(dCounts);
  return rc;
}

static u64 revcomp_kmer(u64 k, u32 K) {
  u64 r = 0;
  for (u32 i = 0; i < K; ++i) {
    r = (r << 2) | (3 - (k & 3));
    k >>= 2;
  }
  return r;
}

// reduce the junction list to final colours (sequential semantics of Jellyfish.cpp:278-289) and append the
// four homopolymer resets of decolourRepeatsFromDBG (utils.cpp:658-669)
static void reduce_colours(const talc_params& p, const u64* jkeys, const i64* jcounts, u64 nj, bool use, std::vector<u64>& ck,
                           std::vector<u32>& cc) {
  std::unordered_map<u64, u32> last;
  if (use) {
    last.reserve(nj * 2 + 8);
    for (u64 i = 0; i < nj; ++i) {
      const u32 v = (u32)(int)jcounts[i];
      if (v < kColouredCountThr) {
        last[jkeys[i]] = v;
        last[revcomp_kmer(jkeys[i], p.K)] = v;
      }
    }
  }
  for (u32 b = 0; b < 4; ++b) {
    u64 homo = 0;
    for (u32 i = 0; i < p.K; ++i) homo = (homo << 2) | b;
    last[homo] = 0;
  }
  ck.reserve(last.size());
  cc.reserve(last.size());
  for (auto& kv : last) {
    ck.push_back(kv.first);
    cc.push_back(kv.second);
  }
}

int talc_table_load_packed(talc_ctx* c, const uint64_t* keys, const int64_t* counts, uint64_t n, const uint64_t* jkeys,
                           const int64_t* jcounts, uint64_t nj, int use_junctions, uint64_t* n_kept) {
  if (!c || (n && (!keys || !counts))) return TALC_ERR_ARG;
  std::vector<u64> k;
  std::vector<u32> v;
  k.reserve(n);
  v.reserve(n);
  const u64 kmask = kmer_mask(c->params.K);
  for (u64 i = 0; i < n; ++i) {
    const u32 cnt = (u32)(int)counts[i];  // std::stoi(count) >= gp_MIN_COUNT compares as unsigned (Jellyfish.cpp:260)
    if (cnt >= c->params.min_count && (keys[i] & ~kmask) == 0) {
      k.push_back(keys[i]);
      v.push_back(cnt);
    }
  }
  std::vector<u64> ck;
  std::vector<u32> cc;
  reduce_colours(c->params, jkeys, jcounts, nj, use_junctions != 0, ck, cc);
  c->provJunctions = use_junctions ? 1u : 0u;
  c->provDumpSize = c->provDumpMtime = c->provJuncSize = c->provJuncMtime = 0;
  return build_table(c, k, v, ck, cc, n_kept);
}

// buildCDBG + decolourRepeatsFromDBG (Jellyfish.cpp:236-295, utils.cpp:658-669) with the text parsed on the GPU
// (dump_gpu.cuh): the entries never visit the host.  The junction dump (small) is parsed the same way, then reduced to
// final colours on the host ("last writer wins, forward before reverse complement" is sequential by nature).
int talc_table_load_dump(talc_ctx* c, const char* dump_path, const char* junction_path, uint64_t* n_lines, uint64_t* n_kept) {
  if (!c || !dump_path) return TALC_ERR_ARG;
  CUDA_TRY(c, cudaSetDevice(c->device));
  DeviceDump d;
  std::string err;
  if (!parse_dump_gpu(dump_path, c->params.K, c->params.min_count, true, c->sms, c->stream, d, err)) {
    c->err = err;
    return TALC_ERR_IO;
  }
  if (n_lines) *n_lines = d.tally.lines;
  std::vector<u64> ck;
  std::vector<u32> cc;
  if (junction_path) {
    DeviceDump j;
    if (!parse_dump_gpu(junction_path, c->params.K, 0, false, c->sms, c->stream, j, err)) {
      d.release();
      c->err = err;
      return TALC_ERR_IO;
    }
    std::vector<u64> jk(j.nLines);
    std::vector<u32> jv(j.nLines);
    if (j.nLines) {
      cudaMemcpy(jk.data(), j.keys, j.nLines * 8, cudaMemcpyDeviceToHost);
      cudaMemcpy(jv.data(), j.counts, j.nLines * 4, cudaMemcpyDeviceToHost);
    }
    j.release();
    std::vector<u64> jk2;
    std::vector<i64> jc2;
    jk2.reserve(jk.size());
    jc2.reserve(jk.size());
    for (size_t i = 0; i < jk.size(); ++i)
      if (jk[i] != kEmptyKey) { jk2.push_back(jk[i]); jc2.push_back((i64)(i32)jv[i]); }
    reduce_colours(c->params, jk2.data(), jc2.data(), jk2.size(), true, ck, cc);
  } else {
    reduce_colours(c->params, nullptr, nullptr, 0, false, ck, cc);
  }
  c->provJunctions = junction_path ? 1u : 0u;
  file_identity(dump_path, c->provDumpSize, c->provDumpMtime);
  file_identity(junction_path, c->provJuncSize, c->provJuncMtime);
  const int rc = build_table_device(c, d.keys, d.counts, d.nLines, d.tally.kept, ck, cc, n_kept);
  d.release();
  return rc;
}

// The round-1 ingest path, kept for A/B timing only (bench.py --time-table-load): threaded host parse of the mapped
// file (dump_parse.hpp), entries copied to the device afterwards.  Same table, bit for bit.
int talc_table_load_dump_host(talc_ctx* c, const char* dump_path, const char* junction_path, uint64_t* n_lines, uint64_t* n_kept) {
  if (!c || !dump_path) return TALC_ERR_ARG;
  DumpEntries d;
  std::string err;
  if (!parse_dump_file(dump_path, c->params.K, c->params.min_count, true, d, err)) {
    c->err = err;
    return TALC_ERR_IO;
  }
  if (n_lines) *n_lines = d.lines;
  std::vector<u64> ck;
  std::vector<u32> cc;
  if (junction_path) {
    DumpEntries j;
    if (!parse_dump_file(junction_path, c->params.K, 0, false, j, err)) {
      c->err = err;
      return TALC_ERR_IO;
    }
    std::vector<i64> jc(j.counts.begin(), j.counts.end());
    reduce_colours(c->params, j.keys.data(), jc.data(), j.keys.size(), true, ck, cc);
  } else {
    reduce_colours(c->params, nullptr, nullptr, 0, false, ck, cc);
  }
  std::vector<u32> v(d.counts.size());
  for (size_t i = 0; i < v.size(); ++i) v[i] = (u32)(int)d.counts[i];
  c->provJunctions = junction_path ? 1u : 0u;
  file_identity(dump_path, c->provDumpSize, c->provDumpMtime);
  file_identity(junction_path, c->provJuncSize, c->provJuncMtime);
  return build_table(c, d.keys, v, ck, cc, n_kept);
}

// ---------------------------------------------------------------------------------- row f3: count k-mers from short reads
static int junction_colours_gpu(talc_ctx* c, const char* junction_path, std::vector<u64>& ck, std::vector<u32>& cc) {
  std::string err;
  if (!junction_path) { reduce_colours(c->params, nullptr, nullptr, 0, false, ck, cc); return TALC_OK; }
  DeviceDump j;
  if (!parse_dump_gpu(junction_path, c->params.K, 0, false, c->sms, c->stream, j, err)) { c->err = err; return TALC_ERR_IO; }
  std::vector<u64> jk(j.nLines);
  std::vector<u32> jv(j.nLines);
  if (j.nLines) {
    cudaMemcpy(jk.data(), j.keys, j.nLines * 8, cudaMemcpyDeviceToHost);
    cudaMemcpy(jv.data(), j.counts, j.nLines * 4, cudaMemcpyDeviceToHost);
  }
  j.release();
  std::vector<u64> jk2;
  std::vector<i64> jc2;
  for (size_t i = 0; i < jk.size(); ++i)
    if (jk[i] != kEmptyKey) { jk2.push_back(jk[i]); jc2.push_back((i64)(i32)jv[i]); }
  reduce_colours(c->params, jk2.data(), jc2.data(), jk2.size(), true, ck, cc);
  return TALC_OK;
}

int talc_table_count_reads(talc_ctx* c, const char* const* paths, int n_paths, uint64_t expected_distinct, const char* junction_path,
                           uint64_t* n_kmers, uint64_t* n_distinct, uint64_t* n_kept) {
  if (!c || !paths || n_paths < 1) return TALC_ERR_ARG;
  CUDA_TRY(c, cudaSetDevice(c->device));
  const u32 K = c->params.K;
  if (expected_distinct == 0) {  // no hint (jellyfish's -s): one distinct k-mer per 4 bytes of input is generous
    for (int i = 0; i < n_paths; ++i) {
      struct stat st;
      if (stat(paths[i], &st) == 0) expected_distinct += (u64)st.st_size / 4;
    }
    if (expected_distinct < (1u << 20)) expected_distinct = 1u << 20;
  }
  u64 cap = 2;
  while (cap < 2 * expected_distinct + 2) cap <<= 1;
  const int blocks = c->sms * 8;
  Slot* big = nullptr;
  CUDA_TRY(c, cudaMalloc((void**)&big, cap * sizeof(Slot)));
  count_fill_empty_kernel<<<blocks, 256, 0, c->stream>>>(big, cap);
  const size_t piece = 64u << 20;
  char *pin = nullptr, *dText = nullptr;
  u8* dFlag = nullptr;
  u64* dStarts = nullptr;
  unsigned long long* dNum = nullptr;  // [0] line count / select count, [1] k-mer occurrences, [2] fail flag, [3] distinct, [4] kept
  void* dTmp = nullptr;
  size_t tmpBytes = 0;
  int rc = TALC_OK;
  auto fail = [&](int code, const std::string& msg) { rc = code; c->err = msg; };
  if (cudaHostAlloc((void**)&pin, piece, cudaHostAllocDefault) != cudaSuccess || cudaMalloc((void**)&dText, 2 * piece + 16) != cudaSuccess ||
      cudaMalloc((void**)&dFlag, 2 * piece) != cudaSuccess || cudaMalloc((void**)&dStarts, (2 * piece / 2 + 2) * 8) != cudaSuccess ||
      cudaMalloc((void**)&dNum, 64) != cudaSuccess)
    fail(TALC_ERR_CUDA, "talc_table_count_reads: out of memory");
  if (rc == TALC_OK) {
    cudaMemsetAsync(dNum, 0, 64, c->stream);
    thrust::counting_iterator<u64> pos0(0);
    cub::DeviceSelect::Flagged(nullptr, tmpBytes, pos0, dFlag, dStarts, (u64*)dNum, (int)(2 * piece), c->stream);
    if (cudaMalloc(&dTmp, tmpBytes + 16) != cudaSuccess) fail(TALC_ERR_CUDA, "talc_table_count_reads: out of memory");
  }
  for (int fi = 0; fi < n_paths && rc == TALC_OK; ++fi) {
    FILE* f = fopen(paths[fi], "rb");
    if (!f) { fail(TALC_ERR_IO, std::string("cannot open ") + paths[fi]); break; }
    u64 carry = 0;  // bytes of an incomplete record at the front of dText
    u32 period = 0;
    bool eof = false;
    while (!eof && rc == TALC_OK) {
      size_t n = fread(pin, 1, piece, f);
      eof = n < piece;
      if (n == 0 && carry == 0) break;
      if (period == 0) {
        size_t q = 0;
        while (q < n && (pin[q] == '\n' || pin[q] == '\r')) ++q;
        if (q < n && pin[q] == '@') period = 4;
        else if (q < n && pin[q] == '>') period = 2;
        else { fail(TALC_ERR_IO, std::string(paths[fi]) + " is neither FASTQ nor FASTA"); break; }
        if (q) { memmove(pin, pin + q, n - q); n -= q; }
      }
      if (n && cudaMemcpyAsync(dText + carry, pin, n, cudaMemcpyHostToDevice, c->stream) != cudaSuccess) { fail(TALC_ERR_CUDA, "copy failed"); break; }
      const u64 size = carry + n;
      cudaMemsetAsync(dNum, 0, 8, c->stream);
      line_flag_kernel<<<blocks, 256, 0, c->stream>>>(dText, size, dFlag, dNum);
      u64 nLines = 0;
      cudaMemcpyAsync(&nLines, dNum, 8, cudaMemcpyDeviceToHost, c->stream);
      if (cudaStreamSynchronize(c->stream) != cudaSuccess) { fail(TALC_ERR_CUDA, "line scan failed"); break; }
      if (nLines > piece) { fail(TALC_ERR_IO, std::string(paths[fi]) + ": lines of fewer than two bytes on average -- not a read file"); break; }
      thrust::counting_iterator<u64> pos(0);
      size_t tb = tmpBytes;
      cub::DeviceSelect::Flagged(dTmp, tb, pos, dFlag, dStarts, (u64*)dNum, (int)size, c->stream);
      // lines that are complete: all of them at the end of the file, else all but the last (which may be cut); records
      // that are complete: a multiple of `period` lines
      u64 usable = eof ? nLines : (nLines ? nLines - 1 : 0);
      usable -= usable % period;
      u64 cut = size;
      if (usable < nLines) {
        cudaMemcpyAsync(&cut, dStarts + usable, 8, cudaMemcpyDeviceToHost, c->stream);
        if (cudaStreamSynchronize(c->stream) != cudaSuccess) { fail(TALC_ERR_CUDA, "line scan failed"); break; }
      }
      if (usable) {
        count_kmers_kernel<<<blocks, 256, 0, c->stream>>>(dText, cut, dStarts, usable, period, K, big, cap - 1, dNum + 1, (u32*)(dNum + 2));
        if (cudaGetLastError() != cudaSuccess) { fail(TALC_ERR_CUDA, "count kernel launch failed"); break; }
      }
      carry = size - cut;
      if (carry > piece) { fail(TALC_ERR_IO, std::string("a record of ") + paths[fi] + " is longer than 64 MiB"); break; }
      if (carry) cudaMemcpyAsync(dText, dText + cut, carry, cudaMemcpyDeviceToDevice, c->stream);  // cut >= carry: no overlap
      if (eof) break;
    }
    fclose(f);
  }
  unsigned long long h[5] = {0, 0, 0, 0, 0};
  if (rc == TALC_OK) {
    count_tally_kernel<<<blocks, 256, 0, c->stream>>>(big, cap, c->params.min_count, dNum + 3, dNum + 4);
    cudaMemcpyAsync(h, dNum, sizeof(h), cudaMemcpyDeviceToHost, c->stream);
    if (cudaStreamSynchronize(c->stream) != cudaSuccess) fail(TALC_ERR_CUDA, std::string("k-mer counting failed: ") + cudaGetErrorString(cudaGetLastError()));
    else if (h[2]) fail(TALC_ERR_CAPACITY, "the counting table is full: raise expected_distinct (jellyfish's -s)");
  }
  if (rc == TALC_OK) {
    if (n_kmers) *n_kmers = h[1];
    if (n_distinct) *n_distinct = h[3];
    u64 fcap = 2;
    while (fcap < 2 * h[4] + 2) fcap <<= 1;
    rc = talc_table_alloc(c, fcap);
    if (rc == TALC_OK) {
      cudaMemsetAsync(dNum, 0, 64, c->stream);
      count_rehash_kernel<<<blocks, 256, 0, c->stream>>>(big, cap, c->params.min_count, c->slots, fcap - 1, (u32*)(dNum + 1));
      std::vector<u64> ck;
      std::vector<u32> cc;
      rc = junction_colours_gpu(c, junction_path, ck, cc);
      c->provJunctions = junction_path ? 1u : 0u;
      c->provDumpSize = c->provDumpMtime = 0;
      file_identity(junction_path, c->provJuncSize, c->provJuncMtime);
      if (rc == TALC_OK) rc = finish_table(c, dNum, ck, cc, n_kept);
    }
  }
  if (pin) cudaFreeHost(pin);
  if (dText) cudaFree(dText);
  if (dFlag) cudaFree(dFlag);
  if (dStarts) cudaFree(dStarts);
  if (dNum) cudaFree(dNum);
  if (dTmp) cudaFree(dTmp);
  cudaFree(big);
  return rc;
}

int talc_dump_write_packed(const char* path, const uint64_t* keys, const int64_t* counts, uint64_t n, uint32_t K) {
  if (!path || (n && (!keys || !counts)) || K < 1 || K > 31) return TALC_ERR_ARG;
  FILE* f = fopen(path, "wb");
  if (!f) return TALC_ERR_IO;
  std::vector<char> buf;
  buf.reserve((size_t)(1u << 22) + 64);
  bool ok = true;
  for (u64 i = 0; i < n && ok; ++i) {
    char line[64];
    u32 p = 0;
    for (u32 j = 0; j < K; ++j) line[p++] = "ACGT"[(keys[i] >> (2 * (K - 1 - j))) & 3ull];
    line[p++] = ' ';
    p += (u32)snprintf(line + p, sizeof(line) - p, "%lld", (long long)counts[i]);
    line[p++] = '\n';
    buf.insert(buf.end(), line, line + p);
    if (buf.size() >= (1u << 22)) { ok = fwrite(buf.data(), 1, buf.size(), f) == buf.size(); buf.clear(); }
  }
  if (ok && !buf.empty()) ok = fwrite(buf.data(), 1, buf.size(), f) == buf.size();
  ok = (fclose(f) == 0) && ok;
  return ok ? TALC_OK : TALC_ERR_IO;
}

int talc_table_lookup(talc_ctx* c, const uint64_t* keys, uint64_t n, uint32_t* counts, uint32_t* colours, uint8_t* found) {
  if (!c || !c->tableReady) return TALC_ERR_NO_TABLE;
  if (!n) return TALC_OK;
  CUDA_TRY(c, cudaSetDevice(c->device));
  u64* dK;
  u32 *dC, *dL;
  u8* dF;
  CUDA_TRY(c, cudaMalloc((void**)&dK, n * 8));
  CUDA_TRY(c, cudaMalloc((void**)&dC, n * 4));
  CUDA_TRY(c, cudaMalloc((void**)&dL, n * 4));
  CUDA_TRY(c, cudaMalloc((void**)&dF, n));
  CUDA_TRY(c, cudaMemcpyAsync(dK, keys, n * 8, cudaMemcpyHostToDevice, c->stream));
  TableView tv{c->slots, c->capacity - 1};
  table_lookup_kernel<<<c->sms * 4, 256, 0, c->stream>>>(tv, dK, n, dC, dL, dF);
  CUDA_TRY(c, cudaGetLastError());
  CUDA_TRY(c, cudaMemcpyAsync(counts, dC, n * 4, cudaMemcpyDeviceToHost, c->stream));
  CUDA_TRY(c, cudaMemcpyAsync(colours, dL, n * 4, cudaMemcpyDeviceToHost, c->stream));
  CUDA_TRY(c, cudaMemcpyAsync(found, dF, n, cudaMemcpyDeviceToHost, c->stream));
  CUDA_TRY(c, cudaStreamSynchronize(c->stream));
  cudaFree(dK); cudaFree(dC); cudaFree(dL); cudaFree(dF);
  return TALC_OK;
}

// One pass of the correction over the reads of A.order (tier 1: the whole batch; tier 2: the reads whose arena was too
// small).  Split mode alternates control_kernel and walk_kernel until every read of the pass is done; the host only
// enqueues rounds and polls one counter every few rounds.  nCtx contexts are in flight, each with its own arena.
static int run_pass(talc_ctx* c, CorrectArgs& A, u32 nCtx, u64* launches) {
  const u32 n = A.nOrder;
  if (!c->splitWalk) {
    u32 blocks = (nCtx + 3) / 4;
    correct_kernel<<<blocks, 128, 0, c->stream>>>(A);
    CUDA_TRY(c, cudaGetLastError());
    if (launches) *launches += 1;
    return TALC_OK;
  }
  CUDA_TRY(c, c->readCtxs.reserve((size_t)nCtx * sizeof(ReadCtx)));
  CUDA_TRY(c, c->roundLists.reserve((size_t)nCtx * 8 + 256));
  ReadCtx* ctxs = (ReadCtx*)c->readCtxs.p;
  u32* dCnt = (u32*)c->roundLists.p;  // [0] nReady, [1] nWalk, [2] taskCursor, [3] finished
  u32* readyList = dCnt + 64;
  u32* walkList = readyList + nCtx;
  CUDA_TRY(c, cudaMemsetAsync(dCnt, 0, 256, c->stream));
  ctx_init_kernel<<<(nCtx + 255) / 256, 256, 0, c->stream>>>(ctxs, nCtx, readyList, dCnt);
  CUDA_TRY(c, cudaGetLastError());
  RoundArgs R;
  R.A = A;
  R.ctxs = ctxs;
  R.readyList = readyList;
  R.nReady = dCnt;
  R.walkList = walkList;
  R.nWalk = dCnt + 1;
  R.taskCursor = dCnt + 2;
  R.finished = dCnt + 3;
  u32 ctlBlocks = (u32)c->sms * c->blocksPerSm;
  if (ctlBlocks * 4 > nCtx) ctlBlocks = (nCtx + 3) / 4;
  u32 walkBlocks = (u32)c->sms * 4;
  if (walkBlocks * 32 > nCtx) walkBlocks = (nCtx + 31) / 32;
  if (getenv("TALC_ROUND_DEBUG")) {  // tuning aid: every round timed and counted on its own (no graph)
    cudaEvent_t e0, e1, e2;
    cudaEventCreate(&e0); cudaEventCreate(&e1); cudaEventCreate(&e2);
    double tc = 0, tw = 0;
    u64 rounds = 0, sumReady = 0, sumWalk = 0;
    u32 h[4];
    for (;;) {
      u32 hr = 0;
      cudaMemcpyAsync(&hr, dCnt, 4, cudaMemcpyDeviceToHost, c->stream);
      cudaMemsetAsync(dCnt + 1, 0, 8, c->stream);
      cudaEventRecord(e0, c->stream);
      control_kernel<<<ctlBlocks, 128, 0, c->stream>>>(R);
      cudaEventRecord(e1, c->stream);
      cudaMemsetAsync(dCnt, 0, 4, c->stream);
      walk_kernel<<<walkBlocks, 256, 0, c->stream>>>(ctxs, walkList, dCnt + 1, readyList, dCnt, c->walkStepCap);
      cudaEventRecord(e2, c->stream);
      cudaMemcpyAsync(h, dCnt, 16, cudaMemcpyDeviceToHost, c->stream);
      CUDA_TRY(c, cudaStreamSynchronize(c->stream));
      float a = 0, b = 0;
      cudaEventElapsedTime(&a, e0, e1);
      cudaEventElapsedTime(&b, e1, e2);
      tc += a; tw += b; ++rounds; sumReady += hr; sumWalk += h[1];
      if (rounds <= 40 || (rounds % 200) == 0 || h[3] >= n)
        fprintf(stderr, "[round %llu] ready %u -> control %.3f ms -> walk %u -> %.3f ms ; finished %u / %u\n",
                (unsigned long long)rounds, hr, a, h[1], b, h[3], n);
      if (h[3] >= n) break;
      if (rounds > 2000000) break;
    }
    fprintf(stderr, "[rounds] %llu rounds: control %.1f ms, walk %.1f ms; tasks %llu (%.1f per round), walks %llu\n",
            (unsigned long long)rounds, tc, tw, (unsigned long long)sumReady, (double)sumReady / rounds, (unsigned long long)sumWalk);
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaEventDestroy(e2);
    c->lastRounds += rounds;
    if (launches) *launches += 2 * rounds + 1;
    return TALC_OK;
  }
  // a chunk of rounds is captured once into a CUDA graph (4 nodes per round) and replayed: the host enqueues one graph
  // and reads one counter per chunk instead of driving every launch
  const u32 chunk = 16;
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  bool captured = cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
  if (captured) {
    for (u32 i = 0; i < chunk; ++i) {
      cudaMemsetAsync(dCnt + 1, 0, 8, c->stream);  // nWalk, taskCursor
      control_kernel<<<ctlBlocks, 128, 0, c->stream>>>(R);
      cudaMemsetAsync(dCnt, 0, 4, c->stream);      // nReady
      walk_kernel<<<walkBlocks, 256, 0, c->stream>>>(ctxs, walkList, dCnt + 1, readyList, dCnt, c->walkStepCap);
    }
    captured = cudaStreamEndCapture(c->stream, &graph) == cudaSuccess && graph != nullptr &&
               cudaGraphInstantiate(&exec, graph, 0) == cudaSuccess;
  }
  if (!captured) {
    if (graph) cudaGraphDestroy(graph);
    c->err = std::string("cannot capture the correction rounds into a CUDA graph: ") + cudaGetErrorString(cudaGetLastError());
    return TALC_ERR_CUDA;
  }
  u64 rounds = 0;
  u32 hFinished = 0;
  int rc = TALC_OK;
  const auto t0 = std::chrono::steady_clock::now();
  for (;;) {
    if (cudaGraphLaunch(exec, c->stream) != cudaSuccess ||
        cudaMemcpyAsync(&hFinished, dCnt + 3, 4, cudaMemcpyDeviceToHost, c->stream) != cudaSuccess ||
        cudaStreamSynchronize(c->stream) != cudaSuccess) {
      c->err = std::string("correction rounds failed: ") + cudaGetErrorString(cudaGetLastError());
      rc = TALC_ERR_CUDA;
      break;
    }
    rounds += chunk;
    if (hFinished >= n) break;
    if (std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() > 600.0) {
      c->err = "correction rounds did not terminate within 600 s (" + std::to_string(hFinished) + " of " + std::to_string(n) + " reads done)";
      rc = TALC_ERR_CUDA;
      break;
    }
  }
  cudaGraphExecDestroy(exec);
  cudaGraphDestroy(graph);
  if (rc) return rc;
  c->lastRounds += rounds;
  if (launches) *launches += 2 * rounds + 1;
  return TALC_OK;
}

// ---------------------------------------------------------------------------------- correction
// shared front end: k-mer offsets, length-sorted order, coverage.  d_bases/d_offs on device.  In reverse mode the reads
// are first reverse-complemented into rcBases (same offsets) and dBases is pointed there for the rest of the batch.
static int prepare_batch(talc_ctx* c, const u8*& dBases, const u64* dOffs, u32 n, u64 totalBases, u64& totalKmers) {
  const u32 K = c->params.K;
  CUDA_TRY(c, c->nk.reserve((size_t)(n + 1) * 8));
  CUDA_TRY(c, c->kmerOff.reserve((size_t)(n + 1) * 8));
  CUDA_TRY(c, c->sortKey.reserve((size_t)n * 4));
  CUDA_TRY(c, c->sortKeyOut.reserve((size_t)n * 4));
  CUDA_TRY(c, c->sortVal.reserve((size_t)n * 4));
  CUDA_TRY(c, c->order.reserve((size_t)n * 4));
  kmer_count_kernel<<<(n + 255) / 256, 256, 0, c->stream>>>(dOffs, n, K, (u64*)c->nk.p, (u32*)c->sortKey.p, (u32*)c->sortVal.p);
  CUDA_TRY(c, cudaGetLastError());
  CUDA_TRY(c, cudaMemsetAsync((u64*)c->nk.p + n, 0, 8, c->stream));
  size_t tmp1 = 0, tmp2 = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, tmp1, (u64*)c->nk.p, (u64*)c->kmerOff.p, n + 1, c->stream);
  cub::DeviceRadixSort::SortPairs(nullptr, tmp2, (u32*)c->sortKey.p, (u32*)c->sortKeyOut.p, (u32*)c->sortVal.p, (u32*)c->order.p,
                                  (int)n, 0, 32, c->stream);
  CUDA_TRY(c, c->cubTmp.reserve(std::max(tmp1, tmp2)));
  size_t tb = c->cubTmp.cap;
  CUDA_TRY(c, cub::DeviceScan::ExclusiveSum(c->cubTmp.p, tb, (u64*)c->nk.p, (u64*)c->kmerOff.p, n + 1, c->stream));
  u64 hk = 0, hEnd = 0;
  CUDA_TRY(c, cudaMemcpyAsync(&hk, (u64*)c->kmerOff.p + n, 8, cudaMemcpyDeviceToHost, c->stream));
  if (c->reverse) CUDA_TRY(c, cudaMemcpyAsync(&hEnd, dOffs + n, 8, cudaMemcpyDeviceToHost, c->stream));
  CUDA_TRY(c, cudaStreamSynchronize(c->stream));
  totalKmers = hk;
  CUDA_TRY(c, c->cov.reserve((size_t)(hk + 4) * 4));
  TableView tv{c->slots, c->capacity - 1};
  const int blocks = c->sms * 8;
  if (c->reverse) {  // sized from the offsets themselves: the caller's buffer is read where they point
    CUDA_TRY(c, c->rcBases.reserve(hEnd + 64));
    revcomp_reads_kernel<<<blocks, 256, 0, c->stream>>>(dBases, dOffs, n, (u8*)c->rcBases.p);
    CUDA_TRY(c, cudaGetLastError());
    dBases = (const u8*)c->rcBases.p;
  }
  CUDA_TRY(c, cudaEventRecord(c->ev[1], c->stream));
  coverage_kernel<<<blocks, 256, 0, c->stream>>>(tv, K, dBases, dOffs, (const u64*)c->kmerOff.p, n, (u32*)c->cov.p);
  CUDA_TRY(c, cudaGetLastError());
  CUDA_TRY(c, cudaEventRecord(c->ev[2], c->stream));
  // processing order of the correction kernel: estimated cost, descending
  cost_key_kernel<<<blocks, 256, 0, c->stream>>>((const u32*)c->cov.p, (const u64*)c->kmerOff.p, dOffs, n, c->P.min_count,
                                                 (u32*)c->sortKey.p, (u32*)c->sortVal.p);
  CUDA_TRY(c, cudaGetLastError());
  tb = c->cubTmp.cap;
  CUDA_TRY(c, cub::DeviceRadixSort::SortPairs(c->cubTmp.p, tb, (u32*)c->sortKey.p, (u32*)c->sortKeyOut.p, (u32*)c->sortVal.p,
                                              (u32*)c->order.p, (int)n, 0, 32, c->stream));
  (void)totalBases;
  return TALC_OK;
}

static int correct_batch_device_impl(talc_ctx* c, const uint8_t* dBases, const uint64_t* dOffs, uint32_t n, uint64_t totalBases,
                                     uint8_t* dOut, uint64_t outCapacity, uint64_t* dOutOffs, uint8_t* dStatus,
                                     talc_counters* counters, u32* dReadStats);
int talc_correct_batch_device(talc_ctx* c, const uint8_t* dBases, const uint64_t* dOffs, uint32_t n, uint64_t totalBases,
                              uint8_t* dOut, uint64_t outCapacity, uint64_t* dOutOffs, uint8_t* dStatus,
                              talc_counters* counters) {
  return correct_batch_device_impl(c, dBases, dOffs, n, totalBases, dOut, outCapacity, dOutOffs, dStatus, counters, nullptr);
}
static int correct_batch_device_impl(talc_ctx* c, const uint8_t* dBases, const uint64_t* dOffs, uint32_t n, uint64_t totalBases,
                                     uint8_t* dOut, uint64_t outCapacity, uint64_t* dOutOffs, uint8_t* dStatus,
                                     talc_counters* counters, u32* dReadStats) {
  if (!c) return TALC_ERR_ARG;
  if (c->parent) lane_follow(c);
  if (!c->tableReady) { c->err = "no k-mer table loaded"; return TALC_ERR_NO_TABLE; }
  CUDA_TRY(c, cudaSetDevice(c->device));
  if (counters) memset(counters, 0, sizeof(*counters));
  if (n == 0) {
    if (dOutOffs) CUDA_TRY(c, cudaMemsetAsync(dOutOffs, 0, 8, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    return TALC_OK;
  }
  CUDA_TRY(c, cudaEventRecord(c->ev[0], c->stream));
  u64 totalKmers = 0;
  int rc = prepare_batch(c, dBases, dOffs, n, totalBases, totalKmers);
  if (rc) return rc;

  // launch geometry.  Monolithic mode: 128-thread blocks (4 warps = 4 reads in flight per block), a multiple of the
  // SM count, no more warps than there are reads.  Split mode: nCtx read contexts in flight, each with its own arena.
  u32 blocksPerSm = c->blocksPerSm;
  u32 blocks = (u32)c->sms * blocksPerSm;
  while (blocks > (u32)c->sms && (u64)(blocks - c->sms) * 4 >= n) blocks -= c->sms;
  const u64 nWarps = c->splitWalk ? (u64)std::min<u32>(n, c->nCtxTier1) : (u64)blocks * 4;
  const u64 outArenaCap = 2 * totalBases + (u64)n * 64 + 4096;
  CUDA_TRY(c, c->arenas.reserve(std::max<size_t>((size_t)nWarps * c->tier1Bytes, (size_t)c->tier2Warps * c->tier2Bytes)));
  CUDA_TRY(c, c->outArena.reserve(outArenaCap));
  CUDA_TRY(c, c->outPos.reserve((size_t)n * 8));
  CUDA_TRY(c, c->outLen.reserve((size_t)n * 4));
  CUDA_TRY(c, c->outLen64.reserve((size_t)(n + 1) * 8));
  CUDA_TRY(c, c->overflowList.reserve((size_t)n * 4));
  CUDA_TRY(c, c->misc.reserve(1024));
  // misc layout (u64 words): [0..kNumCounters) counters | then outCursor | workCounter,nOverflow,outFull (u32)
  unsigned long long* dCounters = (unsigned long long*)c->misc.p;
  unsigned long long* dCursor = dCounters + kNumCounters;
  u32* dWork = (u32*)(dCursor + 1);
  u32* dNOver = dWork + 1;
  u32* dOutFull = dWork + 2;
  CUDA_TRY(c, cudaMemsetAsync(c->misc.p, 0, 1024, c->stream));

  CorrectArgs A;
  A.tv = TableView{c->slots, c->capacity - 1};
  A.cright = CtxView{c->ctxRight, c->ctxCap - 1};
  A.cleft = CtxView{c->ctxLeft, c->ctxCap - 1};
  A.P = c->P;
  A.tabs.lower = c->modelTabs;
  A.tabs.upper = c->modelTabs + kModelTabN;
  A.tabs.sq = c->modelTabs + 2 * kModelTabN;
  A.tabs.n = kModelTabN;
  A.bases = dBases;
  A.offs = dOffs;
  A.kmerOff = (const u64*)c->kmerOff.p;
  A.cov = (const u32*)c->cov.p;
  A.order = (const u32*)c->order.p;
  A.nOrder = n;
  A.arenas = (u8*)c->arenas.p;
  A.arenaBytes = c->tier1Bytes;
  A.outArena = (u8*)c->outArena.p;
  A.outCap = outArenaCap;
  A.outCursor = dCursor;
  A.outPos = (u64*)c->outPos.p;
  A.outLen = (u32*)c->outLen.p;
  A.status = dStatus;
  A.counters = dCounters;
  A.workCounter = dWork;
  A.overflowList = (u32*)c->overflowList.p;
  A.nOverflow = dNOver;
  A.outFull = dOutFull;
  A.readKcycles = nullptr;
  A.readStats = dReadStats;
  DevBuf dbgCycles;
  const bool dbg = getenv("TALC_DEBUG_CYCLES") != nullptr;
  if (dbg) {
    CUDA_TRY(c, dbgCycles.reserve((size_t)n * 4));
    CUDA_TRY(c, cudaMemsetAsync(dbgCycles.p, 0, (size_t)n * 4, c->stream));
    A.readKcycles = (u32*)dbgCycles.p;
  }
  A.wide = 1;
  A.lastTier = 0;
  A.pauseCycles = c->pauseCycles;
  A.inlineInner = c->inlineInner;
  A.inlineBorder = c->inlineBorder;
  u64 launches = 3;
  c->lastRounds = 0;
  {
    const int rcp = run_pass(c, A, (u32)nWarps, &launches);
    if (rcp) return rcp;
  }
  CUDA_TRY(c, cudaEventRecord(c->ev[3], c->stream));
  u32 hOver = 0;
  CUDA_TRY(c, cudaMemcpyAsync(&hOver, dNOver, 4, cudaMemcpyDeviceToHost, c->stream));
  CUDA_TRY(c, cudaStreamSynchronize(c->stream));
  if (hOver > 0) {
    // second tier: only the reads whose first-tier slice was too small, worst-case buffer sizing
    CUDA_TRY(c, cudaMemsetAsync(dWork, 0, 8, c->stream));  // workCounter and nOverflow
    CorrectArgs B = A;
    B.order = (const u32*)c->overflowList.p;  // read in place: tier 2 appends to a second list
    CUDA_TRY(c, c->sortVal.reserve((size_t)n * 4));
    CUDA_TRY(c, cudaMemcpyAsync(c->sortVal.p, c->overflowList.p, (size_t)hOver * 4, cudaMemcpyDeviceToDevice, c->stream));
    B.order = (const u32*)c->sortVal.p;
    B.nOrder = hOver;
    B.arenaBytes = c->tier2Bytes;
    B.lastTier = 1;
    const int rcp = run_pass(c, B, std::max<u32>(1, std::min<u32>(c->tier2Warps, hOver)), &launches);
    if (rcp) return rcp;
  }
  CUDA_TRY(c, cudaEventRecord(c->ev[4], c->stream));
  // input order: exclusive scan of the lengths, then gather
  len_to_u64_kernel<<<(n + 255) / 256, 256, 0, c->stream>>>((const u32*)c->outLen.p, n, (u64*)c->outLen64.p);
  CUDA_TRY(c, cudaMemsetAsync((u64*)c->outLen64.p + n, 0, 8, c->stream));
  size_t tb = c->cubTmp.cap;
  CUDA_TRY(c, cub::DeviceScan::ExclusiveSum(c->cubTmp.p, tb, (u64*)c->outLen64.p, dOutOffs, n + 1, c->stream));
  u64 hTotalOut = 0;
  u32 hOutFull = 0;
  unsigned long long hCtr[kNumCounters];
  CUDA_TRY(c, cudaMemcpyAsync(&hTotalOut, dOutOffs + n, 8, cudaMemcpyDeviceToHost, c->stream));
  CUDA_TRY(c, cudaMemcpyAsync(&hOutFull, dOutFull, 4, cudaMemcpyDeviceToHost, c->stream));
  CUDA_TRY(c, cudaMemcpyAsync(hCtr, dCounters, sizeof(hCtr), cudaMemcpyDeviceToHost, c->stream));
  CUDA_TRY(c, cudaStreamSynchronize(c->stream));
  if (hOutFull) { c->err = "internal output arena too small"; return TALC_ERR_CAPACITY; }
  if (hTotalOut > outCapacity) { c->err = "out_capacity too small for the corrected reads"; return TALC_ERR_CAPACITY; }
  gather_kernel<<<c->sms * 8, 256, 0, c->stream>>>((const u8*)c->outArena.p, (const u64*)c->outPos.p, (const u32*)c->outLen.p,
                                                  dOutOffs, n, dOut, dStatus, c->reverse);
  CUDA_TRY(c, cudaGetLastError());
  CUDA_TRY(c, cudaEventRecord(c->ev[5], c->stream));
  CUDA_TRY(c, cudaStreamSynchronize(c->stream));
  if (dbg) {
    std::vector<u32> kc(n);
    std::vector<u64> ho(n + 1);
    cudaMemcpy(kc.data(), dbgCycles.p, (size_t)n * 4, cudaMemcpyDeviceToHost);
    cudaMemcpy(ho.data(), dOffs, (size_t)(n + 1) * 8, cudaMemcpyDeviceToHost);
    std::vector<u32> idx(n);
    for (u32 i = 0; i < n; ++i) idx[i] = i;
    std::sort(idx.begin(), idx.end(), [&](u32 a, u32 b) { return kc[a] > kc[b]; });
    double sum = 0;
    for (u32 i = 0; i < n; ++i) sum += kc[i];
    fprintf(stderr, "[talc debug] per-read Mcycles: total %.0f  mean %.3f  p50 %.3f  p99 %.3f  max %.3f\n", sum / 1024, sum / 1024 / n,
            kc[idx[n / 2]] / 1024.0, kc[idx[n / 100]] / 1024.0, kc[idx[0]] / 1024.0);
    for (u32 i = 0; i < 8 && i < n; ++i)
      fprintf(stderr, "[talc debug]   slow read %u: %.1f Mcycles, length %llu\n", idx[i], kc[idx[i]] / 1024.0,
              (unsigned long long)(ho[idx[i] + 1] - ho[idx[i]]));
    if (const char* path = getenv("TALC_DEBUG_CYCLES_FILE")) {  // raw u32 kilo-cycles per read, input order
      if (FILE* f = fopen(path, "wb")) {
        fwrite(kc.data(), 4, n, f);
        fclose(f);
      }
    }
    dbgCycles.release();
  }
  if (counters) {
    memcpy(counters, hCtr, sizeof(hCtr));
    counters->reads = n;
    counters->bases_in = totalBases;
    counters->reads_second_tier = hOver;
    counters->kernel_launches = launches + 3;
    counters->rounds = c->lastRounds;
    float ms = 0;
    cudaEventElapsedTime(&ms, c->ev[1], c->ev[2]); counters->ms_coverage = ms;
    cudaEventElapsedTime(&ms, c->ev[2], c->ev[3]); counters->ms_correct = ms;
    cudaEventElapsedTime(&ms, c->ev[3], c->ev[4]); counters->ms_correct_tier2 = ms;
    cudaEventElapsedTime(&ms, c->ev[4], c->ev[5]); counters->ms_gather = ms;
    cudaEventElapsedTime(&ms, c->ev[0], c->ev[5]); counters->ms_total = ms;
  }
  return TALC_OK;
}

int talc_correct_batch(talc_ctx* c, const uint8_t* bases, const uint64_t* offsets, uint32_t n, uint8_t* out,
                       uint64_t outCapacity, uint64_t* outOffsets, uint8_t* status, talc_counters* counters) {
  if (!c || !offsets || !outOffsets || (n && (!bases || !out || !status))) return TALC_ERR_ARG;
  if (!c->tableReady) { c->err = "no k-mer table loaded"; return TALC_ERR_NO_TABLE; }
  CUDA_TRY(c, cudaSetDevice(c->device));
  const u64 total = offsets[n] - offsets[0];
  if (offsets[0] != 0) { c->err = "offsets[0] must be 0"; return TALC_ERR_ARG; }
  CUDA_TRY(c, c->bases.reserve(total + 64));
  CUDA_TRY(c, c->offs.reserve((size_t)(n + 1) * 8));
  CUDA_TRY(c, c->status.reserve(n + 1));
  CUDA_TRY(c, c->outOffs.reserve((size_t)(n + 1) * 8));
  const u64 dOutCap = 2 * total + (u64)n * 64 + 4096;
  CUDA_TRY(c, c->out.reserve(dOutCap));
  CUDA_TRY(c, cudaEventRecord(c->ev[6], c->stream));
  CUDA_TRY(c, cudaMemcpyAsync(c->bases.p, bases, total, cudaMemcpyHostToDevice, c->stream));
  CUDA_TRY(c, cudaMemcpyAsync(c->offs.p, offsets, (size_t)(n + 1) * 8, cudaMemcpyHostToDevice, c->stream));
  CUDA_TRY(c, cudaEventRecord(c->ev[7], c->stream));
  talc_counters local;
  int rc = talc_correct_batch_device(c, (const u8*)c->bases.p, (const u64*)c->offs.p, n, total, (u8*)c->out.p, dOutCap,
                                     (u64*)c->outOffs.p, (u8*)c->status.p, &local);
  if (rc) return rc;
  float msH2D = 0;
  cudaEventElapsedTime(&msH2D, c->ev[6], c->ev[7]);
  CUDA_TRY(c, cudaEventRecord(c->ev[6], c->stream));
  CUDA_TRY(c, cudaMemcpyAsync(outOffsets, c->outOffs.p, (size_t)(n + 1) * 8, cudaMemcpyDeviceToHost, c->stream));
  CUDA_TRY(c, cudaMemcpyAsync(status, c->status.p, n, cudaMemcpyDeviceToHost, c->stream));
  CUDA_TRY(c, cudaStreamSynchronize(c->stream));
  const u64 totalOut = outOffsets[n];
  if (totalOut > outCapacity) { c->err = "out_capacity too small for the corrected reads"; return TALC_ERR_CAPACITY; }
  CUDA_TRY(c, cudaMemcpyAsync(out, c->out.p, totalOut, cudaMemcpyDeviceToHost, c->stream));
  CUDA_TRY(c, cudaEventRecord(c->ev[7], c->stream));
  CUDA_TRY(c, cudaStreamSynchronize(c->stream));
  float msD2H = 0;
  cudaEventElapsedTime(&msD2H, c->ev[6], c->ev[7]);
  if (counters) {
    *counters = local;
    counters->ms_h2d = msH2D;
    counters->ms_d2h = msD2H;
    counters->ms_total = local.ms_total + msH2D + msD2H;
  }
  return TALC_OK;
}

int talc_coverage_batch(talc_ctx* c, const uint8_t* bases, const uint64_t* offsets, uint32_t n, uint32_t* counts,
                        uint64_t countsCapacity) {
  if (!c || !offsets || (n && !bases)) return TALC_ERR_ARG;
  if (c->parent) lane_follow(c);
  if (!c->tableReady) return TALC_ERR_NO_TABLE;
  if (!n) return TALC_OK;
  CUDA_TRY(c, cudaSetDevice(c->device));
  const u64 total = offsets[n];
  CUDA_TRY(c, c->bases.reserve(total + 64));
  CUDA_TRY(c, c->offs.reserve((size_t)(n + 1) * 8));
  CUDA_TRY(c, cudaMemcpyAsync(c->bases.p, bases, total, cudaMemcpyHostToDevice, c->stream));
  CUDA_TRY(c, cudaMemcpyAsync(c->offs.p, offsets, (size_t)(n + 1) * 8, cudaMemcpyHostToDevice, c->stream));
  u64 totalKmers = 0;
  const u8* dBases = (const u8*)c->bases.p;  // the reverse-complemented copy in reverse mode
  int rc = prepare_batch(c, dBases, (const u64*)c->offs.p, n, total, totalKmers);
  if (rc) return rc;
  if (totalKmers > countsCapacity) { c->err = "counts_capacity too small"; return TALC_ERR_CAPACITY; }
  CUDA_TRY(c, cudaMemcpyAsync(counts, c->cov.p, totalKmers * 4, cudaMemcpyDeviceToHost, c->stream));
  CUDA_TRY(c, cudaStreamSynchronize(c->stream));
  return TALC_OK;
}

// ---------------------------------------------------------------------------------- roofline microbenchmark
int talc_bench_random_sectors(talc_ctx* c, uint64_t buffer_bytes, int dependent, uint32_t warps_per_sm, double* gbs,
                              double* ns_per_load) {
  if (!c || !gbs || buffer_bytes < (1u << 20)) return TALC_ERR_ARG;
  CUDA_TRY(c, cudaSetDevice(c->device));
  u64 sectors = 1;
  while (sectors * 2 * 32 <= buffer_bytes) sectors <<= 1;
  void* buf = nullptr;
  unsigned long long* sink = nullptr;
  CUDA_TRY(c, cudaMalloc(&buf, sectors * 32));
  CUDA_TRY(c, cudaMalloc((void**)&sink, 8));
  CUDA_TRY(c, cudaMemsetAsync(buf, 0x5a, sectors * 32, c->stream));
  if (warps_per_sm == 0) warps_per_sm = 64;
  const u32 blocks = (u32)c->sms * ((warps_per_sm + 7) / 8);
  const u32 iters = dependent ? 2048u : 1024u;
  const int ilp = dependent ? 1 : 8;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  float best = 1e30f;
  for (int rep = 0; rep < 4; ++rep) {  // first repetition warms up
    CUDA_TRY(c, cudaEventRecord(e0, c->stream));
    if (dependent) random_sector_kernel<1><<<blocks, 256, 0, c->stream>>>((const ulonglong4*)buf, sectors - 1, iters, 1, sink);
    else random_sector_kernel<8><<<blocks, 256, 0, c->stream>>>((const ulonglong4*)buf, sectors - 1, iters, 0, sink);
    CUDA_TRY(c, cudaGetLastError());
    CUDA_TRY(c, cudaEventRecord(e1, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    if (rep && ms < best) best = ms;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(buf);
  cudaFree(sink);
  const double loads = (double)blocks * 256.0 * iters * ilp;
  *gbs = loads * 32.0 / 1e9 / (best / 1e3);
  if (ns_per_load) *ns_per_load = (double)best * 1e6 / iters;  // per thread: latency of one dependent load (mode 1)
  return TALC_OK;
}

// ---------------------------------------------------------------------------------- self-tests
int talc_test_align(talc_ctx* c, int op, const uint8_t* a, const uint64_t* aOff, const uint8_t* b, const uint64_t* bOff,
                    uint32_t n, int aux, int aux2, int32_t* result) {
  if (!c || !n) return TALC_ERR_ARG;
  CUDA_TRY(c, cudaSetDevice(c->device));
  const u32 arenaBytes = (op == 4) ? (256u << 10) : (1u << 20);
  u8 *dA, *dB, *dAr;
  u64 *dAo, *dBo;
  i32* dR;
  const size_t rn = (size_t)n * (op >= 3 ? 4 : 1);
  CUDA_TRY(c, cudaMalloc((void**)&dA, aOff[n] + 1));
  CUDA_TRY(c, cudaMalloc((void**)&dB, bOff[n] + 1));
  CUDA_TRY(c, cudaMalloc((void**)&dAo, (size_t)(n + 1) * 8));
  CUDA_TRY(c, cudaMalloc((void**)&dBo, (size_t)(n + 1) * 8));
  CUDA_TRY(c, cudaMalloc((void**)&dAr, (size_t)n * arenaBytes));
  CUDA_TRY(c, cudaMalloc((void**)&dR, rn * 4));
  CUDA_TRY(c, cudaMemcpyAsync(dA, a, aOff[n], cudaMemcpyHostToDevice, c->stream));
  CUDA_TRY(c, cudaMemcpyAsync(dB, b, bOff[n], cudaMemcpyHostToDevice, c->stream));
  CUDA_TRY(c, cudaMemcpyAsync(dAo, aOff, (size_t)(n + 1) * 8, cudaMemcpyHostToDevice, c->stream));
  CUDA_TRY(c, cudaMemcpyAsync(dBo, bOff, (size_t)(n + 1) * 8, cudaMemcpyHostToDevice, c->stream));
  test_align_kernel<<<(n + 3) / 4, 128, 0, c->stream>>>(op, dA, dAo, dB, dBo, n, aux, aux2, c->params.K, dAr, arenaBytes, dR);
  CUDA_TRY(c, cudaGetLastError());
  CUDA_TRY(c, cudaMemcpyAsync(result, dR, rn * 4, cudaMemcpyDeviceToHost, c->stream));
  CUDA_TRY(c, cudaStreamSynchronize(c->stream));
  cudaFree(dA); cudaFree(dB); cudaFree(dAo); cudaFree(dBo); cudaFree(dAr); cudaFree(dR);
  return TALC_OK;
}

int talc_test_sort(talc_ctx* c, const int64_t* keys, uint32_t n, uint32_t* perm) {
  if (!c || !n) return TALC_ERR_ARG;
  CUDA_TRY(c, cudaSetDevice(c->device));
  i64* dK;
  u32* dP;
  CUDA_TRY(c, cudaMalloc((void**)&dK, (size_t)n * 8));
  CUDA_TRY(c, cudaMalloc((void**)&dP, (size_t)n * 4));
  CUDA_TRY(c, cudaMemcpyAsync(dK, keys, (size_t)n * 8, cudaMemcpyHostToDevice, c->stream));
  void* dS;
  CUDA_TRY(c, cudaMalloc(&dS, (size_t)n * sizeof(SortKey)));
  test_sort_kernel<<<1, 32, 0, c->stream>>>(dK, n, dP, dS);
  CUDA_TRY(c, cudaGetLastError());
  CUDA_TRY(c, cudaMemcpyAsync(perm, dP, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
  CUDA_TRY(c, cudaStreamSynchronize(c->stream));
  cudaFree(dK); cudaFree(dP); cudaFree(dS);
  return TALC_OK;
}

}  // extern "C"

#include "stream.hpp"
#include "replicate.hpp"
