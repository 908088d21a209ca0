// walk.cuh -- the graph walk of long single-successor stretches, ONE TRAIL PER LANE (device only).
//
// ~97 % of all walk steps (oneMoreStep / oneMoreStepInTheDark, Explorer.cpp:546-687) are ordinary: every trail of a
// frontier of 1..7 trails has exactly one admissible successor, reaches no aim, closes no cycle, and nothing is due to
// be scored or pruned.  Inside the per-read program (correct.cuh, one WARP per read) such a step costs a whole warp
// ~400 instructions for one dependent table probe.  Here the frontiers of different reads walk side by side: a group
// of 8 lanes owns one frontier (lane t = trail t), four frontiers share a warp's instruction stream, and a block of
// this kernel needs 40 registers per thread instead of 241, so an SM holds hundreds of dependent probe chains instead
// of eight.  The per-read program suspends where a long walk starts (Corrector::search_bridge / search_edge return
// kStepYield with the request in Corrector::wq), this kernel advances cur[] / the packed trail sequences / the
// counters in the read's context in HBM, and the control kernel resumes the read from its frames.
//
// The step is the one of Corrector::fast_walk, statement for statement (same probe, same tagger for the rare
// multi-successor bucket, same aim / cycle tests, same double arithmetic in the same order), and like it ends the run
// BEFORE any step that is not ordinary -- the general step of the per-read program then takes that step in full, so
// the result cannot depend on where a run was cut (asserted by the parity tests and by the host emulation of the
// suspend / resume protocol, tests/test_hostemu.py::test_suspend_and_resume_is_result_neutral).
#pragma once
#include "correct.cuh"

namespace talc {

// a read in flight: its program state, its tallies, and which read it is
struct __attribute__((aligned(16))) ReadCtx {
  Corrector cx;
  Counters ctr;
  u32 read;  // index of the read in the batch, kCtxFree when the context is idle
  u32 pad[3];
};
static const u32 kCtxFree = 0xFFFFFFFFu;

#if defined(__CUDACC__)
__device__ __noinline__ double walk_sqrt_cold(u32 c) { return sqrt((double)c); }

__global__ void __launch_bounds__(256) walk_kernel(ReadCtx* __restrict__ ctxs, const u32* __restrict__ walkList, const u32* __restrict__ nWalk,
                                                   u32* __restrict__ readyList, u32* __restrict__ nReady, u32 stepCap) {
#if defined(__CUDA_ARCH__)  // ctx_lookup exists in the device pass only
  const u32 lane = threadIdx.x & 31u, gl = lane & 7u, gbase = lane & ~7u;
  const u32 gmask = 0xFFu << gbase;
  const u32 group = (blockIdx.x * blockDim.x + threadIdx.x) >> 3, nGroups = (gridDim.x * blockDim.x) >> 3;
  const u32 n = *nWalk;
  for (u32 j = group; j < n; j += nGroups) {
    const u32 id = walkList[j];
    ReadCtx* rc = ctxs + id;
    Corrector& cx = rc->cx;  // in HBM; every lane of the group reads the same words
    if (cx.wq.border == 2) {  // a pause, not a walk (Corrector::should_pause): straight back to the control kernel
      if (gl == 0) {
        const u32 pos = atomicAdd(nReady, 1u);
        readyList[pos] = id;
      }
      continue;
    }
    const u32 nT = cx.nCur;
    const bool act = gl < nT;
    const Params P = cx.P;
    const ModelTabs tabs = cx.tabs;
    const u32 k = P.K;
    const bool right = cx.dirRight;
    const bool border = cx.wq.border != 0;
    const CtxView cv = right ? cx.CR : cx.CL;
    const u64 kmask = kmer_mask(k), cmask = kmer_mask(k - 1);
    const u32 stride = (P.cycle_mode == 0) ? k : 1u;
    const u32 pathMax = cx.wq.pathMax, nAims = cx.wq.nAims;
    const AnchorRec* aims = cx.wq.aims;
    // the aim k-mers spread over the 8 lanes of the group (at most 32: walk_eligible); ~0 is not a k-mer (<= 62 bits)
    u64 myAim[4];
#pragma unroll
    for (u32 i = 0; i < 4; ++i) {
      const u32 a = gl + 8u * i;
      myAim[i] = (!border && a < nAims) ? aims[a].kmer : ~0ull;
    }
    Trail* curp = cx.cur;
    const Trail tr = curp[act ? gl : 0];
    u64* const w = cx.slotPool + (u64)tr.slot * cx.slotWords;
    u64 kmer = tr.kmer;
    u32 count = tr.count;
    double dsum = tr.dist;
    u64 rkmer = 0;  // the last k-mer with its bases in reverse order (LEFT walks compare in walk order)
    TALC_ROLLED
    for (u32 i = 0; i < k; ++i) rkmer |= ((kmer >> (2 * i)) & 3ull) << (2 * (k - 1 - i));
    u32 st = cx.wq.step, nSteps = 0;
    const u32 topShift = 2 * (k - 1);
    u32 untilCheck = border ? (kCheckInterval - 1u - (st % kCheckInterval)) : ~0u;  // steps before scoreEdges is due
#pragma unroll 1
    while (st < pathMax) {
      if (untilCheck == 0) break;  // border: (st + 1) % kCheckInterval == 0, scoreEdges is due after this step
      if (nSteps >= stepCap) break;
      const u32 plen = k + st;
      // ---- the four successors of every trail: one sector per trail
      int child = -1;
      u32 childCnt = 0;
      if (act) {
        u32 c4[4], cm;
        ctx_lookup(cv, right ? (kmer & cmask) : (kmer >> 2), c4, cm);
        child = fast_step_child(c4, cm, count, P, tabs);
        const u32 ch0 = (u32)(child < 0 ? 0 : child);
        childCnt = ch0 == 0 ? c4[0] : ch0 == 1 ? c4[1] : ch0 == 2 ? c4[2] : c4[3];
      }
      if (__ballot_sync(gmask, act && child < 0) & gmask) break;  // dead end or branching somewhere: general step
      const u32 ch = (u32)(child < 0 ? 0 : child);
      const u64 ck = right ? (((kmer << 2) | (u64)ch) & kmask) : ((kmer >> 2) | ((u64)ch << topShift));
      if (!border) {  // aim reached by any trail: the general step records the bridge
        bool aim = false;
#pragma unroll 1
        for (u32 q = 0; q < nT; ++q) {
          const u64 cq = __shfl_sync(gmask, ck, gbase + q);
          aim |= (myAim[0] == cq) | (myAim[1] == cq) | (myAim[2] == cq) | (myAim[3] == cq);
        }
        if (__ballot_sync(gmask, aim) & gmask) break;
      }
      // ---- cycle test of every trail against its own sequence, one window per lane of the group
      if (plen > k) {
        const u64 myNeedle = right ? ck : (((rkmer << 2) | (u64)ch) & kmask);
        bool cyc = false;
        TALC_ROLLED
        for (u32 q = 0; q < nT && !cyc; ++q) {
          const u64 needle = __shfl_sync(gmask, myNeedle, gbase + q);
          const u64* wq = (const u64*)__shfl_sync(gmask, (unsigned long long)w, gbase + q);
          TALC_ROLLED
          for (u32 base = 0; (u64)base * stride + k <= plen; base += 8) {
            const u32 p = (base + gl) * stride;
            bool match = false;
            if (p + k <= plen) match = path_kmer_fwd(wq, right ? p : (plen - k - p), k) == needle;
            const u32 mm = (__ballot_sync(gmask, match) >> gbase) & 0xFFu;
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
        if (count != childCnt) {  // a zero numerator adds +0.0
          const double sq = (count < tabs.n) ? tabs.sq[count] : walk_sqrt_cold(count);
          dsum = dsum + fabs((double)count - (double)childCnt) / sq;
        }
      }
      __syncwarp(gmask);  // the appended bases are visible to the group's next cycle test
      if (!right) rkmer = ((rkmer << 2) | (u64)ch) & kmask;
      kmer = ck;
      count = childCnt;
      ++st;
      ++nSteps;
      --untilCheck;
    }
    __syncwarp(gmask);
    if (nSteps && act) {
      curp[gl].kmer = kmer;
      curp[gl].count = count;
      curp[gl].dist = dsum;
    }
    if (gl == 0) {
      if (nSteps) {
        if (border) rc->ctr.steps_border += nSteps;
        else rc->ctr.steps_inner += nSteps;
        rc->ctr.frontier_sum += (u64)nSteps * nT;
        rc->ctr.lookups_walk += 4ull * nSteps * nT;
      }
      cx.wq.step = st;
      const u32 pos = atomicAdd(nReady, 1u);
      readyList[pos] = id;
    }
    __syncwarp(gmask);
  }
#endif
}
#endif

}  // namespace talc
