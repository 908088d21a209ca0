// stream.hpp -- batches of reads streamed through one context with copies, kernels and the caller's own work
// overlapped (SURVEY row f2; replaces the load-everything / write-everything shape of main.cpp:219,310).
//
//   caller thread        talc_stream_submit(i+1): copy into pinned staging, async H2D on the copy-in stream
//   worker thread        batch i: coverage + correction kernels on the context's stream, then async D2H on the
//                        copy-out stream
//   caller thread        talc_stream_next(i-1): pinned result buffers, formatted / written by the caller
//
// A ring of kSlots (= lanes + 2) slots bounds host and device memory whatever the number of reads; results come back in
// submission order.  Included at the end of talc_b200.cu (same translation unit as the context).
#pragma once
#include <condition_variable>
#include <mutex>
#include <sys/mman.h>
#include <thread>

// Page-locked host staging.  Large buffers are anonymous mappings advised to use huge pages and then registered:
// measured on the B200 hosts, 1 GiB costs 0.13-0.16 s that way against 0.47 s through cudaHostAlloc (4 KB pages), and
// copies from it run at the same 56 GB/s (tools/probes/pin_probe.cu).
struct PinBuf {
  void* p = nullptr;
  size_t cap = 0;
  bool mapped = false;  // mmap + cudaHostRegister (else cudaHostAlloc)
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    release();
    size_t want = bytes + bytes / 8 + 4096;
    if (want >= (4u << 20)) {
      want = (want + (2u << 20) - 1) & ~(size_t)((2u << 20) - 1);
      void* q = mmap(nullptr, want, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0);
      if (q != MAP_FAILED) {
        madvise(q, want, MADV_HUGEPAGE);  // advisory: 4 KB pages still work
        if (cudaHostRegister(q, want, cudaHostRegisterPortable) == cudaSuccess) {
          p = q;
          cap = want;
          mapped = true;
          return cudaSuccess;
        }
        (void)cudaGetLastError();
        munmap(q, want);
      }
    }
    cudaError_t e = cudaHostAlloc(&p, want, cudaHostAllocDefault);
    if (e == cudaSuccess) cap = want;
    else p = nullptr;
    return e;
  }
  void release() {
    if (p && mapped) {
      cudaHostUnregister(p);
      munmap(p, cap);
    } else if (p) {
      cudaFreeHost(p);
    }
    p = nullptr;
    cap = 0;
    mapped = false;
  }
};

struct StreamSlot {
  PinBuf hBases, hOffs, hOut, hOutOffs, hStatus, hStats, hStrand, hPieceOff, hBounds;
  DevBuf dBases, dOffs, dOut, dOutOffs, dStatus, dStats, dStrand;
  bool strandAuto = false;  // the batch ran in TALC_STRAND_AUTO: hStrand holds its strands
  bool pieces = false;      // the batch ran with pieces on: hPieceOff / hBounds hold them
  cudaEvent_t h2dDone = nullptr, d2hDone = nullptr;
  u32 n = 0;
  u64 totalBases = 0;
  talc_counters ctr;
  int rc = 0;
  std::string err;
  int state = 0;  // 0 free, 1 submitted, 2 done (D2H in flight or complete), 3 held by the caller
};

struct talc_stream {
  static const int kMaxLanes = 4;
  int kSlots = 4;  // lanes + 2: one batch being filled, one per lane on the device, one held by the caller
  talc_ctx* c = nullptr;
  // Two batches may be on the device at once ("lanes"): the kernels of batch i+1 are queued on their own stream with
  // their own scratch while batch i runs, so that its blocks start on the SMs that the last, longest reads of batch i
  // no longer fill (the per-read program is one warp per read: a batch ends with a tail of a few long reads).  Lane 0
  // is the caller's context, lane 1 a lane of it (talc_ctx_create_lane).
  talc_ctx* lane[kMaxLanes] = {nullptr, nullptr, nullptr, nullptr};
  int nLanes = 1;
  bool wantStats = false;
  std::vector<StreamSlot> slot;
  cudaStream_t copyIn = nullptr, copyOut = nullptr;
  std::thread worker[kMaxLanes];
  std::mutex mu;
  std::condition_variable cv;
  u64 seqSubmit = 0, seqFetch = 0;
  bool closing = false;
  std::string err;
};

static void stream_worker(talc_stream* s, int w) {
  talc_ctx* c = s->lane[w];
  cudaSetDevice(c->device);
  for (u64 seq = (u64)w;; seq += (u64)s->nLanes) {
    StreamSlot* sl = &s->slot[seq % s->kSlots];
    {
      std::unique_lock<std::mutex> lk(s->mu);
      // the slot of batch `seq` is in state 1 only once that very batch has been submitted: its previous tenant
      // (seq - kSlots) has been fetched and released by then
      s->cv.wait(lk, [&] { return s->closing || (s->seqSubmit > seq && sl->state == 1); });
      if (!(s->seqSubmit > seq && sl->state == 1)) return;  // closing and nothing left to run
    }
    int rc = TALC_OK;
    cudaError_t e = cudaStreamWaitEvent(c->stream, sl->h2dDone, 0);
    if (e != cudaSuccess) rc = TALC_ERR_CUDA;
    const bool strandAuto = c->parent ? c->parent->strand == TALC_STRAND_AUTO : c->strand == TALC_STRAND_AUTO;
    if (rc == TALC_OK && strandAuto && (sl->dStrand.reserve(sl->n + 1) != cudaSuccess || sl->hStrand.reserve(sl->n + 1) != cudaSuccess)) {
      rc = TALC_ERR_CUDA;
      c->err = "out of pinned host or device memory for the strands of a batch";
    }
    if (rc == TALC_OK)
      rc = correct_batch_device_impl(c, (const u8*)sl->dBases.p, (const u64*)sl->dOffs.p, sl->n, sl->totalBases, (u8*)sl->dOut.p,
                                     sl->dOut.cap, (u64*)sl->dOutOffs.p, (u8*)sl->dStatus.p, &sl->ctr,
                                     s->wantStats ? (u32*)sl->dStats.p : nullptr, strandAuto ? (u8*)sl->dStrand.p : nullptr);
    sl->strandAuto = rc == TALC_OK && c->lastAuto;
    sl->pieces = rc == TALC_OK && c->lastPieces;
    if (sl->pieces) {
      // the pieces are small (8 bytes a read and a piece) and the context's buffers serve the next batch of this
      // lane: copied out here, on the lane's idle stream, before the next batch is queued
      const u64 total = c->lastPiecesTotal;
      if (sl->hPieceOff.reserve((size_t)(sl->n + 1) * 8) != cudaSuccess || sl->hBounds.reserve((size_t)total * 8 + 8) != cudaSuccess) {
        rc = TALC_ERR_CUDA;
        c->err = "out of pinned host memory for the pieces of a batch";
      } else {
        u64 got = 0;
        rc = talc_last_pieces(c, (uint64_t*)sl->hPieceOff.p, (uint32_t*)sl->hBounds.p, total, &got);
      }
      sl->pieces = rc == TALC_OK;
    }
    if (rc == TALC_OK) {
      // this lane's compute stream is idle here (the call above ends with a synchronize): results leave on the
      // copy-out stream while the next batch computes
      const u64 totalOut = sl->n ? sl->ctr.bases_out : 0;
      bool ok = sl->hOut.reserve(totalOut + 64) == cudaSuccess;
      ok = ok && cudaMemcpyAsync(sl->hOutOffs.p, sl->dOutOffs.p, (size_t)(sl->n + 1) * 8, cudaMemcpyDeviceToHost, s->copyOut) == cudaSuccess;
      if (ok && sl->n) {
        ok = cudaMemcpyAsync(sl->hStatus.p, sl->dStatus.p, sl->n, cudaMemcpyDeviceToHost, s->copyOut) == cudaSuccess;
        if (ok && totalOut) ok = cudaMemcpyAsync(sl->hOut.p, sl->dOut.p, totalOut, cudaMemcpyDeviceToHost, s->copyOut) == cudaSuccess;
        if (ok && s->wantStats)
          ok = cudaMemcpyAsync(sl->hStats.p, sl->dStats.p, (size_t)sl->n * 8, cudaMemcpyDeviceToHost, s->copyOut) == cudaSuccess;
        if (ok && sl->strandAuto)
          ok = cudaMemcpyAsync(sl->hStrand.p, sl->dStrand.p, sl->n, cudaMemcpyDeviceToHost, s->copyOut) == cudaSuccess;
      }
      ok = ok && cudaEventRecord(sl->d2hDone, s->copyOut) == cudaSuccess;
      if (!ok) { rc = TALC_ERR_CUDA; sl->err = "device-to-host copy of a batch failed"; }
    } else {
      sl->err = c->err;
    }
    {
      std::lock_guard<std::mutex> lk(s->mu);
      sl->rc = rc;
      sl->state = 2;
    }
    s->cv.notify_all();
  }
}

extern "C" {

int talc_stream_open(talc_ctx* c, int want_read_stats, talc_stream** out) {
  if (!c || !out) return TALC_ERR_ARG;
  *out = nullptr;
  CUDA_TRY(c, cudaSetDevice(c->device));  // the table may still be loading: it is only needed when a batch runs
  talc_stream* s = new talc_stream;
  s->c = c;
  s->wantStats = want_read_stats != 0;
  s->lane[0] = c;
  int want = 2;  // TALC_STREAM_LANES = 1 .. 4 (1 = one batch at a time, for A/B measurements; 3 or 4 for heavy-tailed inputs)
  if (const char* e = getenv("TALC_STREAM_LANES")) want = std::min(std::max(atoi(e), 1), (int)talc_stream::kMaxLanes);
  if (c->parent) want = 1;  // the caller's context is a lane itself
  s->nLanes = 1;
  while (s->nLanes < want && talc_ctx_create_lane(c, &s->lane[s->nLanes]) == TALC_OK) s->nLanes++;  // fewer if memory is short
  s->kSlots = s->nLanes + 2;
  s->slot = std::vector<StreamSlot>((size_t)s->kSlots);
  bool ok = cudaStreamCreateWithFlags(&s->copyIn, cudaStreamNonBlocking) == cudaSuccess &&
            cudaStreamCreateWithFlags(&s->copyOut, cudaStreamNonBlocking) == cudaSuccess;
  for (auto& sl : s->slot)
    ok = ok && cudaEventCreateWithFlags(&sl.h2dDone, cudaEventDisableTiming) == cudaSuccess &&
         cudaEventCreateWithFlags(&sl.d2hDone, cudaEventDisableTiming) == cudaSuccess;
  if (!ok) {
    c->err = "talc_stream_open: cannot create CUDA streams / events";
    for (int w = 1; w < s->nLanes; ++w) talc_ctx_destroy(s->lane[w]);
    delete s;
    return TALC_ERR_CUDA;
  }
  for (int w = 0; w < s->nLanes; ++w) s->worker[w] = std::thread(stream_worker, s, w);
  *out = s;
  return TALC_OK;
}

// Optional: allocate the pinned host and device buffers of every slot now, for batches of up to max_reads reads and
// max_bases bases (page-locking hundreds of MB takes ~0.05 s per buffer and every other mapping call of the process
// queues behind it: better paid once, before the first batch, than by the first batches -- and not while a table
// loads or NCCL starts up, profiles/r02_summary.md).
int talc_stream_reserve(talc_stream* s, uint32_t max_reads, uint64_t max_bases) {
  if (!s) return TALC_ERR_ARG;
  talc_ctx* c = s->c;
  if (cudaSetDevice(c->device) != cudaSuccess) { s->err = "cudaSetDevice failed"; return TALC_ERR_CUDA; }
  const u64 outCap = 2 * max_bases + (u64)max_reads * 64 + 4096;
  for (auto& sl : s->slot) {
    bool ok = sl.hBases.reserve(max_bases + 64) == cudaSuccess && sl.hOffs.reserve((size_t)(max_reads + 1) * 8) == cudaSuccess &&
              sl.hOutOffs.reserve((size_t)(max_reads + 1) * 8) == cudaSuccess && sl.hStatus.reserve(max_reads + 1) == cudaSuccess &&
              sl.hOut.reserve(max_bases + max_bases / 16 + 64) == cudaSuccess && sl.dBases.reserve(max_bases + 64) == cudaSuccess &&
              sl.dOffs.reserve((size_t)(max_reads + 1) * 8) == cudaSuccess && sl.dOut.reserve(outCap) == cudaSuccess &&
              sl.dOutOffs.reserve((size_t)(max_reads + 1) * 8) == cudaSuccess && sl.dStatus.reserve(max_reads + 1) == cudaSuccess;
    if (ok && s->wantStats) ok = sl.hStats.reserve((size_t)max_reads * 8 + 8) == cudaSuccess && sl.dStats.reserve((size_t)max_reads * 8 + 8) == cudaSuccess;
    if (!ok) { s->err = "talc_stream_reserve: out of pinned host or device memory"; return TALC_ERR_CUDA; }
  }
  return TALC_OK;
}

// Blocks only while all slots are busy (back-pressure).  The caller's buffers are free again on return.
int talc_stream_submit(talc_stream* s, const uint8_t* bases, const uint64_t* offsets, uint32_t n) {
  if (!s || !offsets || (n && !bases) || offsets[0] != 0) return TALC_ERR_ARG;
  talc_ctx* c = s->c;
  StreamSlot* sl = &s->slot[s->seqSubmit % s->kSlots];
  {
    std::unique_lock<std::mutex> lk(s->mu);
    s->cv.wait(lk, [&] { return sl->state == 0; });
  }
  if (cudaSetDevice(c->device) != cudaSuccess) { s->err = "cudaSetDevice failed"; return TALC_ERR_CUDA; }
  const u64 total = offsets[n];
  const u64 outCap = 2 * total + (u64)n * 64 + 4096;
  bool ok = sl->hBases.reserve(total + 64) == cudaSuccess && sl->hOffs.reserve((size_t)(n + 1) * 8) == cudaSuccess &&
            sl->hOutOffs.reserve((size_t)(n + 1) * 8) == cudaSuccess && sl->hStatus.reserve(n + 1) == cudaSuccess &&
            sl->dBases.reserve(total + 64) == cudaSuccess && sl->dOffs.reserve((size_t)(n + 1) * 8) == cudaSuccess &&
            sl->dOut.reserve(outCap) == cudaSuccess && sl->dOutOffs.reserve((size_t)(n + 1) * 8) == cudaSuccess &&
            sl->dStatus.reserve(n + 1) == cudaSuccess;
  if (ok && s->wantStats) ok = sl->hStats.reserve((size_t)n * 8 + 8) == cudaSuccess && sl->dStats.reserve((size_t)n * 8 + 8) == cudaSuccess;
  if (!ok) { s->err = "talc_stream_submit: out of pinned host or device memory"; return TALC_ERR_CUDA; }
  memcpy(sl->hBases.p, bases, total);
  memcpy(sl->hOffs.p, offsets, (size_t)(n + 1) * 8);
  ok = (total == 0 || cudaMemcpyAsync(sl->dBases.p, sl->hBases.p, total, cudaMemcpyHostToDevice, s->copyIn) == cudaSuccess) &&
       cudaMemcpyAsync(sl->dOffs.p, sl->hOffs.p, (size_t)(n + 1) * 8, cudaMemcpyHostToDevice, s->copyIn) == cudaSuccess &&
       cudaEventRecord(sl->h2dDone, s->copyIn) == cudaSuccess;
  if (!ok) { s->err = "talc_stream_submit: host-to-device copy failed"; return TALC_ERR_CUDA; }
  sl->n = n;
  sl->totalBases = total;
  {
    std::lock_guard<std::mutex> lk(s->mu);
    sl->state = 1;
    s->seqSubmit++;
  }
  s->cv.notify_all();
  return TALC_OK;
}

uint64_t talc_stream_pending(talc_stream* s) {
  if (!s) return 0;
  std::lock_guard<std::mutex> lk(s->mu);
  return s->seqSubmit - s->seqFetch;
}

// Result of the oldest batch not yet fetched; blocks until it is complete.  The pointers stay valid until the next
// call to talc_stream_next / talc_stream_close.  read_stats (may be NULL) receives a pointer to n x {solid span,
// regions} when the stream was opened with want_read_stats.
int talc_stream_next(talc_stream* s, const uint8_t** out, const uint64_t** out_offsets, const uint8_t** status, uint32_t* n,
                     const uint32_t** read_stats, talc_counters* counters) {
  if (!s) return TALC_ERR_ARG;
  StreamSlot* sl;
  {
    std::unique_lock<std::mutex> lk(s->mu);
    if (s->seqFetch > 0) {  // release the slot handed out by the previous call
      StreamSlot* prev = &s->slot[(s->seqFetch - 1) % s->kSlots];
      if (prev->state == 3) prev->state = 0;
    }
    if (s->seqFetch == s->seqSubmit) {
      s->cv.notify_all();
      s->err = "talc_stream_next: nothing submitted";
      return TALC_ERR_ARG;
    }
    sl = &s->slot[s->seqFetch % s->kSlots];
    s->cv.notify_all();
    s->cv.wait(lk, [&] { return sl->state == 2; });
    sl->state = 3;
    s->seqFetch++;
  }
  if (sl->rc != TALC_OK) {
    s->err = sl->err;
    return sl->rc;
  }
  cudaSetDevice(s->c->device);
  if (cudaEventSynchronize(sl->d2hDone) != cudaSuccess) { s->err = "talc_stream_next: copy-out failed"; return TALC_ERR_CUDA; }
  if (out) *out = (const uint8_t*)sl->hOut.p;
  if (out_offsets) *out_offsets = (const uint64_t*)sl->hOutOffs.p;
  if (status) *status = (const uint8_t*)sl->hStatus.p;
  if (n) *n = sl->n;
  if (read_stats) *read_stats = s->wantStats ? (const uint32_t*)sl->hStats.p : nullptr;
  if (counters) *counters = sl->ctr;
  return TALC_OK;
}

// the slot handed out by the last talc_stream_next stays in state 3 until the following call
int talc_stream_pieces(talc_stream* s, const uint64_t** piece_off, const uint32_t** bounds) {
  if (!s || !piece_off || !bounds) return TALC_ERR_ARG;
  std::lock_guard<std::mutex> lk(s->mu);
  if (s->seqFetch == 0) { s->err = "talc_stream_pieces: no batch returned yet"; return TALC_ERR_ARG; }
  const StreamSlot* sl = &s->slot[(s->seqFetch - 1) % s->kSlots];
  const bool ok = sl->state == 3 && sl->rc == TALC_OK && sl->pieces;
  *piece_off = ok ? (const uint64_t*)sl->hPieceOff.p : nullptr;
  *bounds = ok ? (const uint32_t*)sl->hBounds.p : nullptr;
  return TALC_OK;
}

int talc_stream_strands(talc_stream* s, const uint8_t** strand) {
  if (!s || !strand) return TALC_ERR_ARG;
  std::lock_guard<std::mutex> lk(s->mu);
  if (s->seqFetch == 0) { s->err = "talc_stream_strands: no batch returned yet"; return TALC_ERR_ARG; }
  const StreamSlot* sl = &s->slot[(s->seqFetch - 1) % s->kSlots];
  *strand = (sl->state == 3 && sl->rc == TALC_OK && sl->strandAuto) ? (const uint8_t*)sl->hStrand.p : nullptr;
  return TALC_OK;
}

const char* talc_stream_last_error(talc_stream* s) { return s ? s->err.c_str() : ""; }

void talc_stream_close(talc_stream* s) {
  if (!s) return;
  {
    std::lock_guard<std::mutex> lk(s->mu);
    s->closing = true;
  }
  s->cv.notify_all();
  for (auto& t : s->worker)
    if (t.joinable()) t.join();
  for (int w = 1; w < s->nLanes; ++w) talc_ctx_destroy(s->lane[w]);
  cudaSetDevice(s->c->device);
  cudaStreamSynchronize(s->copyIn);
  cudaStreamSynchronize(s->copyOut);
  for (auto& sl : s->slot) {
    PinBuf* hb[] = {&sl.hBases, &sl.hOffs, &sl.hOut, &sl.hOutOffs, &sl.hStatus, &sl.hStats, &sl.hStrand, &sl.hPieceOff, &sl.hBounds};
    for (PinBuf* b : hb) b->release();
    DevBuf* db[] = {&sl.dBases, &sl.dOffs, &sl.dOut, &sl.dOutOffs, &sl.dStatus, &sl.dStats, &sl.dStrand};
    for (DevBuf* b : db) b->release();
    if (sl.h2dDone) cudaEventDestroy(sl.h2dDone);
    if (sl.d2hDone) cudaEventDestroy(sl.d2hDone);
  }
  cudaStreamDestroy(s->copyIn);
  cudaStreamDestroy(s->copyOut);
  delete s;
}

}  // extern "C"
