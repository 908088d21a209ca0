// dump_gpu.cuh -- Jellyfish `dump -c` text parsed on the GPU (SURVEY row f1: at 30 M+ lines the getline /
// istringstream / stoi loop of buildCDBG, Jellyfish.cpp:251-269, dominates start-up once correction is fast).
//
// The file goes to HBM through two pinned staging buffers (read and copy overlapped), then
//   line_flag_kernel      one flag per byte: does a line start here?          (streaming, 1 B read + 1 B written per byte)
//   cub::DeviceSelect     the start offsets of all lines, in file order
//   parse_lines_kernel    one thread per line: the two tokens, std::stoi semantics, 2-bit packing
// and the entries stay on the device, indexed by LINE NUMBER (filtered and malformed lines hold kEmptyKey), which is
// what table_insert_kernel needs for "first line wins" (Jellyfish.cpp:262) without any compaction.
//
// Line semantics are those of csrc/dump_parse.hpp (the host parser of round 1, kept for A/B timing): two
// whitespace-separated tokens, anything after them ignored; a count that std::stoi would reject makes the line bad;
// k-mers that are not exactly K letters of ACGT(U), either case, are dropped.
#pragma once
#include <cub/cub.cuh>
#include <thrust/iterator/counting_iterator.h>

#include "defs.cuh"
#include "table.cuh"

namespace talc {

struct DumpCounts {
  unsigned long long lines, bad, dropped, kept;
};

__global__ void line_flag_kernel(const char* __restrict__ text, u64 size, u8* __restrict__ flag, unsigned long long* nLines) {
  const u64 stride = (u64)gridDim.x * blockDim.x;
  u32 mine = 0;
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < size; i += stride) {
    const u8 f = (i == 0 || text[i - 1] == '\n') ? 1 : 0;
    flag[i] = f;
    mine += f;
  }
  mine = __reduce_add_sync(0xffffffffu, mine);
  if ((threadIdx.x & 31) == 0 && mine) atomicAdd(nLines, (unsigned long long)mine);
}

__device__ __forceinline__ bool dump_is_ws(char c) { return c == ' ' || c == '\t' || c == '\r' || c == '\v' || c == '\f'; }

__global__ void parse_lines_kernel(const char* __restrict__ text, u64 size, const u64* __restrict__ starts, u64 nLines, u32 K,
                                   u32 minCount, int filter, u64* __restrict__ keys, u32* __restrict__ counts, DumpCounts* tally) {
  const u64 stride = (u64)gridDim.x * blockDim.x;
  unsigned long long lines = 0, bad = 0, dropped = 0, kept = 0;
  for (u64 li = (u64)blockIdx.x * blockDim.x + threadIdx.x; li < nLines; li += stride) {
    const u64 p = starts[li];
    u64 eol = (li + 1 < nLines) ? starts[li + 1] - 1 : size;  // position of '\n', or the end of an unterminated last line
    if (li + 1 == nLines && size > 0 && text[size - 1] == '\n') eol = size - 1;
    u64 key = kEmptyKey;
    u32 cnt = 0;
    u64 q = p;
    while (q < eol && dump_is_ws(text[q])) ++q;
    const u64 k0 = q;
    while (q < eol && !dump_is_ws(text[q])) ++q;
    const u64 k1 = q;
    while (q < eol && dump_is_ws(text[q])) ++q;
    const u64 c0 = q;
    while (q < eol && !dump_is_ws(text[q])) ++q;
    const u64 c1 = q;
    if (k1 > k0 && c1 > c0) {
      u64 d = c0;
      bool neg = false;
      if (text[d] == '+' || text[d] == '-') { neg = text[d] == '-'; ++d; }
      if (d < c1 && text[d] >= '0' && text[d] <= '9') {  // std::stoi
        i64 v = 0;
        bool rangeOk = true;
        while (d < c1 && text[d] >= '0' && text[d] <= '9') {
          v = v * 10 + (text[d] - '0');
          if (v > 2147483648LL) { rangeOk = false; break; }
          ++d;
        }
        if (neg) v = -v;
        if (rangeOk && v <= 2147483647LL) {
          ++lines;
          const bool keep = !filter || ((u32)(i32)v >= minCount);  // compared as unsigned (Jellyfish.cpp:260)
          if (keep) {
            bool ok = (k1 - k0) == K;
            u64 kk = 0;
            for (u64 s = k0; ok && s < k1; ++s) {
              const u32 c = base_code((u8)text[s]);
              ok = c < 4;
              kk = (kk << 2) | (c & 3);
            }
            if (ok) { key = kk; cnt = (u32)(i32)v; ++kept; }
            else ++dropped;
          }
        } else ++bad;
      } else ++bad;
    } else ++bad;  // fewer than two tokens (an empty line included)
    keys[li] = key;
    counts[li] = cnt;
  }
  // one atomic per warp and counter
  lines = __reduce_add_sync(0xffffffffu, (u32)lines);
  bad = __reduce_add_sync(0xffffffffu, (u32)bad);
  dropped = __reduce_add_sync(0xffffffffu, (u32)dropped);
  kept = __reduce_add_sync(0xffffffffu, (u32)kept);
  if ((threadIdx.x & 31) == 0) {
    if (lines) atomicAdd(&tally->lines, lines);
    if (bad) atomicAdd(&tally->bad, bad);
    if (dropped) atomicAdd(&tally->dropped, dropped);
    if (kept) atomicAdd(&tally->kept, kept);
  }
}

// A canonical dump (`jellyfish count -C`): line i (x, c) stands for the lines 2i (x, c) and 2i+1 (rc(x), c) of a
// directional dump, so that table_insert_kernel's "first line wins" applies to the expansion.  A dropped line (kEmptyKey)
// stays dropped on both.
__global__ void dump_expand_rc_kernel(const u64* __restrict__ keys, const u32* __restrict__ counts, u64 nLines, u32 K,
                                      u64* __restrict__ outKeys, u32* __restrict__ outCounts) {
  const u64 stride = (u64)gridDim.x * blockDim.x;
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < nLines; i += stride) {
    const u64 x = keys[i];
    const u32 v = counts[i];
    outKeys[2 * i] = x;
    outKeys[2 * i + 1] = x == kEmptyKey ? kEmptyKey : kmer_revcomp(x, K);
    outCounts[2 * i] = v;
    outCounts[2 * i + 1] = v;
  }
}

// the text of a file in HBM: fread into two pinned buffers, copies overlapped with the next read
static cudaError_t file_to_device(const char* path, cudaStream_t stream, char** dText, u64* size, std::string& err) {
  *dText = nullptr;
  *size = 0;
  FILE* f = fopen(path, "rb");
  if (!f) { err = std::string("cannot open ") + path; return cudaErrorUnknown; }
  struct stat st;
  if (fstat(fileno(f), &st) != 0) { fclose(f); err = std::string("cannot stat ") + path; return cudaErrorUnknown; }
  const u64 total = (u64)st.st_size;
  cudaError_t e = cudaMalloc((void**)dText, total + 16);
  if (e != cudaSuccess) { fclose(f); err = "cudaMalloc(dump text) failed"; return e; }
  const size_t piece = 32u << 20;
  char* pin[2] = {nullptr, nullptr};
  cudaEvent_t done[2];
  for (int i = 0; i < 2; ++i) {
    e = cudaHostAlloc((void**)&pin[i], piece, cudaHostAllocDefault);
    if (e != cudaSuccess) { err = "cudaHostAlloc(staging) failed"; break; }
    cudaEventCreateWithFlags(&done[i], cudaEventDisableTiming);
  }
  u64 off = 0;
  if (e == cudaSuccess) {
    for (int i = 0; off < total; i ^= 1) {
      cudaEventSynchronize(done[i]);  // the copy that last used this buffer (no-op the first time)
      const size_t n = fread(pin[i], 1, (size_t)std::min<u64>(piece, total - off), f);
      if (n == 0) break;
      e = cudaMemcpyAsync(*dText + off, pin[i], n, cudaMemcpyHostToDevice, stream);
      if (e != cudaSuccess) { err = "copy of the dump text failed"; break; }
      cudaEventRecord(done[i], stream);
      off += n;
    }
  }
  if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
  for (int i = 0; i < 2; ++i) {
    if (pin[i]) { cudaFreeHost(pin[i]); cudaEventDestroy(done[i]); }
  }
  fclose(f);
  if (e == cudaSuccess && off != total) { err = std::string("short read of ") + path; e = cudaErrorUnknown; }
  if (e != cudaSuccess) { cudaFree(*dText); *dText = nullptr; return e; }
  *size = total;
  return cudaSuccess;
}

struct DeviceDump {
  u64* keys = nullptr;    // one per line, kEmptyKey when the line carries no entry
  u32* counts = nullptr;
  u64 nLines = 0;         // physical lines
  DumpCounts tally{0, 0, 0, 0};
  void release() {
    if (keys) cudaFree(keys);
    if (counts) cudaFree(counts);
    keys = nullptr;
    counts = nullptr;
  }
};

// parse a dump file into per-line device arrays; `filter`: apply count >= minCount (the counts dump, not the junction dump)
static bool parse_dump_gpu(const char* path, u32 K, u32 minCount, bool filter, int sms, cudaStream_t stream, DeviceDump& out,
                           std::string& err) {
  char* dText = nullptr;
  u64 size = 0;
  if (file_to_device(path, stream, &dText, &size, err) != cudaSuccess) return false;
  if (size == 0) { cudaFree(dText); return true; }
  const int blocks = sms * 8;
  u8* dFlag = nullptr;
  u64* dStarts = nullptr;
  u64* dNum = nullptr;
  void* dTmp = nullptr;
  DumpCounts* dTally = nullptr;
  bool ok = cudaMalloc((void**)&dFlag, size) == cudaSuccess && cudaMalloc((void**)&dNum, 8) == cudaSuccess &&
            cudaMalloc((void**)&dTally, sizeof(DumpCounts)) == cudaSuccess;
  u64 nLines = 0;
  if (ok) {
    cudaMemsetAsync(dNum, 0, 8, stream);
    line_flag_kernel<<<blocks, 256, 0, stream>>>(dText, size, dFlag, (unsigned long long*)dNum);
    ok = cudaGetLastError() == cudaSuccess && cudaMemcpyAsync(&nLines, dNum, 8, cudaMemcpyDeviceToHost, stream) == cudaSuccess &&
         cudaStreamSynchronize(stream) == cudaSuccess;
  }
  if (ok && nLines) {
    ok = cudaMalloc((void**)&dStarts, nLines * 8) == cudaSuccess && cudaMalloc((void**)&out.keys, nLines * 8) == cudaSuccess &&
         cudaMalloc((void**)&out.counts, nLines * 4) == cudaSuccess;
    // start offsets of the lines in file order: stream compaction of the byte positions, 1 GiB of text at a time
    // (the selection's item count is a 32-bit int in older CUB releases)
    const u64 seg = 1ull << 30;
    size_t tmpBytes = 0;
    if (ok) {
      thrust::counting_iterator<u64> pos0(0);
      cub::DeviceSelect::Flagged(nullptr, tmpBytes, pos0, dFlag, dStarts, dNum, (int)std::min<u64>(seg, size), stream);
      ok = cudaMalloc(&dTmp, tmpBytes + 16) == cudaSuccess;
    }
    u64 written = 0;
    for (u64 s0 = 0; ok && s0 < size; s0 += seg) {
      const int n = (int)std::min<u64>(seg, size - s0);
      thrust::counting_iterator<u64> pos(s0);
      size_t tb = tmpBytes;
      u64 got = 0;
      ok = cub::DeviceSelect::Flagged(dTmp, tb, pos, dFlag + s0, dStarts + written, dNum, n, stream) == cudaSuccess &&
           cudaMemcpyAsync(&got, dNum, 8, cudaMemcpyDeviceToHost, stream) == cudaSuccess && cudaStreamSynchronize(stream) == cudaSuccess;
      written += got;
    }
    ok = ok && written == nLines;
    if (ok) {
      cudaMemsetAsync(dTally, 0, sizeof(DumpCounts), stream);
      parse_lines_kernel<<<blocks, 256, 0, stream>>>(dText, size, dStarts, nLines, K, minCount, filter ? 1 : 0, out.keys, out.counts, dTally);
      ok = cudaGetLastError() == cudaSuccess &&
           cudaMemcpyAsync(&out.tally, dTally, sizeof(DumpCounts), cudaMemcpyDeviceToHost, stream) == cudaSuccess &&
           cudaStreamSynchronize(stream) == cudaSuccess;
    }
  }
  out.nLines = nLines;
  if (dTmp) cudaFree(dTmp);
  if (dFlag) cudaFree(dFlag);
  if (dStarts) cudaFree(dStarts);
  if (dNum) cudaFree(dNum);
  if (dTally) cudaFree(dTally);
  cudaFree(dText);
  if (!ok) {
    err = std::string("GPU parse of ") + path + " failed: " + cudaGetErrorString(cudaGetLastError());
    out.release();
  }
  return ok;
}

}  // namespace talc
