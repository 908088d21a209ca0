// count_gpu.cuh -- k-mer counting on the GPU straight from short-read FASTQ / FASTA (SURVEY row f3).
//
// Replaces the external step the reference's README prescribes (README.md:33-55:
//   jellyfish count --mer K -s 100M -o out.jf reads_1.fq reads_2.fq ; jellyfish dump -c out.jf > out.dump
// -- NON-canonical counts: a k-mer and its reverse complement are counted apart, main.cpp:89) and the ~GB text round
// trip through buildCDBG: every window of K consecutive A/C/G/T (either case) of every read is one occurrence; a
// window holding any other letter is skipped.  The result is the table `dump | buildCDBG` would have produced:
// k-mers with count >= MIN_COUNT, colour 0 (junction colouring is applied afterwards exactly as for a dump).
//
// Files stream through two pinned staging buffers; a piece is cut at a record boundary, its line offsets are found as in
// dump_gpu.cuh, and one thread per sequence line rolls a 2-bit k-mer over the line and bumps an open-addressed counting
// table (16-byte slots, CAS on the key + atomicAdd on the count).  Formats: FASTQ with four lines per record and FASTA
// with one sequence line per record (what short-read pipelines write).  Each file has an orientation (SrOrient): a
// stranded library counts its antisense mates as their reverse complements, an unstranded one counts both strands.
#pragma once
#include "dump_gpu.cuh"

namespace talc {

// Orientation of a short-read file (TALC_SR_* of include/talc_b200.h): what is counted for each window x of a read.
enum SrOrient : int {
  kSrSense = 0,      // x (the reference's recipe)
  kSrAntisense = 1,  // rc(x): reads of the strand opposite to the transcripts (R1 of a dUTP library)
  kSrBoth = 2        // x and rc(x), once when x == rc(x): unstranded libraries, `jellyfish count -C` expanded
};

// one occurrence of `key`: claim its slot (CAS on the key) and bump the count; a full table raises *fail
__device__ __forceinline__ void count_bump(Slot* slots, u64 mask, u64 key, u32* fail) {
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
  if (!hit) { atomicExch(fail, 1u); return; }
  atomicAdd(&hit->count, 1u);
}

// sequence lines are those with li % period == 1.  The windows are the same in every orientation: K consecutive bases
// that base_code reads as A, C, G or T (U counts as T); ORIENT only chooses which key(s) a window adds.
template <int ORIENT>
__global__ void count_kmers_kernel(const char* __restrict__ text, u64 size, const u64* __restrict__ starts, u64 nLines, u32 period,
                                   u32 K, Slot* slots, u64 mask, unsigned long long* nKmers, u32* fail) {
  const u64 stride = (u64)gridDim.x * blockDim.x;
  const u64 kmask = kmer_mask(K);
  unsigned long long mine = 0;
  for (u64 li = (u64)blockIdx.x * blockDim.x + threadIdx.x; li < nLines; li += stride) {
    if (li % period != 1) continue;
    const u64 p = starts[li];
    u64 eol = (li + 1 < nLines) ? starts[li + 1] - 1 : size;
    if (li + 1 == nLines && size > 0 && text[size - 1] == '\n') eol = size - 1;
    u64 km = 0, rc = 0;
    u32 run = 0;  // consecutive valid bases
    for (u64 q = p; q < eol; ++q) {
      const char ch = text[q];
      if (ch == '\r') continue;
      const u32 c = base_code((u8)ch);
      if (c > 3) { run = 0; km = 0; continue; }
      km = ((km << 2) | c) & kmask;
      if (ORIENT != kSrSense) rc = kmer_roll_rc(rc, c, K);
      if (++run < K) continue;
      if (ORIENT != kSrAntisense) {
        ++mine;
        count_bump(slots, mask, km, fail);
      }
      if (ORIENT == kSrAntisense || (ORIENT == kSrBoth && rc != km)) {
        ++mine;
        count_bump(slots, mask, rc, fail);
      }
    }
  }
  mine = __reduce_add_sync(0xffffffffu, (u32)mine);
  if ((threadIdx.x & 31) == 0 && mine) atomicAdd(nKmers, mine);
}
__global__ void count_fill_empty_kernel(Slot* slots, u64 capacity) {
  const u64 stride = (u64)gridDim.x * blockDim.x;
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < capacity; i += stride) {
    slots[i].key = kEmptyKey;
    slots[i].count = 0;
    slots[i].colour = 0;
  }
}
__global__ void count_tally_kernel(const Slot* slots, u64 capacity, u32 minCount, unsigned long long* distinct, unsigned long long* kept) {
  const u64 stride = (u64)gridDim.x * blockDim.x;
  u32 d = 0, k = 0;
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < capacity; i += stride) {
    if (slots[i].key != kEmptyKey) {
      ++d;
      k += slots[i].count >= minCount ? 1 : 0;
    }
  }
  d = __reduce_add_sync(0xffffffffu, d);
  k = __reduce_add_sync(0xffffffffu, k);
  if ((threadIdx.x & 31) == 0) {
    if (d) atomicAdd(distinct, (unsigned long long)d);
    if (k) atomicAdd(kept, (unsigned long long)k);
  }
}
// counting table -> final table: every k-mer with count >= MIN_COUNT (keys are unique: a CAS claim and plain stores);
// counts beyond INT_MAX saturate (the dump's std::stoi could not have read them)
__global__ void count_rehash_kernel(const Slot* src, u64 srcCap, u32 minCount, Slot* dst, u64 mask, u32* fail) {
  const u64 stride = (u64)gridDim.x * blockDim.x;
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < srcCap; i += stride) {
    const Slot s = src[i];
    if (s.key == kEmptyKey || s.count < minCount) continue;
    u64 b = hash_kmer(s.key) & mask & ~1ull;
    Slot* hit = nullptr;
    for (u64 lap = 0; !hit && lap <= mask; lap += 2) {
      for (int j = 0; j < 2 && !hit; ++j) {
        Slot* t = dst + b + j;
        if (atomicCAS((unsigned long long*)&t->key, (unsigned long long)kEmptyKey, (unsigned long long)s.key) == kEmptyKey) hit = t;
      }
      b = (b + 2) & mask;
    }
    if (!hit) { atomicExch(fail, 1u); continue; }
    hit->count = s.count > 0x7FFFFFFFu ? 0x7FFFFFFFu : s.count;
    hit->colour = 0;
  }
}

}  // namespace talc
