// strand_emu.cpp -- --strand auto's per-read decision through the product's TALC_HD helpers (strand_roll_push,
// strand_decide, table_lookup) compiled with g++, so that it can be held against numpy without a GPU.  TEST AID ONLY:
// nothing in the shipped library links this file, and the product has no CPU path.
#include <stdint.h>

#include <vector>

#include "../../talc_b200/csrc/table.cuh"

using namespace talc;

extern "C" {

// The table as the device holds it: pair-aligned linear probing over 16-byte slots, keys with count >= min_count,
// first occurrence wins (the junction colours do not enter the decision).  Then, per read: strand, found_fwd, found_rc.
void emu_orient_reads(uint32_t K, uint32_t min_count, const uint64_t* keys, const int64_t* counts, uint64_t n_keys,
                      const uint8_t* bases, const uint64_t* offsets, uint32_t n_reads, uint8_t* strand,
                      uint32_t* found_fwd, uint32_t* found_rc) {
  u64 cap = 2;
  while (cap < 2 * n_keys + 2) cap <<= 1;
  std::vector<Slot> slots(cap, Slot{kEmptyKey, 0, 0});
  for (u64 i = 0; i < n_keys; ++i) {
    if ((u32)(int)counts[i] < min_count) continue;
    u64 b = hash_kmer(keys[i]) & (cap - 1) & ~1ull;
    for (bool placed = false; !placed; b = (b + 2) & (cap - 1)) {
      for (int j = 0; j < 2 && !placed; ++j) {
        Slot& s = slots[b + j];
        if (s.key == keys[i]) placed = true;
        else if (s.key == kEmptyKey) { s = Slot{keys[i], (u32)(int)counts[i], 0}; placed = true; }
      }
    }
  }
  TableView tv{slots.data(), cap - 1};
  for (u32 r = 0; r < n_reads; ++r) {
    const u8* s = bases + offsets[r];
    const u32 len = (u32)(offsets[r + 1] - offsets[r]);
    u32 nF = 0, nR = 0;
    StrandRoll st = strand_roll_start();
    for (u32 i = 0; i < len; ++i) {
      strand_roll_push(st, s[i], K);
      if (i + 1 < K) continue;
      u32 c = 0, col = 0;
      if (st.runF >= K && table_lookup(tv, st.fwd, c, col) && c != 0) ++nF;
      c = 0;
      if (st.runR >= K && table_lookup(tv, st.rc, c, col) && c != 0) ++nR;
    }
    strand[r] = (u8)strand_decide(nF, nR);
    found_fwd[r] = nF;
    found_rc[r] = nR;
  }
}

}  // extern "C"
