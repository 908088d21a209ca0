// pieces_io_test.cpp -- a C entry point around format_pieces (talc_b200/csrc/host/reads_io.hpp) for tests/test_pieces.py
// (no GPU): the --trim / --split records of one batch, formatted exactly as talc_main.cpp formats them.
#include "../../talc_b200/csrc/host/reads_io.hpp"

extern "C" {

// n records: ids joined with '\n', sequences out[ooffs[r] .. ooffs[r+1]), pieces piece_off[n+1] / bounds.  Returns the
// number of bytes written to dst (-1 if dst_cap is too small); tally[3] = reads kept, pieces, bases.
long pio_format(const char* ids, long n, const unsigned char* out, const unsigned long long* ooffs,
                const unsigned long long* piece_off, const unsigned* bounds, int split, unsigned min_len, char* dst, long dst_cap,
                unsigned long long* tally) {
  Batch b;
  const char* p = ids;
  for (long r = 0; r < n; ++r) {
    const char* e = strchr(p, '\n');
    b.ids.emplace_back(p, e ? (size_t)(e - p) : strlen(p));
    p = e ? e + 1 : p + strlen(p);
  }
  std::vector<uint64_t> oo(ooffs, ooffs + n + 1), po(piece_off, piece_off + n + 1);
  std::string buf;
  PieceTally t;
  format_pieces(b, out, oo.data(), po.data(), bounds, split != 0, min_len, buf, t);
  tally[0] = t.reads;
  tally[1] = t.pieces;
  tally[2] = t.bases;
  if ((long)buf.size() > dst_cap) return -1;
  memcpy(dst, buf.data(), buf.size());
  return (long)buf.size();
}

}  // extern "C"
