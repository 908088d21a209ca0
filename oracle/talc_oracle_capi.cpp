// =============================================================================
// talc_oracle_capi.cpp -- C entry points over the CPU restatement, for ctypes.
// TEST INFRASTRUCTURE ONLY: loaded by tests/, __graft_entry__.smoke() and
// bench.py's cpu_baseline / --impl reference legs.  PARITY UNPINNED.
// =============================================================================
#include <omp.h>

#include <chrono>
#include <cstring>

#include "talc_oracle.hpp"

using namespace talc_oracle;

extern "C" {

struct orc_params {
  uint32_t K, MIN_COUNT, WINDOW_SIZE, MAX_NB_COMPETING_PATHS;
  double ALPHA, SR_ERROR_RATE, MIN_INNER_SCORE, MIN_BORDER_SCORE;
  int32_t cycle_mode, q11_zero_init;
};

static Params to_params(const orc_params* q) {
  Params p;
  p.K = q->K;
  p.MIN_COUNT = q->MIN_COUNT;
  p.WINDOW_SIZE = q->WINDOW_SIZE;
  p.MAX_NB_COMPETING_PATHS = q->MAX_NB_COMPETING_PATHS;
  p.ALPHA = q->ALPHA;
  p.SR_ERROR_RATE = q->SR_ERROR_RATE;
  p.MIN_INNER_SCORE = q->MIN_INNER_SCORE;
  p.MIN_BORDER_SCORE = q->MIN_BORDER_SCORE;
  p.cycle_mode = q->cycle_mode;
  p.q11_zero_init = q->q11_zero_init != 0;
  return p;
}

static std::string unpack(uint64_t key, unsigned K) {
  std::string s(K, 'A');
  for (unsigned i = 0; i < K; ++i) s[i] = "ACGT"[(key >> (2 * (K - 1 - i))) & 3];
  return s;
}

void* orc_table_new(int ordered) { return new Table(ordered != 0); }
void orc_table_free(void* t) { delete (Table*)t; }
uint64_t orc_table_size(void* t) { return ((Table*)t)->size(); }

// text dumps, exactly as the reference reads them
int orc_table_load_dump(void* t, const orc_params* q, const char* dump, const char* junctions) {
  Params p = to_params(q);
  build_cdbg(*(Table*)t, p, dump, junctions ? junctions : "", junctions != nullptr);
  return 0;
}

// 2-bit packed k-mers (first base in the most significant position), dump-line order
int orc_table_build_packed(void* t, const orc_params* q, const uint64_t* keys, const int64_t* counts, uint64_t n,
                           const uint64_t* jkeys, const int64_t* jcounts, uint64_t nj, int use_junctions) {
  Params p = to_params(q);
  std::vector<std::pair<std::string, long long>> km, jm;
  km.reserve(n);
  for (uint64_t i = 0; i < n; ++i) km.emplace_back(unpack(keys[i], p.K), counts[i]);
  for (uint64_t i = 0; i < nj; ++i) jm.emplace_back(unpack(jkeys[i], p.K), jcounts[i]);
  build_cdbg_from_lists(*(Table*)t, p, km, jm, use_junctions != 0);
  return 0;
}

// point lookup of an ASCII k-mer: returns 1 if present
int orc_table_lookup(void* t, const char* kmer, uint32_t* count, uint32_t* colour) {
  const CCount* e = ((Table*)t)->find(to_dna5(kmer));
  *count = e ? e->first : 0;
  *colour = e ? e->second : 0;
  return e != nullptr;
}

// per-read coverage vector (Read.cpp:174-195); returns number of k-mers
uint64_t orc_coverage(void* t, uint32_t K, const char* seq, uint64_t len, uint32_t* counts, uint32_t* colours) {
  Seq s = to_dna5(std::string(seq, len));
  if (len < K) return 0;
  Table* T = (Table*)t;
  uint64_t n = len - K + 1;
  for (uint64_t i = 0; i < n; ++i) {
    const CCount* e = T->find(s.substr(i, K));
    counts[i] = e ? e->first : 0;
    colours[i] = e ? e->second : 0;
  }
  return n;
}

// Batch correction.  bases: concatenated ASCII reads; offsets[n_reads+1].  out must hold out_capacity
// bytes; out_offsets[n_reads+1].  Returns 0, or -1 if out_capacity is too small.
int orc_correct_reads2(void* t, const orc_params* q, const char* bases, const uint64_t* offsets, uint32_t n_reads,
                       int threads, char* out, uint64_t out_capacity, uint64_t* out_offsets, uint8_t* status,
                       char* counters_json, uint64_t counters_cap, double* seconds, uint32_t* read_stats);
int orc_correct_reads(void* t, const orc_params* q, const char* bases, const uint64_t* offsets, uint32_t n_reads,
                      int threads, char* out, uint64_t out_capacity, uint64_t* out_offsets, uint8_t* status,
                      char* counters_json, uint64_t counters_cap, double* seconds) {
  return orc_correct_reads2(t, q, bases, offsets, n_reads, threads, out, out_capacity, out_offsets, status, counters_json,
                            counters_cap, seconds, nullptr);
}
// read_stats (may be null): per read {span of m_InKmersPositions, their number} as Read.cpp:418-433 would print them
int orc_correct_reads2(void* t, const orc_params* q, const char* bases, const uint64_t* offsets, uint32_t n_reads,
                       int threads, char* out, uint64_t out_capacity, uint64_t* out_offsets, uint8_t* status,
                       char* counters_json, uint64_t counters_cap, double* seconds, uint32_t* read_stats) {
  Params p = to_params(q);
  Table* T = (Table*)t;
  if (threads < 1) threads = 1;
  omp_set_num_threads(threads);
  std::vector<Seq> results(n_reads);
  std::vector<Counters> per(threads);
  auto t0 = std::chrono::steady_clock::now();
#pragma omp parallel for schedule(dynamic)
  for (int64_t r = 0; r < (int64_t)n_reads; ++r) {
    Seq s = to_dna5(std::string(bases + offsets[r], offsets[r + 1] - offsets[r]));
    ReadResult rr = correct_read(s, *T, p, per[omp_get_thread_num()]);
    status[r] = (uint8_t)rr.status;
    if (read_stats) { read_stats[2 * r] = rr.stat_span; read_stats[2 * r + 1] = rr.stat_regions; }
    results[r].swap(rr.corrected);
  }
  auto t1 = std::chrono::steady_clock::now();
  if (seconds) *seconds = std::chrono::duration<double>(t1 - t0).count();
  uint64_t pos = 0;
  out_offsets[0] = 0;
  for (uint32_t r = 0; r < n_reads; ++r) {
    if (pos + results[r].size() > out_capacity) return -1;
    memcpy(out + pos, results[r].data(), results[r].size());
    pos += results[r].size();
    out_offsets[r + 1] = pos;
  }
  Counters total;
  for (auto& c : per) total.add(c);
  if (counters_json && counters_cap) {
    std::string j = total.json();
    strncpy(counters_json, j.c_str(), counters_cap - 1);
    counters_json[counters_cap - 1] = 0;
  }
  return 0;
}

// one read with a stage dump (coverage, threshold, regions) for differential debugging
int orc_read_stages(void* t, const orc_params* q, const char* seq, uint64_t len, uint32_t* cov_counts, double* threshold,
                    int32_t* regions_found, int32_t* n_found, int32_t* regions_final, int32_t* n_final, int32_t max_regions,
                    char* trace, uint64_t trace_cap) {
  Params p = to_params(q);
  Counters C;
  StageDump d;
  Seq s = to_dna5(std::string(seq, len));
  ReadResult rr = correct_read(s, *(Table*)t, p, C, &d);
  for (size_t i = 0; i < d.coverage.size(); ++i) cov_counts[i] = d.coverage[i].first;
  *threshold = d.threshold;
  *n_found = (int32_t)std::min<size_t>(d.regions_found.size(), max_regions);
  for (int i = 0; i < *n_found; ++i) {
    regions_found[2 * i] = std::get<0>(d.regions_found[i]);
    regions_found[2 * i + 1] = std::get<1>(d.regions_found[i]);
  }
  *n_final = (int32_t)std::min<size_t>(d.regions_final.size(), max_regions);
  for (int i = 0; i < *n_final; ++i) {
    regions_final[2 * i] = std::get<0>(d.regions_final[i]);
    regions_final[2 * i + 1] = std::get<1>(d.regions_final[i]);
  }
  if (trace && trace_cap) {
    strncpy(trace, d.trace.c_str(), trace_cap - 1);
    trace[trace_cap - 1] = 0;
  }
  return (int)rr.status;
}

// ---- primitives, for unit tests of the device kernels
int orc_nw(const char* a, const char* b) { return nw_score(a, b); }
int orc_lcs(const char* a, const char* b) { return lcs_score(a, b); }
int orc_overlap(const char* ref, const char* cand, int direction_right) {
  return overlap_score(ref, cand, direction_right ? RIGHT : LEFT);
}
void orc_xdrop(const char* query_seg, const char* database_seg, int extend_left, int xdrop, uint64_t* ext_rows,
               uint64_t* ext_cols) {
  size_t r = 0, c = 0;
  xdrop_extend(query_seg, database_seg, extend_left != 0, xdrop, r, c);
  *ext_rows = r;
  *ext_cols = c;
}
// orc_xdrop plus the number of DP cells the extension visited (Counters::cells_xdrop)
void orc_xdrop_counted(const char* query_seg, const char* database_seg, int extend_left, int xdrop, uint64_t* ext_rows,
                       uint64_t* ext_cols, uint64_t* cells) {
  Counters ctr;
  size_t r = 0, c = 0;
  xdrop_extend(query_seg, database_seg, extend_left != 0, xdrop, r, c, &ctr);
  *ext_rows = r;
  *ext_cols = c;
  *cells = ctr.cells_xdrop;
}
// getSeedAndExtension: returns lengths of (refExtension, histExtension), posOnRef, score, stop
void orc_seed_extend(const char* reference, const char* candidate, int xdrop, int direction_right, uint32_t K,
                     int32_t* ref_ext_len, int32_t* hist_ext_len, int32_t* pos_on_ref, double* score, int32_t* stop) {
  auto r = getSeedAndExtension(reference, candidate, xdrop, direction_right ? RIGHT : LEFT, K);
  *ref_ext_len = (int32_t)std::get<0>(r).size();
  *hist_ext_len = (int32_t)std::get<1>(r).size();
  *pos_on_ref = std::get<2>(r);
  *score = std::get<3>(r);
  *stop = std::get<4>(r) ? 1 : 0;
}
long orc_horspool(const char* haystack, const char* needle, int cycle_mode) {
  return horspool_first(haystack, needle, cycle_mode);
}
int orc_is_expected_model(uint32_t nextc, uint32_t cc, double alpha, int classe_expected) {
  Params p;
  p.ALPHA = alpha;
  return isExpectedbyMyModel(nextc, cc, p, classe_expected ? EXPECTED : UNEXPECTED);
}
int orc_is_expected_lastnode(uint32_t nextc, uint32_t cc, double alpha) {
  Params p;
  p.ALPHA = alpha;
  return isExpectedbyMyLastNode(nextc, cc, p);
}
// tags: 0 EXPECTED, 1 UNEXPECTED, 7 BREAKPOINT (Status enum); returns number of tags (0 or 4)
int orc_tag_next_nodes(const orc_params* q, const uint32_t* counts4, const uint32_t* colours4, uint32_t count, int complex_,
                       int32_t* tags4, double* dist4) {
  Params p = to_params(q);
  std::vector<CCount> nc;
  for (int i = 0; i < 4; ++i) nc.push_back(std::make_pair(counts4[i], colours4[i]));
  std::vector<std::pair<Status, double>> tags;
  tagNextNodes(tags, nc, count, p, complex_ != 0);
  for (size_t i = 0; i < tags.size(); ++i) {
    tags4[i] = (int32_t)tags[i].first;
    dist4[i] = tags[i].second;
  }
  return (int)tags.size();
}
void orc_std_sort_perm(const int64_t* keys, uint32_t n, uint32_t* perm) {
  std::vector<long long> k(keys, keys + n);
  std::vector<unsigned> p = std_sort_permutation(k);
  for (uint32_t i = 0; i < n; ++i) perm[i] = p[i];
}

}  // extern "C"
