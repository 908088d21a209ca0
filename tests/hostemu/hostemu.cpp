// hostemu.cpp -- compiles the product's TALC_HD device code with g++ so that its logic can be
// diffed against the oracle on a machine without a GPU.  TEST AID ONLY: nothing in the shipped
// library links this file, and the product has no CPU path.
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "../../talc_b200/csrc/correct.cuh"

using namespace talc;

struct EmuTable {
  std::vector<Slot> slots;
  u64 mask;
  u32 K;
};

static Slot* emu_find(EmuTable* t, u64 key, bool insert) {
  u64 b = hash_kmer(key) & t->mask & ~1ull;
  for (;;) {
    for (int i = 0; i < 2; ++i) {
      Slot& s = t->slots[b + i];
      if (s.key == key) return &s;
      if (s.key == kEmptyKey) {
        if (!insert) return nullptr;
        s.key = key;
        s.count = 0;
        s.colour = 0;
        return &s;
      }
    }
    b = (b + 2) & t->mask;
  }
}

static u64 revcomp(u64 k, u32 K) {
  u64 r = 0;
  for (u32 i = 0; i < K; ++i) {
    r = (r << 2) | (3 - (k & 3));
    k >>= 2;
  }
  return r;
}

extern "C" {

struct emu_params {
  uint32_t K, MIN_COUNT, WINDOW_SIZE, MAX_NB_COMPETING_PATHS;
  double ALPHA, SR_ERROR_RATE, MIN_INNER_SCORE, MIN_BORDER_SCORE;
  int32_t cycle_mode, q11_zero_init;
};
static Params to_params(const emu_params* q) {
  Params p;
  p.K = q->K; p.min_count = q->MIN_COUNT; p.window = q->WINDOW_SIZE; p.max_branches = q->MAX_NB_COMPETING_PATHS;
  p.alpha = q->ALPHA; p.sr_error = q->SR_ERROR_RATE; p.min_inner = q->MIN_INNER_SCORE; p.min_border = q->MIN_BORDER_SCORE;
  p.cycle_mode = q->cycle_mode; p.q11_zero = q->q11_zero_init;
  return p;
}

// sequential build with the reference's semantics (Jellyfish.cpp:236-295, utils.cpp:658-669)
void* emu_table_build(const emu_params* q, const uint64_t* keys, const int64_t* counts, uint64_t n, const uint64_t* jkeys,
                      const int64_t* jcounts, uint64_t nj, int use_junctions) {
  EmuTable* t = new EmuTable;
  t->K = q->K;
  u64 cap = 2;
  while (cap < 2 * n + 2) cap <<= 1;
  t->slots.assign(cap, Slot{kEmptyKey, 0, 0});
  t->mask = cap - 1;
  for (u64 i = 0; i < n; ++i) {
    if ((u32)(int)counts[i] >= q->MIN_COUNT) {
      if (!emu_find(t, keys[i], false)) emu_find(t, keys[i], true)->count = (u32)(int)counts[i];
    }
  }
  if (use_junctions) {
    for (u64 i = 0; i < nj; ++i) {
      if ((u32)(int)jcounts[i] < kColouredCountThr) {
        if (Slot* s = emu_find(t, jkeys[i], false)) s->colour = (u32)(int)jcounts[i];
        if (Slot* s = emu_find(t, revcomp(jkeys[i], q->K), false)) s->colour = (u32)(int)jcounts[i];
      }
    }
  }
  for (u32 b = 0; b < 4; ++b) {
    u64 homo = 0;
    for (u32 i = 0; i < q->K; ++i) homo = (homo << 2) | b;
    if (Slot* s = emu_find(t, homo, false)) s->colour = 0;
  }
  return t;
}
void emu_table_free(void* t) { delete (EmuTable*)t; }

static uint64_t g_yields = 0;
uint64_t emu_yields() { return g_yields; }
int emu_correct_reads(void* tab, const emu_params* q, const uint8_t* bases, const uint64_t* offsets, uint32_t n_reads,
                      uint32_t arena_bytes, int wide, uint8_t* out, uint64_t out_capacity, uint64_t* out_offsets,
                      uint8_t* status, uint64_t* counters /* kNumCounters */) {
  EmuTable* t = (EmuTable*)tab;
  Params P = to_params(q);
  TableView tv;
  tv.slots = t->slots.data();
  tv.mask = t->mask;
  Counters total;
  memset(&total, 0, sizeof(total));
  std::vector<u8> arena(arena_bytes);
  std::vector<u32> cov;
  u64 pos = 0;
  out_offsets[0] = 0;
  for (u32 r = 0; r < n_reads; ++r) {
    ReadView rd;
    rd.s = bases + offsets[r];
    rd.len = (u32)(offsets[r + 1] - offsets[r]);
    // coverage (what the coverage kernel produces)
    cov.clear();
    if (rd.len >= P.K) {
      for (u32 i = 0; i + P.K <= rd.len; ++i) {
        bool ok;
        u64 km = rd.kmer_at(i, P.K, ok);
        u32 c = 0, cl = 0;
        if (ok) table_lookup(tv, km, c, cl);
        cov.push_back(c);
      }
    }
    Corrector* cx = new Corrector;
    cx->T = tv;
    cx->P = P;
    cx->tabs.n = 0;
    cx->tabs.lower = cx->tabs.upper = cx->tabs.sq = nullptr;
    Counters mine;
    memset(&mine, 0, sizeof(mine));
    cx->ctr = &mine;
    ReadJob job;
    job.rd = rd;
    job.cov = cov.data();
    job.arena = arena.data();
    job.arena_bytes = arena_bytes;
    job.wide = (wide & 1) != 0;
    cx->pauseBudget = 0;
    u8 st;
    if (wide & 2) {
      // split mode: the read yields where a long walk starts; the "walk kernel" is the scalar fast path run to its end,
      // then the read resumes from its frames -- the suspend / resume protocol of the device, on one thread
      cx->splitWalk = 1;
      cx->inlineInner = cx->inlineBorder = 6;
      cx->pauseBudget = (wide >> 8) & 0xFF;  // host: pause after every n-th general step (0 = never)
      st = cx->start(job);
      while (st == kReadYield) {
        ++g_yields;
        u32 step = cx->wq.step;
        if (cx->wq.border != 2)  // 2 = a pause, nothing to walk
          cx->fast_walk_scalar(step, cx->wq.pathMax, cx->wq.aims, cx->wq.nAims, cx->wq.border != 0, ~0u);
        cx->walk_done(step);
        st = cx->resume();
      }
    } else if (wide & 4) {
      st = cx->run(job);       // the state machines run through without a yield
    } else {
      st = cx->run_mono(job);  // the straight-line drivers of the monolithic kernel
    }
    mine.cells_nw += cx->dps.cells_nw;
    mine.cells_lcs += cx->dps.cells_lcs;
    mine.cells_ovl += cx->dps.cells_ovl;
    mine.cells_xdrop += cx->dps.cells_xdrop;
    if (st == kReadOverflow) {
      total.reads_overflow++;
    } else {
      const u64* src = (const u64*)&mine;
      u64* dst = (u64*)&total;
      for (int i = 0; i < kNumCounters; ++i) dst[i] += src[i];
      if (st == kReadOk) total.reads_ok++;
    }
    status[r] = st;
    u32 olen;
    if (st == kReadOk) olen = cx->corrected_length();
    else olen = rd.len;
    if (pos + olen > out_capacity) { delete cx; return -1; }
    if (st == kReadOk) cx->emit(out + pos, 0, 1);
    else for (u32 i = 0; i < rd.len; ++i) out[pos + i] = code_char(rd.code(i));
    pos += olen;
    if (st != kReadOverflow) total.bases_out += olen;
    out_offsets[r + 1] = pos;
    delete cx;
  }
  memcpy(counters, &total, sizeof(total));
  return 0;
}

// Two read contexts interleaved on one thread, the way a control warp of the fused kernel multiplexes its block's
// contexts: start A, start B, then resume whichever has been walked, alternating, until both reads are done.  Contexts are
// REUSED from one read to the next (as on the device).  Same outputs as emu_correct_reads.
int emu_correct_interleaved(void* tab, const emu_params* q, const uint8_t* bases, const uint64_t* offsets, uint32_t n_reads,
                            uint32_t arena_bytes, uint8_t* out, uint64_t out_capacity, uint64_t* out_offsets, uint8_t* status,
                            uint64_t* counters) {
  EmuTable* t = (EmuTable*)tab;
  Params P = to_params(q);
  TableView tv;
  tv.slots = t->slots.data();
  tv.mask = t->mask;
  Counters total;
  memset(&total, 0, sizeof(total));
  struct Ctx {
    Corrector cx;
    Counters mine;
    std::vector<u8> arena;
    std::vector<u32> cov;
    u32 read = 0xFFFFFFFFu;
    u8 st = 0;
    bool active = false;
  };
  Ctx* C = new Ctx[2];
  std::vector<std::vector<u8>> results(n_reads);
  u32 next = 0, done = 0;
  auto begin = [&](Ctx& c, u32 r) {
    ReadView rd;
    rd.s = bases + offsets[r];
    rd.len = (u32)(offsets[r + 1] - offsets[r]);
    c.cov.clear();
    if (rd.len >= P.K)
      for (u32 i = 0; i + P.K <= rd.len; ++i) {
        bool ok;
        u64 km = rd.kmer_at(i, P.K, ok);
        u32 cc = 0, cl = 0;
        if (ok) table_lookup(tv, km, cc, cl);
        c.cov.push_back(cc);
      }
    c.arena.resize(arena_bytes);
    c.cx.T = tv;
    c.cx.P = P;
    c.cx.tabs.n = 0;
    c.cx.tabs.lower = c.cx.tabs.upper = c.cx.tabs.sq = nullptr;
    memset(&c.mine, 0, sizeof(c.mine));
    c.cx.ctr = &c.mine;
    c.cx.splitWalk = 1;
    c.cx.inlineInner = 0;
    c.cx.inlineBorder = 6;
    c.cx.pauseBudget = 0;
    ReadJob job;
    job.rd = rd;
    job.cov = c.cov.data();
    job.arena = c.arena.data();
    job.arena_bytes = arena_bytes;
    job.wide = true;
    c.read = r;
    c.active = true;
    c.st = c.cx.start(job);
  };
  auto finish = [&](Ctx& c) {
    const u32 r = c.read;
    const u8 st = c.st;
    c.mine.cells_nw += c.cx.dps.cells_nw;
    c.mine.cells_lcs += c.cx.dps.cells_lcs;
    c.mine.cells_ovl += c.cx.dps.cells_ovl;
    c.mine.cells_xdrop += c.cx.dps.cells_xdrop;
    if (st == kReadOverflow) total.reads_overflow++;
    else {
      const u64* src = (const u64*)&c.mine;
      u64* dst = (u64*)&total;
      for (int i = 0; i < kNumCounters; ++i) dst[i] += src[i];
      if (st == kReadOk) total.reads_ok++;
    }
    status[r] = st;
    const u32 rlen = (u32)(offsets[r + 1] - offsets[r]);
    const u32 olen = st == kReadOk ? c.cx.corrected_length() : rlen;
    results[r].resize(olen);
    if (st == kReadOk) c.cx.emit(results[r].data(), 0, 1);
    else {
      ReadView rd;
      rd.s = bases + offsets[r];
      rd.len = rlen;
      for (u32 i = 0; i < rlen; ++i) results[r][i] = code_char(rd.code(i));
    }
    if (st != kReadOverflow) total.bases_out += olen;
    c.active = false;
    ++done;
  };
  while (done < n_reads) {
    for (int k = 0; k < 2; ++k) {
      Ctx& c = C[k];
      if (!c.active) {
        if (next < n_reads) begin(c, next++);
        else continue;
      } else {  // it yielded last time: walk, then resume
        u32 step = c.cx.wq.step;
        if (c.cx.wq.border != 2)
          c.cx.fast_walk_scalar(step, c.cx.wq.pathMax, c.cx.wq.aims, c.cx.wq.nAims, c.cx.wq.border != 0, ~0u);
        c.cx.walk_done(step);
        c.st = c.cx.resume();
      }
      if (c.st != kReadYield) finish(c);
    }
  }
  u64 pos = 0;
  out_offsets[0] = 0;
  for (u32 r = 0; r < n_reads; ++r) {
    if (pos + results[r].size() > out_capacity) { delete[] C; return -1; }
    memcpy(out + pos, results[r].data(), results[r].size());
    pos += results[r].size();
    out_offsets[r + 1] = pos;
  }
  memcpy(counters, &total, sizeof(total));
  delete[] C;
  return 0;
}

int emu_num_counters() { return kNumCounters; }

// ---- primitives
// ASCII -> the 4-bit packed layout the scoring routines read; the words live until the process ends (test aid)
static SeqView bytes_view(const char* s, u32 n) {
  static thread_local std::vector<std::vector<u64>> keep;
  if (keep.size() > 64) keep.erase(keep.begin(), keep.begin() + 32);
  keep.emplace_back((n + 15) / 16 + 2, 0);
  return pack_ascii4((const u8*)s, n, keep.back().data());
}
static std::vector<u64> pack(const char* s, u32 n) {
  std::vector<u64> w((n + 31) / 32 + 2, 0);
  for (u32 i = 0; i < n; ++i) path_set(w.data(), i, base_code((u8)s[i]) & 3);
  return w;
}
// packed != 0: second sequence is given to the kernel as a packed trail (must be ACGT only)
int emu_nw(const char* a, const char* b, int packed) {
  std::vector<u8> ar(1 << 20);
  Arena A; A.init(ar.data(), (u32)ar.size());
  u32 an = strlen(a), bn = strlen(b);
  std::vector<u64> w = pack(b, bn);
  SeqView vb = packed ? view_of_path(w.data(), bn) : bytes_view(b, bn);
  return -nw_distance(bytes_view(a, an), an, vb, bn, A, nullptr);
}
int emu_lcs(const char* a, const char* b, int packed) {
  std::vector<u8> ar(1 << 20);
  Arena A; A.init(ar.data(), (u32)ar.size());
  u32 an = strlen(a), bn = strlen(b);
  std::vector<u64> w = pack(b, bn);
  SeqView vb = packed ? view_of_path(w.data(), bn) : bytes_view(b, bn);
  return lcs_length(bytes_view(a, an), an, vb, bn, A, nullptr);
}
// walk-order overlap score == the oracle's RIGHT mode; LEFT mode is the same on reversed strings
int emu_overlap(const char* ref, const char* cand) {
  std::vector<u8> ar(1 << 22);
  Arena A; A.init(ar.data(), (u32)ar.size());
  u32 an = strlen(ref), bn = strlen(cand);
  return overlap_score(bytes_view(ref, an), an, bytes_view(cand, bn), bn, A, nullptr);
}
void emu_xdrop(const char* query_seg, const char* database_seg, int xdrop, int wide, uint64_t* ext_rows, uint64_t* ext_cols,
               int* overflow) {
  std::vector<u8> ar(1 << 22);
  Arena A; A.init(ar.data(), (u32)ar.size());
  u32 qn = strlen(query_seg), dn = strlen(database_seg);
  u32 er = 0, ec = 0;
  i32 es = 0;
  xdrop_extend(bytes_view(query_seg, qn), 0, qn, bytes_view(database_seg, dn), 0, dn, xdrop, er, ec, es, A, wide != 0, nullptr);
  *ext_rows = er; *ext_cols = ec; *overflow = (int)A.overflow;
}
// Mirror of xdrop_extend_reg<S> (talc_b200/csrc/xdrop.cuh) with the warp's registers laid out as flat arrays
// indexed by g = S*lane + i; shuffles become neighbour reads, warp reductions become loops.  It shares
// xd_cell / xd_next_window / xd_finish with the device code, so fuzzing it against xdrop_extend_scalar
// validates the band layout, the window updates and the end-position rules without a GPU.
static void xdrop_reg_mirror(const SeqView& query, u32 qoff, u32 qlen, const SeqView& database, u32 doff, u32 dlen, int X,
                             int S, u32& ext_rows, u32& ext_cols, i32& end_score, u64* cells_out) {
  const i32 cols = (i32)qlen + 1, rows = (i32)dlen + 1;
  ext_rows = 0;
  ext_cols = 0;
  end_score = 0;
  if (cells_out) *cells_out = 0;
  if (rows == 1 || cols == 1) return;
  const int G = 32 * S;
  std::vector<i32> vE(G), vO(G), vOld(G, kXdU), nv(G);
  std::vector<u32> qc(G), tc(G);
  for (int g = 0; g < G; ++g) {
    vE[g] = (g == 16 * S) ? 0 : kXdU;
    vO[g] = ((g == 16 * S - 1) | (g == 16 * S)) ? (X >= 1 ? -1 : kXdU) : kXdU;
    const i32 col = 1 - 16 * S + g, row = 1 + 16 * S - g;
    qc[g] = (col >= 1 && col <= (i32)qlen) ? query.code(qoff + (u32)(col - 1)) : 6u;
    tc[g] = (row >= 1 && row <= (i32)dlen) ? database.code(doff + (u32)(row - 1)) : 7u;
  }
  i32 minCol = 1, maxCol = 2, d = 1;
  XdHist h = xd_hist_init();
  u64 cells = 0;
  bool lastOdd;
  for (;;) {
    ++d;
    const i32 m = d >> 1;
    h.push(minCol, maxCol);
    {
      const i32 cb = m - 16 * S;
      const u32 qi = (u32)(m + 16 * S - 1);
      const u32 nq = (qi < qlen) ? query.code(qoff + qi) : 6u;
      i32 loT = INT32_MAX, hiT = INT32_MIN, loC, hiC;
      const XdRow R = xd_row(d, X, minCol, maxCol);
      for (int g = 0; g < G; ++g) {
        const i32 a = g ? vO[g - 1] : kXdU, b = vO[g], dg = vE[g];
        vOld[g] = dg;
        nv[g] = xd_cell(a, b, dg, qc[g] == tc[g], cb + g - minCol, R, loT, hiT);
      }
      xd_window_bounds(loT, hiT, minCol, loC, hiC);
      vE = nv;
      cells += (u64)(maxCol - minCol);
      xd_next_window(d, rows, cols, loC, hiC, minCol, maxCol);
      for (int g = 0; g + 1 < G; ++g) qc[g] = qc[g + 1];
      qc[G - 1] = nq;
    }
    if (!(minCol < maxCol)) { lastOdd = false; break; }
    ++d;
    h.push(minCol, maxCol);
    {
      const i32 cb = m + 1 - 16 * S;
      const u32 ti = (u32)(m + 16 * S);
      const u32 nt = (ti < dlen) ? database.code(doff + ti) : 7u;
      i32 loT = INT32_MAX, hiT = INT32_MIN, loC, hiC;
      const XdRow R = xd_row(d, X, minCol, maxCol);
      for (int g = 0; g < G; ++g) {
        const i32 a = vE[g], b = (g + 1 < G) ? vE[g + 1] : kXdU, dg = vO[g];
        vOld[g] = dg;
        nv[g] = xd_cell(a, b, dg, qc[g] == tc[g], cb + g - minCol, R, loT, hiT);
      }
      xd_window_bounds(loT, hiT, minCol, loC, hiC);
      vO = nv;
      cells += (u64)(maxCol - minCol);
      xd_next_window(d, rows, cols, loC, hiC, minCol, maxCol);
      for (int g = G - 1; g > 0; --g) tc[g] = tc[g - 1];
      tc[0] = nt;
    }
    if (!(minCol < maxCol)) { lastOdd = true; break; }
  }
  if (cells_out) *cells_out = cells;
  const i32 cb3 = xd_col_base(d, S), cb2 = xd_col_base(d - 1, S), cb1 = xd_col_base(d - 2, S);
  auto pick = [&](const std::vector<i32>& v, i32 cb, i32 col) -> i32 {
    const i32 g = col - cb;
    return (g >= 0 && g < G) ? v[g] : kXdU;
  };
  auto at = [&](int which, i32 col) -> i32 {
    if (which == 3) return lastOdd ? pick(vO, cb3, col) : pick(vE, cb3, col);
    return lastOdd ? pick(vE, cb2, col) : pick(vO, cb2, col);
  };
  auto argmax1 = [&](i32 lo, i32 hi, i32& col) -> i32 {
    i32 bv = kXdU;
    col = INT32_MAX;
    for (int g = 0; g < G; ++g) {
      const i32 c = cb1 + g;
      if (c >= lo && c <= hi && vOld[g] > bv) { bv = vOld[g]; col = c; }
    }
    return bv;
  };
  xd_finish(d, h, at, argmax1, ext_rows, ext_cols, end_score);
}
void emu_xdrop_reg(const char* query_seg, const char* database_seg, int xdrop, int S, uint64_t* ext_rows, uint64_t* ext_cols,
                   uint64_t* cells) {
  u32 qn = strlen(query_seg), dn = strlen(database_seg);
  u32 er = 0, ec = 0;
  u64 c = 0;
  i32 es = 0;
  xdrop_reg_mirror(bytes_view(query_seg, qn), 0, qn, bytes_view(database_seg, dn), 0, dn, xdrop, S, er, ec, es, &c);
  *ext_rows = er; *ext_cols = ec; *cells = c;
}
// built-in fuzzer: random related pairs, every admissible S; returns the number of disagreements with the scalar form
int emu_xdrop_reg_fuzz(uint64_t seed, int n_cases, int max_len) {
  u64 s = seed * 0x9E3779B97F4A7C15ull + 1;
  auto rnd = [&]() { s ^= s << 13; s ^= s >> 7; s ^= s << 17; return s; };
  std::vector<u8> ar(1 << 24);
  int bad = 0;
  for (int t = 0; t < n_cases; ++t) {
    const u32 an = 1 + rnd() % max_len;
    std::string a(an, 'A'), b;
    const int alpha = (rnd() % 4 == 0) ? 2 : 4;  // low-complexity pairs make long ties
    for (u32 i = 0; i < an; ++i) a[i] = "ACGT"[rnd() % alpha];
    const u32 errPermille = (u32)(rnd() % 300);
    for (u32 i = 0; i < an; ++i) {
      const u32 r = rnd() % 1000;
      if (r < errPermille / 3) continue;                                  // deletion
      if (r < 2 * errPermille / 3) { b.push_back("ACGT"[rnd() % alpha]); }  // substitution
      else b.push_back(a[i]);
      if (rnd() % 1000 < errPermille / 3) b.push_back("ACGT"[rnd() % alpha]);  // insertion
    }
    if (rnd() % 5 == 0) b.resize(rnd() % (b.size() + 1));
    if (rnd() % 7 == 0) b += std::string(rnd() % 40, 'A');
    if (rnd() % 50 == 0 && !a.empty()) a[rnd() % a.size()] = 'N';
    if (b.empty()) b = "A";
    const int X = (int)(rnd() % 12 == 0 ? rnd() % 270 : rnd() % 40) - 1;
    const bool swap = rnd() & 1;
    const std::string& q = swap ? b : a;
    const std::string& db = swap ? a : b;
    const u32 qoff = rnd() % 3, doff = rnd() % 3;
    if (qoff >= q.size() || doff >= db.size()) continue;
    Arena A; A.init(ar.data(), (u32)ar.size());
    DpStats st; st.cells_xdrop = 0;
    u32 er0 = 0, ec0 = 0;
    i32 es0 = 0;
    const SeqView qv = bytes_view(q.data(), (u32)q.size()), dv = bytes_view(db.data(), (u32)db.size());
    xdrop_extend_scalar(qv, qoff, (u32)q.size() - qoff, dv, doff, (u32)db.size() - doff, X, er0, ec0, es0, A, true, &st);
    {  // the end cell holds the exact edit distance of the two extensions (used instead of a separate NW pass)
      int dist = (int)(er0 > ec0 ? er0 : ec0);
      if (er0 > 0 && ec0 > 0) {
        SeqView qs = qv, ds = dv;
        qs.start += (i32)qoff; ds.start += (i32)doff;
        dist = nw_distance_scalar(qs, ec0, ds, er0, A, nullptr);
      }
      if (es0 != -dist) {
        if (bad < 5) fprintf(stderr, "xdrop end score %d != -distance %d (X=%d q=%s db=%s)\n", es0, dist, X, q.c_str(), db.c_str());
        ++bad;
      }
    }
    for (int S : {1, 2, 4, 8}) {
      if (X > 32 * S - 1) continue;
      u32 er = 0, ec = 0;
      u64 cells = 0;
      i32 es = 0;
      xdrop_reg_mirror(qv, qoff, (u32)q.size() - qoff, dv, doff, (u32)db.size() - doff, X, S, er, ec, es, &cells);
      if (er != er0 || ec != ec0 || cells != st.cells_xdrop || es != es0) {
        if (bad < 5)
          fprintf(stderr, "xdrop mismatch S=%d X=%d q=%s db=%s qoff=%u doff=%u scalar=(%u,%u,%llu) reg=(%u,%u,%llu)\n", S, X,
                  q.c_str(), db.c_str(), qoff, doff, er0, ec0, (unsigned long long)st.cells_xdrop, er, ec,
                  (unsigned long long)cells);
        ++bad;
      }
    }
  }
  return bad;
}
// ---------------------------------------------------------------------------------------------------------
// Groundwork for an incremental border scoring (DESIGN.md "what comes next"): the gapped X-drop with Score(0,-1,-1)
// characterised through a Landau-Vishkin table instead of a cell-by-cell DP.  F[e][k] = furthest row on diagonal
// k = col - row whose cell has edit distance <= e.  A cell survives the X-drop iff its distance is <= X, with the two
// boundary quirks of SeqAn's routine: a first-row / first-column cell at distance d survives only if d < X (or
// d == 1 <= X), and therefore a cell of diagonal +-X survives only if it can be reached without passing through
// that boundary cell.  The window bookkeeping, the cell tally and the end-position rules are then replayed on the
// surviving set.  Fuzzed against xdrop_extend_scalar; F only depends on the sequences, so it can be extended base by
// base as a trail grows instead of re-running the extension from the seed every six steps.
static int g_lv_skip = 2;  // 0: replay every anti-diagonal, 1: jump between any interval boundaries, 2: only outermost ones
static u64 g_lv_steps = 0, g_lv_skipped = 0;
static void xdrop_lv_mirror(const SeqView& query, u32 qoff, u32 qlen, const SeqView& database, u32 doff, u32 dlen, int X,
                            u32& ext_rows, u32& ext_cols, i32& end_score, u64* cells_out) {
  const i32 Q = (i32)qlen, T = (i32)dlen, cols = Q + 1, rows = T + 1;
  ext_rows = ext_cols = 0;
  end_score = 0;
  if (cells_out) *cells_out = 0;
  if (rows == 1 || cols == 1) return;
  const i32 NONE = -1000000;
  const i32 XX = X < 0 ? -1 : X;
  // F[e][k + XX], k in [-e, e]
  std::vector<std::vector<i32>> F((size_t)(XX + 1 > 0 ? XX + 1 : 0), std::vector<i32>((size_t)(2 * (XX > 0 ? XX : 0) + 1), NONE));
  auto slide = [&](i32 r, i32 k) {
    while (r < T && r + k < Q && query.code(qoff + (u32)(r + k)) == database.code(doff + (u32)r)) ++r;
    return r;
  };
  auto inside = [&](i32 r, i32 k) { return r >= 0 && r <= T && r + k >= 0 && r + k <= Q; };
  for (i32 e = 0; e <= XX; ++e) {
    for (i32 k = -e; k <= e; ++k) {
      i32 r = NONE;
      if (e == 0) r = 0;
      else {
        auto get = [&](i32 kk) { return (kk >= -(e - 1) && kk <= e - 1) ? F[e - 1][kk + XX] : NONE; };
        const i32 a = get(k - 1);          // insertion: column + 1, same row
        const i32 b = get(k);              // substitution: row + 1
        const i32 c = get(k + 1);          // deletion: row + 1
        // every cell up to the furthest point of a neighbour diagonal can make the move, so a move that would leave
        // the matrix is clipped to the last row of this diagonal rather than dropped
        const i32 rmax = (T < Q - k) ? T : Q - k, rmin = k < 0 ? -k : 0;
        auto clip = [&](i32 x) { return x > rmax ? rmax : x; };
        if (a != NONE && clip(a) >= rmin) r = clip(a) > r ? clip(a) : r;
        if (b != NONE && clip(b + 1) >= rmin) r = clip(b + 1) > r ? clip(b + 1) : r;
        if (c != NONE && clip(c + 1) >= rmin) r = clip(c + 1) > r ? clip(c + 1) : r;
      }
      if (r != NONE && inside(r, k)) F[e][k + XX] = slide(r, k);
    }
  }
  // distance of a cell, or a large value when it exceeds X
  auto dist = [&](i32 r, i32 c) -> i32 {
    const i32 k = c - r;
    if (k < -XX || k > XX) return 1 << 20;
    for (i32 e = (k < 0 ? -k : k); e <= XX; ++e)
      if (F[e][k + XX] != NONE && F[e][k + XX] >= r) return e;
    return 1 << 20;
  };
  // Surviving cells of diagonal k = the rows [sK[k], fK[k]] (empty when sK > fK): distances do not decrease along a
  // diagonal, so the set is a prefix that ends at the furthest point of level X; it starts at the boundary cell of
  // the diagonal if that one survives (distance |k| < X, or |k| == 1 <= X), else one row further in; and a diagonal
  // +-X (X >= 2) survives at all only if it can be entered beyond its boundary cell.
  std::vector<i32> sK((size_t)(2 * (XX > 0 ? XX : 0) + 1), 1), fK((size_t)(2 * (XX > 0 ? XX : 0) + 1), 0);
  for (i32 k = -XX; k <= XX && XX >= 0; ++k) {
    const i32 ak = k < 0 ? -k : k, first = k < 0 ? -k : 0;
    const bool boundaryOk = (k == 0) || (ak < X) || (ak == 1 && X >= 1);
    i32 s0 = boundaryOk ? first : first + 1, f0 = F[XX][k + XX];
    if (f0 == NONE) { s0 = 1; f0 = 0; }
    if (X >= 2 && ak == X) {
      const i32 r0 = F[X - 1][(k > 0 ? X - 1 : -(X - 1)) + XX];
      const bool ok = r0 != NONE && (k > 0 ? r0 >= 1 : r0 + 1 >= X + 1);
      if (!ok) { s0 = 1; f0 = 0; }
    }
    sK[k + XX] = s0;
    fK[k + XX] = f0;
  }
  auto value = [&](i32 d, i32 c) -> i32 {
    const i32 r = d - c;
    if (c < 0 || r < 0 || c > Q || r > T) return kXdU;
    if (d == 0) return 0;
    const i32 k = c - r;
    if (k < -XX || k > XX) return kXdU;
    if (r < sK[k + XX] || r > fK[k + XX]) return kXdU;
    if (c == 0 || r == 0) return -d;
    return -dist(r, c);
  };
  // replay of the window loop on the surviving set.  Between the O(X) anti-diagonals where a diagonal's interval
  // starts or ends (and before the ends of the sequences clamp the window) the loop is periodic: the windows of
  // anti-diagonals d+2, d+3 are those of d, d+1 moved one column on.  Once that is observed the replay jumps over
  // the rest of the quiet stretch in one step (`skip` below), so its cost is O(X) events, not O(length).
  std::vector<i32> events;
  for (i32 k = -XX; k <= XX && XX >= 0; ++k) {
    if (sK[k + XX] > fK[k + XX]) continue;
    events.push_back(2 * sK[k + XX] + k);
    events.push_back(2 * fK[k + XX] + k);
  }
  std::sort(events.begin(), events.end());
  i32 minCol = 1, maxCol = 2, d = 1;
  XdHist h = xd_hist_init();
  u64 cells = 0;
  u64 skipped = 0;
  while (minCol < maxCol) {
    if (g_lv_skip && d >= 6) {
      // windows of d-2 (h.min2/max2 is d-1's... careful: h.*3 = window of d, h.*2 = d-1, h.*1 = d-2), next = d+1
      const bool periodic = (minCol == h.min2 + 1) && (maxCol == h.max2 + 1) && (h.min3 == h.min1 + 1) && (h.max3 == h.max1 + 1);
      if (periodic) {
        // quiet stretch: until an interval of one of the OUTERMOST surviving diagonals (per parity, looking back over
        // the last four anti-diagonals) ends, or a diagonal outside them starts; inner diagonals come and go freely
        i32 nextEv = INT32_MAX;
        if (g_lv_skip == 2) {
          i32 kmin[2] = {INT32_MAX, INT32_MAX}, kmax[2] = {INT32_MIN, INT32_MIN};
          bool changing = false;
          for (i32 k = -XX; k <= XX; ++k) {
            const i32 s0 = sK[k + XX], f0 = fK[k + XX];
            if (s0 > f0) continue;
            const i32 dS = 2 * s0 + k, dE = 2 * f0 + k;
            if (dS <= d - 4 && dE >= d) {  // alive throughout the observed period
              const int p = k & 1;
              kmin[p] = k < kmin[p] ? k : kmin[p];
              kmax[p] = k > kmax[p] ? k : kmax[p];
            } else if (dE >= d - 4 && dS <= d) changing = true;  // started or ended inside the observed period
          }
          if (!changing && kmin[0] != INT32_MAX && kmin[1] != INT32_MAX) {
            for (i32 k = -XX; k <= XX; ++k) {
              const i32 s0 = sK[k + XX], f0 = fK[k + XX];
              if (s0 > f0) continue;
              const i32 dS = 2 * s0 + k, dE = 2 * f0 + k;
              const int p = k & 1;
              if (k == kmin[p] || k == kmax[p]) nextEv = dE < nextEv ? dE : nextEv;             // an outermost one ends
              if ((k < kmin[p] || k > kmax[p]) && dS > d) nextEv = dS < nextEv ? dS : nextEv;   // one further out starts
              if ((k < kmin[p] || k > kmax[p]) && dS <= d && dE >= d - 4) nextEv = d;           // (cannot happen: not alive)
            }
          } else nextEv = d;
        } else {
          auto it = std::upper_bound(events.begin(), events.end(), d - 4);
          nextEv = (it == events.end()) ? INT32_MAX : *it;
        }
        if (nextEv > d + 6) {
          i64 m = ((i64)(nextEv == INT32_MAX ? (i64)rows + cols : nextEv) - d - 6) / 2;  // double steps that stay clear of it
          const i64 m1 = (i64)rows + minCol - d - 8;  // the database-end clamp d+2-rows stays below minCol
          const i64 m2 = (i64)cols - maxCol - 3;      // the query-end clamp stays above maxCol
          if (m1 < m) m = m1;
          if (m2 < m) m = m2;
          if (m >= 1) {
            // anti-diagonals d+1 .. d+2m: window of d+1 is [minCol,maxCol), of d+2 is [h.min3+1, h.max3+1), ...
            cells += (u64)m * (u64)((maxCol - minCol) + (h.max3 - h.min3));
            skipped += (u64)(2 * m);
            d += (i32)(2 * m);
            minCol += (i32)m; maxCol += (i32)m;
            h.min1 += (i32)m; h.max1 += (i32)m; h.min2 += (i32)m; h.max2 += (i32)m; h.min3 += (i32)m; h.max3 += (i32)m;
          }
        }
      }
    }
    ++d;
    h.push(minCol, maxCol);
    i32 loC = INT32_MAX, hiC = INT32_MIN;
    for (i32 c = minCol; c <= maxCol; ++c) {
      const bool here = (c < maxCol || (d == maxCol)) ? value(d, c) != kXdU : false;  // col maxCol: only the row-0 sentinel
      if (here || value(d - 1, c - 1) != kXdU) { loC = c; break; }
    }
    for (i32 c = maxCol - 1; c >= minCol - 1; --c) {
      const bool here = (c >= minCol || (minCol == 1)) ? value(d, c) != kXdU : false;  // col minCol-1: only the col-0 sentinel
      if (here || value(d - 1, c) != kXdU) { hiC = c; break; }
    }
    cells += (u64)(maxCol - minCol);
    xd_next_window(d, rows, cols, loC, hiC, minCol, maxCol);
  }
  if (cells_out) *cells_out = cells;
  g_lv_steps += (u64)d;
  g_lv_skipped += skipped;
  auto inwin = [&](i32 dd, i32 mn, i32 mx, i32 c) -> i32 {  // the array of anti-diagonal dd: cols [mn-1, mx]
    if (c < mn - 1 || c > mx) return kXdU;
    if (c == mn - 1 && !(mn == 1)) return kXdU;               // low sentinel is only ever the column-0 cell
    if (c == mx && !(dd == mx)) return kXdU;                  // high sentinel is only ever the row-0 cell
    return value(dd, c);
  };
  auto at = [&](int which, i32 c) -> i32 {
    return which == 3 ? inwin(d, h.min3, h.max3, c) : inwin(d - 1, h.min2, h.max2, c);
  };
  auto argmax1 = [&](i32 lo, i32 hi, i32& col) -> i32 {
    i32 bv = kXdU;
    col = INT32_MAX;
    for (i32 c = lo; c <= hi; ++c) {
      const i32 v = inwin(d - 2, h.min1, h.max1, c);
      if (v > bv) { bv = v; col = c; }
    }
    return bv;
  };
  xd_finish(d, h, at, argmax1, ext_rows, ext_cols, end_score);
}
void emu_xdrop_lv_stats(uint64_t* steps, uint64_t* skipped) { *steps = g_lv_steps; *skipped = g_lv_skipped; }
void emu_xdrop_lv_mode(int mode) { g_lv_skip = mode; g_lv_steps = g_lv_skipped = 0; }
// realistic pairs: a read-like sequence against a copy with `err_permille` errors, fixed drop-off
int emu_xdrop_lv_fuzz_realistic(uint64_t seed, int n_cases, int len, int err_permille, int X) {
  u64 s = seed * 0x9E3779B97F4A7C15ull + 11;
  auto rnd = [&]() { s ^= s << 13; s ^= s >> 7; s ^= s << 17; return s; };
  std::vector<u8> ar(1 << 24);
  int bad = 0;
  for (int t = 0; t < n_cases; ++t) {
    std::string a((size_t)len, 'A'), b;
    for (int i = 0; i < len; ++i) a[i] = "ACGT"[rnd() % 4];
    for (int i = 0; i < len; ++i) {
      const u32 r = rnd() % 1000;
      if ((int)r < err_permille * 3 / 10) continue;
      if ((int)r < err_permille * 7 / 10) b.push_back("ACGT"[rnd() % 4]);
      else b.push_back(a[i]);
      if ((int)(rnd() % 1000) < err_permille * 3 / 10) b.push_back("ACGT"[rnd() % 4]);
    }
    if (b.empty()) b = "A";
    Arena A; A.init(ar.data(), (u32)ar.size());
    DpStats st; st.cells_xdrop = 0;
    u32 er0 = 0, ec0 = 0, er = 0, ec = 0;
    i32 es0 = 0, es = 0;
    u64 cells = 0;
    const SeqView qv = bytes_view(a.data(), (u32)a.size()), dv = bytes_view(b.data(), (u32)b.size());
    xdrop_extend_scalar(qv, 0, (u32)a.size(), dv, 0, (u32)b.size(), X, er0, ec0, es0, A, true, &st);
    xdrop_lv_mirror(qv, 0, (u32)a.size(), dv, 0, (u32)b.size(), X, er, ec, es, &cells);
    if (er != er0 || ec != ec0 || es != es0 || cells != st.cells_xdrop) ++bad;
  }
  return bad;
}
int emu_xdrop_lv_fuzz(uint64_t seed, int n_cases, int max_len) {
  u64 s = seed * 0x9E3779B97F4A7C15ull + 7;
  auto rnd = [&]() { s ^= s << 13; s ^= s >> 7; s ^= s << 17; return s; };
  std::vector<u8> ar(1 << 24);
  int bad = 0;
  for (int t = 0; t < n_cases; ++t) {
    const u32 an = 1 + rnd() % max_len;
    std::string a(an, 'A'), b;
    const int alpha = (rnd() % 3 == 0) ? 2 : 4;
    for (u32 i = 0; i < an; ++i) a[i] = "ACGT"[rnd() % alpha];
    const u32 errPermille = (u32)(rnd() % 300);
    for (u32 i = 0; i < an; ++i) {
      const u32 r = rnd() % 1000;
      if (r < errPermille / 3) continue;
      if (r < 2 * errPermille / 3) b.push_back("ACGT"[rnd() % alpha]);
      else b.push_back(a[i]);
      if (rnd() % 1000 < errPermille / 3) b.push_back("ACGT"[rnd() % alpha]);
    }
    if (rnd() % 5 == 0) b.resize(rnd() % (b.size() + 1));
    if (rnd() % 7 == 0) b += std::string(rnd() % 40, 'A');
    if (b.empty()) b = "A";
    const int X = (int)(rnd() % 6 == 0 ? rnd() % 48 : rnd() % 14) - 1;
    const bool swap = rnd() & 1;
    const std::string& q = swap ? b : a;
    const std::string& db = swap ? a : b;
    Arena A; A.init(ar.data(), (u32)ar.size());
    DpStats st; st.cells_xdrop = 0;
    u32 er0 = 0, ec0 = 0, er = 0, ec = 0;
    i32 es0 = 0, es = 0;
    u64 cells = 0;
    const SeqView qv = bytes_view(q.data(), (u32)q.size()), dv = bytes_view(db.data(), (u32)db.size());
    xdrop_extend_scalar(qv, 0, (u32)q.size(), dv, 0, (u32)db.size(), X, er0, ec0, es0, A, true, &st);
    xdrop_lv_mirror(qv, 0, (u32)q.size(), dv, 0, (u32)db.size(), X, er, ec, es, &cells);
    if (er != er0 || ec != ec0 || es != es0 || cells != st.cells_xdrop) {
      if (bad < 8)
        fprintf(stderr, "LV mismatch X=%d q=%s db=%s scalar=(%u,%u,%d,%llu) lv=(%u,%u,%d,%llu)\n", X, q.c_str(), db.c_str(), er0,
                ec0, es0, (unsigned long long)st.cells_xdrop, er, ec, es, (unsigned long long)cells);
      ++bad;
    }
  }
  return bad;
}
// getSeedAndExtension on walk-order strings (RIGHT as is; for LEFT pass reversed strings and right=0)
void emu_seed_extend(const char* reference, const char* candidate, int xdrop, int right, uint32_t K, int32_t* ref_ext,
                     int32_t* cand_ext, int32_t* score, int32_t* stop) {
  std::vector<u8> ar(1 << 22);
  Arena A; A.init(ar.data(), (u32)ar.size());
  u32 rn = strlen(reference), cn = strlen(candidate);
  SeedExt e = seed_and_extension(bytes_view(reference, rn), bytes_view(candidate, cn), xdrop, right != 0, K, A, true, nullptr);
  *ref_ext = e.ref_ext; *cand_ext = e.cand_ext; *score = e.score; *stop = e.stop ? 1 : 0;
}
// talc_test_align_slices on the host: the same views and the same dispatch, with the scalar forms of the primitives
// (ops 0-5; result layout as there).  Returns -1 for an op it does not run.
int emu_align_slices(int op, const uint8_t* reads, const uint64_t* read_off, const int32_t* desc, uint32_t n, int aux,
                     int aux2, uint32_t K, int32_t* result) {
  if (op < 0 || op > 5) return -1;
  std::vector<u8> ar(1 << 22);
  for (u32 i = 0; i < n; ++i) {
    Arena A; A.init(ar.data(), (u32)ar.size());
    SeqView v[2];
    for (u32 s = 0; s < 2; ++s) {
      const int32_t* d = desc + 8 * i + 4 * s;
      ReadView rd;
      rd.s = reads + read_off[d[0]];
      rd.len = (u32)(read_off[d[0] + 1] - read_off[d[0]]);
      v[s] = selftest_view(rd, d[1], d[2], (u32)d[3], 2 * (u64)i + s, A);
    }
    i32 r[4] = {INT32_MIN, 0, 0, 0};
    if (!A.overflow) selftest_align_op(op, v[0], v[1], aux, aux2, K, A, r);
    if (op >= 3) memcpy(result + 4 * i, r, sizeof(r));
    else result[i] = r[0];
  }
  return 0;
}
void emu_std_sort_perm(const int64_t* keys, uint32_t n, uint32_t* perm) {
  for (u32 i = 0; i < n; ++i) perm[i] = i;
  std_sort(perm, perm + n, [keys](const u32& a, const u32& b) { return keys[a] < keys[b]; });
}
int emu_tag_next_nodes(const emu_params* q, const uint32_t* counts4, const uint32_t* colours4, uint32_t count, int complex_,
                       int32_t* tags4, double* dist4) {
  Params P = to_params(q);
  u8 tag[4] = {0, 0, 0, 0};
  const StepBounds sb = step_bounds(count, P);
  int n = tag_next_nodes(counts4, colours4, sb, P, complex_ != 0, tag);
  for (int i = 0; i < n; ++i) { tags4[i] = tag[i] == kExpected ? 0 : tag[i] == kUnexpected ? 1 : 7; dist4[i] = step_dist(count, counts4[i], sb); }
  return n;
}
// talc_test_model on the host: use_tabs = 0 runs the computed path (tabs.n = 0, as the emulated corrector does),
// use_tabs = 1 model tables of kModelTabN counts filled here with model_lower_bound / model_upper_bound
void emu_test_model(const emu_params* q, int op, const uint32_t* args, uint32_t n, int use_tabs, uint64_t* out) {
  Params P = to_params(q);
  std::vector<double> t;
  ModelTabs M;
  M.n = 0;
  M.lower = M.upper = M.sq = nullptr;
  if (use_tabs) {
    t.resize(3 * (size_t)kModelTabN);
    for (u32 c = 0; c < kModelTabN; ++c) {
      t[c] = model_lower_bound(c, P.alpha);
      t[kModelTabN + c] = model_upper_bound(c, P.alpha);
      t[2 * kModelTabN + c] = sqrt((double)c);
    }
    M.lower = t.data();
    M.upper = t.data() + kModelTabN;
    M.sq = t.data() + 2 * kModelTabN;
    M.n = kModelTabN;
  }
  for (u32 i = 0; i < n; ++i) selftest_model_op(op, args + 8 * (u64)i, P, M, out + 9 * (u64)i);
}
}
