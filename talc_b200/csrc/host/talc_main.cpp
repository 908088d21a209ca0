// talc_main.cpp -- the drop-in `talc` command line on top of libtalc_b200.so.
//
// Same interface and the same output files as the reference program (main.cpp:83-325):
//   talc <reads.fa|fq> --SRCounts <dump> [--junctions <dump>] -k <K> [-o <prefix>] [-t <N>] [--reverse] [tunables]
//   <prefix>.config.txt (Settings.cpp:160-185)   <prefix>.stats_basics.txt header (Read.cpp:394-415)
//   <prefix>.log, appended, one line per failed read (io.cpp:105-111; messages main.cpp:290,294)
//   <prefix>.fa, every read in input order, 70 columns (main.cpp:310, io.cpp:50-75)
// Exit codes follow main.cpp: 1 on a parse error (:199) or an empty table (:320), 0 otherwise -- including
// unreadable input (:323).  The work is done on the GPU through the C ABI; there is no CPU path.
// -t is accepted for compatibility and used for host-side FASTA formatting only.
//
// Unlike the reference (loadSeqData holds every read, outputSeqData writes them all at the end: main.cpp:219,310) the
// reads are STREAMED: a reader parses FASTA / FASTQ incrementally into batches (--batch-reads, --batch-bases), each
// batch goes through a talc_stream (copies, kernels and formatting overlapped) and a writer appends the corrected
// records in input order.  Host memory is bounded by the batches in flight, whatever the size of the input.
// Extensions: --gpus N deals the batches round-robin over N devices (table replicated with one NCCL broadcast issued
// by the library, or with peer copies: --replicate peer), --tableCache <file>, --readStats (the per-read rows of Read.cpp:418-433 the reference left disabled
// at main.cpp:305).
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <chrono>
#include <condition_variable>
#include <deque>
#include <fstream>
#include <iostream>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <unistd.h>
#include <vector>

#include "reads_io.hpp"
#include "talc_b200.h"

struct Cli {
  std::string reads, dump, junctions, out = "out", queryMode = "memory", tableCache, replicate = "nccl";
  bool useJunctions = false, reverse = false, readStats = false;
  int threads = 1, gpus = 1;
  long batchReads = 131072, batchBases = 256l << 20;
  talc_params p;
  bool haveK = false, haveSR = false;
};

static bool to_int(const std::string& s, long& v) {
  char* e = nullptr;
  v = strtol(s.c_str(), &e, 10);
  return e && *e == 0 && !s.empty();
}
static bool to_dbl(const std::string& s, double& v) {
  char* e = nullptr;
  v = strtod(s.c_str(), &e);
  return e && *e == 0 && !s.empty();
}

// mirrors the option table of main.cpp:101-195 (SeqAn ArgumentParser: "-x" short and "--long" names)
static int parse(int argc, const char** argv, Cli& c) {
  talc_params_default(&c.p, 21);
  std::vector<std::string> pos;
  for (int i = 1; i < argc; ++i) {
    const std::string a = argv[i];
    auto val = [&](std::string& dst) { if (i + 1 >= argc) return false; dst = argv[++i]; return true; };
    std::string v;
    long n;
    double d;
    if (a == "-h" || a == "--help" || a == "--version") return 2;
    else if (a == "-o" || a == "--output") { if (!val(c.out)) return 1; }
    else if (a == "-k" || a == "--kmerSize") { if (!val(v) || !to_int(v, n) || n < 18 || n > 30) return 1; c.p.K = (uint32_t)n; c.haveK = true; }
    else if (a == "-qm" || a == "--query-mode") { if (!val(c.queryMode) || (c.queryMode != "memory" && c.queryMode != "jellyfish2")) return 1; }
    else if (a == "-SR" || a == "--SRCounts") { if (!val(c.dump)) return 1; c.haveSR = true; }
    else if (a == "-j" || a == "--junctions") { if (!val(c.junctions)) return 1; c.useJunctions = true; }
    else if (a == "--tableCache") { if (!val(c.tableCache)) return 1; }  // extension: binary cache of the built table
    else if (a == "--replicate") { if (!val(c.replicate) || (c.replicate != "nccl" && c.replicate != "peer")) return 1; }
    else if (a == "-jf2" || a == "--pathToJF2") { if (!val(v)) return 1; }
    else if (a == "-MIN_INNER_SCORE" || a == "--MIN_INNER_SCORE") { if (!val(v) || !to_dbl(v, d) || d < 0.3 || d > 0.9) return 1; c.p.min_inner_score = d; }
    else if (a == "-MIN_BORDER_SCORE" || a == "--MIN_BORDER_SCORE") { if (!val(v) || !to_dbl(v, d) || d < 0.5 || d > 0.9) return 1; c.p.min_border_score = d; }
    else if (a == "-MIN_COUNT" || a == "--MIN_COUNT") { if (!val(v) || !to_int(v, n) || n < 2) return 1; c.p.min_count = (uint32_t)n; }
    else if (a == "-SR_ERROR_RATE" || a == "--SR_ERROR_RATE") { if (!val(v) || !to_dbl(v, d) || d < 0.01 || d > 0.1) return 1; c.p.sr_error_rate = d; }
    else if (a == "-WINDOW_SIZE" || a == "--WINDOW_SIZE") { if (!val(v) || !to_int(v, n) || n < 6) return 1; c.p.window_size = (uint32_t)n; }
    else if (a == "-MAX_NB_BRANCHES" || a == "--MAX_NB_BRANCHES") { if (!val(v) || !to_int(v, n) || n < 5) return 1; c.p.max_nb_branches = (uint32_t)n; }
    else if (a == "-ALPHA_FOR_PRED" || a == "--ALPHA_FOR_PRED") { if (!val(v) || !to_dbl(v, d) || d < 0.67) return 1; c.p.alpha = d; }
    else if (a == "-t" || a == "--num_threads") { if (!val(v) || !to_int(v, n) || n < 1) return 1; c.threads = (int)n; }
    else if (a == "-DEBUG_MODE" || a == "--DEBUG_MODE") { if (!val(v)) return 1; }
    else if (a == "-rev" || a == "--reverse") { c.reverse = true; }
    else if (a == "--readStats") { c.readStats = true; }
    else if (a == "--batch-reads") { if (!val(v) || !to_int(v, n) || n < 1) return 1; c.batchReads = n; }
    else if (a == "--batch-bases") { if (!val(v) || !to_int(v, n) || n < 1) return 1; c.batchBases = n; }
    else if (a == "--gpus") { if (!val(v) || !to_int(v, n) || n < 1) return 1; c.gpus = (int)n; }
    else if (a == "--cycle-mode") { if (!val(v) || !to_int(v, n)) return 1; c.p.cycle_mode = (int32_t)n; }
    else if (a.size() > 1 && a[0] == '-') return 1;
    else pos.push_back(a);
  }
  if (pos.size() != 1 || !c.haveK || !c.haveSR) return 1;
  if (c.queryMode != "memory") { std::cerr << "talc: only query mode 'memory' is supported\n"; return 1; }
  c.reads = pos[0];
  return 0;
}

static void write_config(const Cli& c) {  // Settings.cpp:160-185
  std::ofstream f(c.out + ".config.txt", std::ios_base::trunc);
  f << "TALC: Parameters used for sample: " << c.out << "\n"
    << "****************************\n"
    << "INPUT=" << c.reads << "\n"
    << "OUTPUT=" << c.out << "\n"
    << "STATS=" << c.out << ".stats_basics.txt" << "\n"
    << "****************************\n"
    << "KmerSize=" << c.p.K << "\n"
    << "Junction mode activated? " << c.useJunctions << "\n"
    << "queryMode=" << c.queryMode << "\n"
    << "****************************\n"
    << "MIN_INNER_SCORE=" << c.p.min_inner_score << "\n"
    << "MIN_BORDER_SCORE=" << c.p.min_border_score << "\n"
    << "MAX_NB_BRANCHES=" << c.p.max_nb_branches << "\n"
    << "ALPHA=" << c.p.alpha << "\n"
    << "MIN_SR_COUNT=" << c.p.min_count << "\n"
    << "WINDOW_SIZE=" << c.p.window_size << "\n"
    << "****************************" << std::endl;
}
static void write_stats_header(const std::string& path) {  // Read.cpp:394-415
  std::ofstream f(path, std::ios_base::trunc);
  f << "read_name\traw_length\twhead_length\twtail_length\tnbInKmers\tnbSolidKmers\tnbSolidReg\tnbInWeakReg\t"
       "nbInCorrReg\tCorrHead?\tCorrHeadLen\tCorrTail?\tCorrTailLen\tCorrlength\tnbInKmers2\n";
}

int main(int argc, const char** argv) {
  std::cout << "******************************************************\n"
            << "* TALC : Transcriptome-Aware Long Read Correction    *\n"
            << "*        B200 build (libtalc_b200)                   *\n"
            << "******************************************************" << std::endl;
  Cli cli;
  const int pr = parse(argc, argv, cli);
  if (pr == 2) {
    std::cout << "talc <reads> --SRCounts <dump> [--junctions <dump>] -k <K> [-o <prefix>] [-t <N>] [--reverse] [--gpus <N>] [--tableCache <file>]"
                 " [--batch-reads <N>] [--batch-bases <N>] [--readStats] [--replicate nccl|peer]\n";
    return 0;
  }
  if (pr != 0) { std::cerr << "talc: PARSE_ERROR\n"; return 1; }
  write_config(cli);
  write_stats_header(cli.out + ".stats_basics.txt");

  std::cout << "[TALC]: Attempting to load sequences." << std::endl;
  ReadParser parser(cli.reads);
  if (!parser.is_open()) {
    std::cerr << "ERROR: Could not open file " << cli.reads << "\n";
    std::cout << "[TALC]: ISSUE WITH INPUT FILES" << std::endl;
    return 0;  // main.cpp:323 falls off main
  }
  // the first batch is parsed before the table is built: an input that is not FASTA / FASTQ ends the run here, as in
  // the reference (which loads every read first)
  auto first = std::make_shared<Batch>();
  if (!parser.next_batch(*first, (size_t)cli.batchReads, (size_t)cli.batchBases)) {
    std::cout << "[TALC]: ISSUE WITH INPUT FILES" << std::endl;
    return 0;
  }

  const auto tStart = std::chrono::steady_clock::now();
  auto since = [&](std::chrono::steady_clock::time_point t0) { return std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count(); };
  std::vector<talc_ctx*> ctx(cli.gpus, nullptr);
  for (int g = 0; g < cli.gpus; ++g) {  // (one thread per device was measured: no faster, the driver serialises it)
    if (talc_ctx_create(&cli.p, g, &ctx[g]) != 0) {
      std::cerr << "talc: cannot create a GPU context on device " << g << ": " << talc_last_error(nullptr) << "\n";
      return 2;
    }
    // --reverse (main.cpp:253,285-286): the long reads only; the stream's lanes follow their context
    if (cli.reverse && talc_ctx_set_reverse(ctx[g], 1) != 0) {
      std::cerr << "talc: " << talc_last_error(ctx[g]) << "\n";
      return 2;
    }
  }
  const double sCtx = since(tStart);
  const auto tTable = std::chrono::steady_clock::now();
  uint64_t nLines = 0, nKept = 0;
  int rc = -1;
  // --tableCache <file> (extension, SURVEY row f1): reuse the built table if the file exists, else build it from the
  // dump and write the file; a cache made from other --SRCounts / --junctions files (size, mtime), another -k or
  // MIN_COUNT is refused by the library and rebuilt
  if (!cli.tableCache.empty())
    rc = talc_table_load_cache_for(ctx[0], cli.tableCache.c_str(), cli.dump.c_str(),
                                   cli.useJunctions ? cli.junctions.c_str() : nullptr, &nKept);
  if (rc == TALC_ERR_STALE) std::cout << "[TALC]: " << talc_last_error(ctx[0]) << " -> rebuilding it." << std::endl;
  if (rc != 0) {
    rc = talc_table_load_dump(ctx[0], cli.dump.c_str(), cli.useJunctions ? cli.junctions.c_str() : nullptr, &nLines, &nKept);
    if (rc == 0 && nKept > 0 && !cli.tableCache.empty() && talc_table_save(ctx[0], cli.tableCache.c_str()) != 0)
      std::cerr << "talc: " << talc_last_error(ctx[0]) << "\n";
  }
  if (rc != 0) { std::cerr << "talc: " << talc_last_error(ctx[0]) << "\n"; nKept = 0; }
  std::cout << "[TALC]: SR-dBG contains " << nKept << " nodes." << std::endl;
  if (nKept == 0) {
    std::cout << "[TALC]: The de Bruijn Graph is empty...Correction aborted." << std::endl;
    return 1;  // main.cpp:320
  }
  const double sTable = since(tTable);
  const auto tRep = std::chrono::steady_clock::now();
  if (cli.gpus > 1) {
    double ms = 0;
    int usedNccl = 0;
    if (cli.replicate == "peer") {
      // --replicate peer: one cudaMemcpyPeer per replica instead of the NCCL broadcast -- no communicator to set up
      // (~3 s in a process that has not used NCCL yet), at the price of N-1 sequential copies from device 0
      for (int g = 1; g < cli.gpus; ++g)
        if (talc_table_copy(ctx[g], ctx[0]) != 0) {
          std::cerr << "talc: " << talc_last_error(ctx[g]) << "\n";
          return 2;
        }
      std::cout << "[TALC]: k-mer table replicated on " << cli.gpus << " GPUs (peer copies)." << std::endl;
    } else if (talc_table_replicate(ctx.data(), cli.gpus, &ms, &usedNccl) != 0) {
      std::cerr << "talc: " << talc_last_error(ctx[0]) << "\n";
      return 2;
    } else if (usedNccl) std::cout << "[TALC]: k-mer table replicated on " << cli.gpus << " GPUs (one NCCL broadcast, " << ms << " ms)." << std::endl;
    else std::cout << "[TALC]: k-mer table replicated on " << cli.gpus << " GPUs (peer copies; NCCL not found)." << std::endl;
  }
  const double sRep = since(tRep);
  // one stream per device; its pinned staging is page-locked now, one thread per device, and not while the table
  // loads or NCCL starts up: page-locking contends with every other mapping the process makes (measured: table load
  // 0.25 -> 2.7 s, NCCL start-up 1 -> 8 s when run side by side)
  const auto tOpen = std::chrono::steady_clock::now();
  std::vector<talc_stream*> streams(cli.gpus, nullptr);
  {
    std::vector<int> openRc(cli.gpus, 0);
    std::vector<std::thread> openers;
    for (int g = 0; g < cli.gpus; ++g)
      openers.emplace_back([&, g]() {
        openRc[g] = talc_stream_open(ctx[g], cli.readStats ? 1 : 0, &streams[g]);
        if (openRc[g] == 0)
          openRc[g] = talc_stream_reserve(streams[g], (uint32_t)cli.batchReads, (uint64_t)cli.batchBases + (8u << 20));
      });
    for (auto& t : openers) t.join();
    for (int g = 0; g < cli.gpus; ++g) {
      if (openRc[g] != 0) {
        std::cerr << "talc: cannot open a stream on device " << g << ": " << (streams[g] ? talc_stream_last_error(streams[g]) : talc_last_error(ctx[g])) << "\n";
        return 2;
      }
    }
  }
  const double sOpen = since(tOpen);
  const auto tCorr = std::chrono::steady_clock::now();

  // ---- writer: corrected records in input order into <o>.fa.partial, renamed when the run is complete; the failed-read
  // log (input order = the reference's order under -t 1) and the optional stats rows are appended as batches arrive
  const std::string faTmp = cli.out + ".fa.partial";
  FILE* fo = fopen(faTmp.c_str(), "wb");
  if (!fo) { std::cerr << "ERROR: Could not open the file " << cli.out << ".fa\n"; return 0; }
  IdQueue idq;
  int writerRc = 0;
  uint64_t nReads = 0, nResource = 0;
  double sWait = 0, sFormat = 0, sWrite = 0, sParse = 0, sSubmit = 0;  // where the threads of this phase spent their time
  std::thread writer([&]() {
    std::ofstream lg, st;
    std::vector<std::string> parts;
    while (auto b = idq.pop()) {
      talc_stream* s = streams[b->seq % cli.gpus];
      const uint8_t *out = nullptr, *status = nullptr;
      const uint64_t* ooffs = nullptr;
      const uint32_t* stats = nullptr;
      uint32_t n = 0;
      auto t0 = std::chrono::steady_clock::now();
      const int nrc = talc_stream_next(s, &out, &ooffs, &status, &n, &stats, nullptr);
      sWait += since(t0);
      if (nrc != 0 || n != b->ids.size()) {
        std::cerr << "talc: correction failed on device " << (b->seq % cli.gpus) << ": " << talc_stream_last_error(s) << "\n";
        writerRc = 2;
        while (idq.pop()) {}  // keep draining so that the reader does not block for ever
        return;
      }
      for (uint32_t r = 0; r < n; ++r) {
        const uint8_t v = status[r];
        const char* msg = v == TALC_READ_NO_STRUCTURE ? "Unable to define convenient structure."
                          : v == TALC_READ_NO_SOLID   ? "No solid kmer could be found." : nullptr;
        if (msg) {
          if (!lg.is_open()) lg.open(cli.out + ".log", std::ios_base::app);
          lg << "[Read: " << b->ids[r] << " ]: " << msg << std::endl;
        }
        if (v == TALC_READ_RESOURCE) {
          ++nResource;
          std::cerr << "talc: read " << b->ids[r] << " outgrew the scratch arena and is passed through uncorrected\n";
        }
        if (cli.readStats && v != TALC_READ_SHORT) {  // outputBasicReadStats, Read.cpp:418-433 (only reads longer than K)
          if (!st.is_open()) st.open(cli.out + ".stats_basics.txt", std::ios_base::app);
          const uint64_t rawLen = b->offs[r + 1] - b->offs[r];
          st << "\n" << b->ids[r] << "\t" << rawLen << "\t" << (stats ? stats[2 * r] : 0) << "\t" << (stats ? stats[2 * r + 1] : 0)
             << "\t" << (v == TALC_READ_OK ? ooffs[r + 1] - ooffs[r] : 0);
        }
      }
      t0 = std::chrono::steady_clock::now();
      format_fasta(*b, out, ooffs, cli.threads, parts);
      sFormat += since(t0);
      t0 = std::chrono::steady_clock::now();
      for (const auto& p : parts) fwrite(p.data(), 1, p.size(), fo);
      sWrite += since(t0);
      nReads += n;
    }
  });

  // ---- reader / submitter (this thread): batch b goes to device b mod N; submit blocks while that device's ring of
  // slots is full, which bounds the memory in flight
  bool inputOk = true;
  int submitRc = 0;
  uint64_t seq = 0;
  for (std::shared_ptr<Batch> b = first; b && !b->ids.empty();) {
    b->seq = seq;
    talc_stream* s = streams[seq % cli.gpus];
    if (b->offs.size() != b->ids.size() + 1) { inputOk = false; break; }
    auto t0 = std::chrono::steady_clock::now();
    const int src = talc_stream_submit(s, b->bases.data(), b->offs.data(), (uint32_t)b->ids.size());
    sSubmit += since(t0);
    if (src != 0) {
      std::cerr << "talc: " << talc_stream_last_error(s) << "\n";
      submitRc = 2;
      break;
    }
    std::vector<uint8_t>().swap(b->bases);  // the stream holds its own copy; ids and offsets stay for the writer
    idq.push(b);                            // only now: the writer fetches what has been submitted
    ++seq;
    if (writerRc) break;
    auto nb = std::make_shared<Batch>();
    t0 = std::chrono::steady_clock::now();
    const bool parsed = parser.next_batch(*nb, (size_t)cli.batchReads, (size_t)cli.batchBases);
    sParse += since(t0);
    if (!parsed) { inputOk = false; break; }
    b = nb;
  }
  idq.finish();
  writer.join();
  fclose(fo);
  const double sCorr = since(tCorr);
  // error paths release everything in order; a complete run leaves the buffers to the process exit (unpinning and
  // freeing several GB per device one allocation at a time took 0.3 s on one GPU and 2.5 s on two)
  auto teardown = [&]() {
    for (auto* s : streams) talc_stream_close(s);
    for (auto* c : ctx) talc_ctx_destroy(c);
  };
  if (submitRc || writerRc || !inputOk) teardown();
  if (submitRc || writerRc) { remove(faTmp.c_str()); return 2; }
  if (!inputOk) {  // the reference would have failed while loading, before writing anything
    remove(faTmp.c_str());
    std::cout << "[TALC]: ISSUE WITH INPUT FILES" << std::endl;
    return 0;
  }
  if (rename(faTmp.c_str(), (cli.out + ".fa").c_str()) != 0) {
    std::cerr << "ERROR: Could not open the file " << cli.out << ".fa\n";
    return 0;
  }
  std::cout << "[TALC]: " << nReads << " long read(s) processed" << std::endl;
  std::cout << "[TALC]: seconds: contexts " << sCtx << ", table " << sTable << ", replication " << sRep << ", staging " << sOpen << ", correction (read + correct + write) "
            << sCorr << " [reader: parse " << sParse << ", submit " << sSubmit << "; writer: wait " << sWait << ", format " << sFormat
            << ", write " << sWrite << "]" << std::endl;
  std::cout << "[TALC]: Looks like we are done now." << std::endl;
  std::cout.flush();
  std::cerr.flush();
  fflush(nullptr);
  _exit(0);  // outputs are closed and renamed; see the note on teardown above
}
