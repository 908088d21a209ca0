/* talc_b200.h -- C ABI of the B200 correction library (libtalc_b200.so).
 *
 * TALC (lbroseus/TALC) has no plugin / FFI interface of its own; the drop-in surface is the `talc`
 * command line and its output files.  This ABI replaces the *internal seam* of the reference, i.e.
 * exactly the calls main() makes on the hot path (all paths relative to /root/reference/src):
 *
 *   talc_table_load_dump / talc_table_load_packed
 *       <- SR_DBG = buildCDBG(1, dump, jdump); decolourRepeatsFromDBG(SR_DBG, K);   main.cpp:231-232
 *          (Jellyfish.cpp:236-295, utils.cpp:658-669)
 *   talc_correct_batch / talc_correct_batch_device
 *       <- the body of the OpenMP loop over reads                                  main.cpp:247-306
 *          Read r(id,seq); if len>K: r.reCoverage() -> r.defineStructure2() -> r.correct2(); r.getCorrSeq()
 *          (Read.cpp:174-386, Explorer.cpp, Trail.cpp, Trajectory.cpp)
 *   talc_ctx_set_reverse
 *       <- if (reverse) reverseComplement(seq) before, and of the corrected read after, the above   main.cpp:253,285-286
 *   talc_ctx_set_strand / talc_orient_batch / talc_last_strands / talc_stream_strands
 *       <- not in the reference: the strand chosen per read (--strand auto), for inputs of both orientations
 *   talc_ctx_set_pieces / talc_pieces_batch / talc_last_pieces / talc_stream_pieces
 *       <- not in the reference: the table-supported stretches of each corrected read (--trim, --split)
 *   talc_coverage_batch
 *       <- getLRCountsInSR(seq, K, SR_DBG, ..)                                     Jellyfish.cpp:471-496
 *   talc_table_lookup
 *       <- dBG.count(kmer) / dBG.at(kmer)                                          Jellyfish.cpp:317-318,492-493
 *   per-read `status[]` <- the two throwToLog() messages of main.cpp:290,294 (io.cpp:105-111)
 *
 * Conventions: plain pointers and sizes, no C++ or torch types; every function returns 0 on success
 * and a negative code on failure (message via talc_last_error); no exception crosses the boundary.
 * The caller owns every buffer it passes in; the library owns its device memory inside talc_ctx.
 * A context is bound to one CUDA device and is not thread-safe.  There is no CPU fallback: without a
 * usable CUDA device talc_ctx_create fails.
 *
 * k-mers are 2-bit packed into uint64_t with the FIRST base in the MOST significant position
 * (A=0, C=1, G=2, T=3), K <= 31.  Reads are ASCII (ACGTN, either case; anything else reads as N, the
 * way SeqAn converts char -> Dna5); corrected reads come back as upper-case ACGTN.
 */
#ifndef TALC_B200_H
#define TALC_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct talc_ctx talc_ctx;

/* Settings.cpp:33-69 (set by main.cpp:94-195 / Settings.cpp:74-123); defaults via talc_params_default */
typedef struct talc_params {
  uint32_t K;                       /* -k, 18..30 (main.cpp:112-116); up to 31 accepted by the library */
  uint32_t min_count;               /* --MIN_COUNT        gp_MIN_COUNT (2)              */
  uint32_t window_size;             /* --WINDOW_SIZE      gp_WINDOW_SIZE (9)            */
  uint32_t max_nb_branches;         /* --MAX_NB_BRANCHES  gp_MAX_NB_COMPETING_PATHS (7) */
  double alpha;                     /* --ALPHA_FOR_PRED   gp_ALPHA (2.57)               */
  double sr_error_rate;             /* --SR_ERROR_RATE    gp_SR_ERROR_RATE (0.025); the command line takes [0.01, 0.1],
                                       talc_ctx_create refuses NaN and anything outside [0, 0.5] (TALC_ERR_ARG) */
  double min_inner_score;           /* --MIN_INNER_SCORE  (0.7)                         */
  double min_border_score;          /* --MIN_BORDER_SCORE (0.7)                         */
  int32_t cycle_mode;               /* 0: SeqAn2 Horspool over mixed alphabets (default), 1: exact first occurrence */
  int32_t q11_zero_init;            /* Explorer.cpp:705 uninitialised counter behaves as 0 (default 1) */
} talc_params;

/* per-read outcome: main.cpp:262 (short), :290 (no structure), :294 (no solid k-mer) */
enum {
  TALC_READ_OK = 0,
  TALC_READ_NO_SOLID = 1,      /* log: "No solid kmer could be found."            */
  TALC_READ_NO_STRUCTURE = 2,  /* log: "Unable to define convenient structure."   */
  TALC_READ_SHORT = 3,         /* len <= K: passed through, nothing logged        */
  TALC_READ_RESOURCE = 4       /* not in the reference (which has no memory bound): the search of this read outgrew even
                                  the second-tier scratch arena (talc_ctx_set_scratch); the read is passed through
                                  uncorrected and counted in talc_counters.reads_overflow; the batch itself succeeds.
                                  In reverse mode (talc_ctx_set_reverse) it comes back like every other read that is not
                                  TALC_READ_OK: as the reverse complement of its input */
};

/* algorithmic work of a batch (properties of the algorithm on the input, SURVEY 8d) and timings */
typedef struct talc_counters {
  uint64_t lookups_seg, lookups_deg, lookups_walk;
  uint64_t steps_inner, steps_border, frontier_sum;
  uint64_t cells_nw, cells_lcs, cells_ovl, cells_xdrop;
  uint64_t gaps, gaps_bridged, gap_attempts, borders, borders_corrected;
  uint64_t ev_gardening, ev_bridge, ev_edge, ev_cycle;
  uint64_t bases_out, reads_ok, reads_overflow;
  /* filled by the host side of the call */
  uint64_t reads, bases_in, reads_second_tier, kernel_launches;
  uint64_t rounds;   /* control / walk kernel rounds of the call (0 in monolithic mode) */
  double ms_h2d, ms_coverage, ms_correct, ms_correct_tier2, ms_gather, ms_d2h, ms_total;
} talc_counters;

enum {
  TALC_OK = 0,
  TALC_ERR_ARG = -1,
  TALC_ERR_CUDA = -2,
  TALC_ERR_IO = -3,
  TALC_ERR_NO_TABLE = -4,
  TALC_ERR_CAPACITY = -5,   /* an output buffer supplied by the caller is too small */
  TALC_ERR_NCCL = -8,       /* libnccl.so.2 could not be loaded, or an NCCL call failed */
  TALC_ERR_STALE = -7,      /* a table cache made for other inputs / parameters: rebuild from the dump */
  TALC_ERR_SCRATCH = -6     /* reserved (a read that exhausts the second-tier arena is data: TALC_READ_RESOURCE) */
};

void talc_params_default(talc_params* p, uint32_t K);
/* sha256 prefix of the sources this binary was compiled from (talc_b200/build.py refuses a stale prebuilt library) */
const char* talc_build_source_hash(void);

int talc_ctx_create(const talc_params* p, int cuda_device, talc_ctx** out);
void talc_ctx_destroy(talc_ctx* ctx);
const char* talc_last_error(talc_ctx* ctx);   /* ctx may be NULL: last create error */

/* A lane: a second context on the same device that borrows the tables of `parent` and follows its settings, with its
 * own CUDA stream and scratch memory.  Two host threads correcting batches through a context and its lane overlap on
 * the device: a batch ends with a tail of a few long reads (one warp per read), and the other batch's blocks fill the
 * SMs that tail leaves idle (+8 % on the bench workload).  The streamed calls below use a lane internally.  Table
 * loading calls are refused on a lane; destroy it (talc_ctx_destroy) before its parent.  No reference counterpart
 * (the reference's unit of concurrency is the OpenMP thread of main.cpp:247).                                       */
int talc_ctx_create_lane(talc_ctx* parent, talc_ctx** lane);

/* scratch sizing (optional): bytes per thread for the first and second tier, warps (= reads in flight) of the second tier */
int talc_ctx_set_scratch(talc_ctx* ctx, uint32_t tier1_bytes, uint32_t tier2_bytes, uint32_t tier2_threads);

/* execution shape of the correction kernels; 0 keeps a value.  split_walk: 1 (default) = reads are suspendable programs
 * whose long graph walks run in a separate lane-per-trail kernel (csrc/walk.cuh), 2 = one monolithic kernel per batch
 * (the round-1 shape, kept for A/B measurements).  Results are identical (tests/test_gpu_parity.py).  read_contexts =
 * reads in flight in split mode (each owns a first-tier arena), walk_step_cap = steps per frontier and round.  */
int talc_ctx_set_exec(talc_ctx* ctx, uint32_t split_walk, uint32_t read_contexts, uint32_t walk_step_cap);

/* main.cpp:253,285-286 (--reverse): long reads sequenced from the strand opposite to the short reads.  reverse != 0:
 * every read is reverse-complemented (Dna5: ACGT in either case -> complement, anything else -> N) before anything
 * else, the len <= K test included; a corrected read comes back as the reverse complement of its corrected sequence,
 * i.e. in the read's input orientation; every other read comes back as the reverse complement of its input (SURVEY
 * Q24: the reference does not undo the flip for reads it cannot correct).  Coverage (talc_coverage_batch) and the
 * read_stats of the stream describe the reverse-complemented read.  The k-mer table is not affected.  Set on a
 * context, not on a lane (a lane follows its parent, TALC_ERR_ARG on a lane); not while a stream on the context has
 * batches pending.  Default 0.                                                                                     */
int talc_ctx_set_reverse(talc_ctx* ctx, int reverse);

/* Strand mode of the correction (not in the reference; talc --strand).  A k-mer table counted from short reads holds
 * one strand, so a long read finds solid k-mers only on that strand; cDNA long-read libraries mix sense and antisense
 * reads.
 *   TALC_STRAND_FORWARD (default)  every read as it is
 *   TALC_STRAND_REVERSE            talc_ctx_set_reverse(ctx, 1): every read on the opposite strand
 *   TALC_STRAND_AUTO               each read on the strand where it finds more of the table.  For each read, found_fwd
 *                                  = its K-mer windows without N whose k-mer is in the table (count != 0), found_rc =
 *                                  the same for its Dna5 reverse complement (as talc_ctx_set_reverse builds it); strand
 *                                  1 (antisense) iff found_rc > found_fwd, ties (reads shorter than K, all-N reads,
 *                                  reverse palindromes) stay 0.  A strand-1 read is corrected exactly as reverse mode
 *                                  corrects it; EVERY read comes back in its input orientation: a corrected strand-1 read
 *                                  as the reverse complement of its correction, any other strand-1 read as its
 *                                  Dna5-normalised input (unlike reverse mode's Q24), strand-0 reads as in forward mode.
 *                                  Status, offsets and the algorithmic counters are those of forward mode on the batch
 *                                  with every strand-1 read reverse-complemented; the orientation probes are not counted
 *                                  in lookups_seg.  Coverage (talc_coverage_batch) and the read_stats of the stream
 *                                  describe each read on its chosen strand.
 * The same rules as talc_ctx_set_reverse: set on a context, not on a lane (TALC_ERR_ARG; a lane follows its parent),
 * not while a stream on the context has batches pending.  Another mode value is TALC_ERR_ARG.                     */
#define TALC_STRAND_FORWARD 0
#define TALC_STRAND_REVERSE 1
#define TALC_STRAND_AUTO 2
int talc_ctx_set_strand(talc_ctx* ctx, int mode);

/* ---- k-mer table (main.cpp:231-232) -------------------------------------------------------- */
/* Jellyfish `dump -c` text (KMER<ws>COUNT per line), optional junction dump (NULL = none).      */
int talc_table_load_dump(talc_ctx* ctx, const char* dump_path, const char* junction_path, uint64_t* n_lines,
                         uint64_t* n_kept);
/* load_dump parses the text ON THE GPU (row f1: file -> pinned staging -> HBM, one flag per byte, line offsets by
 * stream compaction, one thread per line; entries are inserted straight from device arrays).  load_dump_host is the
 * threaded host parser of round 1, kept for A/B timing; both build the same table bit for bit.                    */
int talc_table_load_dump_host(talc_ctx* ctx, const char* dump_path, const char* junction_path, uint64_t* n_lines,
                              uint64_t* n_kept);
/* Row f3 -- the table counted on the GPU straight from short-read files, replacing `jellyfish count` + `jellyfish dump -c`
 * (README.md:33-55 of the reference) and the text round trip: NON-canonical counts of every window of K consecutive
 * ACGT letters (either case) of every read of every file (paired-end: pass both files); FASTQ with four lines per
 * record or FASTA with one sequence line per record.  The sealed table holds the k-mers with count >= MIN_COUNT, i.e.
 * what buildCDBG keeps of the dump (Jellyfish.cpp:260); junction colours are applied as for a dump (NULL = none).
 * expected_distinct sizes the counting table like jellyfish's -s (0 = derived from the file sizes); TALC_ERR_CAPACITY
 * when it was too small.  n_kmers = occurrences counted, n_distinct = distinct k-mers seen, n_kept = entries kept.   */
int talc_table_count_reads(talc_ctx* ctx, const char* const* paths, int n_paths, uint64_t expected_distinct,
                           const char* junction_path_or_null, uint64_t* n_kmers, uint64_t* n_distinct, uint64_t* n_kept);
/* The same with an orientation per file (not in the reference; talc --SRLibType), so that the table holds one strand of
 * the transcriptome whatever the library: for each window x that SENSE counts (the windows are the same in every mode)
 *   TALC_SR_SENSE      x                                      (talc_table_count_reads: every file SENSE)
 *   TALC_SR_ANTISENSE  rc(x)                                  (R1 of fr-firststrand / dUTP, R2 of fr-secondstrand)
 *   TALC_SR_BOTH       x and rc(x), once when x == rc(x)      (unstranded: `jellyfish count -C`, expanded to both strands)
 * n_kmers = count increments (two per BOTH window that is not its own reverse complement).  With expected_distinct = 0 a
 * BOTH file adds size/2 to the sizing instead of size/4.  Another orient value is TALC_ERR_ARG.                     */
#define TALC_SR_SENSE 0
#define TALC_SR_ANTISENSE 1
#define TALC_SR_BOTH 2
int talc_table_count_reads_oriented(talc_ctx* ctx, const char* const* paths, const int* orient, int n_paths,
                                    uint64_t expected_distinct, const char* junction_path_or_null, uint64_t* n_kmers,
                                    uint64_t* n_distinct, uint64_t* n_kept);
/* load_dump with flags (talc_table_load_dump = flags 0).  TALC_DUMP_CANONICAL: the dump holds canonical counts
 * (`jellyfish count -C`); line i (x, c) stands for the two lines (x, c), (rc(x), c) at 2i and 2i+1, and the usual rules
 * (MIN_COUNT per line, first line wins, junction colours) apply to that expanded dump.  n_lines counts the dump's own
 * lines.  Other flag bits are TALC_ERR_ARG.                                                                          */
#define TALC_DUMP_CANONICAL 1u
int talc_table_load_dump_ex(talc_ctx* ctx, const char* dump_path, const char* junction_path, uint32_t flags,
                            uint64_t* n_lines, uint64_t* n_kept);
/* Jellyfish `dump -c` text of packed k-mers (KMER<space>COUNT\n, given order): the inverse of the parser, for tests,
 * benches and for exporting a table.  Host only.                                                                    */
int talc_dump_write_packed(const char* path, const uint64_t* keys, const int64_t* counts, uint64_t n, uint32_t K);
/* same, from packed k-mers in dump-line order; counts as the dump gives them (int)               */
int talc_table_load_packed(talc_ctx* ctx, const uint64_t* keys, const int64_t* counts, uint64_t n,
                           const uint64_t* jkeys, const int64_t* jcounts, uint64_t nj, int use_junctions,
                           uint64_t* n_kept);
/* replication across GPUs: rank 0 builds, every rank allocates the same capacity, the raw slot
 * array is broadcast (NCCL) between the device pointers below, then each rank seals its copy.     */
int talc_table_info(talc_ctx* ctx, uint64_t* capacity_slots, uint64_t* bytes, uint64_t* n_entries);
int talc_table_alloc(talc_ctx* ctx, uint64_t capacity_slots);
int talc_table_device_ptr(talc_ctx* ctx, void** device_ptr);
int talc_table_seal(talc_ctx* ctx, uint64_t n_entries);
/* the same two steps with a caller-owned DEVICE staging buffer of `bytes` = capacity*16 (e.g. the
 * tensor handed to ncclBroadcast): export copies the sealed table out, import allocates+copies+seals */
int talc_table_export_device(talc_ctx* ctx, void* dst_device, uint64_t bytes);
int talc_table_import_device(talc_ctx* ctx, const void* src_device, uint64_t capacity_slots, uint64_t n_entries);
/* single-process replication: copy src's sealed table to dst's device (peer copy over NVLink)    */
int talc_table_copy(talc_ctx* dst, talc_ctx* src);
/* The collective of the path, owned by the library (SURVEY 8e): ONE ncclBroadcast of the slot array after the build.
 * NCCL is bound at run time (dlopen libnccl.so.2 -- inside torchrun the copy torch loaded, else the system one).
 *   talc_table_replicate   one process, n contexts on n devices: ctxs[0] holds the table, the others receive it
 *                          (ncclCommInitAll + one grouped broadcast; peer copies if NCCL is absent: *used_nccl = 0)
 *   talc_nccl_unique_id /  one process per GPU: rank 0 makes the id, hands its 128 bytes to the other ranks by any
 *   talc_table_broadcast   means, every rank calls talc_table_broadcast(ctx, id, rank, world, root): geometry, then
 *                          the slot array in one broadcast; receivers allocate, receive and seal                   */
int talc_nccl_available(void);
int talc_table_replicate(talc_ctx** ctxs, int n, double* broadcast_ms, int* used_nccl);
int talc_nccl_unique_id(uint8_t id[128]);
int talc_table_broadcast(talc_ctx* ctx, const uint8_t id[128], int rank, int world, int root, double* broadcast_ms);
/* binary cache of the built table (SURVEY 8f row f1: at 30 M+ lines the text parse of buildCDBG,
 * Jellyfish.cpp:251-269, dominates start-up once correction is fast).  save writes the sealed slot array with a
 * small header (magic, K, MIN_COUNT, capacity, entries, provenance); load checks K and MIN_COUNT against the context,
 * uploads the array and seals it -- the result is the table the dump would have built.            */
int talc_table_save(talc_ctx* ctx, const char* path);
int talc_table_load_cache(talc_ctx* ctx, const char* path, uint64_t* n_entries);
/* The header also records whether junction colours were baked in and the size + mtime of the --SRCounts / --junctions
 * files the table was built from.  load_cache_for refuses (TALC_ERR_STALE) a cache made from other inputs, so that a
 * file left over from another run is rebuilt instead of silently used; both loaders check the file size against the
 * header, recount the occupied slots on the device and refuse a table that is more than half full.            */
int talc_table_load_cache_for(talc_ctx* ctx, const char* path, const char* dump_path, const char* junction_path_or_null,
                              uint64_t* n_entries);
/* The header also records the TALC_DUMP_* flags the dump was loaded with (0 in caches written before they existed);
 * load_cache_for_ex refuses (TALC_ERR_STALE) a cache with other flags, load_cache_for is flags = 0.  talc_table_copy
 * and the replication calls carry the flags to the copies.                                                         */
int talc_table_load_cache_for_ex(talc_ctx* ctx, const char* path, const char* dump_path, const char* junction_path_or_null,
                                 uint32_t flags, uint64_t* n_entries);
/* point look-ups from the host (tests, debugging): found[i] in {0,1}                              */
int talc_table_lookup(talc_ctx* ctx, const uint64_t* keys, uint64_t n, uint32_t* counts, uint32_t* colours,
                      uint8_t* found);

/* ---- correction (main.cpp:247-306) ----------------------------------------------------------- */
/* Host buffers.  bases: the reads concatenated; offsets[n_reads+1].  out / out_offsets[n_reads+1] /
 * status[n_reads] receive the corrected reads in input order; uncorrectable reads come back as
 * their (Dna5-normalised) input with a non-zero status.  counters may be NULL.                    */
int talc_correct_batch(talc_ctx* ctx, const uint8_t* bases, const uint64_t* offsets, uint32_t n_reads, uint8_t* out,
                       uint64_t out_capacity, uint64_t* out_offsets, uint8_t* status, talc_counters* counters);
/* Same with every buffer already resident on the context's device (no host<->device copies).      */
int talc_correct_batch_device(talc_ctx* ctx, const uint8_t* d_bases, const uint64_t* d_offsets, uint32_t n_reads,
                              uint64_t total_bases, uint8_t* d_out, uint64_t out_capacity, uint64_t* d_out_offsets,
                              uint8_t* d_status, talc_counters* counters);
/* Per-read coverage vectors only (Read::reCoverage): counts[sum(max(0,len-K+1))], host buffers.   */
int talc_coverage_batch(talc_ctx* ctx, const uint8_t* bases, const uint64_t* offsets, uint32_t n_reads,
                        uint32_t* counts, uint64_t counts_capacity);
/* The decision of TALC_STRAND_AUTO without correcting, in any strand mode (e.g. to orient reads for other tools).
 * Host buffers: offsets[n_reads+1] with offsets[0] == 0, strand[n_reads] in {0,1}; found_fwd[n_reads] and
 * found_rc[n_reads] may be NULL.                                                                                  */
int talc_orient_batch(talc_ctx* ctx, const uint8_t* bases, const uint64_t* offsets, uint32_t n_reads, uint8_t* strand,
                      uint32_t* found_fwd, uint32_t* found_rc);
/* The strands (0 / 1) of the first n reads of the last batch corrected through this context (talc_correct_batch,
 * talc_correct_batch_device, or a stream's batch on this very context or lane); all 0 for a batch corrected in forward
 * or reverse mode.  dst is a host or a device pointer.  TALC_ERR_ARG when n exceeds that batch.                     */
int talc_last_strands(talc_ctx* ctx, uint8_t* dst, uint32_t n);

/* Pieces of the corrected reads that the k-mer table supports (not in the reference; talc --trim / --split).  The rule
 * applies to every read's output, whatever its status.  A window [p, p+K) of the output is solid when its K bytes are
 * ACGT (either case, U as T) and its k-mer is in the table (count != 0) -- for a read that came back flipped (reverse
 * mode: status TALC_READ_OK; auto mode: strand 1) the reverse complement of that k-mer, i.e. the strand the read was
 * corrected on.  A base covered by a solid window is supported; a stretch is a maximal run of supported bases (>= K
 * bases).  Pieces are 0-based, half-open [start, end) in output coordinates:
 *   TALC_PIECES_OFF    (default) nothing is computed: no launch and no copy is added to a correction
 *   TALC_PIECES_TRIM   at most one piece per read, [first supported base, last supported base + 1)
 *   TALC_PIECES_SPLIT  one piece per stretch
 * Pieces shorter than min_len (>= 1) are dropped.  Computed on the device after the correction, from the table already
 * there.  The same rules as talc_ctx_set_strand: set on a context, not on a lane (TALC_ERR_ARG; a lane follows its
 * parent), not while a stream on the context has batches pending.  Another mode or min_len 0 is TALC_ERR_ARG.       */
#define TALC_PIECES_OFF 0
#define TALC_PIECES_TRIM 1
#define TALC_PIECES_SPLIT 2
int talc_ctx_set_pieces(talc_ctx* ctx, int mode, uint32_t min_len);
/* The pieces of the last batch corrected through this context with pieces on (talc_correct_batch(_device), or a
 * stream's batch on this very context or lane), as CSR over that batch's n reads: piece_off[n+1] (piece_off[0] = 0),
 * bounds[2*total] = {start, end} per piece, in read order.  Host or device pointers; piece_off may be NULL, bounds may be
 * NULL when cap is 0.  *total is always set; TALC_ERR_CAPACITY (nothing copied) when total > cap pieces.  TALC_ERR_ARG
 * when that batch ran with pieces off.                                                                              */
int talc_last_pieces(talc_ctx* ctx, uint64_t* piece_off, uint32_t* bounds, uint64_t cap, uint64_t* total);
/* The same rule on any reads, without correcting them (the context's own settings are not used or changed).  Host
 * buffers: bases, offsets[n_reads+1] with offsets[0] == 0, flip[n_reads] (non-zero: judge the read on its reverse
 * complement; NULL: none), mode TALC_PIECES_TRIM or _SPLIT, min_len >= 1; piece_off[n_reads+1], bounds[2*cap] and
 * *total as for talc_last_pieces.  cap = (offsets[n_reads] + n_reads) / (K+1) + 1 is always enough.               */
int talc_pieces_batch(talc_ctx* ctx, const uint8_t* bases, const uint64_t* offsets, uint32_t n_reads, const uint8_t* flip,
                      int mode, uint32_t min_len, uint64_t* piece_off, uint32_t* bounds, uint64_t cap, uint64_t* total);

/* ---- streamed correction (replaces loadSeqData / outputSeqData holding every read: main.cpp:219,310, io.cpp:26-75) ----
 * Batches of reads pass through one context with the host-to-device copy of batch i+1, the kernels of batch i, the
 * device-to-host copy of batch i-1 and the caller's own work (FASTA formatting) overlapped: a ring of slots with pinned
 * staging, two copy streams and one worker thread per lane inside the library.  The stream keeps TWO batches on the
 * device (the context and one lane of it, see talc_ctx_create_lane; environment TALC_STREAM_LANES = 1..4 changes
 * that) and has lanes + 2 slots, four by default.  Host and device memory are bounded by the batch size whatever the
 * number of reads; results come back in submission order.
 *   submit  copies the caller's buffers (free again on return); blocks only while all slots are busy
 *   next    blocks until the oldest unfetched batch is complete; the returned pointers (pinned host memory owned by
 *           the stream) stay valid until the following next / close.  read_stats: per read {span of the final solid
 *           regions in k-mers, number of regions} -- the columns of outputBasicReadStats (Read.cpp:418-433) that need
 *           the kernel -- when the stream was opened with want_read_stats, else NULL.
 * One caller thread per stream; while a stream is open its context must not be used for other correction calls.  */
typedef struct talc_stream talc_stream;
int talc_stream_open(talc_ctx* ctx, int want_read_stats, talc_stream** out);
/* optional: allocate every slot's pinned / device buffers now for batches of up to max_reads reads and max_bases bases
 * (otherwise the first batch through each slot pays for it); may be called while the table is still loading        */
int talc_stream_reserve(talc_stream* s, uint32_t max_reads, uint64_t max_bases);
int talc_stream_submit(talc_stream* s, const uint8_t* bases, const uint64_t* offsets, uint32_t n_reads);
int talc_stream_next(talc_stream* s, const uint8_t** out, const uint64_t** out_offsets, const uint8_t** status,
                     uint32_t* n_reads, const uint32_t** read_stats, talc_counters* counters);
uint64_t talc_stream_pending(talc_stream* s);   /* batches submitted and not yet fetched */
/* strand[n_reads] (see TALC_STRAND_AUTO) of the batch last returned by talc_stream_next, in pinned host memory owned by
 * the stream and valid until the following next / close; NULL for a batch corrected in forward or reverse mode.
 * TALC_ERR_ARG before the first next.                                                                              */
int talc_stream_strands(talc_stream* s, const uint8_t** strand);
/* piece_off[n_reads+1] and bounds[2*piece_off[n_reads]] (see talc_ctx_set_pieces) of the batch last returned by
 * talc_stream_next, in pinned host memory owned by the stream and valid until the following next / close; both NULL
 * for a batch corrected with pieces off.  TALC_ERR_ARG before the first next.                                      */
int talc_stream_pieces(talc_stream* s, const uint64_t** piece_off, const uint32_t** bounds);
const char* talc_stream_last_error(talc_stream* s);
void talc_stream_close(talc_stream* s);

/* ---- roofline microbenchmark (SURVEY 8d: "the random-32 B-sector peak must be measured ... and reported") --------
 * Uniformly random 256-bit read-only loads over a buffer of `buffer_bytes` (rounded down to a power of two; use
 * >= 2 GiB so that the 126 MB L2 does not help).  dependent = 0: eight independent loads in flight per thread, the
 * pattern of the coverage kernel; dependent = 1: one chain per thread, the next address hashed from the loaded sector,
 * the pattern of the graph walk (ns_per_load is then the latency of one hop).  gbs = sectors * 32 B / time.    */
int talc_bench_random_sectors(talc_ctx* ctx, uint64_t buffer_bytes, int dependent, uint32_t warps_per_sm, double* gbs,
                              double* ns_per_load);

/* ---- device self-tests of the scoring primitives (used by tests/ on a GPU) ------------------- */
/* pairs of NUL-free ASCII strings given as (concatenated bytes, offsets[n+1]); op: 0 NW score,
 * 1 LCS length, 2 overlap score (walk order), 3 seed-and-extension (result[4*i..]: ref_ext,
 * cand_ext, score, stop; aux = xdrop, aux2 = direction_right, K from the context)                 */
int talc_test_align(talc_ctx* ctx, int op, const uint8_t* a, const uint64_t* a_off, const uint8_t* b,
                    const uint64_t* b_off, uint32_t n, int aux, int aux2, int32_t* result);
/* the same operations on the views the correction builds.  reads (concatenated bytes, read_off[n_reads+1]) are
 * packed as the corrector packs them (2 bits per base, 4 when the read holds an N); desc[8*i..] = {read, start,
 * step, len} of side a, then of side b.  step +1 / -1: bases start, start+step, ... of the packed read (walk order);
 * step 0: read[start, start+len) (A, C, G, T only) copied into a 2-bit trail slot whose bits past len are random.
 * op 0-2: result[i]; op 3: as above; op 4: X-drop of query a against database b, result[4*i..]: ext_rows,
 * ext_cols, DP cells visited, end score (aux = xdrop); op 5: result[4*i..]: NW score, LCS length of the fused pass;
 * op 6: every aux consecutive pairs form one gardening frontier, the a side of its first pair the reference and the
 * b sides its trails (step 0, equal lengths): result[i] = overlap score of trail i with the shared-prefix stripe
 * reuse of the corrector.  A score of INT32_MIN means the per-pair scratch (2 MB) was too small.                  */
int talc_test_align_slices(talc_ctx* ctx, int op, const uint8_t* reads, const uint64_t* read_off, uint32_t n_reads,
                           const int32_t* desc, uint32_t n, int aux, int aux2, int32_t* result);
/* the successor tables of the walks (one bucket per (K-1)-mer context with the counts of its four successors, derived
 * from the k-mer table at every seal): for each kmers[i], the look-up the walk makes for its successors, right != 0 the
 * k-mers x[1..]+b, else b+x[..K-2]; cnt[4*i+b] = count of successor b (0 when absent), colmask[i] bit b = successor b
 * carries a junction colour.  *ctx_capacity (may be NULL) = buckets per table.  TALC_ERR_NO_TABLE before a seal.     */
int talc_test_successors(talc_ctx* ctx, int right, const uint64_t* kmers, uint32_t n, uint32_t* cnt, uint32_t* colmask,
                         uint64_t* ctx_capacity);
/* the count model of the walk on the context's parameters and device tables (counts below 16384 are tabulated, larger
 * ones computed).  args[8*i..], out[9*i..] (a double as its IEEE bits):
 *   op 0  step bounds of count       args {count}                       out {lower, upperNoise, sqrt(count), lambda,
 *                                                                             noiseModel}
 *   op 1  successor tags             args {count, c[4], colmask, complex} out {n (0 or 4), tag[4] (0 EXPECTED,
 *                                                                             1 UNEXPECTED, 2 BREAKPOINT), dist[4]}
 *   op 2  child of a fast-walk step  args {count, c[4], colmask}        out {child 0..3, or -1 as int64}
 *   op 3  upper bound test           args {nextc, cc}                   out {nextc within the noise interval of cc}
 *   op 4  last-node test             args {nextc, cc}                   out {nextc within both bounds of cc}          */
int talc_test_model(talc_ctx* ctx, int op, const uint32_t* args, uint32_t n, uint64_t* out);
/* permutation produced by the device replica of libstdc++ std::sort on keys[n] (operator<)        */
int talc_test_sort(talc_ctx* ctx, const int64_t* keys, uint32_t n, uint32_t* perm);

#ifdef __cplusplus
}
#endif
#endif /* TALC_B200_H */
