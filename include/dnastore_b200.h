/* dnastore_b200.h -- C ABI of the B200-native batched Viterbi decoder for dnastore's
 * hot path.  extern "C", plain pointers and sizes, integer return codes, no
 * exceptions across the boundary, no torch types.  One decoder handle per device;
 * a handle may be used from one host thread at a time.
 *
 * The reference (ihh/dnastore) has no plugin/FFI interface; the seam this library
 * replaces is (all paths relative to the reference tree):
 *   src/viterbi.h:108       decodeFastSeqs(filename, machine, mutatorParams)
 *   src/viterbi.h:94-102    ViterbiMatrix(machine, inputModel, params, fastSeq),
 *                           traceback(), loglike(), sCell/dCell/tCell
 *   src/viterbi.h:18-40     MachineScores  (flattened into dnab_tables)
 *   src/mutator.h:9-41      MutatorParams / MutatorScores
 *   src/trans.h:83-126      Machine: fromFile, compose, writeJSON, inputAlphabet
 *   t/dnastore.cpp:41-82    the CLI flags that feed them
 * INTEGRATION.md shows the few lines a maintainer would add to the reference to
 * call these entry points instead of its per-read CPU loop.
 *
 * Error convention: functions returning a pointer return NULL on failure, functions
 * returning int return 0 on success and a negative DNAB_E* code on failure; in both
 * cases dnab_last_error() (thread-local) describes what went wrong.
 */
#ifndef DNASTORE_B200_H
#define DNASTORE_B200_H

#include <stddef.h>
#include <stdint.h>

#include "dnab_tables.h"

#ifdef __cplusplus
extern "C" {
#endif

#define DNAB_OK 0
#define DNAB_EINVAL (-1)      /* bad argument / unsupported machine */
#define DNAB_ECUDA (-2)       /* CUDA runtime error, or no usable device */
#define DNAB_EIO (-3)         /* file not found / unreadable */
#define DNAB_ECYCLIC (-4)     /* null-transition cycle: reference throws std::domain_error (src/trans.cpp:631-632) */
#define DNAB_EFORMAT (-5)     /* malformed machine / error-model JSON, non-ACGT read */

/* per-read status written by dnab_viterbi_batch */
#define DNAB_READ_OK 0
#define DNAB_READ_NO_DECODING 1  /* loglike == -inf: reference warns "No valid Viterbi decoding found" and yields "" (src/viterbi.cpp:198-201) */
#define DNAB_READ_OVERFLOW 2     /* decoded string or path did not fit the caller's buffer */
#define DNAB_READ_TRACEBACK_FAILED 3 /* a predecessor record was missing (cannot happen for a finite loglike) */

const char* dnab_last_error(void);
const char* dnab_version(void);
void dnab_free(void* p); /* frees strings/buffers this library returned */

/* ------------------------------------------------------------------------
 * Machine: dnastore's transducer and its JSON format (src/trans.h:83-126).
 * ---------------------------------------------------------------------- */
typedef struct dnab_machine dnab_machine;

dnab_machine* dnab_machine_load(const char* json_path);             /* Machine::fromFile, src/trans.cpp:477-482 */
dnab_machine* dnab_machine_from_json(const char* json_text);        /* Machine::fromJSON, src/trans.cpp:471-475 */
/* Machine::compose(first, second), src/trans.cpp:505-602: first's output feeds second's input. */
dnab_machine* dnab_machine_compose(const dnab_machine* first, const dnab_machine* second);
char* dnab_machine_to_json(const dnab_machine* m);                  /* Machine::writeJSON, src/trans.cpp:402-429; dnab_free() it */
uint32_t dnab_machine_n_states(const dnab_machine* m);
uint32_t dnab_machine_max_left_context(const dnab_machine* m);      /* src/trans.cpp:252-257 */
/* Machine::inputAlphabet(flags) (src/trans.cpp:280-292); flags as in src/trans.h:42-48. Writes a NUL-terminated string. */
int dnab_machine_input_alphabet(const dnab_machine* m, int flags, char* out, size_t cap);
void dnab_machine_free(dnab_machine* m);

/* ------------------------------------------------------------------------
 * Error model: the CLI's flags (t/dnastore.cpp:69-75,119-129).
 * ---------------------------------------------------------------------- */
typedef struct dnab_error_flags {
  int32_t length;      /* -l/--length (default 12): maxDupLen = length/2 */
  int32_t global;      /* --error-global: 1 = global alignment, 0 = local (CLI default) */
  double sub_prob;     /* --error-sub-prob  (.01) */
  double iv_ratio;     /* --error-iv-ratio  (10) */
  double dup_prob;     /* --error-dup-prob  (.001) */
  double del_open;     /* --error-del-open  (.001) */
  double del_ext;      /* --error-del-ext   (.01) */
} dnab_error_flags;

void dnab_error_flags_default(dnab_error_flags* f);

/* ------------------------------------------------------------------------
 * Compile: Machine + error model -> flat tables (host memory).
 * Replaces the per-read MachineScores/MutatorScores/InputModel construction
 * (src/viterbi.cpp:6-14,23-60,309-310; src/mutator.cpp:56-75).
 * ---------------------------------------------------------------------- */
typedef struct dnab_compiled dnab_compiled;

dnab_compiled* dnab_compile(const dnab_machine* m, const dnab_error_flags* flags);
/* Same, with the error model read from an --error-file JSON (src/mutator.cpp:18-30). */
dnab_compiled* dnab_compile_with_error_file(const dnab_machine* m, const char* error_json_path);
const dnab_tables* dnab_compiled_tables(const dnab_compiled* c);
void dnab_compiled_free(dnab_compiled* c);

/* ------------------------------------------------------------------------
 * Decoder: the tables resident on one GPU + the CUDA kernels.
 * ---------------------------------------------------------------------- */
typedef struct dnab_decoder dnab_decoder;

/* Uploads the tables to `device` (CUDA ordinal) and derives the device-side
 * structures (state partition over the thread-block cluster, packed edge words,
 * outgoing lists).  Fails with DNAB_ECUDA when there is no CUDA device: there is
 * NO CPU fallback. */
dnab_decoder* dnab_decoder_create(const dnab_tables* t, int device);
void dnab_decoder_destroy(dnab_decoder* d);

typedef struct dnab_decoder_info {
  uint32_t n_states, k, local;
  uint32_t cluster_size;     /* CTAs cooperating on one read */
  uint32_t states_per_cta;   /* slice of the state space owned by one CTA */
  uint32_t threads_per_cta;
  uint32_t smem_bytes_per_cta;
  uint32_t t_in_smem;        /* 1: duplication (T) columns live in shared memory, 0: in global scratch */
  uint32_t table_in_smem;    /* 1: each CTA keeps its out-table (its slice of the transition table) in shared memory */
  uint32_t s_prev_in_smem;   /* 1: the previous column S(pos-1) is in shared memory, 0: in L2-resident global scratch */
  uint32_t n_clusters;       /* clusters resident at once = reads in flight */
  uint32_t sm_count;
} dnab_decoder_info;
int dnab_decoder_get_info(const dnab_decoder* d, dnab_decoder_info* info);

/* Tuning overrides of the one-read-per-cluster kernel (0 = automatic; t_in_smem_mode 1 shared memory, 2 global scratch),
 * the same as the options "cluster_size", "threads_per_cta" and "t_columns" below; must be set before the first batch. */
int dnab_decoder_configure(dnab_decoder* d, uint32_t cluster_size, uint32_t threads_per_cta, uint32_t t_in_smem_mode);

/* Named options; set before the first batch.
 *   "kernel"          0 automatic (read-batched when the machine fits, else one read per cluster), 1 read-batched
 *                     (viterbi_fill_batch.cu), 2 push closure, one read per cluster (viterbi_fill_push.cu); 3, the
 *                     pull-closure kernel of round 1, was retired and returns DNAB_EINVAL
 *   "team_size"       read-batched kernel: CTAs holding one group of 32 reads (0 = smallest that fits)
 *   "warps_per_cta"   read-batched kernel: 8, 16 or 32
 *   "cluster_size", "threads_per_cta", "t_columns" (1 shared / 2 global), "table" (1 shared / 2 global),
 *   "s_prev" (1 shared / 2 global), "partition" (0 automatic = 3; 1 index runs, 2 DFS runs, 3 DFS chunks dealt,
 *                     4 DFS runs sorted): placements of the one-read-per-cluster push kernel; setting any of them (or
 *                     dnab_decoder_configure) makes "kernel" 0 choose the push kernel
 *   "thin_n", "t_recompute", "queue_cap", "deal_chunks": schedule knobs of the push kernel (tests)
 *   "idle_sleep_ns"   accepted and ignored (it tuned the retired pull-closure kernel)
 *   "async_closure"   read-batched kernel: 0 breadth-first levels with a CTA barrier each, 1 no level barriers (work counter),
 *                     2 (default) automatic = 1, in a team and in a single CTA alike; "batch_idle_ns" back-off of an idle warp;
 *                     "team_slack_pct"
 *   "notify_classes"  read-batched kernel, teams: notification counters per CTA, 1..32 (default 32).  The states of a CTA that have
 *                     transitions from other CTAs are dealt into that many classes; a publishing state notifies the classes of its
 *                     successors and the owner re-relaxes only the notified classes (1 = every transition that crosses CTAs)
 *   "eager_notify"    read-batched kernel, teams: 1 = every notification is also sent once before the release fence (measured slower:
 *                     the extra wake-ups cost more than the fence latency they save), 0 (default)
 *   "persist_l2"      read-batched kernel: 1 gives the rows carried between columns a persisting L2 access-policy window (default 0:
 *                     measured on B200 it DOUBLES the DRAM writes; the rows carry an evict-last cache hint instead)
 *   "pred_budget_mb"  device memory the predecessor records of one launch may take
 * Unknown keys return DNAB_EINVAL. */
int dnab_decoder_set_option(dnab_decoder* d, const char* key, int64_t value);

typedef struct dnab_batch_info {
  uint32_t enabled;            /* 1: batches run on the read-batched kernel */
  uint32_t reads_per_group;    /* 32: the reads of a group are the lanes of a warp */
  uint32_t team_size;          /* CTAs that hold the S and D columns of one group in shared memory */
  uint32_t states_per_cta;
  uint32_t warps_per_cta;
  uint32_t smem_bytes_per_cta;
  uint32_t n_teams;            /* groups in flight */
  uint32_t wide_states;        /* wide states of the machine (see dnab_viterbi_batch); 0 = no side plane */
  double cross_cta_transition_fraction; /* transitions whose source and destination live in different CTAs */
} dnab_batch_info;
int dnab_decoder_get_batch_info(const dnab_decoder* d, dnab_batch_info* info);

/* Reads are packed 2 bits per base, A,C,G,T = 0..3 (src/kmer.h:11-13, src/fastseq.cpp:9-15),
 * base i of a read in bits 2*(i%4).. of byte i/4; read r starts at byte
 * read_byte_off[r] (a multiple of 16) and has read_len[r] bases. */
size_t dnab_packed_size(const int32_t* read_len, int64_t n_reads);  /* bytes needed incl. 16-byte alignment */
/* Packs ASCII reads (concatenated in `bases`, read r = bases[base_off[r] .. base_off[r+1])).
 * Case-insensitive; a non-ACGT character is an error (DNAB_EFORMAT), as in the reference
 * (src/fastseq.cpp:25-39, which terminates the process). */
int dnab_pack_reads(const char* bases, const int64_t* base_off, int64_t n_reads, uint8_t* packed, int64_t* read_byte_off,
                    int32_t* read_len);

/* Batched Viterbi decode with HOST buffers: copies the packed reads to the device,
 * runs fill + traceback there, copies results back (this is the `e2e` path).
 *   loglike[n]          ViterbiMatrix::loglike() (src/viterbi.h:102), fp64, bit-exact
 *   decoded             n * decoded_stride bytes; read r's input-symbol string
 *                       (ViterbiMatrix::traceback(), src/viterbi.cpp:195-304) at
 *                       decoded + r*decoded_stride, NOT NUL-terminated
 *   decoded_len[n]      its length
 *   status[n]           DNAB_READ_*
 *   path / path_len     optional (NULL to skip): traceback cells as int32 triples
 *                       (state, pos, mutState) with mutState 0=S,1=D,2+i=T(i+1)
 *                       (src/viterbi.h:52-56), in traceback order starting at the
 *                       first cell the reference's loop visits; path_stride triples per read
 * Returns DNAB_OK or a negative code.
 *
 * Viterbi decoding takes states of any in- and out-degree that the reference accepts.  The predecessor
 * record of a DP cell is one byte; a state with more candidates than a byte can name, or with more
 * than 255 outgoing transitions, is a WIDE state (nEmit > 126, nEmit + nNull + 2 > 254, 2*nEmit + nNull
 * > 254, or > 255 outgoing transitions): the high byte of its S and D records goes to a side plane
 * sized nWide * 2 bytes per read and column, allocated only for machines that have wide states
 * (dnab_batch_info.wide_states counts them).  Still refused with DNAB_EINVAL, the state named in the
 * error text: a state with more than 65,535 candidates in a record (nEmit + nNull + 3 or
 * 2*nEmit + nNull > 65,535: a wide record is 16 bits, 0xFFFF = none), or with more than 65,535
 * outgoing transitions.  Independently of degree, the tables of one CTA use 16-bit offsets; a
 * machine whose tables exceed them for every placement is refused as not fitting. */
int dnab_viterbi_batch(dnab_decoder* d, int64_t n_reads, const uint8_t* packed, const int64_t* read_byte_off,
                       const int32_t* read_len, double* loglike, char* decoded, int32_t decoded_stride,
                       int32_t* decoded_len, int32_t* status, int32_t* path, int32_t path_stride, int32_t* path_len);

/* Same computation with every buffer already RESIDENT IN DEVICE MEMORY of the
 * decoder's device (pointers are device pointers; path output not available).
 * Asynchronous on `cuda_stream` (a cudaStream_t passed as void*, NULL = default
 * stream); the caller synchronises.  Scratch for the predecessor records is grown
 * on demand and kept in the handle.  max_read_len >= every read_len[r]. */
int dnab_viterbi_batch_device(dnab_decoder* d, int64_t n_reads, int32_t max_read_len, const uint8_t* d_packed,
                              const int64_t* d_read_byte_off, const int32_t* d_read_len, double* d_loglike,
                              char* d_decoded, int32_t decoded_stride, int32_t* d_decoded_len, int32_t* d_status,
                              void* cuda_stream);

/* Debug/parity aid: decode ONE read and also return every DP cell in the reference's
 * layout cell[(k+2)*(pos*n_states+state)+mut] (src/viterbi.h:65-67); cells must hold
 * (len+1)*n_states*(k+2) doubles (host memory). */
int dnab_viterbi_cells(dnab_decoder* d, const uint8_t* packed, int32_t read_len, double* loglike, double* cells);

/* Forward (sum-product) log-likelihood over the same machine-state x DNA-position lattice
 * (SURVEY.md 8a-12).  NOT IN THE REFERENCE: the reference's only forward-backward is the pair-HMM
 * of src/fwdback.cpp (dnab_pairhmm_fb_batch below).  Specified by analogy with ViterbiMatrix's fill
 * (src/viterbi.cpp:62-176): every max becomes the reference's table-based log_sum_exp
 * (src/logsumexp.h:19-74); the closure of a column is solved by synchronous sweeps that stop after
 * the first sweep that changes no cell.  loglike = F_S(end, L) (global mode) or the log-sum over all
 * states of F_S(., L) (local mode).  Host buffers; same packed-read format as dnab_viterbi_batch.
 * sweeps[r] (optional) = closure sweeps summed over the columns of read r; status[r] = 0, or 1 when a
 * closure did not settle within max_sweeps (0 = default 4096).  cells (optional, read 0 only):
 * (len+1)*n_states*(k+2) doubles in the ViterbiMatrix layout. */
int dnab_forward_batch(dnab_decoder* d, int64_t n_reads, const uint8_t* packed, const int64_t* read_byte_off,
                       const int32_t* read_len, int32_t max_sweeps, double* loglike, int64_t* sweeps, int32_t* status,
                       double* cells);

/* Forward AND backward over the machine lattice with the posterior expected counts of the error-model
 * events -- the machine-lattice analogue of FwdBackMatrix::counts (src/fwdback.cpp:154-188): what
 * `--error-counts` computes from given alignments, here summed over every input the machine accepts.
 * NOT IN THE REFERENCE (SURVEY.md 8a-12), specified by oracle/forward_oracle.c, parity unpinned.
 * counts[r*(5+k+16) ...] = nDelOpen, nTanDup, nNoGap, nDelExtend, nDelEnd, nLen[k], nSub[16] (row = machine
 * base, column = observed base), the order of dnab_mutator_counts.  loglike_back[r] = B_S(start, 0), which
 * equals loglike[r] up to the accuracy of the table log_sum_exp. */
int dnab_fwdback_counts_batch(dnab_decoder* d, int64_t n_reads, const uint8_t* packed, const int64_t* read_byte_off,
                              const int32_t* read_len, int32_t max_sweeps, double* loglike, double* loglike_back,
                              double* counts, int32_t* status);

/* Posterior (soft) decoding over the machine lattice (SURVEY.md 8a-12, 8f-4; BASELINE config 5): for every base of every
 * read, the posterior probability, summed over ALL paths (forward x transition x backward / likelihood -- the formula of
 * FwdBackMatrix, src/fwdback.h:92-113, applied to the machine lattice), of the CLASS of the move that emitted it:
 *   class 0        a transition that consumes no input symbol (padding / control-word bases)
 *   class 1..s     a transition that consumes input symbol classes[i] ('0', '1', control letters, ...)
 *   class s+1      a tandem duplication (the base repeats an earlier one, src/viterbi.cpp:102-106)
 * dnab_posterior_classes writes the class characters ("-" + the machine's input symbols + "+") and returns their number.
 * post: row post_off[r] + p, column c = P(class c emitted base p of read r | read); every row sums to 1 up to the accuracy
 * of the reference's table log_sum_exp (2e-3).  decoded (optional, one char per base, same offsets): the most probable
 * class per base -- a soft output for an outer code (doc/trans.tex:947-952,1148-1154), not the Viterbi input string.
 * NOT IN THE REFERENCE; specified by oracle/forward_oracle.c (dnab_oracle_backward_posterior), parity unpinned. */
int dnab_posterior_classes(const dnab_decoder* d, char* classes, size_t cap);
int dnab_posterior_batch(dnab_decoder* d, int64_t n_reads, const uint8_t* packed, const int64_t* read_byte_off,
                         const int32_t* read_len, int32_t max_sweeps, const int64_t* post_off, double* loglike, double* post,
                         char* decoded, int32_t* status);

/* Counters since creation: kernels launched by this library and DP cells filled. */
typedef struct dnab_decoder_stats {
  uint64_t kernel_launches;
  uint64_t fill_launches;
  uint64_t traceback_launches;
  uint64_t reads;
  uint64_t cells;           /* sum over reads of n_states*(len+1)*(k+2) */
  double last_fill_ms;      /* CUDA-event time of the most recent fill kernel (host-buffer path) */
  double last_traceback_ms;
  /* device path, when dnab_decoder_set_timing(d,1): CUDA-event time summed over every fill /
   * traceback launch since the last dnab_decoder_reset_timing (events on the launching stream) */
  double timed_fill_ms;
  double timed_traceback_ms;
  uint64_t timed_fill_launches;
} dnab_decoder_stats;
/* Resolves pending timing events: call only after the stream(s) used have been synchronised. */
int dnab_decoder_get_stats(const dnab_decoder* d, dnab_decoder_stats* s);
int dnab_decoder_set_timing(dnab_decoder* d, int enabled);
int dnab_decoder_reset_timing(dnab_decoder* d);
/* Profiling aid: in-kernel counters (columns, closure sweeps, worklist entries, SM cycles per phase).  When on, the
 * fill runs an instrumented instantiation of the kernel (same results, a few per cent slower); the production
 * instantiation carries no counters at all.  dnab_viterbi_cells uses the instrumented one as well. */
int dnab_decoder_set_debug(dnab_decoder* d, int enabled);
int dnab_decoder_debug_counters(dnab_decoder* d, unsigned long long* out16);

/* ------------------------------------------------------------------------
 * File-level driver: the drop-in for decodeFastSeqs (src/viterbi.cpp:306-320).
 * Reads a FASTA/FASTQ file (plain or gzip; multi-line records concatenated,
 * src/fastseq.cpp:123-148), decodes every record on the decoder's device and
 * returns the decoded strings in input order.
 * ---------------------------------------------------------------------- */
typedef struct dnab_decoded_set dnab_decoded_set;
dnab_decoded_set* dnab_decode_fasta(dnab_decoder* d, const char* fasta_path);
int64_t dnab_decoded_count(const dnab_decoded_set* s);
const char* dnab_decoded_name(const dnab_decoded_set* s, int64_t i);
const char* dnab_decoded_seq(const dnab_decoded_set* s, int64_t i);   /* NUL-terminated */
double dnab_decoded_loglike(const dnab_decoded_set* s, int64_t i);
int32_t dnab_decoded_status(const dnab_decoded_set* s, int64_t i);
void dnab_decoded_free(dnab_decoded_set* s);

/* ------------------------------------------------------------------------
 * Several GPUs of one node, and the ingest/egress pipeline (SURVEY.md 8e, 8f-3).  Reads are independent
 * (src/viterbi.cpp:312-318 carries no state between them), so a batch is cut into chunks that one host thread
 * per device decodes with its own decoder; no collective; results come back in input order.
 * dnab_decode_fasta above is the one-device form of the same pipeline: the file is parsed and packed in bounded
 * chunks by a producer thread (plain or gzip FASTA/FASTQ, src/fastseq.cpp:123-148) into page-locked buffers while the
 * previous chunk is being copied and decoded, and only reads whose decoded string overflowed their slot are re-decoded.
 * ---------------------------------------------------------------------- */
typedef struct dnab_multi_decoder dnab_multi_decoder;
dnab_multi_decoder* dnab_multi_decoder_create(const dnab_tables* t, const int* devices, int n_devices);
void dnab_multi_decoder_destroy(dnab_multi_decoder* m);
int dnab_multi_decoder_count(const dnab_multi_decoder* m);
dnab_decoder* dnab_multi_decoder_at(dnab_multi_decoder* m, int i);            /* for dnab_decoder_set_option / stats */
/* "chunk_reads" (0 = automatic), "decoded_slot_bytes" (bytes reserved per decoded string on the first attempt,
 * 0 = 2*maxLen+256; overflowing reads are re-decoded with 4x); any other key goes to every device's decoder. */
int dnab_multi_decoder_set_option(dnab_multi_decoder* m, const char* key, int64_t value);
/* dnab_viterbi_batch over all devices of m: same buffers and meaning, host memory, path output not available. */
int dnab_viterbi_batch_multi(dnab_multi_decoder* m, int64_t n_reads, const uint8_t* packed, const int64_t* read_byte_off,
                             const int32_t* read_len, double* loglike, char* decoded, int32_t decoded_stride,
                             int32_t* decoded_len, int32_t* status);
dnab_decoded_set* dnab_decode_fasta_multi(dnab_multi_decoder* m, const char* fasta_path);
typedef struct dnab_pipeline_stats {
  int64_t reads, chunks, overflow_reruns;
  double parse_seconds;        /* producer thread: parsing + 2-bit packing */
  double decode_busy_seconds;  /* summed over the device threads: copies + kernels */
  double wall_seconds;
} dnab_pipeline_stats;
int dnab_multi_decoder_last_stats(const dnab_multi_decoder* m, dnab_pipeline_stats* s);


/* ------------------------------------------------------------------------
 * Exact (error-free) decoding on the host: dnastore's -d/--decode-file, --decode-string and
 * --decode-bits (call sites t/dnastore.cpp:185-211).  Not a GPU path: O(L) per read and strictly
 * sequential; kept so that BASELINE config 1 and the reference's testdecode goldens
 * (Makefile:142-144,153,168,176,183) run through this library.
 *   Decoder<Writer>   src/decoder.h:7-190   (expand :54-103, decodeSymbol :130-158,
 *                                            shiftResolvedSymbols :160-184, close :28-47)
 *   BinaryWriter      src/decoder.h:193-240 (bits packed least significant first)
 * ---------------------------------------------------------------------- */
typedef struct dnab_exact_decoder dnab_exact_decoder;
/* Decoder::Decoder (decoder.h:16-22); `m` must outlive the decoder. */
dnab_exact_decoder* dnab_exact_decoder_create(const dnab_machine* m);
/* Decoder::decodeString (decoder.h:186-189): n bases, case-insensitive.  DNAB_EINVAL with
 * dnab_last_error() = the reference's assertion text when a base cannot be decoded or the machine is
 * ambiguous (the reference aborts there). */
int dnab_exact_decoder_feed(dnab_exact_decoder* d, const char* bases, size_t n);
/* Decoder::close (decoder.h:28-47): end of input. */
int dnab_exact_decoder_close(dnab_exact_decoder* d);
/* Input symbols ('0','1','^','$', control letters) resolved since the last call; dnab_free() it. */
char* dnab_exact_decoder_take_symbols(dnab_exact_decoder* d);
/* The reference's "Decoder unresolved ..." warnings so far, one per line; dnab_free() it. */
char* dnab_exact_decoder_warnings(const dnab_exact_decoder* d);
int64_t dnab_exact_decoder_hypotheses(const dnab_exact_decoder* d);   /* |current| of decoder.h:13 */
void dnab_exact_decoder_destroy(dnab_exact_decoder* d);

/* BinaryWriter (decoder.h:193-240): packs the '0'/'1' symbols into bytes (first bit = bit 0), skips
 * '^' '$', warns about anything else.  Returns the number of bytes (written to `bytes` if cap allows, else
 * DNAB_EINVAL); leftover_bits (>= 8 chars incl. NUL) receives the bits of an unfinished last byte, most
 * significant first, as the reference's destructor warning prints them; *warnings (optional): one per line,
 * dnab_free() it. */
int64_t dnab_pack_decoded_symbols(const char* symbols, size_t n, uint8_t* bytes, size_t cap, char* leftover_bits,
                                  char** warnings);
/* -d/--decode-file (t/dnastore.cpp:185-190): every record of a FASTA/FASTQ file through ONE decoder
 * (its state carries over between records, as in the reference), close, then BinaryWriter.
 * *bytes is malloc'ed (dnab_free); *warnings optional, as above. */
int dnab_exact_decode_fasta(const dnab_machine* m, const char* fasta_path, uint8_t** bytes, size_t* n_bytes,
                            char** warnings);

/* ------------------------------------------------------------------------
 * Pair-HMM forward / backward / expected counts (SURVEY.md 8a-10, 8a-11): the reference's
 * only forward-backward, over the (original DNA x observed DNA) lattice of a 2-row
 * alignment, used to train the error model (--error-counts / --fit-error).
 *   ForwardMatrix / BackwardMatrix / FwdBackMatrix::counts   src/fwdback.cpp:43-188
 *   expectedCounts / baumWelchParams                         src/fwdback.cpp:190-230
 *   MutatorParams / MutatorCounts                            src/mutator.h:9-67
 *   log_sum_exp (lookup table)                               src/logsumexp.h:19-86
 * ---------------------------------------------------------------------- */
#define DNAB_MAX_DUP 16

typedef struct dnab_mutator_params {      /* MutatorParams, src/mutator.h:9-31 */
  double p_del_open, p_del_extend, p_tan_dup, p_transition, p_transversion;
  double p_len[DNAB_MAX_DUP];
  int32_t max_dup_len;                    /* pLen.size() */
  int32_t local;
} dnab_mutator_params;

typedef struct dnab_mutator_counts {      /* MutatorCounts, src/mutator.h:43-67 */
  double n_del_open, n_tan_dup, n_no_gap, n_del_extend, n_del_end;
  double n_len[DNAB_MAX_DUP];
  double n_sub[16];                       /* nSub[original base * 4 + observed base] */
  int32_t max_dup_len;
  int32_t reserved;
} dnab_mutator_counts;

/* MutatorParams as the CLI builds it from its flags (t/dnastore.cpp:119-129). */
void dnab_mutator_params_from_flags(const dnab_error_flags* f, dnab_mutator_params* out);
char* dnab_mutator_params_json(const dnab_mutator_params* p);   /* MutatorParams::writeJSON text; dnab_free() it */
char* dnab_mutator_counts_json(const dnab_mutator_counts* c);   /* MutatorCounts::writeJSON text; dnab_free() it */
/* The log(1+exp(-x)) lookup table the device uses (100,001 entries, step 1e-4). */
const double* dnab_lse_table(int32_t* n_entries);

/* A database of 2-row Stockholm alignments prepared for the lattice (readStockholmDatabase,
 * src/stockholm.cpp:154-167; Alignment + GuideAlignmentEnvelope, src/alignpath.cpp:189-204,237-265):
 * tokens of both rows and the envelope coordinates a[0..inLen], b[0..outLen] with
 * inRange(ip,op) <=> |a[ip]-b[op]| <= maxDistance (src/alignpath.h:48-53). */
typedef struct dnab_pair_db dnab_pair_db;
dnab_pair_db* dnab_pair_db_load(const char* stockholm_path);
int64_t dnab_pair_db_count(const dnab_pair_db* db);
int32_t dnab_pair_db_in_len(const dnab_pair_db* db, int64_t i);
int32_t dnab_pair_db_out_len(const dnab_pair_db* db, int64_t i);
const uint8_t* dnab_pair_db_in(const dnab_pair_db* db, int64_t i);     /* tokens 0..3 */
const uint8_t* dnab_pair_db_out(const dnab_pair_db* db, int64_t i);
const int32_t* dnab_pair_db_env_a(const dnab_pair_db* db, int64_t i);  /* in_len+1 entries */
const int32_t* dnab_pair_db_env_b(const dnab_pair_db* db, int64_t i);  /* out_len+1 entries */
void dnab_pair_db_free(dnab_pair_db* db);

/* Forward, backward and expected counts of a batch of alignments on `device` (one GPU thread per
 * alignment, 32 alignments of similar length per warp).  Alignment i: tokens in_tok[in_off[i]..in_off[i+1]), out_tok[out_off[i]..out_off[i+1]),
 * envelope env_a[in_off[i]+i ..] (in_len+1 entries) and env_b[out_off[i]+i ..] (out_len+1 entries).
 * strict != 0 <=> --strict-guides (maxDistance 0, else maxDupLen; src/fwdback.cpp:17).
 * fwd_ll = ForwardMatrix::loglike, back_ll = BackwardMatrix::loglike (bit-identical to the
 * reference: same lookup table, same operand order); counts[i] = FwdBackMatrix::counts(). */
int dnab_pairhmm_fb_batch(int device, const dnab_mutator_params* p, int strict, int64_t n_align, const uint8_t* in_tok,
                          const int64_t* in_off, const uint8_t* out_tok, const int64_t* out_off, const int32_t* env_a,
                          const int32_t* env_b, double* fwd_ll, double* back_ll, dnab_mutator_counts* counts,
                          double* kernel_ms);
/* The batch is run in chunks of alignments whose forward and backward cells fit the device: by default 40 % of the free
 * memory each; `cells` > 0 caps a chunk at that many envelope cells per lane (tuning / testing; 0 = automatic).
 * Results do not depend on it. */
int dnab_pairhmm_set_chunk_cells(int64_t cells);
/* expectedCounts (src/fwdback.cpp:190-209): counts summed and log-likelihoods added in database order. */
int dnab_expected_counts(int device, const dnab_mutator_params* p, const dnab_pair_db* db, int strict,
                         dnab_mutator_counts* total, double* loglike);
/* baumWelchParams (src/fwdback.cpp:211-230) with the Laplace prior the CLI uses (t/dnastore.cpp:137-139). */
int dnab_baum_welch(int device, const dnab_mutator_params* init, const dnab_pair_db* db, int strict,
                    dnab_mutator_params* fitted, int32_t* iterations);

#ifdef __cplusplus
}
#endif
#endif /* DNASTORE_B200_H */
