/*
 * f2q.h — C-ABI of libf2q.so, the B200 (sm_100a) read -> feature -> count engine.
 *
 * This is the drop-in boundary for ONE path of 2FAST2Q (reference v2.8.1): everything that
 * happens between "uncompressed FASTQ bytes" and "per-feature count vector + 5 read statistics".
 * The reference has no FFI; its seam is the Python function
 *     reads_counter(i, raw, features, param, reads_stats, preprocess)      fast2q/fast2q.py:514-582
 * which drives fastq_parser (fast2q.py:306-409), sequence_tinder (:215-285), border_finder
 * (:628-658), features_all_vs_all (:660-690) and mismatch_search_handler (:692-750).
 * The Python host layer (2fast2q_b200/fast2q.py) mirrors reads_counter and calls the entry
 * points below through ctypes.  Each entry point cites the reference lines it replaces.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes only; no C++/torch/Python types cross the boundary.
 *   - every call returns F2Q_OK (0) or a negative F2Q_E* code; text via f2q_last_error().
 *   - CUDA errors are sticky per context.  Nothing here ever falls back to a CPU implementation:
 *     without a usable sm_100 device f2q_create fails with F2Q_ENODEVICE.
 *   - a context = one GPU, one sample in flight, used from one thread at a time.
 *   - the caller owns every host buffer; the library owns all device memory it allocates.
 */
#ifndef F2Q_H_
#define F2Q_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define F2Q_ABI_VERSION 2

#define F2Q_MAX_ITER   8    /* max comma items in --st / --us / --ds (search_iterations, fast2q.py:541,558) */
#define F2Q_MAX_DELIM  64   /* max bytes of one --us / --ds search sequence */

/* error codes */
#define F2Q_OK            0
#define F2Q_EINVAL       -1  /* bad argument / configuration the reference would FATAL on (fast2q.py:555-556) */
#define F2Q_ENOMEM       -2
#define F2Q_ECUDA        -3  /* CUDA runtime/driver error (sticky) */
#define F2Q_ESTATE       -4  /* call out of order (e.g. submit before begin_sample) */
#define F2Q_EUNSUPPORTED -5  /* input outside what the device path implements; never silently approximated */
#define F2Q_ETOOLONG     -6  /* one FASTQ record longer than the carry buffer (see f2q_set_option) */
#define F2Q_ENODEVICE    -7  /* no CUDA device of compute capability 10.x */
#define F2Q_EINTERNAL    -8  /* device-side invariant violated (reported, never ignored) */

/* running mode: fast2q.py:1294-1297 ('C' / 'EC') */
#define F2Q_MODE_COUNT          0
#define F2Q_MODE_EXTRACT_COUNT  1

/*
 * Parameters of the hot path — the subset of the reference's `param` dict that fastq_parser,
 * sequence_tinder and reads_counter read (fast2q.py:538-558, 1112-1129, 1246-1309).
 * Values are the RAW command-line integers; clamping (ph<=0 -> 1, fast2q.py:1118-1125) and the
 * fail-set construction (fast2q.py:1127-1129) happen inside the library exactly as in the reference.
 * Fixed mode (has_up==0 && has_down==0): n_iter = number of --st items, starts[] = those ints.
 * Delimiter mode: n_iter = max(#up, #down) (fast2q.py:558); up/down hold the UPPER-CASED search
 * sequences (fast2q.py:547,550); when both are given their counts must match (fast2q.py:553-556).
 */
typedef struct f2q_config {
    int32_t mode;        /* F2Q_MODE_* */
    int32_t miss;        /* --m   mismatches allowed per feature (Counter mode only) */
    int32_t phred;       /* --ph  */
    int32_t qual_up;     /* --qsu */
    int32_t qual_down;   /* --qsd */
    int32_t miss_up;     /* --msu */
    int32_t miss_down;   /* --msd */
    int32_t length;      /* --l   */
    int32_t n_iter;      /* search_iterations */
    int32_t has_up;      /* --us given */
    int32_t has_down;    /* --ds given */
    int32_t starts[F2Q_MAX_ITER];     /* --st items (fixed mode) */
    int32_t up_len[F2Q_MAX_ITER];
    int32_t down_len[F2Q_MAX_ITER];
    uint8_t up[F2Q_MAX_ITER][F2Q_MAX_DELIM];
    uint8_t down[F2Q_MAX_ITER][F2Q_MAX_DELIM];
} f2q_config;

/* order of the five per-sample statistics (local_read_stats, fast2q.py:310-316) */
#define F2Q_STAT_READS           0
#define F2Q_STAT_PERFECT         1
#define F2Q_STAT_IMPERFECT       2
#define F2Q_STAT_NON_ALIGNED     3
#define F2Q_STAT_QUALITY_FAILED  4
#define F2Q_N_STATS              5

typedef struct f2q_ctx f2q_ctx;

/* ---- library / device ------------------------------------------------------------------- */
int f2q_abi_version(void);
/* number of usable devices (compute capability 10.x); 0 when there is none, never an error */
int f2q_device_count(void);

/*
 * Create a context on `device`.  `stream` is a cudaStream_t the work is enqueued on (so a caller can
 * bracket it with its own events) or NULL for a library-owned stream.
 * Replaces: the per-call parameter derivation of reads_counter (fast2q.py:536-558).
 */
int f2q_create(const f2q_config* cfg, int device, void* stream, f2q_ctx** out);
void f2q_destroy(f2q_ctx* ctx);
const char* f2q_last_error(const f2q_ctx* ctx);   /* ctx may be NULL: last create-time error */

/* tunables; must be set before the first f2q_begin_sample.  Unknown names -> F2Q_EINVAL.
 *   "carry_bytes"     max bytes of one partial FASTQ record carried between submits (default 4 MiB)
 *   "stage_bytes"     size of each internal pinned/device staging slot used by f2q_submit (default 64 MiB)
 *   "stage_slots"     number of staging slots (default 3)
 *   "resolver"        kernel for queued non-exact keys: 0 auto | 1 Hamming-1 neighbour probing | 2 pigeonhole seed
 *                     index | 3 library tile scan (small libraries decide distance-1 keys in the lookup table itself)
 *   "queue_entries"   capacity of the deferred non-exact key queue (default: derived from the chunk size;
 *                     capacity never changes results — overflow is resolved in place)
 *   "force_generic"   1: run every read through the byte-wise generic kernels (cross-check of the packed path)
 *   "row_chunks"      0 auto | 3 | 5 | 7: bytes per tile row / 16 (auto: just below the record length of the sample)
 *   "halo_rows"       0 auto | read-ahead rows at the end of every tile (reads reaching further finish in global memory)
 *   "tile_threads"    128 | 256: threads (= rows) per CTA of the exact look-back kernel (default: 256 for the packed
 *                     single-window policy, 128 for the generic per-read code)
 *   "time_kernels"    1: bracket the tile / resolver / generic launches with CUDA events (see f2q_kernel_times)
 *   "debug_waits"     1: the exact kernel counts the cycles of each of its waits; f2q_end_sample prints them on stderr
 *   "spec"            1 (default): Counter mode parses each chunk with the speculative streaming kernel first and
 *                     falls back to the exact look-back kernel when its line-phase guesses do not verify | 0: exact only
 *   "spec_warps"      12 | 16: warps per CTA of the streaming kernel (one CTA per SM)
 *   "spec_range_tiles" 0 auto | tiles (32 rows each) per speculated range
 *   "flex"            1 (default): search sequences / several windows per read / Extract+Count run on the bit-parallel
 *                     policies of the streaming kernel when the configuration allows | 0: byte-wise generic kernels
 *   "flex_warps"      12 | 16: warps per CTA of the streaming kernel's bit-parallel policies
 *   "resolve_group"   0 auto | 1 | 8 | 32: lanes that resolve one non-exact key together (seed-index resolvers)
 *   "memo_entries"    0 off (default) | power of two: entries of the device memo of resolved non-exact keys; set before
 *                     f2q_set_library.  Worth it when the stream repeats its erroneous keys (real screens do; the host layer
 *                     2fast2q_b200/fast2q.py switches it on), pure overhead when it does not (the synthetic bench streams)
 *   "gpu_inflate"     1 (default): f2q_submit_file inflates bgzip (BGZF) files ON THE DEVICE (k_inflate_bgzf_lanes: the 32
 *                     lanes of a warp inflate 32 blocks in lock step; only the compressed bytes cross PCIe) | 0: on host
 *                     threads, block-parallel | 2: on the device, one free-running thread per block (cross-check, slow)
 *   "gpu_inflate_bits" 0 auto | 8 | 9: index bits of the GPU inflate's literal/length lookup table (8: 640 B of shared memory per
 *                     lane, 11 warps per SM; 9: 1 280 B, 5 warps; auto takes 8 when a batch has more than 5 warps per SM)
 *   "seed_parts"      0 auto | P: segments of the resolver's seed plan (a key within m mismatches agrees with its library
 *                     entry on some P - m of P segments; seeds = all such choices; auto picks P from the library size);
 *                     set before f2q_set_library.  A P that does not fit (P <= m, more than 32 seeds, seeds longer than
 *                     16 symbols) falls back to the classic m + 1 one-segment seeds
 *   "generic_entries" capacity of the queue of reads handed to the byte-wise generic kernel (default: derived)
 *   "ec_slots"        minimum capacity of the Extract+Count packed key table (default: grown on demand)
 */
int f2q_set_option(f2q_ctx* ctx, const char* name, int64_t value);

/*
 * Counter mode library = the keys of the dict built by features_loader (fast2q.py:125-186), i.e. the
 * upper-cased, space-stripped sequences, in file order, duplicates already removed.
 * key i = key_bytes[key_offsets[i] .. key_offsets[i+1]).  Keys may contain any bytes (':' for
 * multi-feature entries).  Builds the device tables that replace binary_converter (fast2q.py:188-213).
 */
int f2q_set_library(f2q_ctx* ctx, const uint8_t* key_bytes, const uint64_t* key_offsets, uint32_t n_keys);

/* ---- one sample (= one FASTQ stream) ------------------------------------------------------ */
/* zero the count vector / statistics / carried state.  Replaces the per-file entry of reads_counter. */
int f2q_begin_sample(f2q_ctx* ctx);

/*
 * Feed the next `nbytes` of the UNCOMPRESSED stream, in file order, from HOST memory.  Chunks may cut
 * records anywhere; the context carries the partial record (fast2q.py:324-328 — a record is every four
 * '\n'-separated lines counted from byte 0).  The copy is staged through internal pinned slots and is
 * asynchronous when host_chunk itself is pinned (f2q_host_alloc); the call may block until a slot frees.
 * is_last != 0 marks end of stream (a final unterminated 4th line still completes a record).
 */
int f2q_submit(f2q_ctx* ctx, const uint8_t* host_chunk, uint64_t nbytes, int is_last);

/*
 * One sequencing file -> the current sample, natively: the file is read (is_gzip == 0) or inflated with zlib (is_gzip != 0;
 * multi-member and zero-padded files as Python's gzip module reads them; bgzip/BGZF files block-parallel on `threads` host
 * threads) straight into page-locked ring buffers near the GPU and submitted from there; the stream is closed (is_last).
 * Replaces the open / gzip.open + `for line in current` of reads_counter / fastq_parser (fast2q.py:566-578, 324).
 * limit_lines > 0 stops after that many lines (preprocess mode parses 10 000 reads = 40 000 lines, fast2q.py:398-400).
 * *complete (may be NULL) = 0 when a gzip stream broke off before its end: every complete line before the break has been
 * parsed and the partial one dropped, as the reference's line iterator does before its EOFError (fast2q.py:405-407).
 * Corrupted deflate data -> F2Q_EINVAL (the reference crashes with zlib.error).  *bytes_out = uncompressed bytes submitted.
 */
int f2q_submit_file(f2q_ctx* ctx, const char* path, int is_gzip, uint64_t limit_lines, int threads, int* complete, uint64_t* bytes_out);

/*
 * One plain or bgzip file as ONE sample parsed by n contexts (on one device or several; no NCCL): the file is cut into byte
 * ranges, context k parses range k on a host thread of its own (`threads` readers are divided among them), and on return
 * ctxs[0] holds the whole sample — counts, statistics, the device error word and, in Extract+Count mode, the merged key
 * table — so f2q_end_sample / f2q_end_sample_async / f2q_ec_size / f2q_ec_drain on ctxs[0] work as after f2q_submit_file.
 * Every other context's sample is closed and empty.  *complete and *bytes_out mean what they mean for f2q_submit_file.
 * Preconditions: n >= 1, no context twice (else F2Q_EINVAL); every context inside a freshly begun sample (else F2Q_ESTATE);
 * all with the same f2q_config bytes and the same library (else F2Q_EINVAL).
 * cuts: NULL splits the file evenly into ranges of at least 64 MiB (a small file uses fewer contexts), or n-1 non-decreasing
 * file offsets (bgzip: rounded up to the next block start); empty ranges are dropped.
 * Protocol: a range that starts mid-file guesses its first record start on the device (the one byte behind its 1st..4th
 * newline where two records of FASTQ shape start); the bytes before it (its head) and the partial record behind the last
 * whole record of the range before (its tail) are parsed on ctxs[0] in file order.  A guess is right exactly when the
 * tail's newlines plus the head's are a multiple of 4; this is checked for every range, so by induction every record is
 * parsed once at its true line phase.  The whole file is parsed again on ctxs[0] alone (the other samples restart empty)
 * for ordinary gzip (nothing to cut at), a bgzip file that is not whole BGZF blocks ending with the end-of-file block, a
 * range with no unique guess, or a failed check: the results are then exactly f2q_submit_file's.
 * f2q_get_info "shards" / "shard_fallback" on ctxs[0] tell how many contexts parsed the sample and whether it fell back.
 */
int f2q_submit_file_sharded(f2q_ctx** ctxs, int n, const char* path, int is_gzip, const uint64_t* cuts, int threads,
                            int* complete, uint64_t* bytes_out);

/* Same, but the chunk already lives in device memory of this context's GPU (resident mode).  The buffer
 * must stay valid and unmodified until the next f2q_end_sample/f2q_sync returns. */
int f2q_submit_device(f2q_ctx* ctx, const void* dptr, uint64_t nbytes, int is_last);

/* block until everything submitted so far has been consumed (device buffers may be reused after) */
int f2q_sync(f2q_ctx* ctx);

/* block until every host chunk handed to f2q_submit so far has been copied off the host: pinned buffers
 * (f2q_host_alloc) may be refilled after this returns, while the kernels that parse the copies still run */
int f2q_sync_copies(f2q_ctx* ctx);

/*
 * Finish the sample: waits, then writes counts[n_keys] (Counter mode; may be NULL in EC mode) and the
 * five statistics.  Replaces the return value of fastq_parser (fast2q.py:409).
 * If the stream was never closed with is_last the carried partial record is dropped, exactly as the
 * reference drops 1–3 left-over lines.
 */
int f2q_end_sample(f2q_ctx* ctx, uint64_t* counts, uint64_t stats[F2Q_N_STATS]);

/*
 * Counter mode, many samples back to back: finish the sample WITHOUT waiting.  The stream is closed (a carried final
 * record is flushed) and [counts[n_keys] | stats[5] | error word] (n_keys + 6 uint64) is copied, stream-ordered, into
 * pinned_out, which must come from f2q_host_alloc.  f2q_begin_sample may follow at once; the numbers are valid after the
 * next f2q_sync (or any later blocking call).  A non-zero error word reports a device-side failure of that sample
 * (low half: kernel error flags, high half: stream state flags; F2Q_ETOOLONG's bit is 2 of the high half).
 */
int f2q_end_sample_async(f2q_ctx* ctx, uint64_t* pinned_out);

/* device address of the uint64 vector [counts[n_keys] | stats[5]] of the current sample, valid after
 * the work was enqueued; for an in-place NCCL all-reduce over ranks (merge_feature_dicts,
 * fast2q.py:439-445, 487-495).  After a reduce call f2q_end_sample as usual. */
int f2q_result_device(f2q_ctx* ctx, void** dptr, uint64_t* n_words);

/* ---- Extract + Count mode (fast2q.py:382-387) -------------------------------------------- */
/* number of distinct keys and total key bytes of the current sample (synchronises) */
int f2q_ec_size(f2q_ctx* ctx, uint64_t* n_keys, uint64_t* key_bytes);
/* copy out keys (concatenated), offsets[n_keys+1] and counts[n_keys]; order unspecified */
int f2q_ec_drain(f2q_ctx* ctx, uint8_t* key_bytes, uint64_t* key_offsets, uint64_t* counts);

/* ---- several GPUs (NCCL over NVLink / NVSwitch) --------------------------------------------------
 * Reads shard over GPUs with no data-path collective (every rank parses its own byte range / its own record-aligned
 * shards); what is exchanged is the per-sample RESULT.  Replaces merge_feature_dicts and the statistics additions of the
 * reference's chunked mode (fast2q.py:439-445, 487-495) and the per-file pool of fast2q.py:1646-1655.
 * libnccl is loaded at run time: f2q_comm_load(path) (or NULL: F2Q_NCCL_LIB, then the default library search).
 * One process per GPU: rank 0 calls f2q_comm_unique_id, ships the 128 bytes to the other ranks by any means, every rank
 * calls f2q_comm_init_rank.  One process, several contexts on distinct devices: f2q_comm_init(ctxs, n).
 * Collective calls take the contexts of THIS process that take part (n = 1 with one process per GPU).
 *   f2q_allreduce_counts  in-place sum over all ranks of [counts | stats], stream-ordered; call it after the last submit of
 *                         the sample, then f2q_end_sample / f2q_end_sample_async as usual (every rank gets the totals)
 *   f2q_ec_merge          Extract+Count: the key tables of all ranks are gathered on every rank and merged on the device
 *                         (counts of equal keys add); f2q_ec_size / f2q_ec_drain then return the merged table on every rank.
 *                         Call it after f2q_end_sample (statistics: sum them with f2q_allreduce_counts before that). */
int f2q_comm_load(const char* libnccl_path);
int f2q_comm_unique_id(uint8_t id128[128]);
int f2q_comm_init_rank(f2q_ctx* ctx, const uint8_t id128[128], int nranks, int rank);
int f2q_comm_init(f2q_ctx** ctxs, int n);
int f2q_comm_destroy(f2q_ctx* ctx);
/* ctx (same device, same process) uses `from`'s communicator, which must outlive it */
int f2q_comm_share(f2q_ctx* ctx, f2q_ctx* from);
int f2q_allreduce_counts(f2q_ctx** ctxs, int n);
int f2q_ec_merge(f2q_ctx** ctxs, int n);

/* ---- pinned host memory for f2q_submit ------------------------------------------------------ */
int f2q_host_alloc(void** ptr, uint64_t nbytes);
/* the same for the chunks of ONE device: on that device's NUMA node (/sys/bus/pci/devices/<bdf>/numa_node; mmap + mbind +
 * cudaHostRegister) when the platform shows more than one node — eight GPUs fed from one socket's memory share that socket's
 * bandwidth.  flags bit 0: write-combined.  *numa_node (may be NULL) = the node the buffer was bound to, -1 when none was
 * (single-node platforms such as VMs).  Free with f2q_host_free. */
int f2q_host_alloc_near(void** ptr, uint64_t nbytes, int device, int flags, int* numa_node);
int f2q_host_free(void* ptr);

/* ---- primitives with public reference counterparts (README.md:259-298; tests/test_mainfunctions.py) ----
 * Device implementations of border_finder (fast2q.py:628-658) and sequence_tinder (:215-285) run on ONE read
 * (context-free: they allocate, launch and free on `device`); used by the host-side helpers of the same names
 * and by the known-answer tests.
 * f2q_border_finder: *pos = first index >= start_place with <= mismatch mismatches, or -1 for the reference's None.
 * f2q_sequence_tinder: cfg supplies up/down/miss_up/miss_down/length/qual_up/qual_down; set_up/set_down optionally
 *   override the delimiter fail sets with explicit 256-bit byte sets (uint64[4], bit b of word b>>6) because the
 *   reference helper takes arbitrary sets.  *found = 0 for the reference's (None, None).
 */
int f2q_border_finder(int device, const uint8_t* seq, uint32_t seq_len, const uint8_t* read, uint32_t read_len,
                      int32_t mismatch, int32_t start_place, int32_t* pos);
int f2q_sequence_tinder(int device, const f2q_config* cfg, int32_t iteration, const uint8_t* read, uint32_t read_len,
                        const uint8_t* qual, uint32_t qual_len, const uint64_t* set_up, const uint64_t* set_down,
                        int32_t* found, int32_t* start, int32_t* end);

/* ---- synthetic FASTQ generator K0 (bench/tests only; SURVEY.md §8d) -------------------------- */
typedef struct f2q_synth_spec {
    uint64_t seed;
    uint64_t first_read;     /* global index of the first read to generate */
    uint64_t n_reads;
    uint32_t read_len;       /* L; record = 2L+18 bytes */
    uint32_t feat_len;       /* guide length placed at read offset 0 */
    uint32_t n_guides;
    /* cumulative class thresholds out of 65536: exact | 1 sub | 2 sub | 3 sub | one N | (rest = random) */
    uint32_t cum_exact, cum_sub1, cum_sub2, cum_sub3, cum_n;
    uint32_t lowq_per_65536; /* fraction of reads that get one low-quality byte */
    /* workload shape: 0 guide at offset 0 + random tail (configs 2, 3; the class thresholds above apply) |
     * 1 Bar-seq: stagger + delim[0] + barcode + delim[1] + pad (config 4) | 2 dual fixed: X at 0, Y at feat_len+10
     * (config 5a) | 3 dual delimiters: delim[0] X delim[1] .. delim[2] Y delim[3] (config 5b).  Shapes 2/3 take
     * 2*n_guides sequences: the X's, then the Y's.  Class mixes of shapes 1-3 are fixed (csrc/synth_gen.h). */
    uint32_t shape;
    uint32_t delim_len[4];
    uint8_t  delim[4][16];
} f2q_synth_spec;
/* writes n_reads*(2L+18) bytes at dptr (device); guides = n_guides*feat_len (shapes 2/3: 2*n_guides*feat_len) ASCII
 * bytes on the HOST.  Asynchronous on the context's stream when n_guides == 0 && guides == NULL re-uses the guide
 * table uploaded by the previous call (per-chunk generation of workloads larger than HBM). */
int f2q_synth_fastq(f2q_ctx* ctx, const f2q_synth_spec* spec, const uint8_t* guides, void* dptr);

/* device memory helpers so that a non-CUDA host language can hold resident chunks */
int f2q_device_alloc(f2q_ctx* ctx, void** dptr, uint64_t nbytes);
int f2q_device_free(f2q_ctx* ctx, void* dptr);
int f2q_memcpy_d2h(f2q_ctx* ctx, void* host, const void* dptr, uint64_t nbytes);
int f2q_memcpy_h2d(f2q_ctx* ctx, void* dptr, const void* host, uint64_t nbytes);

/* number of kernel launches issued by this context so far (bench.py reports it as gpu_launches) */
uint64_t f2q_launch_count(const f2q_ctx* ctx);

/* last finished sample: number of chunks whose speculative parse verified and was committed, and number of chunks the
 * exact look-back kernel had to parse instead (always 0 / every chunk with option "spec" = 0) */
int f2q_spec_counts(const f2q_ctx* ctx, uint64_t* committed, uint64_t* fell_back);

/* last finished sample (f2q_end_sample): lookups of non-exact keys in the device memo of resolved keys and how many of them
 * hit.  The memo is the device analogue of the reference's passed_reads / failed_reads (fast2q.py:724-731, 741, 748): it
 * lives with the library — across chunks and samples of the context — and never changes a count (option "memo_entries"). */
int f2q_memo_counts(const f2q_ctx* ctx, uint64_t* lookups, uint64_t* hits);

/* read-only view of the shapes the context chose, by name (results never depend on them; tests use them to prove which
 * side of a size threshold an input landed on):
 *   "policy"        per-read code of the streaming kernel: 0 byte-wise generic | 1 fast1 (one fixed window, Counter) |
 *                   2 flex_S (bit-parallel, 96-position planes, k <= 1) | 3 flex_B (160-position planes, k <= 3).
 *                   Final after the first submit of a sample (the record length sniffed there can move flex_S to flex_B)
 *   "table"         exact lookup table of the packed library keys: 0 probing | 1 compact | 2 two-choice cuckoo |
 *                   3 cuckoo that also holds every Hamming-1 neighbour
 *   "hist"          this sample's launches used the per-CTA shared-memory histogram: bit 0 the streaming kernel, bit 1 the
 *                   exact kernel
 *   "seed_parts"    segments P of the resolver's seed plan; 0 = the classic m + 1 one-segment seeds (or no seed index)
 *   "flex_table"    1 when the library has the flex tables (every key <= 2 ACGT pieces of <= 32 symbols)
 *   "generic_reads" reads the generic read queue took during the last finished sample (one device-to-host copy per call;
 *                   F2Q_ESTATE inside a sample)
 *   "shards"        contexts that parsed the current / last sample (f2q_submit_file_sharded; 1 otherwise and after a fallback)
 *   "shard_fallback" 1 when f2q_submit_file_sharded parsed the sample again on ctxs[0] alone */
int f2q_get_info(f2q_ctx* ctx, const char* name, int64_t* value);

/* device time of the last finished sample per kernel class, measured with CUDA events on the context's stream
 * (needs option "time_kernels" = 1): [0] fused tile kernel over the chunk (the streaming kernel when "spec" is on),
 * [1] mismatch resolver, [2] generic queue, [3] speculation verify + commit + the exact kernel behind it (which
 * returns at once when the speculation held).  launches[k] = number of event brackets ms[k] sums over. */
int f2q_kernel_times(f2q_ctx* ctx, double ms[4], uint64_t launches[4]);

#ifdef __cplusplus
}
#endif
#endif /* F2Q_H_ */
