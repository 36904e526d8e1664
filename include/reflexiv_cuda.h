/*
 * reflexiv_cuda.h -- C ABI of libreflexiv_cuda, the B200 (sm_100a) implementation of Reflexiv's
 * k-mer counting + de Bruijn contig-extension path.
 *
 * The reference (rhinempi/Reflexiv) has no FFI: the path is a chain of Spark Dataset stages inside
 *   src/main/java/uni/bielefeld/cmg/reflexiv/pipeline/ReflexivDataFrameCounter.java:139-236   (`reflexiv counter`)
 *   src/main/java/uni/bielefeld/cmg/reflexiv/pipeline/ReflexivDSMain.java:123-357            (`reflexiv run`)
 * This header is the seam a Java driver (JNI / Panama FFM, see INTEGRATION.md) binds instead of those
 * stages.  Each entry point names the reference stage(s) it replaces.  Plain pointers and sizes only.
 *
 * Conventions
 *   - every call returns RFX_OK (0) or a negative rfx_status; rfx_last_error() gives the message;
 *     the library never throws, exits or falls back to the CPU;
 *   - host buffers are caller owned and not retained; results are copied into caller buffers;
 *   - one context per driver thread, calls are blocking, the context owns its CUDA stream;
 *   - k-mers are 2 bits per base (A=0 C=1 G=2 T=3, every other character counts as T exactly as
 *     nucleotideValue() does), first base most significant.
 */
#ifndef REFLEXIV_CUDA_H
#define REFLEXIV_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct rfx_ctx rfx_ctx;

typedef enum {
    RFX_OK = 0,
    RFX_E_INVALID = -1,     /* bad argument / unsupported parameter value */
    RFX_E_CUDA = -2,        /* CUDA runtime error (message has the cudaError string) */
    RFX_E_NOMEM = -3,       /* device allocation failed */
    RFX_E_STATE = -4,       /* call out of order (e.g. rfx_assemble before rfx_count) */
    RFX_E_CAPACITY = -5,    /* an internal table overflowed; raise table_capacity */
    RFX_E_GRAPH = -6,       /* k-mer set violates the in/out-degree <= 1 invariant after the fork filters */
    RFX_E_UNSUPPORTED = -7  /* reference behaviour undefined for this option (see DESIGN.md) */
} rfx_status;

/* FASTQ line filter, selects which reference reader is mirrored */
enum {
    RFX_FASTQ_RUN = 0,     /* 4-line state machine: DSFastqFilterWithQual, ReflexivDSMain.java:4048-4072 */
    RFX_FASTQ_COUNTER = 1, /* stateless heuristic:  DSFastqFilterOnlySeq, ReflexivDataFrameCounter.java:243-289 */
    RFX_FASTQ_LINE = 2     /* -infmt line: every line is a read, ReflexivDataFrameCounter.java:184 */
};

/* The parameter block every reference operator closes over: util/DefaultParam.java:54-141. */
typedef struct {
    int32_t struct_size;        /* sizeof(rfx_params), for ABI evolution */
    int32_t kmer_size;          /* -kmer          (31)        1..63 */
    int32_t min_kmer_coverage;  /* -cover         (2)  */
    int32_t max_kmer_coverage;  /* -maxcov        (10000000) */
    int32_t min_error_coverage; /* -error         (8 = 4 * default cover; NOT updated by -cover, Parameter.java:479-487) */
    int32_t min_contig;         /* -mincontig     (500) */
    int32_t front_clip;         /* -clipf         (0) */
    int32_t end_clip;           /* -clipe         (0) */
    int32_t bubble;             /* 1 = fork filters on (default); -bubble clears it -> RFX_E_UNSUPPORTED in rfx_assemble */
    int32_t min_iter;           /* -miniter       (15)  accepted; the extension runs to its fixed point */
    int32_t max_iter;           /* -maxiter       (150) accepted */
    int32_t partitions;         /* -partition     (0)   accepted, no numerical effect */
    int32_t shuffle_partitions; /* -partitionredu (200) accepted, no numerical effect */
    int32_t counter_mode;       /* 1 = `reflexiv counter` filter rule (ReflexivDataFrameCounter.java:202-210):
                                   lower bound only if cover > 1, upper only if maxcov < 10000000;
                                   0 = `reflexiv run` rule (ReflexivDSMain.java:211-216): always both */
    int32_t fastq_mode;         /* RFX_FASTQ_* */
    int32_t device;             /* CUDA device ordinal */
    int32_t minimizer_len;      /* 0 = auto.  super-k-mer minimiser length (<= 16) */
    int32_t reserved0;
    int64_t table_capacity;     /* 0 = auto.  rows reserved for the filtered (k-mer, count) table */
    int64_t bin_target_kmers;   /* 0 = auto.  k-mer instances per counting bin */
} rfx_params;

typedef struct {
    uint64_t n_reads;        /* sequence lines accepted by the FASTQ filter */
    uint64_t n_bases;        /* bases kept after clipping / minimum-length rule */
    uint64_t n_instances;    /* k-mer instances extracted (A2) */
    uint64_t n_distinct;     /* distinct canonical k-mers before the coverage filter (A3) */
    uint64_t n_rows;         /* rows after the coverage filter (A4) */
    uint64_t n_records;      /* super-k-mer records */
    uint64_t n_bins;
    uint64_t n_bin_splits;   /* counting bins that had to be re-run in sub-classes */
    uint64_t n_oriented;     /* oriented k-mers surviving both fork filters (A7, A8) */
    uint64_t n_budget_junctions;   /* junctions whose two flags have different signs as the fork filters left them */
    uint64_t n_budget_admissible;  /* k-mers absorbed by budget walks (clause 3 / 4 merges, ReflexivDSMain.java:3077-3084) */
    uint64_t n_cycles;
    uint64_t n_contigs;
    uint64_t n_contig_bases;
    uint64_t kernel_launches;  /* kernels launched by this context since creation */
    float ms_parse;    /* K1: line split + FASTQ filter + 2-bit encode */
    float ms_partition;/* K2: minimiser binning into super-k-mer records */
    float ms_count;    /* K3+K4: per-bin counting + coverage filter */
    float ms_graph;    /* K5: both orientations, fork filters, neighbour links */
    float ms_extend;   /* K6: list ranking */
    float ms_contigs;  /* K7: contig gather */
    /* single-kernel durations of the last rfx_count (CUDA events around the launch only) */
    float ms_kernel_bin_histogram; /* minimiser scan (bin_scan_fast_kernel / bin_scan_kernel): one GPU: scan + record store into the
                                      bin slabs; sharded: scan + run descriptors + bin histogram */
    float ms_kernel_bin_scatter;   /* emit_records_kernel (sharded runs only): super-k-mer records into the compact layout */
    float ms_kernel_count;         /* count_bins_kernel (pilot, when it runs, + main launch) */
    float reserved1;
} rfx_stats_t;

int rfx_params_default(rfx_params* p);

int rfx_create(rfx_ctx** out, const rfx_params* p);
void rfx_destroy(rfx_ctx* ctx);
const char* rfx_last_error(const rfx_ctx* ctx); /* ctx may be NULL: error of the last failed rfx_create */
int rfx_reset(rfx_ctx* ctx);                     /* forget reads and results, keep device buffers */

/* ---- input ----------------------------------------------------------------------------------
 * replaces spark.read().text + DSFastqFilterWithQual / DSFastqFilterOnlySeq
 * (ReflexivDSMain.java:188-195, ReflexivDataFrameCounter.java:178-188).
 * `buf` is decompressed FASTQ text in host memory; may be called repeatedly, every call must end on a
 * line boundary and (RFX_FASTQ_RUN) on a record boundary. */
int rfx_push_fastq(rfx_ctx* ctx, const uint8_t* buf, size_t len);
/* same, `d_buf` is a CUDA device pointer on the context's device (used when the text is already in HBM).
 * The parser reads whole 64-byte aligned chunks: the allocation must extend to the next 64-byte boundary behind
 * d_buf + len (always true for a cudaMalloc'ed buffer). */
int rfx_push_fastq_device(rfx_ctx* ctx, const uint8_t* d_buf, size_t len);
/* already-split reads: ASCII bases, read i = bases[offsets[i] .. offsets[i+1]) (host memory) */
int rfx_push_reads(rfx_ctx* ctx, const uint8_t* bases, const uint64_t* offsets, uint64_t n_reads);

/* ---- counting ------------------------------------------------------------------------------
 * replaces ReverseComplementKmerBinaryExtractionFromDataset(64) + groupBy("value").count() + coverage filter
 * (ReflexivDataFrameCounter.java:195-210, ReflexivDataFrameCounter64.java:197-212, ReflexivDSMain.java:204-216). */
int rfx_count(rfx_ctx* ctx);
int rfx_counts_size(rfx_ctx* ctx, uint64_t* n_rows, int32_t* words_per_key);
/* keys: n_rows * words_per_key uint64, laid out exactly like the reference's key column so that
 * DSBinaryKmerToString (ReflexivDataFrameCounter.java:405-428, Counter64.java:340-369) decodes them:
 * k <= 31 one word, right aligned; k > 31: k/32+1 words, 32 bases per word, the last word holds k%32
 * bases right aligned.  Row order is unspecified (as in the reference). */
int rfx_counts_copy(rfx_ctx* ctx, uint64_t* keys, uint32_t* counts);
/* `KMER,count\n` rows (the reference's CSV part-file content, A5).  Call with out == NULL to get the size. */
int rfx_counts_csv(rfx_ctx* ctx, char* out, uint64_t cap, uint64_t* n_bytes);
/* load an existing filtered table instead of counting (the -kmerc seam, ReflexivDSMain.java:362-713);
 * keys in the layout rfx_counts_copy produces */
int rfx_load_counts(rfx_ctx* ctx, const uint64_t* keys, const uint32_t* counts, uint64_t n_rows);

/* ---- assembly ------------------------------------------------------------------------------
 * replaces DSKmerReverseComplementLong .. DSExtendReflexivKmerToArrayLoop .. DSKmerToContig
 * (ReflexivDSMain.java:221-338). */
int rfx_assemble(rfx_ctx* ctx);
int rfx_contigs_size(rfx_ctx* ctx, uint64_t* n_contigs, uint64_t* total_bases);
/* bases: total_bases chars ACGT; offsets: n_contigs+1; left/right: the two flags printed in the header
 * ">Contig-<len>-(<left>,<right>)-<idx>" (DSKmerToContig, ReflexivDSMain.java:743-771).
 * Every contig appears on both strands, order unspecified (as in the reference). */
int rfx_contigs_copy(rfx_ctx* ctx, char* bases, uint64_t* offsets, int32_t* left, int32_t* right);
/* surviving oriented k-mers with their fork-filter flags (the Count_<k>_sorted content, SURVEY 8f-2) */
int rfx_oriented_size(rfx_ctx* ctx, uint64_t* n);
int rfx_oriented_copy(rfx_ctx* ctx, uint64_t* keys_hi, uint64_t* keys_lo, int32_t* left, int32_t* right);

/* ---- Count_<k>_sorted (the "left and right sorting" stage of the reference's multi-k workflows) ----
 * Replaces ReflexivDSKmerLeftAndRightSorting.assemblyFromKmer() (pipeline/ReflexivDSKmerLeftAndRightSorting.java:105-243,
 * called from pipeline/Pipelines.java:1309-1313): both orientations of every row of the context's count table go
 * through that class's two fork filters (:432-537, :700-818) and every survivor becomes a row `KMER,1|left|right`
 * (:249-274) with left / right in {-1, max_kmer_size + 3}.  The table is used as it stands: the caller applies the
 * stage's `count <= maxcov` rule (:186-193) when it loads or counts (rfx_params.max_kmer_coverage).
 *   min_error_coverage  param.minErrorCoverage (util/DefaultParam.java:106; Pipelines.java:1412-1416 sets 3 * cover for k >= 61)
 *   min_repeat_fold     param.minRepeatFold    (util/DefaultParam.java:107: 1.5)
 *   max_kmer_size       param.kmerListInt[last] (util/DefaultParam.java:87: 95 for the default list)
 * RFX_E_UNSUPPORTED where the reference itself cannot run: min_error_coverage == 0, (k-1) % 31 == 0.
 * Invalidates the results of rfx_assemble (the graph index and flag arrays are shared).
 * rfx_sort_kmers_sharded (multi-GPU block below) is the same stage on a table sharded across ranks. */
int rfx_sort_kmers(rfx_ctx* ctx, int32_t min_error_coverage, double min_repeat_fold, int32_t max_kmer_size);
int rfx_sorted_size(rfx_ctx* ctx, uint64_t* n_rows);
/* oriented k-mers (right-aligned, hi/lo halves) with their flags; caller buffers of n_rows elements each */
int rfx_sorted_copy(rfx_ctx* ctx, uint64_t* keys_hi, uint64_t* keys_lo, int32_t* left, int32_t* right);
/* the CSV text of Count_<k>_sorted/part-*.csv, formatted on the device; out == NULL: size query */
int rfx_sorted_csv(rfx_ctx* ctx, char* out, uint64_t cap, uint64_t* n_bytes);

/* ---- -stitch: low-coverage read rescue (SURVEY 8f-4) --------------------------------------------
 * Replaces the `if (param.stitch)` branch of ReflexivDSMain.assemblyFromKmer() (pipeline/ReflexivDSMain.java:585-672):
 * DSLowCoverageSubKmerExtraction (:1211-1268) + SubKmerProbRowToHash (:109-118) + the broadcast, the second pass over the
 * FASTQ with DSLowCoverageReadDetection (:1448-1612), DSFilterRepeatLowCoverageFragment (:922-1010), the union and the second
 * extension loop (:640-670).  One GPU.  For k > 31 the reference's own branch (ReflexivDSMain64.java:715-790) can never cut a read -- it
 * looks a Long up in a Hashtable keyed by List<Long> (:1562-1600, :119-131) -- so there the stage returns the plain assembly.
 *   rfx_load_counts | rfx_count  ->  rfx_stitch_begin  ->  rfx_push_fastq* (any number of calls)  ->  rfx_stitch_finish
 * rfx_stitch_begin runs the assembly itself (as rfx_assemble, but every record of the extension is kept whatever its
 * length: the -mincontig rule applies to the stitched set, as in the reference where DSKmerToContig runs last) and puts
 * the (k-1)-mers of the contig ends that are clean and covered at most 4 times into a probe table.  While the stage is
 * open, rfx_push_fastq / rfx_push_fastq_device / rfx_push_reads do not store reads: every sequence line of the `run`
 * FASTQ filter (unclipped, as the reference reads units[1]) is scanned on both strands for a "left extendable" probe
 * followed by a "right extendable" probe of another contig, and the piece between them is kept as a fragment.
 * rfx_stitch_finish keeps one fragment per contig end, joins contig + fragment + contig chains and REPLACES the contigs
 * that rfx_contigs_size / rfx_contigs_copy return.  rfx_reset, rfx_count, rfx_load_counts*, rfx_assemble and rfx_sort_kmers
 * abandon an open stage (its fragments refer to the contigs it was opened on).  The order-dependent choices of the reference (probe collisions, which
 * fragment of a run stays, rings) are fixed as DESIGN.md section 2 lists them. */
typedef struct {
    uint64_t n_probes;      /* keys in the probe table */
    uint64_t n_reads;       /* sequence lines scanned */
    uint64_t n_fragments;   /* fragments cut from reads (both strands) */
    uint64_t n_after_pass1; /* ... one per contig end they leave (DSFilterRepeatLowCoverageFragment) */
    uint64_t n_joined;      /* ... that also won the contig they end on */
    uint64_t n_stitched;    /* records made of more than one piece */
    uint64_t n_rings;       /* closed chains, opened at their smallest first k-mer */
    float ms_stitch;        /* probe table + finish (the read scan is part of ms_parse) */
    float reserved;
} rfx_stitch_stats_t;
int rfx_stitch_begin(rfx_ctx* ctx);
int rfx_stitch_finish(rfx_ctx* ctx);
int rfx_stitch_stats(rfx_ctx* ctx, rfx_stitch_stats_t* out);

int rfx_stats(rfx_ctx* ctx, rfx_stats_t* out);

/* ---- sharded counting (one context per GPU; the caller moves records between GPUs) ------------
 * Bins are laid out shard-major: with B bins in total, shard s owns bins [s*B/n, (s+1)*B/n) and its
 * records are one contiguous device slice.  Sender: rfx_partition(ctx, n, B) then rfx_shard_records()
 * for every s.  The caller exchanges the slices (NCCL all-to-all over NVLink: this replaces the
 * groupBy hash shuffle, ReflexivDataFrameCounter.java:198-200).  Receiver: rfx_begin_shard(ctx, s, n, B),
 * rfx_load_records_device() for every received slice, then rfx_count() re-bins and counts them.
 * B (n_bins_total) must be the same on every rank and a multiple of n; 0 = let the library choose
 * (single-process use only). */
int rfx_partition(rfx_ctx* ctx, int32_t n_shards, uint32_t n_bins_total);
/* the library's own choice of B for `global_instances` k-mer instances over n_shards shards (what rfx_count uses in a
 * single-process run); every rank of a sharded run calls it with the same arguments.  0 on bad arguments. */
uint32_t rfx_choose_bins(rfx_ctx* ctx, uint64_t global_instances, int32_t n_shards);
int rfx_shard_records(rfx_ctx* ctx, int32_t shard, const void** d_ptr, uint64_t* n_bytes);
int rfx_begin_shard(rfx_ctx* ctx, int32_t shard_id, int32_t n_shards, uint32_t n_bins_total);
int rfx_load_records_device(rfx_ctx* ctx, const void* d_records, uint64_t n_bytes);
/* Faster receive path: a sender's slice is already grouped by bin, so if its bin offsets travel with it the receiver
 * needs no re-binning at all -- rfx_count walks every bin as the concatenation of one segment per sender.
 * rfx_shard_bin_offsets: device pointer to the B/n + 1 record offsets (sender-absolute) of shard `shard`.
 * rfx_load_segment_device: append one received slice together with the offsets its sender exported.
 * Do not mix with rfx_load_records_device inside one rfx_begin_shard. */
int rfx_shard_bin_offsets(rfx_ctx* ctx, int32_t shard, const uint64_t** d_offsets, uint32_t* n_offsets);
int rfx_load_segment_device(rfx_ctx* ctx, const void* d_records, uint64_t n_bytes, const uint64_t* d_bin_offsets);
/* Optional zero-copy receive: after rfx_begin_shard, a device buffer of n_bytes owned by the context; slices received
 * into it back to back (sender 0 first) and then announced with rfx_load_segment_device in that order are used in place. */
int rfx_rx_buffer(rfx_ctx* ctx, uint64_t n_bytes, void** d_ptr);
int rfx_record_bytes(rfx_ctx* ctx, int32_t* bytes_per_record);
/* The filtered table as device pointers (valid until the next rfx_count / rfx_load_* / rfx_reset): keys are
 * key_bytes (8 for k <= 31, 16 for k > 31) little-endian right-aligned 2k-bit integers, i.e. the library's internal
 * layout, NOT the reference slot layout of rfx_counts_copy.  Used to move shard tables between GPUs. */
int rfx_counts_device(rfx_ctx* ctx, const void** d_keys, const uint32_t** d_counts, uint64_t* n_rows, int32_t* key_bytes);
/* Replace (append == 0) or extend (append != 0) the table from device memory in that same layout. */
int rfx_load_counts_device(rfx_ctx* ctx, const void* d_keys, const uint32_t* d_counts, uint64_t n_rows, int32_t append);

/* ---- multi-GPU over peer memory (one context per GPU = one rank; NVLink / NVSwitch) ---------------------------------
 * Replaces, across GPUs, the reference's shuffles: groupBy("value") (ReflexivDataFrameCounter.java:198-200,
 * ReflexivDSMain.java:207-209) and every sort("k-1") of the fork filters and of the extension loop
 * (ReflexivDSMain.java:232, 244, 261-326).  After rfx_shard_init all device buffers of the context live in one arena;
 * rfx_shard_export / rfx_shard_connect let every rank map every other rank's arena (CUDA IPC between processes, plain
 * pointers inside one process -- ranks may even share a device, which is how a one-GPU box tests the path).  The kernels
 * then read and write peer HBM directly: no collective library on the data path.
 *   every rank:  rfx_shard_init -> rfx_shard_export -> [caller gathers the world * RFX_SHARD_HANDLE_BYTES bytes] ->
 *                rfx_shard_connect -> { rfx_reset, rfx_push_fastq*, rfx_count_sharded, rfx_assemble_sharded, results }*
 * rfx_count_sharded / rfx_assemble_sharded are collective: every rank must call them (from its own host thread or
 * process); they meet in cross-GPU barriers and fail with RFX_E_STATE if a peer never arrives.  Ranks that share a device
 * inside one process meet on the host instead and need CUDA_MODULE_LOADING=EAGER in the environment (no kernel may be
 * loaded lazily while a peer on the same device waits).  rfx_assemble_sharded needs a table sharded by minimiser bin: the
 * one rfx_count_sharded leaves, or a loaded one after rfx_shard_table:
 *   every rank:  ... rfx_shard_connect -> { rfx_reset, rfx_load_counts* (any slice, may be empty), rfx_shard_table,
 *                rfx_assemble_sharded | rfx_sort_kmers_sharded, results }*
 * On return from rfx_count_sharded / rfx_shard_table the context holds its shard of the global table (the rows whose
 * minimiser bin it owns; rfx_counts_* work on it); after rfx_assemble_sharded it holds the contigs whose first k-mer it owns
 * (rfx_contigs_* work on them), after rfx_sort_kmers_sharded the Count_<k>_sorted rows of its shard (rfx_sorted_* work on
 * them): the union over the ranks is the result of the single-GPU calls. */
#define RFX_SHARD_HANDLE_BYTES 128
#define RFX_SHARD_MAX_RANKS 8
typedef struct {
    int32_t rank, world;
    uint64_t arena_bytes, arena_used;
    uint64_t n_instances_global;  /* k-mer instances extracted by all ranks */
    uint64_t n_shard_instances;   /* ... that fell into this rank's bins */
    uint64_t n_rows_global, n_oriented_global, n_contigs_global, n_contig_bases_global;  /* after rfx_sort_kmers_sharded:
                                     n_oriented_global = Count_<k>_sorted rows of all ranks, no contigs */
    uint64_t n_remote_probes;     /* neighbour requests of peers this rank answered from its index (last rfx_assemble_sharded
                                     or rfx_sort_kmers_sharded) */
    uint64_t n_l1_splitters, n_l2_splitters;
    float ms_comm;                /* barriers + value exchanges of the last sharded calls */
    int32_t fell_back;            /* last rfx_assemble_sharded met a closed path: rank 0 assembled the whole table */
} rfx_shard_stats_t;
/* Arena size: rfx_shard_table needs about twice its share of the table in the arena
 * (send buffer + new table, 2 * (8 or 16 + 4) bytes a row), plus the loaded slice when the new table outgrows it.
 * rfx_sort_kmers_sharded needs, besides the shard table, about 106 bytes per own row (two oriented k-mers of 37 bytes:
 * flags, alive byte, output flags, work list; 32 bytes of minima and index) plus the request / answer channels, world *
 * (global rows / world + 65536) * (32 or 48) bytes, plus the replicated presence bits, 2 bytes per global row (8 at least
 * per bin). */
int rfx_shard_init(rfx_ctx* ctx, int32_t rank, int32_t world, uint64_t arena_bytes /* 0: half of the free device memory */);
int rfx_shard_export(rfx_ctx* ctx, void* handle /* RFX_SHARD_HANDLE_BYTES */);
int rfx_shard_connect(rfx_ctx* ctx, const void* handles /* world * RFX_SHARD_HANDLE_BYTES, rank order */, int32_t world);
/* optional: the total number of minimiser bins (a multiple of world, same on every rank; rfx_choose_bins).  Known up
 * front it lets rfx_push_fastq scan each uploaded chunk straight into the slabs; otherwise the ranks agree on it. */
int rfx_shard_set_bins(rfx_ctx* ctx, uint32_t n_bins_total);
/* Collective counting from the pushed reads.  A rank whose reads put most records into a few bins (poly-A / poly-G,
 * microsatellites) scans them a second time with an overflow list of the size the first scan counted.  If its arena cannot
 * hold that list, EVERY rank returns RFX_E_CAPACITY at once (raise arena_bytes in rfx_shard_init); any other failure of one
 * rank's partition or count is likewise returned by every rank, with that rank's code.  The contexts stay usable. */
int rfx_count_sharded(rfx_ctx* ctx);
/* Collective re-shard of a loaded table: every rank holds a slice loaded with rfx_load_counts / rfx_load_counts_device
 * (slices may be empty and uneven); on return every rank holds exactly the rows whose minimiser bin it owns, as after
 * rfx_count_sharded.  Rows are neither merged nor de-duplicated, their order inside a shard is unspecified.  The bin
 * count B is the one of rfx_shard_set_bins if the caller set one (the same on every rank), else
 * rfx_choose_bins(ctx, 64 * global rows, world) -- what counting from reads picks at typical coverage, ~100 rows a bin.
 * A rank without a table, a different k or a B that is no multiple of world makes EVERY rank fail with the same error
 * (RFX_E_STATE / RFX_E_INVALID) after the first exchange.  rfx_stats: ms_partition is the call's time. */
int rfx_shard_table(rfx_ctx* ctx);
int rfx_assemble_sharded(rfx_ctx* ctx);
/* Collective Count_<k>_sorted on a table sharded by minimiser bin (after rfx_count_sharded or rfx_shard_table): the same
 * arguments, domain and results as rfx_sort_kmers.  On return every rank holds the sorted rows of its own shard
 * (rfx_sorted_size / rfx_sorted_copy / rfx_sorted_csv); their union over the ranks equals, bit for bit, what rfx_sort_kmers
 * gives on one context holding the whole table.  Like rfx_sort_kmers it takes the index and the flag arrays over: the
 * contigs of an earlier rfx_assemble_sharded are gone (RFX_E_STATE), a later rfx_assemble_sharded rebuilds them.  The ranks
 * agree on their arguments before any barrier, so a misuse makes EVERY rank fail with the same error at once: arguments
 * that differ between ranks RFX_E_INVALID, a rank without a sharded table RFX_E_STATE, min_error_coverage == 0 or
 * (k-1) % 31 == 0 RFX_E_UNSUPPORTED, more than 2^28 rows on a rank RFX_E_CAPACITY.  rfx_stats: ms_graph is the call's time;
 * rfx_shard_stats: ms_comm and n_remote_probes cover the call. */
int rfx_sort_kmers_sharded(rfx_ctx* ctx, int32_t min_error_coverage, double min_repeat_fold, int32_t max_kmer_size);
int rfx_shard_stats(rfx_ctx* ctx, rfx_shard_stats_t* out);

/* number of CUDA devices the library can use (a launcher maps ranks to devices with it) */
int rfx_device_count(int32_t* n_devices);

const char* rfx_version(void);

#ifdef __cplusplus
}
#endif
#endif /* REFLEXIV_CUDA_H */
