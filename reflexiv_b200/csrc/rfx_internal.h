// rfx_internal.h -- context layout and host-side helpers shared by the .cu files of libreflexiv_cuda.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <string>

#include "../../include/reflexiv_cuda.h"
#include "rfx_core.h"

namespace rfx {

// growable device buffer; contents are NOT preserved on growth unless keep == true
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    bool in_arena = false;  // carved out of the context's peer-visible arena (sharded runs): never cudaFree'd on its own
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

struct Ctx;
int ctx_fail(Ctx* c, int code, const char* fmt, ...);
int devbuf_reserve(Ctx* c, DevBuf& b, size_t bytes, bool keep = false);
void devbuf_free(DevBuf& b);

#define RFX_CUDA(c, expr)                                                                          \
    do {                                                                                           \
        cudaError_t e_ = (expr);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return ctx_fail((c), RFX_E_CUDA, "%s failed at %s:%d: %s", #expr, __FILE__, __LINE__, \
                            cudaGetErrorString(e_));                                               \
    } while (0)
#define RFX_TRY(expr)                 \
    do {                              \
        int rc_ = (expr);             \
        if (rc_ != RFX_OK) return rc_; \
    } while (0)

// ---- record segments of the counting kernel ----
// One entry per (segment, bin): where the bin's records inside that segment start (absolute address, possibly in a peer
// GPU's memory) and how many there are.  Built by build_ext_kernel from at most RFX_MAX_SEG segment descriptions.
#define RFX_MAX_SEG 16
#define RFX_MAX_RANKS 8
#define RFX_PUB_SLOTS 56
struct SegExt {
    unsigned long long addr;
    uint32_t cnt, pad;
};
struct ExtSrc {
    const uint64_t* rec;       // record array of the segment
    const uint32_t* slab_cnt;  // slab layout: records of bin b at rec[b * slab_cap ..], min(slab_cnt[b], slab_cap) of them
    const uint64_t* off;       // offset layout: records of bin b at rec[off[b] - off_sub .. off[b + 1] - off_sub)
    uint64_t off_sub;          // subtracted from the offsets (a received slice carries its sender's absolute offsets)
    uint32_t slab_cap;         // != 0: slab layout
    uint32_t bin_base;         // the segment's arrays are indexed by bin_base + (bin of the table)
};
struct ExtSrcs {
    ExtSrc s[RFX_MAX_SEG];
};

struct StageTimer {
    cudaEvent_t a = nullptr, b = nullptr;
};

struct Ctx {
    rfx_params prm;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;  // H2D of the next FASTQ chunk overlaps the parse of the current one
    cudaEvent_t copy_done[2] = {nullptr, nullptr};
    std::string err;
    uint64_t launches = 0;

    // derived
    int k = 31;
    bool wide = false;  // k > 31: 128-bit keys
    int recw = 2;       // 64-bit words per super-k-mer record
    int m = 13;         // minimiser length
    uint32_t max_nk = 26;

    // ---- reads (packed 2-bit) ----
    DevBuf text;        // staging for host FASTQ text
    DevBuf line_start;  // u64[n_lines + 1]
    DevBuf line_at;     // u8[n_lines + 1] line starts with '@'
    DevBuf nl_masks;    // ulonglong2[n_chunks] newline mask + newline-followed-by-'@' mask of every 64-byte chunk of the text
    DevBuf seq_flag;    // u32[n_lines]  NOT_A_READ, or the effective length of the read on that line
    DevBuf scan_ws;     // scan workspace
    DevBuf rd_src;      // u64[new reads] text offset of each read of the current push (scratch)
    DevBuf rd_len;      // u32[n_reads]   effective length (0 = contributes nothing)
    DevBuf rd_woff;     // u64[n_reads]   first word in `packed`
    DevBuf packed;      // u64[n_words + pad]
    uint64_t n_reads = 0, n_words = 0, n_bases = 0, n_instances = 0;

    // ---- super-k-mer records ----
    DevBuf bin_off;     // u64[n_bins + 1]
    DevBuf bin_cursor;  // u64[n_bins]
    DevBuf records;     // u64[n_records * recw]
    DevBuf run_desc;    // u32[slots][n_reads]  (bin << 8 | n_kmers) per run, read-interleaved
    DevBuf rd_runs;     // u32[n_reads] runs per read
    uint32_t n_bins = 0;
    int32_t n_shards = 1;
    uint64_t n_records = 0;
    bool have_records = false;
    // single-pass (slab) layout: bin b = records[b * slab_cap ..] (first min(count, slab_cap) records) + an exactly
    // partitioned overflow segment in rx_records; slab_cap == 0: compact two-pass layout described by bin_off
    uint32_t slab_cap = 0;
    uint64_t n_ovf = 0;
    // streamed slab partition (rfx_push_fastq): geometry fixed from the first chunk, reads scanned as they arrive
    bool sp_active = false;
    uint32_t sp_cap = 0;
    uint64_t sp_ovf_cap = 0, sp_done = 0;
    float sp_kernel_ms = 0;
    DevBuf ovf_rec, ovf_bin;
    uint32_t forced_bins = 0;  // total bin count imposed by the caller (sharded runs), 0 = choose
    // records received from other shards (rfx_begin_shard / rfx_load_records_device)
    DevBuf rx_records;
    uint64_t rx_bytes = 0;
    int32_t shard_id = -1;
    // per-sender segments (rfx_load_segment_device): record base in rx_records + the sender's bin offsets
    DevBuf seg_ext;       // SegExt[n_seg][n_bins]: what the counting kernel walks
    DevBuf seg_off;       // u64[n_seg][bps + 1]
    DevBuf seg_base;      // u64[n_seg]
    uint64_t seg_base_host[64];
    int32_t n_seg = 0;

    // ---- filtered count table ----
    DevBuf keys;        // KT[table_cap]  right-aligned canonical k-mers
    DevBuf counts;      // u32[table_cap]
    DevBuf dstat;       // u64[16] device-side counters
    uint64_t table_cap = 0, n_rows = 0, n_distinct = 0, n_bin_splits = 0, n_shard_instances = 0;
    int count_geometry = 0;           // 0: unknown (run the pilot), 1: small table, 2: large table -- survives rfx_reset
    uint32_t count_geometry_bins = 0; // bin count of the run the pilot looked at
    uint32_t bin_shrink = 1;          // 1, 2, 4: bins this much smaller than the default (a run that had to split > 1 % of its bins asks the next
                                      // run on this context for smaller ones: noisy reads) -- survives rfx_reset, not used by sharded runs
    bool have_counts = false;

    // ---- de Bruijn graph over oriented k-mers (id = 2*row + strand) ----
    DevBuf ht;          // u32[ht_cap] row index or 0xffffffff
    uint64_t ht_cap = 0;
    DevBuf g_rowbin, g_binrows, g_hoff, g_bloom;
    uint64_t g_bloom_mask = 0;  // bin-local index: bin of every row, rows per bin, region offsets
    uint32_t g_bins = 0;
    int g_m = 11;
    DevBuf rflag, lflag;  // i32[2*n_rows]
    DevBuf eff_l, eff_r;  // i32[2*n_rows] flags after the budget walks (only when a fork winner survived)
    DevBuf alive;         // u8[2*n_rows]  bit0: survives right filter, bit1: survives both
    DevBuf succ, pred;    // u32[2*n_rows]
    DevBuf ad[2];         // u64[2*n_rows] packed (ancestor, distance) for pointer jumping, double buffered
    DevBuf spl_id;        // u32[2*n_rows] splitter index of a node (NONE where it is not one: sharded runs only write that)
    DevBuf spl_node;      // u32[2*n_rows] node of a splitter
    DevBuf loc;           // u64[2*n_rows] (owning splitter, offset from it)
    DevBuf sp_ad[2];      // u64[2*n_rows] packed (ancestor, distance) over the splitter list
    DevBuf cmin[2];
    DevBuf spl_tail;      // u64[2*n_rows] per splitter: (last node, nodes) of a segment that ends its chain, ~0 for the others
    DevBuf spl_chain;     // u64[2*n_rows] per splitter: (right flag of the tail, chain length) at a chain's first splitter, 0 elsewhere
    DevBuf chain_len;     // u32[2*n_rows] at heads (sharded chain ranking)
    DevBuf ctg_idx;       // u32[2*n_rows] contig index or NONE: per splitter on one GPU, at heads in a sharded run
    DevBuf ctg_off;       // u64[n_contigs + 1]
    DevBuf ctg_left, ctg_right;  // i32[n_contigs]
    DevBuf ctg_bases;     // char[total]
    uint64_t n_oriented = 0, n_budget = 0, n_budget_adm = 0, n_cycles = 0, n_contigs = 0, n_contig_bases = 0;
    bool have_contigs = false;

    // ---- Count_<k>_sorted (rfx_sort_kmers): flags of the oriented k-mers that survive that stage's filters (alive & 2) ----
    DevBuf srt_left, srt_right;  // i32[2*n_rows]
    uint64_t n_sorted = 0;
    bool have_sorted = false;

    // ---- -stitch (rfx_stitch.cu): contig-end probes, fragments cut from the reads, chains over contigs ----
    bool st_active = false;      // between rfx_stitch_begin and rfx_stitch_finish: pushed reads are scanned, not stored
    DevBuf st_keys, st_vals;     // u64 / u32 [st_cap] open-addressing probe table: (k-1)-mer -> contig << 1 | direction
    DevBuf st_bloom;             // u32[2^19 / 32] Bloom filter over the probe keys (64 KB: answers from the L1)
    DevBuf st_firstk;            // u64[n_contigs] first k-mer of every contig (orders probes and opens rings)
    DevBuf st_ctr;               // u64[8] device counters
    DevBuf st_len, st_woff;      // read table of the chunk being scanned (scratch)
    DevBuf st_hits;              // fragments found in the chunk being scanned
    DevBuf st_frags, st_codes;   // all fragments so far: descriptors + 2-bit codes, one per byte
    DevBuf st_nxt, st_prv, st_role, st_outlen, st_outright, st_slot;
    uint64_t st_cap = 0, st_nfrag = 0, st_ncodes = 0, st_reads = 0;
    uint64_t st_stat[6] = {0, 0, 0, 0, 0, 0};  // probes, fragments, after pass 1, joined on both sides, stitched records, rings
    float ms_stitch = 0;

    // ---- sharded runs over peer memory (rfx_shard.cu): one context per GPU, every device buffer of the context lives in
    // ONE cudaMalloc'ed arena that the other ranks map (CUDA IPC between processes, plain pointers inside a process) ----
    int sh_rank = -1, sh_world = 0;
    uint8_t* arena = nullptr;
    uint64_t arena_bytes = 0, arena_used = 0, arena_base = 0;  // arena_base: behind the control block and the published-value staging
    uint8_t* peer_base[RFX_MAX_RANKS] = {nullptr};  // arena of every rank as seen from this device (own: arena)
    bool peer_ipc[RFX_MAX_RANKS] = {false};         // opened through cudaIpcOpenMemHandle
    unsigned long long sh_epoch = 0;                // barriers passed
    unsigned long long sh_epoch2 = 0;               // in-kernel barriers passed (ShardCtl::flags2)
    unsigned long long sh_exchanges = 0;            // value exchanges made (parity picks the published block)
    unsigned long long* d_pub = nullptr;            // device staging: everybody's published block, gathered by one kernel
    unsigned long long* h_pub = nullptr;            // pinned: own published values + everybody's after an exchange
    uint32_t sh_bins = 0;                           // total bin count of sharded counting (0: agreed on per run)
    uint32_t sh_bins_run = 0;                       // ... the one in force for the slab scan (rfx_partition.cu: slab_begin)
    uint64_t sh_inst_global = 0;                    // k-mer instances extracted by all ranks
    uint64_t sh_rows_global = 0;                    // rows of all shard tables (known to every rank after rfx_count_sharded / rfx_shard_table)
    DevBuf sh_send;                                 // rfx_shard_table: the loaded rows grouped by owner, pulled by the owners
    cudaEvent_t ev_comm[2] = {nullptr, nullptr};
    float ms_comm = 0;                              // cross-GPU barriers + value exchanges of the last sharded calls
    void* hbar = nullptr;                           // host-side barrier of ranks that share a device inside one process
    unsigned long long hbar_key = 0;
    struct GShard* gshard = nullptr;                // state of the sharded graph stages

    float ms[6] = {0, 0, 0, 0, 0, 0};
    float ms_kernel[3] = {0, 0, 0};  // histogram, scatter, count: last launch only
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    cudaEvent_t evk[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
};

// device-side counter slots in Ctx::dstat
enum {
    DS_OUT_CURSOR = 0,
    DS_DISTINCT = 1,
    DS_INSTANCES = 2,
    DS_OVERFLOW = 3,
    DS_SPLITS = 4,
    DS_BUDGET = 5,
    DS_BUDGET_ADM = 6,
    DS_GRAPH_ERR = 7,
    DS_CHANGED = 8,
    DS_CYCLE_NODES = 9,
    DS_CYCLES = 10,
    DS_ORIENTED = 11,
    DS_SPILL = 12,
    DS_NSPL = 13,
    DS_FQ_STATE = 14,  // lineMark carried between the chunks of one rfx_push_fastq call
    DS_TICKET = 15,    // next bin handed to a counting CTA
    DS_OVF_RECORDS = 20,
    DS_SCAN_TODO = 21,    // the register-resident scan left reads to the general kernel  // records that did not fit their slab (single-pass partition)
    DS_OVF_WHY = 16,   // 4 slots: why counting bins were split (table full, probe exhausted, tag collision, narrow probe exhausted)
    DS_FLAGGED = 23,      // surviving oriented k-mers with a non-negative flag (fork winners): budget walks needed
    DS_ABSORBED = 27,     // k-mers absorbed by budget walks
    DS_RANK_CUR = 22,     // which of the two (ancestor, distance) buffers holds the result of rank_all_kernel
    DS_RANK_FLAGS = 24,
    DS_READ_TOTALS = 28,  // 2 slots: bases kept and k-mer instances of the reads being appended   // 3 rotating 'something changed' flags of rank_all_kernel
    DS_XBAR_ERR = 30,     // a cross-GPU barrier timed out (rfx_shard.cu)
    DS_NL2 = 32,          // level-2 splitters of the sharded chain ranking (rfx_shard_graph.cuh)
    DS_REMOTE = 33,       // neighbour probes answered from a peer's index
    DS_SG_CYCLE = 34,
    DS_WORK = 35,         // 3 slots: nodes the first pass of a sharded K5 kernel put off (their probe goes to a peer)     // a closed path was seen
    DS_FQ_NLINES = 39,    // 4 slots read back together by rfx_fastq.cu: lines of the chunk, violations of the regular 4-line layout,
    DS_FQ_IRREGULAR = 40, //   position (mod 4) of the sequence lines, lineMark behind the chunk if the layout is regular
    DS_FQ_SEQPOS = 41,
    DS_FQ_NEXT = 42,
    DS_REACHED = 43,      // nodes the splitter walks stamped: all alive nodes unless some sit on a closed path without a splitter
    DS_NSLOTS = 48
};

static const uint32_t NONE32 = 0xffffffffu;

// SMs of the current device (148 on a B200), queried once per device: launch grids are sized in multiples of it
inline unsigned sm_count() {
    static int cached[64] = {0};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64) dev = 0;
    if (!cached[dev]) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n < 1) n = 148;
        cached[dev] = n;
    }
    return (unsigned)cached[dev];
}

// stage entry points (each in its own .cu)
int stage_parse_fastq(Ctx* c, const uint8_t* d_text, size_t len, bool first_chunk = true, bool more_follows = false);
int stage_push_reads(Ctx* c, const uint8_t* h_bases, const uint64_t* h_offsets, uint64_t n_reads);
int stage_partition(Ctx* c, int n_shards);
int stage_partition_slab(Ctx* c, uint64_t ovf_need = 0);
int stage_stream_partition_begin(Ctx* c, uint64_t est_instances, uint64_t est_reads);
int stage_stream_partition_scan(Ctx* c);
int stage_rebin(Ctx* c);
int stage_adopt_segments(Ctx* c);
int stage_count(Ctx* c);
int stage_count_segments(Ctx* c, const ExtSrcs& S, int n_seg, uint32_t n_bins, bool check_instances);
int stage_graph(Ctx* c);
int stage_sorted(Ctx* c, int min_error_coverage, double min_repeat_fold, int max_kmer_size);
int stage_stitch_begin(Ctx* c);
int stitch_scan_reads(Ctx* c, const uint8_t* d_text, const uint64_t* rd_src, const uint32_t* rd_len, uint64_t n_reads);
int stage_stitch_finish(Ctx* c);
uint32_t choose_bin_count(const Ctx* c, uint64_t instances, int n_shards);
void set_minimizer(Ctx* c, uint32_t n_bins_total);  // c->m from the TOTAL bin count (rfx_partition.cu)
int stage_count_sharded(Ctx* c);
int stage_shard_table(Ctx* c);
int stage_assemble_sharded(Ctx* c);
int stage_sorted_sharded(Ctx* c, int min_error_coverage, double min_repeat_fold, int max_kmer_size);
void shard_release(Ctx* c);

inline void stage_begin(Ctx* c) { cudaEventRecord(c->ev0, c->stream); }
inline float stage_end(Ctx* c) {
    float ms = 0;
    cudaEventRecord(c->ev1, c->stream);
    cudaEventSynchronize(c->ev1);
    cudaEventElapsedTime(&ms, c->ev0, c->ev1);
    return ms;
}

}  // namespace rfx

struct rfx_ctx : rfx::Ctx {};
