// rfx_api.cu -- the C ABI of libreflexiv_cuda (include/reflexiv_cuda.h): context life cycle,
// host <-> device copies, result layout conversion.  No compute lives here except small formatting
// kernels (CSV rows, oriented k-mer export).
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "rfx_internal.h"
#include "rfx_scan.cuh"
#include "rfx_shard.h"

namespace rfx {

static thread_local std::string g_create_error;

int ctx_fail(Ctx* c, int code, const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (c) c->err = buf;
    else g_create_error = buf;
    return code;
}

int devbuf_reserve(Ctx* c, DevBuf& b, size_t bytes, bool keep) {
    if (bytes <= b.cap) return RFX_OK;
    size_t want = bytes;
    if (keep && b.cap) want = bytes > b.cap * 2 ? bytes : b.cap * 2;  // appended buffers grow geometrically
    want = (want + 255) & ~(size_t)255;
    if (c && c->arena) {
        // sharded run: bump allocation inside the peer-visible arena.  No cudaMalloc / cudaFree while other ranks may sit in
        // a cross-GPU barrier (both can synchronise the whole device); an outgrown block is only given up, the arena
        // is sized for the run (rfx_shard_init).
        if (!keep || !b.cap) want += want / 8;  // head room, so that slightly different sizes from step to step do not move the block
        want = (want + 255) & ~(size_t)255;
        if (c->arena_used + want > c->arena_bytes)
            return ctx_fail(c, RFX_E_NOMEM, "peer-visible arena exhausted (%llu of %llu bytes used, %zu more needed): raise arena_bytes in rfx_shard_init",
                            (unsigned long long)c->arena_used, (unsigned long long)c->arena_bytes, want);
        void* p = c->arena + c->arena_used;
        c->arena_used += want;
        if (b.p && keep && b.cap) cudaMemcpyAsync(p, b.p, b.cap, cudaMemcpyDeviceToDevice, c->stream);
        if (b.p && !b.in_arena) { if (c->stream) cudaStreamSynchronize(c->stream); cudaFree(b.p); }
        b.p = p;
        b.cap = want;
        b.in_arena = true;
        return RFX_OK;
    }
    if (b.p && !(keep && b.cap)) {
        // contents are not needed: give the old block back first, so that growing a 45 GB buffer by 2 % does not need 90 GB
        if (c && c->stream) cudaStreamSynchronize(c->stream);
        cudaFree(b.p);
        b.p = nullptr;
        b.cap = 0;
    }
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return ctx_fail(c, RFX_E_NOMEM, "cudaMalloc(%zu bytes) failed: %s", want, cudaGetErrorString(e));
    }
    if (b.p) {
        if (c && c->stream) cudaStreamSynchronize(c->stream);
        cudaMemcpy(p, b.p, b.cap, cudaMemcpyDeviceToDevice);
        cudaFree(b.p);
    }
    b.p = p;
    b.cap = want;
    return RFX_OK;
}

void devbuf_free(DevBuf& b) {
    if (b.p && !b.in_arena) cudaFree(b.p);
    b.in_arena = false;
    b.p = nullptr;
    b.cap = 0;
}

void free_all_buffers(Ctx* c) {
    DevBuf* all[] = {&c->text, &c->line_start, &c->line_at, &c->nl_masks, &c->seq_flag, &c->scan_ws, &c->rd_len, &c->rd_woff, &c->packed, &c->bin_off, &c->bin_cursor,
                     &c->records, &c->keys, &c->counts, &c->dstat, &c->ht, &c->rflag, &c->lflag, &c->alive, &c->succ, &c->pred, &c->ad[0],
                     &c->ad[1], &c->rd_src, &c->spl_id, &c->spl_node, &c->loc, &c->sp_ad[0], &c->sp_ad[1], &c->cmin[0], &c->cmin[1], &c->spl_tail, &c->spl_chain, &c->chain_len, &c->ctg_idx, &c->ctg_off,
                     &c->ctg_left, &c->ctg_right, &c->ctg_bases, &c->rx_records, &c->run_desc, &c->rd_runs, &c->seg_off, &c->seg_base, &c->ovf_rec, &c->ovf_bin, &c->g_rowbin, &c->g_binrows, &c->g_hoff, &c->g_bloom, &c->srt_left, &c->srt_right, &c->eff_l, &c->eff_r, &c->seg_ext,
                     &c->st_keys, &c->st_vals, &c->st_bloom, &c->st_firstk, &c->st_ctr, &c->st_len, &c->st_woff, &c->st_hits, &c->st_frags, &c->st_codes, &c->st_nxt, &c->st_prv,
                     &c->st_role, &c->st_outlen, &c->st_outright, &c->st_slot, &c->sh_send};
    for (DevBuf* b : all) devbuf_free(*b);
}

// ---- CSV rows: "KMER,count\n" (DSBinaryKmerToString + write().csv, ReflexivDataFrameCounter.java:405-428, 222-233)
__device__ __forceinline__ uint32_t dec_digits(uint32_t v) {
    uint32_t d = 1;
    while (v >= 10) { v /= 10; d++; }
    return d;
}
struct CsvIn {
    const uint32_t* counts;
    int k;
    __device__ __forceinline__ uint64_t operator()(uint64_t i) const { return (uint64_t)k + 2 + dec_digits(counts[i]); }
};
template <class KT> struct CsvOut {
    const KT* keys;
    const uint32_t* counts;
    int k;
    char* out;
    __device__ __forceinline__ void operator()(uint64_t i, uint64_t excl, uint64_t len) const {
        char* p = out + excl;
        const KT key = keys[i];
        for (int j = 0; j < k; j++) p[j] = "ACGT"[(uint32_t)(key >> (2 * (k - 1 - j))) & 3u];
        p[k] = ',';
        uint32_t v = counts[i];
        for (int j = (int)len - 2; j > k; j--) { p[j] = (char)('0' + v % 10); v /= 10; }
        p[len - 1] = '\n';
    }
};

// ---- oriented k-mer export ----
struct AliveIn {
    const uint8_t* alive;
    __device__ __forceinline__ uint64_t operator()(uint64_t x) const { return (alive[x] & 2) ? 1 : 0; }
};
template <class KT> struct OrientedOut {
    const KT* keys;
    int k;
    const int32_t* lflag;
    const int32_t* rflag;
    uint64_t* hi;
    uint64_t* lo;
    int32_t* left;
    int32_t* right;
    __device__ __forceinline__ void operator()(uint64_t x, uint64_t excl, uint64_t v) const {
        if (!v) return;
        KT key = keys[x >> 1];
        if (x & 1) key = revcomp(key, k);
        const u128 wide = (u128)key;
        hi[excl] = (uint64_t)(wide >> 64);
        lo[excl] = (uint64_t)wide;
        left[excl] = lflag[x];
        right[excl] = rflag[x];
    }
};

// ---- Count_<k>_sorted rows: "KMER,1|left|right\n" (DSBinaryFullKmerArrayToString, ReflexivDSKmerLeftAndRightSorting.java:249-274;
// DSSubKmerToFullKmer sets every marker to 1, :1323) ----
__device__ __forceinline__ uint32_t dec_width(int32_t v) { return v < 0 ? 1u + dec_digits((uint32_t)(-(int64_t)v)) : dec_digits((uint32_t)v); }
__device__ __forceinline__ char* put_dec(char* p, int32_t v) {
    if (v < 0) *p++ = '-';
    uint32_t u = v < 0 ? (uint32_t)(-(int64_t)v) : (uint32_t)v;
    const uint32_t d = dec_digits(u);
    for (int j = (int)d - 1; j >= 0; j--) { p[j] = (char)('0' + u % 10); u /= 10; }
    return p + d;
}
struct SortedCsvIn {
    const uint8_t* alive;
    const int32_t* left;
    const int32_t* right;
    int k;
    __device__ __forceinline__ uint64_t operator()(uint64_t x) const {
        return (alive[x] & 2) ? (uint64_t)k + 3 + dec_width(left[x]) + 1 + dec_width(right[x]) + 1 : 0;
    }
};
template <class KT> struct SortedCsvOut {
    const KT* keys;
    const int32_t* left;
    const int32_t* right;
    int k;
    char* out;
    __device__ __forceinline__ void operator()(uint64_t x, uint64_t excl, uint64_t len) const {
        if (!len) return;
        char* p = out + excl;
        KT key = keys[x >> 1];
        if (x & 1) key = revcomp(key, k);
        for (int j = 0; j < k; j++) p[j] = "ACGT"[(uint32_t)(key >> (2 * (k - 1 - j))) & 3u];
        p += k;
        *p++ = ','; *p++ = '1'; *p++ = '|';
        p = put_dec(p, left[x]);
        *p++ = '|';
        p = put_dec(p, right[x]);
        *p = '\n';
    }
};

static int derive(Ctx* c) {
    const rfx_params& p = c->prm;
    if (p.kmer_size < 1 || p.kmer_size > 63) return ctx_fail(c, RFX_E_INVALID, "kmer_size %d outside 1..63", p.kmer_size);
    if (p.front_clip < 0 || p.end_clip < 0) return ctx_fail(c, RFX_E_INVALID, "negative clip");
    c->k = p.kmer_size;
    c->wide = c->k > 31;
    c->recw = rec_words_for_k(c->k);
    c->max_nk = (uint32_t)rec_max_kmers(c->recw, c->k);
    int m = p.minimizer_len > 0 ? p.minimizer_len : 11;
    if (m > 16) m = 16;
    if (m > c->k) m = c->k;
    c->m = m;
    return RFX_OK;
}

}  // namespace rfx

using namespace rfx;

extern "C" {

const char* rfx_version(void) { return "reflexiv_cuda 0.1 (sm_100a)"; }

int rfx_params_default(rfx_params* p) {
    if (!p) return RFX_E_INVALID;
    memset(p, 0, sizeof(*p));
    p->struct_size = (int32_t)sizeof(rfx_params);
    p->kmer_size = 31;            // DefaultParam.java:78
    p->min_kmer_coverage = 2;     // :104
    p->max_kmer_coverage = 10000000;  // :105
    p->min_error_coverage = 8;    // :106 (4 * minKmerCoverage at construction)
    p->min_contig = 500;          // :108
    p->bubble = 1;                // :109
    p->min_iter = 15;             // :116
    p->max_iter = 150;            // :115
    p->partitions = 0;            // :114
    p->shuffle_partitions = 200;  // :123
    p->fastq_mode = RFX_FASTQ_RUN;
    return RFX_OK;
}

int rfx_create(rfx_ctx** out, const rfx_params* p) {
    if (!out || !p) return ctx_fail(nullptr, RFX_E_INVALID, "rfx_create: null argument");
    if (p->struct_size != (int32_t)sizeof(rfx_params)) return ctx_fail(nullptr, RFX_E_INVALID, "rfx_create: rfx_params size mismatch");
    rfx_ctx* c = new rfx_ctx();
    c->prm = *p;
    int rc = derive(c);
    if (rc != RFX_OK) { g_create_error = c->err; delete c; return rc; }
    cudaError_t e = cudaSetDevice(p->device);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreate(&c->ev0);
    if (e == cudaSuccess) e = cudaEventCreate(&c->ev1);
    for (int i = 0; i < 6 && e == cudaSuccess; i++) e = cudaEventCreate(&c->evk[i]);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking);
    for (int i = 0; i < 2 && e == cudaSuccess; i++) e = cudaEventCreateWithFlags(&c->copy_done[i], cudaEventDisableTiming);
    if (e != cudaSuccess) {
        // no CPU fallback: without a usable CUDA device the library refuses to create a context
        rc = ctx_fail(nullptr, RFX_E_CUDA, "rfx_create: CUDA device %d unusable: %s", p->device, cudaGetErrorString(e));
        delete c;
        return rc;
    }
    rc = devbuf_reserve(c, c->dstat, DS_NSLOTS * sizeof(uint64_t));
    if (rc != RFX_OK) { g_create_error = c->err; rfx_destroy(c); return rc; }
    *out = c;
    return RFX_OK;
}

void rfx_destroy(rfx_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->prm.device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    free_all_buffers(c);
    shard_release(c);
    if (c->ev0) cudaEventDestroy(c->ev0);
    if (c->ev1) cudaEventDestroy(c->ev1);
    for (int i = 0; i < 6; i++) if (c->evk[i]) cudaEventDestroy(c->evk[i]);
    for (int i = 0; i < 2; i++) if (c->copy_done[i]) cudaEventDestroy(c->copy_done[i]);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

const char* rfx_last_error(const rfx_ctx* c) { return c ? c->err.c_str() : g_create_error.c_str(); }

int rfx_reset(rfx_ctx* c) {
    if (!c) return RFX_E_INVALID;
    if (c->arena) {
        // Sharded runs: buffers are bump-allocated in the peer-visible arena and nothing of a finished run is needed any more
        // (every sharded call ends behind a cross-rank barrier, so no peer still reads them): hand the whole arena back, the
        // next run lays its buffers out afresh.  Without this a context that is fed data sets of growing size would creep
        // through its arena, since an outgrown block is only given up, never reused.
        cudaSetDevice(c->prm.device);
        if (c->stream) cudaStreamSynchronize(c->stream);
        DevBuf keep = c->dstat;
        c->dstat = DevBuf();
        free_all_buffers(c);
        c->dstat = keep;
        shard_graph_reset(c);
        c->arena_used = c->arena_base;
    }
    c->n_reads = c->n_words = c->n_bases = c->n_instances = 0;
    c->n_records = 0; c->n_bins = 0; c->have_records = false; c->slab_cap = 0; c->n_ovf = 0; c->sp_active = false;
    c->n_rows = c->n_distinct = c->n_bin_splits = 0; c->have_counts = false;
    c->have_contigs = false; c->have_sorted = false; c->st_active = false;
    c->rx_bytes = 0; c->shard_id = -1; c->n_seg = 0;
    for (float& m : c->ms) m = 0;
    return RFX_OK;
}

int rfx_push_fastq_device(rfx_ctx* c, const uint8_t* d_buf, size_t len) {
    if (!c || (!d_buf && len)) return RFX_E_INVALID;
    cudaSetDevice(c->prm.device);
    if (c->st_active) return stage_parse_fastq(c, d_buf, len, true, false);  // reads of the stitch stage: scanned, nothing is kept
    c->have_records = false; c->have_counts = false; c->have_contigs = false; c->have_sorted = false; c->sp_active = false;
    return stage_parse_fastq(c, d_buf, len, true, false);
}

// Host text is uploaded in chunks of whole lines on a copy stream while the compute stream parses and encodes the
// previous chunk (PCIe is the bound of the end-to-end path: 1 GB of FASTQ per 3 M reads).  The FASTQ state machine's
// lineMark is carried from chunk to chunk on the device, so chunking never changes which lines are reads.
int rfx_push_fastq(rfx_ctx* c, const uint8_t* buf, size_t len) {
    if (!c || (!buf && len)) return RFX_E_INVALID;
    if (len == 0) return RFX_OK;
    cudaSetDevice(c->prm.device);
    if (!c->st_active) { c->have_records = false; c->have_counts = false; c->have_contigs = false; c->have_sorted = false; }
    RFX_TRY(devbuf_reserve(c, c->text, len + 128));
    uint8_t* d_text = c->text.as<uint8_t>();
    // chunk boundaries: just behind a newline; the last chunk keeps at least two lines
    size_t target = (size_t)96 << 20;
    if (const char* e = getenv("RFX_FASTQ_CHUNK_BYTES")) { const long long v = atoll(e); if (v >= 64) target = (size_t)v; }  // tests force many chunks
    std::vector<size_t> cuts;
    cuts.push_back(0);
    size_t last_ok = len;
    {   // position just behind the third-last newline: no earlier chunk may end after it
        size_t p = len, seen = 0;
        while (p > 0 && seen < 3) { p--; if (buf[p] == '\n') seen++; }
        last_ok = seen == 3 ? p + 1 : 0;
    }
    while (len - cuts.back() > target + target / 2) {
        size_t want = cuts.back() + target;
        if (want > last_ok) break;
        const void* nl = memchr(buf + want, '\n', last_ok > want ? last_ok - want : 0);
        if (!nl) break;
        const size_t cut = (size_t)((const uint8_t*)nl - buf) + 1;
        if (cut > last_ok || cut <= cuts.back()) break;
        cuts.push_back(cut);
    }
    cuts.push_back(len);
    const size_t n_chunks = cuts.size() - 1;
    // With several chunks and nothing pushed before, the single-GPU partition follows the upload: bin geometry from the
    // first chunk scaled to the whole text, every chunk's reads scanned while the next chunk is still on the bus.
    // (A later rfx_partition -- sharded runs -- or another push simply discards that work.)
    const char* sp_env = getenv("RFX_STREAM_PARTITION");
    bool stream_part = n_chunks >= 2 && c->n_reads == 0 && !c->st_active && !(sp_env && !strcmp(sp_env, "0"));
    c->sp_active = false;
    // every error path waits for the copy stream: the next chunk's upload may still be reading the caller's buffer,
    // and the header promises that host buffers are not touched after the call returns
    auto body = [&]() -> int {
        RFX_CUDA(c, cudaMemsetAsync(d_text + len, 0, 128, c->copy_stream));
        RFX_CUDA(c, cudaMemcpyAsync(d_text, buf, cuts[1], cudaMemcpyHostToDevice, c->copy_stream));
        RFX_CUDA(c, cudaEventRecord(c->copy_done[0], c->copy_stream));
        for (size_t i = 0; i < n_chunks; i++) {
            if (i + 1 < n_chunks) {
                RFX_CUDA(c, cudaMemcpyAsync(d_text + cuts[i + 1], buf + cuts[i + 1], cuts[i + 2] - cuts[i + 1], cudaMemcpyHostToDevice, c->copy_stream));
                RFX_CUDA(c, cudaEventRecord(c->copy_done[(i + 1) & 1], c->copy_stream));
            }
            RFX_CUDA(c, cudaStreamWaitEvent(c->stream, c->copy_done[i & 1], 0));
            RFX_TRY(stage_parse_fastq(c, d_text + cuts[i], cuts[i + 1] - cuts[i], i == 0, i + 1 < n_chunks));
            if (stream_part) {
                if (i == 0) {
                    if (c->n_reads == 0) { stream_part = false; continue; }
                    const double scale = 1.02 * (double)len / (double)cuts[1];
                    RFX_TRY(stage_stream_partition_begin(c, (uint64_t)((double)c->n_instances * scale) + 1, (uint64_t)((double)c->n_reads * scale) + 1));
                }
                RFX_TRY(stage_stream_partition_scan(c));
            }
        }
        return RFX_OK;
    };
    const int rc = body();
    if (rc != RFX_OK) cudaStreamSynchronize(c->copy_stream);
    return rc;
}

int rfx_push_reads(rfx_ctx* c, const uint8_t* bases, const uint64_t* offsets, uint64_t n_reads) {
    if (!c || !offsets || (!bases && n_reads && offsets[n_reads])) return RFX_E_INVALID;
    cudaSetDevice(c->prm.device);
    if (!c->st_active) { c->have_records = false; c->have_counts = false; c->have_contigs = false; c->have_sorted = false; c->sp_active = false; }
    return stage_push_reads(c, bases, offsets, n_reads);
}

int rfx_partition(rfx_ctx* c, int32_t n_shards, uint32_t n_bins_total) {
    if (!c) return RFX_E_INVALID;
    cudaSetDevice(c->prm.device);
    c->forced_bins = n_bins_total;
    return stage_partition(c, n_shards);
}

uint32_t rfx_choose_bins(rfx_ctx* c, uint64_t global_instances, int32_t n_shards) {
    if (!c || n_shards < 1) return 0;
    return choose_bin_count(c, global_instances, n_shards);
}

int rfx_count(rfx_ctx* c) {
    if (!c) return RFX_E_INVALID;
    cudaSetDevice(c->prm.device);
    c->st_active = false;  // an open stitch stage is abandoned: its fragments refer to the contigs it was opened on
    if (c->shard_id >= 0 && c->n_seg > 0) RFX_TRY(stage_adopt_segments(c));
    else if (c->shard_id >= 0) RFX_TRY(stage_rebin(c));
    else if (!c->have_records) {
        // one GPU, records stay local: single-pass slab partition; inputs with very heavy bins fall back to two passes
        const char* e = getenv("RFX_PARTITION");
        const bool two_pass = e && !strcmp(e, "twopass");
        if (!two_pass) RFX_TRY(stage_partition_slab(c));
        if (two_pass || !c->have_records) RFX_TRY(stage_partition(c, 1));
    }
    return stage_count(c);
}

int rfx_counts_size(rfx_ctx* c, uint64_t* n_rows, int32_t* words_per_key) {
    if (!c) return RFX_E_INVALID;
    if (!c->have_counts) return ctx_fail(c, RFX_E_STATE, "no count table");
    if (n_rows) *n_rows = c->n_rows;
    if (words_per_key) *words_per_key = c->k <= 31 ? 1 : c->k / 32 + 1;
    return RFX_OK;
}

int rfx_counts_copy(rfx_ctx* c, uint64_t* keys, uint32_t* counts) {
    if (!c) return RFX_E_INVALID;
    if (!c->have_counts) return ctx_fail(c, RFX_E_STATE, "no count table");
    cudaSetDevice(c->prm.device);
    const uint64_t n = c->n_rows;
    if (n == 0) return RFX_OK;
    if (counts) RFX_CUDA(c, cudaMemcpyAsync(counts, c->counts.p, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
    if (keys) {
        if (!c->wide) {
            RFX_CUDA(c, cudaMemcpyAsync(keys, c->keys.p, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, c->stream));
        } else {
            // internal: one right-aligned 2k-bit integer.  reference (Counter64.java:417-440): k/32+1 words,
            // 32 bases per word, the last word holds k%32 bases right aligned.
            std::vector<u128> tmp(n);
            RFX_CUDA(c, cudaMemcpyAsync(tmp.data(), c->keys.p, n * sizeof(u128), cudaMemcpyDeviceToHost, c->stream));
            RFX_CUDA(c, cudaStreamSynchronize(c->stream));
            const int res = c->k - 32;
            const uint64_t resmask = res ? (uint64_t)(((u128)1 << (2 * res)) - 1) : 0;
            for (uint64_t i = 0; i < n; i++) {
                keys[2 * i] = (uint64_t)(tmp[i] >> (2 * res));
                keys[2 * i + 1] = (uint64_t)tmp[i] & resmask;
            }
        }
    }
    RFX_CUDA(c, cudaStreamSynchronize(c->stream));
    return RFX_OK;
}

int rfx_load_counts(rfx_ctx* c, const uint64_t* keys, const uint32_t* counts, uint64_t n_rows) {
    if (!c || (n_rows && (!keys || !counts))) return RFX_E_INVALID;
    cudaSetDevice(c->prm.device);
    c->st_active = false;
    const size_t ksz = c->wide ? sizeof(u128) : sizeof(uint64_t);
    RFX_TRY(devbuf_reserve(c, c->keys, (n_rows + 1) * ksz));
    RFX_TRY(devbuf_reserve(c, c->counts, (n_rows + 1) * sizeof(uint32_t)));
    if (n_rows) {
        if (!c->wide) {
            RFX_CUDA(c, cudaMemcpyAsync(c->keys.p, keys, n_rows * sizeof(uint64_t), cudaMemcpyHostToDevice, c->stream));
        } else {
            std::vector<u128> tmp(n_rows);
            const int res = c->k - 32;
            for (uint64_t i = 0; i < n_rows; i++) tmp[i] = ((u128)keys[2 * i] << (2 * res)) | keys[2 * i + 1];
            RFX_CUDA(c, cudaMemcpyAsync(c->keys.p, tmp.data(), n_rows * sizeof(u128), cudaMemcpyHostToDevice, c->stream));
            RFX_CUDA(c, cudaStreamSynchronize(c->stream));
        }
        RFX_CUDA(c, cudaMemcpyAsync(c->counts.p, counts, n_rows * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
    }
    RFX_CUDA(c, cudaStreamSynchronize(c->stream));
    c->n_rows = n_rows;
    c->table_cap = n_rows + 1;
    c->have_counts = true;
    c->have_contigs = false; c->have_sorted = false;
    return RFX_OK;
}

int rfx_counts_csv(rfx_ctx* c, char* out, uint64_t cap, uint64_t* n_bytes) {
    if (!c || !n_bytes) return RFX_E_INVALID;
    if (!c->have_counts) return ctx_fail(c, RFX_E_STATE, "no count table");
    cudaSetDevice(c->prm.device);
    cudaStream_t st = c->stream;
    const uint64_t n = c->n_rows;
    if (n == 0) { *n_bytes = 0; return RFX_OK; }
    ScanPlan<uint64_t> plan;
    RFX_TRY(devbuf_reserve(c, c->scan_ws, ScanPlan<uint64_t>::workspace_elems(n) * sizeof(uint64_t)));
    plan.bind(n, c->scan_ws.as<uint64_t>());
    CsvIn in{c->counts.as<uint32_t>(), c->k};
    scan_prepare(plan, in, OpAddU64{}, (uint64_t)0, st);
    c->launches += 2 * plan.levels;
    uint64_t total = 0;
    RFX_CUDA(c, cudaMemcpyAsync(&total, plan.total, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    RFX_CUDA(c, cudaStreamSynchronize(st));
    *n_bytes = total;
    if (!out) return RFX_OK;
    if (cap < total) return ctx_fail(c, RFX_E_INVALID, "rfx_counts_csv: buffer of %llu bytes, need %llu", (unsigned long long)cap, (unsigned long long)total);
    DevBuf txt;
    RFX_TRY(devbuf_reserve(c, txt, total + 16));
    if (!c->wide) scan_apply(plan, in, CsvOut<uint64_t>{c->keys.as<uint64_t>(), c->counts.as<uint32_t>(), c->k, txt.as<char>()}, OpAddU64{}, (uint64_t)0, st);
    else scan_apply(plan, in, CsvOut<u128>{c->keys.as<u128>(), c->counts.as<uint32_t>(), c->k, txt.as<char>()}, OpAddU64{}, (uint64_t)0, st);
    c->launches += 1;
    cudaError_t e = cudaMemcpyAsync(out, txt.p, total, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    devbuf_free(txt);
    if (e != cudaSuccess) return ctx_fail(c, RFX_E_CUDA, "rfx_counts_csv: %s", cudaGetErrorString(e));
    return RFX_OK;
}

int rfx_assemble(rfx_ctx* c) {
    if (!c) return RFX_E_INVALID;
    cudaSetDevice(c->prm.device);
    c->st_active = false;  // an open stitch stage is abandoned: its fragments refer to the contigs it was opened on
    return stage_graph(c);
}

int rfx_contigs_size(rfx_ctx* c, uint64_t* n_contigs, uint64_t* total_bases) {
    if (!c) return RFX_E_INVALID;
    if (!c->have_contigs) return ctx_fail(c, RFX_E_STATE, "no contigs (call rfx_assemble)");
    if (n_contigs) *n_contigs = c->n_contigs;
    if (total_bases) *total_bases = c->n_contig_bases;
    return RFX_OK;
}

int rfx_contigs_copy(rfx_ctx* c, char* bases, uint64_t* offsets, int32_t* left, int32_t* right) {
    if (!c) return RFX_E_INVALID;
    if (!c->have_contigs) return ctx_fail(c, RFX_E_STATE, "no contigs (call rfx_assemble)");
    cudaSetDevice(c->prm.device);
    cudaStream_t st = c->stream;
    const uint64_t n = c->n_contigs;
    if (offsets) RFX_CUDA(c, cudaMemcpyAsync(offsets, c->ctg_off.p, (n + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    if (n) {
        if (bases) RFX_CUDA(c, cudaMemcpyAsync(bases, c->ctg_bases.p, c->n_contig_bases, cudaMemcpyDeviceToHost, st));
        if (left) RFX_CUDA(c, cudaMemcpyAsync(left, c->ctg_left.p, n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        if (right) RFX_CUDA(c, cudaMemcpyAsync(right, c->ctg_right.p, n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    }
    RFX_CUDA(c, cudaStreamSynchronize(st));
    return RFX_OK;
}

int rfx_oriented_size(rfx_ctx* c, uint64_t* n) {
    if (!c || !n) return RFX_E_INVALID;
    if (!c->have_contigs) return ctx_fail(c, RFX_E_STATE, "no graph (call rfx_assemble)");
    *n = c->n_oriented;
    return RFX_OK;
}

// survivors (alive & 2) with their two flags, in oid order
static int copy_survivors(Ctx* c, const char* who, uint64_t m, const int32_t* d_lflag, const int32_t* d_rflag, uint64_t* keys_hi, uint64_t* keys_lo, int32_t* left,
                          int32_t* right) {
    cudaSetDevice(c->prm.device);
    cudaStream_t st = c->stream;
    const uint64_t n = 2 * c->n_rows;
    if (m == 0) return RFX_OK;
    ScanPlan<uint64_t> plan;
    RFX_TRY(devbuf_reserve(c, c->scan_ws, ScanPlan<uint64_t>::workspace_elems(n) * sizeof(uint64_t)));
    plan.bind(n, c->scan_ws.as<uint64_t>());
    AliveIn in{c->alive.as<uint8_t>()};
    scan_prepare(plan, in, OpAddU64{}, (uint64_t)0, st);
    DevBuf tmp;
    RFX_TRY(devbuf_reserve(c, tmp, m * 24 + 64));
    uint64_t* d_hi = tmp.as<uint64_t>();
    uint64_t* d_lo = d_hi + m;
    int32_t* d_l = reinterpret_cast<int32_t*>(d_lo + m);
    int32_t* d_r = d_l + m;
    if (!c->wide) scan_apply(plan, in, OrientedOut<uint64_t>{c->keys.as<uint64_t>(), c->k, d_lflag, d_rflag, d_hi, d_lo, d_l, d_r}, OpAddU64{}, (uint64_t)0, st);
    else scan_apply(plan, in, OrientedOut<u128>{c->keys.as<u128>(), c->k, d_lflag, d_rflag, d_hi, d_lo, d_l, d_r}, OpAddU64{}, (uint64_t)0, st);
    c->launches += 2 * plan.levels + 1;
    cudaMemcpyAsync(keys_hi, d_hi, m * 8, cudaMemcpyDeviceToHost, st);
    cudaMemcpyAsync(keys_lo, d_lo, m * 8, cudaMemcpyDeviceToHost, st);
    cudaMemcpyAsync(left, d_l, m * 4, cudaMemcpyDeviceToHost, st);
    cudaMemcpyAsync(right, d_r, m * 4, cudaMemcpyDeviceToHost, st);
    cudaError_t e = cudaStreamSynchronize(st);
    devbuf_free(tmp);
    if (e != cudaSuccess) return ctx_fail(c, RFX_E_CUDA, "%s: %s", who, cudaGetErrorString(e));
    return RFX_OK;
}

int rfx_oriented_copy(rfx_ctx* c, uint64_t* keys_hi, uint64_t* keys_lo, int32_t* left, int32_t* right) {
    if (!c || !keys_hi || !keys_lo || !left || !right) return RFX_E_INVALID;
    if (!c->have_contigs) return ctx_fail(c, RFX_E_STATE, "no graph (call rfx_assemble)");
    return copy_survivors(c, "rfx_oriented_copy", c->n_oriented, c->lflag.as<int32_t>(), c->rflag.as<int32_t>(), keys_hi, keys_lo, left, right);
}

// ---- Count_<k>_sorted (SURVEY 8f-2; ReflexivDSKmerLeftAndRightSorting.java:105-243) ----
int rfx_sort_kmers(rfx_ctx* c, int32_t min_error_coverage, double min_repeat_fold, int32_t max_kmer_size) {
    if (!c) return RFX_E_INVALID;
    cudaSetDevice(c->prm.device);
    c->st_active = false;  // an open stitch stage is abandoned: its fragments refer to the contigs it was opened on
    return stage_sorted(c, min_error_coverage, min_repeat_fold, max_kmer_size);
}

int rfx_sorted_size(rfx_ctx* c, uint64_t* n_rows) {
    if (!c || !n_rows) return RFX_E_INVALID;
    if (!c->have_sorted) return ctx_fail(c, RFX_E_STATE, "no sorted rows (call rfx_sort_kmers)");
    *n_rows = c->n_sorted;
    return RFX_OK;
}

int rfx_sorted_copy(rfx_ctx* c, uint64_t* keys_hi, uint64_t* keys_lo, int32_t* left, int32_t* right) {
    if (!c || !keys_hi || !keys_lo || !left || !right) return RFX_E_INVALID;
    if (!c->have_sorted) return ctx_fail(c, RFX_E_STATE, "no sorted rows (call rfx_sort_kmers)");
    return copy_survivors(c, "rfx_sorted_copy", c->n_sorted, c->srt_left.as<int32_t>(), c->srt_right.as<int32_t>(), keys_hi, keys_lo, left, right);
}

int rfx_sorted_csv(rfx_ctx* c, char* out, uint64_t cap, uint64_t* n_bytes) {
    if (!c || !n_bytes) return RFX_E_INVALID;
    if (!c->have_sorted) return ctx_fail(c, RFX_E_STATE, "no sorted rows (call rfx_sort_kmers)");
    cudaSetDevice(c->prm.device);
    cudaStream_t st = c->stream;
    const uint64_t n = 2 * c->n_rows;
    if (c->n_sorted == 0) { *n_bytes = 0; return RFX_OK; }
    ScanPlan<uint64_t> plan;
    RFX_TRY(devbuf_reserve(c, c->scan_ws, ScanPlan<uint64_t>::workspace_elems(n) * sizeof(uint64_t)));
    plan.bind(n, c->scan_ws.as<uint64_t>());
    SortedCsvIn in{c->alive.as<uint8_t>(), c->srt_left.as<int32_t>(), c->srt_right.as<int32_t>(), c->k};
    scan_prepare(plan, in, OpAddU64{}, (uint64_t)0, st);
    c->launches += 2 * plan.levels;
    uint64_t total = 0;
    RFX_CUDA(c, cudaMemcpyAsync(&total, plan.total, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    RFX_CUDA(c, cudaStreamSynchronize(st));
    *n_bytes = total;
    if (!out) return RFX_OK;
    if (cap < total) return ctx_fail(c, RFX_E_INVALID, "rfx_sorted_csv: buffer of %llu bytes, need %llu", (unsigned long long)cap, (unsigned long long)total);
    DevBuf txt;
    RFX_TRY(devbuf_reserve(c, txt, total + 16));
    if (!c->wide) scan_apply(plan, in, SortedCsvOut<uint64_t>{c->keys.as<uint64_t>(), c->srt_left.as<int32_t>(), c->srt_right.as<int32_t>(), c->k, txt.as<char>()}, OpAddU64{}, (uint64_t)0, st);
    else scan_apply(plan, in, SortedCsvOut<u128>{c->keys.as<u128>(), c->srt_left.as<int32_t>(), c->srt_right.as<int32_t>(), c->k, txt.as<char>()}, OpAddU64{}, (uint64_t)0, st);
    c->launches += 1;
    cudaError_t e = cudaMemcpyAsync(out, txt.p, total, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    devbuf_free(txt);
    if (e != cudaSuccess) return ctx_fail(c, RFX_E_CUDA, "rfx_sorted_csv: %s", cudaGetErrorString(e));
    return RFX_OK;
}

int rfx_stitch_begin(rfx_ctx* c) {
    if (!c) return RFX_E_INVALID;
    cudaSetDevice(c->prm.device);
    return stage_stitch_begin(c);
}

int rfx_stitch_finish(rfx_ctx* c) {
    if (!c) return RFX_E_INVALID;
    cudaSetDevice(c->prm.device);
    return stage_stitch_finish(c);
}

int rfx_stitch_stats(rfx_ctx* c, rfx_stitch_stats_t* out) {
    if (!c || !out) return RFX_E_INVALID;
    memset(out, 0, sizeof(*out));
    out->n_probes = c->st_stat[0];
    out->n_reads = c->st_reads;
    out->n_fragments = c->st_stat[1];
    out->n_after_pass1 = c->st_stat[2];
    out->n_joined = c->st_stat[3];
    out->n_stitched = c->st_stat[4];
    out->n_rings = c->st_stat[5];
    out->ms_stitch = c->ms_stitch;
    return RFX_OK;
}

int rfx_stats(rfx_ctx* c, rfx_stats_t* s) {
    if (!c || !s) return RFX_E_INVALID;
    memset(s, 0, sizeof(*s));
    s->n_reads = c->n_reads; s->n_bases = c->n_bases; s->n_instances = c->n_instances; s->n_distinct = c->n_distinct;
    s->n_rows = c->n_rows; s->n_records = c->n_records; s->n_bins = c->n_bins; s->n_bin_splits = c->n_bin_splits;
    s->n_oriented = c->n_oriented; s->n_budget_junctions = c->n_budget; s->n_budget_admissible = c->n_budget_adm;
    s->n_cycles = c->n_cycles; s->n_contigs = c->n_contigs; s->n_contig_bases = c->n_contig_bases;
    s->kernel_launches = c->launches;
    s->ms_parse = c->ms[0]; s->ms_partition = c->ms[1]; s->ms_count = c->ms[2];
    s->ms_graph = c->ms[3]; s->ms_extend = c->ms[4]; s->ms_contigs = c->ms[5];
    s->ms_kernel_bin_histogram = c->ms_kernel[0]; s->ms_kernel_bin_scatter = c->ms_kernel[1]; s->ms_kernel_count = c->ms_kernel[2];
    return RFX_OK;
}

// ---- sharded counting ---------------------------------------------------------------------------
int rfx_record_bytes(rfx_ctx* c, int32_t* bytes_per_record) {
    if (!c || !bytes_per_record) return RFX_E_INVALID;
    *bytes_per_record = c->recw * 8;
    return RFX_OK;
}

int rfx_shard_records(rfx_ctx* c, int32_t shard, const void** d_ptr, uint64_t* n_bytes) {
    if (!c || !d_ptr || !n_bytes) return RFX_E_INVALID;
    if (!c->have_records) return ctx_fail(c, RFX_E_STATE, "rfx_shard_records: call rfx_partition first");
    if (shard < 0 || shard >= c->n_shards) return ctx_fail(c, RFX_E_INVALID, "shard %d outside 0..%d", shard, c->n_shards - 1);
    cudaSetDevice(c->prm.device);
    const uint32_t bps = c->n_bins / (uint32_t)c->n_shards;
    uint64_t lo = 0, hi = 0;
    RFX_CUDA(c, cudaMemcpyAsync(&lo, c->bin_off.as<uint64_t>() + (uint64_t)shard * bps, 8, cudaMemcpyDeviceToHost, c->stream));
    RFX_CUDA(c, cudaMemcpyAsync(&hi, c->bin_off.as<uint64_t>() + (uint64_t)(shard + 1) * bps, 8, cudaMemcpyDeviceToHost, c->stream));
    RFX_CUDA(c, cudaStreamSynchronize(c->stream));
    *d_ptr = c->records.as<uint64_t>() + lo * c->recw;
    *n_bytes = (hi - lo) * c->recw * 8;
    return RFX_OK;
}

int rfx_begin_shard(rfx_ctx* c, int32_t shard_id, int32_t n_shards, uint32_t n_bins_total) {
    if (!c || n_shards < 1 || shard_id < 0 || shard_id >= n_shards || n_bins_total == 0 || n_bins_total % (uint32_t)n_shards)
        return c ? ctx_fail(c, RFX_E_INVALID, "rfx_begin_shard: bad shard geometry") : RFX_E_INVALID;
    c->shard_id = shard_id; c->n_shards = n_shards; c->forced_bins = n_bins_total;
    c->rx_bytes = 0; c->n_seg = 0;
    c->have_records = false; c->have_counts = false; c->have_contigs = false; c->have_sorted = false;
    return RFX_OK;
}

int rfx_load_records_device(rfx_ctx* c, const void* d_records, uint64_t n_bytes) {
    if (!c || (!d_records && n_bytes)) return RFX_E_INVALID;
    if (c->shard_id < 0) return ctx_fail(c, RFX_E_STATE, "rfx_load_records_device: call rfx_begin_shard first");
    if (n_bytes % (uint64_t)(c->recw * 8)) return ctx_fail(c, RFX_E_INVALID, "record bytes not a multiple of %d", c->recw * 8);
    cudaSetDevice(c->prm.device);
    RFX_TRY(devbuf_reserve(c, c->rx_records, c->rx_bytes + n_bytes + 16, true));
    if (n_bytes) RFX_CUDA(c, cudaMemcpyAsync(c->rx_records.as<uint8_t>() + c->rx_bytes, d_records, n_bytes, cudaMemcpyDeviceToDevice, c->stream));
    RFX_CUDA(c, cudaStreamSynchronize(c->stream));
    c->rx_bytes += n_bytes;
    return RFX_OK;
}

int rfx_rx_buffer(rfx_ctx* c, uint64_t n_bytes, void** d_ptr) {
    if (!c || !d_ptr) return RFX_E_INVALID;
    if (c->shard_id < 0) return ctx_fail(c, RFX_E_STATE, "rfx_rx_buffer: call rfx_begin_shard first");
    if (c->rx_bytes) return ctx_fail(c, RFX_E_STATE, "rfx_rx_buffer: segments were already loaded");
    cudaSetDevice(c->prm.device);
    RFX_TRY(devbuf_reserve(c, c->rx_records, n_bytes + 16));
    *d_ptr = c->rx_records.p;
    return RFX_OK;
}

int rfx_counts_device(rfx_ctx* c, const void** d_keys, const uint32_t** d_counts, uint64_t* n_rows, int32_t* key_bytes) {
    if (!c) return RFX_E_INVALID;
    if (!c->have_counts) return ctx_fail(c, RFX_E_STATE, "no count table");
    if (d_keys) *d_keys = c->keys.p;
    if (d_counts) *d_counts = c->counts.as<uint32_t>();
    if (n_rows) *n_rows = c->n_rows;
    if (key_bytes) *key_bytes = c->wide ? 16 : 8;
    return RFX_OK;
}

int rfx_load_counts_device(rfx_ctx* c, const void* d_keys, const uint32_t* d_counts, uint64_t n_rows, int32_t append) {
    if (!c || (n_rows && (!d_keys || !d_counts))) return RFX_E_INVALID;
    cudaSetDevice(c->prm.device);
    c->st_active = false;
    const size_t ksz = c->wide ? 16 : 8;
    const uint64_t base = (append && c->have_counts) ? c->n_rows : 0;
    RFX_TRY(devbuf_reserve(c, c->keys, (base + n_rows + 1) * ksz, base > 0));
    RFX_TRY(devbuf_reserve(c, c->counts, (base + n_rows + 1) * sizeof(uint32_t), base > 0));
    if (n_rows) {
        RFX_CUDA(c, cudaMemcpyAsync(c->keys.as<uint8_t>() + base * ksz, d_keys, n_rows * ksz, cudaMemcpyDeviceToDevice, c->stream));
        RFX_CUDA(c, cudaMemcpyAsync(c->counts.as<uint32_t>() + base, d_counts, n_rows * sizeof(uint32_t), cudaMemcpyDeviceToDevice, c->stream));
    }
    RFX_CUDA(c, cudaStreamSynchronize(c->stream));
    c->n_rows = base + n_rows;
    c->table_cap = c->n_rows + 1;
    c->have_counts = true;
    c->have_contigs = false; c->have_sorted = false;
    return RFX_OK;
}

int rfx_shard_bin_offsets(rfx_ctx* c, int32_t shard, const uint64_t** d_offsets, uint32_t* n_offsets) {
    if (!c || !d_offsets || !n_offsets) return RFX_E_INVALID;
    if (!c->have_records) return ctx_fail(c, RFX_E_STATE, "rfx_shard_bin_offsets: call rfx_partition first");
    if (shard < 0 || shard >= c->n_shards) return ctx_fail(c, RFX_E_INVALID, "shard %d outside 0..%d", shard, c->n_shards - 1);
    const uint32_t bps = c->n_bins / (uint32_t)c->n_shards;
    *d_offsets = c->bin_off.as<uint64_t>() + (uint64_t)shard * bps;
    *n_offsets = bps + 1;
    return RFX_OK;
}

int rfx_load_segment_device(rfx_ctx* c, const void* d_records, uint64_t n_bytes, const uint64_t* d_bin_offsets) {
    if (!c || (!d_records && n_bytes) || !d_bin_offsets) return RFX_E_INVALID;
    if (c->shard_id < 0) return ctx_fail(c, RFX_E_STATE, "rfx_load_segment_device: call rfx_begin_shard first");
    if (c->n_seg >= RFX_MAX_SEG) return ctx_fail(c, RFX_E_INVALID, "more than %d segments", RFX_MAX_SEG);
    if (c->n_seg == 0 && c->rx_bytes) return ctx_fail(c, RFX_E_STATE, "do not mix rfx_load_records_device and rfx_load_segment_device");
    if (n_bytes % (uint64_t)(c->recw * 8)) return ctx_fail(c, RFX_E_INVALID, "record bytes not a multiple of %d", c->recw * 8);
    cudaSetDevice(c->prm.device);
    const uint32_t bps = c->forced_bins / (uint32_t)c->n_shards;
    RFX_TRY(devbuf_reserve(c, c->rx_records, c->rx_bytes + n_bytes + 16, true));
    RFX_TRY(devbuf_reserve(c, c->seg_off, (size_t)(c->n_seg + 1) * (bps + 1) * sizeof(uint64_t), true));
    // a slice received straight into rfx_rx_buffer() memory is already where it belongs
    if (n_bytes && d_records != (const void*)(c->rx_records.as<uint8_t>() + c->rx_bytes))
        RFX_CUDA(c, cudaMemcpyAsync(c->rx_records.as<uint8_t>() + c->rx_bytes, d_records, n_bytes, cudaMemcpyDeviceToDevice, c->stream));
    RFX_CUDA(c, cudaMemcpyAsync(c->seg_off.as<uint64_t>() + (size_t)c->n_seg * (bps + 1), d_bin_offsets, (size_t)(bps + 1) * sizeof(uint64_t),
                                cudaMemcpyDeviceToDevice, c->stream));
    RFX_CUDA(c, cudaStreamSynchronize(c->stream));
    c->seg_base_host[c->n_seg] = c->rx_bytes / (uint64_t)(c->recw * 8);
    c->n_seg++;
    c->rx_bytes += n_bytes;
    return RFX_OK;
}

}  // extern "C"
