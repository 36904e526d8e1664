// rfx_counts_csv.cu -- rfx_load_counts_csv: Count_<k> text (KmerBinarizer rows, ReflexivDSMain.java:3872-3948) parsed on the device
// into the context's count table.
//
// Host text is uploaded in chunks of whole lines into a ring of two staging slots on the copy stream while the compute stream parses
// the previous chunk, so the device memory the call needs besides the table grows with the chunk size, not with the text.  Per chunk:
//   text --newline masks + scan (rfx_newline.cuh, rfx_scan.cuh)--> newline positions --decode_count_rows_kernel--> key, count, keep flag
//   per line --order-preserving compaction (scan over the keep flags)--> appended to keys[] / counts[]
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "rfx_internal.h"
#include "rfx_scan.cuh"

#include "rfx_counts_csv.cuh"

namespace rfx {

struct CsvNewlineMaskIn {  // pass 1: the newlines of a 64-byte chunk, counted, the mask left behind
    TextView tv;
    uint64_t* masks;
    __device__ __forceinline__ uint64_t operator()(uint64_t chunk) const {
        const uint64_t m = newline_mask64(tv, chunk);
        masks[chunk] = m;
        return __popcll(m);
    }
};
struct CsvMaskCountIn {  // pass 2
    const uint64_t* masks;
    __device__ __forceinline__ uint64_t operator()(uint64_t chunk) const { return __popcll(masks[chunk]); }
};
struct CsvNewlineOut {
    const uint64_t* masks;
    uint64_t* nl_pos;  // position of the i-th newline
    __device__ __forceinline__ void operator()(uint64_t chunk, uint64_t excl, uint64_t v) const {
        if (!v) return;
        uint64_t m = masks[chunk];
        while (m) {
            nl_pos[excl++] = chunk * 64 + (uint64_t)lowest_bit(m);
            m &= m - 1;
        }
    }
};

// One thread per line: line i is [nl_pos[i - 1] + 1, nl_pos[i]), the last one ends at len when the text does not end with '\n'.
template <class KT>
__global__ void __launch_bounds__(256) decode_count_rows_kernel(const uint8_t* __restrict__ text, uint64_t len, const uint64_t* __restrict__ nl_pos, uint64_t n_nl,
                                                                uint64_t n_lines, int k, long long min_count, long long max_count, KT* __restrict__ row_key,
                                                                uint32_t* __restrict__ row_count, uint8_t* __restrict__ keep, unsigned long long* first_bad) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_lines; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t b = i ? nl_pos[i - 1] + 1 : 0, e = i < n_nl ? nl_pos[i] : len;
        const CsvRow r = decode_count_row(text, b, e, k);
        if (r.kind == CSV_BAD) atomicMin(first_bad, (unsigned long long)i);
        row_key[i] = (KT)r.key;
        row_count[i] = r.count;
        keep[i] = r.kind == CSV_ROW && (long long)r.count >= min_count && (long long)r.count <= max_count;  // ReflexivDSMain.java:405-412
    }
}

struct KeepIn {
    const uint8_t* keep;
    __device__ __forceinline__ uint64_t operator()(uint64_t i) const { return keep[i]; }
};
template <class KT> struct KeepOut {
    const KT* row_key;
    const uint32_t* row_count;
    KT* keys;  // the table behind its rows so far
    uint32_t* counts;
    __device__ __forceinline__ void operator()(uint64_t i, uint64_t excl, uint64_t v) const {
        if (!v) return;
        keys[excl] = row_key[i];
        counts[excl] = row_count[i];
    }
};

static unsigned csv_grid(uint64_t n) {
    const uint64_t g = (n + 255) / 256, cap = (uint64_t)sm_count() * 16;
    return (unsigned)(g < 1 ? 1 : g > cap ? cap : g);
}

// One chunk of whole lines at d_text (16-byte aligned), appended behind the c->n_rows rows of the table.  *lines_before: lines of the
// call in front of this chunk (for the error message), advanced by the chunk's lines.
template <class KT>
static int csv_chunk(Ctx* c, const uint8_t* d_text, size_t len, bool ends_with_newline, int64_t min_count, int64_t max_count, uint64_t* lines_before) {
    cudaStream_t st = c->stream;
    if (len == 0) return RFX_OK;
    TextView tv;
    tv.aligned = d_text;
    tv.delta = 0;
    tv.len = len;
    const uint64_t n_blocks = (len + 63) / 64;
    // 1. newline positions
    ScanPlan<uint64_t> nl;
    RFX_TRY(devbuf_reserve(c, c->scan_ws, ScanPlan<uint64_t>::workspace_elems(n_blocks) * sizeof(uint64_t)));
    RFX_TRY(devbuf_reserve(c, c->nl_masks, n_blocks * sizeof(uint64_t)));
    nl.bind(n_blocks, c->scan_ws.as<uint64_t>());
    uint64_t* masks = c->nl_masks.as<uint64_t>();
    scan_prepare(nl, CsvNewlineMaskIn{tv, masks}, OpAddU64{}, (uint64_t)0, st);
    c->launches += 2 * nl.levels;
    uint64_t n_nl = 0;
    RFX_CUDA(c, cudaMemcpyAsync(&n_nl, nl.total, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    RFX_CUDA(c, cudaStreamSynchronize(st));
    const uint64_t n_lines = n_nl + (ends_with_newline ? 0 : 1);
    RFX_TRY(devbuf_reserve(c, c->line_start, (n_nl + 1) * sizeof(uint64_t)));
    uint64_t* nl_pos = c->line_start.as<uint64_t>();
    scan_apply(nl, CsvMaskCountIn{masks}, CsvNewlineOut{masks, nl_pos}, OpAddU64{}, (uint64_t)0, st);
    c->launches += 1;
    // 2. every line decoded: key, count, keep flag; the first malformed line in DS_CSV_BAD
    const size_t key_bytes = (n_lines * sizeof(KT) + 255) & ~(size_t)255, count_bytes = (n_lines * sizeof(uint32_t) + 255) & ~(size_t)255;
    RFX_TRY(devbuf_reserve(c, c->csv_rows, key_bytes + count_bytes + n_lines));
    KT* row_key = c->csv_rows.as<KT>();
    uint32_t* row_count = reinterpret_cast<uint32_t*>(c->csv_rows.as<uint8_t>() + key_bytes);
    uint8_t* keep = c->csv_rows.as<uint8_t>() + key_bytes + count_bytes;
    unsigned long long* first_bad = c->dstat.as<unsigned long long>() + DS_CSV_BAD;
    RFX_CUDA(c, cudaMemsetAsync(first_bad, 0xff, sizeof(uint64_t), st));
    decode_count_rows_kernel<KT><<<csv_grid(n_lines), 256, 0, st>>>(d_text, len, nl_pos, n_nl, n_lines, c->k, (long long)min_count, (long long)max_count, row_key,
                                                                     row_count, keep, first_bad);
    c->launches += 1;
    // 3. kept rows appended in line order
    ScanPlan<uint64_t> kp;
    RFX_TRY(devbuf_reserve(c, c->scan_ws, ScanPlan<uint64_t>::workspace_elems(n_lines) * sizeof(uint64_t)));
    kp.bind(n_lines, c->scan_ws.as<uint64_t>());
    scan_prepare(kp, KeepIn{keep}, OpAddU64{}, (uint64_t)0, st);
    c->launches += 2 * kp.levels;
    uint64_t got[2] = {0, 0};  // kept rows, first malformed line
    RFX_CUDA(c, cudaMemcpyAsync(&got[0], kp.total, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    RFX_CUDA(c, cudaMemcpyAsync(&got[1], first_bad, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    RFX_CUDA(c, cudaStreamSynchronize(st));
    if (got[1] != ~0ull)
        return ctx_fail(c, RFX_E_INVALID, "rfx_load_counts_csv: line %llu: malformed k-mer count row (no ',' or fewer than %d characters in front of it)",
                        (unsigned long long)(*lines_before + got[1] + 1), c->k);
    *lines_before += n_lines;
    const uint64_t base = c->n_rows;
    if (got[0] == 0) return RFX_OK;
    RFX_TRY(devbuf_reserve(c, c->keys, (base + got[0] + 1) * sizeof(KT), base > 0));
    RFX_TRY(devbuf_reserve(c, c->counts, (base + got[0] + 1) * sizeof(uint32_t), base > 0));
    scan_apply(kp, KeepIn{keep}, KeepOut<KT>{row_key, row_count, c->keys.as<KT>() + base, c->counts.as<uint32_t>() + base}, OpAddU64{}, (uint64_t)0, st);
    c->launches += 1;
    c->n_rows = base + got[0];
    return RFX_OK;
}

int stage_load_counts_csv(Ctx* c, const uint8_t* buf, size_t len, int64_t min_count, int64_t max_count, bool append) {
    c->st_active = false;  // an open stitch stage is abandoned: its fragments refer to the contigs it was opened on
    c->have_contigs = false; c->have_sorted = false;
    if (!(append && c->have_counts)) c->n_rows = 0;
    c->have_counts = false;  // until the call succeeds: a failed call leaves no table
    // chunks of whole lines, each ending just behind a '\n' (the last one at the end of the text)
    size_t target = (size_t)16 << 20;
    if (const char* e = getenv("RFX_CSV_CHUNK_BYTES")) { const long long v = atoll(e); if (v >= 64) target = (size_t)v; }  // tests force many chunks
    std::vector<size_t> cuts(1, 0);
    while (len - cuts.back() > target) {
        const size_t want = cuts.back() + target;
        const void* nl = memchr(buf + want, '\n', len - want);
        if (!nl || (size_t)((const uint8_t*)nl - buf) + 1 >= len) break;
        cuts.push_back((size_t)((const uint8_t*)nl - buf) + 1);
    }
    cuts.push_back(len);
    const size_t n_chunks = cuts.size() - 1;
    size_t slot = 0;
    for (size_t i = 0; i < n_chunks; i++) slot = cuts[i + 1] - cuts[i] > slot ? cuts[i + 1] - cuts[i] : slot;
    slot = (slot + 64 + 255) & ~(size_t)255;  // the newline masks read whole 64-byte blocks, the row decoder whole 16-byte blocks
    RFX_TRY(devbuf_reserve(c, c->text, 2 * slot));
    uint8_t* ring = c->text.as<uint8_t>();
    const size_t ksz = c->wide ? sizeof(u128) : sizeof(uint64_t);
    stage_begin(c);
    // Slot s of the ring is refilled for chunk i + 1 only after the host has waited for chunk i - 1's decode (csv_chunk synchronises
    // before its scatter, which no longer reads the text).  Every error path waits for the copy stream: the next chunk's upload may
    // still be reading the caller's buffer.
    auto body = [&]() -> int {
        uint64_t lines = 0;
        if (len) {
            RFX_CUDA(c, cudaMemcpyAsync(ring, buf, cuts[1], cudaMemcpyHostToDevice, c->copy_stream));
            RFX_CUDA(c, cudaEventRecord(c->copy_done[0], c->copy_stream));
        }
        for (size_t i = 0; i < n_chunks && len; i++) {
            if (i + 1 < n_chunks) {
                RFX_CUDA(c, cudaMemcpyAsync(ring + ((i + 1) & 1) * slot, buf + cuts[i + 1], cuts[i + 2] - cuts[i + 1], cudaMemcpyHostToDevice, c->copy_stream));
                RFX_CUDA(c, cudaEventRecord(c->copy_done[(i + 1) & 1], c->copy_stream));
            }
            RFX_CUDA(c, cudaStreamWaitEvent(c->stream, c->copy_done[i & 1], 0));
            const size_t n = cuts[i + 1] - cuts[i];
            const bool nl_end = buf[cuts[i + 1] - 1] == '\n';
            if (c->wide) RFX_TRY(csv_chunk<u128>(c, ring + (i & 1) * slot, n, nl_end, min_count, max_count, &lines));
            else RFX_TRY(csv_chunk<uint64_t>(c, ring + (i & 1) * slot, n, nl_end, min_count, max_count, &lines));
        }
        RFX_TRY(devbuf_reserve(c, c->keys, (c->n_rows + 1) * ksz, true));
        RFX_TRY(devbuf_reserve(c, c->counts, (c->n_rows + 1) * sizeof(uint32_t), true));
        RFX_CUDA(c, cudaStreamSynchronize(c->stream));
        return RFX_OK;
    };
    const int rc = body();
    c->ms[0] += stage_end(c);
    if (rc != RFX_OK) {
        cudaStreamSynchronize(c->copy_stream);
        c->n_rows = 0;
        return rc;
    }
    c->table_cap = c->n_rows + 1;
    c->have_counts = true;
    return RFX_OK;
}

}  // namespace rfx

using namespace rfx;

extern "C" int rfx_load_counts_csv(rfx_ctx* c, const uint8_t* text, size_t len, int64_t min_count, int64_t max_count, int32_t append) {
    if (!c || (!text && len)) return RFX_E_INVALID;
    cudaSetDevice(c->prm.device);
    return stage_load_counts_csv(c, text, len, min_count, max_count, append != 0);
}
