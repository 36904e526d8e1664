// rfx_testhooks.cu -- TEST-ONLY access to intermediate device state of a libreflexiv_cuda context (packed reads, super-k-mer
// records, which partition ran): copies to host.  Built as tests/hooks/librfx_testhooks.so from the library's internal header; not part of
// the product library or its ABI.
#include "../../reflexiv_b200/csrc/rfx_internal.h"

using namespace rfx;

int rfx::ctx_fail(Ctx* c, int code, const char* fmt, ...) { (void)fmt; if (c) c->err = "test hook failed"; return code; }

extern "C" {
int rfx_debug_reads(rfx_ctx* c, uint64_t* n_reads, uint64_t* total_words, uint32_t* lens, uint64_t* word_offsets, uint64_t* words) {
    if (!c) return RFX_E_INVALID;
    cudaSetDevice(c->prm.device);
    if (n_reads) *n_reads = c->n_reads;
    if (total_words) *total_words = c->n_words;
    if (lens && c->n_reads) RFX_CUDA(c, cudaMemcpy(lens, c->rd_len.p, c->n_reads * 4, cudaMemcpyDeviceToHost));
    if (word_offsets && c->n_reads) RFX_CUDA(c, cudaMemcpy(word_offsets, c->rd_woff.p, c->n_reads * 8, cudaMemcpyDeviceToHost));
    if (words && c->n_words) RFX_CUDA(c, cudaMemcpy(words, c->packed.p, c->n_words * 8, cudaMemcpyDeviceToHost));
    return RFX_OK;
}

int rfx_debug_records(rfx_ctx* c, uint64_t* n_records, uint32_t* n_bins, uint64_t* bin_offsets, uint64_t* records) {
    if (!c) return RFX_E_INVALID;
    if (!c->have_records) return ctx_fail(c, RFX_E_STATE, "no records");
    cudaSetDevice(c->prm.device);
    if (n_records) *n_records = c->n_records;
    if (n_bins) *n_bins = c->n_bins;
    if (bin_offsets) RFX_CUDA(c, cudaMemcpy(bin_offsets, c->bin_off.p, ((size_t)c->n_bins + 1) * 8, cudaMemcpyDeviceToHost));
    if (records && c->n_records) RFX_CUDA(c, cudaMemcpy(records, c->records.p, c->n_records * c->recw * 8, cudaMemcpyDeviceToHost));
    return RFX_OK;
}

// Which partition the last count ran on, read after the call returned (nothing is launched):
//   out[0] slab capacity (0: compact two-pass layout)   out[1] records that missed their slab (also those the list had no room for)
//   out[2] capacity of the overflow list                out[3] bins          out[4] records
//   out[5] dstat[DS_SPILL] (the two-pass scan left reads to the spill pass; cleared when counting starts)
//   out[6] arena bytes in use (sharded contexts)        out[7] arena offset of the overflow list's records, out[8] bytes of its two blocks
int rfx_debug_partition(rfx_ctx* c, uint64_t* out) {
    if (!c || !out) return RFX_E_INVALID;
    cudaSetDevice(c->prm.device);
    uint64_t spill = 0;
    RFX_CUDA(c, cudaStreamSynchronize(c->stream));
    if (c->dstat.p) RFX_CUDA(c, cudaMemcpy(&spill, c->dstat.as<uint64_t>() + DS_SPILL, sizeof(spill), cudaMemcpyDeviceToHost));
    out[0] = c->slab_cap; out[1] = c->n_ovf; out[2] = c->sp_ovf_cap; out[3] = c->n_bins; out[4] = c->n_records; out[5] = spill;
    out[6] = c->arena ? c->arena_used : 0;
    out[7] = c->arena && c->ovf_rec.p ? (uint64_t)(c->ovf_rec.as<uint8_t>() - c->arena) : 0;
    out[8] = c->ovf_rec.cap + c->ovf_bin.cap;
    return RFX_OK;
}

}
