// rfx_stitch.cu -- `reflexiv run -stitch`: the low-coverage read rescue of ReflexivDSMain.java:585-672 (SURVEY 8f-4); for k > 31 the
// reference's own branch can never cut a read (see stage_stitch_begin) and the stage is the plain assembly.
//
//   reference (pipeline/ReflexivDSMain.java)                          here
//   DSLowCoverageSubKmerExtraction :1211-1268 + collect +            probe_first_kernel / probe_insert_kernel: an open-addressing
//     SubKmerProbRowToHash :109-118 + broadcast :596                   table of contig-end (k-1)-mers in HBM (it stays in the L2)
//   second spark.read().text + DSFastqFilterWithQual :601-606         the K1 line scan + state machine of rfx_fastq.cu, unclipped
//   DSLowCoverageReadDetection :1448-1612                             stitch_scan_kernel: one thread per (read, strand) rolls the
//                                                                       (k-1)-mer over the TEXT (the reverse strand goes through
//                                                                       complementary() as in the reference: 'N' stays 'N' -> 3)
//   reflexivKmerExtractionFromLowCoverageFragment :1541-1595          stitch_copy_kernel: fragment bases as 2-bit codes
//   DSFilterRepeatLowCoverageFragment x 2 :629-638, :922-1010         frag_pick_kernel (one fragment leaves a contig, one arrives)
//   union + sort + DSExtendReflexivKmerToArrayLoop loop :640-670      chains over CONTIGS: heads, rings, lengths, one gather
//   DSKmerToContig :743-771                                           the same keep rule, then the contig arrays are replaced
//
// Spark's arrival order decides four things in the reference; the order fixed here is the one oracle/stitch_oracle.c states
// (probe collisions, which fragment of a run stays, which of several fragments joins a contig, where a ring is opened).
#include <string.h>

#include "rfx_internal.h"
#include "rfx_scan.cuh"
#include "rfx_shard.h"
#include "rfx_stitch_kernels.cuh"

namespace rfx {

using namespace stitch;

namespace {

unsigned grid_for_n(uint64_t n, unsigned per_block = 256) {
    uint64_t g = (n + per_block - 1) / per_block;
    if (g < 1) g = 1;
    const uint64_t cap = (uint64_t)sm_count() * 16u;
    return (unsigned)(g > cap ? cap : g);
}

// device counters of the stitch stage (Ctx::st_ctr): [0] hits of the chunk, [1] codes of the chunk, [2] probes put, [3] keys in
// the table, [4] after pass 1, [5] joined on both sides, [6] stitched records, [7] rings
enum { SC_HITS = 0, SC_CODES = 1, SC_PUT = 2, SC_KEYS = 3, SC_PASS1 = 4, SC_BOTH = 5, SC_STITCHED = 6, SC_RINGS = 7, SC_N = 8 };

}  // namespace

int stage_stitch_begin(Ctx* c) {
    // k > 31 (ReflexivDSMain64.java:715-790): DSLowCoverageReadDetection rolls the read's (k-1)-mer into ONE Long and asks a
    // Hashtable<List<Long>, Integer> for it (:1562-1600 against SubKmerProbRowToHash :119-131) -- a Long never equals a List, so
    // no read is ever cut there and the branch leaves the contigs as they are.  Same here: the stage opens with an empty probe table.
    const bool no_probe_can_match = c->k > 31;
    if (c->arena) return ctx_fail(c, RFX_E_UNSUPPORTED, "rfx_stitch_begin runs on one GPU: a sharded context stitches with rfx_stitch_begin_sharded");
    if (!c->have_counts) return ctx_fail(c, RFX_E_STATE, "rfx_stitch_begin: no count table (call rfx_count or rfx_load_counts first)");
    // every record of the extension takes part, whatever its length (the minContig rule is applied to the stitched set)
    const int32_t min_contig = c->prm.min_contig;
    c->prm.min_contig = 0;
    const int rc = stage_graph(c);
    c->prm.min_contig = min_contig;
    RFX_TRY(rc);
    cudaStream_t st = c->stream;
    stage_begin(c);
    const uint64_t n = c->n_contigs;
    uint64_t cap = 1024;
    while (cap < 4 * n + 16) cap <<= 1;  // at most 2 probes per contig: load <= 0.5
    RFX_TRY(devbuf_reserve(c, c->st_keys, cap * sizeof(uint64_t)));
    RFX_TRY(devbuf_reserve(c, c->st_vals, cap * sizeof(uint32_t)));
    RFX_TRY(devbuf_reserve(c, c->st_firstk, (n + 1) * sizeof(uint64_t)));
    RFX_TRY(devbuf_reserve(c, c->st_ctr, SC_N * sizeof(uint64_t)));
    RFX_TRY(devbuf_reserve(c, c->st_bloom, ST_BLOOM_BITS / 8));
    RFX_CUDA(c, cudaMemsetAsync(c->st_bloom.p, 0, ST_BLOOM_BITS / 8, st));
    c->st_cap = cap;
    RFX_CUDA(c, cudaMemsetAsync(c->st_keys.p, 0xff, cap * sizeof(uint64_t), st));
    RFX_CUDA(c, cudaMemsetAsync(c->st_vals.p, 0xff, cap * sizeof(uint32_t), st));
    RFX_CUDA(c, cudaMemsetAsync(c->st_ctr.p, 0, SC_N * sizeof(uint64_t), st));
    unsigned long long* ctr = c->st_ctr.as<unsigned long long>();
    if (n && !no_probe_can_match) {
        probe_first_kernel<<<grid_for_n(n), 256, 0, st>>>(c->ctg_off.as<uint64_t>(), c->ctg_bases.as<char>(), n, c->k, c->st_firstk.as<uint64_t>());
        probe_insert_kernel<<<grid_for_n(n), 256, 0, st>>>(c->ctg_off.as<uint64_t>(), c->ctg_bases.as<char>(), c->ctg_left.as<int32_t>(), c->ctg_right.as<int32_t>(), n,
                                                          c->k, c->st_firstk.as<uint64_t>(), c->st_keys.as<uint64_t>(), c->st_vals.as<uint32_t>(), cap - 1, c->st_bloom.as<uint32_t>(), ctr + SC_PUT);
        count_keys_kernel<<<grid_for_n(cap), 256, 0, st>>>(c->st_keys.as<uint64_t>(), cap, ctr + SC_KEYS);
        c->launches += 3;
    }
    uint64_t h[SC_N];
    RFX_CUDA(c, cudaMemcpyAsync(h, c->st_ctr.p, sizeof(h), cudaMemcpyDeviceToHost, st));
    RFX_CUDA(c, cudaStreamSynchronize(st));
    c->ms_stitch = stage_end(c);
    c->st_stat[0] = h[SC_KEYS];
    for (int i = 1; i < 6; i++) c->st_stat[i] = 0;
    c->st_nfrag = 0; c->st_ncodes = 0; c->st_reads = 0;
    c->st_active = true;
    c->st_sharded = false;
    return RFX_OK;
}

// Called by the K1 read-table pass (rfx_fastq.cu) for the reads of one chunk of text while the stitch stage is open.
int stitch_scan_reads(Ctx* c, const uint8_t* d_text, const uint64_t* rd_src, const uint32_t* rd_len, uint64_t n_reads) {
    c->st_reads += n_reads;
    if (n_reads == 0 || c->st_stat[0] == 0) return RFX_OK;  // no probe: no read can be cut
    cudaStream_t st = c->stream;
    unsigned long long* ctr = c->st_ctr.as<unsigned long long>();
    uint64_t hit_cap = c->st_hits.cap / sizeof(Hit);
    if (hit_cap < 4096) { RFX_TRY(devbuf_reserve(c, c->st_hits, 4096 * sizeof(Hit))); hit_cap = c->st_hits.cap / sizeof(Hit); }
    uint64_t h[2];
    for (int attempt = 0;; attempt++) {
        RFX_CUDA(c, cudaMemsetAsync(ctr, 0, 2 * sizeof(uint64_t), st));
        stitch_scan_kernel<<<grid_for_n(n_reads), 256, 0, st>>>(d_text, rd_src, rd_len, n_reads, c->k, c->st_keys.as<uint64_t>(), c->st_vals.as<uint32_t>(), c->st_cap - 1,
                                                                  c->st_bloom.as<uint32_t>(), c->st_hits.as<Hit>(), hit_cap, ctr);
        c->launches++;
        RFX_CUDA(c, cudaMemcpyAsync(h, ctr, sizeof(h), cudaMemcpyDeviceToHost, st));
        RFX_CUDA(c, cudaStreamSynchronize(st));
        if (h[0] <= hit_cap) break;
        if (attempt) return ctx_fail(c, RFX_E_STATE, "internal: the fragment list overflowed twice");
        RFX_TRY(devbuf_reserve(c, c->st_hits, h[0] * sizeof(Hit)));  // (at most 2 per read) and once more with room for all
        hit_cap = c->st_hits.cap / sizeof(Hit);
    }
    if (h[0] == 0) return RFX_OK;
    RFX_TRY(devbuf_reserve(c, c->st_frags, (c->st_nfrag + h[0]) * sizeof(Frag), true));
    RFX_TRY(devbuf_reserve(c, c->st_codes, c->st_ncodes + h[1] + 16, true));
    stitch_copy_kernel<<<grid_for_n(h[0] * 32), 256, 0, st>>>(d_text, c->st_hits.as<Hit>(), h[0], c->k, c->st_keys.as<uint64_t>(), c->st_vals.as<uint32_t>(), c->st_cap - 1,
                                                            c->st_codes.as<uint8_t>(), c->st_ncodes, c->st_frags.as<Frag>(), c->st_nfrag);
    c->launches++;
    RFX_CUDA(c, cudaStreamSynchronize(st));  // the text buffer may be reused by the caller's next chunk
    c->st_nfrag += h[0];
    c->st_ncodes += h[1];
    return RFX_OK;
}

int stage_stitch_finish(Ctx* c) {
    if (!c->st_active) return ctx_fail(c, RFX_E_STATE, "rfx_stitch_finish: no stitch stage open (call rfx_stitch_begin first)");
    if (c->st_sharded) return ctx_fail(c, RFX_E_STATE, "rfx_stitch_finish: the open stage is a sharded one (finish it with rfx_stitch_finish_sharded on every rank)");
    c->st_active = false;
    cudaStream_t st = c->stream;
    const uint64_t n = c->n_contigs, nf = c->st_nfrag;
    c->st_stat[1] = nf;
    if (nf >= 0xffffffffull) return ctx_fail(c, RFX_E_CAPACITY, "more than 2^32 fragments");
    if (n == 0) return RFX_OK;
    stage_begin(c);
    unsigned long long* ctr = c->st_ctr.as<unsigned long long>();
    RFX_TRY(devbuf_reserve(c, c->st_nxt, n * sizeof(uint32_t)));
    RFX_TRY(devbuf_reserve(c, c->st_prv, n * sizeof(uint32_t)));
    RFX_TRY(devbuf_reserve(c, c->st_role, n));
    RFX_TRY(devbuf_reserve(c, c->st_outlen, n * sizeof(uint64_t)));
    RFX_TRY(devbuf_reserve(c, c->st_outright, n * sizeof(int32_t)));
    RFX_TRY(devbuf_reserve(c, c->st_slot, n * sizeof(uint64_t)));
    uint32_t *nxt = c->st_nxt.as<uint32_t>(), *prv = c->st_prv.as<uint32_t>();
    uint8_t* role = c->st_role.as<uint8_t>();
    const Frag* f = c->st_frags.as<Frag>();
    const uint8_t* codes = c->st_codes.as<uint8_t>();
    fill_u32_kernel<<<grid_for_n(n), 256, 0, st>>>(nxt, n, NONE32);
    fill_u32_kernel<<<grid_for_n(n), 256, 0, st>>>(prv, n, NONE32);
    RFX_CUDA(c, cudaMemsetAsync(role, 0, n, st));
    c->launches += 2;
    if (nf) {
        frag_pick_kernel<<<grid_for_n(nf), 256, 0, st>>>(f, codes, nf, 0, nullptr, nxt);
        frag_pick_kernel<<<grid_for_n(nf), 256, 0, st>>>(f, codes, nf, 1, nxt, prv);
        count_picked_kernel<<<grid_for_n(nf), 256, 0, st>>>(f, nf, nxt, prv, ctr + SC_PASS1);
        c->launches += 3;
    }
    chain_heads_kernel<<<grid_for_n(n), 256, 0, st>>>(n, nxt, prv, f, role);
    ring_heads_kernel<<<grid_for_n(n), 256, 0, st>>>(n, nxt, prv, f, c->st_firstk.as<uint64_t>(), role, ctr + SC_RINGS);
    chain_sizes_kernel<<<grid_for_n(n), 256, 0, st>>>(n, c->k, c->prm.min_contig, c->ctg_off.as<uint64_t>(), c->ctg_left.as<int32_t>(), c->ctg_right.as<int32_t>(), nxt, prv, f,
                                                     role, c->st_outlen.as<uint64_t>(), c->st_outright.as<int32_t>(), ctr + SC_STITCHED);
    c->launches += 3;
    ScanPlan<U64x3> plan;
    RFX_TRY(devbuf_reserve(c, c->scan_ws, ScanPlan<U64x3>::workspace_elems(n) * sizeof(U64x3)));
    plan.bind(n, c->scan_ws.as<U64x3>());
    KeepIn in{c->st_outlen.as<uint64_t>()};
    scan_prepare(plan, in, OpAddU64x3{}, U64x3{0, 0, 0}, st);
    c->launches += 2 * plan.levels;
    U64x3 tot;
    uint64_t h[SC_N];
    RFX_CUDA(c, cudaMemcpyAsync(&tot, plan.total, sizeof(tot), cudaMemcpyDeviceToHost, st));
    RFX_CUDA(c, cudaMemcpyAsync(h, ctr, sizeof(h), cudaMemcpyDeviceToHost, st));
    RFX_CUDA(c, cudaStreamSynchronize(st));
    DevBuf n_off, n_left, n_right, n_bases;
    int rc = RFX_OK;
    do {
        if ((rc = devbuf_reserve(c, n_off, (tot.a + 1) * sizeof(uint64_t))) != RFX_OK) break;
        if ((rc = devbuf_reserve(c, n_left, (tot.a + 1) * sizeof(int32_t))) != RFX_OK) break;
        if ((rc = devbuf_reserve(c, n_right, (tot.a + 1) * sizeof(int32_t))) != RFX_OK) break;
        if ((rc = devbuf_reserve(c, n_bases, tot.b + 16)) != RFX_OK) break;
        KeepOut out{c->ctg_left.as<int32_t>(), c->st_outright.as<int32_t>(), n_off.as<uint64_t>(), c->st_slot.as<uint64_t>(), n_left.as<int32_t>(), n_right.as<int32_t>()};
        scan_apply(plan, in, out, OpAddU64x3{}, U64x3{0, 0, 0}, st);
        set_end_kernel<<<1, 1, 0, st>>>(n_off.as<uint64_t>() + tot.a, plan.total);
        unsigned blocks = (unsigned)(n < (uint64_t)sm_count() * 8u ? (n ? n : 1) : (uint64_t)sm_count() * 8u);
        chain_gather_kernel<<<blocks, 256, 0, st>>>(n, c->k, c->ctg_off.as<uint64_t>(), c->ctg_bases.as<char>(), nxt, prv, f, codes, c->st_slot.as<uint64_t>(),
                                                    n_off.as<uint64_t>(), n_bases.as<char>());
        c->launches += 3;
        const cudaError_t e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) { rc = ctx_fail(c, RFX_E_CUDA, "stitch gather failed: %s", cudaGetErrorString(e)); break; }
    } while (0);
    if (rc != RFX_OK) { devbuf_free(n_off); devbuf_free(n_left); devbuf_free(n_right); devbuf_free(n_bases); return rc; }
    // the stitched set replaces the contigs of the extension
    devbuf_free(c->ctg_off); devbuf_free(c->ctg_left); devbuf_free(c->ctg_right); devbuf_free(c->ctg_bases);
    c->ctg_off = n_off; c->ctg_left = n_left; c->ctg_right = n_right; c->ctg_bases = n_bases;
    c->n_contigs = tot.a;
    c->n_contig_bases = tot.b;
    c->ms_stitch += stage_end(c);
    c->st_stat[2] = h[SC_PASS1]; c->st_stat[3] = h[SC_BOTH]; c->st_stat[4] = h[SC_STITCHED]; c->st_stat[5] = h[SC_RINGS];
    return RFX_OK;
}

// ---- across ranks ---------------------------------------------------------------------------------------------------------
// The reads are the large input; probes, fragments and contig metadata are small.  So every rank keeps its reads and its
// contigs where they are and replicates the small things: begin pulls every rank's per-contig summary (first k-mer, first and
// last (k-1)-mer, offsets, flags) and builds the same probe table over global contig ids (the ranks' contigs in rank order);
// every rank scans its own reads against it; finish pulls every rank's fragments, runs the picks and the chain heads over all
// contigs, and keeps, sizes and gathers the records whose head it owns, reading contig bases from their owner's arena.
// The result does not depend on how contigs and reads are split: the probe order, the fragment order (length, 2-bit sequence,
// index -- two fragments equal in length and sequence share their end (k-1)-mers, so their contigs, and which copy wins
// changes nothing) and the ring heads (smallest first k-mer) compare contents, never where a contig or a fragment came from.
static unsigned long long arena_off(const Ctx* c, const DevBuf& b) { return b.p ? (unsigned long long)(b.as<uint8_t>() - c->arena) : 0ull; }

int stage_stitch_begin_sharded(Ctx* c) {
    if (c->sh_world < 1 || !c->arena || !c->peer_base[c->sh_rank])
        return ctx_fail(c, RFX_E_STATE, "rfx_stitch_begin_sharded: call rfx_shard_init / rfx_shard_connect first");
    const int world = c->sh_world;
    unsigned long long mine[8];
    static_assert(sizeof(mine) / sizeof(mine[0]) <= PUB_VALS, "the summary exchange fits the published block");
    PubVals all;
    c->st_active = false; c->st_sharded = false;
    c->ms_comm = 0;
    // 1. what every rank holds and was asked for, before the assembly starts
    const bool sharded = c->have_counts && c->n_bins && c->n_bins % (uint32_t)world == 0;
    const int rc0 = sharded ? RFX_OK
                            : ctx_fail(c, RFX_E_STATE, "rfx_stitch_begin_sharded: this rank holds no table sharded by minimiser bin (rfx_count_sharded, or rfx_load_counts* and rfx_shard_table first)");
    mine[0] = (unsigned long long)c->k;
    mine[1] = (unsigned long long)(uint32_t)c->prm.min_contig;
    RFX_TRY(shard_exchange(c, rc0, 2, mine, all));
    for (int r = 1; r < world; r++) {
        if (all.at(r, 0) != all.at(0, 0)) return ctx_fail(c, RFX_E_INVALID, "rfx_stitch_begin_sharded: rank %d has k = %llu, rank 0 k = %llu", r, all.at(r, 0), all.at(0, 0));
        if (all.at(r, 1) != all.at(0, 1)) return ctx_fail(c, RFX_E_INVALID, "rfx_stitch_begin_sharded: rank %d has min_contig = %d, rank 0 %d", r, (int)all.at(r, 1), (int)all.at(0, 1));
    }
    // 2. the sharded assembly, every record kept (the minContig rule is applied to the stitched set)
    const float comm0 = c->ms_comm;
    const int32_t min_contig = c->prm.min_contig;
    c->prm.min_contig = 0;
    const int arc = stage_assemble_sharded(c);
    c->prm.min_contig = min_contig;
    c->ms_comm += comm0;
    RFX_TRY(arc);
    cudaStream_t st = c->stream;
    stage_begin(c);
    const bool no_probe_can_match = c->k > 31;  // (see stage_stitch_begin)
    const uint64_t n = c->n_contigs;
    // 3. the own summary, published with the contig counts
    const int rc1 = [&]() -> int {
        RFX_TRY(devbuf_reserve(c, c->st_lfirstk, (n + 1) * sizeof(uint64_t)));
        RFX_TRY(devbuf_reserve(c, c->st_lends, (2 * n + 2) * sizeof(uint64_t)));
        if (n && !no_probe_can_match) {
            probe_first_kernel<<<grid_for_n(n), 256, 0, st>>>(c->ctg_off.as<uint64_t>(), c->ctg_bases.as<char>(), n, c->k, c->st_lfirstk.as<uint64_t>());
            contig_ends_kernel<<<grid_for_n(n), 256, 0, st>>>(c->ctg_off.as<uint64_t>(), c->ctg_bases.as<char>(), n, c->k, c->st_lends.as<uint64_t>());
            c->launches += 2;
        } else if (n) {
            RFX_CUDA(c, cudaMemsetAsync(c->st_lfirstk.p, 0, n * sizeof(uint64_t), st));
            RFX_CUDA(c, cudaMemsetAsync(c->st_lends.p, 0, 2 * n * sizeof(uint64_t), st));
        }
        RFX_CUDA(c, cudaGetLastError());
        return RFX_OK;
    }();
    mine[0] = n;
    mine[1] = c->n_contig_bases;
    mine[2] = arena_off(c, c->ctg_off);
    mine[3] = arena_off(c, c->ctg_left);
    mine[4] = arena_off(c, c->ctg_right);
    mine[5] = arena_off(c, c->ctg_bases);
    mine[6] = arena_off(c, c->st_lfirstk);
    mine[7] = arena_off(c, c->st_lends);
    RFX_TRY(shard_exchange(c, rc1, 8, mine, all));
    c->st_ctg_lo[0] = 0; c->st_base_lo[0] = 0;
    for (int r = 0; r < world; r++) {
        c->st_ctg_lo[r + 1] = c->st_ctg_lo[r] + all.at(r, 0);
        c->st_base_lo[r + 1] = c->st_base_lo[r] + all.at(r, 1);
        c->st_bases_at[r] = all.at(r, 5);
    }
    const uint64_t N = c->st_ctg_lo[world];
    if (N > 0x7fffffffull) return ctx_fail(c, RFX_E_CAPACITY, "rfx_stitch_begin_sharded: %llu contigs, a probe holds the id of at most 2^31 - 1", (unsigned long long)N);
    // 4. everybody's summary -> the replicated per-contig arrays and the probe table over global ids
    uint64_t cap = 1024;
    while (cap < 4 * N + 16) cap <<= 1;  // at most 2 probes per contig: load <= 0.5
    uint64_t h[SC_N] = {0};
    const uint64_t g_end = c->st_base_lo[world];
    const int rc2 = [&]() -> int {
        RFX_TRY(devbuf_reserve(c, c->st_keys, cap * sizeof(uint64_t)));
        RFX_TRY(devbuf_reserve(c, c->st_vals, cap * sizeof(uint32_t)));
        RFX_TRY(devbuf_reserve(c, c->st_firstk, (N + 1) * sizeof(uint64_t)));
        RFX_TRY(devbuf_reserve(c, c->st_ctr, SC_N * sizeof(uint64_t)));
        RFX_TRY(devbuf_reserve(c, c->st_bloom, ST_BLOOM_BITS / 8));
        RFX_TRY(devbuf_reserve(c, c->st_goff, (N + 1) * sizeof(uint64_t)));
        RFX_TRY(devbuf_reserve(c, c->st_gends, (2 * N + 2) * sizeof(uint64_t)));
        RFX_TRY(devbuf_reserve(c, c->st_gleft, (N + 1) * sizeof(int32_t)));
        RFX_TRY(devbuf_reserve(c, c->st_gright, (N + 1) * sizeof(int32_t)));
        RFX_CUDA(c, cudaMemsetAsync(c->st_bloom.p, 0, ST_BLOOM_BITS / 8, st));
        RFX_CUDA(c, cudaMemsetAsync(c->st_keys.p, 0xff, cap * sizeof(uint64_t), st));
        RFX_CUDA(c, cudaMemsetAsync(c->st_vals.p, 0xff, cap * sizeof(uint32_t), st));
        RFX_CUDA(c, cudaMemsetAsync(c->st_ctr.p, 0, SC_N * sizeof(uint64_t), st));
        for (int r = 0; r < world; r++) {
            const uint64_t nr = all.at(r, 0), lo = c->st_ctg_lo[r];
            if (!nr) continue;
            const uint8_t* pb = c->peer_base[r];
            RFX_CUDA(c, cudaMemcpyAsync(c->st_firstk.as<uint64_t>() + lo, pb + all.at(r, 6), nr * sizeof(uint64_t), cudaMemcpyDefault, st));
            RFX_CUDA(c, cudaMemcpyAsync(c->st_gends.as<uint64_t>() + 2 * lo, pb + all.at(r, 7), 2 * nr * sizeof(uint64_t), cudaMemcpyDefault, st));
            RFX_CUDA(c, cudaMemcpyAsync(c->st_gleft.as<int32_t>() + lo, pb + all.at(r, 3), nr * sizeof(int32_t), cudaMemcpyDefault, st));
            RFX_CUDA(c, cudaMemcpyAsync(c->st_gright.as<int32_t>() + lo, pb + all.at(r, 4), nr * sizeof(int32_t), cudaMemcpyDefault, st));
            rebase_off_kernel<<<grid_for_n(nr), 256, 0, st>>>(reinterpret_cast<const uint64_t*>(pb + all.at(r, 2)), nr, c->st_base_lo[r], c->st_goff.as<uint64_t>() + lo);
            c->launches++;
        }
        RFX_CUDA(c, cudaMemcpyAsync(c->st_goff.as<uint64_t>() + N, &g_end, sizeof(uint64_t), cudaMemcpyHostToDevice, st));
        unsigned long long* ctr = c->st_ctr.as<unsigned long long>();
        if (N && !no_probe_can_match) {
            probe_insert_ends_kernel<<<grid_for_n(N), 256, 0, st>>>(c->st_goff.as<uint64_t>(), c->st_gends.as<uint64_t>(), c->st_gleft.as<int32_t>(), c->st_gright.as<int32_t>(), N,
                                                                   c->st_firstk.as<uint64_t>(), c->st_keys.as<uint64_t>(), c->st_vals.as<uint32_t>(), cap - 1,
                                                                   c->st_bloom.as<uint32_t>(), ctr + SC_PUT);
            count_keys_kernel<<<grid_for_n(cap), 256, 0, st>>>(c->st_keys.as<uint64_t>(), cap, ctr + SC_KEYS);
            c->launches += 2;
        }
        RFX_CUDA(c, cudaMemcpyAsync(h, c->st_ctr.p, sizeof(h), cudaMemcpyDeviceToHost, st));
        const cudaError_t e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) return ctx_fail(c, RFX_E_CUDA, "rfx_stitch_begin_sharded: probe table failed: %s", cudaGetErrorString(e));
        return RFX_OK;
    }();
    // 5. nobody may reuse its summary before every rank has pulled it; every rank built the same table
    mine[0] = h[SC_KEYS];
    RFX_TRY(shard_exchange(c, rc2, 1, mine, all));
    for (int r = 1; r < world; r++)
        if (all.at(r, 0) != all.at(0, 0)) return ctx_fail(c, RFX_E_STATE, "internal: rank %d built a probe table of %llu keys, rank 0 one of %llu", r, all.at(r, 0), all.at(0, 0));
    c->ms_stitch = stage_end(c);
    c->st_cap = cap;
    c->st_stat[0] = h[SC_KEYS];
    for (int i = 1; i < 6; i++) c->st_stat[i] = 0;
    c->st_nfrag = 0; c->st_ncodes = 0; c->st_reads = 0;
    c->st_active = true;
    c->st_sharded = true;
    return RFX_OK;
}

int stage_stitch_finish_sharded(Ctx* c) {
    if (c->sh_world < 1 || !c->arena || !c->peer_base[c->sh_rank])
        return ctx_fail(c, RFX_E_STATE, "rfx_stitch_finish_sharded: call rfx_shard_init / rfx_shard_connect first");
    const int world = c->sh_world, me = c->sh_rank;
    unsigned long long mine[4];
    PubVals all;
    const bool open = c->st_active && c->st_sharded;
    c->st_active = false; c->st_sharded = false;
    c->ms_comm = 0;
    const int rc0 = open ? RFX_OK : ctx_fail(c, RFX_E_STATE, "rfx_stitch_finish_sharded: no sharded stitch stage open on this rank (call rfx_stitch_begin_sharded first)");
    const uint64_t nf = c->st_nfrag;
    c->st_stat[1] = nf;
    // 1. every rank's fragments: how many, where
    mine[0] = nf;
    mine[1] = c->st_ncodes;
    mine[2] = nf ? arena_off(c, c->st_frags) : 0ull;
    mine[3] = nf ? arena_off(c, c->st_codes) : 0ull;
    RFX_TRY(shard_exchange(c, rc0, 4, mine, all));
    uint64_t frag_lo[RFX_MAX_RANKS + 1], code_lo[RFX_MAX_RANKS + 1];
    frag_lo[0] = code_lo[0] = 0;
    for (int r = 0; r < world; r++) { frag_lo[r + 1] = frag_lo[r] + all.at(r, 0); code_lo[r + 1] = code_lo[r] + all.at(r, 1); }
    const uint64_t NF = frag_lo[world], NC = code_lo[world];
    if (NF >= 0xffffffffull) return ctx_fail(c, RFX_E_CAPACITY, "rfx_stitch_finish_sharded: %llu fragments over all ranks, at most 2^32 - 2", (unsigned long long)NF);
    const uint64_t N = c->st_ctg_lo[world], lo = c->st_ctg_lo[me], hi = c->st_ctg_lo[me + 1], n_own = hi - lo;
    cudaStream_t st = c->stream;
    stage_begin(c);
    // 2. pull, pick and chain over all contigs; keep, size and gather the own heads
    U64x3 tot{0, 0, 0};
    uint64_t h[SC_N] = {0};
    DevBuf n_off, n_left, n_right, n_bases;
    const int rc1 = [&]() -> int {
        RFX_TRY(devbuf_reserve(c, c->st_gfrags, (NF + 1) * sizeof(Frag)));
        RFX_TRY(devbuf_reserve(c, c->st_gcodes, NC + 16));
        RFX_TRY(devbuf_reserve(c, c->st_nxt, (N + 1) * sizeof(uint32_t)));
        RFX_TRY(devbuf_reserve(c, c->st_prv, (N + 1) * sizeof(uint32_t)));
        RFX_TRY(devbuf_reserve(c, c->st_role, N + 1));
        RFX_TRY(devbuf_reserve(c, c->st_outlen, (n_own + 1) * sizeof(uint64_t)));
        RFX_TRY(devbuf_reserve(c, c->st_outright, (n_own + 1) * sizeof(int32_t)));
        RFX_TRY(devbuf_reserve(c, c->st_slot, (n_own + 1) * sizeof(uint64_t)));
        Frag* f = c->st_gfrags.as<Frag>();
        uint8_t* codes = c->st_gcodes.as<uint8_t>();
        for (int r = 0; r < world; r++) {
            const uint64_t nr = all.at(r, 0);
            if (!nr) continue;
            const uint8_t* pb = c->peer_base[r];
            frag_pull_kernel<<<grid_for_n(nr), 256, 0, st>>>(reinterpret_cast<const Frag*>(pb + all.at(r, 2)), nr, code_lo[r], f + frag_lo[r]);
            c->launches++;
            if (all.at(r, 1)) RFX_CUDA(c, cudaMemcpyAsync(codes + code_lo[r], pb + all.at(r, 3), all.at(r, 1), cudaMemcpyDefault, st));
        }
        unsigned long long* ctr = c->st_ctr.as<unsigned long long>();
        RFX_CUDA(c, cudaMemsetAsync(ctr + SC_PASS1, 0, (SC_N - SC_PASS1) * sizeof(uint64_t), st));
        uint32_t *nxt = c->st_nxt.as<uint32_t>(), *prv = c->st_prv.as<uint32_t>();
        uint8_t* role = c->st_role.as<uint8_t>();
        if (N) {
            fill_u32_kernel<<<grid_for_n(N), 256, 0, st>>>(nxt, N, NONE32);
            fill_u32_kernel<<<grid_for_n(N), 256, 0, st>>>(prv, N, NONE32);
            RFX_CUDA(c, cudaMemsetAsync(role, 0, N, st));
            c->launches += 2;
        }
        if (NF) {
            frag_pick_kernel<<<grid_for_n(NF), 256, 0, st>>>(f, codes, NF, 0, nullptr, nxt);
            frag_pick_kernel<<<grid_for_n(NF), 256, 0, st>>>(f, codes, NF, 1, nxt, prv);
            count_picked_kernel<<<grid_for_n(NF), 256, 0, st>>>(f, NF, nxt, prv, ctr + SC_PASS1);
            c->launches += 3;
        }
        if (N) {
            chain_heads_kernel<<<grid_for_n(N), 256, 0, st>>>(N, nxt, prv, f, role);
            c->launches++;
        }
        ScanPlan<U64x3> plan;
        KeepIn in{c->st_outlen.as<uint64_t>()};
        if (n_own) {
            ring_heads_range_kernel<<<grid_for_n(n_own), 256, 0, st>>>(lo, hi, N, nxt, prv, f, c->st_firstk.as<uint64_t>(), role, ctr + SC_RINGS);
            chain_sizes_range_kernel<<<grid_for_n(n_own), 256, 0, st>>>(lo, hi, N, c->k, c->prm.min_contig, c->st_goff.as<uint64_t>(), c->st_gleft.as<int32_t>(),
                                                                        c->st_gright.as<int32_t>(), nxt, prv, f, role, c->st_outlen.as<uint64_t>(),
                                                                        c->st_outright.as<int32_t>(), ctr + SC_STITCHED);
            c->launches += 2;
            RFX_TRY(devbuf_reserve(c, c->scan_ws, ScanPlan<U64x3>::workspace_elems(n_own) * sizeof(U64x3)));
            plan.bind(n_own, c->scan_ws.as<U64x3>());
            scan_prepare(plan, in, OpAddU64x3{}, U64x3{0, 0, 0}, st);
            c->launches += 2 * plan.levels;
            RFX_CUDA(c, cudaMemcpyAsync(&tot, plan.total, sizeof(tot), cudaMemcpyDeviceToHost, st));
        }
        RFX_CUDA(c, cudaMemcpyAsync(h, ctr, sizeof(h), cudaMemcpyDeviceToHost, st));
        cudaError_t e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) return ctx_fail(c, RFX_E_CUDA, "rfx_stitch_finish_sharded: chains failed: %s", cudaGetErrorString(e));
        RFX_TRY(devbuf_reserve(c, n_off, (tot.a + 1) * sizeof(uint64_t)));
        RFX_TRY(devbuf_reserve(c, n_left, (tot.a + 1) * sizeof(int32_t)));
        RFX_TRY(devbuf_reserve(c, n_right, (tot.a + 1) * sizeof(int32_t)));
        RFX_TRY(devbuf_reserve(c, n_bases, tot.b + 16));
        if (!n_own) {
            RFX_CUDA(c, cudaMemsetAsync(n_off.p, 0, sizeof(uint64_t), st));
            return RFX_OK;
        }
        KeepOut out{c->st_gleft.as<int32_t>() + lo, c->st_outright.as<int32_t>(), n_off.as<uint64_t>(), c->st_slot.as<uint64_t>(), n_left.as<int32_t>(), n_right.as<int32_t>()};
        scan_apply(plan, in, out, OpAddU64x3{}, U64x3{0, 0, 0}, st);
        set_end_kernel<<<1, 1, 0, st>>>(n_off.as<uint64_t>() + tot.a, plan.total);
        CtgSources P;
        memset(&P, 0, sizeof(P));
        P.n = world;
        P.off = c->st_goff.as<uint64_t>();
        for (int r = 0; r < world; r++) P.bases[r] = reinterpret_cast<const char*>(c->peer_base[r] + c->st_bases_at[r]);
        for (int r = 0; r <= world; r++) { P.ctg_lo[r] = c->st_ctg_lo[r]; P.base_lo[r] = c->st_base_lo[r]; }
        const unsigned blocks = (unsigned)(n_own < (uint64_t)sm_count() * 8u ? n_own : (uint64_t)sm_count() * 8u);
        chain_gather_peer_kernel<<<blocks, 256, 0, st>>>(lo, hi, N, c->k, P, nxt, prv, f, codes, c->st_slot.as<uint64_t>(), n_off.as<uint64_t>(), n_bases.as<char>());
        c->launches += 3;
        e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) return ctx_fail(c, RFX_E_CUDA, "rfx_stitch_finish_sharded: gather failed: %s", cudaGetErrorString(e));
        return RFX_OK;
    }();
    // 3. nobody returns (and may recycle its arena) while a peer still reads its contig bases; the global record counts
    mine[0] = tot.a;
    mine[1] = tot.b;
    const int rc2 = shard_exchange(c, rc1, 2, mine, all);
    if (rc2 != RFX_OK) { devbuf_free(n_off); devbuf_free(n_left); devbuf_free(n_right); devbuf_free(n_bases); return rc2; }
    // the stitched records of the own heads replace the own contigs
    devbuf_free(c->ctg_off); devbuf_free(c->ctg_left); devbuf_free(c->ctg_right); devbuf_free(c->ctg_bases);
    c->ctg_off = n_off; c->ctg_left = n_left; c->ctg_right = n_right; c->ctg_bases = n_bases;
    c->n_contigs = tot.a;
    c->n_contig_bases = tot.b;
    shard_graph_set_contigs_global(c, all.sum(0), all.sum(1));
    c->ms_stitch += stage_end(c);
    c->st_stat[2] = h[SC_PASS1]; c->st_stat[3] = h[SC_BOTH]; c->st_stat[4] = h[SC_STITCHED]; c->st_stat[5] = h[SC_RINGS];
    return RFX_OK;
}

}  // namespace rfx
