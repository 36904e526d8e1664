// stitch_sharded_emu.cpp -- TEST-ONLY: runs the kernels of reflexiv_b200/csrc/rfx_stitch_kernels.cuh on the host, thread by
// thread, in the order rfx_stitch.cu launches them for rfx_stitch_begin_sharded / rfx_stitch_finish_sharded, for W simulated
// ranks.  A rank's "peer pointers" are the other ranks' host arrays; the pulls a rank does with cudaMemcpyAsync are memcpy.
// Checked against oracle/stitch_oracle.c on a machine without a GPU (see stitch_emu.cpp for the shim); tests/test_stitch_sharded_cpu.py
// compiles it into a temporary directory.
// Not part of libreflexiv_cuda; nothing in reflexiv_b200/ uses it.
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <vector>

#define RFX_STITCH_HOSTEMU 1
#define __global__
#define __device__
#define __forceinline__ inline
#define __restrict__
#define __launch_bounds__(x)
struct EmuDim { unsigned x = 1, y = 1, z = 1; };
static EmuDim blockIdx, threadIdx, gridDim, blockDim;
template <class T> static inline T __ldg(const T* p) { return *p; }
static inline unsigned long long atomicCAS(unsigned long long* p, unsigned long long cmp, unsigned long long v) { unsigned long long o = *p; if (o == cmp) *p = v; return o; }
static inline uint32_t atomicCAS(uint32_t* p, uint32_t cmp, uint32_t v) { uint32_t o = *p; if (o == cmp) *p = v; return o; }
static inline unsigned long long atomicAdd(unsigned long long* p, unsigned long long v) { unsigned long long o = *p; *p += v; return o; }
static inline uint32_t atomicOr(uint32_t* p, uint32_t v) { uint32_t o = *p; *p |= v; return o; }
static inline void __syncwarp() {}
namespace rfx {
struct U64x3 { uint64_t a, b, c; };
static const uint32_t NONE32 = 0xffffffffu;
}  // namespace rfx

#include "../../reflexiv_b200/csrc/rfx_stitch_kernels.cuh"

using namespace rfx;
using namespace rfx::stitch;

template <class F> static void launch(unsigned grid, unsigned block, F f) {
    gridDim.x = grid; blockDim.x = block;
    for (unsigned b = 0; b < grid; b++)
        for (unsigned t = 0; t < block; t++) { blockIdx.x = b; threadIdx.x = t; f(); }
}

namespace {

struct Rank {
    // input: the contigs the sharded assembly left on this rank, the reads pushed to it
    uint64_t n = 0;
    const uint64_t* off = nullptr;
    const char* bases = nullptr;
    const int32_t *cl = nullptr, *cr = nullptr;
    uint64_t n_reads = 0;
    const uint64_t* starts = nullptr;
    std::vector<uint32_t> elen;
    // begin
    std::vector<uint64_t> lfirstk, lends, firstk, goff, gends, keys;
    std::vector<int32_t> gleft, gright;
    std::vector<uint32_t> vals, bloom;
    unsigned long long ctr[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    // scan
    std::vector<Frag> frags;
    std::vector<uint8_t> codes;
};

}  // namespace

extern "C" {

struct EmuStitchOut {
    uint64_t n_contigs;
    uint64_t* off;
    char* bases;
    int32_t *left, *right;
    uint64_t stats[6];  // probes, fragments, after pass 1, joined on both sides, stitched records, rings
};

void emu_stitch_sharded_free(EmuStitchOut* o, int world) {
    for (int r = 0; r < world; r++) { free(o[r].off); free(o[r].bases); free(o[r].left); free(o[r].right); memset(&o[r], 0, sizeof(o[r])); }
}

// Rank r holds n[r] contigs (off[r], bases[r], cl[r], cr[r]) and the n_reads[r] reads at starts[r] / lens[r] of `text` (one
// FASTQ text for all: any split on record boundaries).  hit_cap0: first capacity of a rank's fragment list.
int emu_stitch_sharded(int world, const uint64_t* n, const uint64_t* const* off, const char* const* bases, const int32_t* const* cl, const int32_t* const* cr,
                       const uint8_t* text, const uint64_t* n_reads, const uint64_t* const* starts, const uint32_t* const* lens, int k, int min_contig,
                       uint64_t hit_cap0, EmuStitchOut* out) {
    memset(out, 0, sizeof(*out) * (size_t)world);
    if (k < 2 || k > 31 || world < 1 || world > 8) return -1;
    const unsigned G = 3, B = 64;
    std::vector<Rank> R(world);
    uint64_t text_len = 0;
    for (int r = 0; r < world; r++) {
        Rank& q = R[r];
        q.n = n[r]; q.off = off[r]; q.bases = bases[r]; q.cl = cl[r]; q.cr = cr[r];
        q.n_reads = n_reads[r]; q.starts = starts[r];
        q.elen.assign(q.n_reads ? q.n_reads : 1, 0);
        for (uint64_t i = 0; i < q.n_reads; i++) {
            q.elen[i] = ((int64_t)lens[r][i] - (k - 1) <= 1) ? 0u : lens[r][i];  // effective_read_len(len, k - 1, 0, 0)
            if (q.starts[i] + lens[r][i] > text_len) text_len = q.starts[i] + lens[r][i];
        }
    }
    // the scan reads the text in aligned 4-byte words: give it the slack the device buffer has
    std::vector<uint8_t> padded(text_len + 16, 0);
    if (text_len) memcpy(padded.data() + 8, text, text_len);
    text = padded.data() + 8;

    // ---- stage_stitch_begin_sharded: 3. the own summary ----
    for (Rank& q : R) {
        q.lfirstk.assign(q.n + 1, 0);
        q.lends.assign(2 * q.n + 2, 0);
        if (q.n) {
            launch(G, B, [&] { probe_first_kernel(q.off, q.bases, q.n, k, q.lfirstk.data()); });
            launch(G, B, [&] { contig_ends_kernel(q.off, q.bases, q.n, k, q.lends.data()); });
        }
    }
    std::vector<uint64_t> ctg_lo(world + 1, 0), base_lo(world + 1, 0);
    for (int r = 0; r < world; r++) { ctg_lo[r + 1] = ctg_lo[r] + R[r].n; base_lo[r + 1] = base_lo[r] + R[r].off[R[r].n]; }
    const uint64_t N = ctg_lo[world];
    uint64_t cap = 1024;
    while (cap < 4 * N + 16) cap <<= 1;
    // 4. everybody's summary -> the replicated arrays and the probe table
    for (Rank& q : R) {
        q.keys.assign(cap, ~0ull); q.vals.assign(cap, NONE32); q.bloom.assign(ST_BLOOM_BITS / 32, 0);
        q.firstk.assign(N + 1, 0); q.goff.assign(N + 1, 0); q.gends.assign(2 * N + 2, 0); q.gleft.assign(N + 1, 0); q.gright.assign(N + 1, 0);
        for (int r = 0; r < world; r++) {
            const Rank& p = R[r];
            const uint64_t lo = ctg_lo[r];
            if (!p.n) continue;
            memcpy(q.firstk.data() + lo, p.lfirstk.data(), p.n * sizeof(uint64_t));
            memcpy(q.gends.data() + 2 * lo, p.lends.data(), 2 * p.n * sizeof(uint64_t));
            memcpy(q.gleft.data() + lo, p.cl, p.n * sizeof(int32_t));
            memcpy(q.gright.data() + lo, p.cr, p.n * sizeof(int32_t));
            launch(G, B, [&] { rebase_off_kernel(p.off, p.n, base_lo[r], q.goff.data() + lo); });
        }
        q.goff[N] = base_lo[world];
        if (N) {
            launch(G, B, [&] { probe_insert_ends_kernel(q.goff.data(), q.gends.data(), q.gleft.data(), q.gright.data(), N, q.firstk.data(), q.keys.data(), q.vals.data(), cap - 1,
                                                        q.bloom.data(), &q.ctr[2]); });
            launch(G, B, [&] { count_keys_kernel(q.keys.data(), cap, &q.ctr[3]); });
        }
    }
    for (int r = 0; r < world; r++)
        if (R[r].ctr[3] != R[0].ctr[3]) return -3;  // every rank built the same table

    // ---- stitch_scan_reads on every rank's own reads ----
    for (Rank& q : R) {
        if (!q.n_reads || !q.ctr[3]) continue;
        std::vector<Hit> hits(hit_cap0 ? hit_cap0 : 1);
        for (int attempt = 0;; attempt++) {
            q.ctr[0] = q.ctr[1] = 0;
            launch(G, B, [&] { stitch_scan_kernel(text, q.starts, q.elen.data(), q.n_reads, k, q.keys.data(), q.vals.data(), cap - 1, q.bloom.data(), hits.data(), hits.size(), q.ctr); });
            if (q.ctr[0] <= hits.size()) break;
            if (attempt) return -2;
            hits.resize(q.ctr[0]);
        }
        if (!q.ctr[0]) continue;
        q.frags.resize(q.ctr[0]);
        q.codes.resize(q.ctr[1] + 16);
        launch(G, B, [&] { stitch_copy_kernel(text, hits.data(), q.ctr[0], k, q.keys.data(), q.vals.data(), cap - 1, q.codes.data(), 0, q.frags.data(), 0); });
        q.codes.resize(q.ctr[1]);
    }

    // ---- stage_stitch_finish_sharded ----
    std::vector<uint64_t> frag_lo(world + 1, 0), code_lo(world + 1, 0);
    for (int r = 0; r < world; r++) { frag_lo[r + 1] = frag_lo[r] + R[r].frags.size(); code_lo[r + 1] = code_lo[r] + R[r].codes.size(); }
    const uint64_t NF = frag_lo[world], NC = code_lo[world];
    for (int me = 0; me < world; me++) {
        Rank& q = R[me];
        const uint64_t lo = ctg_lo[me], hi = ctg_lo[me + 1], n_own = hi - lo;
        std::vector<Frag> f(NF + 1);
        std::vector<uint8_t> codes(NC + 16, 0);
        for (int r = 0; r < world; r++) {
            const Rank& p = R[r];
            if (p.frags.empty()) continue;
            launch(G, B, [&] { frag_pull_kernel(p.frags.data(), p.frags.size(), code_lo[r], f.data() + frag_lo[r]); });
            memcpy(codes.data() + code_lo[r], p.codes.data(), p.codes.size());
        }
        unsigned long long ctr[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        std::vector<uint32_t> nxt(N + 1), prv(N + 1);
        std::vector<uint8_t> role(N + 1, 0);
        std::vector<uint64_t> out_len(n_own + 1), slot(n_own + 1);
        std::vector<int32_t> out_right(n_own + 1);
        if (N) {
            launch(G, B, [&] { fill_u32_kernel(nxt.data(), N, NONE32); });
            launch(G, B, [&] { fill_u32_kernel(prv.data(), N, NONE32); });
        }
        if (NF) {
            launch(G, B, [&] { frag_pick_kernel(f.data(), codes.data(), NF, 0, nullptr, nxt.data()); });
            launch(G, B, [&] { frag_pick_kernel(f.data(), codes.data(), NF, 1, nxt.data(), prv.data()); });
            launch(G, B, [&] { count_picked_kernel(f.data(), NF, nxt.data(), prv.data(), &ctr[4]); });
        }
        if (N) launch(G, B, [&] { chain_heads_kernel(N, nxt.data(), prv.data(), f.data(), role.data()); });
        EmuStitchOut& o = out[me];
        o.stats[0] = q.ctr[3];
        o.stats[1] = q.frags.size();
        o.stats[2] = ctr[4]; o.stats[3] = ctr[5];
        if (n_own) {
            launch(G, B, [&] { ring_heads_range_kernel(lo, hi, N, nxt.data(), prv.data(), f.data(), q.firstk.data(), role.data(), &ctr[7]); });
            launch(G, B, [&] { chain_sizes_range_kernel(lo, hi, N, k, min_contig, q.goff.data(), q.gleft.data(), q.gright.data(), nxt.data(), prv.data(), f.data(), role.data(),
                                                        out_len.data(), out_right.data(), &ctr[6]); });
        }
        o.stats[4] = ctr[6]; o.stats[5] = ctr[7];
        // the transform-scan of rfx_scan.cuh over the own heads, element by element
        KeepIn in{out_len.data()};
        U64x3 tot{0, 0, 0};
        for (uint64_t c = 0; c < n_own; c++) { const U64x3 v = in(c); tot.a += v.a; tot.b += v.b; }
        o.off = (uint64_t*)malloc((tot.a + 1) * sizeof(uint64_t));
        o.left = (int32_t*)malloc((tot.a + 1) * sizeof(int32_t));
        o.right = (int32_t*)malloc((tot.a + 1) * sizeof(int32_t));
        o.bases = (char*)malloc(tot.b + 16);
        KeepOut ko{q.gleft.data() + lo, out_right.data(), o.off, slot.data(), o.left, o.right};
        U64x3 acc{0, 0, 0};
        for (uint64_t c = 0; c < n_own; c++) { const U64x3 v = in(c); ko(c, acc, v); acc.a += v.a; acc.b += v.b; }
        o.off[tot.a] = tot.b;
        o.n_contigs = tot.a;
        if (!n_own) continue;
        CtgSources P;
        memset(&P, 0, sizeof(P));
        P.n = world;
        P.off = q.goff.data();
        for (int r = 0; r < world; r++) P.bases[r] = R[r].bases;
        for (int r = 0; r <= world; r++) { P.ctg_lo[r] = ctg_lo[r]; P.base_lo[r] = base_lo[r]; }
        launch(5, 32, [&] { chain_gather_peer_kernel(lo, hi, N, k, P, nxt.data(), prv.data(), f.data(), codes.data(), slot.data(), o.off, o.bases); });
    }
    return 0;
}
}
