// rfx_graph.cu -- K5 (both orientations, fork filters, neighbour links), K6 (list ranking of the unitig
// chains), K7 (contig gather).
//
// Replaces, in ReflexivDSMain.java (paths relative to .../reflexiv/pipeline/):
//   DSKmerReverseComplementLong :3849-3869        both orientations of every kept k-mer
//   DSForwardSubKmerExtraction :3625-3644 + sort + DSFilterForkSubKmer(WithErrorCorrection) :3375-3483
//   DSReflectedSubKmerExtractionFromForward :3661-3685 + sort + DSFilterForkReflectedSubKmer(...) :3489-3616
//   DSkmerRandomReflection :3688-3792, DSExtendReflexivKmer :3011-3362, ...ToArrayFirstTime :2559-3004,
//   ...ToArrayLoop :1746-2551 and the driver loop :261-326   (>= 18 global sorts in the reference)
//   DSBinaryReflexivKmerArrayToString :855-900, DSKmerToContig :743-771
//
// Data layout in HBM: the filtered table (keys[], counts[]) is the only copy of the k-mers.  An
// oriented k-mer is an id  oid = 2*row + strand  (strand 1 = reverse complement of keys[row]); every
// per-node array (flags, links, ranks) is indexed by oid.  A 32-bit open-addressing index (ht[]) maps a
// canonical k-mer to its row.  K5 probes it once per node for the 4 possible successors and stores them (N(Y), below);
// both fork filters and the links read their neighbour sets from there.
//
// After the two fork filters every (k-1)-mer has at most one surviving out-edge and one in-edge, so
// the reference's sort-and-merge iteration converges to the maximal paths of that graph; pointer
// jumping computes (head, rank) for every node in O(log n) rounds instead.
#include <cooperative_groups.h>
#include <stdlib.h>
#include <string.h>

#include "rfx_internal.h"
#include "rfx_graph.cuh"
#include "rfx_scan.cuh"

namespace rfx {

// The index is local to minimiser bins: a row lives in the hash region of the bin its canonical minimiser hashes to
// (regions are back to back in ht[], 4 * rows + 2 slots each).  A neighbour shares k-1 bases with the node that asks
// for it, so its minimiser -- hence its region -- is almost always the node's own: the probes of the adjacency pass
// (and of the fork filters' direct fallback) stay inside a few hundred bytes that the neighbouring threads (rows come
// out of the counting kernel grouped by bin) have just touched, instead of landing anywhere in a table of hundreds of
// megabytes.  The
// asking node computes the m-mer hashes of its own k-mer once; a candidate's minimiser is then the minimum over the
// shared (k-1)-mer plus one new m-mer.  (The same bin -> owner map is what lets a sharded run route a probe.)
template <class KT> struct Graph {
    const KT* keys;
    const uint32_t* counts;
    uint64_t n_rows;
    uint32_t* ht;
    const uint64_t* hoff;  // [g_bins + 1] first slot of every bin's region
    uint32_t g_bins;       // 1: the whole table is one region of cap0 slots (tables that fit L2)
    uint32_t cap0;
    int k, m;
    // presence bits (one hash, >= 16 bits per row): three of four probes ask for a k-mer that does not exist, and
    // most of those are answered from this small array (16 MB at config 2) without touching the index or the keys
    uint32_t* bloom;
    uint64_t bloom_mask;  // number of bits - 1 (power of two), 0: no filter

    __device__ __forceinline__ uint32_t bin_of(uint32_t hmin) const { return (uint32_t)(((uint64_t)fmix32(hmin ^ 0x7f4a7c15u) * g_bins) >> 32); }
    __device__ __forceinline__ uint32_t mm_hash(uint32_t mm) const { return mm_hash_m(mm, m); }
    __device__ __forceinline__ void minima(KT X, uint32_t& pre_min, uint32_t& suf_min) const { kmer_minima<KT>(X, k, m, pre_min, suf_min); }
    __device__ __forceinline__ uint32_t last_mm(KT S, uint32_t b) const { return last_mm_of<KT>(S, b, m); }
    __device__ __forceinline__ uint32_t first_mm(KT S, uint32_t a) const { return first_mm_of<KT>(S, a, k, m); }
    __device__ __forceinline__ uint32_t lookup(KT canon, uint32_t hmin) const {
        const uint64_t kh = key_hash(canon);
        if (bloom_mask) {
            const uint64_t bit = (kh >> 13) & bloom_mask;
            if (!((bloom[bit >> 5] >> (bit & 31u)) & 1u)) return NONE32;
        }
        uint64_t lo = 0;
        uint32_t cap = cap0;
        if (g_bins > 1) {
            const uint32_t b = bin_of(hmin);
            lo = hoff[b];
            cap = (uint32_t)(hoff[b + 1] - lo);
        }
        uint32_t slot = (uint32_t)(((uint64_t)(uint32_t)(kh >> 20) * cap) >> 32);
        while (true) {
            const uint32_t v = ht[lo + slot];
            if (v == NONE32) return NONE32;
            if (keys[v] == canon) return v;
            slot = slot + 1 == cap ? 0u : slot + 1;
        }
    }
    __device__ __forceinline__ KT oriented(uint32_t oid) const {
        const KT key = keys[oid >> 1];
        return (oid & 1u) ? revcomp(key, k) : key;
    }
    // oriented id of the oriented k-mer Z (whose minimiser hash is hmin), NONE32 if its canonical form is not in the table
    __device__ __forceinline__ uint32_t find(KT Z, uint32_t hmin, uint32_t* cnt) const {
        const KT zc = revcomp(Z, k);
        const bool fwd = !(zc < Z);
        const uint32_t r = lookup(fwd ? Z : zc, hmin);
        if (r == NONE32) return NONE32;
        *cnt = counts[r];
        return 2u * r + (fwd ? 0u : 1u);
    }
};

// index build: bin of every row + rows per bin, region offsets by scan, insertion
template <class KT> __global__ void row_bin_kernel(Graph<KT> G, uint32_t* __restrict__ row_bin, uint32_t* __restrict__ bin_rows) {
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < G.n_rows; r += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t a, b;
        G.minima(G.keys[r], a, b);
        // minimiser of the whole k-mer: the first m-mer is in the prefix part, the last one in the suffix part
        const uint32_t bin = G.bin_of(a < b ? a : b);
        row_bin[r] = bin;
        atomicAdd(&bin_rows[bin], 1u);
    }
}
struct RegionIn {
    const uint32_t* bin_rows;
    __device__ __forceinline__ uint64_t operator()(uint64_t i) const { return 4ull * bin_rows[i] + 2ull; }
};
struct RegionOut {
    uint64_t* hoff;
    __device__ __forceinline__ void operator()(uint64_t i, uint64_t excl, uint64_t) const { hoff[i] = excl; }
};
__global__ void set_last_region_kernel(uint64_t* hoff, uint64_t g_bins, const uint64_t* total) { hoff[g_bins] = *total; }

template <class KT> __global__ void ht_build_kernel(Graph<KT> G, const uint32_t* __restrict__ row_bin) {
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < G.n_rows; r += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t lo = 0;
        uint32_t cap = G.cap0;
        if (G.g_bins > 1) {
            const uint32_t b = row_bin[r];
            lo = G.hoff[b];
            cap = (uint32_t)(G.hoff[b + 1] - lo);
        }
        const uint64_t kh = key_hash(G.keys[r]);
        if (G.bloom_mask) {
            const uint64_t bit = (kh >> 13) & G.bloom_mask;
            atomicOr(&G.bloom[bit >> 5], 1u << (bit & 31u));
        }
        uint32_t slot = (uint32_t)(((uint64_t)(uint32_t)(kh >> 20) * cap) >> 32);
        while (atomicCAS(&G.ht[lo + slot], NONE32, (uint32_t)r) != NONE32) slot = slot + 1 == cap ? 0u : slot + 1;
    }
}

// ---- K5: adjacency, fork filters, links ---------------------------------------------------------------------------
// The index is probed once per oriented k-mer: the adjacency pass stores N(Y), the oriented ids of the 4 possible
// successors suffix(Y)·b of every oriented k-mer Y (slot b, NONE32 where absent), 16 B per oriented id.  Every
// neighbour set the filters and the links need is one of these sets, read at the node or at a neighbour:
//   successors of Y              N(Y)
//   predecessors of Y            { rc(z) : z in N(Y^1) }                 (Y^1: the other strand, the same row)
//   right group  prefix(Y)·b     N(P), P any predecessor of Y           (slot b)
//   left group   a·suffix(Y)     { rc(z) : z in N(S^1) }, S any successor of Y   (slot 3 - a holds rc(a·suffix(Y)))
// so a node costs 4 index probes instead of 10.  A node without a predecessor (successor) has no stored set that names
// its right (left) group; it probes its siblings directly.  On clean data those are the chain ends; on noisy data the
// error tips.
// The even ids' sets are in s[0], the odd ids' in s[1], both indexed by row.
struct Adj {
    uint4* s[2];
    __device__ __forceinline__ uint4* set(uint64_t oid) const { return ((oid & 1u) ? s[1] : s[0]) + (oid >> 1); }  // (a select: no local copy of s)
    __device__ __forceinline__ uint4 out(uint32_t oid) const { return *set(oid); }
};
__device__ __forceinline__ uint32_t adj_slot(const uint4& v, uint32_t b) { return b == 0 ? v.x : b == 1 ? v.y : b == 2 ? v.z : v.w; }

template <class KT> __device__ __forceinline__ bool is_palindrome(const Graph<KT>& G, KT Z) { return !(G.k & 1) && revcomp(Z, G.k) == Z; }
// oriented id of revcomp(Z), given z = find(Z): the other strand of z's row -- except for a palindromic row, which is
// one node: find returns its even id, and the odd id is not a node (alive = 0)
template <class KT> __device__ __forceinline__ uint32_t rc_oid(const Graph<KT>& G, uint32_t z, KT Z) { return is_palindrome(G, Z) ? z : z ^ 1u; }

template <class KT>
__global__ void __launch_bounds__(256) adjacency_kernel(Graph<KT> G, Adj A, uint64_t n) {
    const KT sufmask = mask_bases<KT>(G.k - 1);
    for (uint64_t oid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; oid < n; oid += (uint64_t)gridDim.x * blockDim.x) {
        const KT X = G.oriented((uint32_t)oid);
        const KT suffix = X & sufmask;
        uint32_t pre_min = 0, suf_min = 0;
        if (G.g_bins > 1) G.minima(X, pre_min, suf_min);
        uint32_t s[4];
#pragma unroll
        for (uint32_t b = 0; b < 4; b++) {
            uint32_t cz;
            const uint32_t hl = G.g_bins > 1 ? G.last_mm(suffix, b) : 0u;
            s[b] = G.find((suffix << 2) | (KT)b, hl < suf_min ? hl : suf_min, &cz);
        }
        *A.set(oid) = make_uint4(s[0], s[1], s[2], s[3]);
    }
}

// counts of the group prefix(X)·b by probing the 3 siblings of X (own: X's count)
template <class KT> __device__ __forceinline__ void probe_right_group(const Graph<KT>& G, KT X, uint32_t own, uint32_t cnt[4]) {
    const KT prefix = X >> 2;
    const uint32_t myb = (uint32_t)X & 3u;
    uint32_t pre_min = 0, suf_min = 0;
    if (G.g_bins > 1) G.minima(X, pre_min, suf_min);
#pragma unroll
    for (uint32_t b = 0; b < 4; b++) {
        if (b == myb) { cnt[b] = own; continue; }
        const KT Z = (prefix << 2) | (KT)b;
        const KT zc = revcomp(Z, G.k);
        const uint32_t hl = G.g_bins > 1 ? G.last_mm(prefix, b) : 0u;
        const uint32_t r = G.lookup(zc < Z ? zc : Z, hl < pre_min ? hl : pre_min);
        cnt[b] = r == NONE32 ? 0u : G.counts[r];
    }
}
// counts of the right-filter survivors among a·suffix(X) by probing the 3 siblings of X (own: X's count)
template <class KT> __device__ __forceinline__ void probe_left_group(const Graph<KT>& G, KT X, const uint8_t* alive, uint32_t own, uint32_t cnt[4]) {
    const int top = 2 * (G.k - 1);
    const KT suffix = X & mask_bases<KT>(G.k - 1);
    const uint32_t mya = (uint32_t)(X >> top) & 3u;
    uint32_t pre_min = 0, suf_min = 0;
    if (G.g_bins > 1) G.minima(X, pre_min, suf_min);
#pragma unroll
    for (uint32_t a = 0; a < 4; a++) {
        if (a == mya) { cnt[a] = own; continue; }
        uint32_t cz = 0;
        const uint32_t hf = G.g_bins > 1 ? G.first_mm(suffix, a) : 0u;
        const uint32_t oz = G.find(((KT)a << top) | suffix, hf < suf_min ? hf : suf_min, &cz);
        cnt[a] = (oz != NONE32 && (alive[oz] & 1)) ? cz : 0u;
    }
}

// The alive byte of an oriented k-mer: bit0 survives the right fork filter, bit1 survives both, bit2 right flag < 0,
// bit3 left flag < 0.  The sign bits are all a neighbour needs to know about a node's flags (junction_joins), so in
// a sharded run one byte per node is the only per-node state that crosses GPUs.
//
// A7.
template <class KT>
__global__ void __launch_bounds__(256) right_filter_kernel(Graph<KT> G, Adj A, int E, uint8_t* __restrict__ alive, int32_t* __restrict__ rflag, uint64_t n) {
    const KT sufmask = mask_bases<KT>(G.k - 1);
    for (uint64_t oid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; oid < n; oid += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t row = (uint32_t)(oid >> 1);
        const KT key = G.keys[row];
        const KT rc = revcomp(key, G.k);
        if ((oid & 1u) && rc == key) { alive[oid] = 0; rflag[oid] = 0; continue; }  // palindrome: one node, not two
        const KT X = (oid & 1u) ? rc : key;
        const KT prefix = X >> 2;
        const uint32_t myb = (uint32_t)X & 3u;
        // a predecessor: the reverse complement of a successor of revcomp(X), whose out-set is stored next to X's
        const KT rpre = ((oid & 1u) ? key : rc) & sufmask;  // revcomp(prefix(X))
        const uint4 in = A.out((uint32_t)oid ^ 1u);
        uint32_t z = NONE32, zc = 0;
#pragma unroll
        for (int c = 3; c >= 0; c--)
            if (adj_slot(in, c) != NONE32) { z = adj_slot(in, c); zc = c; }
        const uint32_t own = G.counts[row];
        uint32_t cnt[4];
        if (z != NONE32) {
            const uint4 grp = A.out(rc_oid(G, z, (rpre << 2) | (KT)zc));
#pragma unroll
            for (uint32_t b = 0; b < 4; b++) cnt[b] = b == myb ? own : adj_slot(grp, b) == NONE32 ? 0u : G.counts[adj_slot(grp, b) >> 1];
        } else {
            probe_right_group(G, X, own, cnt);
        }
        bool dup[4];
#pragma unroll
        for (uint32_t b = 0; b < 4; b++) dup[b] = is_palindrome(G, (prefix << 2) | (KT)b);
        const ForkResult res = right_fork(cnt, dup, E, G.k - 1);
        alive[oid] = (uint8_t)(((res.winner == (int)myb) ? 1 : 0) | (res.flag < 0 ? 4 : 0));
        rflag[oid] = res.flag;
    }
}

// A8.
template <class KT>
__global__ void __launch_bounds__(256) left_filter_kernel(Graph<KT> G, Adj A, int E, uint8_t* alive, int32_t* __restrict__ lflag, uint64_t n) {
    const int top = 2 * (G.k - 1);
    const KT sufmask = mask_bases<KT>(G.k - 1);
    for (uint64_t oid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; oid < n; oid += (uint64_t)gridDim.x * blockDim.x) {
        lflag[oid] = 0;
        if (!(alive[oid] & 1)) continue;
        const KT X = G.oriented((uint32_t)oid);
        const KT suffix = X & sufmask;
        const uint32_t mya = (uint32_t)(X >> top) & 3u;
        const uint4 out = A.out((uint32_t)oid);
        uint32_t s = NONE32, sb = 0;
#pragma unroll
        for (int b = 3; b >= 0; b--)
            if (adj_slot(out, b) != NONE32) { s = adj_slot(out, b); sb = b; }
        const uint32_t own = G.counts[oid >> 1];
        uint32_t cnt[4];
        if (s != NONE32) {
            const uint4 grp = A.out(rc_oid(G, s, (suffix << 2) | (KT)sb));
#pragma unroll
            for (uint32_t a = 0; a < 4; a++) {
                const uint32_t z = adj_slot(grp, 3 - a);
                const uint32_t oz = (a == mya || z == NONE32) ? NONE32 : rc_oid(G, z, ((KT)a << top) | suffix);
                cnt[a] = a == mya ? own : (oz != NONE32 && (alive[oz] & 1)) ? G.counts[z >> 1] : 0u;
            }
        } else {
            probe_left_group(G, X, alive, own, cnt);
        }
        const ForkResult res = left_fork(cnt, E, G.k - 1);
        if (res.winner == (int)mya) { alive[oid] = (uint8_t)((alive[oid] & 4) | 3 | (res.flag < 0 ? 8 : 0)); lflag[oid] = res.flag; }
    }
}

// ---- Count_<k>_sorted (SURVEY 8f-2): the fork filters of ReflexivDSKmerLeftAndRightSorting.java ----------------
// Every node probes its siblings in the index; what differs from A7 / A8 is the rule (sorted_right_fork /
// sorted_left_fork, rfx_core.h) and that the left filter needs, from every candidate, the coverage and the right flag the right filter left on it.
template <class KT>
__global__ void sorted_right_kernel(Graph<KT> G, int E, double fold, int X, uint8_t* __restrict__ alive, int32_t* __restrict__ cov, int32_t* __restrict__ rflag,
                                    uint64_t n) {
    for (uint64_t oid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; oid < n; oid += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t row = (uint32_t)(oid >> 1);
        const KT key = G.keys[row];
        const KT rc = revcomp(key, G.k);
        if ((oid & 1u) && rc == key) { alive[oid] = 0; continue; }  // palindrome: one node, not two
        const KT Xk = (oid & 1u) ? rc : key;
        const KT prefix = Xk >> 2;
        const uint32_t myb = (uint32_t)Xk & 3u;
        uint32_t pre_min = 0, suf_min = 0;
        if (G.g_bins > 1) G.minima(Xk, pre_min, suf_min);
        uint32_t cnt[4];
        bool dup[4];
#pragma unroll
        for (uint32_t b = 0; b < 4; b++) {
            if (b == myb) { cnt[b] = G.counts[row]; dup[b] = (rc == key); }
            else {
                const KT Z = (prefix << 2) | (KT)b;
                const KT zc = revcomp(Z, G.k);
                const uint32_t hl = G.g_bins > 1 ? G.last_mm(prefix, b) : 0u;
                const uint32_t r = G.lookup(zc < Z ? zc : Z, hl < pre_min ? hl : pre_min);
                cnt[b] = r == NONE32 ? 0u : G.counts[r];
                dup[b] = (Z == zc);
            }
        }
        const SortedFork res = sorted_right_fork(cnt, dup, E, fold, X);
        const bool won = res.winner == (int)myb;
        alive[oid] = won ? 1 : 0;
        if (won) { cov[oid] = res.left; rflag[oid] = res.right; }
    }
}

template <class KT>
__global__ void sorted_left_kernel(Graph<KT> G, int E, double fold, int X, uint8_t* alive, const int32_t* __restrict__ cov, const int32_t* __restrict__ rflag,
                                   int32_t* __restrict__ out_left, int32_t* __restrict__ out_right, uint64_t n) {
    const int top = 2 * (G.k - 1);
    const KT sufmask = mask_bases<KT>(G.k - 1);
    for (uint64_t oid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; oid < n; oid += (uint64_t)gridDim.x * blockDim.x) {
        if (!(alive[oid] & 1)) continue;
        const KT Xk = G.oriented((uint32_t)oid);
        const KT suffix = Xk & sufmask;
        const uint32_t mya = (uint32_t)(Xk >> top) & 3u;
        uint32_t pre_min = 0, suf_min = 0;
        if (G.g_bins > 1) G.minima(Xk, pre_min, suf_min);
        int32_t cv[4], rf[4];
#pragma unroll
        for (uint32_t a = 0; a < 4; a++) {
            if (a == mya) { cv[a] = cov[oid]; rf[a] = rflag[oid]; }
            else {
                uint32_t cz = 0;
                const uint32_t hf = G.g_bins > 1 ? G.first_mm(suffix, a) : 0u;
                const uint32_t oz = G.find(((KT)a << top) | suffix, hf < suf_min ? hf : suf_min, &cz);
                const bool there = oz != NONE32 && (alive[oz] & 1);
                cv[a] = there ? cov[oz] : 0;
                rf[a] = there ? rflag[oz] : 0;
            }
        }
        const SortedFork res = sorted_left_fork(cv, rf, E, fold, X);
        if (res.winner == (int)mya) { alive[oid] = 3; out_left[oid] = res.left; out_right[oid] = res.right; }  // bit 0 stays: others still read it
    }
}

// Neighbour links.  succ/pred are preset to NONE32.  A node writes its successor's pred[] and EVERY junction is linked
// (raw links): which of them hold is decided afterwards (budget walks + junction_finalize_kernel) and only matters when
// some flag is non-negative, i.e. a real fork survived (DS_FLAGGED).
__global__ void __launch_bounds__(256) link_kernel(Adj A, const uint8_t* __restrict__ alive, const int32_t* __restrict__ lflag, const int32_t* __restrict__ rflag,
                                                   uint32_t* __restrict__ succ, uint32_t* pred, unsigned long long* dstat, uint64_t n) {
    for (uint64_t oid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; oid < n; oid += (uint64_t)gridDim.x * blockDim.x) {
        if (!(alive[oid] & 2)) continue;
        const uint4 out = A.out((uint32_t)oid);
        uint32_t next = NONE32;
        int n_cand = 0;
#pragma unroll
        for (uint32_t b = 0; b < 4; b++) {
            const uint32_t oy = adj_slot(out, b);
            if (oy != NONE32 && (alive[oy] & 2)) { next = oy; n_cand++; }
        }
        if (n_cand > 1) { atomicExch(&dstat[DS_GRAPH_ERR], 1ull); continue; }
        if (lflag[oid] >= 0 || rflag[oid] >= 0) atomicAdd(&dstat[DS_FLAGGED], 1ull);
        if (next != NONE32) {
            const bool joins = junction_joins(rflag[oid], lflag[next]);
            if (!joins) atomicAdd(&dstat[DS_BUDGET], 1ull);
            if (next == (uint32_t)oid) {
                if (joins) atomicAdd(&dstat[DS_CYCLES], 1ull);  // 1-cycle: a record never merges with itself
            } else {
                succ[oid] = next;
                if (atomicExch(&pred[next], (uint32_t)oid) != NONE32) atomicExch(&dstat[DS_GRAPH_ERR], 2ull);
            }
        }
    }
}

// ---- budget walks (A9, clauses 3 / 4: ReflexivDSMain.java:3077-3084, flag rule of reflexivExtend :3265-3279) ----------
// A fork winner's flag k-1 facing a clean end is a budget: the flagged fragment absorbs clean k-mers one at a time, the
// budget shrinks by one per k-mer and overwrites the flag of the new outer end; it stops in front of a non-negative
// facing flag (clause 2 joins there) or when it is used up.  Canonical schedule (DESIGN.md, oracle: budget_scan): along
// a path   E(v) = (face(v) < 0 && E(prev(v)) >= 1) ? E(prev(v)) - 1 : budget(v),   once along succ (budget = right flag,
// face = left flag) and once along pred.  Fork winners are rare, so the recurrence is evaluated from them: a thread per
// node with a budget first decides whether an upstream walk absorbs it (it looks upstream until a node that cannot be
// absorbed, a path end, or k-1 budget-less nodes in a row -- no walk survives those), then, if not, walks downstream
// writing the effective flags of what it absorbs and marking the junctions it went through (alive bit 4 / 5 on the
// junction's left node).  On a closed path where every walk may wrap around, the fork winner with the smallest oriented
// k-mer starts fresh (oracle: loop_start).
template <class KT, int DIR>
__global__ void budget_walk_kernel(Graph<KT> G, uint64_t n, uint8_t* alive, const int32_t* __restrict__ bud, const int32_t* __restrict__ face,
                                   const uint32_t* __restrict__ nxt, const uint32_t* __restrict__ prv, int32_t* eff, int bmax, unsigned long long* dstat) {
    for (uint64_t x = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; x < n; x += (uint64_t)gridDim.x * blockDim.x) {
        if (!(alive[x] & 2) || bud[x] < 0) continue;
        const uint32_t s = (uint32_t)x;
        if (nxt[s] == NONE32) continue;  // nothing downstream to absorb
        uint32_t stop = s;
        bool fresh = true;
        if (face[s] < 0 && prv[s] != NONE32) {
            uint32_t u = prv[s], start = NONE32;
            int gap = 0;
            while (true) {
                if (u == s) break;  // closed path without a fixed point: smallest fork winner starts
                gap = bud[u] < 0 ? gap + 1 : 0;
                if (face[u] >= 0 || prv[u] == NONE32 || gap >= bmax) { start = u; break; }
                u = prv[u];
            }
            if (start == NONE32) {
                uint32_t m = s;
                KT mk = G.oriented(s);
                for (u = prv[s]; u != s; u = prv[u])
                    if (bud[u] >= 0) { const KT ku = G.oriented(u); if (ku < mk) { mk = ku; m = u; } }
                start = m;
                stop = m;
            }
            if (start != s) {
                int32_t E = bud[start];
                for (uint32_t v = nxt[start]; v != s; v = nxt[v]) E = (face[v] < 0 && E >= 1) ? E - 1 : bud[v];
                fresh = !(E >= 1);  // face[s] < 0 here
            }
        }
        if (!fresh) continue;  // absorbed: the walk that takes it writes its flag
        int32_t rem = bud[s];
        uint32_t cur = s;
        unsigned long long taken = 0;
        while (rem >= 1) {
            const uint32_t z = nxt[cur];
            if (z == NONE32 || z == stop || z == s || face[z] >= 0) break;
            rem--;
            eff[z] = rem;
            alive_or(alive, DIR == 0 ? cur : z, DIR == 0 ? 16u : 32u);
            taken++;
            cur = z;
        }
        if (taken) atomicAdd(&dstat[DS_ABSORBED], taken);
    }
}
// which junctions hold: a walk went through, or the effective flags have the same sign
__global__ void junction_finalize_kernel(uint64_t n, const uint8_t* __restrict__ alive, const int32_t* __restrict__ eff_l, const int32_t* __restrict__ eff_r,
                                         uint32_t* succ, uint32_t* pred) {
    for (uint64_t x = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; x < n; x += (uint64_t)gridDim.x * blockDim.x) {
        if (!(alive[x] & 2)) continue;
        const uint32_t y = succ[x];
        if (y == NONE32) continue;
        if ((alive[x] & 48) || junction_joins(eff_r[x], eff_l[y])) continue;
        succ[x] = NONE32;
        pred[y] = NONE32;
    }
}

// ---- K6: pointer jumping towards the head ------------------------------------------------------
// One 64-bit word per node: low half = current ancestor, high half = distance to it, so a jump costs one random
// 8-byte read.  Double buffered (Jacobi), so every round is deterministic.

__global__ void rank_init_kernel(uint64_t n, const uint32_t* __restrict__ pred, uint64_t* __restrict__ ad) {
    for (uint64_t x = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; x < n; x += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t p = pred[x];
        ad[x] = p == NONE32 ? ad_pack((uint32_t)x, 0u) : ad_pack(p, 1u);
    }
}
__global__ void rank_step_kernel(uint64_t n, const uint64_t* __restrict__ ad_in, uint64_t* __restrict__ ad_out, unsigned long long* dstat) {
    bool changed = false;
    for (uint64_t x = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; x < n; x += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t mine = ad_in[x];
        const uint32_t a = (uint32_t)mine;
        if (a == (uint32_t)x) { ad_out[x] = mine; continue; }
        const uint64_t up = ad_in[a];
        const uint32_t aa = (uint32_t)up;
        ad_out[x] = ad_pack(aa, (uint32_t)(mine >> 32) + (uint32_t)(up >> 32));
        changed |= (aa != a);
    }
    if (__any_sync(0xffffffffu, changed) && (threadIdx.x & 31) == 0) atomicExch(&dstat[DS_CHANGED], 1ull);
}
// All pointer-jumping rounds over the splitter list in ONE cooperative launch: the list is small (a few MB), so a round
// is a few microseconds of work and what used to cost was 20-odd launches and the host reading a "changed" flag every
// fourth one.  Grid-wide barrier between rounds; three rotating flags tell every block whether the round changed
// anything (a flag is cleared one round before it is used and read one round after).
__global__ void __launch_bounds__(256) rank_all_kernel(const unsigned long long* m_ptr, uint64_t* ad0, uint64_t* ad1, unsigned long long* dstat) {
    cooperative_groups::grid_group grid = cooperative_groups::this_grid();
    const uint64_t m = *m_ptr;
    int max_rounds = 2;
    while ((1ull << max_rounds) < m + 1) max_rounds++;
    max_rounds += 2;
    unsigned long long* flags = dstat + DS_RANK_FLAGS;
    uint64_t* in = ad0;
    uint64_t* out = ad1;
    int cur = 0;
    for (int round = 0; round < max_rounds; round++) {
        if (blockIdx.x == 0 && threadIdx.x == 0) flags[(round + 1) % 3] = 0ull;
        bool changed = false;
        for (uint64_t x = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; x < m; x += (uint64_t)gridDim.x * blockDim.x) {
            const uint64_t mine = in[x];
            const uint32_t a = (uint32_t)mine;
            if (a == (uint32_t)x) { out[x] = mine; continue; }
            const uint64_t up = in[a];
            const uint32_t aa = (uint32_t)up;
            out[x] = ad_pack(aa, (uint32_t)(mine >> 32) + (uint32_t)(up >> 32));
            changed |= (aa != a);
        }
        if (__any_sync(0xffffffffu, changed) && (threadIdx.x & 31) == 0) atomicExch(&flags[round % 3], 1ull);
        grid.sync();
        uint64_t* t = in; in = out; out = t;
        cur ^= 1;
        if (*(volatile unsigned long long*)&flags[round % 3] == 0ull) break;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) dstat[DS_RANK_CUR] = (unsigned long long)cur;
}

// ---- K6 (work-efficient variant): rank through a sample of splitters ------------------------------------------
// Heads and one node in 16 (hash of the id) are splitters.  Each splitter walks its successors up to the next
// splitter, stamping (owner, offset) on the way: every node is touched once.  Only the splitter list (n/16 entries,
// L2 resident) goes through pointer jumping; a last pass adds the offsets.  ~2 random accesses per node instead of
// one per node per round.
__device__ __forceinline__ bool is_random_splitter(uint32_t x) { return (fmix32(x ^ 0xa5a5a5a5u) & 15u) == 0u; }

__global__ void splitter_select_kernel(uint64_t n, const uint8_t* __restrict__ alive, const uint32_t* __restrict__ pred, uint32_t* __restrict__ spl_id,
                                       uint32_t* __restrict__ spl_node, uint64_t* __restrict__ sp_ad, unsigned long long* dstat) {
    for (uint64_t x = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; x < n; x += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t id = NONE32;
        if ((alive[x] & 2) && (pred[x] == NONE32 || is_random_splitter((uint32_t)x))) {
            id = (uint32_t)atomicAdd(&dstat[DS_NSPL], 1ull);
            spl_node[id] = (uint32_t)x;
            sp_ad[id] = ad_pack(id, 0u);
        }
        spl_id[x] = id;
    }
}
__global__ void splitter_walk_kernel(const unsigned long long* m_ptr, const uint32_t* __restrict__ spl_node, const uint32_t* __restrict__ succ,
                                     const uint32_t* __restrict__ spl_id, uint64_t* __restrict__ loc, uint64_t* sp_ad) {
    const uint64_t m = *m_ptr;  // number of splitters, still on the device: no host round trip between select and walk
    for (uint64_t id = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; id < m; id += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t x = spl_node[id];
        uint32_t off = 0;
        loc[x] = ad_pack((uint32_t)id, 0u);
        uint32_t y = succ[x];
        while (y != NONE32) {
            // a node with a predecessor is a splitter iff its id hashes to one (heads are never walked into)
            if (is_random_splitter(y)) { sp_ad[spl_id[y]] = ad_pack((uint32_t)id, off + 1u); break; }  // my segment ends in front of it
            off++;
            loc[y] = ad_pack((uint32_t)id, off);
            y = succ[y];
        }
    }
}
__global__ void rank_finalize_kernel(uint64_t n, const uint8_t* __restrict__ alive, const uint32_t* __restrict__ pred, const uint64_t* __restrict__ loc,
                                     const uint64_t* sp_ad0, const uint64_t* sp_ad1, const uint32_t* __restrict__ spl_node, uint64_t* __restrict__ ad,
                                     unsigned long long* dstat) {
    const uint64_t* sp_ad = dstat[DS_RANK_CUR] ? sp_ad1 : sp_ad0;
    bool on_cycle = false;
    for (uint64_t x = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; x < n; x += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t l = loc[x];
        if (!(alive[x] & 2)) { ad[x] = ad_pack((uint32_t)x, 0u); continue; }
        if (l == ~0ull) { ad[x] = ad_pack((uint32_t)x, 0u); on_cycle = true; continue; }  // never reached: cycle without a splitter
        const uint64_t v = sp_ad[(uint32_t)l];
        const uint32_t head = spl_node[(uint32_t)v];
        ad[x] = ad_pack(head, (uint32_t)(v >> 32) + (uint32_t)(l >> 32));
        if ((l >> 32) == 0) on_cycle |= pred[head] != NONE32;  // splitters check that their chain's head really is one
    }
    if (__any_sync(0xffffffffu, on_cycle) && (threadIdx.x & 31) == 0) atomicExch(&dstat[DS_CYCLE_NODES], 1ull);
}

// nodes whose final ancestor is not a true head (pred == NONE) sit on a cycle
__global__ void cycle_mark_kernel(uint64_t n, const uint8_t* __restrict__ alive, const uint32_t* __restrict__ pred, const uint64_t* __restrict__ ad,
                                  uint32_t* __restrict__ lab, uint32_t* __restrict__ ptr, unsigned long long* dstat) {
    for (uint64_t x = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; x < n; x += (uint64_t)gridDim.x * blockDim.x) {
        const bool cyc = (alive[x] & 2) && pred[x] != NONE32 && pred[(uint32_t)ad[x]] != NONE32;
        lab[x] = cyc ? (uint32_t)x : NONE32;
        ptr[x] = cyc ? pred[x] : NONE32;
        if (cyc) atomicAdd(&dstat[DS_CYCLE_NODES], 1ull);
    }
}
template <class KT>
__global__ void cycle_min_step_kernel(Graph<KT> G, const uint32_t* __restrict__ lab_in, const uint32_t* __restrict__ ptr_in,
                                      uint32_t* __restrict__ lab_out, uint32_t* __restrict__ ptr_out) {
    const uint64_t n = 2 * G.n_rows;
    for (uint64_t x = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; x < n; x += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t p = ptr_in[x];
        if (p == NONE32) { lab_out[x] = NONE32; ptr_out[x] = NONE32; continue; }
        const uint32_t la = lab_in[x], lb = lab_in[p];
        lab_out[x] = (la == lb || G.oriented(la) < G.oriented(lb)) ? la : lb;
        ptr_out[x] = ptr_in[p];
    }
}
// CANONICAL ORDER: a cycle is opened in front of its smallest oriented k-mer (oracle: assemble_canonical)
__global__ void cycle_cut_kernel(uint64_t n, const uint32_t* __restrict__ lab, uint32_t* succ, uint32_t* pred, unsigned long long* dstat) {
    for (uint64_t x = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; x < n; x += (uint64_t)gridDim.x * blockDim.x) {
        if (lab[x] == (uint32_t)x) {
            const uint32_t p = pred[x];
            succ[p] = NONE32;
            pred[x] = NONE32;
            atomicAdd(&dstat[DS_CYCLES], 1ull);
        }
    }
}

__global__ void tails_kernel(uint64_t n, const uint8_t* __restrict__ alive, const uint32_t* __restrict__ succ, const uint64_t* __restrict__ ad,
                             uint32_t* __restrict__ chain_len, uint32_t* __restrict__ tail_of) {
    for (uint64_t x = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; x < n; x += (uint64_t)gridDim.x * blockDim.x) {
        if ((alive[x] & 2) && succ[x] == NONE32) {
            const uint64_t v = ad[x];
            const uint32_t h = (uint32_t)v;
            chain_len[h] = (uint32_t)(v >> 32) + 1u;
            tail_of[h] = (uint32_t)x;
        }
    }
}

// ---- K7: contigs ----------------------------------------------------------------------------------
struct ContigIn {
    const uint8_t* alive;
    const uint32_t* pred;
    const uint32_t* chain_len;
    const uint32_t* tail_of;
    const int32_t* lflag;
    const int32_t* rflag;
    int k, min_contig;
    __device__ __forceinline__ U64x3 operator()(uint64_t x) const {
        if (!(alive[x] & 2)) return U64x3{0, 0, 0};
        if (pred[x] != NONE32) return U64x3{0, 0, 1};
        const uint64_t len = (uint64_t)chain_len[x] + (uint64_t)k - 1;
        // DSKmerToContig, ReflexivDSMain.java:749-754
        const bool keep = !(lflag[x] <= -10000000 && rflag[tail_of[x]] <= -10000000) && len >= (uint64_t)min_contig;
        return keep ? U64x3{1, len, 1} : U64x3{0, 0, 1};
    }
};
struct ContigOut {
    const uint32_t* tail_of;
    const int32_t* lflag;
    const int32_t* rflag;
    uint32_t* ctg_idx;
    uint64_t* ctg_off;
    int32_t* ctg_left;
    int32_t* ctg_right;
    __device__ __forceinline__ void operator()(uint64_t x, U64x3 excl, U64x3 v) const {
        ctg_idx[x] = v.a ? (uint32_t)excl.a : NONE32;
        if (v.a) {
            ctg_off[excl.a] = excl.b;
            ctg_left[excl.a] = lflag[x];
            ctg_right[excl.a] = rflag[tail_of[x]];
        }
    }
};

template <class KT>
__global__ void gather_contigs_kernel(Graph<KT> G, const uint8_t* __restrict__ alive, const uint64_t* __restrict__ ad,
                                      const uint32_t* __restrict__ ctg_idx, const uint64_t* __restrict__ ctg_off, char* __restrict__ out) {
    const uint64_t n = 2 * G.n_rows;
    for (uint64_t x = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; x < n; x += (uint64_t)gridDim.x * blockDim.x) {
        if (!(alive[x] & 2)) continue;
        const uint64_t v = ad[x];
        const uint32_t h = (uint32_t)v;
        const uint32_t ci = ctg_idx[h];
        if (ci == NONE32) continue;
        const KT X = G.oriented((uint32_t)x);
        char* dst = out + ctg_off[ci];
        dst[(uint64_t)(G.k - 1) + (uint32_t)(v >> 32)] = "ACGT"[(uint32_t)X & 3u];
        if (h == (uint32_t)x)
            for (int j = 0; j < G.k - 1; j++) dst[j] = "ACGT"[(uint32_t)(X >> (2 * (G.k - 1 - j))) & 3u];
    }
}

__global__ void set_u64_kernel(uint64_t* p, const U64x3* tot) { *p = tot->b; }
__global__ void set_value_kernel(unsigned long long* p, unsigned long long v) { *p = v; }

struct AliveBoth {
    const uint8_t* alive;
    __device__ __forceinline__ uint64_t operator()(uint64_t x) const { return (alive[x] & 2) ? 1 : 0; }
};

static unsigned grid_n(uint64_t n) {
    uint64_t g = (n + 255) / 256;
    if (g < 1) g = 1;
    const uint64_t cap = (uint64_t)sm_count() * 16u;
    return (unsigned)(g > cap ? cap : g);
}

template <class KT> static Graph<KT> make_graph(Ctx* c) {
    return Graph<KT>{c->keys.as<KT>(), c->counts.as<uint32_t>(), c->n_rows, c->ht.as<uint32_t>(), c->g_hoff.as<uint64_t>(), c->g_bins, c->g_bins > 1 ? 0u : (uint32_t)c->ht_cap, c->k, c->g_m,
                     c->g_bloom.as<uint32_t>(), c->g_bloom_mask};
}

// builds the bin-local index over the whole table (asynchronous on the context's stream)
template <class KT> static int build_index(Ctx* c) {
    cudaStream_t st = c->stream;
    const uint64_t n_rows = c->n_rows;
    // Presence bits (>= 16 per row) answer most probes as long as they stay (mostly) cache resident: up to 2^30 bits
    // (128 MB, 64 M rows) the table is ONE region behind that filter.  Beyond that a filter access is just one more
    // trip to HBM (measured at 1.5 * 10^8 rows: 102 ms with it, 76 ms without), and what helps instead is locality:
    // regions per minimiser bin, no filter.
    uint64_t bits = 1024;
    while (bits < 16 * n_rows) bits <<= 1;
    const char* force = getenv("RFX_GRAPH_INDEX");  // "local" / "global": tests exercise both on small inputs
    const bool local = force ? !strcmp(force, "local") : bits > (1024ull << 20);
    uint64_t gb = n_rows / 32;
    if (gb < 64) gb = 64;
    if (gb > (1ull << 26)) gb = 1ull << 26;
    if (!local) gb = 1;
    c->g_bins = (uint32_t)gb;
    int m = gb > 65536 ? 15 : 11;  // many more minimiser values than bins (as in rfx_partition.cu: set_minimizer)
    if (m > c->k - 1) m = c->k - 1;
    c->g_m = m;
    RFX_TRY(devbuf_reserve(c, c->g_rowbin, (n_rows + 1) * sizeof(uint32_t)));
    RFX_TRY(devbuf_reserve(c, c->g_binrows, gb * sizeof(uint32_t)));
    RFX_TRY(devbuf_reserve(c, c->g_hoff, (gb + 1) * sizeof(uint64_t)));
    const uint64_t slots = 4 * n_rows + 2 * gb;  // load factor <= 1/4 in every region: most probes are for absent neighbours
    RFX_TRY(devbuf_reserve(c, c->ht, slots * sizeof(uint32_t)));
    c->ht_cap = slots;
    RFX_CUDA(c, cudaMemsetAsync(c->ht.p, 0xff, slots * sizeof(uint32_t), st));
    c->g_bloom_mask = (!local || force) && bits <= (1024ull << 20) ? bits - 1 : 0;
    if (c->g_bloom_mask) {
        RFX_TRY(devbuf_reserve(c, c->g_bloom, bits / 8));
        RFX_CUDA(c, cudaMemsetAsync(c->g_bloom.p, 0, bits / 8, st));
    }
    Graph<KT> G = make_graph<KT>(c);
    if (local) {
        RFX_CUDA(c, cudaMemsetAsync(c->g_binrows.p, 0, gb * sizeof(uint32_t), st));
        if (n_rows) row_bin_kernel<KT><<<grid_n(n_rows), 256, 0, st>>>(G, c->g_rowbin.as<uint32_t>(), c->g_binrows.as<uint32_t>());
        ScanPlan<uint64_t> plan;
        RFX_TRY(devbuf_reserve(c, c->scan_ws, ScanPlan<uint64_t>::workspace_elems(gb) * sizeof(uint64_t)));
        plan.bind(gb, c->scan_ws.as<uint64_t>());
        RegionIn in{c->g_binrows.as<uint32_t>()};
        scan_prepare(plan, in, OpAddU64{}, (uint64_t)0, st);
        scan_apply(plan, in, RegionOut{c->g_hoff.as<uint64_t>()}, OpAddU64{}, (uint64_t)0, st);
        set_last_region_kernel<<<1, 1, 0, st>>>(c->g_hoff.as<uint64_t>(), gb, plan.total);
        c->launches += 2 + 2 * plan.levels;
    }
    if (n_rows) ht_build_kernel<KT><<<grid_n(n_rows), 256, 0, st>>>(G, c->g_rowbin.as<uint32_t>());
    c->launches++;
    return RFX_OK;
}

template <class KT> static int graph_impl(Ctx* c) {
    cudaStream_t st = c->stream;
    const uint64_t n_rows = c->n_rows, n = 2 * n_rows;
    unsigned long long* dstat = c->dstat.as<unsigned long long>();
    uint64_t h[DS_NSLOTS];
    RFX_CUDA(c, cudaMemsetAsync(c->dstat.p, 0, DS_NSLOTS * sizeof(uint64_t), st));
    c->n_oriented = c->n_budget = c->n_budget_adm = c->n_cycles = c->n_contigs = c->n_contig_bases = 0;
    c->have_sorted = false;  // index, alive bytes and flag arrays are rebuilt below
    if (n_rows == 0) {
        RFX_TRY(devbuf_reserve(c, c->ctg_off, sizeof(uint64_t)));
        RFX_CUDA(c, cudaMemsetAsync(c->ctg_off.p, 0, sizeof(uint64_t), st));
        c->have_contigs = true;
        return RFX_OK;
    }
    if (n >= 0xffffffffull) return ctx_fail(c, RFX_E_CAPACITY, "more than 2^31 rows: oriented ids do not fit 32 bits");

    // ---- K5 ----
    stage_begin(c);
    RFX_TRY(devbuf_reserve(c, c->rflag, n * sizeof(int32_t)));
    RFX_TRY(devbuf_reserve(c, c->lflag, n * sizeof(int32_t)));
    RFX_TRY(devbuf_reserve(c, c->alive, n));
    RFX_TRY(devbuf_reserve(c, c->succ, n * sizeof(uint32_t)));
    RFX_TRY(devbuf_reserve(c, c->pred, n * sizeof(uint32_t)));
    RFX_TRY(devbuf_reserve(c, c->tail_of, n * sizeof(uint32_t)));  // doubles as open_next until the tails pass
    RFX_TRY(devbuf_reserve(c, c->ad[0], n * sizeof(uint64_t)));
    for (int i = 0; i < 2; i++) RFX_TRY(devbuf_reserve(c, c->sp_ad[i], n * sizeof(uint64_t)));
    RFX_TRY(devbuf_reserve(c, c->spl_id, n * sizeof(uint32_t)));
    RFX_TRY(devbuf_reserve(c, c->spl_node, n * sizeof(uint32_t)));
    RFX_TRY(devbuf_reserve(c, c->loc, n * sizeof(uint64_t)));
    RFX_TRY(devbuf_reserve(c, c->chain_len, n * sizeof(uint32_t)));
    RFX_TRY(devbuf_reserve(c, c->ctg_idx, n * sizeof(uint32_t)));
    int rc = RFX_OK;
    do {
        if ((rc = build_index<KT>(c)) != RFX_OK) break;
        Graph<KT> G = make_graph<KT>(c);
        cudaMemsetAsync(c->succ.p, 0xff, n * sizeof(uint32_t), st);
        cudaMemsetAsync(c->pred.p, 0xff, n * sizeof(uint32_t), st);
        cudaMemsetAsync(c->chain_len.p, 0, n * sizeof(uint32_t), st);
        cudaMemsetAsync(c->tail_of.p, 0xff, n * sizeof(uint32_t), st);
        const int E = c->prm.min_error_coverage;
        uint8_t* alive = c->alive.as<uint8_t>();
        int32_t* lflag = c->lflag.as<int32_t>();
        int32_t* rflag = c->rflag.as<int32_t>();
        uint32_t* succ = c->succ.as<uint32_t>();
        uint32_t* pred = c->pred.as<uint32_t>();
        // the out-sets live in the splitter buffers, which nothing reads before K6 writes them
        const Adj A{{c->sp_ad[0].as<uint4>(), c->sp_ad[1].as<uint4>()}};
        adjacency_kernel<KT><<<grid_n(n), 256, 0, st>>>(G, A, n);
        right_filter_kernel<KT><<<grid_n(n), 256, 0, st>>>(G, A, E, alive, rflag, n);
        left_filter_kernel<KT><<<grid_n(n), 256, 0, st>>>(G, A, E, alive, lflag, n);
        link_kernel<<<grid_n(n), 256, 0, st>>>(A, alive, lflag, rflag, succ, pred, dstat, n);
        c->launches += 4;
        cudaMemcpyAsync(h, c->dstat.p, sizeof(h), cudaMemcpyDeviceToHost, st);
        cudaError_t e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) { rc = ctx_fail(c, RFX_E_CUDA, "graph kernels failed: %s", cudaGetErrorString(e)); break; }
        c->ms[3] += stage_end(c);
        if (h[DS_GRAPH_ERR]) { rc = ctx_fail(c, RFX_E_GRAPH, "fork filters left a (k-1)-mer with degree > 1 (code %llu)", (unsigned long long)h[DS_GRAPH_ERR]); break; }
        c->n_budget = h[DS_BUDGET];
        if (h[DS_FLAGGED]) {
            // real forks survived the filters: budget walks, then cut the junctions that do not hold (still part of K5's time)
            stage_begin(c);
            if ((rc = devbuf_reserve(c, c->eff_l, n * sizeof(int32_t))) != RFX_OK) break;
            if ((rc = devbuf_reserve(c, c->eff_r, n * sizeof(int32_t))) != RFX_OK) break;
            cudaMemcpyAsync(c->eff_l.p, lflag, n * sizeof(int32_t), cudaMemcpyDeviceToDevice, st);
            cudaMemcpyAsync(c->eff_r.p, rflag, n * sizeof(int32_t), cudaMemcpyDeviceToDevice, st);
            budget_walk_kernel<KT, 0><<<grid_n(n), 256, 0, st>>>(G, n, alive, rflag, lflag, succ, pred, c->eff_r.as<int32_t>(), c->k - 1, dstat);
            budget_walk_kernel<KT, 1><<<grid_n(n), 256, 0, st>>>(G, n, alive, lflag, rflag, pred, succ, c->eff_l.as<int32_t>(), c->k - 1, dstat);
            junction_finalize_kernel<<<grid_n(n), 256, 0, st>>>(n, alive, c->eff_l.as<int32_t>(), c->eff_r.as<int32_t>(), succ, pred);
            c->launches += 3;
            e = cudaStreamSynchronize(st);
            if (e != cudaSuccess) { rc = ctx_fail(c, RFX_E_CUDA, "budget walks failed: %s", cudaGetErrorString(e)); break; }
            c->ms[3] += stage_end(c);
            lflag = c->eff_l.as<int32_t>();  // the contig stage reads the effective flags of heads and tails
            rflag = c->eff_r.as<int32_t>();
        }

        // ---- K6 ----
        stage_begin(c);
        int limit = 2;
        while ((1ull << limit) < n + 1) limit++;
        limit += 2;
        int cur = 0;
        for (int attempt = 0; attempt < 2; attempt++) {
            cur = 0;
            {
                uint32_t* spl_id = c->spl_id.as<uint32_t>();
                uint32_t* spl_node = c->spl_node.as<uint32_t>();
                uint64_t* loc = c->loc.as<uint64_t>();
                cudaMemsetAsync(dstat + DS_NSPL, 0, sizeof(uint64_t), st);
                cudaMemsetAsync(loc, 0xff, n * sizeof(uint64_t), st);
                splitter_select_kernel<<<grid_n(n), 256, 0, st>>>(n, alive, pred, spl_id, spl_node, c->sp_ad[0].as<uint64_t>(), dstat);
                // select -> walk -> jumping rounds -> finalize; the splitter count stays on the device
                splitter_walk_kernel<<<sm_count() * 16, 256, 0, st>>>(dstat + DS_NSPL, spl_node, succ, spl_id, loc, c->sp_ad[0].as<uint64_t>());
                cudaMemsetAsync(dstat + DS_RANK_FLAGS, 0, 3 * sizeof(uint64_t), st);
                cudaMemsetAsync(dstat + DS_RANK_CUR, 0, sizeof(uint64_t), st);
                if (n <= (16ull << 20) && !c->arena) {  // (a rank of a sharded run may share its device with a peer that waits in a barrier: no co-resident grid)
                    // up to ~10^6 splitters: every round in one cooperative launch, no host round trip at all
                    const unsigned long long* m_ptr = dstat + DS_NSPL;
                    uint64_t* a0 = c->sp_ad[0].as<uint64_t>();
                    uint64_t* a1 = c->sp_ad[1].as<uint64_t>();
                    unsigned long long* ds = dstat;
                    void* args[] = {(void*)&m_ptr, (void*)&a0, (void*)&a1, (void*)&ds};
                    e = cudaLaunchCooperativeKernel((void*)rank_all_kernel, dim3(sm_count() * 4), dim3(256), args, 0, st);
                    if (e != cudaSuccess) break;
                } else {
                    // long lists: one launch per round over as many threads as entries (the co-resident grid of the
                    // cooperative kernel has too few loads in flight); the host looks at the "changed" flag every 4 rounds
                    uint64_t m = 0;
                    cudaMemcpyAsync(&m, dstat + DS_NSPL, sizeof(uint64_t), cudaMemcpyDeviceToHost, st);
                    e = cudaStreamSynchronize(st);
                    if (e != cudaSuccess) break;
                    int scur = 0;
                    if (m) {
                        int slimit = 2;
                        while ((1ull << slimit) < m + 1) slimit++;
                        slimit += 2;
                        for (int round = 0; round < slimit;) {
                            cudaMemsetAsync(dstat + DS_CHANGED, 0, sizeof(uint64_t), st);
                            for (int q = 0; q < 4 && round < slimit; q++, round++) {
                                rank_step_kernel<<<grid_n(m), 256, 0, st>>>(m, c->sp_ad[scur].as<uint64_t>(), c->sp_ad[scur ^ 1].as<uint64_t>(), dstat);
                                c->launches++;
                                scur ^= 1;
                            }
                            uint64_t changed = 0;
                            cudaMemcpyAsync(&changed, dstat + DS_CHANGED, sizeof(uint64_t), cudaMemcpyDeviceToHost, st);
                            e = cudaStreamSynchronize(st);
                            if (e != cudaSuccess) break;
                            if (!changed) break;
                        }
                        if (e != cudaSuccess) break;
                    }
                    set_value_kernel<<<1, 1, 0, st>>>(dstat + DS_RANK_CUR, (unsigned long long)scur);
                }
                cudaMemsetAsync(dstat + DS_CYCLE_NODES, 0, sizeof(uint64_t), st);
                rank_finalize_kernel<<<grid_n(n), 256, 0, st>>>(n, alive, pred, loc, c->sp_ad[0].as<uint64_t>(), c->sp_ad[1].as<uint64_t>(), spl_node, c->ad[0].as<uint64_t>(), dstat);
                c->launches++;
                c->launches += 3;
                uint64_t any_cycle = 0;
                cudaMemcpyAsync(&any_cycle, dstat + DS_CYCLE_NODES, sizeof(uint64_t), cudaMemcpyDeviceToHost, st);
                e = cudaStreamSynchronize(st);
                if (e != cudaSuccess || !any_cycle) break;
            }
            if (attempt == 1) break;
            // cycles: every junction of a closed path joins, no node is a head
            RFX_TRY(devbuf_reserve(c, c->cmin[0], 2 * n * sizeof(uint32_t)));
            RFX_TRY(devbuf_reserve(c, c->cmin[1], 2 * n * sizeof(uint32_t)));
            uint32_t* lab[2] = {c->cmin[0].as<uint32_t>(), c->cmin[1].as<uint32_t>()};
            uint32_t* ptr[2] = {lab[0] + n, lab[1] + n};
            cudaMemsetAsync(dstat + DS_CYCLE_NODES, 0, sizeof(uint64_t), st);
            cycle_mark_kernel<<<grid_n(n), 256, 0, st>>>(n, alive, pred, c->ad[cur].as<uint64_t>(), lab[0], ptr[0], dstat);
            c->launches++;
            uint64_t cyc_nodes = 0;
            cudaMemcpyAsync(&cyc_nodes, dstat + DS_CYCLE_NODES, sizeof(uint64_t), cudaMemcpyDeviceToHost, st);
            e = cudaStreamSynchronize(st);
            if (e != cudaSuccess || cyc_nodes == 0) break;
            int b = 0;
            for (int round = 0; round < limit; round++) {
                cycle_min_step_kernel<KT><<<grid_n(n), 256, 0, st>>>(G, lab[b], ptr[b], lab[b ^ 1], ptr[b ^ 1]);
                c->launches++;
                b ^= 1;
            }
            cycle_cut_kernel<<<grid_n(n), 256, 0, st>>>(n, lab[b], succ, pred, dstat);
            c->launches++;
        }
        if (e != cudaSuccess) { rc = ctx_fail(c, RFX_E_CUDA, "list ranking failed: %s", cudaGetErrorString(e)); break; }
        const uint64_t* ad = c->ad[cur].as<uint64_t>();
        tails_kernel<<<grid_n(n), 256, 0, st>>>(n, alive, succ, ad, c->chain_len.as<uint32_t>(), c->tail_of.as<uint32_t>());
        c->launches += 1;
        e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) { rc = ctx_fail(c, RFX_E_CUDA, "chain kernels failed: %s", cudaGetErrorString(e)); break; }
        c->ms[4] += stage_end(c);

        // ---- K7 ----
        stage_begin(c);
        ScanPlan<U64x3> plan;
        if ((rc = devbuf_reserve(c, c->scan_ws, ScanPlan<U64x3>::workspace_elems(n) * sizeof(U64x3))) != RFX_OK) break;
        plan.bind(n, c->scan_ws.as<U64x3>());
        ContigIn in{alive, pred, c->chain_len.as<uint32_t>(), c->tail_of.as<uint32_t>(), lflag, rflag, c->k, c->prm.min_contig};
        scan_prepare(plan, in, OpAddU64x3{}, U64x3{0, 0, 0}, st);
        c->launches += 2 * plan.levels;
        U64x3 tot;
        cudaMemcpyAsync(&tot, plan.total, sizeof(tot), cudaMemcpyDeviceToHost, st);
        cudaMemcpyAsync(h, c->dstat.p, sizeof(h), cudaMemcpyDeviceToHost, st);
        e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) { rc = ctx_fail(c, RFX_E_CUDA, "contig scan failed: %s", cudaGetErrorString(e)); break; }
        if ((rc = devbuf_reserve(c, c->ctg_off, (tot.a + 1) * sizeof(uint64_t))) != RFX_OK) break;
        if ((rc = devbuf_reserve(c, c->ctg_left, (tot.a + 1) * sizeof(int32_t))) != RFX_OK) break;
        if ((rc = devbuf_reserve(c, c->ctg_right, (tot.a + 1) * sizeof(int32_t))) != RFX_OK) break;
        if ((rc = devbuf_reserve(c, c->ctg_bases, tot.b + 16)) != RFX_OK) break;
        ContigOut out{c->tail_of.as<uint32_t>(), lflag, rflag, c->ctg_idx.as<uint32_t>(), c->ctg_off.as<uint64_t>(), c->ctg_left.as<int32_t>(),
                      c->ctg_right.as<int32_t>()};
        scan_apply(plan, in, out, OpAddU64x3{}, U64x3{0, 0, 0}, st);
        set_u64_kernel<<<1, 1, 0, st>>>(c->ctg_off.as<uint64_t>() + tot.a, plan.total);
        gather_contigs_kernel<KT><<<grid_n(n), 256, 0, st>>>(G, alive, ad, c->ctg_idx.as<uint32_t>(), c->ctg_off.as<uint64_t>(), c->ctg_bases.as<char>());
        c->launches += 3;
        e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) { rc = ctx_fail(c, RFX_E_CUDA, "contig gather failed: %s", cudaGetErrorString(e)); break; }
        c->ms[5] += stage_end(c);
        c->n_contigs = tot.a;
        c->n_contig_bases = tot.b;
        c->n_oriented = tot.c;
        c->n_budget_adm = h[DS_ABSORBED];
        c->n_cycles = h[DS_CYCLES];
        c->have_contigs = true;
    } while (0);
    return rc;
}

template <class KT> static int sorted_impl(Ctx* c, int E, double fold, int X) {
    cudaStream_t st = c->stream;
    const uint64_t n = 2 * c->n_rows;
    c->n_sorted = 0;
    c->have_contigs = false;  // the index, the alive bytes and the flag arrays are taken over
    if (n == 0) { c->have_sorted = true; return RFX_OK; }
    if (n >= 0xffffffffull) return ctx_fail(c, RFX_E_CAPACITY, "more than 2^31 rows: oriented ids do not fit 32 bits");
    stage_begin(c);
    RFX_TRY(devbuf_reserve(c, c->rflag, n * sizeof(int32_t)));
    RFX_TRY(devbuf_reserve(c, c->lflag, n * sizeof(int32_t)));
    RFX_TRY(devbuf_reserve(c, c->alive, n));
    RFX_TRY(devbuf_reserve(c, c->srt_left, n * sizeof(int32_t)));
    RFX_TRY(devbuf_reserve(c, c->srt_right, n * sizeof(int32_t)));
    RFX_TRY(build_index<KT>(c));
    Graph<KT> G = make_graph<KT>(c);
    uint8_t* alive = c->alive.as<uint8_t>();
    int32_t* cov = c->lflag.as<int32_t>();
    int32_t* rflag = c->rflag.as<int32_t>();
    sorted_right_kernel<KT><<<grid_n(n), 256, 0, st>>>(G, E, fold, X, alive, cov, rflag, n);
    sorted_left_kernel<KT><<<grid_n(n), 256, 0, st>>>(G, E, fold, X, alive, cov, rflag, c->srt_left.as<int32_t>(), c->srt_right.as<int32_t>(), n);
    c->launches += 2;
    // survivors
    ScanPlan<uint64_t> plan;
    RFX_TRY(devbuf_reserve(c, c->scan_ws, ScanPlan<uint64_t>::workspace_elems(n) * sizeof(uint64_t)));
    plan.bind(n, c->scan_ws.as<uint64_t>());
    scan_prepare(plan, AliveBoth{alive}, OpAddU64{}, (uint64_t)0, st);
    c->launches += 2 * plan.levels;
    uint64_t total = 0;
    RFX_CUDA(c, cudaMemcpyAsync(&total, plan.total, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return ctx_fail(c, RFX_E_CUDA, "sorted-stage kernels failed: %s", cudaGetErrorString(e));
    c->ms[3] += stage_end(c);
    c->n_sorted = total;
    c->have_sorted = true;
    return RFX_OK;
}

// the working domain of the reference's sorting stage (rfx_sort_kmers, rfx_sort_kmers_sharded)
static int sorted_domain(Ctx* c, const char* who, int E, double fold, int max_kmer_size) {
    if (E == 0)
        return ctx_fail(c, RFX_E_UNSUPPORTED,
                        "min_error_coverage 0 selects DSFilterForkSubKmer, which reads five columns from a three-column row "
                        "(ReflexivDSKmerLeftAndRightSorting.java:366-407) and cannot run in the reference");
    if (c->k < 2 || (c->k - 1) % 31 == 0)
        return ctx_fail(c, RFX_E_UNSUPPORTED, "k = %d: DSForwardSubKmerExtraction takes the last base from the wrong block when (k-1) %% 31 == 0 "
                        "(ReflexivDSKmerLeftAndRightSorting.java:930-936)", c->k);
    if (!(fold > 0) || max_kmer_size < 1 || max_kmer_size + 3 >= 30000) return ctx_fail(c, RFX_E_INVALID, "%s: bad fold / max_kmer_size", who);
    return RFX_OK;
}

int stage_sorted(Ctx* c, int E, double fold, int max_kmer_size) {
    if (!c->have_counts) return ctx_fail(c, RFX_E_STATE, "rfx_sort_kmers: no count table (call rfx_count or rfx_load_counts first)");
    RFX_TRY(sorted_domain(c, "rfx_sort_kmers", E, fold, max_kmer_size));
    return c->wide ? sorted_impl<u128>(c, E, fold, max_kmer_size + 3) : sorted_impl<uint64_t>(c, E, fold, max_kmer_size + 3);
}

int stage_graph(Ctx* c) {
    if (!c->have_counts) return ctx_fail(c, RFX_E_STATE, "rfx_assemble: no count table (call rfx_count or rfx_load_counts first)");
    if (!c->prm.bubble)
        return ctx_fail(c, RFX_E_UNSUPPORTED,
                        "-bubble: with the fork filters off the reference feeds marker-less extensions into DSkmerRandomReflection "
                        "(ReflexivDSMain.java:3634 vs 3716) and its output is undefined");
    if (c->k < 2) return ctx_fail(c, RFX_E_INVALID, "assembly needs k >= 2");
    return c->wide ? graph_impl<u128>(c) : graph_impl<uint64_t>(c);
}

}  // namespace rfx

#include "rfx_shard_graph.cuh"
