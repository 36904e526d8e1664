// rfx_graph.cuh -- device helpers shared by the single-GPU graph stages (rfx_graph.cu) and the sharded ones (rfx_shard_graph.cu).
#pragma once
#include "rfx_internal.h"

namespace rfx {

// ---- minimiser arithmetic of a k-mer's neighbours --------------------------------------------------------------
// hash of the canonical form of an m-mer given right aligned
__device__ __forceinline__ uint32_t mm_hash_m(uint32_t mm, int m) {
    uint32_t r = brev32(mm);
    r = ((r >> 1) & 0x55555555u) | ((r & 0x55555555u) << 1);
    r = (~r) >> (32 - 2 * m);
    return mmer_hash(mm < r ? mm : r);
}
// minima of the m-mer hashes inside the first / the last k-1 bases of X
template <class KT> __device__ __forceinline__ void kmer_minima(KT X, int k, int m, uint32_t& pre_min, uint32_t& suf_min) {
    const uint32_t mmask = (m >= 16) ? 0xffffffffu : ((1u << (2 * m)) - 1u);
    const int mtop = 2 * (m - 1), w = k - m + 1;
    KT Y = X << (8 * (int)sizeof(KT) - 2 * k);  // first base in the top two bits
    uint32_t mf = 0, mr = 0;
    pre_min = 0xffffffffu; suf_min = 0xffffffffu;
    for (int t = 0; t < k; t++) {
        const uint32_t v = (uint32_t)(Y >> (8 * (int)sizeof(KT) - 2)) & 3u;
        Y <<= 2;
        mf = ((mf << 2) | v) & mmask;
        mr = (mr >> 2) | ((v ^ 3u) << mtop);
        if (t >= m - 1) {
            const int j = t - m + 1;
            const uint32_t h = mmer_hash(mf < mr ? mf : mr);
            if (j <= w - 2) pre_min = h < pre_min ? h : pre_min;
            if (j >= 1) suf_min = h < suf_min ? h : suf_min;
        }
    }
}
// minimiser bin of a row (a canonical k-mer): the smaller of its two minima, or its one m-mer when m == k (that m-mer lies
// in neither the prefix nor the suffix part).  The shard that owns the bin owns the row: rfx_shard_table routes rows by it
// and the sharded graph stages expect every row there.  The two minima are returned as well.
template <class KT> __device__ __forceinline__ uint32_t row_bin(KT key, int k, int m, uint32_t n_bins, uint32_t& pre_min, uint32_t& suf_min) {
    kmer_minima<KT>(key, k, m, pre_min, suf_min);
    uint32_t h = pre_min < suf_min ? pre_min : suf_min;
    if (m == k) h = mm_hash_m((uint32_t)key, m);
    return bin_of_minimizer(h, n_bins);
}
// hash of the last m-mer of (S + b) / the first m-mer of (a + S), S a right-aligned (k-1)-mer
template <class KT> __device__ __forceinline__ uint32_t last_mm_of(KT S, uint32_t b, int m) {
    const uint32_t low = (m >= 17) ? 0u : ((uint32_t)S & ((m >= 16) ? 0x3fffffffu : ((1u << (2 * (m - 1))) - 1u)));
    return mm_hash_m((low << 2) | b, m);
}
template <class KT> __device__ __forceinline__ uint32_t first_mm_of(KT S, uint32_t a, int k, int m) {
    const uint32_t top = (uint32_t)(S >> (2 * (k - 1 - (m - 1)))) & ((1u << (2 * (m - 1))) - 1u);
    return mm_hash_m((a << (2 * (m - 1))) | top, m);
}

// ---- list ranking by pointer jumping (rfx_graph.cu) ------------------------------------------------------------
__device__ __forceinline__ uint64_t ad_pack(uint32_t anc, uint32_t dist) { return (uint64_t)anc | ((uint64_t)dist << 32); }

// A7 / A8 junction bookkeeping bits of the alive byte: bit0 survives the right filter, bit1 survives both, bit2 right
// flag < 0, bit3 left flag < 0, bit4 / bit5: a budget walk along succ / pred went through the junction behind this node
__device__ __forceinline__ void alive_or(uint8_t* alive, uint64_t i, uint32_t bit) {
    atomicOr(reinterpret_cast<unsigned int*>(alive + (i & ~(uint64_t)3)), bit << (8u * (uint32_t)(i & 3u)));
}

}  // namespace rfx
