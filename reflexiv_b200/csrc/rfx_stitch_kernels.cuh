// rfx_stitch_kernels.cuh -- the kernels of the -stitch stage (rfx_stitch.cu has the map to the reference and the host side).
// Kept in a header of their own so that tests/hostemu can run the SAME kernel bodies thread by thread on the host
// (RFX_STITCH_HOSTEMU: a test-only shim supplies blockIdx / atomicCAS / ... ; the product never defines it).
#pragma once
#include <stdint.h>
#ifndef RFX_STITCH_HOSTEMU
#include "rfx_internal.h"
#include "rfx_scan.cuh"
#elif !defined(__grid_constant__)
#define __grid_constant__
#endif

namespace rfx {
namespace stitch {

constexpr uint64_t ST_EMPTY = ~0ull;

struct Hit {          // a fragment found in the chunk being scanned
    uint64_t src;     // text offset of the READ
    uint64_t off;     // offset of its codes behind the codes of earlier chunks
    uint32_t rlen;    // read length
    uint32_t start;   // first position of the fragment in the scanned strand
    uint32_t len;
    uint32_t left_ctg, right_ctg;
    uint32_t strand;  // 1: the reverse-complement string was scanned
};
struct Frag {
    uint64_t off;     // into the code array
    uint32_t len, left_ctg, right_ctg, pad;
};

__device__ __forceinline__ uint32_t nv(uint8_t c) { return c == 'A' ? 0u : c == 'C' ? 1u : c == 'G' ? 2u : 3u; }  // nucleotideValue, :1597-1609
__device__ __forceinline__ uint8_t complementary(uint8_t a) {  // :1527-1539
    if (a == 'A' || a == 'a') return 'T';
    if (a == 'T' || a == 't' || a == 'U' || a == 'u') return 'A';
    if (a == 'C' || a == 'c') return 'G';
    if (a == 'G' || a == 'g') return 'C';
    return 'N';
}
__device__ __forceinline__ uint64_t st_hash(uint64_t x) {
    x ^= x >> 31; x *= 0x7fb5d329728ea185ull; x ^= x >> 27; x *= 0x81dadef4bc2dd44dull; x ^= x >> 33;
    return x;
}

// A Bloom filter over the probe keys (64 KB, two bits per key) in front of the table: almost every (k-1)-mer of a read is no
// contig end, and the filter answers that from the L1 where the table itself only fits the L2.
constexpr uint32_t ST_BLOOM_BITS = 1u << 19;
__device__ __forceinline__ void bloom_set(uint32_t* bloom, uint64_t key) {
    const uint32_t x = (uint32_t)key ^ (uint32_t)(key >> 31);
    const uint32_t a = (x * 0x9E3779B1u) >> 13, b = (x * 0x85EBCA6Bu) >> 13;  // 19 bits each (ST_BLOOM_BITS), as bloom_maybe below
    atomicOr(&bloom[a >> 5], 1u << (a & 31));
    atomicOr(&bloom[b >> 5], 1u << (b & 31));
}

// ---- S1: probes ---------------------------------------------------------------------------------
__global__ void probe_first_kernel(const uint64_t* __restrict__ off, const char* __restrict__ bases, uint64_t n, int k, uint64_t* __restrict__ firstk) {
    for (uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; c < n; c += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t len = off[c + 1] - off[c];
        uint64_t f = 0;
        if (len >= (uint64_t)k)
            for (int j = 0; j < k; j++) f = (f << 2) | nv((uint8_t)bases[off[c] + j]);
        firstk[c] = f;
    }
}

// value = contig << 1 | direction (1: the contig's first (k-1)-mer, "right extendable"; 0: its last, "left extendable").
// Of the probes with one key the largest (first k-mer of the contig, direction 0 over 1) stays: Hashtable.put keeps the last.
__device__ __forceinline__ bool probe_after(uint32_t a, uint32_t b, const uint64_t* firstk) {
    const uint64_t fa = firstk[a >> 1], fb = firstk[b >> 1];
    if (fa != fb) return fa > fb;
    if ((a >> 1) != (b >> 1)) return (a >> 1) > (b >> 1);  // (two contigs never start with the same k-mer; a total order all the same)
    return (a & 1u) < (b & 1u);
}
__device__ void probe_insert(uint64_t key, uint32_t val, uint64_t* keys, uint32_t* vals, uint64_t mask, const uint64_t* firstk, uint32_t* bloom) {
    bloom_set(bloom, key);
    uint64_t s = st_hash(key) & mask;
    for (;;) {
        const unsigned long long prev = atomicCAS((unsigned long long*)&keys[s], (unsigned long long)ST_EMPTY, (unsigned long long)key);
        if (prev == ST_EMPTY || prev == key) break;
        s = (s + 1) & mask;
    }
    uint32_t cur = vals[s];
    for (;;) {
        if (cur != NONE32 && !probe_after(val, cur, firstk)) return;
        const uint32_t seen = atomicCAS(&vals[s], cur, val);
        if (seen == cur) return;
        cur = seen;
    }
}
// the probes of contig c (its first (k-1)-mer a, its last b) for the ends that are clean and covered <= 4 times (the caller
// has checked the length)
__device__ __forceinline__ void probe_contig(uint64_t c, int32_t cl, int32_t cr, uint64_t a, uint64_t b, uint64_t* keys, uint32_t* vals, uint64_t mask,
                                             const uint64_t* firstk, uint32_t* bloom, unsigned long long* n_probes) {
    const bool l = cl >= -5 && cl < 0, r = cr >= -5 && cr < 0;
    if (l) probe_insert(a, (uint32_t)(c << 1) | 1u, keys, vals, mask, firstk, bloom);
    if (r) probe_insert(b, (uint32_t)(c << 1), keys, vals, mask, firstk, bloom);
    if (l || r) atomicAdd(n_probes, (unsigned long long)l + (unsigned long long)r);
}
__global__ void probe_insert_kernel(const uint64_t* __restrict__ off, const char* __restrict__ bases, const int32_t* __restrict__ cl,
                                    const int32_t* __restrict__ cr, uint64_t n, int k, const uint64_t* __restrict__ firstk, uint64_t* keys,
                                    uint32_t* vals, uint64_t mask, uint32_t* bloom, unsigned long long* n_probes) {
    const int sk = k - 1;
    for (uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; c < n; c += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t len = off[c + 1] - off[c];
        if (len < 61) continue;  // :1229
        if (!(cl[c] >= -5 && cl[c] < 0) && !(cr[c] >= -5 && cr[c] < 0)) continue;
        uint64_t a = 0, b = 0;
        for (int j = 0; j < sk; j++) {
            a = (a << 2) | nv((uint8_t)bases[off[c] + j]);
            b = (b << 2) | nv((uint8_t)bases[off[c + 1] - sk + j]);
        }
        probe_contig(c, cl[c], cr[c], a, b, keys, vals, mask, firstk, bloom, n_probes);
    }
}

// ---- S1 across ranks (rfx_stitch_begin_sharded): every rank summarises its own contigs, pulls everybody's summary and builds
// the same probe table over global contig ids (a rank's prefix + its local index)
// ends[2c], ends[2c + 1]: the first and the last (k-1)-mer of contig c (0 for a contig too short to probe)
__global__ void contig_ends_kernel(const uint64_t* __restrict__ off, const char* __restrict__ bases, uint64_t n, int k, uint64_t* __restrict__ ends) {
    const int sk = k - 1;
    for (uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; c < n; c += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t a = 0, b = 0;
        if (off[c + 1] - off[c] >= 61)
            for (int j = 0; j < sk; j++) {
                a = (a << 2) | nv((uint8_t)bases[off[c] + j]);
                b = (b << 2) | nv((uint8_t)bases[off[c + 1] - sk + j]);
            }
        ends[2 * c] = a;
        ends[2 * c + 1] = b;
    }
}
// a rank's contig offsets (possibly in a peer's memory) -> its slice of the global offsets, moved by `add` bases
__global__ void rebase_off_kernel(const uint64_t* __restrict__ src, uint64_t n, uint64_t add, uint64_t* __restrict__ dst) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) dst[i] = src[i] + add;
}
// probe_insert_kernel over the pulled summaries: global offsets, ends, flags
__global__ void probe_insert_ends_kernel(const uint64_t* __restrict__ off, const uint64_t* __restrict__ ends, const int32_t* __restrict__ cl,
                                         const int32_t* __restrict__ cr, uint64_t n, const uint64_t* __restrict__ firstk, uint64_t* keys, uint32_t* vals,
                                         uint64_t mask, uint32_t* bloom, unsigned long long* n_probes) {
    for (uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; c < n; c += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t len = off[c + 1] - off[c];
        if (len < 61) continue;  // :1229
        probe_contig(c, cl[c], cr[c], ends[2 * c], ends[2 * c + 1], keys, vals, mask, firstk, bloom, n_probes);
    }
}
__global__ void count_keys_kernel(const uint64_t* __restrict__ keys, uint64_t cap, unsigned long long* n) {
    unsigned long long m = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < cap; i += (uint64_t)gridDim.x * blockDim.x) m += keys[i] != ST_EMPTY;
    if (m) atomicAdd(n, m);
}

__device__ __forceinline__ uint32_t probe_lookup_h(uint64_t key, uint64_t h, const uint64_t* __restrict__ keys, const uint32_t* __restrict__ vals, uint64_t mask) {
    uint64_t s = h & mask;
    for (;;) {
        const uint64_t kk = __ldg(&keys[s]);
        if (kk == key) return __ldg(&vals[s]);
        if (kk == ST_EMPTY) return NONE32;
        s = (s + 1) & mask;
    }
}

__device__ __forceinline__ uint32_t probe_lookup(uint64_t key, const uint64_t* __restrict__ keys, const uint32_t* __restrict__ vals, uint64_t mask) {
    return probe_lookup_h(key, st_hash(key), keys, vals, mask);
}

// Both codes of a text byte in one table entry: bits 0-1 nucleotideValue(c) (the forward strand), bits 2-3
// nucleotideValue(complementary(c)) (the reverse-complement STRING of the reference: lower case folded, U = T, anything else 'N' -> 3).
__device__ const uint8_t ST_CODES[256] = {
    15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15,
    15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15,
    15, 12, 15, 9, 15, 15, 15, 6, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 3, 3, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15,
    15, 15, 15, 11, 15, 15, 15, 7, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 3, 3, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15,
    15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15,
    15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15,
    15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15,
    15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15, 15,
};

// the window hash of the Bloom filter: cheap, because nearly every window of a read ends here
__device__ __forceinline__ uint32_t bloom_fold(uint64_t w) { return (uint32_t)w ^ (uint32_t)(w >> 31); }
__device__ __forceinline__ bool bloom_maybe(const uint32_t* __restrict__ bloom, uint64_t w) {
    const uint32_t x = bloom_fold(w);
    const uint32_t a = (x * 0x9E3779B1u) >> 13;
    if (!((__ldg(&bloom[a >> 5]) >> (a & 31)) & 1u)) return false;
    const uint32_t b = (x * 0x85EBCA6Bu) >> 13;
    return (__ldg(&bloom[b >> 5]) >> (b & 31)) & 1u;
}

// ---- S2: reads ----------------------------------------------------------------------------------
// One thread per read walks the text ONCE, in aligned 4-byte words, and rolls two windows: the (k-1)-mer of the forward strand
// and the (k-1)-mer the reverse-complement string shows at the mirrored position (window ending at i  <->  window ending at
// L + k - 3 - i of the other strand).  DSLowCoverageReadDetection scans each strand front to back and keeps the FIRST direction-0
// hit (its contig is remembered) and the LAST direction-1 hit of another contig (:1497-1531); that is: left = the smallest hit
// position of direction 0, right = the largest direction-1 position behind it whose contig differs from left's -- a rule without
// an order, so the reverse strand can be collected back to front: the last direction-0 hit met is its `left`, and of the
// direction-1 hits only the first met and the first met of another contig can be its `right`.
__global__ void __launch_bounds__(256) stitch_scan_kernel(const uint8_t* __restrict__ text, const uint64_t* __restrict__ rd_src, const uint32_t* __restrict__ rd_len,
                                                          uint64_t n_reads, int k, const uint64_t* __restrict__ keys, const uint32_t* __restrict__ vals, uint64_t mask,
                                                          const uint32_t* __restrict__ bloom, Hit* hits, uint64_t hit_cap, unsigned long long* ctr /* [0] hits, [1] codes */) {
    const int sk = k - 1;
    const uint64_t kmask = (1ull << (2 * sk)) - 1;
    const int top = 2 * (sk - 1);
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n_reads; r += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t L = rd_len[r];  // 0 when readLength - (k-1) <= 1 (:1473)
        if (L == 0) continue;
        const uint64_t src = rd_src[r];
        const uintptr_t a0 = (uintptr_t)(text + src), a1 = a0 + L;
        // forward strand
        uint32_t f_probed = NONE32;
        int f_left = -1, f_right = -1;
        // reverse strand, positions in ITS coordinates
        uint32_t r_lctg = NONE32, ra_ctg = NONE32, rb_ctg = NONE32;
        int r_left = -1, ra_pos = -1, rb_pos = -1;
        uint64_t wf = 0, wr = 0;
        int i = 0;
        for (uintptr_t wa = a0 & ~(uintptr_t)3; wa < a1; wa += 4) {
            const uint32_t word = __ldg(reinterpret_cast<const uint32_t*>(wa));  // (inside the text buffer: it is read in whole 64-byte chunks)
#pragma unroll
            for (int b = 0; b < 4; b++) {
                const uintptr_t a = wa + b;
                if (a < a0 || a >= a1) continue;
                const uint32_t cc = ST_CODES[(word >> (8 * b)) & 0xffu];
                wf = ((wf << 2) | (cc & 3u)) & kmask;
                wr = (wr >> 2) | ((uint64_t)(cc >> 2) << top);
                if (i >= sk - 1) {
                    if (bloom_maybe(bloom, wf)) {
                        const uint32_t v = probe_lookup(wf, keys, vals, mask);
                        if (v != NONE32) {
                            if (!(v & 1u)) {
                                if (f_left < 0) { f_probed = v >> 1; f_left = i; }
                            } else if (f_probed != (v >> 1)) {
                                f_right = i;
                            }
                        }
                    }
                    if (bloom_maybe(bloom, wr)) {
                        const uint32_t v = probe_lookup(wr, keys, vals, mask);
                        if (v != NONE32) {
                            const int ip = (int)L + sk - 2 - i;  // where the reverse strand shows this window
                            if (!(v & 1u)) { r_left = ip; r_lctg = v >> 1; }
                            else if (ra_pos < 0) { ra_pos = ip; ra_ctg = v >> 1; }
                            else if (rb_pos < 0 && (v >> 1) != ra_ctg) { rb_pos = ip; rb_ctg = v >> 1; }
                        }
                    }
                }
                i++;
            }
        }
        int r_right = -1;
        if (r_left >= 0) {
            if (ra_pos >= 0 && ra_ctg != r_lctg) r_right = ra_pos;
            else if (rb_pos >= 0 && rb_ctg != r_lctg) r_right = rb_pos;
        }
        if (f_left >= 0 && f_right >= 0 && f_left < f_right) {
            const uint32_t start = (uint32_t)(f_left - sk + 1), len = (uint32_t)f_right + 1u - start;
            const unsigned long long idx = atomicAdd(&ctr[0], 1ull);
            const unsigned long long o = atomicAdd(&ctr[1], (unsigned long long)len);
            if (idx < hit_cap) hits[idx] = Hit{src, o, L, start, len, 0u, 0u, 0u};
        }
        if (r_left >= 0 && r_right >= 0 && r_left < r_right) {
            const uint32_t start = (uint32_t)(r_left - sk + 1), len = (uint32_t)r_right + 1u - start;
            const unsigned long long idx = atomicAdd(&ctr[0], 1ull);
            const unsigned long long o = atomicAdd(&ctr[1], (unsigned long long)len);
            if (idx < hit_cap) hits[idx] = Hit{src, o, L, start, len, 0u, 0u, 1u};
        }
    }
}

// one warp per fragment: bases -> 2-bit codes (one per byte), the descriptor, and the two contigs whose probes cut it
__global__ void __launch_bounds__(256) stitch_copy_kernel(const uint8_t* __restrict__ text, const Hit* __restrict__ hits, uint64_t n_hits, int k,
                                                          const uint64_t* __restrict__ keys, const uint32_t* __restrict__ vals, uint64_t mask,
                                                          uint8_t* __restrict__ codes, uint64_t code_base, Frag* __restrict__ frags, uint64_t frag_base) {
    const int lane = threadIdx.x & 31;
    const int sk = k - 1;
    for (uint64_t h = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; h < n_hits; h += ((uint64_t)gridDim.x * blockDim.x) >> 5) {
        const Hit H = hits[h];
        const uint8_t* rd = text + H.src;
        uint8_t* dst = codes + code_base + H.off;
        for (uint32_t j = lane; j < H.len; j += 32) {
            const uint32_t i = H.start + j;
            dst[j] = (uint8_t)(H.strand ? nv(complementary(rd[H.rlen - 1 - i])) : nv(rd[i]));
        }
        __syncwarp();
        if (lane == 0) {
            uint64_t a = 0, b = 0;
            for (int j = 0; j < sk; j++) {
                const uint32_t i0 = H.start + j, i1 = H.start + H.len - sk + j;
                a = (a << 2) | (H.strand ? nv(complementary(rd[H.rlen - 1 - i0])) : nv(rd[i0]));
                b = (b << 2) | (H.strand ? nv(complementary(rd[H.rlen - 1 - i1])) : nv(rd[i1]));
            }
            frags[frag_base + h] = Frag{code_base + H.off, H.len, probe_lookup(a, keys, vals, mask) >> 1, probe_lookup(b, keys, vals, mask) >> 1, 0u};
        }
    }
}

// ---- S3 / S4 --------------------------------------------------------------------------------------
// CANONICAL ORDER: the shorter fragment, then the smaller 2-bit sequence, then (identical fragments) the smaller index
__device__ bool frag_before(uint32_t a, uint32_t b, const Frag* __restrict__ f, const uint8_t* __restrict__ codes) {
    const Frag A = f[a], B = f[b];
    if (A.len != B.len) return A.len < B.len;
    const uint8_t *x = codes + A.off, *y = codes + B.off;
    for (uint32_t j = 0; j < A.len; j++)
        if (x[j] != y[j]) return x[j] < y[j];
    return a < b;
}
// side 0: nxt[left contig] = the fragment that leaves it (pass 1 of DSFilterRepeatLowCoverageFragment: one record per first
// (k-1)-mer); side 1: prv[right contig] = the one of the pass-1 survivors that joins it (the extension merges one pair of a run)
__global__ void frag_pick_kernel(const Frag* __restrict__ f, const uint8_t* __restrict__ codes, uint64_t n, int side, const uint32_t* __restrict__ nxt_in,
                                 uint32_t* slot) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        if (side == 1 && nxt_in[f[i].left_ctg] != (uint32_t)i) continue;
        uint32_t* s = &slot[side ? f[i].right_ctg : f[i].left_ctg];
        uint32_t cur = *s;
        for (;;) {
            if (cur != NONE32 && !frag_before((uint32_t)i, cur, f, codes)) break;
            const uint32_t seen = atomicCAS(s, cur, (uint32_t)i);
            if (seen == cur) break;
            cur = seen;
        }
    }
}

// the contig a record continues with behind contig c, NONE32 at its end
__device__ __forceinline__ uint32_t next_ctg(uint32_t c, const uint32_t* nxt, const uint32_t* prv, const Frag* f) {
    const uint32_t g = nxt[c];
    if (g == NONE32) return NONE32;
    const uint32_t b = f[g].right_ctg;
    return prv[b] == g ? b : NONE32;
}
// role: 0 lone contig, 1 head of a chain, 2 inner member (visited from a head), 3 head of a ring
__global__ void chain_heads_kernel(uint64_t n, const uint32_t* __restrict__ nxt, const uint32_t* __restrict__ prv, const Frag* __restrict__ f, uint8_t* role) {
    for (uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; c < n; c += (uint64_t)gridDim.x * blockDim.x) {
        if (prv[c] != NONE32) continue;
        role[c] = nxt[c] != NONE32 ? 1 : 0;
        uint64_t steps = 0;  // (every walk below is bounded by the number of contigs: a chain cannot be longer)
        for (uint32_t cur = next_ctg((uint32_t)c, nxt, prv, f); cur != NONE32 && steps < n; cur = next_ctg(cur, nxt, prv, f), steps++) role[cur] = 2;
    }
}
// what no head reached lies on a ring: its member with the smallest first k-mer becomes the head (a record never meets itself)
__device__ __forceinline__ void ring_head_at(uint64_t c, uint64_t n, const uint32_t* __restrict__ nxt, const uint32_t* __restrict__ prv, const Frag* __restrict__ f,
                                             const uint64_t* __restrict__ firstk, uint8_t* role, unsigned long long* n_rings) {
    if (prv[c] == NONE32 || role[c] == 2) return;
    bool smallest = true;
    uint64_t steps = 0;
    for (uint32_t cur = next_ctg((uint32_t)c, nxt, prv, f); cur != (uint32_t)c && cur != NONE32 && steps < n; cur = next_ctg(cur, nxt, prv, f), steps++)
        if (firstk[cur] < firstk[c] || (firstk[cur] == firstk[c] && cur < (uint32_t)c)) { smallest = false; break; }
    if (smallest) { role[c] = 3; atomicAdd(n_rings, 1ull); }
}
__global__ void ring_heads_kernel(uint64_t n, const uint32_t* __restrict__ nxt, const uint32_t* __restrict__ prv, const Frag* __restrict__ f,
                                  const uint64_t* __restrict__ firstk, uint8_t* role, unsigned long long* n_rings) {
    for (uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; c < n; c += (uint64_t)gridDim.x * blockDim.x) ring_head_at(c, n, nxt, prv, f, firstk, role, n_rings);
}
// length, right flag and keep decision (DSKmerToContig :749-754) of the record every head stands for
__device__ __forceinline__ void chain_size_at(uint64_t c, uint64_t n, int k, int min_contig, const uint64_t* __restrict__ off, const int32_t* __restrict__ cl,
                                              const int32_t* __restrict__ cr, const uint32_t* __restrict__ nxt, const uint32_t* __restrict__ prv, const Frag* __restrict__ f,
                                              const uint8_t* __restrict__ role, uint64_t* out_len, int32_t* out_right, unsigned long long* n_stitched) {
    const uint64_t sk = (uint64_t)k - 1;
    uint64_t len = 0;
    int32_t right = 0;
    const uint8_t ro = role[c];
    if (ro != 2 && !(ro == 0 && prv[c] != NONE32)) {  // (role 0 with an arriving fragment: a ring member that is not its head)
        len = off[c + 1] - off[c];
        right = cr[c];
        uint32_t cur = (uint32_t)c;
        for (uint64_t steps = 0; nxt[cur] != NONE32 && steps < n; steps++) {
            const Frag F = f[nxt[cur]];
            len += F.len - sk;
            right = -10000000;
            if (prv[F.right_ctg] != nxt[cur]) break;  // another fragment joined the contig this one ends on
            cur = F.right_ctg;
            if (cur == (uint32_t)c) break;            // ring closed: the closing fragment ends the record
            len += off[cur + 1] - off[cur] - sk;
            right = cr[cur];
        }
        if (nxt[c] != NONE32) atomicAdd(n_stitched, 1ull);
        if ((cl[c] <= -10000000 && right <= -10000000) || len < (uint64_t)min_contig) len = 0;
    }
    *out_len = len;
    *out_right = right;
}
__global__ void chain_sizes_kernel(uint64_t n, int k, int min_contig, const uint64_t* __restrict__ off, const int32_t* __restrict__ cl,
                                   const int32_t* __restrict__ cr, const uint32_t* __restrict__ nxt, const uint32_t* __restrict__ prv, const Frag* __restrict__ f,
                                   const uint8_t* __restrict__ role, uint64_t* out_len, int32_t* out_right, unsigned long long* n_stitched) {
    for (uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; c < n; c += (uint64_t)gridDim.x * blockDim.x)
        chain_size_at(c, n, k, min_contig, off, cl, cr, nxt, prv, f, role, &out_len[c], &out_right[c], n_stitched);
}
struct KeepIn {
    const uint64_t* out_len;
    __device__ __forceinline__ U64x3 operator()(uint64_t c) const { return out_len[c] ? U64x3{1, out_len[c], 0} : U64x3{0, 0, 0}; }
};
struct KeepOut {
    const int32_t* cl;
    const int32_t* out_right;
    uint64_t *new_off, *slot_of;
    int32_t *new_left, *new_right;
    __device__ __forceinline__ void operator()(uint64_t c, U64x3 excl, U64x3 v) const {
        slot_of[c] = v.a ? excl.a : ~0ull;
        if (v.a) { new_off[excl.a] = excl.b; new_left[excl.a] = cl[c]; new_right[excl.a] = out_right[c]; }
    }
};
__global__ void set_end_kernel(uint64_t* p, const U64x3* tot) { *p = tot->b; }
// the record of head c, written by the threads of one block: contig, fragment extension, contig minus its first k-1 bases, ...
// bases_of(g): the first base of contig g
template <class BasesOf>
__device__ __forceinline__ void gather_record(uint64_t c, uint64_t n, int k, const uint64_t* __restrict__ off, BasesOf bases_of, const uint32_t* __restrict__ nxt,
                                              const uint32_t* __restrict__ prv, const Frag* __restrict__ f, const uint8_t* __restrict__ codes, char* __restrict__ dst) {
    const uint64_t sk = (uint64_t)k - 1;
    uint64_t l0 = off[c + 1] - off[c];
    const char* src = bases_of((uint32_t)c);
    for (uint64_t j = threadIdx.x; j < l0; j += blockDim.x) dst[j] = src[j];
    dst += l0;
    uint32_t cur = (uint32_t)c;
    for (uint64_t steps = 0; nxt[cur] != NONE32 && steps < n; steps++) {
        const Frag F = f[nxt[cur]];
        for (uint64_t j = threadIdx.x; j + sk < F.len; j += blockDim.x) dst[j] = "ACGT"[codes[F.off + sk + j]];
        dst += F.len - sk;
        if (prv[F.right_ctg] != nxt[cur]) break;
        cur = F.right_ctg;
        if (cur == (uint32_t)c) break;
        l0 = off[cur + 1] - off[cur] - sk;
        src = bases_of(cur) + sk;
        for (uint64_t j = threadIdx.x; j < l0; j += blockDim.x) dst[j] = src[j];
        dst += l0;
    }
}
struct LocalBases {
    const uint64_t* off;
    const char* bases;
    __device__ __forceinline__ const char* operator()(uint32_t g) const { return bases + off[g]; }
};
// one block per record
__global__ void __launch_bounds__(256) chain_gather_kernel(uint64_t n, int k, const uint64_t* __restrict__ off, const char* __restrict__ bases,
                                                           const uint32_t* __restrict__ nxt, const uint32_t* __restrict__ prv, const Frag* __restrict__ f,
                                                           const uint8_t* __restrict__ codes, const uint64_t* __restrict__ slot_of,
                                                           const uint64_t* __restrict__ new_off, char* __restrict__ out) {
    for (uint64_t c = blockIdx.x; c < n; c += gridDim.x) {
        if (slot_of[c] == ~0ull) continue;
        gather_record(c, n, k, off, LocalBases{off, bases}, nxt, prv, f, codes, out + new_off[slot_of[c]]);
    }
}

// ---- S3 / S4 across ranks (rfx_stitch_finish_sharded): every rank holds all fragments and the replicated per-contig arrays
// over global ids, runs the picks and chain_heads_kernel over all of them, and the kernels below over the heads [lo, hi) it owns.
// Per-head outputs (out_len, out_right, slot_of) are indexed by c - lo.
__global__ void ring_heads_range_kernel(uint64_t lo, uint64_t hi, uint64_t n, const uint32_t* __restrict__ nxt, const uint32_t* __restrict__ prv,
                                        const Frag* __restrict__ f, const uint64_t* __restrict__ firstk, uint8_t* role, unsigned long long* n_rings) {
    for (uint64_t c = lo + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; c < hi; c += (uint64_t)gridDim.x * blockDim.x) ring_head_at(c, n, nxt, prv, f, firstk, role, n_rings);
}
__global__ void chain_sizes_range_kernel(uint64_t lo, uint64_t hi, uint64_t n, int k, int min_contig, const uint64_t* __restrict__ off, const int32_t* __restrict__ cl,
                                         const int32_t* __restrict__ cr, const uint32_t* __restrict__ nxt, const uint32_t* __restrict__ prv, const Frag* __restrict__ f,
                                         const uint8_t* __restrict__ role, uint64_t* out_len, int32_t* out_right, unsigned long long* n_stitched) {
    for (uint64_t c = lo + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; c < hi; c += (uint64_t)gridDim.x * blockDim.x)
        chain_size_at(c, n, k, min_contig, off, cl, cr, nxt, prv, f, role, &out_len[c - lo], &out_right[c - lo], n_stitched);
}
// where every rank's contigs are: global ids [ctg_lo[r], ctg_lo[r + 1]) hold bases [base_lo[r], base_lo[r + 1]) of the global
// offsets, stored from bases[r] on (the rank's own contig bases, as seen from this device: possibly a peer's memory)
struct CtgSources {
    const char* bases[8];
    unsigned long long ctg_lo[9], base_lo[9];
    int n;
    const uint64_t* off;  // global offsets
    __device__ __forceinline__ const char* operator()(uint32_t g) const {
        int r = 0;
        while (r + 1 < n && (unsigned long long)g >= ctg_lo[r + 1]) r++;
        return bases[r] + (off[g] - base_lo[r]);
    }
};
// one block per own head: the pieces of its record are read where they lie, contig bases from their owner over peer memory
__global__ void __launch_bounds__(256) chain_gather_peer_kernel(uint64_t lo, uint64_t hi, uint64_t n, int k, const __grid_constant__ CtgSources P,
                                                                const uint32_t* __restrict__ nxt, const uint32_t* __restrict__ prv, const Frag* __restrict__ f,
                                                                const uint8_t* __restrict__ codes, const uint64_t* __restrict__ slot_of,
                                                                const uint64_t* __restrict__ new_off, char* __restrict__ out) {
    for (uint64_t c = lo + blockIdx.x; c < hi; c += gridDim.x) {
        if (slot_of[c - lo] == ~0ull) continue;
        gather_record(c, n, k, P.off, P, nxt, prv, f, codes, out + new_off[slot_of[c - lo]]);
    }
}
// a rank's fragments (possibly in a peer's memory) -> their place in the global list, code offsets moved by `add`
__global__ void frag_pull_kernel(const Frag* __restrict__ src, uint64_t n, uint64_t add, Frag* __restrict__ dst) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        Frag F = src[i];
        F.off += add;
        dst[i] = F;
    }
}
__global__ void fill_u32_kernel(uint32_t* p, uint64_t n, uint32_t v) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) p[i] = v;
}
__global__ void count_picked_kernel(const Frag* __restrict__ f, uint64_t n, const uint32_t* __restrict__ nxt, const uint32_t* __restrict__ prv, unsigned long long* out) {
    unsigned long long a = 0, b = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const bool alive = nxt[f[i].left_ctg] == (uint32_t)i;
        a += alive;
        b += alive && prv[f[i].right_ctg] == (uint32_t)i;
    }
    if (a) atomicAdd(&out[0], a);
    if (b) atomicAdd(&out[1], b);
}


}  // namespace stitch
}  // namespace rfx
