// rfx_shard_graph.cuh -- the graph stages (K5, K6, K7) of a sharded run: every rank keeps ITS rows of the filtered table
// (the rows whose minimiser bin it owns, exactly as rfx_count_sharded left them), the index over them and all per-node
// state; whatever a node needs from another rank it reads -- or writes -- in that rank's HBM over NVLink / NVSwitch.
// Included at the end of rfx_graph.cu (same translation unit: Graph<KT>, the index build and the rule functions are shared).
//
// Replaces, across GPUs, the global sort("k-1") shuffles of ReflexivDSMain.java:232, 244 (fork filters) and :261-326 (one
// or two per pass of the extension loop).
//
//   ids        a node is  gid = rank << 29 | (2 * row + strand)  with `row` local to its rank; links, ancestors and
//              splitter ids all use that form, so following a chain across GPUs is following a pointer.
//   owner      of a k-mer = owner of the bin its canonical minimiser hashes to (rfx_core.h: bin_of_minimizer), the very
//              map the counting stage shards by.  A neighbour shares k-1 bases with the node that asks for it, so the
//              asking node knows the neighbour's minimiser -- and owner -- after hashing ONE more m-mer.
//   probes     every rank holds a copy of every rank's presence bits (16 bits per row, pulled once per run: 2 B per
//              row instead of the 12 B per row of the table).  Three of four probes ask for a k-mer that does not
//              exist and end there; about 90 % of the rest stay on the rank (same minimiser).  What is left is ASKED of
//              the owner: the first pass of a K5 kernel writes a 16-byte request into the owner's inbox (a posted
//              store over NVLink), the owner looks the k-mer up in its own index and stores the answer (count, node,
//              alive byte) into the asker's answer box, a second pass finishes the nodes that were waiting.  One
//              request / response exchange per filter pass, no round trip ever waits on the link (random reads of a
//              peer's index from inside the kernels were measured first: 8.5 G/s per GPU between 2 GPUs, 1.3 G/s with
//              8 GPUs all asking at once -- the link pass alone took 2.7 ms; profiles/).
//   chains     level-1 splitters = heads, a 1-in-64 sample and every node whose predecessor lives on another rank, so a
//              level-1 segment never leaves its GPU and the walk that stamps it is purely local.  Level-2 splitters = heads
//              and 1 in 8 of the level-1 splitters; they walk the level-1 list (one 8-byte peer read and one 8-byte peer
//              write per hop).  Only the level-2 list (about 1 % of the nodes) goes through pointer jumping, each round
//              one small kernel + one cross-GPU barrier.
//   contigs    stay with the owner of their head: the tail tells the head its length and right flag, the owner sizes
//              and lays out its contigs, every node writes its base into the owner's buffer.
//   cycles     a closed path has no head: the ranks notice (a node without ancestor, or an ancestor that is no head)
//              and rank 0 pulls the shard tables and runs the single-GPU stages on the whole table (rare).
#pragma once

#include <string>
#include <utility>
#include <vector>

#include "rfx_shard.h"

namespace rfx {

constexpr uint32_t GID_MASK = 0x1fffffffu;
__host__ __device__ __forceinline__ uint32_t gid_make(int r, uint32_t l) { return ((uint32_t)r << 29) | l; }
__host__ __device__ __forceinline__ int gid_rank(uint32_t g) { return (int)(g >> 29); }
__host__ __device__ __forceinline__ uint32_t gid_loc(uint32_t g) { return g & GID_MASK; }

// what a rank needs to know of a rank (itself included); every address as seen from THIS device
struct SGPeer {
    const void* keys;
    const uint32_t* counts;
    const uint32_t* ht;
    const uint32_t* filter; // that rank's presence bits in ITS memory (only used to pull its slice)
    uint8_t* alive;
    int32_t *lflag, *rflag, *eff_l, *eff_r;
    uint32_t *succ, *pred;
    uint32_t* nxt_l1;  // per node whose successor lives on another rank: that successor's level-1 splitter (written by its owner)
    ulonglong2* l1_ent;  // per level-1 splitter: x = next level-1 splitter (gid form: rank, index) | nodes of the segment << 32, y = its level-2 index or NONE
    uint64_t* l1_loc;    // per level-1 splitter: (level-2 splitter that walked over it, nodes in front of it)
    uint64_t* l2_up[2];
    uint32_t* l2_node;
    uint64_t* l2_fin;  // per level-2 splitter: (head node, nodes in front of it)
    uint32_t* chain_len;
    int32_t* tail_rf;
    uint32_t* ctg_idx;
    uint64_t* ctg_off;
    char* ctg_bases;
    uint8_t* inbox;          // requests of every rank to this one: channel r at r * chan_cap (SGReq<KT>)
    uint4* respbox;          // answers of every rank to this one: channel q at q * chan_cap
    unsigned long long* req_cnt;  // [3 stages][RFX_MAX_RANKS]: requests this rank sent to every rank
    uint32_t ht_cap, pad;
};
struct SGView {
    SGPeer p[RFX_MAX_RANKS];
    int me, world, k, m;
    uint32_t B, bps;
    // Presence bits of ALL ranks' rows, one region of `rb` bits per minimiser bin (16 bits per row on average), the
    // whole array replicated on every rank (a rank fills the regions of its own bins, the others pull them: 2 B per row).
    // A node's neighbours mostly share its minimiser -- its bin -- and rows sit in the table grouped by bin, so the probes of
    // neighbouring threads fall into the same few hundred bytes; the array is streamed through once instead of being hit at
    // random (at 8 GPUs it is 8 x the size of one rank's rows and no longer fits the L2).
    const uint32_t* filter;
    uint32_t rb;       // bits per region (a multiple of 64)
    uint64_t inv_bps;  // ceil(2^64 / bps): bin -> owner without a division
    uint64_t chan_cap; // requests one rank may send to one rank per stage
    __device__ __forceinline__ int owner_of_bin(uint32_t bin) const { return bps == 1u ? (int)bin : (int)__umul64hi((uint64_t)bin, inv_bps); }
};

// what sg_publish exchanges: arena offsets first, then values
enum {
    GP_KEYS, GP_COUNTS, GP_HT, GP_BLOOM, GP_ALIVE, GP_LFLAG, GP_RFLAG, GP_EFFL, GP_EFFR, GP_SUCC, GP_PRED, GP_NXTL1, GP_L1ENT, GP_L1LOC, GP_L2UP0,
    GP_L2UP1, GP_L2NODE, GP_L2FIN, GP_CHAINLEN, GP_TAILRF, GP_CTGIDX, GP_CTGOFF, GP_CTGBASES, GP_INBOX, GP_RESPBOX, GP_REQCNT, GP_NPTR,
    GP_NROWS = GP_NPTR, GP_HTCAP, GP_BLOOMMASK, GP_HOST,  // GP_HOST: 6 host values, then up to 6 device values
    GP_NHOST = 6, GP_DEV = GP_HOST + GP_NHOST, GP_NDEV = 6, GP_END = GP_DEV + GP_NDEV
};
static_assert(GP_END <= PUB_VALS, "published block too small");

struct GShard {
    DevBuf rmin, work, pend_ref, inbox, respbox, req_cnt, nxt_l1, l1_ent, l1_loc, l1_fin, l1_dst, l2_l1, l2_node, l2_up[2], l2_fin, tail_rf, pubsrc, all_keys, all_counts;
    uint64_t n_remote = 0, n_l1 = 0, n_l2 = 0, n_rows_global = 0, n_oriented_global = 0, n_contigs_global = 0, n_bases_global = 0;
    uint64_t chan_cap = 0;
    int fell_back = 0;
    uint32_t rb = 64;
};

// ---- neighbour lookup ------------------------------------------------------------------------------------------------
struct SGProbe {
    uint32_t gid;    // oriented node (NONE32: no such k-mer)
    uint32_t count;
    uint32_t alive;  // its alive byte (when asked for)
    uint32_t w;      // word w of an owner's answer: the candidate's right flag in the sorted filters' serve mode (0 otherwise)
};
// a request to the owner of a k-mer / its answer
template <class KT> struct alignas(16) SGReq {
    KT key;        // canonical form
    uint32_t oid;  // asking node (local id on the sender) | bit 31: the asked orientation IS the canonical form
    uint32_t pad;
};
static_assert(sizeof(SGReq<uint64_t>) == 16 && sizeof(SGReq<u128>) == 32, "requests are 16 / 32 bytes");
constexpr uint32_t SG_REF_MASK = 0x1fffffffu;
constexpr uint32_t SG_REF_ASK = 0x80000000u;  // | owner: a candidate that still has to be asked for (only inside pass 1)

// row of a canonical k-mer in THIS rank's index, NONE32 if absent
template <class KT> __device__ __forceinline__ uint32_t sg_lookup_own(const SGPeer& Me, KT canon, uint64_t kh) {
    const KT* keys = reinterpret_cast<const KT*>(Me.keys);
    const uint32_t cap = Me.ht_cap;
    uint32_t slot = (uint32_t)(((uint64_t)(uint32_t)(kh >> 20) * cap) >> 32);
    while (true) {
        const uint32_t v = Me.ht[slot];
        if (v == NONE32) return NONE32;
        if (keys[v] == canon) return v;
        slot = slot + 1 == cap ? 0u : slot + 1;
    }
}
// The oriented k-mer Z = the (k-1)-mer it shares with the asking node (minimum h_side over its m-mers, bin bin_side) plus
// one new m-mer (hash h_new).
//   PASS 1  a candidate in this rank's bins is looked up.  One in a peer's bins that passes the presence bits is marked
//           (ref = SG_REF_ASK | owner); sg_finish_pass1 turns the marks of a block into requests in the owners' inboxes and
//           ref = owner << 29 | position, which says where the answer will be.  The node has to wait.
//   PASS 2  (nodes that waited) a candidate with a ref takes the owner's answer, the others are looked up again.
// SORTED: a local candidate is read as sg_serve_kernel<SORTED> answers for a remote one: count = its lflag, w = its rflag.
template <class KT, int PASS, bool WANT_ALIVE, bool SORTED = false>
__device__ __forceinline__ SGProbe sg_probe(const SGView& V, KT Z, uint32_t h_new, uint32_t h_side, uint32_t bin_side, uint32_t oid, int stage, uint32_t& ref,
                                            unsigned long long* dstat) {
    SGProbe out{NONE32, 0u, 0u, 0u};
    if (PASS == 2 && ref != NONE32) {
        const uint4 a = V.p[V.me].respbox[(uint64_t)(ref >> 29) * V.chan_cap + (ref & SG_REF_MASK)];

        out.gid = a.y == NONE32 ? NONE32 : gid_make((int)(ref >> 29), a.y);
        out.count = a.x; out.alive = a.z; out.w = a.w;
        return out;
    }
    const KT zc = revcomp(Z, V.k);
    const bool fwd = !(zc < Z);
    const KT canon = fwd ? Z : zc;
    const uint32_t bin = h_new < h_side ? bin_of_minimizer(h_new, V.B) : bin_side;
    const uint64_t kh = key_hash(canon);
    const uint64_t bit = (uint64_t)bin * V.rb + (((uint64_t)(uint32_t)kh * V.rb) >> 32);
    if (!((V.filter[bit >> 5] >> (bit & 31u)) & 1u)) return out;
    const int r = V.owner_of_bin(bin);
    if (r != V.me) {
        if (PASS == 1) ref = SG_REF_ASK | (uint32_t)r;  // asked of rank r once the block has reserved its channel positions (sg_finish_pass1)
        return out;  // (PASS 2: not reached -- such a candidate has a ref)
    }
    const SGPeer& Me = V.p[V.me];
    const uint32_t v = sg_lookup_own<KT>(Me, canon, kh);
    if (v == NONE32) return out;
    const uint32_t y = 2u * v + (fwd ? 0u : 1u);
    out.gid = gid_make(V.me, y);
    out.count = SORTED ? (uint32_t)Me.lflag[y] : Me.counts[v];
    if (WANT_ALIVE) out.alive = Me.alive[y];
    if (SORTED) out.w = (uint32_t)Me.rflag[y];
    return out;
}
// The owner's side: every request of every peer is looked up in the own index, the answer goes into the asker's answer box.
// LINK: a surviving node that is asked for by its predecessor notes that predecessor (the asker links to it in its second pass).
// SORTED (left filter of rfx_sort_kmers_sharded): the answer is {coverage, node, alive byte, right flag} as the right filter left
// them on the node (lflag / rflag) instead of {count, node, alive byte, 0}.
template <class KT, bool LINK, bool SORTED = false>
__global__ void __launch_bounds__(256) sg_serve_kernel(const __grid_constant__ SGView V, int stage, unsigned long long* dstat) {
    const SGPeer& Me = V.p[V.me];
    unsigned long long served = 0;
    for (int q = 1; q < V.world; q++) {
        const int r = (V.me + q) % V.world;  // sender
        const unsigned long long cnt_raw = *reinterpret_cast<const volatile unsigned long long*>(&V.p[r].req_cnt[stage * RFX_MAX_RANKS + V.me]);
        const uint64_t cnt = cnt_raw < V.chan_cap ? cnt_raw : V.chan_cap;
        const SGReq<KT>* in = reinterpret_cast<const SGReq<KT>*>(Me.inbox) + (uint64_t)r * V.chan_cap;
        uint4* out = V.p[r].respbox + (uint64_t)V.me * V.chan_cap;
        for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < cnt; i += (uint64_t)gridDim.x * blockDim.x) {
            const SGReq<KT> rq = in[i];
            const uint32_t v = sg_lookup_own<KT>(Me, rq.key, key_hash(rq.key));
            uint4 a = make_uint4(0u, NONE32, 0u, 0u);
            if (v != NONE32) {
                const uint32_t y = 2u * v + ((rq.oid & 0x80000000u) ? 0u : 1u);
                a.x = SORTED ? (uint32_t)Me.lflag[y] : Me.counts[v]; a.y = y; a.z = Me.alive[y];
                if (SORTED) a.w = (uint32_t)Me.rflag[y];
                if (LINK && (a.z & 2)) Me.pred[y] = gid_make(r, rq.oid & SG_REF_MASK);  // the left filter left at most one predecessor
            }
            out[i] = a;  // posted store into the asker's memory
            served++;
        }
    }
    __syncwarp();
    served = __reduce_add_sync(0xffffffffu, (uint32_t)served);
    if ((threadIdx.x & 31) == 0 && served) atomicAdd(&dstat[DS_REMOTE], served);
}
// the two passes of a K5 kernel: pass 1 runs over the own nodes and lists the ones that wait for answers, pass 2 runs over that list
struct SGWork {
    uint32_t* list;               // waiting nodes (pass 1 appends, pass 2 reads)
    uint4* refs;                  // per waiting node: where the answers for its four candidates are (NONE32: not asked)
    unsigned long long* counter;  // entries in the list (device)
};
template <int PASS> __device__ __forceinline__ uint64_t sg_work_count(uint64_t n, const SGWork& W) { return PASS == 1 ? n : (uint64_t)*W.counter; }
// End of a pass-1 iteration, called by every thread of the block: the marked candidates become requests (positions in the
// channels reserved per block: one global atomic per owner and block, the lanes rank themselves in shared memory) and the
// nodes that wait go onto the work list with the places of their answers.  zfun(b) rebuilds candidate b of this thread's node.
template <class KT, class ZFun>
__device__ __forceinline__ void sg_finish_pass1(const SGView& V, const SGWork& W, int stage, uint32_t oid, uint32_t (&ref)[4], ZFun zfun, unsigned long long* dstat) {
    __shared__ uint32_t s_req[RFX_MAX_RANKS], s_wait;
    __shared__ unsigned long long s_rbase[RFX_MAX_RANKS], s_wbase;
    const uint32_t lane = threadIdx.x & 31u;
    if (threadIdx.x < RFX_MAX_RANKS) s_req[threadIdx.x] = 0;
    if (threadIdx.x == RFX_MAX_RANKS) s_wait = 0;
    __syncthreads();
    uint32_t lpos[4];
    bool waits = false;
#pragma unroll
    for (int b = 0; b < 4; b++) {
        lpos[b] = 0;
        if (ref[b] != NONE32) { waits = true; lpos[b] = atomicAdd(&s_req[ref[b] & 7u], 1u); }
    }
    const uint32_t wm = __ballot_sync(0xffffffffu, waits);
    uint32_t wbase = 0;
    if (lane == 0 && wm) wbase = atomicAdd(&s_wait, (uint32_t)__popc(wm));
    wbase = __shfl_sync(0xffffffffu, wbase, 0);
    __syncthreads();
    if (threadIdx.x < RFX_MAX_RANKS && s_req[threadIdx.x])
        s_rbase[threadIdx.x] = atomicAdd(&V.p[V.me].req_cnt[stage * RFX_MAX_RANKS + threadIdx.x], (unsigned long long)s_req[threadIdx.x]);
    if (threadIdx.x == RFX_MAX_RANKS && s_wait) s_wbase = atomicAdd(W.counter, (unsigned long long)s_wait);
    __syncthreads();
    if (!waits) return;
#pragma unroll
    for (int b = 0; b < 4; b++) {
        if (ref[b] == NONE32) continue;
        const uint32_t r = ref[b] & 7u;
        const unsigned long long i = s_rbase[r] + lpos[b];
        if (i < V.chan_cap) {
            const KT Z = zfun((uint32_t)b);
            const KT zc = revcomp(Z, V.k);
            const bool fwd = !(zc < Z);
            SGReq<KT> q;
            q.key = fwd ? Z : zc; q.oid = oid | (fwd ? 0x80000000u : 0u); q.pad = 0;
            reinterpret_cast<SGReq<KT>*>(V.p[r].inbox)[(uint64_t)V.me * V.chan_cap + i] = q;  // posted store into the owner's memory
            ref[b] = (r << 29) | (uint32_t)i;
        } else {
            atomicExch(&dstat[DS_GRAPH_ERR], 4ull);
            ref[b] = NONE32;
        }
    }
    const unsigned long long at = s_wbase + wbase + __popc(wm & ((1u << lane) - 1u));
    W.list[at] = oid;
    W.refs[at] = make_uint4(ref[0], ref[1], ref[2], ref[3]);
}
__device__ __forceinline__ void sg_work_pop(const SGWork& W, uint64_t i, uint32_t& oid, uint32_t (&ref)[4]) {
    oid = W.list[i];
    const uint4 r = W.refs[i];
    ref[0] = r.x; ref[1] = r.y; ref[2] = r.z; ref[3] = r.w;
}

template <class KT> __device__ __forceinline__ KT sg_oriented(const SGView& V, uint32_t g) {
    const uint32_t l = gid_loc(g);
    const KT key = reinterpret_cast<const KT*>(V.p[gid_rank(g)].keys)[l >> 1];
    return (l & 1u) ? revcomp(key, V.k) : key;
}

// Per row, once: the minima of the m-mer hashes inside the first / the last k-1 bases of the canonical k-mer with their bins
// (the reverse strand sees the same two swapped: m-mer hashes are strand symmetric).  A neighbour's minimiser -- hence its bin
// and owner -- is then min(one new m-mer, one of the two).  The row's own bin must belong to this rank, or neighbours would
// look for it elsewhere (checked); its presence bit is set in that bin's region.
template <class KT>
__global__ void sg_row_minima_kernel(const KT* __restrict__ keys, uint64_t n_rows, int k, int m, uint32_t B, uint32_t bin_lo, uint32_t bin_hi, uint32_t rb,
                                     uint4* __restrict__ rmin, uint32_t* filter, unsigned long long* dstat) {
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n_rows; r += (uint64_t)gridDim.x * blockDim.x) {
        const KT key = keys[r];
        uint32_t a, b;
        const uint32_t bin = row_bin<KT>(key, k, m, B, a, b);
        rmin[r] = make_uint4(a, b, bin_of_minimizer(a, B), bin_of_minimizer(b, B));
        if (bin < bin_lo || bin >= bin_hi) atomicExch(&dstat[DS_GRAPH_ERR], 3ull);
        const uint64_t bit = (uint64_t)bin * rb + (((uint64_t)(uint32_t)key_hash(key) * rb) >> 32);
        atomicOr(&filter[bit >> 5], 1u << (bit & 31u));
    }
}

// ---- K5: A7, A8, links (rules: rfx_core.h; the single-GPU kernels of rfx_graph.cu, neighbours in a peer's bins asked by message) ----
template <class KT, int PASS>
__global__ void __launch_bounds__(256, 8) sg_right_filter_kernel(const __grid_constant__ SGView V, int E, uint64_t n, const uint4* __restrict__ rmin, SGWork W, unsigned long long* dstat) {
    const SGPeer& Me = V.p[V.me];
    const KT* keys = reinterpret_cast<const KT*>(Me.keys);
    const uint64_t count = sg_work_count<PASS>(n, W);
    for (uint64_t i0 = (uint64_t)blockIdx.x * blockDim.x; i0 < count; i0 += (uint64_t)gridDim.x * blockDim.x) {  // block-uniform trip count (sg_work_push)
        const uint64_t i = i0 + threadIdx.x;
        uint32_t ref[4] = {NONE32, NONE32, NONE32, NONE32};
        uint32_t oid = 0;
        KT prefix = 0;
        if (i < count) {
            if (PASS == 1) oid = (uint32_t)i; else sg_work_pop(W, i, oid, ref);
            const uint32_t row = oid >> 1;
            const KT key = keys[row];
            const KT rc = revcomp(key, V.k);
            if ((oid & 1u) && rc == key) { Me.alive[oid] = 0; Me.rflag[oid] = 0; }  // palindrome: one node, not two
            else {
                const KT X = (oid & 1u) ? rc : key;
                prefix = X >> 2;
                const uint32_t myb = (uint32_t)X & 3u;
                const uint4 mm = rmin[row];
                const uint32_t pre_min = (oid & 1u) ? mm.y : mm.x, pre_bin = (oid & 1u) ? mm.w : mm.z;
                uint32_t cnt[4];
                bool dup[4];
#pragma unroll
                for (uint32_t b = 0; b < 4; b++) {
                    if (b == myb) { cnt[b] = Me.counts[row]; dup[b] = (rc == key); }
                    else {
                        const KT Z = (prefix << 2) | (KT)b;
                        const SGProbe pr = sg_probe<KT, PASS, false>(V, Z, last_mm_of<KT>(prefix, b, V.m), pre_min, pre_bin, oid, 0, ref[b], dstat);
                        cnt[b] = pr.gid == NONE32 ? 0u : pr.count;
                        dup[b] = (Z == revcomp(Z, V.k));
                    }
                }
                if (PASS == 2 || (ref[0] & ref[1] & ref[2] & ref[3]) == NONE32) {
                    const ForkResult res = right_fork(cnt, dup, E, V.k - 1);
                    Me.alive[oid] = (uint8_t)(((res.winner == (int)myb) ? 1 : 0) | (res.flag < 0 ? 4 : 0));
                    Me.rflag[oid] = res.flag;
                }
            }
        }
        if (PASS == 1) sg_finish_pass1<KT>(V, W, 0, oid, ref, [&](uint32_t b) { return (KT)((prefix << 2) | (KT)b); }, dstat);
    }
}

template <class KT, int PASS>
__global__ void __launch_bounds__(256, 8) sg_left_filter_kernel(const __grid_constant__ SGView V, int E, uint64_t n, const uint4* __restrict__ rmin, SGWork W, unsigned long long* dstat) {
    const SGPeer& Me = V.p[V.me];
    const int top = 2 * (V.k - 1);
    const KT sufmask = mask_bases<KT>(V.k - 1);
    const uint64_t count = sg_work_count<PASS>(n, W);
    for (uint64_t i0 = (uint64_t)blockIdx.x * blockDim.x; i0 < count; i0 += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t i = i0 + threadIdx.x;
        uint32_t ref[4] = {NONE32, NONE32, NONE32, NONE32};
        uint32_t oid = 0;
        KT suffix = 0;
        if (i < count) {
            if (PASS == 1) { oid = (uint32_t)i; Me.lflag[oid] = 0; } else sg_work_pop(W, i, oid, ref);
            if (Me.alive[oid] & 1) {
                const KT X = sg_oriented<KT>(V, gid_make(V.me, oid));
                suffix = X & sufmask;
                const uint32_t mya = (uint32_t)(X >> top) & 3u;
                const uint4 mm = rmin[oid >> 1];
                const uint32_t suf_min = (oid & 1u) ? mm.x : mm.y, suf_bin = (oid & 1u) ? mm.z : mm.w;
                uint32_t cnt[4];
#pragma unroll
                for (uint32_t a = 0; a < 4; a++) {
                    if (a == mya) cnt[a] = Me.counts[oid >> 1];
                    else {
                        const SGProbe pr = sg_probe<KT, PASS, true>(V, ((KT)a << top) | suffix, first_mm_of<KT>(suffix, a, V.k, V.m), suf_min, suf_bin, oid, 1, ref[a], dstat);
                        cnt[a] = (pr.gid != NONE32 && (pr.alive & 1)) ? pr.count : 0u;
                    }
                }
                if (PASS == 2 || (ref[0] & ref[1] & ref[2] & ref[3]) == NONE32) {
                    const ForkResult res = left_fork(cnt, E, V.k - 1);
                    if (res.winner == (int)mya) { Me.alive[oid] = (uint8_t)((Me.alive[oid] & 4) | 3 | (res.flag < 0 ? 8 : 0)); Me.lflag[oid] = res.flag; }
                }
            }
        }
        if (PASS == 1) sg_finish_pass1<KT>(V, W, 1, oid, ref, [&](uint32_t a) { return (KT)(((KT)a << top) | suffix); }, dstat);
    }
}

// Raw links over every junction (which of them hold is decided by the budget walks, as on one GPU).  A successor in a peer's
// bins: the owner, asked for it, notes this node as its predecessor while it answers (sg_serve_kernel<LINK>); the alive byte in
// the answer carries the sign of the successor's left flag, which is all the junction test needs.
template <class KT, int PASS>
__global__ void __launch_bounds__(256, 8) sg_link_kernel(const __grid_constant__ SGView V, uint64_t n, const uint4* __restrict__ rmin, SGWork W, unsigned long long* dstat) {
    const SGPeer& Me = V.p[V.me];
    const KT sufmask = mask_bases<KT>(V.k - 1);
    const uint64_t count = sg_work_count<PASS>(n, W);
    for (uint64_t i0 = (uint64_t)blockIdx.x * blockDim.x; i0 < count; i0 += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t i = i0 + threadIdx.x;
        uint32_t ref[4] = {NONE32, NONE32, NONE32, NONE32};
        uint32_t oid = 0;
        KT suffix = 0;
        if (i < count) {
            if (PASS == 1) oid = (uint32_t)i; else sg_work_pop(W, i, oid, ref);
            const int32_t my_l = Me.lflag[oid], my_r = Me.rflag[oid];
            if (PASS == 1) { Me.eff_l[oid] = my_l; Me.eff_r[oid] = my_r; }
            if (Me.alive[oid] & 2) {
                const uint32_t self = gid_make(V.me, oid);
                const KT X = sg_oriented<KT>(V, self);
                suffix = X & sufmask;
                const uint4 mm = rmin[oid >> 1];
                const uint32_t suf_min = (oid & 1u) ? mm.x : mm.y, suf_bin = (oid & 1u) ? mm.z : mm.w;
                uint32_t next = NONE32;
                bool next_l_neg = false;
                int n_cand = 0;
#pragma unroll
                for (uint32_t b = 0; b < 4; b++) {
                    const SGProbe pr = sg_probe<KT, PASS, true>(V, (suffix << 2) | (KT)b, last_mm_of<KT>(suffix, b, V.m), suf_min, suf_bin, oid, 2, ref[b], dstat);
                    if (pr.gid != NONE32 && (pr.alive & 2)) { next = pr.gid; next_l_neg = (pr.alive & 8) != 0; n_cand++; }
                }
                if (PASS == 2 || (ref[0] & ref[1] & ref[2] & ref[3]) == NONE32) {
                    if (n_cand > 1) atomicExch(&dstat[DS_GRAPH_ERR], 1ull);
                    else {
                        if (my_l >= 0 || my_r >= 0) atomicAdd(&dstat[DS_FLAGGED], 1ull);
                        if (next != NONE32) {
                            const bool joins = (my_r < 0) == next_l_neg;  // junction_joins on the signs
                            if (!joins) atomicAdd(&dstat[DS_BUDGET], 1ull);
                            if (next == self) {
                                if (joins) atomicAdd(&dstat[DS_CYCLES], 1ull);  // 1-cycle: a record never merges with itself
                            } else {
                                Me.succ[oid] = next;
                                if (gid_rank(next) == V.me && atomicExch(&Me.pred[gid_loc(next)], self) != NONE32) atomicExch(&dstat[DS_GRAPH_ERR], 2ull);
                            }
                        }
                    }
                }
            }
        }
        if (PASS == 1) sg_finish_pass1<KT>(V, W, 2, oid, ref, [&](uint32_t b) { return (KT)((suffix << 2) | (KT)b); }, dstat);
    }
}

// ---- Count_<k>_sorted across ranks (rfx_sort_kmers_sharded; the single-GPU sorted_right_kernel / sorted_left_kernel) -------
// The probes, requests and answers of A7 / A8 (request stages 0 and 1), the rules sorted_right_fork / sorted_left_fork.  The
// right filter leaves the coverage it carries on in lflag and the right flag in rflag; the left filter needs both of every
// candidate: a local one's from the own arrays, a remote one's from its owner (sg_serve_kernel<SORTED>: {lflag, node, alive, rflag}).
template <class KT, int PASS>
__global__ void __launch_bounds__(256, 8) sg_sorted_right_kernel(const __grid_constant__ SGView V, int E, double fold, int Xf, uint64_t n, const uint4* __restrict__ rmin,
                                                                 SGWork W, unsigned long long* dstat) {
    const SGPeer& Me = V.p[V.me];
    const KT* keys = reinterpret_cast<const KT*>(Me.keys);
    const uint64_t count = sg_work_count<PASS>(n, W);
    for (uint64_t i0 = (uint64_t)blockIdx.x * blockDim.x; i0 < count; i0 += (uint64_t)gridDim.x * blockDim.x) {  // block-uniform trip count
        const uint64_t i = i0 + threadIdx.x;
        uint32_t ref[4] = {NONE32, NONE32, NONE32, NONE32};
        uint32_t oid = 0;
        KT prefix = 0;
        if (i < count) {
            if (PASS == 1) oid = (uint32_t)i; else sg_work_pop(W, i, oid, ref);
            const uint32_t row = oid >> 1;
            const KT key = keys[row];
            const KT rc = revcomp(key, V.k);
            if ((oid & 1u) && rc == key) Me.alive[oid] = 0;  // palindrome: one node, not two
            else {
                const KT Xk = (oid & 1u) ? rc : key;
                prefix = Xk >> 2;
                const uint32_t myb = (uint32_t)Xk & 3u;
                const uint4 mm = rmin[row];
                const uint32_t pre_min = (oid & 1u) ? mm.y : mm.x, pre_bin = (oid & 1u) ? mm.w : mm.z;
                uint32_t cnt[4];
                bool dup[4];
#pragma unroll
                for (uint32_t b = 0; b < 4; b++) {
                    if (b == myb) { cnt[b] = Me.counts[row]; dup[b] = (rc == key); }
                    else {
                        const KT Z = (prefix << 2) | (KT)b;
                        const SGProbe pr = sg_probe<KT, PASS, false>(V, Z, last_mm_of<KT>(prefix, b, V.m), pre_min, pre_bin, oid, 0, ref[b], dstat);
                        cnt[b] = pr.gid == NONE32 ? 0u : pr.count;
                        dup[b] = (Z == revcomp(Z, V.k));
                    }
                }
                if (PASS == 2 || (ref[0] & ref[1] & ref[2] & ref[3]) == NONE32) {
                    const SortedFork res = sorted_right_fork(cnt, dup, E, fold, Xf);
                    const bool won = res.winner == (int)myb;
                    Me.alive[oid] = won ? 1 : 0;
                    if (won) { Me.lflag[oid] = res.left; Me.rflag[oid] = res.right; }
                }
            }
        }
        if (PASS == 1) sg_finish_pass1<KT>(V, W, 0, oid, ref, [&](uint32_t b) { return (KT)((prefix << 2) | (KT)b); }, dstat);
    }
}

// A remote candidate's coverage and right flag are read only by its owner's stage-1 serve, which runs behind the barrier that
// follows every rank's right pass 2: they are final there without a barrier of their own.  Local ones are final once this
// rank's right pass 2 is (stream order).  The winner writes srt_left / srt_right, never lflag / rflag, which peers may still ask for.
template <class KT, int PASS>
__global__ void __launch_bounds__(256, 8) sg_sorted_left_kernel(const __grid_constant__ SGView V, int E, double fold, int Xf, uint64_t n, const uint4* __restrict__ rmin,
                                                                SGWork W, int32_t* __restrict__ out_left, int32_t* __restrict__ out_right, unsigned long long* dstat) {
    const SGPeer& Me = V.p[V.me];
    const int top = 2 * (V.k - 1);
    const KT sufmask = mask_bases<KT>(V.k - 1);
    const uint64_t count = sg_work_count<PASS>(n, W);
    for (uint64_t i0 = (uint64_t)blockIdx.x * blockDim.x; i0 < count; i0 += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t i = i0 + threadIdx.x;
        uint32_t ref[4] = {NONE32, NONE32, NONE32, NONE32};
        uint32_t oid = 0;
        KT suffix = 0;
        if (i < count) {
            if (PASS == 1) oid = (uint32_t)i; else sg_work_pop(W, i, oid, ref);
            if (Me.alive[oid] & 1) {
                const KT Xk = sg_oriented<KT>(V, gid_make(V.me, oid));
                suffix = Xk & sufmask;
                const uint32_t mya = (uint32_t)(Xk >> top) & 3u;
                const uint4 mm = rmin[oid >> 1];
                const uint32_t suf_min = (oid & 1u) ? mm.x : mm.y, suf_bin = (oid & 1u) ? mm.z : mm.w;
                int32_t cv[4], rf[4];
#pragma unroll
                for (uint32_t a = 0; a < 4; a++) {
                    cv[a] = 0; rf[a] = 0;
                    if (a == mya) { cv[a] = Me.lflag[oid]; rf[a] = Me.rflag[oid]; }
                    else {
                        const SGProbe pr = sg_probe<KT, PASS, true, true>(V, ((KT)a << top) | suffix, first_mm_of<KT>(suffix, a, V.k, V.m), suf_min, suf_bin, oid, 1, ref[a], dstat);
                        if (pr.gid != NONE32 && (pr.alive & 1)) { cv[a] = (int32_t)pr.count; rf[a] = (int32_t)pr.w; }
                    }
                }
                if (PASS == 2 || (ref[0] & ref[1] & ref[2] & ref[3]) == NONE32) {
                    const SortedFork res = sorted_left_fork(cv, rf, E, fold, Xf);
                    if (res.winner == (int)mya) { Me.alive[oid] = 3; out_left[oid] = res.left; out_right[oid] = res.right; }  // bit 0 stays: others still read it
                }
            }
        }
        if (PASS == 1) sg_finish_pass1<KT>(V, W, 1, oid, ref, [&](uint32_t a) { return (KT)(((KT)a << top) | suffix); }, dstat);
    }
}

// ---- budget walks across ranks (rfx_graph.cu: budget_walk_kernel, every array read through its owner) ----------------------
struct SGWalkArrays {  // DIR 0: bud = rflag, face = lflag, nxt = succ, prv = pred, eff = eff_r;  DIR 1: mirrored
    __device__ __forceinline__ static int32_t bud(const SGView& V, int DIR, uint32_t g) { return (DIR == 0 ? V.p[gid_rank(g)].rflag : V.p[gid_rank(g)].lflag)[gid_loc(g)]; }
    __device__ __forceinline__ static int32_t face(const SGView& V, int DIR, uint32_t g) { return (DIR == 0 ? V.p[gid_rank(g)].lflag : V.p[gid_rank(g)].rflag)[gid_loc(g)]; }
    __device__ __forceinline__ static uint32_t nxt(const SGView& V, int DIR, uint32_t g) { return (DIR == 0 ? V.p[gid_rank(g)].succ : V.p[gid_rank(g)].pred)[gid_loc(g)]; }
    __device__ __forceinline__ static uint32_t prv(const SGView& V, int DIR, uint32_t g) { return (DIR == 0 ? V.p[gid_rank(g)].pred : V.p[gid_rank(g)].succ)[gid_loc(g)]; }
};
template <class KT, int DIR> __global__ void sg_budget_walk_kernel(const __grid_constant__ SGView V, uint64_t n, int bmax, unsigned long long* dstat) {
    typedef SGWalkArrays W;
    const SGPeer& Me = V.p[V.me];
    for (uint64_t x = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; x < n; x += (uint64_t)gridDim.x * blockDim.x) {
        if (!(Me.alive[x] & 2)) continue;
        const uint32_t s = gid_make(V.me, (uint32_t)x);
        if (W::bud(V, DIR, s) < 0) continue;
        if (W::nxt(V, DIR, s) == NONE32) continue;  // nothing downstream to absorb
        uint32_t stop = s;
        bool fresh = true;
        if (W::face(V, DIR, s) < 0 && W::prv(V, DIR, s) != NONE32) {
            uint32_t u = W::prv(V, DIR, s), start = NONE32;
            int gap = 0;
            while (true) {
                if (u == s) break;  // closed path without a fixed point: smallest fork winner starts
                gap = W::bud(V, DIR, u) < 0 ? gap + 1 : 0;
                if (W::face(V, DIR, u) >= 0 || W::prv(V, DIR, u) == NONE32 || gap >= bmax) { start = u; break; }
                u = W::prv(V, DIR, u);
            }
            if (start == NONE32) {
                uint32_t mn = s;
                KT mk = sg_oriented<KT>(V, s);
                for (u = W::prv(V, DIR, s); u != s; u = W::prv(V, DIR, u))
                    if (W::bud(V, DIR, u) >= 0) { const KT ku = sg_oriented<KT>(V, u); if (ku < mk) { mk = ku; mn = u; } }
                start = mn;
                stop = mn;
            }
            if (start != s) {
                int32_t Eb = W::bud(V, DIR, start);
                for (uint32_t v = W::nxt(V, DIR, start); v != s; v = W::nxt(V, DIR, v)) Eb = (W::face(V, DIR, v) < 0 && Eb >= 1) ? Eb - 1 : W::bud(V, DIR, v);
                fresh = !(Eb >= 1);  // face[s] < 0 here
            }
        }
        if (!fresh) continue;  // absorbed: the walk that takes it writes its flag
        int32_t rem = W::bud(V, DIR, s);
        uint32_t cur = s;
        unsigned long long taken = 0;
        while (rem >= 1) {
            const uint32_t z = W::nxt(V, DIR, cur);
            if (z == NONE32 || z == stop || z == s || W::face(V, DIR, z) >= 0) break;
            rem--;
            (DIR == 0 ? V.p[gid_rank(z)].eff_r : V.p[gid_rank(z)].eff_l)[gid_loc(z)] = rem;
            const uint32_t j = DIR == 0 ? cur : z;  // the junction's left node
            alive_or(V.p[gid_rank(j)].alive, gid_loc(j), DIR == 0 ? 16u : 32u);
            taken++;
            cur = z;
        }
        if (taken) atomicAdd(&dstat[DS_ABSORBED], taken);
    }
}
__global__ void sg_junction_finalize_kernel(const __grid_constant__ SGView V, uint64_t n) {
    const SGPeer& Me = V.p[V.me];
    for (uint64_t x = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; x < n; x += (uint64_t)gridDim.x * blockDim.x) {
        if (!(Me.alive[x] & 2)) continue;
        const uint32_t y = Me.succ[x];
        if (y == NONE32) continue;
        if ((Me.alive[x] & 48) || junction_joins(Me.eff_r[x], V.p[gid_rank(y)].eff_l[gid_loc(y)])) continue;
        Me.succ[x] = NONE32;
        V.p[gid_rank(y)].pred[gid_loc(y)] = NONE32;
    }
}

// ---- K6: two levels of splitters ----------------------------------------------------------------------------------------
__device__ __forceinline__ bool sg_l1_sample(uint32_t x) { return (fmix32(x ^ 0xa5a5a5a5u) & 63u) == 0u; }
__device__ __forceinline__ bool sg_l2_sample(uint32_t l1_gid) { return (fmix32(l1_gid ^ 0x3c6ef372u) & 7u) == 0u; }

__global__ void sg_select_kernel(const __grid_constant__ SGView V, uint64_t n, uint32_t* __restrict__ spl_id, uint32_t* __restrict__ spl_node, uint32_t* __restrict__ l2_l1,
                                 unsigned long long* dstat) {
    const SGPeer& Me = V.p[V.me];
    for (uint64_t x0 = (uint64_t)blockIdx.x * blockDim.x; x0 < n; x0 += (uint64_t)gridDim.x * blockDim.x) {  // block-uniform trip count
        const uint64_t x = x0 + threadIdx.x;
        uint32_t p = 0;
        bool s1 = false;
        if (x < n && (Me.alive[x] & 2)) {
            p = Me.pred[x];
            s1 = p == NONE32 || gid_rank(p) != V.me || sg_l1_sample((uint32_t)x);
        }
        const uint32_t id = (uint32_t)block_reserve(s1, &dstat[DS_NSPL]);
        const bool s2 = s1 && (p == NONE32 || sg_l2_sample(gid_make(V.me, id)));
        const uint32_t j = (uint32_t)block_reserve(s2, &dstat[DS_NL2]);
        if (s1) {
            spl_node[id] = (uint32_t)x;
            if (s2) {
                l2_l1[j] = id;
                Me.l2_node[j] = (uint32_t)x;
                Me.l2_up[0][j] = ad_pack(gid_make(V.me, j), 0u);  // a non-head is overwritten by the level-2 walk that reaches it
            }
            Me.l1_ent[id].y = (unsigned long long)j;  // NONE32 unless level 2
            // the predecessor lives on another rank: tell it where its segment ends (a posted store; its walk never has to ask)
            if (p != NONE32 && gid_rank(p) != V.me) V.p[gid_rank(p)].nxt_l1[gid_loc(p)] = gid_make(V.me, id);
        }
        if (x < n) spl_id[x] = s1 ? id : NONE32;
    }
}
// level-1 walk: purely local; the segment ends in front of the next level-1 splitter (on this rank or the first node on another)
__global__ void sg_l1_walk_kernel(const __grid_constant__ SGView V, uint64_t m1, const uint32_t* __restrict__ spl_id, const uint32_t* __restrict__ spl_node, uint64_t* __restrict__ loc) {
    const SGPeer& Me = V.p[V.me];
    for (uint64_t id = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; id < m1; id += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t x = spl_node[id];
        uint32_t off = 0, next = NONE32;
        loc[x] = ad_pack((uint32_t)id, 0u);
        uint32_t y = Me.succ[x];
        while (y != NONE32) {
            if (gid_rank(y) != V.me) { next = Me.nxt_l1[x]; break; }  // left here by the successor's owner (sg_select_kernel)
            const uint32_t yl = gid_loc(y);
            const uint32_t s = spl_id[yl];
            if (s != NONE32) { next = gid_make(V.me, s); break; }
            off++;
            loc[yl] = ad_pack((uint32_t)id, off);
            x = yl;
            y = Me.succ[yl];
        }
        Me.l1_ent[id].x = ad_pack(next, off + 1u);
    }
}
// level-2 walk over the level-1 list: stamps (owner, nodes in front) on every level-1 splitter it passes, ends at the next level-2 splitter
__global__ void sg_l2_walk_kernel(const __grid_constant__ SGView V, uint64_t m2, const uint32_t* __restrict__ l2_l1) {
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < m2; j += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t self = gid_make(V.me, (uint32_t)j);
        const uint32_t a = l2_l1[j];
        uint32_t dist = 0;
        V.p[V.me].l1_loc[a] = ad_pack(self, 0u);
        unsigned long long nl = V.p[V.me].l1_ent[a].x;
        while (true) {  // one 16-byte read and one 8-byte store per hop, most of them in a peer's memory
            const uint32_t nx = (uint32_t)nl;
            dist += (uint32_t)(nl >> 32);
            if (nx == NONE32) break;
            const SGPeer& Q = V.p[gid_rank(nx)];
            const ulonglong2 e = Q.l1_ent[gid_loc(nx)];
            const uint32_t t = (uint32_t)e.y;
            if (t != NONE32) { Q.l2_up[0][t] = ad_pack(self, dist); break; }
            Q.l1_loc[gid_loc(nx)] = ad_pack(self, dist);
            nl = e.x;
        }
    }
}
// one round of pointer jumping over the level-2 list (Jacobi: everybody reads buffer `in`, writes its own entries of `out`)
__global__ void sg_l2_jump_kernel(const __grid_constant__ SGView V, uint64_t m2, int in) {
    const SGPeer& Me = V.p[V.me];
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < m2; j += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t mine = Me.l2_up[in][j];
        const uint32_t a = (uint32_t)mine;
        if (a == gid_make(V.me, (uint32_t)j)) { Me.l2_up[in ^ 1][j] = mine; continue; }
        const uint64_t up = V.p[gid_rank(a)].l2_up[in][gid_loc(a)];
        Me.l2_up[in ^ 1][j] = ad_pack((uint32_t)up, (uint32_t)(mine >> 32) + (uint32_t)(up >> 32));
    }
}
// Measured alternative (RFX_JUMP_FUSED=1; slower, see the call site): all rounds in ONE cooperative launch per rank (ranks on
// different devices only): between two rounds a grid-wide barrier, a cross-GPU barrier taken by block 0 (every rank writes the
// round's epoch into every rank's flags2[] and waits for its own to fill up) and another grid-wide barrier.
// The (ancestor, distance) words change under the kernel's feet by design, so they are read around the L1.
__global__ void __launch_bounds__(256) sg_l2_jump_all_kernel(const __grid_constant__ SGView V, PeerBases P, uint64_t m2, int rounds, unsigned long long epoch0,
                                                             unsigned long long* dstat) {
    cooperative_groups::grid_group grid = cooperative_groups::this_grid();
    const SGPeer& Me = V.p[V.me];
    int cur = 0;
    for (int r = 0; r < rounds; r++) {
        for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < m2; j += (uint64_t)gridDim.x * blockDim.x) {
            const uint64_t mine = *reinterpret_cast<const volatile uint64_t*>(&Me.l2_up[cur][j]);
            const uint32_t a = (uint32_t)mine;
            uint64_t out = mine;
            if (a != gid_make(V.me, (uint32_t)j)) {
                const uint64_t up = *reinterpret_cast<const volatile uint64_t*>(&V.p[gid_rank(a)].l2_up[cur][gid_loc(a)]);
                out = ad_pack((uint32_t)up, (uint32_t)(mine >> 32) + (uint32_t)(up >> 32));
            }
            Me.l2_up[cur ^ 1][j] = out;
        }
        __threadfence_system();
        grid.sync();
        if (blockIdx.x == 0 && (int)threadIdx.x < P.n) {
            const unsigned long long epoch = epoch0 + (unsigned long long)r + 1ull;
            const int q = threadIdx.x;
            __threadfence_system();
            *reinterpret_cast<volatile unsigned long long*>(&reinterpret_cast<ShardCtl*>(P.base[q])->flags2[P.me]) = epoch;
            const volatile unsigned long long* mine = &reinterpret_cast<ShardCtl*>(P.base[P.me])->flags2[q];
            const long long t0 = clock64();
            while (*mine < epoch) {
                if (clock64() - t0 > 40000000000ll) { dstat[DS_XBAR_ERR] = 1ull; break; }
                __nanosleep(100);
            }
            __threadfence_system();
        }
        grid.sync();
        cur ^= 1;
    }
}
__global__ void sg_l2_fin_kernel(const __grid_constant__ SGView V, uint64_t m2, int res, unsigned long long* dstat) {
    const SGPeer& Me = V.p[V.me];
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < m2; j += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t v = Me.l2_up[res][j];
        const uint32_t a = (uint32_t)v;
        const uint32_t head = gid_make(gid_rank(a), V.p[gid_rank(a)].l2_node[gid_loc(a)]);
        if (V.p[gid_rank(head)].pred[gid_loc(head)] != NONE32) atomicExch(&dstat[DS_SG_CYCLE], 1ull);  // the chain's first splitter is no head
        Me.l2_fin[j] = ad_pack(head, (uint32_t)(v >> 32));
    }
}
__global__ void sg_l1_fin_kernel(const __grid_constant__ SGView V, uint64_t m1, uint64_t* __restrict__ l1_fin, unsigned long long* dstat) {
    const SGPeer& Me = V.p[V.me];
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m1; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t l = Me.l1_loc[i];
        if (l == ~0ull) { atomicExch(&dstat[DS_SG_CYCLE], 1ull); l1_fin[i] = ~0ull; continue; }  // no level-2 walk came by: closed path
        const uint32_t o = (uint32_t)l;
        const uint64_t f = V.p[gid_rank(o)].l2_fin[gid_loc(o)];
        l1_fin[i] = ad_pack((uint32_t)f, (uint32_t)(f >> 32) + (uint32_t)(l >> 32));
    }
}
__global__ void sg_node_fin_kernel(const __grid_constant__ SGView V, uint64_t n, const uint64_t* __restrict__ loc, const uint64_t* __restrict__ l1_fin, uint64_t* __restrict__ ad,
                                   unsigned long long* dstat) {
    const SGPeer& Me = V.p[V.me];
    for (uint64_t x = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; x < n; x += (uint64_t)gridDim.x * blockDim.x) {
        if (!(Me.alive[x] & 2)) continue;
        const uint64_t l = loc[x];
        if (l == ~0ull) { atomicExch(&dstat[DS_SG_CYCLE], 1ull); continue; }  // no level-1 walk came by: closed path inside this rank
        const uint64_t f = l1_fin[(uint32_t)l];
        if (f == ~0ull) continue;
        const uint32_t d = (uint32_t)(f >> 32) + (uint32_t)(l >> 32);
        ad[x] = ad_pack((uint32_t)f, d);
        if (Me.succ[x] == NONE32) {  // tail: tell the head (wherever it lives) how long its chain is and what its right flag is
            const uint32_t h = (uint32_t)f;
            V.p[gid_rank(h)].chain_len[gid_loc(h)] = d + 1u;
            V.p[gid_rank(h)].tail_rf[gid_loc(h)] = Me.eff_r[x];
        }
    }
}

// ---- K7 -------------------------------------------------------------------------------------------------------------------
struct SContigIn {
    const uint8_t* alive;
    const uint32_t* pred;
    const uint32_t* chain_len;
    const int32_t* lflag;    // effective left flag of the head
    const int32_t* tail_rf;  // effective right flag of the chain's tail, stored at the head
    int k, min_contig;
    __device__ __forceinline__ U64x3 operator()(uint64_t x) const {
        if (!(alive[x] & 2)) return U64x3{0, 0, 0};
        if (pred[x] != NONE32) return U64x3{0, 0, 1};
        const uint64_t len = (uint64_t)chain_len[x] + (uint64_t)k - 1;
        const bool keep = !(lflag[x] <= -10000000 && tail_rf[x] <= -10000000) && len >= (uint64_t)min_contig;  // DSKmerToContig, ReflexivDSMain.java:749-754
        return keep ? U64x3{1, len, 1} : U64x3{0, 0, 1};
    }
};
struct SContigOut {
    const int32_t* lflag;
    const int32_t* tail_rf;
    uint32_t* ctg_idx;
    uint64_t* ctg_off;
    int32_t* ctg_left;
    int32_t* ctg_right;
    __device__ __forceinline__ void operator()(uint64_t x, U64x3 excl, U64x3 v) const {
        ctg_idx[x] = v.a ? (uint32_t)excl.a : NONE32;
        if (v.a) {
            ctg_off[excl.a] = excl.b;
            ctg_left[excl.a] = lflag[x];
            ctg_right[excl.a] = tail_rf[x];
        }
    }
};
// where the bases of a level-1 segment go: address of its first node's last base inside the head owner's buffer (0: contig not kept)
__global__ void sg_l1_dst_kernel(const __grid_constant__ SGView V, uint64_t m1, const uint64_t* __restrict__ l1_fin, unsigned long long* __restrict__ l1_dst) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m1; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t f = l1_fin[i];
        unsigned long long d = 0;
        if (f != ~0ull) {
            const uint32_t h = (uint32_t)f;
            const SGPeer& Q = V.p[gid_rank(h)];
            const uint32_t ci = Q.ctg_idx[gid_loc(h)];
            if (ci != NONE32) d = (unsigned long long)(Q.ctg_bases + Q.ctg_off[ci] + (uint64_t)(V.k - 1) + (uint32_t)(f >> 32));
        }
        l1_dst[i] = d;
    }
}
// one thread per node: its base goes to where its segment starts + its offset (a one-byte store, often into a peer's memory)
template <class KT>
__global__ void sg_gather_nodes_kernel(const __grid_constant__ SGView V, uint64_t n, const uint64_t* __restrict__ loc, const unsigned long long* __restrict__ l1_dst) {
    const SGPeer& Me = V.p[V.me];
    for (uint64_t x = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; x < n; x += (uint64_t)gridDim.x * blockDim.x) {
        if (!(Me.alive[x] & 2)) continue;
        const uint64_t l = loc[x];
        if (l == ~0ull) continue;
        const unsigned long long d = l1_dst[(uint32_t)l];
        if (!d) continue;
        const KT X = sg_oriented<KT>(V, gid_make(V.me, (uint32_t)x));
        char* dst = reinterpret_cast<char*>(d) + (uint32_t)(l >> 32);
        *dst = "ACGT"[(uint32_t)X & 3u];
        if (Me.pred[x] == NONE32)  // head: its contig lives on this rank; the first k-1 bases come from it as well
            for (int j = 0; j < V.k - 1; j++) dst[j - (V.k - 1)] = "ACGT"[(uint32_t)(X >> (2 * (V.k - 1 - j))) & 3u];
    }
}
// One thread per level-1 segment: the bases of its nodes (the head's segment: the first k-1 bases of the contig as well) are
// packed into 8-byte words and OR-ed into the owner's buffer (zeroed by the owner; words are shared with the neighbouring
// segments, which other ranks write): about one posted atomic per 8 bases instead of one store per base -- on this
// workload all ranks write into the buffers of the two ranks that own the two strands of the chromosome.
template <class KT>
__global__ void sg_gather_kernel(const __grid_constant__ SGView V, uint64_t m1, const uint32_t* __restrict__ spl_node, const unsigned long long* __restrict__ l1_dst) {
    const SGPeer& Me = V.p[V.me];
    for (uint64_t id = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; id < m1; id += (uint64_t)gridDim.x * blockDim.x) {
        unsigned long long addr = l1_dst[id];
        if (!addr) continue;
        uint32_t x = spl_node[id];
        const uint32_t len = (uint32_t)(Me.l1_ent[id].x >> 32);
        unsigned long long word = 0;
        auto put = [&](uint32_t code) {
            word |= (unsigned long long)(uint8_t)"ACGT"[code] << (8u * (uint32_t)(addr & 7ull));
            addr++;
            if (!(addr & 7ull)) { atomicOr(reinterpret_cast<unsigned long long*>(addr - 8ull), word); word = 0; }
        };
        KT X = sg_oriented<KT>(V, gid_make(V.me, x));
        if (Me.pred[x] == NONE32) {  // head
            addr -= (unsigned long long)(V.k - 1);
            for (int j = 0; j < V.k - 1; j++) put((uint32_t)(X >> (2 * (V.k - 1 - j))) & 3u);
        }
        for (uint32_t t = 0;;) {
            put((uint32_t)X & 3u);
            if (++t == len) break;
            x = gid_loc(Me.succ[x]);  // the segment stays on this rank
            X = sg_oriented<KT>(V, gid_make(V.me, x));
        }
        if (addr & 7ull) atomicOr(reinterpret_cast<unsigned long long*>(addr & ~7ull), word);
    }
}

// ---- host side ------------------------------------------------------------------------------------------------------------
// RFX_SHARD_PROF=1: event marks between the phases of rfx_assemble_sharded / rfx_sort_kmers_sharded, printed by rank 0 when
// the call returns
struct SGProf {
    const char* what = "rfx_assemble_sharded";
    bool on = false;
    cudaStream_t st = nullptr;
    std::vector<std::pair<const char*, cudaEvent_t>> marks;
    void mark(const char* name) {
        if (!on) return;
        cudaEvent_t e;
        cudaEventCreate(&e);
        cudaEventRecord(e, st);
        marks.push_back({name, e});
    }
    void report(int rank) {
        if (!on) return;
        cudaStreamSynchronize(st);
        std::string line = std::string(what) + " rank " + std::to_string(rank) + " [ms]:";
        for (size_t i = 1; i < marks.size(); i++) {
            float ms = 0;
            cudaEventElapsedTime(&ms, marks[i - 1].second, marks[i].second);
            char buf[96];
            snprintf(buf, sizeof(buf), " %s %.3f", marks[i].first, ms);
            line += buf;
        }
        fprintf(stderr, "%s\n", line.c_str());
        for (auto& m : marks) cudaEventDestroy(m.second);
        marks.clear();
    }
};

// publish the status `rc`, the arena offsets of this rank's graph buffers + values; rebuild the view of everybody's buffers
static int sg_publish(Ctx* c, int rc, SGView& V, const unsigned long long host_vals[GP_NHOST], int n_dev, const int* dev_slots, PubVals& all) {
    GShard* gs = c->gshard;
    unsigned long long mine[GP_DEV];
    auto off_of = [&](const void* p) -> unsigned long long { return p ? (unsigned long long)((const uint8_t*)p - c->arena) : ~0ull; };
    const void* ptrs[GP_NPTR] = {c->keys.p, c->counts.p, c->ht.p, c->g_bloom.p, c->alive.p, c->lflag.p, c->rflag.p, c->eff_l.p, c->eff_r.p, c->succ.p, c->pred.p, gs->nxt_l1.p,
                                 gs->l1_ent.p, gs->l1_loc.p, gs->l2_up[0].p, gs->l2_up[1].p, gs->l2_node.p, gs->l2_fin.p, c->chain_len.p, gs->tail_rf.p,
                                 c->ctg_idx.p, c->ctg_off.p, c->ctg_bases.p, gs->inbox.p, gs->respbox.p, gs->req_cnt.p};
    for (int i = 0; i < GP_NPTR; i++) mine[i] = off_of(ptrs[i]);
    mine[GP_NROWS] = c->n_rows;
    mine[GP_HTCAP] = c->ht_cap;
    mine[GP_BLOOMMASK] = 0;
    for (int i = 0; i < GP_NHOST; i++) mine[GP_HOST + i] = host_vals ? host_vals[i] : 0ull;
    // device values (at GP_DEV + i): copied right behind the host values by one small copy each
    RFX_TRY(shard_exchange(c, rc, GP_DEV, mine, all, n_dev, dev_slots));
    V.me = c->sh_rank; V.world = c->sh_world; V.k = c->k; V.m = c->m;
    V.B = c->n_bins; V.bps = c->n_bins / (uint32_t)c->sh_world;
    V.filter = c->g_bloom.as<uint32_t>();
    V.rb = gs->rb;
    V.inv_bps = V.bps > 1 ? ~0ull / V.bps + 1ull : 0ull;
    V.chan_cap = gs->chan_cap;
    for (int r = 0; r < RFX_MAX_RANKS; r++) {
        SGPeer& P = V.p[r];
        memset(&P, 0, sizeof(P));
        if (r >= c->sh_world) continue;
        uint8_t* base = c->peer_base[r];
        auto at = [&](int slot) -> uint8_t* { return all.at(r, slot) == ~0ull ? nullptr : base + all.at(r, slot); };
        P.keys = at(GP_KEYS); P.counts = (const uint32_t*)at(GP_COUNTS); P.ht = (const uint32_t*)at(GP_HT); P.filter = (const uint32_t*)at(GP_BLOOM);
        P.alive = at(GP_ALIVE); P.lflag = (int32_t*)at(GP_LFLAG); P.rflag = (int32_t*)at(GP_RFLAG); P.eff_l = (int32_t*)at(GP_EFFL); P.eff_r = (int32_t*)at(GP_EFFR);
        P.succ = (uint32_t*)at(GP_SUCC); P.pred = (uint32_t*)at(GP_PRED); P.nxt_l1 = (uint32_t*)at(GP_NXTL1);
        P.l1_ent = (ulonglong2*)at(GP_L1ENT); P.l1_loc = (uint64_t*)at(GP_L1LOC);
        P.l2_up[0] = (uint64_t*)at(GP_L2UP0); P.l2_up[1] = (uint64_t*)at(GP_L2UP1); P.l2_node = (uint32_t*)at(GP_L2NODE); P.l2_fin = (uint64_t*)at(GP_L2FIN);
        P.chain_len = (uint32_t*)at(GP_CHAINLEN); P.tail_rf = (int32_t*)at(GP_TAILRF); P.ctg_idx = (uint32_t*)at(GP_CTGIDX); P.ctg_off = (uint64_t*)at(GP_CTGOFF);
        P.ctg_bases = (char*)at(GP_CTGBASES);
        P.inbox = at(GP_INBOX); P.respbox = (uint4*)at(GP_RESPBOX); P.req_cnt = (unsigned long long*)at(GP_REQCNT);
        P.ht_cap = (uint32_t)all.at(r, GP_HTCAP);
    }
    return RFX_OK;
}

// a closed path somewhere: rank 0 pulls every shard table and runs the single-GPU stages over the whole table
template <class KT> static int sg_fallback_whole_table(Ctx* c, const SGView& V, const PubVals& all) {
    GShard* gs = c->gshard;
    cudaStream_t st = c->stream;
    gs->fell_back = 1;
    int rc = RFX_OK;
    if (c->sh_rank == 0) {
        const uint64_t tot = all.sum(GP_NROWS);
        RFX_TRY(devbuf_reserve(c, gs->all_keys, (tot + 1) * sizeof(KT)));
        RFX_TRY(devbuf_reserve(c, gs->all_counts, (tot + 1) * sizeof(uint32_t)));
        uint64_t pos = 0;
        for (int r = 0; r < c->sh_world; r++) {
            const uint64_t nr = all.at(r, GP_NROWS);
            if (nr) {
                RFX_CUDA(c, cudaMemcpyAsync(gs->all_keys.as<KT>() + pos, V.p[r].keys, nr * sizeof(KT), cudaMemcpyDefault, st));
                RFX_CUDA(c, cudaMemcpyAsync(gs->all_counts.as<uint32_t>() + pos, V.p[r].counts, nr * sizeof(uint32_t), cudaMemcpyDefault, st));
            }
            pos += nr;
        }
        DevBuf own_keys = c->keys, own_counts = c->counts;
        const uint64_t own_rows = c->n_rows;
        c->keys = gs->all_keys; c->counts = gs->all_counts; c->n_rows = tot;
        rc = graph_impl<KT>(c);
        gs->all_keys = c->keys; gs->all_counts = c->counts;
        c->keys = own_keys; c->counts = own_counts; c->n_rows = own_rows;
        c->have_contigs = false;  // alive / flags describe the whole table, not this rank's rows: only the contigs are kept
    } else {
        RFX_TRY(devbuf_reserve(c, c->ctg_off, sizeof(uint64_t)));
        RFX_CUDA(c, cudaMemsetAsync(c->ctg_off.p, 0, sizeof(uint64_t), st));
        c->n_contigs = c->n_contig_bases = c->n_oriented = c->n_budget = c->n_budget_adm = c->n_cycles = 0;
    }
    return rc;
}

// The buffers of the K5 prologue (sg_k5_prologue), and the sizes every rank computes the same.  A failure comes back as a
// code: the rank still publishes it.
template <class KT> static int sg_k5_reserve(Ctx* c, bool chains) {
    GShard* gs = c->gshard;
    const int world = c->sh_world;
    const uint64_t n_rows = c->n_rows, n = 2 * n_rows, nn = n ? n : 1;
    RFX_TRY(devbuf_reserve(c, c->rflag, nn * sizeof(int32_t)));
    RFX_TRY(devbuf_reserve(c, c->lflag, nn * sizeof(int32_t)));
    RFX_TRY(devbuf_reserve(c, c->alive, nn + 8));
    RFX_TRY(devbuf_reserve(c, gs->rmin, (n_rows + 1) * sizeof(uint4)));
    if (chains) {
        RFX_TRY(devbuf_reserve(c, c->eff_l, nn * sizeof(int32_t)));
        RFX_TRY(devbuf_reserve(c, c->eff_r, nn * sizeof(int32_t)));
        RFX_TRY(devbuf_reserve(c, c->succ, nn * sizeof(uint32_t)));
        RFX_TRY(devbuf_reserve(c, c->pred, nn * sizeof(uint32_t)));
        RFX_TRY(devbuf_reserve(c, c->spl_id, nn * sizeof(uint32_t)));
        RFX_TRY(devbuf_reserve(c, c->spl_node, nn * sizeof(uint32_t)));
        RFX_TRY(devbuf_reserve(c, c->loc, nn * sizeof(uint64_t)));
        RFX_TRY(devbuf_reserve(c, c->ad[0], nn * sizeof(uint64_t)));
        RFX_TRY(devbuf_reserve(c, c->chain_len, nn * sizeof(uint32_t)));
        RFX_TRY(devbuf_reserve(c, c->ctg_idx, nn * sizeof(uint32_t)));
        RFX_TRY(devbuf_reserve(c, gs->tail_rf, nn * sizeof(int32_t)));
        RFX_TRY(devbuf_reserve(c, gs->l1_ent, nn * sizeof(ulonglong2)));
        RFX_TRY(devbuf_reserve(c, gs->nxt_l1, nn * sizeof(uint32_t)));
        RFX_TRY(devbuf_reserve(c, gs->l1_loc, nn * sizeof(uint64_t)));
        RFX_TRY(devbuf_reserve(c, gs->l1_fin, nn * sizeof(uint64_t)));
        RFX_TRY(devbuf_reserve(c, gs->l1_dst, nn * sizeof(uint64_t)));
        RFX_TRY(devbuf_reserve(c, gs->l2_l1, nn * sizeof(uint32_t)));
        RFX_TRY(devbuf_reserve(c, gs->l2_node, nn * sizeof(uint32_t)));
        for (int i = 0; i < 2; i++) RFX_TRY(devbuf_reserve(c, gs->l2_up[i], nn * sizeof(uint64_t)));
        RFX_TRY(devbuf_reserve(c, gs->l2_fin, nn * sizeof(uint64_t)));
        RFX_TRY(devbuf_reserve(c, c->ctg_off, sizeof(uint64_t)));
        RFX_TRY(devbuf_reserve(c, c->ctg_bases, 16));
    }
    // the own index: one region, load factor <= 1/4.  Presence bits: a region per minimiser bin of ALL ranks (SGView), the
    // region size from the global row count rfx_count_sharded left behind, so that every rank computes the same
    const uint32_t B = c->n_bins;
    {
        const uint64_t per_bin = (c->sh_rows_global + B - 1) / B;
        uint64_t rb = (16 * per_bin + 63) / 64 * 64;
        if (rb < 64) rb = 64;
        if (rb > (1u << 24)) rb = 1u << 24;
        gs->rb = (uint32_t)rb;
    }
    const uint64_t filter_bytes = (uint64_t)B * gs->rb / 8;
    const uint64_t slots = 4 * n_rows + 2;
    RFX_TRY(devbuf_reserve(c, c->ht, slots * sizeof(uint32_t)));
    RFX_TRY(devbuf_reserve(c, c->g_bloom, filter_bytes + 64));
    RFX_TRY(devbuf_reserve(c, gs->work, nn * sizeof(uint32_t)));
    RFX_TRY(devbuf_reserve(c, gs->pend_ref, nn * sizeof(uint4)));
    // request / answer channels: one per (sender, receiver) pair, reused by the three K5 stages
    gs->chan_cap = world > 1 ? c->sh_rows_global / (uint64_t)world + 65536 : 1;  // the same on every rank: a channel is addressed from both ends
    RFX_TRY(devbuf_reserve(c, gs->inbox, (size_t)world * gs->chan_cap * sizeof(SGReq<KT>)));
    RFX_TRY(devbuf_reserve(c, gs->respbox, (size_t)world * gs->chan_cap * sizeof(uint4)));
    RFX_TRY(devbuf_reserve(c, gs->req_cnt, 3 * RFX_MAX_RANKS * sizeof(unsigned long long)));
    c->ht_cap = slots; c->g_bins = 1; c->g_m = c->m; c->g_bloom_mask = 0;
    return RFX_OK;
}

// The K5 prologue of rfx_assemble_sharded and rfx_sort_kmers_sharded: the per-node arrays of the fork filters, the index over
// the own rows, the presence bits of all ranks and the request / answer channels, published to the peers.  `chains`: also the
// buffers of the chain ranking and the contigs (K6, K7) and their presets.  Every rank must call it (a barrier when world > 1),
// with the status it has so far (`rc`): a rank that already failed reserves nothing and only publishes its code.
template <class KT> static int sg_k5_prologue(Ctx* c, int rc, bool chains, SGView& V, PubVals& all, SGProf& prof) {
    cudaStream_t st = c->stream;
    GShard* gs = c->gshard;
    const int world = c->sh_world;
    const uint64_t n_rows = c->n_rows, n = 2 * n_rows, nn = n ? n : 1;
    unsigned long long* dstat = c->dstat.as<unsigned long long>();
    if (rc == RFX_OK) rc = sg_k5_reserve<KT>(c, chains);
    // everything is allocated: tell the others where (nothing behind these addresses is valid yet)
    RFX_TRY(sg_publish(c, rc, V, nullptr, 0, nullptr, all));
    gs->n_rows_global = all.sum(GP_NROWS);
    const uint32_t B = c->n_bins, bps = B / (uint32_t)world;
    const uint64_t slice_bytes = (uint64_t)bps * gs->rb / 8, slots = c->ht_cap;
    prof.mark("reserve+publish1");
    // own presence bits (+ the per-row minima) first: the peers pull them while this rank builds its index
    RFX_CUDA(c, cudaMemsetAsync(gs->req_cnt.p, 0, 3 * RFX_MAX_RANKS * sizeof(unsigned long long), st));
    RFX_CUDA(c, cudaMemsetAsync(c->g_bloom.as<uint8_t>() + (size_t)c->sh_rank * slice_bytes, 0, slice_bytes, st));
    if (n_rows) {
        sg_row_minima_kernel<KT><<<grid_n(n_rows), 256, 0, st>>>(c->keys.as<KT>(), n_rows, c->k, c->m, B, (uint32_t)c->sh_rank * bps, (uint32_t)(c->sh_rank + 1) * bps,
                                                                gs->rb, gs->rmin.as<uint4>(), c->g_bloom.as<uint32_t>(), dstat);
        c->launches++;
    }
    if (world > 1) {
        RFX_TRY(shard_barrier(c));  // every rank's presence bits are complete
        RFX_CUDA(c, cudaEventRecord(c->copy_done[0], st));
        RFX_CUDA(c, cudaStreamWaitEvent(c->copy_stream, c->copy_done[0], 0));
        for (int q = 1; q < world && slice_bytes; q++) {  // every rank starts with another peer
            const int r = (c->sh_rank + q) % world;
            RFX_CUDA(c, cudaMemcpyAsync(c->g_bloom.as<uint8_t>() + (size_t)r * slice_bytes, reinterpret_cast<const uint8_t*>(V.p[r].filter) + (size_t)r * slice_bytes, slice_bytes,
                                        cudaMemcpyDefault, c->copy_stream));
        }
        RFX_CUDA(c, cudaEventRecord(c->copy_done[1], c->copy_stream));
    }
    prof.mark("filter_bits");
    RFX_CUDA(c, cudaMemsetAsync(c->ht.p, 0xff, slots * sizeof(uint32_t), st));
    if (n_rows) {
        Graph<KT> G = make_graph<KT>(c);
        G.bloom_mask = 0;
        ht_build_kernel<KT><<<grid_n(n_rows), 256, 0, st>>>(G, nullptr);
        c->launches++;
    }
    if (chains) {
        cudaMemsetAsync(c->succ.p, 0xff, nn * sizeof(uint32_t), st);
        cudaMemsetAsync(c->pred.p, 0xff, nn * sizeof(uint32_t), st);
        cudaMemsetAsync(c->chain_len.p, 0, nn * sizeof(uint32_t), st);
        cudaMemsetAsync(gs->tail_rf.p, 0, nn * sizeof(int32_t), st);
        cudaMemsetAsync(c->loc.p, 0xff, nn * sizeof(uint64_t), st);
        cudaMemsetAsync(gs->l1_loc.p, 0xff, nn * sizeof(uint64_t), st);
    }
    cudaMemsetAsync(c->alive.p, 0, nn + 8, st);
    prof.mark("memsets+index");
    if (world > 1) RFX_CUDA(c, cudaStreamWaitEvent(st, c->copy_done[1], 0));  // the peers' presence bits have arrived
    prof.mark("filter_wait");
    return RFX_OK;
}

// `rc`: the entry checks of this rank, published by the prologue
template <class KT> static int sharded_graph_impl(Ctx* c, int rc) {
    cudaStream_t st = c->stream;
    if (!c->gshard) c->gshard = new GShard();
    GShard* gs = c->gshard;
    const int world = c->sh_world;
    const uint64_t n_rows = c->n_rows, n = 2 * n_rows, nn = n ? n : 1;
    unsigned long long* dstat = c->dstat.as<unsigned long long>();
    PubVals all;
    RFX_CUDA(c, cudaMemsetAsync(c->dstat.p, 0, DS_NSLOTS * sizeof(uint64_t), st));
    c->n_oriented = c->n_budget = c->n_budget_adm = c->n_cycles = c->n_contigs = c->n_contig_bases = 0;
    c->have_sorted = false; c->have_contigs = false;
    c->ms_comm = 0;
    gs->fell_back = 0;

    SGProf prof;
    prof.on = getenv("RFX_SHARD_PROF") != nullptr && c->sh_rank == 0;
    prof.st = st;
    prof.mark("start");
    // ---- K5 ----
    stage_begin(c);
    SGView V;
    RFX_TRY(sg_k5_prologue<KT>(c, rc, true, V, all, prof));
    // (the peers' indexes are first touched by the answering kernels, behind the barrier that follows the first pass)
    const int E = c->prm.min_error_coverage;
    const uint4* rmin = gs->rmin.as<uint4>();
    // every K5 stage: pass 1 over the own nodes (requests out), [barrier], the owners answer, [barrier], pass 2 over the nodes that waited
    const unsigned g2 = sm_count() * 8u;
    SGWork W[3];
    for (int i = 0; i < 3; i++) W[i] = SGWork{gs->work.as<uint32_t>(), gs->pend_ref.as<uint4>(), dstat + DS_WORK + i};
    if (n) sg_right_filter_kernel<KT, 1><<<grid_n(n), 256, 0, st>>>(V, E, n, rmin, W[0], dstat);
    prof.mark("right");
    if (world > 1) {
        RFX_TRY(shard_barrier(c));
        sg_serve_kernel<KT, false><<<g2, 256, 0, st>>>(V, 0, dstat);
        RFX_TRY(shard_barrier(c));
        prof.mark("right_serve");
        if (n) sg_right_filter_kernel<KT, 2><<<g2, 256, 0, st>>>(V, E, n, rmin, W[0], dstat);
        prof.mark("right2");
    }
    if (n) sg_left_filter_kernel<KT, 1><<<grid_n(n), 256, 0, st>>>(V, E, n, rmin, W[1], dstat);
    prof.mark("left");
    if (world > 1) {
        RFX_TRY(shard_barrier(c));
        sg_serve_kernel<KT, false><<<g2, 256, 0, st>>>(V, 1, dstat);
        RFX_TRY(shard_barrier(c));
        prof.mark("left_serve");
        if (n) sg_left_filter_kernel<KT, 2><<<g2, 256, 0, st>>>(V, E, n, rmin, W[1], dstat);
        prof.mark("left2");
    }
    if (n) sg_link_kernel<KT, 1><<<grid_n(n), 256, 0, st>>>(V, n, rmin, W[2], dstat);
    prof.mark("link");
    if (world > 1) {
        RFX_TRY(shard_barrier(c));
        sg_serve_kernel<KT, true><<<g2, 256, 0, st>>>(V, 2, dstat);
        RFX_TRY(shard_barrier(c));
        prof.mark("link_serve");
        if (n) sg_link_kernel<KT, 2><<<g2, 256, 0, st>>>(V, n, rmin, W[2], dstat);
        prof.mark("link2");
    }
    c->launches += 9;
    {
        const int slots_dev[3] = {DS_FLAGGED, DS_GRAPH_ERR, DS_REMOTE};
        RFX_TRY(sg_publish(c, RFX_OK, V, nullptr, 3, slots_dev, all));  // [barrier] every pred[] has its remote writes
    }
    prof.mark("publish2");
    const unsigned long long flagged = all.sum(GP_DEV + 0), gerr = all.sum(GP_DEV + 1);
    gs->n_remote = all.at(c->sh_rank, GP_DEV + 2);
    if (gerr) return ctx_fail(c, RFX_E_GRAPH, "sharded fork filters: a (k-1)-mer with degree > 1 (codes 1, 2), a row on a rank that does not own its minimiser bin (3) or a request channel that overflowed (4); codes add up to %llu", gerr);
    if (flagged) {
        if (n) {
            sg_budget_walk_kernel<KT, 0><<<grid_n(n), 256, 0, st>>>(V, n, c->k - 1, dstat);
            sg_budget_walk_kernel<KT, 1><<<grid_n(n), 256, 0, st>>>(V, n, c->k - 1, dstat);
        }
        RFX_TRY(shard_barrier(c));
        if (n) sg_junction_finalize_kernel<<<grid_n(n), 256, 0, st>>>(V, n);
        c->launches += 3;
        // the barrier inside the next exchange orders the cuts before the splitter selection of the peers
    }

    // ---- K6 ----
    RFX_TRY(shard_barrier(c));
    RFX_TRY(shard_check(c, "sharded fork filters"));
    c->ms[3] += stage_end(c);
    prof.mark("budget+bar+sync");
    stage_begin(c);
    if (n) sg_select_kernel<<<grid_n(n), 256, 0, st>>>(V, n, c->spl_id.as<uint32_t>(), c->spl_node.as<uint32_t>(), gs->l2_l1.as<uint32_t>(), dstat);
    c->launches++;
    {
        const int slots_dev[2] = {DS_NSPL, DS_NL2};
        RFX_TRY(sg_publish(c, RFX_OK, V, nullptr, 2, slots_dev, all));  // [barrier] spl_id / l2_of of every rank are final
    }
    prof.mark("select+publish3");
    const uint64_t m1 = all.at(c->sh_rank, GP_DEV + 0);
    const uint64_t m2 = all.at(c->sh_rank, GP_DEV + 1);
    const uint64_t m2_all = all.sum(GP_DEV + 1);
    gs->n_l1 = m1; gs->n_l2 = m2;
    int rounds = 1;
    while ((1ull << rounds) < m2_all + 1) rounds++;
    rounds += 1;
    if (m1) sg_l1_walk_kernel<<<grid_n(m1), 256, 0, st>>>(V, m1, c->spl_id.as<uint32_t>(), c->spl_node.as<uint32_t>(), c->loc.as<uint64_t>());
    prof.mark("l1_walk");
    RFX_TRY(shard_barrier(c));
    prof.mark("bar");
    if (m2) {
        uint64_t g2 = (m2 + 63) / 64;
        if (g2 > sm_count() * 32u) g2 = sm_count() * 32u;
        sg_l2_walk_kernel<<<(unsigned)g2, 64, 0, st>>>(V, m2, gs->l2_l1.as<uint32_t>());
    }
    prof.mark("l2_walk");
    RFX_TRY(shard_barrier(c));
    prof.mark("bar");
    c->launches += 2;
    int cur = 0;
    if (world > 1 && !c->hbar && getenv("RFX_JUMP_FUSED")) {
        // measured alternative, off by default: every round inside one cooperative launch (sg_l2_jump_all_kernel).  At 2 GPUs
        // 0.61 ms against 0.31 ms for one small kernel + one barrier kernel per round: two grid-wide barriers per round cost more
        // than the two launches they replace.
        PeerBases PB = peer_bases(c);
        uint64_t m2v = m2;
        int rv = rounds;
        unsigned long long e0 = c->sh_epoch2;
        unsigned long long* ds = dstat;
        unsigned blocks = (unsigned)((m2 + 255) / 256);
        if (blocks < 1) blocks = 1;
        if (blocks > sm_count()) blocks = sm_count();
        void* args[] = {(void*)&V, (void*)&PB, (void*)&m2v, (void*)&rv, (void*)&e0, (void*)&ds};
        RFX_CUDA(c, cudaLaunchCooperativeKernel((void*)sg_l2_jump_all_kernel, dim3(blocks), dim3(256), args, 0, st));
        c->sh_epoch2 += (unsigned long long)rounds;
        c->launches++;
        cur = rounds & 1;  // (the last round ends behind a cross-GPU barrier: every rank's result is complete and visible)
    } else {
        for (int r = 0; r < rounds; r++) {
            if (m2) sg_l2_jump_kernel<<<grid_n(m2), 256, 0, st>>>(V, m2, cur);
            RFX_TRY(shard_barrier(c));
            c->launches++;
            cur ^= 1;
        }
    }
    prof.mark("l2_jump_rounds");
    if (m2) sg_l2_fin_kernel<<<grid_n(m2), 256, 0, st>>>(V, m2, cur, dstat);
    RFX_TRY(shard_barrier(c));
    prof.mark("l2_fin+bar");
    if (m1) sg_l1_fin_kernel<<<grid_n(m1), 256, 0, st>>>(V, m1, gs->l1_fin.as<uint64_t>(), dstat);
    if (n) sg_node_fin_kernel<<<grid_n(n), 256, 0, st>>>(V, n, c->loc.as<uint64_t>(), gs->l1_fin.as<uint64_t>(), c->ad[0].as<uint64_t>(), dstat);
    c->launches += 3;
    {
        const int slots_dev[5] = {DS_SG_CYCLE, DS_BUDGET, DS_ABSORBED, DS_CYCLES, DS_XBAR_ERR};
        RFX_TRY(sg_publish(c, RFX_OK, V, nullptr, 5, slots_dev, all));  // [barrier] every head knows its chain's length and right flag
    }
    prof.mark("l1_fin+node_fin+publish4");
    c->ms[4] += stage_end(c);
    const unsigned long long any_cycle = all.sum(GP_DEV + 0);
    c->n_budget = all.at(c->sh_rank, GP_DEV + 1);
    c->n_budget_adm = all.at(c->sh_rank, GP_DEV + 2);
    c->n_cycles = all.at(c->sh_rank, GP_DEV + 3);
    if (any_cycle) {
        stage_begin(c);
        const int frc = sg_fallback_whole_table<KT>(c, V, all);
        c->ms[5] += stage_end(c);
        // The barrier of this publish also keeps every peer from touching its table before rank 0 has read it: rank 0 enqueues
        // it behind its copies.
        unsigned long long hv[GP_NHOST] = {c->n_contigs, c->n_contig_bases, c->n_oriented, 0, 0, 0};
        RFX_TRY(sg_publish(c, frc, V, hv, 0, nullptr, all));
        gs->n_contigs_global = all.sum(GP_HOST + 0);
        gs->n_bases_global = all.sum(GP_HOST + 1);
        gs->n_oriented_global = all.sum(GP_HOST + 2);
        c->have_contigs = true;
        return RFX_OK;
    }

    // ---- K7 ----
    stage_begin(c);
    // the own contigs' layout; a rank that cannot reserve it still publishes, with its code
    U64x3 tot{0, 0, 0};
    const int lrc = [&]() -> int {
        ScanPlan<U64x3> plan;
        RFX_TRY(devbuf_reserve(c, c->scan_ws, ScanPlan<U64x3>::workspace_elems(nn) * sizeof(U64x3)));
        plan.bind(n, c->scan_ws.as<U64x3>());
        SContigIn in{c->alive.as<uint8_t>(), c->pred.as<uint32_t>(), c->chain_len.as<uint32_t>(), c->eff_l.as<int32_t>(), gs->tail_rf.as<int32_t>(), c->k, c->prm.min_contig};
        if (n) {
            scan_prepare(plan, in, OpAddU64x3{}, U64x3{0, 0, 0}, st);
            c->launches += 2 * plan.levels;
            RFX_CUDA(c, cudaMemcpyAsync(&tot, plan.total, sizeof(tot), cudaMemcpyDeviceToHost, st));
            cudaError_t e = cudaStreamSynchronize(st);
            if (e != cudaSuccess) return ctx_fail(c, RFX_E_CUDA, "sharded contig scan failed: %s", cudaGetErrorString(e));
        }
        prof.mark("contig_scan");
        RFX_TRY(devbuf_reserve(c, c->ctg_off, (tot.a + 1) * sizeof(uint64_t)));
        RFX_TRY(devbuf_reserve(c, c->ctg_left, (tot.a + 1) * sizeof(int32_t)));
        RFX_TRY(devbuf_reserve(c, c->ctg_right, (tot.a + 1) * sizeof(int32_t)));
        RFX_TRY(devbuf_reserve(c, c->ctg_bases, tot.b + 16));
        RFX_CUDA(c, cudaMemsetAsync(c->ctg_bases.p, 0, tot.b + 16, st));  // the bases arrive as OR-ed words (sg_gather_kernel)
        if (n) {
            SContigOut out{c->eff_l.as<int32_t>(), gs->tail_rf.as<int32_t>(), c->ctg_idx.as<uint32_t>(), c->ctg_off.as<uint64_t>(), c->ctg_left.as<int32_t>(), c->ctg_right.as<int32_t>()};
            scan_apply(plan, in, out, OpAddU64x3{}, U64x3{0, 0, 0}, st);
            set_u64_kernel<<<1, 1, 0, st>>>(c->ctg_off.as<uint64_t>() + tot.a, plan.total);
            c->launches += 2;
        } else {
            RFX_CUDA(c, cudaMemsetAsync(c->ctg_off.p, 0, sizeof(uint64_t), st));
        }
        return RFX_OK;
    }();
    c->n_contigs = tot.a; c->n_contig_bases = tot.b; c->n_oriented = tot.c;
    {
        unsigned long long hv[GP_NHOST] = {tot.a, tot.b, tot.c, 0, 0, 0};
        RFX_TRY(sg_publish(c, lrc, V, hv, 0, nullptr, all));  // [barrier] contig tables laid out, buffers published
    }
    gs->n_contigs_global = all.sum(GP_HOST + 0);
    gs->n_bases_global = all.sum(GP_HOST + 1);
    gs->n_oriented_global = all.sum(GP_HOST + 2);
    prof.mark("scan_apply+publish5");
    if (m1) sg_l1_dst_kernel<<<grid_n(m1), 256, 0, st>>>(V, m1, gs->l1_fin.as<uint64_t>(), gs->l1_dst.as<unsigned long long>());
    {
        const char* gv = getenv("RFX_GATHER");  // "nodes" / "segments": measured both ways (profiles/)
        const bool by_segment = gv ? !strcmp(gv, "segments") : world > 2;
        if (by_segment) { if (m1) sg_gather_kernel<KT><<<grid_n(m1), 128, 0, st>>>(V, m1, c->spl_node.as<uint32_t>(), gs->l1_dst.as<unsigned long long>()); }
        else if (n) sg_gather_nodes_kernel<KT><<<grid_n(n), 256, 0, st>>>(V, n, c->loc.as<uint64_t>(), gs->l1_dst.as<unsigned long long>());
    }
    c->launches += 2;
    RFX_TRY(shard_barrier(c));  // every base of the own contigs has arrived
    prof.mark("l1_dst+gather+bar");
    RFX_TRY(shard_check(c, "sharded assembly"));
    c->ms[5] += stage_end(c);
    prof.report(c->sh_rank);
    c->have_contigs = true;
    return RFX_OK;
}

int stage_assemble_sharded(Ctx* c) {
    if (c->sh_world < 1 || !c->peer_base[c->sh_rank]) return ctx_fail(c, RFX_E_STATE, "rfx_assemble_sharded: call rfx_shard_init / rfx_shard_connect first");
    int rc = RFX_OK;
    if (!c->have_counts) rc = ctx_fail(c, RFX_E_STATE, "rfx_assemble_sharded: no count table (call rfx_count_sharded first)");
    else if (!c->prm.bubble) rc = ctx_fail(c, RFX_E_UNSUPPORTED, "-bubble: undefined in the reference (see rfx_assemble)");
    else if (c->k < 2) rc = ctx_fail(c, RFX_E_INVALID, "assembly needs k >= 2");
    else if (2 * c->n_rows >= GID_MASK) rc = ctx_fail(c, RFX_E_CAPACITY, "sharded assembly: more than 2^28 rows on one rank");
    else if (!c->n_bins || c->n_bins % (uint32_t)c->sh_world)
        rc = ctx_fail(c, RFX_E_STATE, "sharded assembly needs the table of rfx_count_sharded (rows sharded by minimiser bin)");
    return c->wide ? sharded_graph_impl<u128>(c, rc) : sharded_graph_impl<uint64_t>(c, rc);
}

// ---- Count_<k>_sorted across ranks (rfx_sort_kmers_sharded) -------------------------------------------------------------
// The K5 prologue of the assembly (no chain or contig buffers), the two sorted filters as request / answer passes, the
// survivors counted as on one GPU.  A closing exchange makes a channel overflow or a misplaced row on any rank fail every rank.
template <class KT> static int sharded_sorted_impl(Ctx* c, int E, double fold, int Xf) {
    cudaStream_t st = c->stream;
    if (!c->gshard) c->gshard = new GShard();
    GShard* gs = c->gshard;
    const int world = c->sh_world;
    const uint64_t n = 2 * c->n_rows, nn = n ? n : 1;
    unsigned long long* dstat = c->dstat.as<unsigned long long>();
    PubVals all;
    RFX_CUDA(c, cudaMemsetAsync(c->dstat.p, 0, DS_NSLOTS * sizeof(uint64_t), st));
    c->n_sorted = 0;
    c->have_sorted = false; c->have_contigs = false;  // the index, the alive bytes and the flag arrays are taken over
    gs->fell_back = 0; gs->n_l1 = gs->n_l2 = 0; gs->n_contigs_global = gs->n_bases_global = 0;

    SGProf prof;
    prof.what = "rfx_sort_kmers_sharded";
    prof.on = getenv("RFX_SHARD_PROF") != nullptr && c->sh_rank == 0;
    prof.st = st;
    prof.mark("start");
    int rc = devbuf_reserve(c, c->srt_left, nn * sizeof(int32_t));
    if (rc == RFX_OK) rc = devbuf_reserve(c, c->srt_right, nn * sizeof(int32_t));
    SGView V;
    RFX_TRY(sg_k5_prologue<KT>(c, rc, false, V, all, prof));
    const uint4* rmin = gs->rmin.as<uint4>();
    // pass 1 over the own nodes (requests out), [barrier], the owners answer, [barrier], pass 2 over the nodes that waited
    const unsigned g2 = sm_count() * 8u;
    const SGWork W0{gs->work.as<uint32_t>(), gs->pend_ref.as<uint4>(), dstat + DS_WORK + 0};
    const SGWork W1{gs->work.as<uint32_t>(), gs->pend_ref.as<uint4>(), dstat + DS_WORK + 1};
    int32_t* out_l = c->srt_left.as<int32_t>();
    int32_t* out_r = c->srt_right.as<int32_t>();
    if (n) sg_sorted_right_kernel<KT, 1><<<grid_n(n), 256, 0, st>>>(V, E, fold, Xf, n, rmin, W0, dstat);
    prof.mark("right");
    if (world > 1) {
        RFX_TRY(shard_barrier(c));
        sg_serve_kernel<KT, false><<<g2, 256, 0, st>>>(V, 0, dstat);
        RFX_TRY(shard_barrier(c));
        prof.mark("right_serve");
        if (n) sg_sorted_right_kernel<KT, 2><<<g2, 256, 0, st>>>(V, E, fold, Xf, n, rmin, W0, dstat);
        prof.mark("right2");
    }
    if (n) sg_sorted_left_kernel<KT, 1><<<grid_n(n), 256, 0, st>>>(V, E, fold, Xf, n, rmin, W1, out_l, out_r, dstat);
    prof.mark("left");
    if (world > 1) {
        // the first barrier follows every rank's right pass 2: the coverages and right flags this serve answers with are final
        RFX_TRY(shard_barrier(c));
        sg_serve_kernel<KT, false, true><<<g2, 256, 0, st>>>(V, 1, dstat);
        RFX_TRY(shard_barrier(c));
        prof.mark("left_serve");
        if (n) sg_sorted_left_kernel<KT, 2><<<g2, 256, 0, st>>>(V, E, fold, Xf, n, rmin, W1, out_l, out_r, dstat);
        prof.mark("left2");
    }
    c->launches += world > 1 ? 6 : 2;
    // survivors (alive & 2), as rfx_sort_kmers counts them
    uint64_t total = 0;
    const int rc_scan = n ? devbuf_reserve(c, c->scan_ws, ScanPlan<uint64_t>::workspace_elems(n) * sizeof(uint64_t)) : RFX_OK;
    if (n && rc_scan == RFX_OK) {
        ScanPlan<uint64_t> plan;
        plan.bind(n, c->scan_ws.as<uint64_t>());
        scan_prepare(plan, AliveBoth{c->alive.as<uint8_t>()}, OpAddU64{}, (uint64_t)0, st);
        c->launches += 2 * plan.levels;
        RFX_CUDA(c, cudaMemcpyAsync(&total, plan.total, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    }
    cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return ctx_fail(c, RFX_E_CUDA, "sharded sorted-stage kernels failed: %s", cudaGetErrorString(e));
    prof.mark("survivors");
    // [barrier] every rank is done with its channels; survivors and error words of all ranks
    {
        const unsigned long long mine[1] = {total};
        const int slots_dev[2] = {DS_GRAPH_ERR, DS_REMOTE};  // values 1, 2
        RFX_TRY(shard_exchange(c, rc_scan, 1, mine, all, 2, slots_dev));
    }
    prof.mark("exchange");
    const unsigned long long gerr = all.sum(1);
    gs->n_remote = all.at(c->sh_rank, 2);
    gs->n_oriented_global = all.sum(0);
    c->ms[3] = stage_end(c);
    prof.report(c->sh_rank);
    if (gerr) return ctx_fail(c, RFX_E_GRAPH, "sharded sorted filters: a row on a rank that does not own its minimiser bin (code 3) or a request channel that overflowed (4); codes add up to %llu", gerr);
    c->n_sorted = total;
    c->have_sorted = true;
    return RFX_OK;
}

int stage_sorted_sharded(Ctx* c, int E, double fold, int max_kmer_size) {
    if (c->sh_world < 1 || !c->peer_base[c->sh_rank]) return ctx_fail(c, RFX_E_STATE, "rfx_sort_kmers_sharded: call rfx_shard_init / rfx_shard_connect first");
    const int world = c->sh_world;
    unsigned long long mine[6];
    static_assert(sizeof(mine) / sizeof(mine[0]) <= PUB_VALS, "the agreement exchange fits the published block");
    PubVals all;
    c->ms_comm = 0;
    stage_begin(c);
    // What every rank holds and was asked for, before any barrier or buffer.  Every rank checks every rank's values in the same
    // order, so that all ranks return the same error together.
    const bool sharded = c->have_counts && c->n_bins && c->n_bins % (uint32_t)world == 0;
    const int rc = sharded ? RFX_OK
                           : ctx_fail(c, RFX_E_STATE, "rfx_sort_kmers_sharded: this rank holds no table sharded by minimiser bin (rfx_count_sharded, or rfx_load_counts* and rfx_shard_table first)");
    unsigned long long fold_bits = 0;
    memcpy(&fold_bits, &fold, sizeof(fold_bits));
    mine[0] = (unsigned long long)c->k;
    mine[1] = c->n_bins;
    mine[2] = (uint32_t)E;
    mine[3] = fold_bits;
    mine[4] = (uint32_t)max_kmer_size;
    mine[5] = c->have_counts ? c->n_rows : 0;
    RFX_TRY(shard_exchange(c, rc, 6, mine, all));
    static const char* what[5] = {"k", "bin count", "min_error_coverage", "min_repeat_fold", "max_kmer_size"};
    for (int r = 1; r < world; r++)
        for (int s = 0; s < 5; s++)
            if (all.at(r, s) != all.at(0, s)) return ctx_fail(c, RFX_E_INVALID, "rfx_sort_kmers_sharded: rank %d has another %s than rank 0", r, what[s]);
    RFX_TRY(sorted_domain(c, "rfx_sort_kmers_sharded", E, fold, max_kmer_size));
    for (int r = 0; r < world; r++)
        if (2 * all.at(r, 5) >= GID_MASK) return ctx_fail(c, RFX_E_CAPACITY, "rfx_sort_kmers_sharded: rank %d holds more than 2^28 rows", r);
    return c->wide ? sharded_sorted_impl<u128>(c, E, fold, max_kmer_size + 3) : sharded_sorted_impl<uint64_t>(c, E, fold, max_kmer_size + 3);
}

void shard_graph_reset(Ctx* c) {
    if (c->gshard) *c->gshard = GShard();  // (all of its buffers live in the arena: nothing to free)
}

void shard_graph_release(Ctx* c) {
    delete c->gshard;
    c->gshard = nullptr;
}

void shard_graph_stats(Ctx* c, rfx_shard_stats_t* out) {
    if (!c->gshard) return;
    const GShard* gs = c->gshard;
    out->n_rows_global = gs->n_rows_global;
    out->n_oriented_global = gs->n_oriented_global;
    out->n_contigs_global = gs->n_contigs_global;
    out->n_contig_bases_global = gs->n_bases_global;
    out->n_remote_probes = gs->n_remote;
    out->n_l1_splitters = gs->n_l1;
    out->n_l2_splitters = gs->n_l2;
    out->fell_back = gs->fell_back;
}

}  // namespace rfx
