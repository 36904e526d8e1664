// rfx_count.cu -- K3 + K4: per-bin k-mer counting in shared memory, coverage-filter compaction.
//
// Replaces groupBy("value").count() + filter(count >= min && count <= max)
//   (ReflexivDataFrameCounter.java:198-210, ReflexivDataFrameCounter64.java:200-212, ReflexivDSMain.java:207-216).
//
// One CTA owns one minimiser bin at a time (bins are handed out by an atomic ticket, so a heavy bin never
// holds up a static schedule).  Per bin:
//   A   every thread hashes its super-k-mer records whole into a shared-memory table whose slot word carries a
//       21-bit tag and the index of the record that claimed the slot: a record that meets its own tag compares
//       itself with the claimant's record (staged in shared memory) on the spot, so identical records -- the
//       same genome window seen by many reads -- collapse exactly into one entry with a multiplicity;
//   B   the distinct records are expanded: a warp takes 32 entries, prefix-sums their k-mer counts and walks
//       the flattened (record, k-mer) space 32 k-mers per step -- shuffle binary search for the source record,
//       record words fetched by shuffle, the k-mer cut straight out of the 2-bit stream, brev-based reverse
//       complement -- and adds the record's multiplicity to the canonical k-mer's slot of an open-addressing
//       table in shared memory.
//         k <= 31: 64-bit atomicCAS claims the slot with the key itself;
//         k  > 31: a 32-bit tag CAS claims the slot and the claimant publishes the 128-bit key (pass B1);
//                  after a barrier pass B2 walks the same k-mers again, finds the slot whose FULL key
//                  matches and counts.  A key swallowed by a tag collision in B1 is not found in B2: the bin
//                  is re-run in sub-classes (different hash bits separate the pair), so counts stay exact.
//   K4  only rows inside the coverage bounds leave shared memory.
// Both tables keep a list of their occupied slots, so clearing and compaction cost what the bin holds, not
// what the table could hold; that is what lets bins be small (one chunk, few barriers) and the table be
// sized for noisy reads (one error-carrying k-mer in four is a singleton) at the same time.
// A bin whose distinct k-mers still do not fit is re-run in 2 or 4 sub-classes chosen by independent hash
// bits, recursively, so the result is exact for any input.
#include <stdlib.h>
#include <string.h>

#include <type_traits>

#include "rfx_internal.h"

namespace rfx {

constexpr int CNT_STACK = 64;

struct CountArgs {
    // bin b = concatenation over segments s of ext[s * n_bins + b].cnt records starting at the absolute address
    // ext[s * n_bins + b].addr -- a local slab, an exactly partitioned overflow list, a slice received through NCCL or
    // a PEER GPU's slab read in place over NVLink (rfx_shard.cu): the kernel does not care, its producer warp issues
    // one bulk copy per non-empty segment (build_ext_kernel fills the table)
    const SegExt* ext;
    int n_seg;
    uint32_t n_bins;
    int k;
    uint32_t min_count, max_count;
    void* out_keys;
    uint32_t* out_counts;
    unsigned long long* dstat;
    unsigned long long out_cap;
    // tickets t = 0 .. n_tickets-1 map to bins t * bin_stride (the full run: n_tickets = n_bins, stride 1)
    uint32_t n_tickets, bin_stride;
    int dry;  // pilot run: count and report statistics, write no rows
};

constexpr int MAX_SEG = RFX_MAX_SEG;

// slot hash + tag of a whole record (tag 0 = empty slot)
template <int RECW> __device__ __forceinline__ void record_hash(const uint64_t (&w)[RECW], uint32_t& slot_h, uint32_t& tag) {
    uint32_t x = hash_lane_a((uint32_t)w[0], (uint32_t)(w[0] >> 32), (uint32_t)w[1], (uint32_t)(w[1] >> 32));
    if (RECW == 4) x = hash_lane_b((uint32_t)w[2] ^ x, (uint32_t)(w[2] >> 32), (uint32_t)w[3], (uint32_t)(w[3] >> 32));
    const uint64_t p = (uint64_t)x * 0xD3A2646Cu;
    slot_h = (uint32_t)p ^ (uint32_t)(p >> 32);
    tag = (uint32_t)(p >> 32) * 0xFD7046C5u | 1u;
}

// The shared-memory k-mer table of one CTA.
template <bool WIDE, int CAP> struct KmerTable {
    static constexpr int KMAX = CAP * 3 / 4;  // distinct k-mers the table accepts before the bin is split
    unsigned long long* keys;  // narrow: the key, ~0 = empty.   wide: high 64 bits of the key
    unsigned long long* keys_lo;  // wide only
    uint32_t* tags;               // wide only: 0 = empty
    uint32_t* cnts;
    uint16_t* klist;              // occupied slots in claim order
    uint32_t* n_distinct;
    volatile uint32_t* overflow;
    unsigned long long* why;  // DS_OVF_WHY counters

    __device__ __forceinline__ void flag(int reason) const {
        if (!*overflow) atomicAdd(&why[reason], 1ull);
        *overflow = 1u;
    }
    __device__ __forceinline__ void note_claim(uint32_t slot) const {
        const uint32_t i = atomicAdd(n_distinct, 1u);
        if (i < (uint32_t)KMAX) klist[i] = (uint16_t)slot;
        else flag(0);
    }
    // narrow: claim-or-find with the key itself, then count
    __device__ __forceinline__ void add(uint64_t key, uint32_t h, uint32_t mult) const {
        uint32_t slot = h & (CAP - 1);
        for (int probe = 0; probe < CAP; probe++) {
            unsigned long long cur = keys[slot];
            if (cur != key) {
                if (cur != ~0ull) { slot = (slot + 1) & (CAP - 1); continue; }
                if (*overflow) return;
                cur = atomicCAS(&keys[slot], ~0ull, (unsigned long long)key);
                if (cur == ~0ull) note_claim(slot);
                else if (cur != key) { slot = (slot + 1) & (CAP - 1); continue; }
            }
            atomicAdd(&cnts[slot], mult);
            return;
        }
        flag(3);
    }
    // wide, pass B1: claim by tag, publish the key (an equal tag is presumed to be the same key; B2 verifies)
    __device__ __forceinline__ void claim(u128 key, uint32_t h, uint32_t tag) const {
        uint32_t slot = h & (CAP - 1);
        for (int probe = 0; probe < CAP; probe++) {
            uint32_t cur = tags[slot];
            if (cur == 0u) {
                if (*overflow) return;
                cur = atomicCAS(&tags[slot], 0u, tag);
                if (cur == 0u) {
                    keys[slot] = (unsigned long long)(uint64_t)(key >> 64);
                    keys_lo[slot] = (unsigned long long)(uint64_t)key;
                    note_claim(slot);
                    return;
                }
            }
            if (cur == tag) return;
            slot = (slot + 1) & (CAP - 1);
        }
        flag(1);
    }
    // wide, pass B2: find the slot whose full key matches, count
    __device__ __forceinline__ void count(u128 key, uint32_t h, uint32_t tag, uint32_t mult) const {
        const unsigned long long hi = (uint64_t)(key >> 64), lo = (uint64_t)key;
        uint32_t slot = h & (CAP - 1);
        for (int probe = 0; probe < CAP; probe++) {
            const uint32_t cur = tags[slot];
            if (cur == 0u) break;
            if (cur == tag && keys[slot] == hi && keys_lo[slot] == lo) { atomicAdd(&cnts[slot], mult); return; }
            slot = (slot + 1) & (CAP - 1);
        }
        flag(2);  // swallowed by a tag collision in B1
    }
};

// PHASE 0: narrow add.  PHASE 1: wide claim.  PHASE 2: wide count.
template <bool WIDE, int CAP, int PHASE> struct KmerSink {
    KmerTable<WIDE, CAP> T;
    uint32_t depth, cval;
    __device__ __forceinline__ void operator()(uint64_t key, uint32_t mult) const {
        uint32_t cls;
        const uint32_t h = narrow_hash(key, cls);
        if (depth == 0 || (cls >> (24u - depth)) == cval) T.add(key, h, mult);
    }
    __device__ __forceinline__ void operator()(u128 key, uint32_t mult) const {
        const uint64_t hi = (uint64_t)(key >> 64), lo = (uint64_t)key;
        // two independent 32-bit lanes: slot = low bits of h1, class = its top bits, tag = h2
        const uint32_t h1 = hash_lane_a((uint32_t)hi, (uint32_t)(hi >> 32), (uint32_t)lo, (uint32_t)(lo >> 32));
        const uint32_t h2 = hash_lane_b((uint32_t)hi, (uint32_t)(hi >> 32), (uint32_t)lo, (uint32_t)(lo >> 32));
        if (depth != 0 && (h1 >> (32u - depth)) != cval) return;
        if (PHASE == 1) T.claim(key, h1, h2 | 1u);
        else T.count(key, h1, h2 | 1u, mult);
    }
};

// Warp-cooperative expansion of up to 32 records (one per lane: words w[], nk k-mers, multiplicity mult; nk = 0 for
// an idle lane) into canonical k-mers: sink(key, mult) is called once per k-mer, 32 k-mers per step.
template <bool WIDE, class Sink>
__device__ __forceinline__ void expand_warp(const uint64_t* w, uint32_t nk, uint32_t mult, int k, int lane, const Sink& sink, volatile uint32_t* overflow) {
    uint32_t pi = nk;  // inclusive prefix of k-mer counts over the warp's 32 records
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const uint32_t o = __shfl_up_sync(0xffffffffu, pi, d); if (lane >= d) pi += o; }
    const uint32_t total = __shfl_sync(0xffffffffu, pi, 31);
    // Source record of k-mer t: the non-empty records are lanes 0 .. r-1 (idle lanes only trail), so it is
    // (number of records that start at or before t) - 1.  Per step every record that starts inside the step's window
    // of 32 k-mers sets one bit; one warp-wide OR and a popcount replace a binary search over the prefix sums.
    const uint32_t pe = pi - nk;  // exclusive prefix: first k-mer of this lane's record
    uint32_t base = 0;            // records that start before the window
    for (uint32_t t0 = 0; t0 < total; t0 += 32) {
        const uint32_t t = t0 + lane;
        const uint32_t rel = pe - t0;
        const uint32_t heads = __reduce_or_sync(0xffffffffu, (nk != 0u && rel < 32u) ? (1u << rel) : 0u);
        const uint32_t s = (base + (uint32_t)__popc(heads & (0xffffffffu >> (31 - lane))) - 1u) & 31u;
        base += (uint32_t)__popc(heads);
        const uint32_t pes = __shfl_sync(0xffffffffu, pe, s);
        const uint32_t ms = __shfl_sync(0xffffffffu, mult, s);
        const uint32_t off = t - pes;  // k-mer index inside the record
        if (!WIDE) {
            const uint64_t ws[2] = {__shfl_sync(0xffffffffu, w[0], s), __shfl_sync(0xffffffffu, w[1], s)};
            if (t < total) {
                const uint64_t fwd = rec_kmer_at<uint64_t, 2>(ws, off, k);
                const uint64_t rc = revcomp(fwd, k);
                sink(fwd < rc ? fwd : rc, ms);
            }
        } else {
            const uint64_t ws[4] = {__shfl_sync(0xffffffffu, w[0], s), __shfl_sync(0xffffffffu, w[1], s), __shfl_sync(0xffffffffu, w[2], s),
                                    __shfl_sync(0xffffffffu, w[3], s)};
            if (t < total) {
                const u128 fwd = rec_kmer_at<u128, 4>(ws, off, k);
                const u128 rc = revcomp(fwd, k);
                sink(fwd < rc ? fwd : rc, ms);  // forward on a tie (Counter64.java:686)
            }
        }
        if (__any_sync(0xffffffffu, *overflow)) break;
    }
}

// ---- bulk-copy / mbarrier plumbing (PTX; sm_90+) ----------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* b, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(b)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* b, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* b) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(b)) : "memory"); }
__device__ __forceinline__ void mbar_wait(uint64_t* b, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}" ::"r"(smem_u32(b)), "r"(parity) : "memory");
}
// global -> shared bulk copy (TMA engine, SASS UBLKCP); bytes % 16 == 0, both addresses 16-byte aligned
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src), "r"(bytes),
                 "r"(smem_u32(bar))
                 : "memory");
}
template <int N> __device__ __forceinline__ void compute_barrier() { asm volatile("bar.sync 1, %0;" ::"n"(N) : "memory"); }

constexpr int CNT_STAGES = 2;
constexpr uint32_t BIN_END = 0xffffffffu;

// what the producer warp hands over per bin
struct BinDesc {
    unsigned long long seg_beg[MAX_SEG];  // address of the bin's first record inside each segment
    uint32_t seg_pre[MAX_SEG + 1];        // bin-local index of the first record of each segment
    uint32_t bin;
};

// issue the bulk copies that bring records [cbeg, cbeg + cn) of the bin into `dst`; one thread
template <int RECW>
__device__ __forceinline__ void issue_chunk(const CountArgs& A, const BinDesc& D, int n_seg, uint32_t cbeg, uint32_t cn, uint64_t* dst, uint64_t* bar) {
    mbar_expect_tx(bar, cn * (uint32_t)(RECW * 8));
    const uint32_t cend = cbeg + cn;
    for (int s = 0; s < n_seg; s++) {
        const uint32_t lo = D.seg_pre[s] > cbeg ? D.seg_pre[s] : cbeg;
        const uint32_t hi = D.seg_pre[s + 1] < cend ? D.seg_pre[s + 1] : cend;
        if (lo < hi)
            bulk_g2s(dst + (size_t)(lo - cbeg) * RECW, reinterpret_cast<const uint64_t*>(D.seg_beg[s]) + (size_t)(lo - D.seg_pre[s]) * RECW, (hi - lo) * (uint32_t)(RECW * 8), bar);
    }
}

// NT compute threads + one producer warp.  The producer draws bin tickets, reads the bin's segment offsets and
// bulk-copies its first chunk of records into one of CNT_STAGES shared-memory buffers while the compute warps are
// still busy with the previous bin; full[]/empty[] mbarriers hand the stages back and forth.
template <bool WIDE, int CAP, int RCAP, int NT, int PER_SM>
__global__ void __launch_bounds__(NT + 32, PER_SM) count_bins_kernel(CountArgs A) {
    using KT = typename std::conditional<WIDE, u128, uint64_t>::type;
    constexpr int RECW = WIDE ? 4 : 2;
    constexpr int CHUNK = RCAP * 3 / 4;
    static_assert(CHUNK % NT == 0, "chunk must be a whole number of records per thread");
    constexpr int PER_THREAD = CHUNK / NT;
    constexpr int NW = NT / 32;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint64_t* rbuf = reinterpret_cast<uint64_t*>(smem_raw);  // [CNT_STAGES][CHUNK * RECW]
    unsigned long long* keys = reinterpret_cast<unsigned long long*>(rbuf + (size_t)CNT_STAGES * CHUNK * RECW);
    unsigned long long* keys_lo = keys + CAP;
    uint32_t* tags = reinterpret_cast<uint32_t*>(keys + (WIDE ? 2 * CAP : CAP));
    uint32_t* cnts = tags + (WIDE ? CAP : 0);
    uint32_t* rtag = cnts + CAP;
    uint32_t* rmult = rtag + RCAP;
    uint16_t* ulist = reinterpret_cast<uint16_t*>(rmult + RCAP);  // [CHUNK] claimed slots of the chunk, in claim order
    uint16_t* klist = ulist + CHUNK; // [KMAX]
    __shared__ uint32_t s_distinct[2], s_nuniq[2], s_overflow, s_sp, s_npass, s_cursor, s_early;
    __shared__ uint32_t s_stack_val[CNT_STACK], s_stack_depth[CNT_STACK];
    __shared__ unsigned long long s_out_base;
    __shared__ BinDesc s_desc[CNT_STAGES];
    __shared__ __align__(8) uint64_t s_full[CNT_STAGES], s_empty[CNT_STAGES], s_aux;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int k = A.k;
    const int n_seg = A.n_seg;

    if (tid == 0) {
        for (int i = 0; i < CNT_STAGES; i++) { mbar_init(&s_full[i], 1); mbar_init(&s_empty[i], 1); }
        mbar_init(&s_aux, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp < NW) {
        for (int i = tid; i < CAP; i += NT) { if (WIDE) tags[i] = 0u; else keys[i] = ~0ull; cnts[i] = 0u; }
        for (int i = tid; i < RCAP; i += NT) { rtag[i] = 0u; rmult[i] = 0u; }
        if (tid == 0) { s_distinct[0] = s_distinct[1] = 0; s_nuniq[0] = s_nuniq[1] = 0; s_overflow = 0; }
    }
    __syncthreads();

    if (warp == NW) {
        // ---------------- producer warp ----------------
        uint32_t it = 0;
        while (true) {
            unsigned long long t = 0;
            if (lane == 0) t = atomicAdd(&A.dstat[DS_TICKET], 1ull);
            t = __shfl_sync(0xffffffffu, t, 0);
            const bool end = t >= (unsigned long long)A.n_tickets;
            const uint32_t bin = end ? 0u : (uint32_t)t * A.bin_stride;
            // per-segment extent of the bin: lanes over segments
            uint32_t tot = 0;
            unsigned long long my_beg[(MAX_SEG + 31) / 32];
            uint32_t my_cnt[(MAX_SEG + 31) / 32], my_pre[(MAX_SEG + 31) / 32];
#pragma unroll
            for (int r = 0; r < (MAX_SEG + 31) / 32; r++) {
                const int sg = r * 32 + lane;
                my_beg[r] = 0; my_cnt[r] = 0;
                if (!end && sg < n_seg) {
                    const SegExt e = A.ext[(size_t)sg * A.n_bins + bin];
                    my_beg[r] = e.addr;
                    my_cnt[r] = e.cnt;
                }
                uint32_t incl = my_cnt[r];
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) { const uint32_t o = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += o; }
                my_pre[r] = tot + incl - my_cnt[r];
                tot += __shfl_sync(0xffffffffu, incl, 31);
            }
            if (!end && tot == 0) continue;  // empty bin: nothing to hand over
            const int st = (int)(it % CNT_STAGES);
            if (it >= (uint32_t)CNT_STAGES) mbar_wait(&s_empty[st], ((it / CNT_STAGES) - 1) & 1);
            BinDesc& D = s_desc[st];
#pragma unroll
            for (int r = 0; r < (MAX_SEG + 31) / 32; r++) {
                const int sg = r * 32 + lane;
                if (sg < n_seg) { D.seg_beg[sg] = my_beg[r]; D.seg_pre[sg] = my_pre[r]; }
            }
            if (lane == 0) { D.seg_pre[n_seg] = tot; D.bin = end ? BIN_END : bin; }
            __syncwarp();
            if (lane == 0) {
                if (end) mbar_arrive(&s_full[st]);
                else issue_chunk<RECW>(A, D, n_seg, 0u, tot < (uint32_t)CHUNK ? tot : (uint32_t)CHUNK, rbuf + (size_t)st * CHUNK * RECW, &s_full[st]);
            }
            if (end) break;
            it++;
        }
        return;
    }

    // ---------------- compute warps ----------------
    // Counters are double buffered by bin parity, so the common case -- one class, one staged chunk -- needs no barrier
    // beyond the ones that separate A | B | K4: thread 0 clears the other parity's counters right behind the
    // first barrier of a bin, when nobody can still be reading them.
    auto clear_all = [&]() {
        for (int i = tid; i < CAP; i += NT) { if (WIDE) tags[i] = 0u; else keys[i] = ~0ull; cnts[i] = 0u; }
        for (int i = tid; i < RCAP; i += NT) { rtag[i] = 0u; rmult[i] = 0u; }
    };
    uint32_t aux_phase = 0;
    for (uint32_t it = 0;; it++) {
        const int st = (int)(it % CNT_STAGES);
        const int par = (int)(it & 1u);
        mbar_wait(&s_full[st], (it / CNT_STAGES) & 1);
        const BinDesc& D = s_desc[st];
        if (D.bin == BIN_END) break;
        const uint64_t* buf = rbuf + (size_t)st * CHUNK * RECW;
        const uint32_t n_rec = D.seg_pre[n_seg];
        uint32_t* const nuniq = &s_nuniq[par];
        const KmerTable<WIDE, CAP> T{keys, keys_lo, tags, cnts, klist, &s_distinct[par], &s_overflow, A.dstat + DS_OVF_WHY};

        // A | B of one chunk of `cn` records sitting in `buf` (`fast`: thread 0 also clears the other parity behind the first barrier)
        auto run_chunk = [&](uint32_t cn, uint32_t depth, uint32_t cval, bool fast) {
            // ---- A: collapse identical records ----
            // One 32-bit word per slot carries a 21-bit tag AND the chunk-local index of the record that claimed the
            // slot, so a later record with the same tag compares itself with the claimant's record (in the staged
            // buffer) on the spot: a proper hash insert with full-key compare, no confirmation pass.
            constexpr uint32_t IDX_BITS = 11, IDX_MASK = (1u << IDX_BITS) - 1u;
            static_assert(CHUNK <= (1 << IDX_BITS), "record index must fit the slot word");
#pragma unroll
            for (int j = 0; j < PER_THREAD; j++) {
                const uint32_t li = (uint32_t)j * NT + tid;  // chunk-local record index
                if (li < cn) {
                    uint64_t v[RECW];
#pragma unroll
                    for (int q = 0; q < RECW; q += 2) {
                        const ulonglong2 x = *reinterpret_cast<const ulonglong2*>(buf + (size_t)li * RECW + q);
                        v[q] = x.x; v[q + 1] = x.y;
                    }
                    uint32_t h, tag;
                    record_hash<RECW>(v, h, tag);
                    const uint32_t word = ((tag | (1u << IDX_BITS)) & ~IDX_MASK) | li;  // never 0
                    uint32_t slot = h & (RCAP - 1);
                    while (true) {  // at most CHUNK < RCAP entries: an empty slot always exists
                        uint32_t cur = rtag[slot];
                        if (cur == 0u) {
                            cur = atomicCAS(&rtag[slot], 0u, word);
                            if (cur == 0u) { ulist[atomicAdd(nuniq, 1u)] = (uint16_t)slot; break; }
                        }
                        if (((cur ^ word) & ~IDX_MASK) == 0u) {
                            const uint64_t* o = buf + (size_t)(cur & IDX_MASK) * RECW;
                            bool same = true;
#pragma unroll
                            for (int q = 0; q < RECW; q += 2) {
                                const ulonglong2 x = *reinterpret_cast<const ulonglong2*>(o + q);
                                same = same && x.x == v[q] && x.y == v[q + 1];
                            }
                            if (same) break;
                        }
                        slot = (slot + 1) & (RCAP - 1);
                    }
                    atomicAdd(&rmult[slot], 1u);
                }
            }
            compute_barrier<NT>();
            // (s_overflow is NOT reset here: warps past this barrier may already be flagging it in phase B.  It is zero on
            // entry to every bin: cleared at kernel start, and by whoever consumed it -- the split path below)
            if (fast && tid == 0) { s_nuniq[par ^ 1] = 0; s_distinct[par ^ 1] = 0; s_npass = 0; s_cursor = 0; }
            // ---- B: expand the distinct records, spread evenly over the warps ----
            const int n_uniq = (int)*nuniq;
            int per = (n_uniq + NW - 1) / NW;
            per = per < 4 ? 4 : per > 32 ? 32 : per;
#pragma unroll 1
            for (int pass = 0; pass < (WIDE ? 2 : 1); pass++) {
                const bool last = pass == (WIDE ? 1 : 0);
                for (int ubase = warp * per; ubase < n_uniq; ubase += NW * per) {
                    if (__any_sync(0xffffffffu, *(volatile uint32_t*)&s_overflow)) break;  // warp-uniform: shuffles follow
                    const int u = ubase + lane;
                    uint32_t mult = 0, nk = 0;
                    uint64_t w[RECW];
#pragma unroll
                    for (int q = 0; q < RECW; q++) w[q] = 0ull;
                    if (lane < per && u < n_uniq) {
                        const uint32_t e = ulist[u];
                        mult = rmult[e];
                        const uint32_t li = rtag[e] & ((1u << 11) - 1u);
                        if (last) { rtag[e] = 0u; rmult[e] = 0u; }  // the slot is this lane's alone: leave it clean
                        if (mult) {
#pragma unroll
                            for (int q = 0; q < RECW; q += 2) {
                                const ulonglong2 x = *reinterpret_cast<const ulonglong2*>(buf + (size_t)li * RECW + q);
                                w[q] = x.x; w[q + 1] = x.y;
                            }
                            nk = (uint32_t)(w[0] >> 48);
                        }
                    }
                    if (!WIDE) expand_warp<false>(w, nk, mult, k, lane, KmerSink<WIDE, CAP, 0>{T, depth, cval}, &s_overflow);
                    else if (pass == 0) expand_warp<true>(w, nk, mult, k, lane, KmerSink<WIDE, CAP, 1>{T, depth, cval}, &s_overflow);
                    else expand_warp<true>(w, nk, mult, k, lane, KmerSink<WIDE, CAP, 2>{T, depth, cval}, &s_overflow);
                }
                compute_barrier<NT>();
            }
        };

        bool slow = n_rec > (uint32_t)CHUNK, resume_split = false;
        if (!slow) {
            // ---- fast path: the whole bin is the staged chunk, depth 0 ----
            run_chunk(n_rec, 0u, 0u, true);
            // (run_chunk ended on a barrier: the stage and the record-tag table are free, the k-mer table is complete)
            const bool ovf = s_overflow != 0;
            const uint32_t nd = s_distinct[par] < (uint32_t)KmerTable<WIDE, CAP>::KMAX ? s_distinct[par] : (uint32_t)KmerTable<WIDE, CAP>::KMAX;
            if (!ovf) {
                if (tid == 0) mbar_arrive(&s_empty[st]);
                // K4: coverage filter + compaction over the occupied slots, all warps (its two counters were cleared
                // behind the bin's first barrier)
                uint32_t mine = 0, inst = 0;
                for (uint32_t i = tid; i < nd; i += NT) {
                    const uint32_t c = cnts[klist[i]];
                    inst += c;
                    mine += (c >= A.min_count && c <= A.max_count) ? 1u : 0u;
                }
#pragma unroll
                for (int d = 16; d > 0; d >>= 1) { mine += __shfl_xor_sync(0xffffffffu, mine, d); inst += __shfl_xor_sync(0xffffffffu, inst, d); }
                if (lane == 0) {
                    if (mine) atomicAdd(&s_npass, mine);
                    if (inst) atomicAdd(&A.dstat[DS_INSTANCES], (unsigned long long)inst);
                }
                compute_barrier<NT>();
                if (tid == 0) {
                    const uint32_t tot = s_npass;
                    s_out_base = (tot && !A.dry) ? atomicAdd(&A.dstat[DS_OUT_CURSOR], (unsigned long long)tot) : 0ull;
                    atomicAdd(&A.dstat[DS_DISTINCT], (unsigned long long)nd);
                    if (!A.dry && s_out_base + tot > A.out_cap) atomicExch(&A.dstat[DS_OVERFLOW], 1ull);
                }
                compute_barrier<NT>();
                const bool room = !A.dry && s_out_base + s_npass <= A.out_cap;
                for (uint32_t i0 = (uint32_t)warp * 32u; i0 < nd; i0 += NT) {
                    const uint32_t i = i0 + lane;
                    bool keep = false;
                    uint32_t c = 0, slot = 0;
                    if (i < nd) { slot = klist[i]; c = cnts[slot]; keep = c >= A.min_count && c <= A.max_count; }
                    const uint32_t ball = __ballot_sync(0xffffffffu, keep);
                    uint32_t base = 0;
                    if (lane == 0 && ball) base = atomicAdd(&s_cursor, (uint32_t)__popc(ball));
                    base = __shfl_sync(0xffffffffu, base, 0);
                    if (i < nd) {
                        if (keep && room) {
                            const unsigned long long o = s_out_base + base + (uint32_t)__popc(ball & ((1u << lane) - 1u));
                            if (!WIDE) reinterpret_cast<uint64_t*>(A.out_keys)[o] = keys[slot];
                            else reinterpret_cast<KT*>(A.out_keys)[o] = ((u128)keys[slot] << 64) | keys_lo[slot];
                            A.out_counts[o] = c;
                        }
                        if (WIDE) tags[slot] = 0u; else keys[slot] = ~0ull;
                        cnts[slot] = 0u;
                    }
                }
                continue;
            }
            // the table overflowed: split depth 0 in two and let the general loop run the halves
            compute_barrier<NT>();
            if (tid == 0) {
                s_sp = 0;
                for (uint32_t c = 0; c < 2u; c++) { s_stack_val[s_sp] = c; s_stack_depth[s_sp] = 1u; s_sp++; }
                atomicAdd(&A.dstat[DS_SPLITS], 1ull);
            }
            clear_all();
            slow = true; resume_split = true;
        }
        // ---- general path: several chunks and / or sub-classes ----
        bool staged = !resume_split;  // the buffer holds chunk 0 of the bin
        compute_barrier<NT>();  // every thread has left the previous bin before the stack is re-armed
        if (tid == 0) {
            if (!resume_split) { s_sp = 1; s_stack_val[0] = 0; s_stack_depth[0] = 0; }
            s_nuniq[par ^ 1] = 0; s_distinct[par ^ 1] = 0;
        }
        while (true) {
            compute_barrier<NT>();
            if (s_sp == 0) break;
            const uint32_t depth = s_stack_depth[s_sp - 1], cval = s_stack_val[s_sp - 1];
            compute_barrier<NT>();
            if (tid == 0) { s_sp--; s_distinct[par] = 0; s_overflow = 0; s_npass = 0; s_cursor = 0; s_early = 0; }
            for (uint32_t cbeg = 0; cbeg < n_rec; cbeg += CHUNK) {
                const uint32_t cn = n_rec - cbeg < (uint32_t)CHUNK ? n_rec - cbeg : (uint32_t)CHUNK;
                if (tid == 0) s_nuniq[par] = 0;
                if (!(staged && cbeg == 0)) {
                    // later chunks and sub-class re-runs: fetched on demand (every thread is past its reads of the buffer)
                    compute_barrier<NT>();
                    if (tid == 0) issue_chunk<RECW>(A, D, n_seg, cbeg, cn, const_cast<uint64_t*>(buf), &s_aux);
                    mbar_wait(&s_aux, aux_phase);
                    aux_phase ^= 1u;
                    staged = false;
                }
                compute_barrier<NT>();
                if (s_overflow) break;
                run_chunk(cn, depth, cval, false);
                if (s_overflow && tid == 0 && 2 * (cbeg + cn) <= n_rec) s_early = 1;  // overflowed within the first half
            }
            compute_barrier<NT>();
            if (s_overflow) {
                // too many distinct k-mers for the table: split this class by the next hash bit(s)
                const uint32_t bits = s_early ? 2u : 1u;
                compute_barrier<NT>();
                if (tid == 0) {
                    if (depth + bits > 20 || s_sp + (1u << bits) > CNT_STACK) {
                        atomicExch(&A.dstat[DS_OVERFLOW], 2ull);
                    } else {
                        for (uint32_t c = 0; c < (1u << bits); c++) { s_stack_val[s_sp] = (cval << bits) | c; s_stack_depth[s_sp] = depth + bits; s_sp++; }
                        atomicAdd(&A.dstat[DS_SPLITS], 1ull);
                    }
                }
                clear_all();
                staged = false;
                continue;
            }
            if (n_rec > (uint32_t)CHUNK) staged = false;
            // ---- K4: coverage filter + compaction over the occupied slots ----
            const uint32_t nd = s_distinct[par] < (uint32_t)KmerTable<WIDE, CAP>::KMAX ? s_distinct[par] : (uint32_t)KmerTable<WIDE, CAP>::KMAX;
            uint32_t mine = 0, inst = 0;
            for (uint32_t i = tid; i < nd; i += NT) {
                const uint32_t c = cnts[klist[i]];
                inst += c;
                mine += (c >= A.min_count && c <= A.max_count) ? 1u : 0u;
            }
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) { mine += __shfl_xor_sync(0xffffffffu, mine, d); inst += __shfl_xor_sync(0xffffffffu, inst, d); }
            if (lane == 0) {
                if (mine) atomicAdd(&s_npass, mine);
                if (inst) atomicAdd(&A.dstat[DS_INSTANCES], (unsigned long long)inst);
            }
            compute_barrier<NT>();
            if (tid == 0) {
                const uint32_t tot = s_npass;
                s_out_base = (tot && !A.dry) ? atomicAdd(&A.dstat[DS_OUT_CURSOR], (unsigned long long)tot) : 0ull;
                atomicAdd(&A.dstat[DS_DISTINCT], (unsigned long long)nd);
                if (!A.dry && s_out_base + tot > A.out_cap) atomicExch(&A.dstat[DS_OVERFLOW], 1ull);
            }
            compute_barrier<NT>();
            const bool room = !A.dry && s_out_base + s_npass <= A.out_cap;
            for (uint32_t i0 = (uint32_t)warp * 32u; i0 < nd; i0 += NT) {
                const uint32_t i = i0 + lane;
                bool keep = false;
                uint32_t c = 0, slot = 0;
                if (i < nd) {
                    slot = klist[i];
                    c = cnts[slot];
                    keep = c >= A.min_count && c <= A.max_count;
                }
                const uint32_t ball = __ballot_sync(0xffffffffu, keep);
                uint32_t base = 0;
                if (lane == 0 && ball) base = atomicAdd(&s_cursor, (uint32_t)__popc(ball));
                base = __shfl_sync(0xffffffffu, base, 0);
                if (i < nd) {
                    if (keep && room) {
                        const unsigned long long o = s_out_base + base + (uint32_t)__popc(ball & ((1u << lane) - 1u));
                        if (!WIDE) reinterpret_cast<uint64_t*>(A.out_keys)[o] = keys[slot];
                        else reinterpret_cast<KT*>(A.out_keys)[o] = ((u128)keys[slot] << 64) | keys_lo[slot];
                        A.out_counts[o] = c;
                    }
                    if (WIDE) tags[slot] = 0u; else keys[slot] = ~0ull;
                    cnts[slot] = 0u;
                }
            }
        }
        // the class loop left through a compute barrier: every thread is done with the stage
        if (tid == 0) { mbar_arrive(&s_empty[st]); s_nuniq[par] = 0; s_distinct[par] = 0; }
    }
}

// ---------------------------------------------------------------------------------------------------------------------------
// The measured alternative (north_star: "hash table or radix / sort + run-length, picked by measurement"): count a bin by
// SORTING.  One CTA per bin ticket: the k-mers of the bin's super-k-mer records are expanded into shared memory (one
// shared-memory atomic per record claims its range), sorted by a bitonic network, and equal neighbours are run-length counted;
// rows inside the coverage bounds go out through one global atomic per warp.  No table, no probing, no tag collisions, no
// splitting: a bin with more k-mers than the array holds is done in P passes over its records, pass p keeping the k-mers of
// hash class p (class sizes are measured first, P doubles until every class fits).  Work per bin is O(T log^2 T) whatever
// the data look like -- against the hash kernel's O(T) on clean reads (where equal super-k-mers collapse before a k-mer is
// touched) and its probing / splitting cost on noisy ones, where every second instance is a k-mer of its own.
// ---------------------------------------------------------------------------------------------------------------------------
template <bool WIDE, int CAPS, int NT>
__global__ void __launch_bounds__(NT) sort_bins_kernel(CountArgs A) {
    using KT = typename std::conditional<WIDE, u128, uint64_t>::type;
    constexpr int RECW = WIDE ? 4 : 2;
    constexpr int MAXP = 64;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    KT* skey = reinterpret_cast<KT*>(smem_raw);  // [CAPS]
    __shared__ uint32_t s_fill, s_total, s_bin, s_hist[MAXP];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int k = A.k;
    while (true) {
        __syncthreads();
        if (tid == 0) {
            const unsigned long long t = atomicAdd(&A.dstat[DS_TICKET], 1ull);
            s_bin = t < (unsigned long long)A.n_tickets ? (uint32_t)t * A.bin_stride : BIN_END;
            s_total = 0;
        }
        __syncthreads();
        const uint32_t bin = s_bin;
        if (bin == BIN_END) break;
        // k-mer instances of the bin
        uint32_t mine = 0;
        for (int sg = 0; sg < A.n_seg; sg++) {
            const SegExt e = A.ext[(size_t)sg * A.n_bins + bin];
            const uint64_t* rec = reinterpret_cast<const uint64_t*>(e.addr);
            for (uint32_t i = tid; i < e.cnt; i += NT) mine += (uint32_t)(rec[(size_t)i * RECW] >> 48);
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, d);
        if (lane == 0 && mine) atomicAdd(&s_total, mine);
        __syncthreads();
        const uint32_t T = s_total;
        if (T == 0) continue;
        if (tid == 0) atomicAdd(&A.dstat[DS_INSTANCES], (unsigned long long)T);
        // passes: one if everything fits, else hash classes whose sizes are measured before anything is written
        uint32_t P = 1;
        if (T > (uint32_t)CAPS) {
            P = 2;
            while ((uint64_t)P * (uint64_t)(CAPS * 3 / 4) < (uint64_t)T && P < (uint32_t)MAXP) P <<= 1;
            while (true) {
                __syncthreads();
                if (tid < MAXP) s_hist[tid] = 0;
                __syncthreads();
                for (int sg = 0; sg < A.n_seg; sg++) {
                    const SegExt e = A.ext[(size_t)sg * A.n_bins + bin];
                    const uint64_t* rec = reinterpret_cast<const uint64_t*>(e.addr);
                    for (uint32_t i = tid; i < e.cnt; i += NT)
                        rec_foreach_kmer<KT, RECW>(rec + (size_t)i * RECW, k, [&](KT key) { atomicAdd(&s_hist[(uint32_t)(key_hash(key) >> 40) & (P - 1u)], 1u); });
                }
                __syncthreads();
                bool fits = true;
                for (uint32_t q = 0; q < P; q++) fits = fits && s_hist[q] <= (uint32_t)CAPS;
                if (fits) break;
                // one k-mer more than CAPS times in a bin (poly-A / poly-G reads, microsatellites): no split helps, the host
                // counts the run again with the hash kernel, which collapses identical records before it touches a k-mer
                if (P >= (uint32_t)MAXP) { if (tid == 0) atomicExch(&A.dstat[DS_OVERFLOW], 2ull); break; }
                P <<= 1;
            }
            if (tid == 0) atomicAdd(&A.dstat[DS_SPLITS], 1ull);
        }
        for (uint32_t p = 0; p < P; p++) {
            __syncthreads();
            if (tid == 0) s_fill = 0;
            __syncthreads();
            for (int sg = 0; sg < A.n_seg; sg++) {
                const SegExt e = A.ext[(size_t)sg * A.n_bins + bin];
                const uint64_t* rec = reinterpret_cast<const uint64_t*>(e.addr);
                for (uint32_t i = tid; i < e.cnt; i += NT) {
                    const uint64_t* r = rec + (size_t)i * RECW;
                    if (P == 1) {
                        uint32_t at = atomicAdd(&s_fill, (uint32_t)(r[0] >> 48));
                        rec_foreach_kmer<KT, RECW>(r, k, [&](KT key) { if (at < (uint32_t)CAPS) skey[at] = key; at++; });
                    } else {
                        rec_foreach_kmer<KT, RECW>(r, k, [&](KT key) {
                            if (((uint32_t)(key_hash(key) >> 40) & (P - 1u)) == p) {
                                const uint32_t at = atomicAdd(&s_fill, 1u);
                                if (at < (uint32_t)CAPS) skey[at] = key;
                            }
                        });
                    }
                }
            }
            __syncthreads();
            const uint32_t n = s_fill < (uint32_t)CAPS ? s_fill : (uint32_t)CAPS;
            if (n == 0) continue;
            uint32_t N2 = 32;
            while (N2 < n) N2 <<= 1;
            for (uint32_t i = n + tid; i < N2; i += NT) skey[i] = ~(KT)0;  // no k-mer has all bits set (k <= 63)
            __syncthreads();
            // bitonic network, ascending
            for (uint32_t k2 = 2; k2 <= N2; k2 <<= 1) {
                for (uint32_t j = k2 >> 1; j > 0; j >>= 1) {
                    for (uint32_t t = tid; t < (N2 >> 1); t += NT) {
                        const uint32_t i = ((t & ~(j - 1u)) << 1) | (t & (j - 1u)), ixj = i | j;
                        const KT a = skey[i], b = skey[ixj];
                        if ((a > b) == ((i & k2) == 0u)) { skey[i] = b; skey[ixj] = a; }
                    }
                    __syncthreads();
                }
            }
            // run lengths, coverage filter, rows out
            uint32_t nd = 0;
            for (uint32_t i0 = (uint32_t)warp * 32u; i0 < n; i0 += NT) {
                const uint32_t i = i0 + lane;
                bool keep = false;
                uint32_t c = 0;
                KT key = 0;
                if (i < n) {
                    key = skey[i];
                    if (i == 0 || skey[i - 1] != key) {
                        c = 1;
                        while (i + c < n && skey[i + c] == key) c++;
                        nd++;
                        keep = c >= A.min_count && c <= A.max_count;
                    }
                }
                const uint32_t ball = __ballot_sync(0xffffffffu, keep);
                if (ball) {
                    unsigned long long base = 0;
                    if (lane == 0) base = atomicAdd(&A.dstat[DS_OUT_CURSOR], (unsigned long long)__popc(ball));
                    base = __shfl_sync(0xffffffffu, base, 0);
                    if (keep) {
                        const unsigned long long o = base + (uint32_t)__popc(ball & ((1u << lane) - 1u));
                        if (o < A.out_cap) { reinterpret_cast<KT*>(A.out_keys)[o] = key; A.out_counts[o] = c; }
                        else atomicExch(&A.dstat[DS_OVERFLOW], 1ull);
                    }
                }
            }
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) nd += __shfl_xor_sync(0xffffffffu, nd, d);
            if (lane == 0 && nd) atomicAdd(&A.dstat[DS_DISTINCT], (unsigned long long)nd);
        }
    }
}
template <bool WIDE, int CAPS, int NT> static cudaError_t launch_sort_count(const CountArgs& A, cudaStream_t st) {
    const size_t smem = (size_t)CAPS * (WIDE ? 16 : 8);
    cudaError_t e = cudaFuncSetAttribute(sort_bins_kernel<WIDE, CAPS, NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    unsigned grid = sm_count() * 3u;  // 64 KB of keys per CTA
    if (grid > A.n_tickets) grid = A.n_tickets;
    sort_bins_kernel<WIDE, CAPS, NT><<<grid, NT, smem, st>>>(A);
    return cudaGetLastError();
}

// (segment, bin) -> extent, for every layout the records may be in (rfx_internal.h: ExtSrc)
__global__ void build_ext_kernel(ExtSrcs S, int n_seg, uint32_t n_bins, int recw, SegExt* __restrict__ ext) {
    const uint64_t total = (uint64_t)n_seg * n_bins;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (uint64_t)gridDim.x * blockDim.x) {
        const int sg = (int)(i / n_bins);
        const uint32_t b = (uint32_t)(i % n_bins);
        const ExtSrc& x = S.s[sg];
        const uint64_t gb = (uint64_t)x.bin_base + b;
        SegExt e;
        e.pad = 0;
        if (x.slab_cap) {
            const uint32_t cn = x.slab_cnt[gb];
            e.cnt = cn < x.slab_cap ? cn : x.slab_cap;
            e.addr = (unsigned long long)(x.rec + gb * x.slab_cap * (uint64_t)recw);
        } else {
            const uint64_t o = x.off[gb], oe = x.off[gb + 1];
            e.cnt = (uint32_t)(oe - o);
            e.addr = (unsigned long long)(x.rec + (o - x.off_sub) * (uint64_t)recw);
        }
        ext[i] = e;
    }
}

// geometry (shared memory per CTA -> CTAs per SM):
//   k <= 31, small: 2 x 768 x 16 B record stages + 2048 x 12 B k-mer table + lists + 1024-entry record table = 61 KB -> 3
//   k <= 31, large: the same with a 4096-slot k-mer table                                                    = 87 KB -> 2
//   k  > 31:        2 x 192 x 32 B record stages + 2048 x 24 B k-mer table + lists + 256-entry record table  = 66 KB -> 3
template <bool WIDE, int CAP, int RCAP, int NT, int PER_SM> static cudaError_t launch_count(const CountArgs& A, cudaStream_t st) {
    const size_t smem = (size_t)CNT_STAGES * (RCAP * 3 / 4) * (WIDE ? 32 : 16) + (size_t)CAP * (WIDE ? 24 : 12) + (size_t)RCAP * 8 +
                        (size_t)(RCAP * 3 / 4) * 2 + (size_t)(CAP * 3 / 4) * 2;
    cudaError_t e = cudaFuncSetAttribute(count_bins_kernel<WIDE, CAP, RCAP, NT, PER_SM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    unsigned grid = sm_count() * PER_SM;
    if (grid > A.n_tickets) grid = A.n_tickets;
    count_bins_kernel<WIDE, CAP, RCAP, NT, PER_SM><<<grid, NT + 32, smem, st>>>(A);
    return cudaGetLastError();
}

// offsets of the first bin of every received slice (its sender's absolute offset of that bin)
__global__ void seg_first_offsets_kernel(const uint64_t* seg_off, int n_seg, uint32_t bps, uint64_t* out) {
    if ((int)threadIdx.x < n_seg) out[threadIdx.x] = seg_off[(size_t)threadIdx.x * (bps + 1)];
}

// the locally held records in whatever layout the partition left them
int stage_count(Ctx* c) {
    if (!c->have_records) return ctx_fail(c, RFX_E_STATE, "rfx_count: no records (push reads first)");
    ExtSrcs S;
    memset(&S, 0, sizeof(S));
    int n_seg = 1;
    const bool segmented = c->shard_id >= 0 && c->n_seg > 0;
    if (segmented) {
        // slices received through NCCL, each grouped by bin with its sender's offsets (rfx_load_segment_device)
        if (c->n_seg > RFX_MAX_SEG) return ctx_fail(c, RFX_E_INVALID, "more than %d record segments", RFX_MAX_SEG);
        uint64_t first[RFX_MAX_SEG];
        const uint32_t bps = c->n_bins;
        RFX_TRY(devbuf_reserve(c, c->seg_base, 64 * sizeof(uint64_t)));
        seg_first_offsets_kernel<<<1, 32, 0, c->stream>>>(c->seg_off.as<uint64_t>(), c->n_seg, bps, c->seg_base.as<uint64_t>());
        RFX_CUDA(c, cudaMemcpyAsync(first, c->seg_base.p, (size_t)c->n_seg * sizeof(uint64_t), cudaMemcpyDeviceToHost, c->stream));
        RFX_CUDA(c, cudaStreamSynchronize(c->stream));
        n_seg = c->n_seg;
        for (int i = 0; i < n_seg; i++) {
            S.s[i].rec = c->rx_records.as<uint64_t>() + c->seg_base_host[i] * (uint64_t)c->recw;
            S.s[i].off = c->seg_off.as<uint64_t>() + (size_t)i * (bps + 1);
            S.s[i].off_sub = first[i];
        }
    } else if (c->slab_cap) {
        // single-pass partition: slab segment + (maybe) the exactly partitioned overflow list
        S.s[0].rec = c->records.as<uint64_t>();
        S.s[0].slab_cnt = c->bin_cursor.as<uint32_t>();
        S.s[0].slab_cap = c->slab_cap;
        if (c->n_ovf) {
            S.s[1].rec = c->rx_records.as<uint64_t>();
            S.s[1].off = c->bin_off.as<uint64_t>();
            n_seg = 2;
        }
    } else {
        S.s[0].rec = c->records.as<uint64_t>();
        S.s[0].off = c->bin_off.as<uint64_t>();
    }
    return stage_count_segments(c, S, n_seg, c->n_bins, true);
}

int stage_count_segments(Ctx* c, const ExtSrcs& S, int n_seg, uint32_t n_bins, bool check_instances) {
    cudaStream_t st = c->stream;
    stage_begin(c);
    // effective coverage bounds (A4)
    uint32_t minc = (uint32_t)(c->prm.min_kmer_coverage < 0 ? 0 : c->prm.min_kmer_coverage);
    uint32_t maxc = (uint32_t)c->prm.max_kmer_coverage;
    if (c->prm.counter_mode) {
        if (c->prm.min_kmer_coverage <= 1) minc = 0;
        if (c->prm.max_kmer_coverage >= 10000000) maxc = 0xffffffffu;
    }
    if (minc < 1) minc = 1;
    // capacity of the filtered table
    uint64_t cap = c->prm.table_capacity > 0 ? (uint64_t)c->prm.table_capacity : 0;
    if (!cap) {
        // every surviving row needs >= minc instances; keep a floor for tiny inputs
        uint64_t inst = c->n_instances ? c->n_instances : c->n_records * c->max_nk;
        if (!check_instances) inst += inst / 4 + 4096;  // a shard's share of the global instances: about the local count
        cap = inst / minc + 1024;
        const uint64_t soft = 1ull << 31;  // 2 G rows (24-40 GB): beyond this the caller must say so
        if (cap > soft) cap = soft;
    }
    const size_t ksz = c->wide ? sizeof(u128) : sizeof(uint64_t);
    RFX_TRY(devbuf_reserve(c, c->keys, cap * ksz));
    RFX_TRY(devbuf_reserve(c, c->counts, cap * sizeof(uint32_t)));
    c->table_cap = cap;
    RFX_CUDA(c, cudaMemsetAsync(c->dstat.p, 0, DS_NSLOTS * sizeof(uint64_t), st));
    RFX_TRY(devbuf_reserve(c, c->seg_ext, ((size_t)n_seg * n_bins + 1) * sizeof(SegExt)));
    if (n_bins) {
        uint64_t g = ((uint64_t)n_seg * n_bins + 255) / 256;
        if (g > sm_count() * 16u) g = sm_count() * 16u;
        build_ext_kernel<<<(unsigned)g, 256, 0, st>>>(S, n_seg, n_bins, c->recw, c->seg_ext.as<SegExt>());
        c->launches++;
    }
    CountArgs A;
    A.ext = c->seg_ext.as<SegExt>();
    A.n_seg = n_seg;
    A.n_bins = n_bins;
    A.k = c->k;
    A.min_count = minc; A.max_count = maxc;
    A.out_keys = c->keys.p; A.out_counts = c->counts.as<uint32_t>();
    A.dstat = c->dstat.as<unsigned long long>();
    A.out_cap = cap;
    A.n_tickets = n_bins; A.bin_stride = 1; A.dry = 0;
    const bool any = check_instances ? c->n_records != 0 : n_bins != 0;
    bool sorted_run = false;
    if (any) {
        cudaEventRecord(c->evk[4], st);
        cudaError_t le;
        const char* variant = getenv("RFX_COUNT_VARIANT");  // skip the pilot and force a kernel (tests, tuning)
        std::string vs = variant ? variant : "";
        // Which kernel: "small" / "large" (hash tables of 2048 / 4096 slots, k <= 31), "hash" (k > 31), "sort" (sort_bins_kernel).
        // Unless forced, k <= 31 runs a pilot: ~300 evenly spaced bins are counted by the hash kernel without writing anything,
        // and the distinct k-mers per bin pick the table geometry.  The sort kernel is the measured alternative and LOSES in
        // every regime tried (one B200, profiles/r2_count_hash_vs_sort.md: clean configs[1] 36.9 ms against 1.2; k = 61 with
        // 1 % errors, where every second instance is a k-mer of its own, 24.4 ms against 9.6), so it is only taken when asked
        // for: RFX_COUNT_VARIANT=sort, or RFX_SORT_RATIO=<x> (the pilot then picks it where distinct / instances > x).
        // The choice is kept per context while the bin count stays the same (a driver pushing batch after batch of one data
        // set) and dropped when a run splits more than 1 % of its bins.
        const char* rs = getenv("RFX_SORT_RATIO");
        if (vs.empty() && c->count_geometry && c->count_geometry_bins == n_bins) {
            vs = c->count_geometry == 1 ? "small" : c->count_geometry == 2 ? "large" : c->count_geometry == 3 ? "hash" : "sort";
        } else if (vs.empty() && c->wide && !rs) {
            vs = "hash";
        } else if (vs.empty()) {
            CountArgs P = A;
            P.n_tickets = n_bins < 296u ? n_bins : 296u;
            P.bin_stride = n_bins / P.n_tickets;
            P.dry = 1;
            le = c->wide ? launch_count<true, 2048, 256, 192, 3>(P, st) : launch_count<false, 4096, 1024, 384, 2>(P, st);
            if (le != cudaSuccess) return ctx_fail(c, RFX_E_CUDA, "count pilot launch failed: %s", cudaGetErrorString(le));
            uint64_t ph[DS_NSLOTS];
            RFX_CUDA(c, cudaMemcpyAsync(ph, c->dstat.p, sizeof(ph), cudaMemcpyDeviceToHost, st));
            RFX_CUDA(c, cudaStreamSynchronize(st));
            RFX_CUDA(c, cudaMemsetAsync(c->dstat.p, 0, DS_NSLOTS * sizeof(uint64_t), st));
            c->launches++;
            const uint64_t per_bin = ph[DS_DISTINCT] / P.n_tickets;
            const double ratio = ph[DS_INSTANCES] ? (double)ph[DS_DISTINCT] / (double)ph[DS_INSTANCES] : 0.0;
            if (rs && ratio > atof(rs)) vs = "sort";
            else if (c->wide) vs = "hash";
            else vs = (per_bin <= 600 && ph[DS_SPLITS] == 0) ? "small" : "large";
            c->count_geometry = vs == "small" ? 1 : vs == "large" ? 2 : vs == "hash" ? 3 : 4;
            c->count_geometry_bins = n_bins;
        }
        sorted_run = vs == "sort";
        if (sorted_run) le = c->wide ? launch_sort_count<true, 4096, 256>(A, st) : launch_sort_count<false, 8192, 256>(A, st);
        else if (c->wide) le = launch_count<true, 2048, 256, 192, 3>(A, st);
        else if (vs == "small") le = launch_count<false, 2048, 1024, 384, 3>(A, st);
        else if (vs == "large") le = launch_count<false, 4096, 1024, 384, 2>(A, st);
        else return ctx_fail(c, RFX_E_INVALID, "RFX_COUNT_VARIANT must be small, large, hash or sort");
        if (le != cudaSuccess) return ctx_fail(c, RFX_E_CUDA, "count kernel launch failed: %s", cudaGetErrorString(le));
        cudaEventRecord(c->evk[5], st);
        c->launches++;
    }
    uint64_t h[DS_NSLOTS];
    RFX_CUDA(c, cudaMemcpyAsync(h, c->dstat.p, sizeof(h), cudaMemcpyDeviceToHost, st));
    cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return ctx_fail(c, RFX_E_CUDA, "count kernel failed: %s", cudaGetErrorString(e));
    if (sorted_run && h[DS_OVERFLOW] == 2) {
        // The sort kernel met a k-mer that fills a hash class beyond its array on its own (one poly-A k-mer of a run of a few
        // thousand reads does).  Count the whole run again with the hash kernel, from zeroed counters and output cursor, and
        // remember that kernel, not the sort kernel, for this context's next runs.
        RFX_CUDA(c, cudaMemsetAsync(c->dstat.p, 0, DS_NSLOTS * sizeof(uint64_t), st));
        const cudaError_t le = c->wide ? launch_count<true, 2048, 256, 192, 3>(A, st) : launch_count<false, 4096, 1024, 384, 2>(A, st);
        if (le != cudaSuccess) return ctx_fail(c, RFX_E_CUDA, "count kernel launch failed: %s", cudaGetErrorString(le));
        cudaEventRecord(c->evk[5], st);
        c->launches++;
        if (c->count_geometry == 4) c->count_geometry = c->wide ? 3 : 2;
        RFX_CUDA(c, cudaMemcpyAsync(h, c->dstat.p, sizeof(h), cudaMemcpyDeviceToHost, st));
        e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) return ctx_fail(c, RFX_E_CUDA, "count kernel failed: %s", cudaGetErrorString(e));
    }
    c->ms[2] += stage_end(c);
    c->ms_kernel[2] = 0;
    if (any) cudaEventElapsedTime(&c->ms_kernel[2], c->evk[4], c->evk[5]);
    if (h[DS_OVERFLOW] == 2)
        return ctx_fail(c, RFX_E_CAPACITY, "a counting bin could not be split further (splits %llu: table full %llu, probe exhausted %llu, tag collision %llu, %llu)",
                        (unsigned long long)h[DS_SPLITS], (unsigned long long)h[DS_OVF_WHY], (unsigned long long)h[DS_OVF_WHY + 1],
                        (unsigned long long)h[DS_OVF_WHY + 2], (unsigned long long)h[DS_OVF_WHY + 3]);
    if (h[DS_OVERFLOW] == 1 || h[DS_OUT_CURSOR] > cap)
        return ctx_fail(c, RFX_E_CAPACITY, "filtered table needs %llu rows, capacity %llu: raise table_capacity",
                        (unsigned long long)h[DS_OUT_CURSOR], (unsigned long long)cap);
    c->n_rows = h[DS_OUT_CURSOR];
    c->n_distinct = h[DS_DISTINCT];
    c->n_bin_splits = h[DS_SPLITS];
    if (c->n_bin_splits * 100 > n_bins) {
        c->count_geometry = 0;  // the remembered geometry no longer fits the data: pilot again next time
        if (c->bin_shrink < 4) c->bin_shrink *= 2;  // ... and smaller bins (rfx_partition.cu: choose_bin_count)
    }
    c->n_shard_instances = h[DS_INSTANCES];
    if (!check_instances) {}  // a shard counts the instances of ITS bins, not those of the reads this rank scanned
    else if (c->n_instances == 0) c->n_instances = h[DS_INSTANCES];
    else if (h[DS_INSTANCES] != c->n_instances)
        return ctx_fail(c, RFX_E_STATE, "internal: counted %llu k-mer instances, extracted %llu", (unsigned long long)h[DS_INSTANCES],
                        (unsigned long long)c->n_instances);
    c->have_counts = true;
    c->have_contigs = false; c->have_sorted = false;
    return RFX_OK;
}

}  // namespace rfx
