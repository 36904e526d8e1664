// rfx_partition.cu -- K2: rolling minimiser scan of the packed reads, super-k-mer records binned by
// canonical minimiser.
//
// This is the device-side replacement of the map side of
//   ReverseComplementKmerBinaryExtractionFromDataset + groupBy("value") hash shuffle
//   (ReflexivDataFrameCounter.java:195-200, ReflexivDSMain.java:204-209):
// instead of materialising every k-mer instance as an 8/16-byte key and shuffling it, consecutive
// k-mers that share a minimiser bin travel together as one 16/32-byte record (about 1.5 B per k-mer
// instance), and all instances of one canonical k-mer are guaranteed to land in one bin because the
// bin is a function of the strand-symmetric minimiser of the k-mer.
//
// One GPU: ONE pass over the reads -- the scan kernel cuts every run's record out of the read and stores it at
// bin * cap + atomicAdd(cursor[bin]) ("slab" layout, SlabFactory).  Runs that are exchanged between GPUs through NCCL
// (rfx_partition) take two passes: descriptors + bin histogram, prefix scan, then emit_records_kernel scatters the
// records into the compact shard-major layout.  One thread walks one read; the register-resident fast path keeps the
// whole sliding-minimum state in registers, the general kernel keeps a lane-interleaved ring in shared memory.
#include "rfx_internal.h"
#include "rfx_scan.cuh"

namespace rfx {

constexpr int PART_THREADS = 128;

// Pass 1 (the only pass that walks the bases): every run of k-mers that share a bin becomes one 32-bit descriptor
// (bin << 8 | n_kmers) plus a 16-bit start position, both in read-interleaved arrays (slot i of read r at
// [i * stride + r]: coalesced across the reads of a warp), and bumps its bin's record count.  A read with more runs
// than descriptor slots (or longer than 65535 k-mers) only counts its extra runs (spill_cnt); pass 2 re-scans such reads.
struct EmitDesc {
    uint32_t* desc;  // already offset by the read index
    uint16_t* pos;   // same layout: first k-mer of the run
    uint64_t stride;
    uint32_t max_slots;
    uint32_t* bin_cnt;
    uint32_t* spill_cnt;
    uint32_t n;        // runs seen
    uint32_t stored;   // runs that got a descriptor (always a prefix of the read's runs)
    RFX_HD void operator()(uint32_t bin, uint32_t first_kmer, uint32_t n_k) {
#if defined(__CUDA_ARCH__)
        if (n < max_slots && first_kmer < 65536u) {
            atomicAdd(&bin_cnt[bin], 1u);  // result unused: compiles to a fire-and-forget RED
            desc[(uint64_t)n * stride] = (bin << 8) | n_k;
            pos[(uint64_t)n * stride] = (uint16_t)first_kmer;
            stored++;
        } else {
            atomicAdd(&spill_cnt[bin], 1u);
        }
        n++;
#else
        (void)bin; (void)first_kmer; (void)n_k;
#endif
    }
};

// The 32 reads of a warp advance in lock step, one base per iteration.  The per-base work (roll the m-mer, hash it,
// sliding minimum) is branch free; what happens only about once per ten k-mers -- the minimiser changes -- is merely
// queued (position + minimiser hash, a few instructions on the few lanes concerned) in a lane-interleaved
// shared-memory queue.  The queues are drained by the whole warp together (at the end of the reads, or when one fills
// up): bin lookup, run cutting and descriptor emission then run with most lanes busy instead of ~3 of 32.
// Semantics are exactly those of bin_scan_read() (rfx_core.h), which the host harness and the spill pass still use.
constexpr int SCAN_Q = 20;  // queued minimiser changes per read between two drains
constexpr uint32_t SCAN_TODO = 0xffffffffu;  // rd_runs marker: left to the general kernel by the fast path

struct RunState {
    uint32_t run_bin, run_start;
    bool have;
};

// what pass 1 does with a run is a template parameter of the scan kernels: a *Factory travels as kernel argument and
// makes the per-read emitter
struct DescFactory {
    uint32_t* desc;
    uint16_t* pos;
    uint64_t stride;
    uint32_t max_slots;
    uint32_t* bin_cnt;
    uint32_t* spill_cnt;
    typedef EmitDesc Emit;
    static constexpr bool kNeedsRuns = true;  // rd_runs[] feeds pass 2
    __device__ __forceinline__ EmitDesc make(uint64_t r, const uint64_t*) const { return EmitDesc{desc + r, pos + r, stride, max_slots, bin_cnt, spill_cnt, 0u, 0u}; }
};

// Single-pass partition ("slab" layout): bin b owns the fixed range [b * cap, (b + 1) * cap) of the record array, so a
// run's record can be cut and stored the moment pass 1 sees it -- one atomic on the bin's cursor, no descriptors,
// no second pass over the reads, no prefix scan.  Records that do not fit their slab go to a small overflow list
// (with their bin), which is partitioned exactly afterwards and reaches the counting kernel as a second segment.
template <int RECW> struct EmitSlab {
    const uint64_t* rd;
    uint64_t* records;
    uint32_t* bin_cnt;
    uint32_t cap;
    uint64_t* ovf_rec;
    uint32_t* ovf_bin;
    unsigned long long* ovf_cursor;  // dstat[DS_OVF_RECORDS]
    unsigned long long ovf_cap;
    int k;
    uint32_t n, stored;
    // The record is cut and stored the moment its run ends.  Deferring the store behind the next run's atomic (so
    // that the two round trips overlap) was measured and is slower: 1.06 ms instead of 1.00 ms with the pending run in
    // four registers, 1.48 ms with its read words prefetched as well (the scan is register bound: 72 registers at 7
    // blocks per SM; 64 registers / 8 blocks: 1.02 ms).
    __device__ __forceinline__ void operator()(uint32_t bin, uint32_t first_kmer, uint32_t n_k) {
        const uint32_t rank = atomicAdd(&bin_cnt[bin], 1u);
        uint64_t rec[RECW];
        rec_build<RECW>(rd, first_kmer, n_k, k, rec);
        uint64_t* dst;
        if (rank < cap) {
            dst = records + ((uint64_t)bin * cap + rank) * RECW;
        } else {
            const unsigned long long o = atomicAdd(ovf_cursor, 1ull);
            if (o >= ovf_cap) return;  // the host sees cursor > capacity and falls back to the two-pass partition
            ovf_bin[o] = bin;
            dst = ovf_rec + o * RECW;
        }
#pragma unroll
        for (int i = 0; i < RECW; i += 2) *reinterpret_cast<ulonglong2*>(dst + i) = make_ulonglong2(rec[i], rec[i + 1]);
    }
};
template <int RECW> struct SlabFactory {
    uint64_t* records;
    uint32_t* bin_cnt;
    uint32_t cap;
    uint64_t* ovf_rec;
    uint32_t* ovf_bin;
    unsigned long long* ovf_cursor;
    unsigned long long ovf_cap;
    int k;
    typedef EmitSlab<RECW> Emit;
    static constexpr bool kNeedsRuns = false;
    __device__ __forceinline__ EmitSlab<RECW> make(uint64_t, const uint64_t* rd) const {
        return EmitSlab<RECW>{rd, records, bin_cnt, cap, ovf_rec, ovf_bin, ovf_cursor, ovf_cap, k, 0u, 0u};
    }
};

template <class Emit> __device__ __forceinline__ void emit_run(Emit& em, uint32_t bin, uint32_t first, uint32_t n_k, uint32_t max_nk) {
    while (n_k > max_nk) { em(bin, first, max_nk); first += max_nk; n_k -= max_nk; }  // same cuts as the streaming rule
    em(bin, first, n_k);
}

// FIXED: the default geometry (k = 31, m = 11, w = 21) as compile-time constants, so masks, shifts and the block
// length fold into immediates; any other (k, m) takes the run-time version of the same code.
template <bool FIXED, class Factory>
__global__ void __launch_bounds__(PART_THREADS)
    bin_scan_kernel(const uint64_t* __restrict__ packed, const uint32_t* __restrict__ rd_len, const uint64_t* __restrict__ rd_woff, uint64_t n_reads,
                    BinParams P, Factory F, uint32_t* __restrict__ rd_runs, unsigned long long* dstat, int only_todo) {
    extern __shared__ uint32_t scan_smem[];
    if (only_todo && dstat[DS_SCAN_TODO] == 0ull) return;  // the fast path took every warp
    const int k = FIXED ? 31 : P.k, m = FIXED ? 11 : P.m, w = FIXED ? 21 : P.w;
    uint32_t* ring = scan_smem + threadIdx.x;                                   // [2*w][PART_THREADS]
    uint32_t* qh = scan_smem + 2 * w * PART_THREADS + threadIdx.x;              // [SCAN_Q][PART_THREADS] minimiser hash
    uint32_t* qp = qh + SCAN_Q * PART_THREADS;                                  // [SCAN_Q][PART_THREADS] k-mer index
    const uint32_t mmask = (m >= 16) ? 0xffffffffu : ((1u << (2 * m)) - 1u);
    const int mtop = 2 * (m - 1);
    const uint32_t rs = PART_THREADS;
    for (uint64_t base = (uint64_t)blockIdx.x * PART_THREADS; base < n_reads; base += (uint64_t)gridDim.x * PART_THREADS) {
        const uint64_t r = base + threadIdx.x;
        uint32_t len = r < n_reads ? rd_len[r] : 0u;
        if (len < (uint32_t)k) len = 0;
        // second pass behind bin_scan_fast_kernel: only the reads it left behind
        const bool mine = r < n_reads && (!only_todo || rd_runs[r] == SCAN_TODO);
        if (only_todo && !__any_sync(0xffffffffu, mine)) continue;
        if (!mine) len = 0;
        const uint64_t* rd = packed + (r < n_reads ? rd_woff[r] : 0ull);
        uint32_t maxlen = len;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) maxlen = max(maxlen, __shfl_xor_sync(0xffffffffu, maxlen, d));
        typename Factory::Emit em = F.make(r, rd);
        RunState rst{0u, 0u, false};
        uint32_t mf = 0, mr = 0, qn = 0, prev_h = 0;
        uint64_t cur = 0;
        uint32_t* blk_cur = ring;
        uint32_t* blk_prev = ring + (uint32_t)w * rs;
        int pib = 0;
        uint32_t pmin = 0xffffffffu;
        auto drain = [&]() {
            uint32_t maxq = qn;
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) maxq = max(maxq, __shfl_xor_sync(0xffffffffu, maxq, d));
            for (uint32_t t = 0; t < maxq; t++) {
                if (t < qn) {
                    const uint32_t i = qp[t * rs];
                    const uint32_t bin = bin_of_minimizer(qh[t * rs], P.n_bins);
                    if (!rst.have) { rst.have = true; rst.run_bin = bin; rst.run_start = i; }
                    else if (bin != rst.run_bin) {
                        emit_run(em, rst.run_bin, rst.run_start, i - rst.run_start, P.max_nk);
                        rst.run_bin = bin; rst.run_start = i;
                    }
                }
            }
            qn = 0;
        };
        for (uint32_t e = 0; e < maxlen; e++) {
            if (e < len) {
                if ((e & 31u) == 0) cur = rd[e >> 5];
                const uint32_t v = (uint32_t)(cur >> 62);
                cur <<= 2;
                mf = ((mf << 2) | v) & mmask;
                mr = (mr >> 2) | ((v ^ 3u) << mtop);
                if (e + 1 >= (uint32_t)m) {
                    const uint32_t j = e + 1 - (uint32_t)m;  // m-mer index
                    const uint32_t h = mmer_hash(mf < mr ? mf : mr);
                    blk_cur[(uint32_t)pib * rs] = h;
                    pmin = h < pmin ? h : pmin;
                    if (j + 1 >= (uint32_t)w) {
                        uint32_t hmin = pmin;
                        if (pib != w - 1) {
                            const uint32_t sfx = blk_prev[(uint32_t)(pib + 1) * rs];
                            hmin = sfx < hmin ? sfx : hmin;
                        }
                        const uint32_t i = j + 1 - (uint32_t)w;  // k-mer index
                        if (i == 0 || hmin != prev_h) {        // minimiser changed: remember where, decide later
                            prev_h = hmin;
                            qh[qn * rs] = hmin;
                            qp[qn * rs] = i;
                            qn++;
                        }
                    }
                    if (++pib == w) {
                        uint32_t sm = 0xffffffffu;
                        for (int t = w - 1; t >= 0; t--) {
                            const uint32_t x = blk_cur[(uint32_t)t * rs];
                            sm = x < sm ? x : sm;
                            blk_cur[(uint32_t)t * rs] = sm;
                        }
                        uint32_t* tmp = blk_cur; blk_cur = blk_prev; blk_prev = tmp;
                        pib = 0; pmin = 0xffffffffu;
                    }
                }
            }
            if (__any_sync(0xffffffffu, qn >= (uint32_t)SCAN_Q)) drain();
        }
        drain();
        if (rst.have) emit_run(em, rst.run_bin, rst.run_start, len - (uint32_t)k + 1u - rst.run_start, P.max_nk);
        if (mine && Factory::kNeedsRuns) {
            const bool spill = em.n > em.stored;
            rd_runs[r] = em.stored | (spill ? 0x80000000u : 0u);  // top bit: this read needs the spill pass
            if (spill) atomicExch(&dstat[DS_SPILL], 1ull);
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Fast path of pass 1 for compile-time (K, M): the whole sliding-minimum state lives in registers.
// The m-mers of a read are taken in blocks of W = K - M + 1 (van Herk / Gil-Werman): 32 bases starting at the block
// are funnelled into one 64-bit window, so every base, shift and mask inside the fully unrolled block is an
// immediate; the block's W hashes stay in registers until its suffix minima are formed at the block end, and the
// minimum of a k-mer's window is min(prefix minimum of this block, suffix minimum of the previous block).  The 32 reads
// of a warp share one position schedule, the one of the LONGEST of them: a shorter read (quality-trimmed data) walks along
// to the end -- its window loads are clamped to its own words -- and simply stops queueing minimiser changes behind its
// last k-mer, so ragged warps stay on this path at the price of the padding (reads of 100..150 bases: 17 %).  Only reads
// beyond 60 000 bases go to the general kernel above (SCAN_TODO).  Results are bit-identical to bin_scan_read() (rfx_core.h).
// ---------------------------------------------------------------------------------------------------------------
constexpr int FAST_Q = 40;  // queued minimiser changes per read between two drains (a block adds at most W)

template <int M, int W> struct FastScan {
    uint32_t mfl, mr;        // rolling m-mer: forward left-aligned in the top 2M bits, reverse complement right-aligned
    uint32_t sfx[W + 1];     // suffix minima of the previous block, sfx[W] = +inf
    uint32_t prev_h, qn;
    uint32_t nk;             // k-mers of THIS lane's read: changes at or behind it are not queued
    uint32_t* qh;            // [FAST_Q][PART_THREADS] lane-interleaved
    uint16_t* qp;

    __device__ __forceinline__ void roll(uint32_t v) {
        mfl = (mfl << 2) | (v << (32 - 2 * M));
        mr = (mr >> 2) | ((v ^ 3u) << (2 * (M - 1)));
    }
    // MODE 0: first block (its last m-mer completes k-mer 0), 1: full block, 2: last, partial block of `lim` m-mers
    template <int MODE> __device__ __forceinline__ void block(uint64_t win, uint32_t i0, int lim) {
        uint32_t hb[W];
        uint32_t pre = 0xffffffffu;
#pragma unroll
        for (int p = 0; p < W; p++) {
            if (MODE == 2 && p >= lim) break;
            roll((uint32_t)(win >> (62 - 2 * p)) & 3u);
            const uint32_t f = mfl >> (32 - 2 * M);
            const uint32_t h = mmer_hash(f < mr ? f : mr);
            hb[p] = h;
            pre = h < pre ? h : pre;
            if (MODE != 0 || p == W - 1) {
                uint32_t hmin = pre;
                if (p != W - 1) hmin = sfx[p + 1] < hmin ? sfx[p + 1] : hmin;
                if ((MODE == 0 || hmin != prev_h) && i0 + (uint32_t)p < nk) {  // minimiser changed (or first k-mer): remember where, decide later
                    prev_h = hmin;
                    qh[qn * PART_THREADS] = hmin;
                    qp[qn * PART_THREADS] = (uint16_t)(i0 + (uint32_t)p);
                    qn++;
                }
            }
        }
        if (MODE != 2) {
            sfx[W - 1] = hb[W - 1];
#pragma unroll
            for (int t = W - 2; t >= 0; t--) sfx[t] = hb[t] < sfx[t + 1] ? hb[t] : sfx[t + 1];
        }
    }
};

template <int K, int M, class Factory>
__global__ void __launch_bounds__(PART_THREADS, 7)  // 72 registers: seven blocks per SM, which is also what the 30 KB of queues allow
    bin_scan_fast_kernel(const uint64_t* __restrict__ packed, const uint32_t* __restrict__ rd_len, const uint64_t* __restrict__ rd_woff, uint64_t n_reads,
                         BinParams P, Factory F, uint32_t* __restrict__ rd_runs, unsigned long long* dstat) {
    constexpr int W = K - M + 1;
    static_assert(W <= 32 && M <= 16 && M >= 2, "one 64-bit window per block");
    __shared__ uint32_t s_qh[FAST_Q * PART_THREADS];
    __shared__ uint16_t s_qp[FAST_Q * PART_THREADS];
    for (uint64_t base = (uint64_t)blockIdx.x * PART_THREADS; base < n_reads; base += (uint64_t)gridDim.x * PART_THREADS) {
        const uint64_t r = base + threadIdx.x;
        const bool valid = r < n_reads;
        if (!__any_sync(0xffffffffu, valid)) continue;  // (valid lanes are a prefix of the warp: lane 0 is one of them)
        const uint32_t len = valid ? rd_len[r] : 0u;
        uint32_t len0 = len;  // the longest read of the warp sets the schedule
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) len0 = max(len0, __shfl_xor_sync(0xffffffffu, len0, d));
        if (len0 > 60000u) {
            if (valid) rd_runs[r] = SCAN_TODO;
            if ((threadIdx.x & 31) == 0) atomicExch(&dstat[DS_SCAN_TODO], 1ull);
            continue;
        }
        if (len0 < (uint32_t)K) {  // no k-mer in any of the 32 reads
            if (valid) rd_runs[r] = 0u;
            continue;
        }
        // the lanes behind the last read walk lane 0's read along (same schedule, nothing emitted)
        const uint64_t woff = __shfl_sync(0xffffffffu, valid ? rd_woff[r] : 0ull, valid ? (int)(threadIdx.x & 31) : 0);
        const uint64_t* rd = packed + woff;
        typename Factory::Emit em = F.make(r, rd);
        RunState rst{0u, 0u, false};
        FastScan<M, W> S;
        S.mfl = 0; S.mr = 0; S.prev_h = 0; S.qn = 0;
        S.nk = len >= (uint32_t)K ? len - (uint32_t)K + 1u : 0u;
        S.qh = s_qh + threadIdx.x; S.qp = s_qp + threadIdx.x;
        const uint64_t last_pos = (uint64_t)len;  // window loads never leave the read's own words (+ the one behind them)
        auto window = [&](uint64_t pos) { return packed_window(rd, pos < last_pos ? pos : last_pos); };
#pragma unroll
        for (int t = 0; t <= W; t++) S.sfx[t] = 0xffffffffu;
        // the whole warp drains its queues together: bin lookup, run cutting and record emission run with most lanes busy
        auto drain = [&](bool final, uint32_t n_kmers) {
            uint32_t maxq = S.qn;
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) maxq = max(maxq, __shfl_xor_sync(0xffffffffu, maxq, d));
            for (uint32_t t = 0; t < maxq; t++) {
                if (valid && t < S.qn) {
                    const uint32_t i = S.qp[t * PART_THREADS];
                    const uint32_t bin = bin_of_minimizer(S.qh[t * PART_THREADS], P.n_bins);
                    if (!rst.have) { rst.have = true; rst.run_bin = bin; rst.run_start = i; }
                    else if (bin != rst.run_bin) {
                        emit_run(em, rst.run_bin, rst.run_start, i - rst.run_start, P.max_nk);
                        rst.run_bin = bin; rst.run_start = i;
                    }
                }
            }
            S.qn = 0;
            if (valid && final && rst.have) emit_run(em, rst.run_bin, rst.run_start, n_kmers - rst.run_start, P.max_nk);
        };
        {   // the first M - 1 bases complete no m-mer
            const uint64_t w0 = rd[0];
#pragma unroll
            for (int t = 0; t < M - 1; t++) S.roll((uint32_t)(w0 >> (62 - 2 * t)) & 3u);
        }
        const uint32_t n_mmers = len0 - (uint32_t)M + 1u;
        const uint32_t n_full = n_mmers / (uint32_t)W, rem = n_mmers % (uint32_t)W;
        // the 64-bit base window of block b + 1 is requested before block b is worked on: its latency (the first touch of
        // a read's words misses L1) hides behind ~500 instructions instead of stalling the warp at every block start
        uint64_t win = window((uint64_t)(M - 1));
        uint64_t win_next = (n_full > 1 || rem) ? window((uint64_t)(M - 1) + (uint64_t)W) : 0ull;
        S.template block<0>(win, 0u - (uint32_t)(W - 1), W);
        for (uint32_t b = 1; b < n_full; b++) {
            win = win_next;
            if (b + 1 < n_full || rem) win_next = window((uint64_t)(M - 1) + (uint64_t)(b + 1) * W);
            S.template block<1>(win, b * W - (uint32_t)(W - 1), W);
            if (__any_sync(0xffffffffu, S.qn > (uint32_t)(FAST_Q - W))) drain(false, 0u);
        }
        if (rem) {
            if (__any_sync(0xffffffffu, S.qn > (uint32_t)(FAST_Q - W))) drain(false, 0u);
            S.template block<2>(win_next, n_full * W - (uint32_t)(W - 1), (int)rem);
        }
        drain(true, S.nk);
        if (!valid) continue;
        if (Factory::kNeedsRuns) {
            const bool spill = em.n > em.stored;
            rd_runs[r] = em.stored | (spill ? 0x80000000u : 0u);
            if (spill) atomicExch(&dstat[DS_SPILL], 1ull);
        } else {
            rd_runs[r] = 0u;  // done (anything but SCAN_TODO)
        }
    }
}

// re-scan of a read with more runs than descriptor slots: runs [max_slots, n) go behind the ranked records of their bin
template <int RECW> struct EmitSpill {
    const uint64_t* rd;
    const uint64_t* bin_off;
    const uint32_t* bin_cnt;
    uint32_t* spill_cur;
    uint64_t* records;
    uint32_t max_slots;
    uint32_t n;
    int k;
    RFX_HD void operator()(uint32_t bin, uint32_t first_kmer, uint32_t n_k) {
#if defined(__CUDA_ARCH__)
        const bool stored = n < max_slots && first_kmer < 65536u;  // same test as pass 1
        n++;
        if (stored) return;
        const uint64_t slot = bin_off[bin] + bin_cnt[bin] + atomicAdd(&spill_cur[bin], 1u);
        uint64_t rec[RECW];
        rec_build<RECW>(rd, first_kmer, n_k, k, rec);
        uint64_t* dst = records + slot * RECW;
#pragma unroll
        for (int i = 0; i < RECW; i += 2) *reinterpret_cast<ulonglong2*>(dst + i) = make_ulonglong2(rec[i], rec[i + 1]);
#else
        (void)bin; (void)first_kmer; (void)n_k;
#endif
    }
};

// Pass 2: per-record work only.  A block owns 32 consecutive reads at a time; its 8 warps take the descriptor slots
// round robin (lane = read, so descriptor loads are coalesced and the 32 reads' packed words -- 1.3 KB -- are fetched
// from HBM once and then served by L1 to all 8 warps).  Each thread claims a place in its run's bin with one atomic
// and cuts the 16/32-byte record out of the read.
template <int RECW>
__global__ void __launch_bounds__(256)
    emit_records_kernel(const uint64_t* __restrict__ packed, const uint64_t* __restrict__ rd_woff, uint64_t n_reads, const uint64_t* __restrict__ bin_off,
                        uint32_t* __restrict__ cursor, const uint32_t* __restrict__ desc, const uint16_t* __restrict__ pos, uint64_t stride,
                        uint32_t max_slots, const uint32_t* __restrict__ rd_runs, uint64_t* __restrict__ records, int k) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t n_tiles = (n_reads + 31) / 32;
    for (uint64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const uint64_t r = tile * 32 + lane;
        uint32_t n = 0;
        const uint64_t* rd = packed;
        if (r < n_reads) { n = rd_runs[r] & 0x7fffffffu; rd = packed + rd_woff[r]; }
        uint32_t nmax = n;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) nmax = max(nmax, __shfl_xor_sync(0xffffffffu, nmax, d));
        // two runs per thread per step: both descriptor loads, both atomics and both stores are in flight together
        for (uint32_t i = warp; i < nmax; i += 16) {
            const uint32_t i2 = i + 8;
            const bool a = i < n, b = i2 < n;
            uint32_t d1 = 0, d2 = 0, f1 = 0, f2 = 0;
            if (a) { const uint64_t idx = (uint64_t)i * stride + r; d1 = desc[idx]; f1 = pos[idx]; }
            if (b) { const uint64_t idx = (uint64_t)i2 * stride + r; d2 = desc[idx]; f2 = pos[idx]; }
            uint64_t s1 = 0, s2 = 0;
            if (a) s1 = bin_off[d1 >> 8] + atomicAdd(&cursor[d1 >> 8], 1u);
            if (b) s2 = bin_off[d2 >> 8] + atomicAdd(&cursor[d2 >> 8], 1u);
            uint64_t rec1[RECW], rec2[RECW];
            if (a) rec_build<RECW>(rd, f1, d1 & 255u, k, rec1);
            if (b) rec_build<RECW>(rd, f2, d2 & 255u, k, rec2);
            if (a) {
                uint64_t* dst = records + s1 * RECW;
#pragma unroll
                for (int q = 0; q < RECW; q += 2) *reinterpret_cast<ulonglong2*>(dst + q) = make_ulonglong2(rec1[q], rec1[q + 1]);
            }
            if (b) {
                uint64_t* dst = records + s2 * RECW;
#pragma unroll
                for (int q = 0; q < RECW; q += 2) *reinterpret_cast<ulonglong2*>(dst + q) = make_ulonglong2(rec2[q], rec2[q + 1]);
            }
        }
    }
}

// reads that did not fit their descriptor slots: re-scan, emit the runs pass 1 could not store
template <int RECW>
__global__ void __launch_bounds__(PART_THREADS)
    emit_spill_kernel(const uint64_t* __restrict__ packed, const uint32_t* __restrict__ rd_len, const uint64_t* __restrict__ rd_woff, uint64_t n_reads,
                      BinParams P, const uint64_t* __restrict__ bin_off, const uint32_t* __restrict__ bin_cnt, uint32_t* __restrict__ spill_cur,
                      uint32_t max_slots, const uint32_t* __restrict__ rd_runs, uint64_t* __restrict__ records) {
    extern __shared__ uint32_t ring_smem[];
    for (uint64_t r = (uint64_t)blockIdx.x * PART_THREADS + threadIdx.x; r < n_reads; r += (uint64_t)gridDim.x * PART_THREADS) {
        if (!(rd_runs[r] >> 31)) continue;
        const uint32_t len = rd_len[r];
        const uint64_t* rd = packed + rd_woff[r];
        EmitSpill<RECW> sp{rd, bin_off, bin_cnt, spill_cur, records, max_slots, 0u, P.k};
        bin_scan_read(rd, len, P, ring_smem + threadIdx.x, (uint32_t)PART_THREADS, sp);
    }
}

struct BinCount2In {
    const uint32_t* cnt;
    const uint32_t* spill;
    __device__ __forceinline__ uint64_t operator()(uint64_t i) const { return (uint64_t)cnt[i] + spill[i]; }
};
struct BinOffset2Out {
    uint64_t* off;
    __device__ __forceinline__ void operator()(uint64_t i, uint64_t excl, uint64_t) const { off[i] = excl; }
};

// bin ids are laid out shard-major: bin b belongs to shard b / bins_per_shard, so every shard's
// records are one contiguous slice of the record array (what the all-to-all sends).
struct BinCountIn {
    const unsigned long long* cnt;
    __device__ __forceinline__ uint64_t operator()(uint64_t i) const { return cnt[i]; }
};
struct BinOffsetOut {
    uint64_t* off;
    unsigned long long* cursor;
    __device__ __forceinline__ void operator()(uint64_t i, uint64_t excl, uint64_t) const {
        off[i] = excl;
        cursor[i] = excl;
    }
};

__global__ void set_last_offset_kernel(uint64_t* off, uint64_t n_bins, const uint64_t* total) { off[n_bins] = *total; }

// Bins are sized so that one bin is one chunk of the counting kernel (rfx_count.cu) and its distinct k-mers fit the
// shared-memory table even when every fourth (k = 31) or second (k = 61) instance is a sequencing-error singleton.
uint32_t choose_bin_count(const Ctx* c, uint64_t instances, int n_shards) {
    uint64_t target = c->prm.bin_target_kmers > 0 ? (uint64_t)c->prm.bin_target_kmers : (c->wide ? 2048 : 6144);
    // Noisy reads fill a bin with k-mers of their own (1 % errors at k = 31: every fourth instance): the shared-memory table
    // overflows and the bin is re-run in sub-classes.  Measured (one B200, gpurun_out/r2_n_*.json, r2_w_*.json): k = 31 with 1 % errors
    // counts in 3.4 ms with bins of 3072 instances against 6.1 ms with 6144; k = 61: 7.4 against 9.6 ms; clean reads prefer the
    // large bins (k = 61: 3.0 against 3.5 ms).  So a context whose last run split more than 1 % of its bins halves them.
    if (c->prm.bin_target_kmers <= 0 && c->sh_world == 0 && n_shards == 1) target /= c->bin_shrink;
    uint64_t nb = (instances + target - 1) / target;
    if (nb < 64) nb = 64;
    if (nb > (1u << 24)) nb = 1u << 24;
    // multiple of the shard count so every shard owns the same number of bins
    nb = (nb + n_shards - 1) / n_shards * n_shards;
    return (uint32_t)nb;
}

// Minimiser length.  Bins are whole minimiser values, so there must be many more values than bins or the bins come
// out uneven: 4^11 / 2 = 2.1 M canonical 11-mers serve up to 2^16 bins, beyond that 15-mers (5.4 * 10^8 values).  The
// rule depends on the TOTAL bin count only, so every rank of a sharded run derives the same m.
void set_minimizer(Ctx* c, uint32_t n_bins_total) {
    int m = c->prm.minimizer_len > 0 ? c->prm.minimizer_len : (n_bins_total > 65536u ? 15 : 11);
    if (m > 16) m = 16;
    if (m > c->k) m = c->k;
    c->m = m;
}

static uint32_t choose_bins(Ctx* c, int n_shards) {
    if (c->forced_bins) return c->forced_bins;
    return choose_bin_count(c, c->n_instances, n_shards);
}

// pass 1 with either emitter: the register-resident scan for the default geometry, then (or instead) the general kernel
template <class Factory> static int launch_scan(Ctx* c, const BinParams& P, const Factory& F, uint64_t read_off, uint64_t n_reads) {
    cudaStream_t st = c->stream;
    unsigned grid = (unsigned)((n_reads + PART_THREADS - 1) / PART_THREADS);
    if (grid < 1) grid = 1;
    // one tile of PART_THREADS reads per block as long as that stays below 148 * 256 blocks: with 7 blocks resident per
    // SM a block-strided loop of 2-3 tiles per block ends in a ragged last wave (measured at config 2: capped at
    // 148 * 64 blocks 1.028 ms, one tile per block 1.006 ms)
    const unsigned grid_cap = sm_count() * 256u;
    if (grid > grid_cap) grid = grid_cap;
    const uint32_t* rd_len = c->rd_len.as<uint32_t>() + read_off;
    const uint64_t* rd_woff = c->rd_woff.as<uint64_t>() + read_off;
    const size_t smem = (size_t)2 * P.w * PART_THREADS * sizeof(uint32_t);           // sliding-minimum ring
    const size_t smem_scan = smem + (size_t)2 * SCAN_Q * PART_THREADS * sizeof(uint32_t);  // + the change queues
    const bool fixed = P.k == 31 && P.m == 11, fast15 = P.k == 31 && P.m == 15;
    RFX_CUDA(c, cudaFuncSetAttribute(bin_scan_kernel<true, Factory>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_scan));
    RFX_CUDA(c, cudaFuncSetAttribute(bin_scan_kernel<false, Factory>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_scan));
    const unsigned grid2 = grid < sm_count() * 4u ? grid : sm_count() * 4u;  // follow-up pass: usually nothing to do
    if (fixed) {
        // register-resident scan for every warp of equal-length reads, then the general kernel for what it left behind
        bin_scan_fast_kernel<31, 11, Factory><<<grid, PART_THREADS, 0, st>>>(c->packed.as<uint64_t>(), rd_len, rd_woff,
                                                                             n_reads, P, F, c->rd_runs.as<uint32_t>(), c->dstat.as<unsigned long long>());
        bin_scan_kernel<true, Factory><<<grid2, PART_THREADS, smem_scan, st>>>(c->packed.as<uint64_t>(), rd_len, rd_woff,
                                                                              n_reads, P, F, c->rd_runs.as<uint32_t>(), c->dstat.as<unsigned long long>(), 1);
        c->launches += 2;
    } else if (fast15) {
        // large inputs (more than 2^16 bins): same register-resident scan with 15-mers
        bin_scan_fast_kernel<31, 15, Factory><<<grid, PART_THREADS, 0, st>>>(c->packed.as<uint64_t>(), rd_len, rd_woff,
                                                                             n_reads, P, F, c->rd_runs.as<uint32_t>(), c->dstat.as<unsigned long long>());
        bin_scan_kernel<false, Factory><<<grid2, PART_THREADS, smem_scan, st>>>(c->packed.as<uint64_t>(), rd_len, rd_woff,
                                                                               n_reads, P, F, c->rd_runs.as<uint32_t>(), c->dstat.as<unsigned long long>(), 1);
        c->launches += 2;
    } else {
        bin_scan_kernel<false, Factory><<<grid, PART_THREADS, smem_scan, st>>>(c->packed.as<uint64_t>(), rd_len, rd_woff,
                                                                               n_reads, P, F, c->rd_runs.as<uint32_t>(), c->dstat.as<unsigned long long>(), 0);
        c->launches++;
    }
    RFX_CUDA(c, cudaGetLastError());
    return RFX_OK;
}

// ---- single-pass partition into slabs (one GPU, records stay local) -------------------------------------------
struct SlabCountIn {
    const uint32_t* cnt;
    __device__ __forceinline__ uint64_t operator()(uint64_t i) const { return cnt[i]; }
};
struct OvfCountIn {
    const uint32_t* cnt;
    uint32_t cap;
    __device__ __forceinline__ uint64_t operator()(uint64_t i) const { return cnt[i] > cap ? cnt[i] - cap : 0u; }
};
template <int RECW>
__global__ void ovf_scatter_kernel(const uint64_t* __restrict__ ovf_rec, const uint32_t* __restrict__ ovf_bin, uint64_t n, const uint64_t* __restrict__ off,
                                   uint32_t* __restrict__ cursor, uint64_t* __restrict__ out) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t b = ovf_bin[i];
        const uint64_t slot = off[b] + atomicAdd(&cursor[b], 1u);
#pragma unroll
        for (int q = 0; q < RECW; q += 2) *reinterpret_cast<ulonglong2*>(out + slot * RECW + q) = *reinterpret_cast<const ulonglong2*>(ovf_rec + i * RECW + q);
    }
}

// The slab partition in three steps, so that the scan can follow the reads as they arrive (rfx_push_fastq uploads the
// text in chunks: the reads of chunk i are scanned while chunk i + 1 is still crossing PCIe):
//   slab_begin   bin geometry and slabs from an (estimated) instance / read count
//   slab_scan    the minimiser scan over reads [off, off + n), records stored as they are cut
//   slab_finish  totals, overflow segment; leaves c->have_records false when the overflow list did not suffice
//                (caller falls back to the two-pass path)
static int slab_begin(Ctx* c, uint64_t est_instances, uint64_t est_reads) {
    cudaStream_t st = c->stream;
    c->n_shards = 1;
    // sharded runs over peer memory: every rank scans into slabs over ALL bins of the run (rfx_shard.cu)
    c->n_bins = (c->sh_world > 0 && c->sh_bins_run) ? c->sh_bins_run : choose_bin_count(c, est_instances, 1);
    set_minimizer(c, c->n_bins);
    const int w = c->k - c->m + 1;
    const size_t nb = c->n_bins;
    // expected records: one run per (w + 1) / 2 k-mers plus one cut per read; slabs hold twice the average bin
    const uint64_t est = est_instances * 2 / (uint64_t)(w + 1) + est_reads + 1;
    uint64_t cap = ((c->wide ? 3 : 2) * est / nb + 8 + 3) & ~(uint64_t)3;  // k > 31: few minimiser loci per bin, uneven bins
    if (cap > 0x7fffffffull) cap = 0x7fffffffull;
    const uint64_t ovf_cap = est / ((c->wide || c->sh_world > 0) ? 3 : 8) + 4096;
    RFX_TRY(devbuf_reserve(c, c->bin_cursor, nb * 4 * sizeof(uint32_t)));
    RFX_TRY(devbuf_reserve(c, c->records, (nb * cap * c->recw + 2) * sizeof(uint64_t)));
    RFX_TRY(devbuf_reserve(c, c->ovf_rec, (ovf_cap * c->recw + 2) * sizeof(uint64_t)));
    RFX_TRY(devbuf_reserve(c, c->ovf_bin, ovf_cap * sizeof(uint32_t)));
    RFX_CUDA(c, cudaMemsetAsync(c->bin_cursor.p, 0, nb * 4 * sizeof(uint32_t), st));
    RFX_CUDA(c, cudaMemsetAsync(c->dstat.as<uint64_t>() + DS_OVF_RECORDS, 0, 2 * sizeof(uint64_t), st));  // + DS_SCAN_TODO
    c->sp_cap = (uint32_t)cap; c->sp_ovf_cap = ovf_cap; c->sp_done = 0; c->sp_kernel_ms = 0;
    return RFX_OK;
}

static int slab_scan(Ctx* c, uint64_t read_off, uint64_t n) {
    if (n == 0) return RFX_OK;
    cudaStream_t st = c->stream;
    BinParams P;
    P.k = c->k; P.m = c->m; P.w = c->k - c->m + 1; P.n_bins = c->n_bins; P.max_nk = c->max_nk;
    RFX_TRY(devbuf_reserve(c, c->rd_runs, (size_t)(n + 1) * sizeof(uint32_t)));
    uint32_t* bin_cnt = c->bin_cursor.as<uint32_t>();
    cudaEventRecord(c->evk[0], st);
    if (c->recw == 2) {
        SlabFactory<2> F{c->records.as<uint64_t>(), bin_cnt, c->sp_cap, c->ovf_rec.as<uint64_t>(), c->ovf_bin.as<uint32_t>(),
                         c->dstat.as<unsigned long long>() + DS_OVF_RECORDS, c->sp_ovf_cap, c->k};
        RFX_TRY(launch_scan(c, P, F, read_off, n));
    } else {
        SlabFactory<4> F{c->records.as<uint64_t>(), bin_cnt, c->sp_cap, c->ovf_rec.as<uint64_t>(), c->ovf_bin.as<uint32_t>(),
                         c->dstat.as<unsigned long long>() + DS_OVF_RECORDS, c->sp_ovf_cap, c->k};
        RFX_TRY(launch_scan(c, P, F, read_off, n));
    }
    cudaEventRecord(c->evk[1], st);
    cudaError_t e = cudaEventSynchronize(c->evk[1]);
    if (e != cudaSuccess) return ctx_fail(c, RFX_E_CUDA, "slab scan failed: %s", cudaGetErrorString(e));
    float ms = 0;
    cudaEventElapsedTime(&ms, c->evk[0], c->evk[1]);
    c->sp_kernel_ms += ms;
    c->sp_done = read_off + n;
    return RFX_OK;
}

static int slab_finish(Ctx* c) {
    cudaStream_t st = c->stream;
    const size_t nb = c->n_bins;
    const uint64_t cap = c->sp_cap;
    uint32_t* bin_cnt = c->bin_cursor.as<uint32_t>();
    uint32_t* ovf_cursor_bin = bin_cnt + nb;
    uint64_t n_records = 0, n_ovf = 0;
    c->ms_kernel[0] = c->sp_kernel_ms; c->ms_kernel[1] = 0;
    c->slab_cap = 0;
    if (c->n_reads) {
        // total records (statistics) and the overflow count
        ScanPlan<uint64_t> plan;
        RFX_TRY(devbuf_reserve(c, c->scan_ws, ScanPlan<uint64_t>::workspace_elems(c->n_bins) * sizeof(uint64_t)));
        plan.bind(c->n_bins, c->scan_ws.as<uint64_t>());
        scan_prepare(plan, SlabCountIn{bin_cnt}, OpAddU64{}, (uint64_t)0, st);
        c->launches += plan.levels;
        RFX_CUDA(c, cudaMemcpyAsync(&n_records, plan.total, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
        RFX_CUDA(c, cudaMemcpyAsync(&n_ovf, c->dstat.as<uint64_t>() + DS_OVF_RECORDS, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
        RFX_CUDA(c, cudaStreamSynchronize(st));
        if (n_ovf > c->sp_ovf_cap) return RFX_OK;  // a few very heavy bins (or a bad size estimate): this input needs the exact layout
        c->n_ovf = n_ovf;
        if (n_ovf) {
            // exact partition of the overflow list -> segment 1 of the counting kernel
            RFX_TRY(devbuf_reserve(c, c->bin_off, (nb + 1) * sizeof(uint64_t)));
            RFX_TRY(devbuf_reserve(c, c->rx_records, (n_ovf * c->recw + 2) * sizeof(uint64_t)));
            scan_prepare(plan, OvfCountIn{bin_cnt, (uint32_t)cap}, OpAddU64{}, (uint64_t)0, st);
            scan_apply(plan, OvfCountIn{bin_cnt, (uint32_t)cap}, BinOffset2Out{c->bin_off.as<uint64_t>()}, OpAddU64{}, (uint64_t)0, st);
            set_last_offset_kernel<<<1, 1, 0, st>>>(c->bin_off.as<uint64_t>(), c->n_bins, plan.total);
            unsigned g2 = (unsigned)((n_ovf + 255) / 256);
            if (g2 > sm_count() * 16u) g2 = sm_count() * 16u;
            if (c->recw == 2) ovf_scatter_kernel<2><<<g2, 256, 0, st>>>(c->ovf_rec.as<uint64_t>(), c->ovf_bin.as<uint32_t>(), n_ovf, c->bin_off.as<uint64_t>(), ovf_cursor_bin, c->rx_records.as<uint64_t>());
            else ovf_scatter_kernel<4><<<g2, 256, 0, st>>>(c->ovf_rec.as<uint64_t>(), c->ovf_bin.as<uint32_t>(), n_ovf, c->bin_off.as<uint64_t>(), ovf_cursor_bin, c->rx_records.as<uint64_t>());
            c->launches += 2 * plan.levels + 2;
            cudaError_t e = cudaStreamSynchronize(st);
            if (e != cudaSuccess) return ctx_fail(c, RFX_E_CUDA, "slab partition failed: %s", cudaGetErrorString(e));
        }
    }
    c->slab_cap = (uint32_t)cap;
    c->n_records = n_records;
    c->have_records = true;
    return RFX_OK;
}

// streamed use (rfx_push_fastq): sizes come from the first chunk, scaled to the whole text
int stage_stream_partition_begin(Ctx* c, uint64_t est_instances, uint64_t est_reads) {
    stage_begin(c);
    int rc = slab_begin(c, est_instances, est_reads);
    c->sp_active = rc == RFX_OK;
    c->ms[1] += stage_end(c);
    return rc;
}
int stage_stream_partition_scan(Ctx* c) {
    if (!c->sp_active) return RFX_OK;
    stage_begin(c);
    int rc = slab_scan(c, c->sp_done, c->n_reads - c->sp_done);
    c->ms[1] += stage_end(c);
    return rc;
}

// One GPU, records stay local.  Uses what the streamed scans already did when they cover every read.
int stage_partition_slab(Ctx* c) {
    stage_begin(c);
    int rc = RFX_OK;
    const bool bins_fit = !(c->sh_world > 0 && c->sh_bins_run) || c->n_bins == c->sh_bins_run;
    if (!(c->sp_active && c->sp_done == c->n_reads && c->n_reads && bins_fit)) {
        rc = slab_begin(c, c->n_instances, c->n_reads);
        if (rc == RFX_OK) rc = slab_scan(c, 0, c->n_reads);
    }
    c->sp_active = false;
    if (rc == RFX_OK) rc = slab_finish(c);
    c->ms[1] += stage_end(c);
    return rc;
}

int stage_partition(Ctx* c, int n_shards) {
    cudaStream_t st = c->stream;
    if (n_shards < 1) return ctx_fail(c, RFX_E_INVALID, "n_shards must be >= 1");
    stage_begin(c);
    c->sp_active = false;  // whatever a streamed slab scan did is not used by the compact layout
    c->n_shards = n_shards;
    c->n_bins = choose_bins(c, n_shards);
    if (c->n_bins % (uint32_t)n_shards) return ctx_fail(c, RFX_E_INVALID, "n_bins_total %u is not a multiple of n_shards %d", c->n_bins, n_shards);
    set_minimizer(c, c->n_bins);
    BinParams P;
    P.k = c->k; P.m = c->m; P.w = c->k - c->m + 1; P.n_bins = c->n_bins; P.max_nk = c->max_nk;
    // descriptor slots per read: twice the expected number of runs (a run is about (w+1)/2 k-mers), 8..64
    const uint64_t avg_nk = c->n_reads ? c->n_instances / c->n_reads : 0;
    uint64_t slots = 2 * (avg_nk / (uint64_t)((P.w + 1) / 2 + 1) + 1) + 4;
    if (slots < 8) slots = 8;
    if (slots > 64) slots = 64;
    const uint64_t stride = (c->n_reads + 31) & ~(uint64_t)31;
    const size_t nb = c->n_bins;
    RFX_TRY(devbuf_reserve(c, c->bin_off, (nb + 1) * sizeof(uint64_t)));
    RFX_TRY(devbuf_reserve(c, c->bin_cursor, nb * 4 * sizeof(uint32_t)));  // ranked count | spill count | cursor | spill cursor
    RFX_TRY(devbuf_reserve(c, c->run_desc, (size_t)(slots * stride + 64) * (sizeof(uint32_t) + sizeof(uint16_t))));
    RFX_TRY(devbuf_reserve(c, c->rd_runs, (size_t)(c->n_reads + 1) * sizeof(uint32_t)));
    RFX_CUDA(c, cudaMemsetAsync(c->bin_cursor.p, 0, nb * 4 * sizeof(uint32_t), st));
    RFX_CUDA(c, cudaMemsetAsync(c->dstat.as<uint64_t>() + DS_SPILL, 0, sizeof(uint64_t), st));
    RFX_CUDA(c, cudaMemsetAsync(c->dstat.as<uint64_t>() + DS_SCAN_TODO, 0, sizeof(uint64_t), st));
    uint32_t* bin_cnt = c->bin_cursor.as<uint32_t>();
    uint32_t* spill_cnt = bin_cnt + nb;
    uint32_t* cursor = spill_cnt + nb;
    uint32_t* spill_cur = cursor + nb;
    uint32_t* desc = c->run_desc.as<uint32_t>();
    uint16_t* pos = reinterpret_cast<uint16_t*>(desc + slots * stride + 32);
    const size_t smem = (size_t)2 * P.w * PART_THREADS * sizeof(uint32_t);           // sliding-minimum ring (spill pass)
    unsigned grid = (unsigned)((c->n_reads + PART_THREADS - 1) / PART_THREADS);
    if (grid < 1) grid = 1;
    if (grid > sm_count() * 64u) grid = sm_count() * 64u;
    c->slab_cap = 0;
    if (c->n_reads) {
        cudaEventRecord(c->evk[0], st);
        RFX_TRY(launch_scan(c, P, DescFactory{desc, pos, stride, (uint32_t)slots, bin_cnt, spill_cnt}, 0, c->n_reads));
        cudaEventRecord(c->evk[1], st);
    }
    // exclusive scan of the per-bin record counts -> bin offsets
    ScanPlan<uint64_t> plan;
    RFX_TRY(devbuf_reserve(c, c->scan_ws, ScanPlan<uint64_t>::workspace_elems(c->n_bins) * sizeof(uint64_t)));
    plan.bind(c->n_bins, c->scan_ws.as<uint64_t>());
    scan_prepare(plan, BinCount2In{bin_cnt, spill_cnt}, OpAddU64{}, (uint64_t)0, st);
    uint64_t n_records = 0, spill = 0;
    RFX_CUDA(c, cudaMemcpyAsync(&n_records, plan.total, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    RFX_CUDA(c, cudaMemcpyAsync(&spill, c->dstat.as<uint64_t>() + DS_SPILL, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    RFX_CUDA(c, cudaStreamSynchronize(st));
    scan_apply(plan, BinCount2In{bin_cnt, spill_cnt}, BinOffset2Out{c->bin_off.as<uint64_t>()}, OpAddU64{}, (uint64_t)0, st);
    set_last_offset_kernel<<<1, 1, 0, st>>>(c->bin_off.as<uint64_t>(), c->n_bins, plan.total);
    c->launches += 2 * plan.levels + 2;
    RFX_TRY(devbuf_reserve(c, c->records, (n_records * c->recw + 2) * sizeof(uint64_t)));
    if (c->n_reads && n_records) {
        const uint64_t n_tiles = (c->n_reads + 31) / 32;
        unsigned g2 = (unsigned)(n_tiles > sm_count() * 64u ? sm_count() * 64u : n_tiles);
        cudaEventRecord(c->evk[2], st);
        if (c->recw == 2)
            emit_records_kernel<2><<<g2, 256, 0, st>>>(c->packed.as<uint64_t>(), c->rd_woff.as<uint64_t>(), c->n_reads, c->bin_off.as<uint64_t>(), cursor, desc, pos,
                                                       stride, (uint32_t)slots, c->rd_runs.as<uint32_t>(), c->records.as<uint64_t>(), c->k);
        else
            emit_records_kernel<4><<<g2, 256, 0, st>>>(c->packed.as<uint64_t>(), c->rd_woff.as<uint64_t>(), c->n_reads, c->bin_off.as<uint64_t>(), cursor, desc, pos,
                                                       stride, (uint32_t)slots, c->rd_runs.as<uint32_t>(), c->records.as<uint64_t>(), c->k);
        c->launches++;
        if (spill) {
            if (c->recw == 2) {
                RFX_CUDA(c, cudaFuncSetAttribute(emit_spill_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                emit_spill_kernel<2><<<grid, PART_THREADS, smem, st>>>(c->packed.as<uint64_t>(), c->rd_len.as<uint32_t>(), c->rd_woff.as<uint64_t>(), c->n_reads, P,
                                                                       c->bin_off.as<uint64_t>(), bin_cnt, spill_cur, (uint32_t)slots, c->rd_runs.as<uint32_t>(),
                                                                       c->records.as<uint64_t>());
            } else {
                RFX_CUDA(c, cudaFuncSetAttribute(emit_spill_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                emit_spill_kernel<4><<<grid, PART_THREADS, smem, st>>>(c->packed.as<uint64_t>(), c->rd_len.as<uint32_t>(), c->rd_woff.as<uint64_t>(), c->n_reads, P,
                                                                       c->bin_off.as<uint64_t>(), bin_cnt, spill_cur, (uint32_t)slots, c->rd_runs.as<uint32_t>(),
                                                                       c->records.as<uint64_t>());
            }
            c->launches++;
        }
        cudaEventRecord(c->evk[3], st);
    }
    cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return ctx_fail(c, RFX_E_CUDA, "partition failed: %s", cudaGetErrorString(e));
    c->ms_kernel[0] = c->ms_kernel[1] = 0;
    if (c->n_reads) cudaEventElapsedTime(&c->ms_kernel[0], c->evk[0], c->evk[1]);
    if (c->n_reads && n_records) cudaEventElapsedTime(&c->ms_kernel[1], c->evk[2], c->evk[3]);
    c->n_records = n_records;
    c->have_records = true;
    c->ms[1] += stage_end(c);
    return RFX_OK;
}

// ---- receiving side of a sharded run: group received records by (local) bin ----------------------
template <int RECW, bool SCATTER>
__global__ void rebin_kernel(const uint64_t* __restrict__ rx, uint64_t n_rec, BinParams P, uint32_t bin_base, uint32_t n_local,
                             unsigned long long* __restrict__ bin_cursor, uint64_t* __restrict__ records, unsigned long long* dstat) {
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n_rec; r += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t rec[RECW];
#pragma unroll
        for (int i = 0; i < RECW; i += 2) {
            const ulonglong2 v = *reinterpret_cast<const ulonglong2*>(rx + r * RECW + i);
            rec[i] = v.x; rec[i + 1] = v.y;
        }
        const uint32_t bin = rec_first_bin<RECW>(rec, P) - bin_base;
        if (bin >= n_local) { atomicExch(&dstat[DS_GRAPH_ERR], 3ull); continue; }  // record sent to the wrong shard
        const unsigned long long slot = atomicAdd(&bin_cursor[bin], 1ull);
        if (SCATTER) {
#pragma unroll
            for (int i = 0; i < RECW; i += 2) *reinterpret_cast<ulonglong2*>(records + slot * RECW + i) = make_ulonglong2(rec[i], rec[i + 1]);
        }
    }
}

int stage_rebin(Ctx* c) {
    cudaStream_t st = c->stream;
    stage_begin(c);
    const uint32_t bps = c->forced_bins / (uint32_t)c->n_shards;
    const uint64_t n_rec = c->rx_bytes / (uint64_t)(c->recw * 8);
    set_minimizer(c, c->forced_bins);
    BinParams P;
    P.k = c->k; P.m = c->m; P.w = c->k - c->m + 1; P.n_bins = c->forced_bins; P.max_nk = c->max_nk;
    c->n_bins = bps;
    RFX_TRY(devbuf_reserve(c, c->bin_off, ((size_t)bps + 1) * sizeof(uint64_t)));
    RFX_TRY(devbuf_reserve(c, c->bin_cursor, (size_t)bps * sizeof(uint64_t)));
    RFX_TRY(devbuf_reserve(c, c->records, (n_rec * c->recw + 2) * sizeof(uint64_t)));
    RFX_CUDA(c, cudaMemsetAsync(c->bin_cursor.p, 0, (size_t)bps * sizeof(uint64_t), st));
    RFX_CUDA(c, cudaMemsetAsync(c->dstat.p, 0, DS_NSLOTS * sizeof(uint64_t), st));
    auto* cursor = c->bin_cursor.as<unsigned long long>();
    auto* dstat = c->dstat.as<unsigned long long>();
    const uint32_t base = (uint32_t)c->shard_id * bps;
    unsigned grid = (unsigned)((n_rec + 255) / 256);
    if (grid < 1) grid = 1;
    if (grid > sm_count() * 16u) grid = sm_count() * 16u;
    if (n_rec) {
        if (c->recw == 2) rebin_kernel<2, false><<<grid, 256, 0, st>>>(c->rx_records.as<uint64_t>(), n_rec, P, base, bps, cursor, nullptr, dstat);
        else rebin_kernel<4, false><<<grid, 256, 0, st>>>(c->rx_records.as<uint64_t>(), n_rec, P, base, bps, cursor, nullptr, dstat);
        c->launches++;
    }
    ScanPlan<uint64_t> plan;
    RFX_TRY(devbuf_reserve(c, c->scan_ws, ScanPlan<uint64_t>::workspace_elems(bps) * sizeof(uint64_t)));
    plan.bind(bps, c->scan_ws.as<uint64_t>());
    scan_prepare(plan, BinCountIn{cursor}, OpAddU64{}, (uint64_t)0, st);
    scan_apply(plan, BinCountIn{cursor}, BinOffsetOut{c->bin_off.as<uint64_t>(), cursor}, OpAddU64{}, (uint64_t)0, st);
    set_last_offset_kernel<<<1, 1, 0, st>>>(c->bin_off.as<uint64_t>(), bps, plan.total);
    c->launches += 2 * plan.levels + 2;
    if (n_rec) {
        if (c->recw == 2) rebin_kernel<2, true><<<grid, 256, 0, st>>>(c->rx_records.as<uint64_t>(), n_rec, P, base, bps, cursor, c->records.as<uint64_t>(), dstat);
        else rebin_kernel<4, true><<<grid, 256, 0, st>>>(c->rx_records.as<uint64_t>(), n_rec, P, base, bps, cursor, c->records.as<uint64_t>(), dstat);
        c->launches++;
    }
    uint64_t err = 0;
    RFX_CUDA(c, cudaMemcpyAsync(&err, dstat + DS_GRAPH_ERR, 8, cudaMemcpyDeviceToHost, st));
    cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return ctx_fail(c, RFX_E_CUDA, "rebin failed: %s", cudaGetErrorString(e));
    if (err) return ctx_fail(c, RFX_E_INVALID, "received a record whose bin is not owned by shard %d", c->shard_id);
    c->n_records = n_rec;
    c->n_instances = 0;  // unknown on the receiving side; rfx_count fills it in
    c->have_records = true;
    c->ms[1] += stage_end(c);
    return RFX_OK;
}

// Receiving side, fast path: every sender's slice arrived grouped by bin together with its bin offsets, so the
// received buffer is used as is; rfx_count walks bin b as the concatenation of segment(s, b) over the senders s.
__global__ void check_segments_kernel(const uint64_t* seg_off, int n_seg, uint32_t bps, const uint64_t* seg_base, uint64_t total_records,
                                      unsigned long long* dstat) {
    // offsets must be monotone and the segments must tile the received records exactly
    uint64_t expect = 0;
    for (int s = 0; s < n_seg; s++) {
        const uint64_t* o = seg_off + (size_t)s * (bps + 1);
        if (seg_base[s] != expect) atomicExch(&dstat[DS_GRAPH_ERR], 4ull);
        for (uint32_t b = threadIdx.x; b < bps; b += blockDim.x)
            if (o[b + 1] < o[b]) atomicExch(&dstat[DS_GRAPH_ERR], 4ull);
        expect += o[bps] - o[0];
    }
    if (expect != total_records) atomicExch(&dstat[DS_GRAPH_ERR], 4ull);
}

int stage_adopt_segments(Ctx* c) {
    cudaStream_t st = c->stream;
    const uint32_t bps = c->forced_bins / (uint32_t)c->n_shards;
    const uint64_t n_rec = c->rx_bytes / (uint64_t)(c->recw * 8);
    RFX_TRY(devbuf_reserve(c, c->seg_base, 64 * sizeof(uint64_t)));
    RFX_CUDA(c, cudaMemcpyAsync(c->seg_base.p, c->seg_base_host, (size_t)c->n_seg * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
    RFX_CUDA(c, cudaMemsetAsync(c->dstat.as<uint64_t>() + DS_GRAPH_ERR, 0, sizeof(uint64_t), st));
    check_segments_kernel<<<1, 256, 0, st>>>(c->seg_off.as<uint64_t>(), c->n_seg, bps, c->seg_base.as<uint64_t>(), n_rec, c->dstat.as<unsigned long long>());
    c->launches++;
    uint64_t err = 0;
    RFX_CUDA(c, cudaMemcpyAsync(&err, c->dstat.as<uint64_t>() + DS_GRAPH_ERR, 8, cudaMemcpyDeviceToHost, st));
    RFX_CUDA(c, cudaStreamSynchronize(st));
    if (err) return ctx_fail(c, RFX_E_INVALID, "received segments do not tile the record buffer");
    c->n_bins = bps;
    c->n_records = n_rec;
    c->n_instances = 0;  // unknown on the receiving side; rfx_count fills it in
    c->have_records = true;
    return RFX_OK;
}

}  // namespace rfx
