// rfx_shard.cu -- multi-GPU runs over peer memory: one context ("rank") per GPU, every rank's device buffers live in one
// arena that the other ranks map (CUDA IPC between processes, plain pointers inside one process), and the kernels of the
// hot path read / write the peers' HBM directly over NVLink / NVSwitch instead of going through a collective library:
//
//   counting   replaces Spark's groupBy hash shuffle (ReflexivDataFrameCounter.java:198-200, ReflexivDSMain.java:207-209).
//              Every rank scans ITS reads into super-k-mer slabs over ALL minimiser bins (the single-GPU one-pass scan);
//              after one cross-GPU barrier the owner of a bin counts it by pulling the bin's records out of every rank's
//              slab with cp.async.bulk (TMA engine) straight into the shared memory of its counting CTA: the exchange IS
//              the load of the counting kernel -- no send buffers, no second copy, no all-to-all.
//   graph      replaces the global sort("k-1") shuffles of the fork filters and of the extension loop
//              (ReflexivDSMain.java:232, 244, 261-326).  A rank keeps its own rows and the index over them; a neighbour
//              probe that leaves the rank (the candidate's minimiser bin belongs to another shard) is first screened
//              against a replicated presence filter and then answered by reading the owner's index over NVLink.
//              Chains are ranked through two levels of splitters; contigs stay with the owner of their head
//              (rfx_shard_graph.cu).
//
// Cross-GPU synchronisation is a flag barrier in peer memory (one small kernel per rank, ~6 us on NVSwitch); small
// values travel through a published block at the start of every arena.
#include <stdlib.h>
#include <string.h>
#include <unistd.h>

#include <chrono>
#include <condition_variable>
#include <map>
#include <mutex>

#include "rfx_graph.cuh"
#include "rfx_internal.h"
#include "rfx_shard.h"

namespace rfx {

// ---- barrier -----------------------------------------------------------------------------------------------------
// Rank `me` writes `epoch` into slot `me` of every rank's flag array and waits until all slots of its own array have
// reached it.  Launched on the context's stream, so everything the rank enqueued before is complete (and, with the
// system-scope fences, visible to the peers) when a peer sees the flag.  A peer that never arrives (a failed rank) ends
// the wait after ~20 s with an error instead of hanging the GPU.
__global__ void xbarrier_kernel(PeerBases P, unsigned long long epoch, unsigned long long* err) {
    const int r = threadIdx.x;
    if (r < P.n) {
        __threadfence_system();
        *reinterpret_cast<volatile unsigned long long*>(&reinterpret_cast<ShardCtl*>(P.base[r])->flags[P.me]) = epoch;
        const volatile unsigned long long* mine = &reinterpret_cast<ShardCtl*>(P.base[P.me])->flags[r];
        const long long t0 = clock64();
        while (*mine < epoch) {
            if (clock64() - t0 > 40000000000ll) {
                *err = 1ull;
                printf("libreflexiv_cuda: rank %d waited ~20 s in barrier %llu for rank %d (its flag says %llu)\n", P.me, epoch, r, *mine);
                break;
            }
            __nanosleep(200);
        }
        __threadfence_system();
    }
}

// Ranks that are threads of ONE process and share a device (how a one-GPU box runs the multi-rank path) meet on the host
// instead: a rank spinning on the GPU would compete with the very kernels it is waiting for (measured: with two ranks
// spinning, the counting kernels of the other ranks on the device do not get to run).
struct HostBarrier {
    std::mutex m;
    std::condition_variable cv;
    int n = 0, arrived = 0, refs = 0;
    unsigned long long gen = 0;
    bool broken = false;
};
static std::mutex g_hb_mutex;
static std::map<unsigned long long, HostBarrier*> g_hb;

static HostBarrier* host_barrier_join(unsigned long long key, int n) {
    std::lock_guard<std::mutex> g(g_hb_mutex);
    HostBarrier*& hb = g_hb[key];
    if (!hb) { hb = new HostBarrier(); hb->n = n; }
    hb->refs++;
    return hb;
}
static void host_barrier_leave(unsigned long long key, HostBarrier* hb) {
    std::lock_guard<std::mutex> g(g_hb_mutex);
    {
        std::lock_guard<std::mutex> l(hb->m);
        hb->broken = true;  // whoever still waits for this rank gives up
    }
    hb->cv.notify_all();
    if (--hb->refs == 0) { g_hb.erase(key); delete hb; }
}
static bool host_barrier_wait(HostBarrier* hb) {
    std::unique_lock<std::mutex> l(hb->m);
    if (hb->broken) return false;
    const unsigned long long my_gen = hb->gen;
    if (++hb->arrived == hb->n) {
        hb->arrived = 0;
        hb->gen++;
        l.unlock();
        hb->cv.notify_all();
        return true;
    }
    const bool ok = hb->cv.wait_for(l, std::chrono::seconds(20), [&] { return hb->gen != my_gen || hb->broken; });
    if (!ok || hb->gen == my_gen) { hb->broken = true; l.unlock(); hb->cv.notify_all(); return false; }
    return true;
}

// everybody's published slots [0, n) -> one local block, so that the host needs ONE device-to-host copy
__global__ void gather_pub_kernel(PeerBases P, int par, int n, unsigned long long* __restrict__ out) {
    for (int i = threadIdx.x; i < P.n * n; i += blockDim.x) {
        const int r = i / n, s = i % n;
        out[(size_t)r * RFX_PUB_SLOTS + s] = *reinterpret_cast<const volatile unsigned long long*>(&reinterpret_cast<const ShardCtl*>(P.base[r])->pub[par][s]);
    }
}

PeerBases peer_bases(const Ctx* c) {
    PeerBases P;
    P.n = c->sh_world; P.me = c->sh_rank;
    for (int r = 0; r < RFX_MAX_RANKS; r++) P.base[r] = r < c->sh_world ? c->peer_base[r] : nullptr;
    return P;
}

int shard_barrier(Ctx* c) {
    c->sh_epoch++;
    if (c->hbar) {
        cudaError_t e = cudaStreamSynchronize(c->stream);
        if (e != cudaSuccess) return ctx_fail(c, RFX_E_CUDA, "kernels in front of a cross-rank barrier failed: %s", cudaGetErrorString(e));
        if (!host_barrier_wait(reinterpret_cast<HostBarrier*>(c->hbar)))
            return ctx_fail(c, RFX_E_STATE, "barrier %llu: a peer rank did not arrive (it failed or was never started)", c->sh_epoch);
        return RFX_OK;
    }
    xbarrier_kernel<<<1, 32, 0, c->stream>>>(peer_bases(c), c->sh_epoch, c->dstat.as<unsigned long long>() + DS_XBAR_ERR);
    c->launches++;
    RFX_CUDA(c, cudaGetLastError());
    return RFX_OK;
}

int shard_check(Ctx* c, const char* what) {
    unsigned long long err = 0;
    RFX_CUDA(c, cudaMemcpyAsync(&err, c->dstat.as<unsigned long long>() + DS_XBAR_ERR, sizeof(err), cudaMemcpyDeviceToHost, c->stream));
    cudaError_t e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) return ctx_fail(c, RFX_E_CUDA, "%s failed: %s", what, cudaGetErrorString(e));
    if (err) return ctx_fail(c, RFX_E_STATE, "%s: a peer rank did not reach the barrier (it failed or was never started)", what);
    return RFX_OK;
}

// Slot 0 of the published block: the status (-rc), then the n host values, then the n_dev device counters.  Every exchange
// starts at slot 0 of the half its parity picks, and a caller reads back only what that exchange wrote.  One host
// synchronisation.
int shard_exchange(Ctx* c, int rc, int n, const unsigned long long* mine, PubVals& all, int n_dev, const int* dev_slots) {
    cudaEventRecord(c->ev_comm[0], c->stream);
    unsigned long long* h = c->h_pub;  // [0, SLOTS): staging of the own values, [SLOTS, ...): everybody's
    h[0] = (unsigned long long)-rc;
    for (int i = 0; i < n; i++) h[1 + i] = mine[i];
    ShardCtl* own = reinterpret_cast<ShardCtl*>(c->arena);
    const int par = (int)(c->sh_exchanges++ & 1u);
    RFX_CUDA(c, cudaMemcpyAsync(&own->pub[par][0], h, (size_t)(1 + n) * sizeof(unsigned long long), cudaMemcpyHostToDevice, c->stream));
    for (int i = 0; i < n_dev; i++)
        RFX_CUDA(c, cudaMemcpyAsync(&own->pub[par][1 + n + i], c->dstat.as<unsigned long long>() + dev_slots[i], sizeof(unsigned long long), cudaMemcpyDeviceToDevice, c->stream));
    RFX_TRY(shard_barrier(c));
    gather_pub_kernel<<<1, 256, 0, c->stream>>>(peer_bases(c), par, 1 + n + n_dev, c->d_pub);
    c->launches++;
    RFX_CUDA(c, cudaMemcpyAsync(h + RFX_PUB_SLOTS, c->d_pub, (size_t)c->sh_world * RFX_PUB_SLOTS * sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
    cudaEventRecord(c->ev_comm[1], c->stream);
    RFX_TRY(shard_check(c, "shard exchange"));
    float ms = 0;
    cudaEventElapsedTime(&ms, c->ev_comm[0], c->ev_comm[1]);
    c->ms_comm += ms;
    all.world = c->sh_world;
    for (int r = 0; r < c->sh_world; r++) {
        const unsigned long long* v = h + (size_t)(r + 1) * RFX_PUB_SLOTS;
        if (v[0]) {  // the lowest failing rank keeps its own message
            const int code = -(int)v[0];
            return r == c->sh_rank ? rc : ctx_fail(c, code, "rank %d failed with error %d in this collective call", r, code);
        }
        for (int i = 0; i < n + n_dev; i++) all.v[r][i] = v[1 + i];
    }
    return RFX_OK;
}

void shard_release(Ctx* c) {
    if (c->hbar) { host_barrier_leave(c->hbar_key, reinterpret_cast<HostBarrier*>(c->hbar)); c->hbar = nullptr; }
    for (int r = 0; r < RFX_MAX_RANKS; r++) {
        if (c->peer_ipc[r] && c->peer_base[r]) cudaIpcCloseMemHandle(c->peer_base[r]);
        c->peer_base[r] = nullptr; c->peer_ipc[r] = false;
    }
    if (c->h_pub) { cudaFreeHost(c->h_pub); c->h_pub = nullptr; }
    for (int i = 0; i < 2; i++) if (c->ev_comm[i]) { cudaEventDestroy(c->ev_comm[i]); c->ev_comm[i] = nullptr; }
    shard_graph_release(c);
    if (c->arena) { cudaFree(c->arena); c->arena = nullptr; }
    c->sh_rank = -1; c->sh_world = 0;
}

// ---- sharded counting ----------------------------------------------------------------------------------------------
int stage_count_sharded(Ctx* c) {
    if (c->sh_world < 1 || !c->peer_base[c->sh_rank]) return ctx_fail(c, RFX_E_STATE, "rfx_count_sharded: call rfx_shard_init / rfx_shard_connect first");
    const int world = c->sh_world, me = c->sh_rank;
    unsigned long long mine[8];
    static_assert(sizeof(mine) / sizeof(mine[0]) <= PUB_VALS, "the slab exchange fits the published block");
    PubVals all;
    c->ms_comm = 0;
    // 1. the bin count every rank uses: given by the caller, or agreed on from the global number of k-mer instances
    uint32_t B = c->sh_bins;
    if (!B) {
        mine[0] = c->n_instances;
        RFX_TRY(shard_exchange(c, RFX_OK, 1, mine, all));
        B = choose_bin_count(c, all.sum(0), world);
    }
    int prc = B % (uint32_t)world ? ctx_fail(c, RFX_E_INVALID, "sharded counting: %u bins are not a multiple of %d ranks", B, world) : RFX_OK;
    const uint32_t bps = B / (uint32_t)world;
    // 2. own reads -> slabs over all B bins (the streamed scan of rfx_push_fastq already did it when it ran with B bins)
    c->sh_bins_run = B;
    c->shard_id = -1; c->n_seg = 0;
    if (prc == RFX_OK) prc = stage_partition_slab(c);
    if (prc == RFX_OK && !c->have_records) {
        // A few minimiser bins hold most of this rank's records (low-complexity reads: poly-A / poly-G, microsatellites) and the
        // overflow list was too small.  Unlike one GPU there is no compact layout to fall back to, but the scan counted every
        // record that missed its slab: one more scan with a list of exactly that many records always fits.
        const unsigned long long need = c->n_ovf;
        prc = stage_partition_slab(c, need);
        if (prc == RFX_E_NOMEM) {
            const std::string why = c->err;
            prc = ctx_fail(c, RFX_E_CAPACITY, "sharded counting: the overflow list of this rank's heavy minimiser bins (%llu records) does not fit: %s", need, why.c_str());
        } else if (prc == RFX_OK && !c->have_records) {
            prc = ctx_fail(c, RFX_E_STATE, "internal: the re-scan overflowed its list of %llu records (%llu)", need, (unsigned long long)c->n_ovf);
        }
    }
    c->sh_bins_run = c->sh_bins;
    // 3. tell the others where the slabs are, or that this rank has none
    auto off_of = [&](const void* p) -> unsigned long long { return p ? (unsigned long long)((const uint8_t*)p - c->arena) : 0ull; };
    mine[0] = off_of(c->records.p);
    mine[1] = off_of(c->bin_cursor.p);
    mine[2] = c->slab_cap;
    mine[3] = c->n_ovf ? off_of(c->rx_records.p) : 0ull;
    mine[4] = c->n_ovf ? off_of(c->bin_off.p) : 0ull;
    mine[5] = c->n_ovf;
    mine[6] = B;
    mine[7] = c->n_instances;
    RFX_TRY(shard_exchange(c, prc, 8, mine, all));
    // 4. count the own bins out of everybody's slabs (and overflow lists)
    ExtSrcs S;
    memset(&S, 0, sizeof(S));
    int n_seg = 0;
    for (int r = 0; r < world; r++) {
        if (all.at(r, 6) != B) return ctx_fail(c, RFX_E_STATE, "sharded counting: rank %d uses %llu bins, this rank %u", r, all.at(r, 6), B);
        ExtSrc& a = S.s[n_seg++];
        a.rec = reinterpret_cast<const uint64_t*>(c->peer_base[r] + all.at(r, 0));
        a.slab_cnt = reinterpret_cast<const uint32_t*>(c->peer_base[r] + all.at(r, 1));
        a.slab_cap = (uint32_t)all.at(r, 2);
        a.bin_base = (uint32_t)me * bps;
        if (all.at(r, 5)) {
            ExtSrc& o = S.s[n_seg++];
            o.rec = reinterpret_cast<const uint64_t*>(c->peer_base[r] + all.at(r, 3));
            o.off = reinterpret_cast<const uint64_t*>(c->peer_base[r] + all.at(r, 4));
            o.bin_base = (uint32_t)me * bps;
        }
    }
    c->sh_inst_global = all.sum(7);
    const int crc = stage_count_segments(c, S, n_seg, bps, false);
    // 5. nobody may touch its slabs again before every rank has counted; the same exchange tells everybody the global row count
    mine[0] = c->n_rows;
    RFX_TRY(shard_exchange(c, crc, 1, mine, all));
    c->sh_rows_global = all.sum(0);
    c->n_bins = B;
    return RFX_OK;
}

// ---- re-sharding a loaded table (rfx_shard_table) ------------------------------------------------------------------
// A Count_<k> table read from disk arrives in arbitrary slices.  Every rank routes its rows to the owner of their minimiser
// bin (the very map the sharded graph stages expect), scatters them grouped by owner into a send buffer in its arena, and
// every owner pulls its rows out of every rank's send buffer with one kernel: the table is then laid out as
// rfx_count_sharded leaves it.  About 12 B per row (k <= 31) cross the links once.
template <class KT>
__global__ void table_route_kernel(const KT* __restrict__ keys, uint64_t n_rows, int k, int m, uint32_t B, uint32_t bps, uint8_t* __restrict__ owner,
                                   unsigned long long* __restrict__ hist) {
    __shared__ unsigned int s_hist[RFX_MAX_RANKS];
    if (threadIdx.x < RFX_MAX_RANKS) s_hist[threadIdx.x] = 0;
    __syncthreads();
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n_rows; r += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t a, b;
        const uint32_t o = row_bin<KT>(keys[r], k, m, B, a, b) / bps;
        owner[r] = (uint8_t)o;
        atomicAdd(&s_hist[o], 1u);
    }
    __syncthreads();
    if (threadIdx.x < RFX_MAX_RANKS && s_hist[threadIdx.x]) atomicAdd(&hist[threadIdx.x], (unsigned long long)s_hist[threadIdx.x]);
}

// rows -> send buffer grouped by owner; the lanes of a warp that go to the same owner take their places with one atomic
template <class KT>
__global__ void table_scatter_kernel(const KT* __restrict__ keys, const uint32_t* __restrict__ counts, const uint8_t* __restrict__ owner, uint64_t n_rows,
                                     unsigned long long* __restrict__ cursor, KT* __restrict__ out_keys, uint32_t* __restrict__ out_counts) {
    const unsigned lane = threadIdx.x & 31u;
    const uint64_t warps = (uint64_t)gridDim.x * (blockDim.x >> 5);
    for (uint64_t base = ((uint64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * 32u; base < n_rows; base += warps * 32u) {
        const uint64_t r = base + lane;
        const bool valid = r < n_rows;
        const int o = valid ? (int)owner[r] : -1;
        const unsigned same = __match_any_sync(0xffffffffu, o);
        const int leader = __ffs(same) - 1;
        unsigned long long at = 0;
        if (valid && (int)lane == leader) at = atomicAdd(&cursor[o], (unsigned long long)__popc(same));
        at = __shfl_sync(0xffffffffu, at, leader);
        if (valid) {
            at += (unsigned long long)__popc(same & ((1u << lane) - 1u));
            out_keys[at] = keys[r];
            out_counts[at] = counts[r];
        }
    }
}

// what an owner pulls: sender q's rows for it start at keys[q] / counts[q] (addresses as seen from this device) and land at
// [start[q], start[q + 1]) of the new table
struct TablePull {
    const void* keys[RFX_MAX_RANKS];
    const uint32_t* counts[RFX_MAX_RANKS];
    unsigned long long start[RFX_MAX_RANKS + 1];
    int n;
};
template <class KT>
__global__ void table_pull_kernel(const __grid_constant__ TablePull P, KT* __restrict__ keys, uint32_t* __restrict__ counts) {
    const uint64_t total = P.start[P.n];
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (uint64_t)gridDim.x * blockDim.x) {
        int q = 0;
        while (i >= P.start[q + 1]) q++;
        const uint64_t j = i - P.start[q];
        keys[i] = reinterpret_cast<const KT*>(P.keys[q])[j];
        counts[i] = P.counts[q][j];
    }
}

static unsigned table_grid(uint64_t n) {
    const uint64_t g = (n + 255) / 256, cap = (uint64_t)sm_count() * 8;
    return (unsigned)(g < 1 ? 1 : g > cap ? cap : g);
}

// send buffer: [histogram per owner | cursor per owner] (256 B), keys (16-byte aligned), counts, owner of every row
static size_t send_keys_off() { return 256; }
static size_t send_counts_off(uint64_t n, size_t ksz) { return send_keys_off() + ((n * ksz + 255) & ~(size_t)255); }
static size_t send_owner_off(uint64_t n, size_t ksz) { return send_counts_off(n, ksz) + ((n * sizeof(uint32_t) + 255) & ~(size_t)255); }

template <class KT> static int table_route_scatter(Ctx* c, uint32_t B, uint32_t bps, unsigned long long* hist) {
    cudaStream_t st = c->stream;
    const uint64_t n = c->n_rows;
    const size_t ksz = sizeof(KT);
    RFX_TRY(devbuf_reserve(c, c->sh_send, send_owner_off(n, ksz) + n + 256));
    uint8_t* s = c->sh_send.as<uint8_t>();
    unsigned long long* d_hist = reinterpret_cast<unsigned long long*>(s);
    uint8_t* owner = s + send_owner_off(n, ksz);
    RFX_CUDA(c, cudaMemsetAsync(d_hist, 0, RFX_MAX_RANKS * sizeof(unsigned long long), st));
    if (n) {
        table_route_kernel<KT><<<table_grid(n), 256, 0, st>>>(c->keys.as<KT>(), n, c->k, c->m, B, bps, owner, d_hist);
        c->launches++;
        RFX_CUDA(c, cudaGetLastError());
    }
    RFX_CUDA(c, cudaMemcpyAsync(hist, d_hist, RFX_MAX_RANKS * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    RFX_CUDA(c, cudaStreamSynchronize(st));
    unsigned long long cur[RFX_MAX_RANKS], sum = 0;
    for (int o = 0; o < RFX_MAX_RANKS; o++) { cur[o] = sum; sum += hist[o]; }
    if (sum != n) return ctx_fail(c, RFX_E_STATE, "rfx_shard_table: routed %llu of %llu rows", sum, (unsigned long long)n);
    if (n) {
        RFX_CUDA(c, cudaMemcpyAsync(d_hist + RFX_MAX_RANKS, cur, sizeof(cur), cudaMemcpyHostToDevice, st));
        table_scatter_kernel<KT><<<table_grid(n), 256, 0, st>>>(c->keys.as<KT>(), c->counts.as<uint32_t>(), owner, n, d_hist + RFX_MAX_RANKS,
                                                                reinterpret_cast<KT*>(s + send_keys_off()), reinterpret_cast<uint32_t*>(s + send_counts_off(n, ksz)));
        c->launches++;
        RFX_CUDA(c, cudaGetLastError());
    }
    return RFX_OK;
}

template <class KT> static int table_pull(Ctx* c, const TablePull& P) {
    const uint64_t recv = P.start[P.n];
    RFX_TRY(devbuf_reserve(c, c->keys, (recv + 1) * sizeof(KT)));
    RFX_TRY(devbuf_reserve(c, c->counts, (recv + 1) * sizeof(uint32_t)));
    if (recv) {
        table_pull_kernel<KT><<<table_grid(recv), 256, 0, c->stream>>>(P, c->keys.as<KT>(), c->counts.as<uint32_t>());
        c->launches++;
        RFX_CUDA(c, cudaGetLastError());
    }
    return RFX_OK;
}

int stage_shard_table(Ctx* c) {
    if (c->sh_world < 1 || !c->peer_base[c->sh_rank]) return ctx_fail(c, RFX_E_STATE, "rfx_shard_table: call rfx_shard_init / rfx_shard_connect first");
    const int world = c->sh_world, me = c->sh_rank;
    unsigned long long mine[2 + RFX_MAX_RANKS];
    static_assert(sizeof(mine) / sizeof(mine[0]) <= PUB_VALS, "the routing exchange fits the published block");
    PubVals all;
    c->st_active = false;
    c->ms_comm = 0;
    stage_begin(c);
    // 1. what every rank holds.  Every rank checks every rank's values in the same order, so that all ranks return the same
    //    error together
    const int rc_have = c->have_counts ? RFX_OK : ctx_fail(c, RFX_E_STATE, "rfx_shard_table: no count table on this rank (every rank loads a slice first, an empty one will do)");
    mine[0] = c->have_counts ? c->n_rows : 0;
    mine[1] = (unsigned long long)c->k;
    mine[2] = c->sh_bins;
    RFX_TRY(shard_exchange(c, rc_have, 3, mine, all));
    uint64_t rows_global = 0;
    for (int r = 0; r < world; r++) {
        if (all.at(r, 1) != all.at(0, 1)) return ctx_fail(c, RFX_E_INVALID, "rfx_shard_table: rank %d has k = %llu, rank 0 k = %llu", r, all.at(r, 1), all.at(0, 1));
        if (all.at(r, 2) != all.at(0, 2)) return ctx_fail(c, RFX_E_INVALID, "rfx_shard_table: rank %d set %llu bins, rank 0 %llu", r, all.at(r, 2), all.at(0, 2));
        rows_global += all.at(r, 0);
    }
    // the bin count: the caller's, or the one counting from reads picks for this many rows at typical coverage (~100 rows a bin)
    uint32_t B = (uint32_t)all.at(0, 2);
    if (!B) B = choose_bin_count(c, 64 * rows_global, world);
    if (B % (uint32_t)world) return ctx_fail(c, RFX_E_INVALID, "rfx_shard_table: %u bins are not a multiple of %d ranks", B, world);
    const uint32_t bps = B / (uint32_t)world;
    set_minimizer(c, B);
    // 2. own rows -> send buffer grouped by owner
    unsigned long long hist[RFX_MAX_RANKS] = {0};
    const int rc_send = c->wide ? table_route_scatter<u128>(c, B, bps, hist) : table_route_scatter<uint64_t>(c, B, bps, hist);
    const size_t ksz = c->wide ? sizeof(u128) : sizeof(uint64_t);
    const unsigned long long send_at = c->sh_send.p ? (unsigned long long)(c->sh_send.as<uint8_t>() - c->arena) : 0ull;
    mine[0] = send_at + send_keys_off();
    mine[1] = send_at + send_counts_off(c->n_rows, ksz);
    for (int o = 0; o < world; o++) mine[2 + o] = hist[o];
    RFX_TRY(shard_exchange(c, rc_send, 2 + world, mine, all));
    uint64_t sent = 0;
    for (int r = 0; r < world; r++)
        for (int o = 0; o < world; o++) sent += all.at(r, 2 + o);
    if (sent != rows_global) return ctx_fail(c, RFX_E_STATE, "rfx_shard_table: %llu rows routed, %llu loaded", (unsigned long long)sent, (unsigned long long)rows_global);
    // 3. pull the own rows out of every rank's send buffer
    TablePull P;
    memset(&P, 0, sizeof(P));
    P.n = world;
    for (int q = 0; q < world; q++) {
        uint64_t before = 0;  // rows of sender q that go to lower ranks
        for (int o = 0; o < me; o++) before += all.at(q, 2 + o);
        P.keys[q] = c->peer_base[q] + all.at(q, 0) + before * ksz;
        P.counts[q] = reinterpret_cast<const uint32_t*>(c->peer_base[q] + all.at(q, 1)) + before;
        P.start[q + 1] = P.start[q] + all.at(q, 2 + me);
    }
    const uint64_t recv = P.start[world];
    const int rc_recv = c->wide ? table_pull<u128>(c, P) : table_pull<uint64_t>(c, P);
    // 4. nobody may reuse its send buffer before every owner has pulled: one more exchange, which also checks the total
    mine[0] = recv;
    RFX_TRY(shard_exchange(c, rc_recv, 1, mine, all));
    const uint64_t received = all.sum(0);
    if (received != rows_global) return ctx_fail(c, RFX_E_STATE, "rfx_shard_table: %llu rows received, %llu sent", (unsigned long long)received, (unsigned long long)rows_global);
    c->ms[1] = stage_end(c);
    c->sh_rows_global = rows_global;
    c->n_rows = recv;
    c->table_cap = recv + 1;
    c->n_bins = B;
    c->have_counts = true;
    c->have_contigs = false; c->have_sorted = false;
    return RFX_OK;
}

}  // namespace rfx

using namespace rfx;

extern "C" {

int rfx_shard_init(rfx_ctx* c, int32_t rank, int32_t world, uint64_t arena_bytes) {
    if (!c || world < 1 || world > RFX_MAX_RANKS || rank < 0 || rank >= world) return c ? ctx_fail(c, RFX_E_INVALID, "rfx_shard_init: rank %d of %d (at most %d ranks)", rank, world, RFX_MAX_RANKS) : RFX_E_INVALID;
    if (c->arena) return ctx_fail(c, RFX_E_STATE, "rfx_shard_init: already initialised");
    cudaSetDevice(c->prm.device);
    if (!arena_bytes) {
        size_t fr = 0, tot = 0;
        RFX_CUDA(c, cudaMemGetInfo(&fr, &tot));
        arena_bytes = fr / 2;
    }
    arena_bytes = (arena_bytes + 4095) & ~(uint64_t)4095;
    if (arena_bytes < (1u << 20)) return ctx_fail(c, RFX_E_INVALID, "rfx_shard_init: arena of %llu bytes is too small", (unsigned long long)arena_bytes);
    RFX_CUDA(c, cudaStreamSynchronize(c->stream));
    // buffers allocated so far move into the arena when they are next reserved: start from a clean slate
    {
        DevBuf keep = c->dstat;
        c->dstat = DevBuf();
        rfx_reset(c);
        free_all_buffers(c);
        c->dstat = keep;
    }
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, arena_bytes);
    if (e != cudaSuccess) { cudaGetLastError(); return ctx_fail(c, RFX_E_NOMEM, "rfx_shard_init: cudaMalloc(%llu bytes) failed: %s", (unsigned long long)arena_bytes, cudaGetErrorString(e)); }
    RFX_CUDA(c, cudaMemset(p, 0, sizeof(ShardCtl)));
    RFX_CUDA(c, cudaHostAlloc(reinterpret_cast<void**>(&c->h_pub), (size_t)(RFX_MAX_RANKS + 1) * RFX_PUB_SLOTS * sizeof(unsigned long long), cudaHostAllocDefault));
    for (int i = 0; i < 2; i++) RFX_CUDA(c, cudaEventCreate(&c->ev_comm[i]));
    c->arena = (uint8_t*)p;
    c->arena_bytes = arena_bytes;
    c->arena_used = (sizeof(ShardCtl) + 255) & ~(size_t)255;
    c->d_pub = reinterpret_cast<unsigned long long*>(c->arena + c->arena_used);  // staging of everybody's published block
    c->arena_used += ((size_t)RFX_MAX_RANKS * RFX_PUB_SLOTS * sizeof(unsigned long long) + 255) & ~(size_t)255;
    c->arena_base = c->arena_used;
    c->sh_rank = rank; c->sh_world = world; c->sh_epoch = 0; c->sh_epoch2 = 0; c->sh_exchanges = 0;
    for (int r = 0; r < RFX_MAX_RANKS; r++) { c->peer_base[r] = nullptr; c->peer_ipc[r] = false; }
    return RFX_OK;
}

int rfx_shard_export(rfx_ctx* c, void* blob) {
    if (!c || !blob) return RFX_E_INVALID;
    if (!c->arena) return ctx_fail(c, RFX_E_STATE, "rfx_shard_export: call rfx_shard_init first");
    cudaSetDevice(c->prm.device);
    ShardBlob b;
    memset(&b, 0, sizeof(b));
    cudaIpcMemHandle_t h;
    RFX_CUDA(c, cudaIpcGetMemHandle(&h, c->arena));
    memcpy(b.handle, &h, sizeof(h));
    b.arena_bytes = c->arena_bytes;
    b.rank = c->sh_rank; b.device = c->prm.device;
    b.pid = (long long)getpid();
    b.ptr = (unsigned long long)c->arena;
    memcpy(blob, &b, sizeof(b));
    return RFX_OK;
}

int rfx_shard_connect(rfx_ctx* c, const void* blobs, int32_t world) {
    if (!c || !blobs) return RFX_E_INVALID;
    if (!c->arena || world != c->sh_world) return ctx_fail(c, RFX_E_STATE, "rfx_shard_connect: call rfx_shard_init with the same world size first");
    cudaSetDevice(c->prm.device);
    const ShardBlob* B = reinterpret_cast<const ShardBlob*>(blobs);
    for (int r = 0; r < world; r++) {
        if (B[r].rank != r) return ctx_fail(c, RFX_E_INVALID, "rfx_shard_connect: handle %d belongs to rank %d", r, B[r].rank);
        if (r == c->sh_rank) { c->peer_base[r] = c->arena; continue; }
        if (B[r].pid == (long long)getpid()) {
            // same process: the pointer itself; another device needs peer access switched on once
            if (B[r].device != c->prm.device) {
                int can = 0;
                RFX_CUDA(c, cudaDeviceCanAccessPeer(&can, c->prm.device, B[r].device));
                if (!can) return ctx_fail(c, RFX_E_CUDA, "device %d cannot access device %d", c->prm.device, B[r].device);
                cudaError_t e = cudaDeviceEnablePeerAccess(B[r].device, 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return ctx_fail(c, RFX_E_CUDA, "cudaDeviceEnablePeerAccess(%d): %s", B[r].device, cudaGetErrorString(e));
                cudaGetLastError();
            }
            c->peer_base[r] = reinterpret_cast<uint8_t*>(B[r].ptr);
        } else {
            cudaIpcMemHandle_t h;
            memcpy(&h, B[r].handle, sizeof(h));
            void* p = nullptr;
            cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
            if (e != cudaSuccess) return ctx_fail(c, RFX_E_CUDA, "cudaIpcOpenMemHandle(rank %d): %s", r, cudaGetErrorString(e));
            c->peer_base[r] = (uint8_t*)p;
            c->peer_ipc[r] = true;
        }
    }
    // all ranks in this process and two of them on one device: barriers on the host (see HostBarrier)
    bool one_process = true, shared_device = false;
    for (int r = 0; r < world; r++) {
        one_process = one_process && B[r].pid == (long long)getpid();
        for (int q = 0; q < r; q++) shared_device = shared_device || B[q].device == B[r].device;
    }
    if (one_process && shared_device && world > 1 && !c->hbar) {
        c->hbar_key = B[0].ptr;
        c->hbar = host_barrier_join(c->hbar_key, world);
    }
    return RFX_OK;
}

int rfx_shard_set_bins(rfx_ctx* c, uint32_t n_bins_total) {
    if (!c) return RFX_E_INVALID;
    if (c->sh_world < 1) return ctx_fail(c, RFX_E_STATE, "rfx_shard_set_bins: call rfx_shard_init first");
    if (n_bins_total % (uint32_t)c->sh_world) return ctx_fail(c, RFX_E_INVALID, "n_bins_total %u is not a multiple of %d ranks", n_bins_total, c->sh_world);
    c->sh_bins = n_bins_total;
    c->sh_bins_run = n_bins_total;  // the streamed scan of rfx_push_fastq uses it as well
    return RFX_OK;
}

int rfx_count_sharded(rfx_ctx* c) {
    if (!c) return RFX_E_INVALID;
    cudaSetDevice(c->prm.device);
    c->st_active = false;  // an open stitch stage is abandoned: its fragments refer to the contigs it was opened on
    return stage_count_sharded(c);
}

int rfx_shard_table(rfx_ctx* c) {
    if (!c) return RFX_E_INVALID;
    cudaSetDevice(c->prm.device);
    return stage_shard_table(c);
}

int rfx_assemble_sharded(rfx_ctx* c) {
    if (!c) return RFX_E_INVALID;
    cudaSetDevice(c->prm.device);
    c->st_active = false;  // an open stitch stage is abandoned: its fragments refer to the contigs it was opened on
    return stage_assemble_sharded(c);
}

int rfx_stitch_begin_sharded(rfx_ctx* c) {
    if (!c) return RFX_E_INVALID;
    cudaSetDevice(c->prm.device);
    return stage_stitch_begin_sharded(c);
}

int rfx_stitch_finish_sharded(rfx_ctx* c) {
    if (!c) return RFX_E_INVALID;
    cudaSetDevice(c->prm.device);
    return stage_stitch_finish_sharded(c);
}

int rfx_sort_kmers_sharded(rfx_ctx* c, int32_t min_error_coverage, double min_repeat_fold, int32_t max_kmer_size) {
    if (!c) return RFX_E_INVALID;
    cudaSetDevice(c->prm.device);
    c->st_active = false;  // an open stitch stage is abandoned, as in rfx_sort_kmers
    return stage_sorted_sharded(c, min_error_coverage, min_repeat_fold, max_kmer_size);
}

int rfx_device_count(int32_t* n_devices) {
    if (!n_devices) return RFX_E_INVALID;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); *n_devices = 0; return RFX_E_CUDA; }
    *n_devices = n;
    return RFX_OK;
}

int rfx_shard_stats(rfx_ctx* c, rfx_shard_stats_t* out) {
    if (!c || !out) return RFX_E_INVALID;
    memset(out, 0, sizeof(*out));
    out->rank = c->sh_rank; out->world = c->sh_world;
    out->arena_bytes = c->arena_bytes; out->arena_used = c->arena_used;
    out->n_instances_global = c->sh_inst_global;
    out->n_shard_instances = c->n_shard_instances;
    out->ms_comm = c->ms_comm;
    shard_graph_stats(c, out);
    return RFX_OK;
}

}  // extern "C"
