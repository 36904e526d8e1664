// rfx_scan.cuh -- order-preserving transform-scan over an index range, hand-written (no CUB).
//
//   prefix(i) = in(0) (+) in(1) (+) ... (+) in(i-1)          (+) = any associative Op, not
//   out(i, prefix(i), in(i))                                   necessarily commutative
//
// Three phases: (A) one aggregate per tile, (B) exclusive scan of the aggregates (recursive),
// (C) re-read the tile, combine with the tile prefix, hand each element to `out`.
// `prepare()` runs A+B and returns the grand total, so callers can size outputs before `apply()`.
// Elements are laid out warp-striped: a warp owns 32*ITEMS consecutive elements and walks them 32 at
// a time, so global loads made by `in` are coalesced and the scan order is the index order.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace rfx {

constexpr int SCAN_WARPS = 8;
constexpr int SCAN_ITEMS = 8;
constexpr int SCAN_TILE = SCAN_WARPS * 32 * SCAN_ITEMS;  // 2048 elements per block

// shuffles for the element types we scan
__device__ __forceinline__ uint32_t shfl_up_any(uint32_t v, int d) { return __shfl_up_sync(0xffffffffu, v, d); }
__device__ __forceinline__ uint64_t shfl_up_any(uint64_t v, int d) { return __shfl_up_sync(0xffffffffu, v, d); }
__device__ __forceinline__ uint32_t shfl_idx_any(uint32_t v, int l) { return __shfl_sync(0xffffffffu, v, l); }
__device__ __forceinline__ uint64_t shfl_idx_any(uint64_t v, int l) { return __shfl_sync(0xffffffffu, v, l); }

struct U64x3 {
    uint64_t a, b, c;
};
__device__ __forceinline__ U64x3 shfl_up_any(U64x3 v, int d) {
    U64x3 r;
    r.a = __shfl_up_sync(0xffffffffu, v.a, d); r.b = __shfl_up_sync(0xffffffffu, v.b, d); r.c = __shfl_up_sync(0xffffffffu, v.c, d);
    return r;
}
__device__ __forceinline__ U64x3 shfl_idx_any(U64x3 v, int l) {
    U64x3 r;
    r.a = __shfl_sync(0xffffffffu, v.a, l); r.b = __shfl_sync(0xffffffffu, v.b, l); r.c = __shfl_sync(0xffffffffu, v.c, l);
    return r;
}

struct OpAddU64 {
    __device__ __forceinline__ uint64_t operator()(uint64_t x, uint64_t y) const { return x + y; }
};
struct OpAddU64x3 {
    __device__ __forceinline__ U64x3 operator()(U64x3 x, U64x3 y) const { return U64x3{x.a + y.a, x.b + y.b, x.c + y.c}; }
};

template <class T, class Op> __device__ __forceinline__ T warp_scan_incl(T v, Op op, int lane) {
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        T o = shfl_up_any(v, d);
        if (lane >= d) v = op(o, v);
    }
    return v;
}

// Phase A: agg[block] = fold of the block's tile.  live (optional): the element count as the device knows it, n is then
// an upper bound and the tiles behind it are empty.
template <class T, class Op, class In>
__global__ void __launch_bounds__(SCAN_WARPS * 32) scan_agg_kernel(uint64_t n, const unsigned long long* live, In in, Op op, T ident, T* __restrict__ agg) {
    if (live && *live < n) n = *live;
    if ((uint64_t)blockIdx.x * SCAN_TILE >= n) {
        if (threadIdx.x == 0) agg[blockIdx.x] = ident;
        return;
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint64_t base = (uint64_t)blockIdx.x * SCAN_TILE + (uint64_t)warp * 32 * SCAN_ITEMS;
    T acc = ident;
#pragma unroll
    for (int it = 0; it < SCAN_ITEMS; it++) {
        const uint64_t i = base + (uint64_t)it * 32 + lane;
        T v = i < n ? in(i) : ident;
        T s = warp_scan_incl(v, op, lane);
        acc = op(acc, shfl_idx_any(s, 31));
    }
    __shared__ T wagg[SCAN_WARPS];
    if (lane == 0) wagg[warp] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        T a = wagg[0];
        for (int w = 1; w < SCAN_WARPS; w++) a = op(a, wagg[w]);
        agg[blockIdx.x] = a;
    }
}

// Phase C: out(i, exclusive prefix, value)
template <class T, class Op, class In, class Out>
__global__ void __launch_bounds__(SCAN_WARPS * 32)
    scan_apply_kernel(uint64_t n, const unsigned long long* live, In in, Out out, Op op, T ident, const T* __restrict__ tile_prefix) {
    if (live && *live < n) n = *live;
    if ((uint64_t)blockIdx.x * SCAN_TILE >= n) return;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint64_t base = (uint64_t)blockIdx.x * SCAN_TILE + (uint64_t)warp * 32 * SCAN_ITEMS;
    T v[SCAN_ITEMS], s[SCAN_ITEMS];
    T acc = ident;
#pragma unroll
    for (int it = 0; it < SCAN_ITEMS; it++) {
        const uint64_t i = base + (uint64_t)it * 32 + lane;
        v[it] = i < n ? in(i) : ident;
        s[it] = warp_scan_incl(v[it], op, lane);
        acc = op(acc, shfl_idx_any(s[it], 31));
    }
    __shared__ T wagg[SCAN_WARPS];
    if (lane == 0) wagg[warp] = acc;
    __syncthreads();
    T carry = tile_prefix ? tile_prefix[blockIdx.x] : ident;
    for (int w = 0; w < warp; w++) carry = op(carry, wagg[w]);
#pragma unroll
    for (int it = 0; it < SCAN_ITEMS; it++) {
        const uint64_t i = base + (uint64_t)it * 32 + lane;
        T prev = shfl_up_any(s[it], 1);
        T excl = lane == 0 ? carry : op(carry, prev);
        if (i < n) out(i, excl, v[it]);
        carry = op(carry, shfl_idx_any(s[it], 31));
    }
}

template <class T> struct ScanInArray {
    const T* p;
    __device__ __forceinline__ T operator()(uint64_t i) const { return p[i]; }
};
template <class T> struct ScanOutArray {
    T* p;
    __device__ __forceinline__ void operator()(uint64_t i, T excl, T) const { p[i] = excl; }
};

// Workspace: level l holds ceil(n / TILE^(l+1)) aggregates, scanned in place into exclusive prefixes.
template <class T> struct ScanPlan {
    uint64_t n = 0;
    int levels = 0;
    uint64_t count[6] = {0};
    T* agg[6] = {nullptr};
    T* total = nullptr;  // device, 1 element
    // element count on the device, when the host does not know it yet: n (from bind) is then an upper bound
    const unsigned long long* live = nullptr;
    static size_t workspace_elems(uint64_t n) {
        size_t tot = 1;
        uint64_t c = n;
        while (c > 1) { c = (c + SCAN_TILE - 1) / SCAN_TILE; tot += c; if (c == 1) break; }
        return tot + 8;
    }
    void bind(uint64_t n_, T* ws) {
        n = n_; levels = 0; live = nullptr;
        uint64_t c = n;
        T* p = ws;
        total = p; p += 1;
        do {
            c = (c + SCAN_TILE - 1) / SCAN_TILE;
            if (c == 0) c = 1;
            count[levels] = c; agg[levels] = p; p += c; levels++;
        } while (c > 1 && levels < 6);
    }
};

template <class T> __global__ void scan_copy_total_kernel(const T* src, T* dst) { *dst = *src; }

// Phases A + B.  After this, plan.agg[0][b] is the exclusive prefix of tile b and *plan.total the grand total.
template <class T, class Op, class In>
void scan_prepare(ScanPlan<T>& plan, In in, Op op, T ident, cudaStream_t st) {
    if (plan.n == 0) { cudaMemsetAsync(plan.total, 0, sizeof(T), st); return; }
    scan_agg_kernel<T, Op, In><<<(unsigned)plan.count[0], SCAN_WARPS * 32, 0, st>>>(plan.n, plan.live, in, op, ident, plan.agg[0]);
    for (int l = 1; l < plan.levels; l++) {
        ScanInArray<T> src{plan.agg[l - 1]};
        scan_agg_kernel<T, Op, ScanInArray<T>><<<(unsigned)plan.count[l], SCAN_WARPS * 32, 0, st>>>(plan.count[l - 1], nullptr, src, op, ident, plan.agg[l]);
    }
    // top level has exactly one aggregate = the grand total
    scan_copy_total_kernel<T><<<1, 1, 0, st>>>(plan.agg[plan.levels - 1], plan.total);
    // walk down: turn each level's aggregates into exclusive prefixes, in place
    for (int l = plan.levels - 1; l >= 1; l--) {
        ScanInArray<T> src{plan.agg[l - 1]};
        ScanOutArray<T> dst{plan.agg[l - 1]};
        const T* pre = (l == plan.levels - 1) ? nullptr : plan.agg[l];
        scan_apply_kernel<T, Op, ScanInArray<T>, ScanOutArray<T>>
            <<<(unsigned)plan.count[l], SCAN_WARPS * 32, 0, st>>>(plan.count[l - 1], nullptr, src, dst, op, ident, pre);
    }
}

// Phase C over the original elements.
template <class T, class Op, class In, class Out>
void scan_apply(ScanPlan<T>& plan, In in, Out out, Op op, T ident, cudaStream_t st) {
    if (plan.n == 0) return;
    const T* pre = plan.levels == 1 ? nullptr : plan.agg[0];
    // with a single level there is one tile and its prefix is the identity
    if (plan.levels >= 1 && plan.count[0] > 1) pre = plan.agg[0];
    scan_apply_kernel<T, Op, In, Out><<<(unsigned)plan.count[0], SCAN_WARPS * 32, 0, st>>>(plan.n, plan.live, in, out, op, ident, pre);
}

}  // namespace rfx
