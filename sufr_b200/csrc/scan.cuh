// Device-wide inclusive scan with functor input/output (reduce -> spine -> apply).
//
// Used for every order-preserving compaction on the path (active-group compaction, shard
// selection, suffix filter) and for the max scans of the refinement stages.
// Three launches, two coalesced reads of the input functor, no inter-block dependencies
// (so no forward-progress assumptions).  The operator must be associative; it need not commute.
#pragma once
#include <type_traits>
#include <utility>

#include "common.cuh"

namespace sufr {
namespace scan {

constexpr int BLOCK = 256;
constexpr int ITEMS = 16;
constexpr int CHUNK = BLOCK * ITEMS;

struct SumU32 {
    using T = uint32_t;
    __host__ __device__ static T identity() { return 0; }
    __device__ T operator()(T a, T b) const { return a + b; }
};
struct SumU64 {
    using T = unsigned long long;
    __host__ __device__ static T identity() { return 0; }
    __device__ T operator()(T a, T b) const { return a + b; }
};
struct MaxU32 {
    using T = uint32_t;
    __host__ __device__ static T identity() { return 0; }
    __device__ T operator()(T a, T b) const { return a > b ? a : b; }
};

// Input functors whose values are flags declare it, and the kernels scan them with warp votes instead of shuffles
// (two ballots and two popcounts per row of 32 against thirty-odd shuffle / add / select instructions):
//   static constexpr bool kFlags = true      SumU32: in(i) is 0 or 1;  SumU64: in(i) is 0 or 1 | (head << 32), the
//                                            compactions' "selected, and first of its group" pair
//   static constexpr bool kLastIndex = true  MaxU32: in(i) is i or 0 (the scan = index of the latest flagged element)
template <typename In, typename = void>
struct is_flags : std::false_type {};
template <typename In>
struct is_flags<In, std::enable_if_t<In::kFlags>> : std::true_type {};
template <typename In, typename = void>
struct is_last_index : std::false_type {};
template <typename In>
struct is_last_index<In, std::enable_if_t<In::kLastIndex>> : std::true_type {};

template <typename Op>
__device__ __forceinline__ typename Op::T warp_inclusive(typename Op::T v, Op op, int lane) {
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        typename Op::T o = __shfl_up_sync(0xffffffffu, v, off);
        if (lane >= off) v = op(o, v);
    }
    return v;
}

// Inclusive scan across the 256 threads of a block. `smem` holds 8 warp totals. Returns the block total
// through `total` (valid in every thread).
template <typename Op>
__device__ __forceinline__ typename Op::T block_inclusive(typename Op::T v, Op op, typename Op::T* smem,
                                                         typename Op::T& total) {
    using T = typename Op::T;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    T incl = warp_inclusive(v, op, lane);
    __syncthreads();  // protect smem reuse across calls
    if (lane == 31) smem[warp] = incl;
    __syncthreads();
    T prefix = Op::identity();
    T run = smem[0];
#pragma unroll
    for (int w = 1; w < BLOCK / 32; w++) {
        if (w == warp) prefix = run;
        run = op(run, smem[w]);
    }
    total = run;
    if (warp > 0) incl = op(prefix, incl);
    return incl;
}

// Layout of a chunk: warp w owns the 32 * ITEMS consecutive elements [w * 32 * ITEMS, ...), as ITEMS rows of 32; lane l
// reads element row * 32 + l, so every access the input / output functors make with consecutive indices is coalesced
// (a thread that owned ITEMS consecutive elements would stride its warp's loads by ITEMS elements).
// Scan order inside the warp is row-major: a warp scan per row, a running prefix over the rows.
template <typename Op>
__device__ __forceinline__ typename Op::T warp_reduce_in_order(typename Op::T v, Op op) {
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        typename Op::T o = __shfl_down_sync(0xffffffffu, v, off);
        v = op(v, o);  // lane 0 ends with e0 (+) e1 (+) ... (+) e31; the other lanes are not used
    }
    return v;
}

template <typename Op, typename In>
__global__ void __launch_bounds__(BLOCK) reduce_kernel(uint64_t n, In in, Op op, typename Op::T* partials) {
    using T = typename Op::T;
    __shared__ T smem[BLOCK / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t w0 = (uint64_t)blockIdx.x * CHUNK + (uint64_t)warp * (32 * ITEMS) + lane;
    T v[ITEMS];
#pragma unroll
    for (int k = 0; k < ITEMS; k++) {
        const uint64_t i = w0 + (uint64_t)k * 32;
        v[k] = i < n ? in(i) : Op::identity();
    }
    T acc = Op::identity();
    if constexpr (is_flags<In>::value) {
        uint32_t c0 = 0, c1 = 0;
#pragma unroll
        for (int k = 0; k < ITEMS; k++) {
            c0 += __popc(__ballot_sync(0xffffffffu, (uint32_t)v[k] & 1u));
            if constexpr (sizeof(T) == 8) c1 += __popc(__ballot_sync(0xffffffffu, (uint32_t)((unsigned long long)v[k] >> 32) & 1u));
        }
        if constexpr (sizeof(T) == 8) acc = (T)(c0 | ((unsigned long long)c1 << 32));
        else acc = (T)c0;
    } else if constexpr (is_last_index<In>::value) {
        uint32_t last = 0;
#pragma unroll
        for (int k = 0; k < ITEMS; k++) {
            const uint32_t hb = __ballot_sync(0xffffffffu, v[k] != 0);
            if (hb) last = (uint32_t)(w0 - lane) + k * 32 + (31 - __clz((int)hb));
        }
        acc = (T)last;
    } else {
#pragma unroll
        for (int k = 0; k < ITEMS; k++) acc = op(acc, warp_reduce_in_order(v[k], op));  // meaningful in lane 0
    }
    if (lane == 0) smem[warp] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        T total = smem[0];
#pragma unroll
        for (int w = 1; w < BLOCK / 32; w++) total = op(total, smem[w]);
        partials[blockIdx.x] = total;
    }
}

// Single block: exclusive scan of the per-chunk partials, in place. `total_out` receives the grand total.
template <typename Op>
__global__ void __launch_bounds__(BLOCK) spine_kernel(uint32_t nblocks, Op op, typename Op::T* partials,
                                                      typename Op::T* total_out) {
    using T = typename Op::T;
    __shared__ T smem[BLOCK / 32];
    T carry = Op::identity();
    for (uint32_t base = 0; base < nblocks; base += BLOCK) {
        uint32_t i = base + threadIdx.x;
        T v = i < nblocks ? partials[i] : Op::identity();
        T total;
        T incl = block_inclusive(v, op, smem, total);
        // exclusive = carry (+) inclusive of the previous thread
        T prev = __shfl_up_sync(0xffffffffu, incl, 1);
        __shared__ T last_of_warp[BLOCK / 32];
        __syncthreads();
        if ((threadIdx.x & 31) == 31) last_of_warp[threadIdx.x >> 5] = incl;
        __syncthreads();
        T excl;
        if (threadIdx.x == 0) excl = Op::identity();
        else if ((threadIdx.x & 31) == 0) excl = last_of_warp[(threadIdx.x >> 5) - 1];
        else excl = prev;
        if (i < nblocks) partials[i] = op(carry, excl);
        carry = op(carry, total);
    }
    if (threadIdx.x == 0 && total_out) *total_out = carry;
}

// out(i, v, inclusive) is called for every i < n; for sum scans exclusive = inclusive - v.
// An output functor that reads memory should split itself into `Staged load(i, v, inclusive)` and `store(i, v, inclusive, staged)`:
// a load inside out() sits between the stores of the rows before and after it, so the sixteen rows of a thread would
// wait for sixteen memory round trips one after the other; with the split all loads are in flight before the first store.
template <typename Out, typename T, typename = void>
struct has_staged_load : std::false_type {};
template <typename Out, typename T>
struct has_staged_load<Out, T, std::void_t<decltype(std::declval<const Out&>().load(uint64_t(0), std::declval<T>(), std::declval<T>()))>>
    : std::true_type {};

// An output functor that keeps per-block state (a shared-memory histogram, say) declares
// `static constexpr bool kBlockHooks = true` and gets `begin()` before the block's first load and `finish()` after its
// last store; both are called by every thread of the block, and finish() may synchronise the block.
template <typename Out, typename = void>
struct has_block_hooks : std::false_type {};
template <typename Out>
struct has_block_hooks<Out, std::enable_if_t<Out::kBlockHooks>> : std::true_type {};

// the last phase of apply_kernel: row k of the warp, value v, inclusive scan value incl
template <typename Out, typename T, typename Rows>
__device__ __forceinline__ void emit_rows(const Out& out, uint64_t n, uint64_t w0, const Rows& rows) {
    if constexpr (has_staged_load<Out, T>::value) {
        decltype(out.load(uint64_t(0), T(), T())) staged[ITEMS];
#pragma unroll
        for (int k = 0; k < ITEMS; k++) {
            const uint64_t i = w0 + (uint64_t)k * 32;
            if (i < n) staged[k] = out.load(i, rows.value(k), rows.inclusive(k));
        }
#pragma unroll
        for (int k = 0; k < ITEMS; k++) {
            const uint64_t i = w0 + (uint64_t)k * 32;
            if (i < n) out.store(i, rows.value(k), rows.inclusive(k), staged[k]);
        }
    } else {
#pragma unroll
        for (int k = 0; k < ITEMS; k++) {
            const uint64_t i = w0 + (uint64_t)k * 32;
            if (i < n) out(i, rows.value(k), rows.inclusive(k));
        }
    }
}

template <typename Op, typename In, typename Out>
__global__ void __launch_bounds__(BLOCK) apply_kernel(uint64_t n, In in, Op op, const typename Op::T* partials,
                                                      Out out) {
    using T = typename Op::T;
    __shared__ T smem[BLOCK / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t w0 = (uint64_t)blockIdx.x * CHUNK + (uint64_t)warp * (32 * ITEMS) + lane;
    if constexpr (has_block_hooks<Out>::value) out.begin();
    if constexpr (is_flags<In>::value) {
        // ---- flags: votes.  b0 / b1 = the row's ballots of bit 0 / bit 32; counts before a row are warp-uniform.
        constexpr bool kPair = sizeof(T) == 8;
        struct Rows {
            uint32_t b0[ITEMS], b1[kPair ? ITEMS : 1], pre0[ITEMS], pre1[kPair ? ITEMS : 1];
            uint32_t lane, le;
            __device__ T value(int k) const {
                if constexpr (kPair) return (T)(((b0[k] >> lane) & 1u) | ((unsigned long long)((b1[k] >> lane) & 1u) << 32));
                else return (T)((b0[k] >> lane) & 1u);
            }
            __device__ T inclusive(int k) const {
                const uint32_t c0 = pre0[k] + __popc(b0[k] & le);
                if constexpr (kPair) return (T)(c0 | ((unsigned long long)(pre1[k] + __popc(b1[k] & le)) << 32));
                else return (T)c0;
            }
        } rows;
        rows.lane = lane;
        rows.le = 0xffffffffu >> (31 - lane);
#pragma unroll
        for (int k = 0; k < ITEMS; k++) {
            const uint64_t i = w0 + (uint64_t)k * 32;
            const T v = i < n ? in(i) : T(0);
            rows.b0[k] = __ballot_sync(0xffffffffu, (uint32_t)v & 1u);
            if constexpr (kPair) rows.b1[k] = __ballot_sync(0xffffffffu, (uint32_t)((unsigned long long)v >> 32) & 1u);
        }
        uint32_t c0 = 0, c1 = 0;
#pragma unroll
        for (int k = 0; k < ITEMS; k++) {
            rows.pre0[k] = c0;
            c0 += __popc(rows.b0[k]);
            if constexpr (kPair) { rows.pre1[k] = c1; c1 += __popc(rows.b1[k]); }
        }
        if (lane == 0) smem[warp] = kPair ? (T)(c0 | ((unsigned long long)c1 << 32)) : (T)c0;
        __syncthreads();
        T prefix = partials[blockIdx.x];
#pragma unroll
        for (int w = 0; w < BLOCK / 32; w++)
            if (w < warp) prefix += smem[w];
#pragma unroll
        for (int k = 0; k < ITEMS; k++) {
            rows.pre0[k] += (uint32_t)prefix;
            if constexpr (kPair) rows.pre1[k] += (uint32_t)((unsigned long long)prefix >> 32);
        }
        emit_rows<Out, T>(out, n, w0, rows);
    } else if constexpr (is_last_index<In>::value) {
        // ---- index of the latest flagged element: the highest set bit of the row's ballot at or below the lane
        struct Rows {
            uint32_t hb[ITEMS], carry[ITEMS];  // carry = latest flagged index before the row
            uint32_t lane, le, base;
            __device__ T value(int k) const { return ((hb[k] >> lane) & 1u) ? base + k * 32 + lane : 0u; }
            __device__ T inclusive(int k) const {
                const uint32_t m = hb[k] & le;
                return m ? base + k * 32 + (31 - __clz((int)m)) : carry[k];
            }
        } rows;
        rows.lane = lane;
        rows.le = 0xffffffffu >> (31 - lane);
        rows.base = (uint32_t)(w0 - lane);
        uint32_t last = 0;
#pragma unroll
        for (int k = 0; k < ITEMS; k++) {
            const uint64_t i = w0 + (uint64_t)k * 32;
            rows.hb[k] = __ballot_sync(0xffffffffu, i < n && in(i) != 0);
            rows.carry[k] = last;
            if (rows.hb[k]) last = rows.base + k * 32 + (31 - __clz((int)rows.hb[k]));
        }
        if (lane == 0) smem[warp] = last;
        __syncthreads();
        T prefix = partials[blockIdx.x];
#pragma unroll
        for (int w = 0; w < BLOCK / 32; w++)
            if (w < warp) prefix = op(prefix, smem[w]);
#pragma unroll
        for (int k = 0; k < ITEMS; k++) rows.carry[k] = op(prefix, rows.carry[k]);
        emit_rows<Out, T>(out, n, w0, rows);
    } else {
        struct Rows {
            T v[ITEMS], s[ITEMS];
            __device__ T value(int k) const { return v[k]; }
            __device__ T inclusive(int k) const { return s[k]; }
        } rows;
#pragma unroll
        for (int k = 0; k < ITEMS; k++) {
            const uint64_t i = w0 + (uint64_t)k * 32;
            rows.v[k] = i < n ? in(i) : Op::identity();
        }
#pragma unroll
        for (int k = 0; k < ITEMS; k++) rows.s[k] = warp_inclusive(rows.v[k], op, lane);
        // running prefix over the rows of this warp (the row totals are warp-uniform)
        T wtotal = Op::identity();
#pragma unroll
        for (int k = 0; k < ITEMS; k++) {
            const T row = __shfl_sync(0xffffffffu, rows.s[k], 31);
            rows.s[k] = op(wtotal, rows.s[k]);
            wtotal = op(wtotal, row);
        }
        if (lane == 0) smem[warp] = wtotal;
        __syncthreads();
        T prefix = partials[blockIdx.x];
#pragma unroll
        for (int w = 0; w < BLOCK / 32; w++)
            if (w < warp) prefix = op(prefix, smem[w]);
#pragma unroll
        for (int k = 0; k < ITEMS; k++) rows.s[k] = op(prefix, rows.s[k]);
        emit_rows<Out, T>(out, n, w0, rows);
    }
    if constexpr (has_block_hooks<Out>::value) out.finish();
}

inline size_t partials_count(uint64_t n) { return (size_t)div_up(n, CHUNK) + 1; }
// Where a scan_reduce or inclusive_scan over n elements leaves its grand total in `partials`.
template <typename T>
inline T* total_ptr(T* partials, uint64_t n) { return partials + div_up(n, CHUNK); }

// Two-step form: scan_reduce leaves the exclusive chunk prefixes in `partials` (and the grand total in its last
// element) so that the caller can size its outputs before scan_apply runs the second pass.
template <typename Op, typename In>
void scan_reduce(uint64_t n, In in, Op op, typename Op::T* partials, cudaStream_t stream) {
    if (n == 0) {
        typename Op::T id = Op::identity();
        SUFR_CUDA_CHECK(cudaMemcpyAsync(partials, &id, sizeof(id), cudaMemcpyHostToDevice, stream));
        return;
    }
    uint32_t nblocks = div_up_u32(n, CHUNK);
    reduce_kernel<Op, In><<<nblocks, BLOCK, 0, stream>>>(n, in, op, partials);
    SUFR_KERNEL_CHECK();
    spine_kernel<Op><<<1, BLOCK, 0, stream>>>(nblocks, op, partials, partials + nblocks);
    SUFR_KERNEL_CHECK();
}
template <typename Op, typename In, typename Out>
void scan_apply(uint64_t n, In in, Op op, Out out, const typename Op::T* partials, cudaStream_t stream) {
    if (n == 0) return;
    uint32_t nblocks = div_up_u32(n, CHUNK);
    apply_kernel<Op, In, Out><<<nblocks, BLOCK, 0, stream>>>(n, in, op, partials, out);
    SUFR_KERNEL_CHECK();
}

// `partials` must hold partials_count(n) elements; the last one receives the grand total.
template <typename Op, typename In, typename Out>
void inclusive_scan(uint64_t n, In in, Op op, Out out, typename Op::T* partials, cudaStream_t stream) {
    if (n == 0) {
        typename Op::T id = Op::identity();
        SUFR_CUDA_CHECK(cudaMemcpyAsync(partials, &id, sizeof(id), cudaMemcpyHostToDevice, stream));
        return;
    }
    uint32_t nblocks = div_up_u32(n, CHUNK);
    reduce_kernel<Op, In><<<nblocks, BLOCK, 0, stream>>>(n, in, op, partials);
    SUFR_KERNEL_CHECK();
    spine_kernel<Op><<<1, BLOCK, 0, stream>>>(nblocks, op, partials, partials + nblocks);
    SUFR_KERNEL_CHECK();
    apply_kernel<Op, In, Out><<<nblocks, BLOCK, 0, stream>>>(n, in, op, partials, out);
    SUFR_KERNEL_CHECK();
}

}  // namespace scan
}  // namespace sufr
