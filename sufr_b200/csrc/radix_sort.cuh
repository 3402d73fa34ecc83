// Hand-written stable LSD radix sort of (key, value) pairs, 8-bit digits.
//
// Per pass:  count    (digit histogram of the run of tiles each scatter block owns -> [digit][block] matrix;
//                      several counting blocks per scatter block, merged with global atomics)
//            scan     (exclusive scan of the matrix, digit-major)
//            scatter  (osort::onesweep_kernel, onesweep.cuh: per tile warp-level vote ranking -> block digit
//                      offsets -> shared-memory exchange -> coalesced scatter of keys, then values;
//                      the next tile arrives by a TMA bulk copy while this one is processed)
// One persistent scatter block of 512 threads per SM, tiles of 8192 records: every block owns a contiguous run of
// tiles, so the only global state is the 256 x G count matrix (no inter-block dependencies, no look-back spinning).
// Tile size and block shape were chosen from tools/ubench/sort_bench.cu on B200 (profiles/r2_sort_bench_*.txt):
// per-pass time is 5.6 ms + 16 ns per tile at 2^30 records, so the largest tile that fits two buffers in 227 KB of
// shared memory wins.
//
// Algorithmic bytes per pass and element: sizeof(K) (count read) + 2*(sizeof(K)+sizeof(V)) (scatter read + write).
#pragma once
#include <algorithm>
#include <utility>
#include <vector>

#include "common.cuh"
#include "onesweep.cuh"

namespace sufr {
namespace rsort {

constexpr int RADIX_BITS = osort::RADIX_BITS;
constexpr int RADIX = osort::RADIX;

template <typename K, typename V>
struct Tuning {
    static constexpr int BLOCK = 512;
    static constexpr int IPT = (sizeof(K) + sizeof(V) > 12) ? 12 : 16;  // two tile buffers within 227 KB
    static constexpr int CTAS = 1;
    static constexpr int TILE = BLOCK * IPT;
};


// counts[d * owners + o] += records with digit d in sub-range `sub` of owner o's run of records
template <typename K>
__global__ void __launch_bounds__(256) count_kernel(const K* __restrict__ keys, uint64_t n, int shift, uint32_t dmask,
                                                    uint32_t* __restrict__ counts, uint64_t owner_records,
                                                    uint32_t owners, uint32_t subs, uint64_t sub_records) {
    constexpr int WARPS = 8;
    __shared__ uint32_t hist[WARPS][RADIX];
    for (int i = threadIdx.x; i < WARPS * RADIX; i += 256) (&hist[0][0])[i] = 0;
    __syncthreads();
    const int warp = threadIdx.x >> 5;
    const uint32_t owner = blockIdx.x / subs, sub = blockIdx.x % subs;
    uint64_t obeg = (uint64_t)owner * owner_records, oend = obeg + owner_records;
    if (oend > n) oend = n;
    uint64_t begin = obeg + (uint64_t)sub * sub_records, end = begin + sub_records;
    if (end > oend) end = oend;
    for (uint64_t i0 = begin + threadIdx.x; i0 < end; i0 += 256 * 4) {
        K k[4];
#pragma unroll
        for (int u = 0; u < 4; u++) k[u] = i0 + 256 * u < end ? keys[i0 + 256 * u] : (K)0;  // four loads in flight
#pragma unroll
        for (int u = 0; u < 4; u++)
            if (i0 + 256 * u < end) atomicAdd(&hist[warp][osort::digit_of(k[u], shift, dmask)], 1u);
    }
    __syncthreads();
    uint32_t acc = 0;
#pragma unroll
    for (int w = 0; w < WARPS; w++) acc += hist[w][threadIdx.x];
    if (acc) atomicAdd(&counts[(uint64_t)threadIdx.x * owners + owner], acc);
}

// Exclusive scan of `len` u32 counts in place (single block).
__global__ void __launch_bounds__(1024) scan_counts_kernel(uint32_t* counts, uint32_t len) {
    __shared__ uint32_t warp_tot[32];
    __shared__ uint32_t carry_s;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (uint32_t base = 0; base < len; base += 1024) {
        uint32_t i = base + threadIdx.x;
        uint32_t v = i < len ? counts[i] : 0;
        uint32_t incl = v;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            uint32_t o = __shfl_up_sync(0xffffffffu, incl, off);
            if (lane >= off) incl += o;
        }
        if (lane == 31) warp_tot[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            uint32_t t = warp_tot[lane];
            uint32_t ti = t;
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                uint32_t o = __shfl_up_sync(0xffffffffu, ti, off);
                if (lane >= off) ti += o;
            }
            warp_tot[lane] = ti - t;  // exclusive warp prefix
        }
        __syncthreads();
        uint32_t carry = carry_s;
        uint32_t excl = carry + warp_tot[warp] + incl - v;
        if (i < len) counts[i] = excl;
        __syncthreads();
        if (threadIdx.x == 1023) carry_s = excl + v;
        __syncthreads();
    }
}

struct Plan {
    uint32_t grid = 0;             // scatter blocks (= owners of the count matrix)
    uint32_t tiles_per_block = 0;
    uint32_t subs = 1;             // counting blocks per scatter block
    uint64_t sub_records = 0;
};

template <typename K, typename V>
inline Plan make_plan(uint64_t n) {
    using T = Tuning<K, V>;
    const uint64_t tiles = div_up(n ? n : 1, T::TILE);
    const uint64_t max_grid = (uint64_t)num_sms() * T::CTAS;
    Plan p;
    p.grid = (uint32_t)std::min<uint64_t>(tiles, max_grid);
    p.tiles_per_block = (uint32_t)div_up(tiles, p.grid);
    p.grid = (uint32_t)div_up(tiles, p.tiles_per_block);
    const uint64_t owner_records = (uint64_t)p.tiles_per_block * T::TILE;
    // about eight counting blocks per SM, each with at least 4096 records
    uint64_t subs = std::max<uint64_t>(1, (uint64_t)num_sms() * 8 / p.grid);
    subs = std::min<uint64_t>(subs, std::max<uint64_t>(1, owner_records / 4096));
    p.subs = (uint32_t)subs;
    p.sub_records = div_up(owner_records, subs);
    return p;
}

inline size_t counts_words() { return (size_t)RADIX * std::max(num_sms(), kNumSMs) * 4; }

// Sorts on key bits [begin_bit, end_bit).  Buffers ping-pong; returns true when the sorted data ended
// up in (keys_b, vals_b).  `counts` needs counts_words() u32.  `launches` (optional) is incremented
// by the number of kernels launched.  With `first_counts_ready` the caller has filled (and scanned) the
// count matrix of the first pass itself, for the plan make_plan<K, V>(n) returns.
using EventPairs = std::vector<std::pair<cudaEvent_t, cudaEvent_t>>;

template <typename K, typename V>
bool sort_pairs(K* keys_a, K* keys_b, V* vals_a, V* vals_b, uint64_t n, int begin_bit, int end_bit,
                uint32_t* counts, cudaStream_t stream, uint64_t* launches = nullptr,
                EventPairs* scatter_events = nullptr) {
    using T = Tuning<K, V>;
    using Cfg = osort::PassConfig<K, V, T::BLOCK, T::IPT>;
    if (n == 0 || end_bit <= begin_bit) return false;
    if (n > 0xFFFFFFFFull) throw Error(3, "rsort: more than 2^32 records need 64-bit write cursors");
    const Plan p = make_plan<K, V>(n);
    auto kern = osort::onesweep_kernel<K, V, T::BLOCK, T::IPT, T::CTAS>;
    static bool attr_set[64] = {};  // per instantiation and device
    allow_dynamic_smem(kern, Cfg::dyn_smem, attr_set);
    const uint64_t owner_records = (uint64_t)p.tiles_per_block * T::TILE;
    bool in_b = false;
    for (int bit = begin_bit; bit < end_bit; bit += RADIX_BITS) {
        const int nb = end_bit - bit < RADIX_BITS ? end_bit - bit : RADIX_BITS;
        const uint32_t dmask = (1u << nb) - 1u;
        K* kin = in_b ? keys_b : keys_a;
        K* kout = in_b ? keys_a : keys_b;
        V* vin = in_b ? vals_b : vals_a;
        V* vout = in_b ? vals_a : vals_b;
        SUFR_CUDA_CHECK(cudaMemsetAsync(counts, 0, (size_t)RADIX * p.grid * sizeof(uint32_t), stream));
        count_kernel<K><<<p.grid * p.subs, 256, 0, stream>>>(kin, n, bit, dmask, counts, owner_records, p.grid, p.subs,
                                                             p.sub_records);
        SUFR_KERNEL_CHECK();
        scan_counts_kernel<<<1, 1024, 0, stream>>>(counts, (uint32_t)RADIX * p.grid);
        SUFR_KERNEL_CHECK();
        cudaEvent_t e0 = nullptr, e1 = nullptr;
        if (scatter_events) {
            SUFR_CUDA_CHECK(cudaEventCreate(&e0));
            SUFR_CUDA_CHECK(cudaEventCreate(&e1));
            SUFR_CUDA_CHECK(cudaEventRecord(e0, stream));
        }
        kern<<<p.grid, T::BLOCK, Cfg::dyn_smem, stream>>>(kin, kout, vin, vout, n, bit, dmask, counts, p.tiles_per_block);
        SUFR_KERNEL_CHECK();
        if (scatter_events) {
            SUFR_CUDA_CHECK(cudaEventRecord(e1, stream));
            scatter_events->push_back({e0, e1});
        }
        if (launches) *launches += 3;
        in_b = !in_b;
    }
    return in_b;
}

}  // namespace rsort
}  // namespace sufr
