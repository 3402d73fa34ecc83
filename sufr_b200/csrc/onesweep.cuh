// The scatter kernel of the stable LSD radix sort of (key, value) pairs, 8-bit digits (driver: radix_sort.cuh).
//
// onesweep_kernel ranks the records of a tile (one vote per digit bit + a per-warp counter chain: stable), exchanges
// them through shared memory and writes digit-contiguous runs.  Every block owns a run of consecutive tiles and takes
// its write cursors from the exclusive scan of a [digit][block] count matrix, filled by a counting pass over the keys.
// The next tile arrives by TMA bulk copies (cp.async.bulk + mbarrier) while this one is processed: one elected thread
// issues two copies per tile instead of every thread issuing a dozen cp.async, which matters in a kernel bound by
// instruction issue.  The name is historical: a one-sweep variant (decoupled look-back over tile status words, the
// next digit counted on the way out) and other ways of staging a tile were measured on B200 with
// tools/ubench/sort_bench.cu and lost (profiles/r2_sort_bench_*.txt).  Per-pass time is 5.6 ms + 16 ns per tile at
// 2^30 records, so large tiles win; at that size the look-back saved less than its cost (8.5 ms against 7.7 + 1.3 ms
// with the counting pass), and on small tiles its chain serialises.  The count matrix is deterministic and has no
// spin-waits.  The removed variants are in the history up to commit 44af2d3.
//
// Algorithmic bytes per pass and element: 2 * (sizeof(K) + sizeof(V)) (+ sizeof(K) for the counting pass).
#pragma once
#include "common.cuh"

namespace sufr {
namespace osort {

constexpr int RADIX_BITS = 8;
constexpr int RADIX = 1 << RADIX_BITS;

// ------------------------------------------------------------------ TMA bulk copy global -> shared, mbarrier
__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t arrivals) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(arrivals) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_addr(dst)),
                 "l"(src), "r"(bytes), "r"(smem_addr(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "OSORT_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra OSORT_DONE;\n"
        "bra OSORT_WAIT;\n"
        "OSORT_DONE:\n"
        "}\n" ::"r"(smem_addr(bar)),
        "r"(parity)
        : "memory");
}
// generic-proxy accesses of shared memory (ld / st by threads) before, async-proxy accesses (bulk copy) after
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

template <typename K>
__device__ __forceinline__ uint32_t digit_of(K key, int shift, uint32_t dmask) {
    return (uint32_t)(key >> shift) & dmask;
}

// ------------------------------------------------------------------ one pass
template <typename K, typename V, int BLOCK, int IPT>
struct PassConfig {
    static constexpr int TILE = BLOCK * IPT;
    static constexpr int WARPS = BLOCK / 32;
    static constexpr size_t record = sizeof(K) + sizeof(V);
    static constexpr size_t dyn_smem = 2 * record * TILE;  // exchange buffer + staged next tile
};

// Every block owns `tiles_per_block` consecutive tiles and takes its starting offsets from a scanned [digit][block]
// count matrix `bases`.  Records are held in registers between the staging buffer and the exchange buffer.
template <typename K, typename V, int BLOCK, int IPT, int MINCTAS>
__global__ void __launch_bounds__(BLOCK, MINCTAS)
    onesweep_kernel(const K* __restrict__ kin, K* __restrict__ kout, const V* __restrict__ vin, V* __restrict__ vout,
                    uint64_t n, int shift, uint32_t dmask, const uint32_t* __restrict__ bases, uint32_t tiles_per_block) {
    using Cfg = PassConfig<K, V, BLOCK, IPT>;
    constexpr int TILE = Cfg::TILE, WARPS = Cfg::WARPS;
    static_assert(BLOCK >= RADIX && BLOCK % 32 == 0, "thread d owns digit d");
    static_assert(TILE <= 65535, "tile-local slots are 16-bit");
    __shared__ uint16_t wc[WARPS][RADIX];  // per-warp digit counters -> tile-local start of (warp, digit)
    __shared__ uint32_t goff[RADIX];       // global index = goff[d] + tile-local slot (mod 2^32)
    __shared__ uint32_t wtot[RADIX / 32];
    __shared__ uint32_t running[RADIX];    // global write cursor of each digit for this block
    __shared__ __align__(8) uint64_t bar;
    extern __shared__ __align__(128) unsigned char dyn[];
    K* exk = reinterpret_cast<K*>(dyn);
    V* exv = reinterpret_cast<V*>(dyn + sizeof(K) * TILE);
    K* pk = reinterpret_cast<K*>(dyn + Cfg::record * TILE);
    V* pv = reinterpret_cast<V*>(dyn + Cfg::record * TILE + sizeof(K) * TILE);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t lt_mask = (1u << lane) - 1u;
    const uint64_t total_tiles = (n + TILE - 1) / TILE;

    if (tid < RADIX) running[tid] = bases[(uint64_t)tid * gridDim.x + blockIdx.x];
    if (tid == 0) {
        mbar_init(&bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    auto issue = [&](uint64_t t) {  // one thread: stage tile t
        const uint64_t tb = t * TILE;
        const uint32_t cnt = (n - tb) < (uint64_t)TILE ? (uint32_t)(n - tb) : (uint32_t)TILE;
        const uint32_t kb = (cnt * (uint32_t)sizeof(K) + 15u) & ~15u, vb = (cnt * (uint32_t)sizeof(V) + 15u) & ~15u;
        fence_proxy_async();
        mbar_expect_tx(&bar, kb + vb);
        bulk_g2s(pk, kin + tb, kb, &bar);
        bulk_g2s(pv, vin + tb, vb, &bar);
    };

    uint64_t tile = (uint64_t)blockIdx.x * tiles_per_block;
    const uint64_t last_tile = tile + tiles_per_block < total_tiles ? tile + tiles_per_block : total_tiles;
    if (tile >= last_tile) tile = total_tiles;
    uint32_t parity = 0;
    if (tid == 0 && tile < total_tiles) issue(tile);
    while (tile < total_tiles) {
        const uint64_t tbase = tile * TILE;
        const uint32_t count = (n - tbase) < (uint64_t)TILE ? (uint32_t)(n - tbase) : (uint32_t)TILE;

        K key[IPT];
        V val[IPT];
        mbar_wait(&bar, parity);
        parity ^= 1u;
        if (count < (uint32_t)TILE) {  // block-uniform: padding records get the largest key
            for (uint32_t i = count + tid; i < (uint32_t)TILE; i += BLOCK) pk[i] = ~(K)0;
            __syncthreads();
        }
#pragma unroll
        for (int i = 0; i < IPT; i++) {
            const uint32_t idx = warp * (32 * IPT) + i * 32 + lane;
            key[i] = pk[idx];
            val[i] = pv[idx];
        }
        for (int i = tid; i < WARPS * RADIX / 2; i += BLOCK) reinterpret_cast<uint32_t*>(&wc[0][0])[i] = 0;
        __syncthreads();  // (A) counters zero, staged records copied to registers
        const uint64_t next = tile + 1 < last_tile ? tile + 1 : total_tiles;
        if (tid == 0 && next < total_tiles) issue(next);

        // ---- rank inside the warp's slice of the tile, rows in tile order => stable
        uint32_t dpack[(IPT + 3) / 4];   // digits, four per register
        uint32_t spack[(IPT + 1) / 2];   // tile-local ranks inside (warp, digit), two per register
#pragma unroll
        for (int i = 0; i < (IPT + 3) / 4; i++) dpack[i] = 0;
#pragma unroll
        for (int i = 0; i < (IPT + 1) / 2; i++) spack[i] = 0;
#pragma unroll
        for (int i = 0; i < IPT; i++) {
            const uint32_t d = digit_of(key[i], shift, dmask);
            unsigned peers = 0xffffffffu;
#pragma unroll
            for (int b = 0; b < RADIX_BITS; b++) {
                const bool bit = (d >> b) & 1u;
                const unsigned vote = __ballot_sync(0xffffffffu, bit);
                peers &= bit ? vote : ~vote;
            }
            const int leader = __ffs(peers) - 1;
            uint32_t old = 0;
            if (lane == leader) {
                old = wc[warp][d];
                wc[warp][d] = (uint16_t)(old + __popc(peers));
            }
            old = __shfl_sync(0xffffffffu, old, leader);
            const uint32_t slot = old + __popc(peers & lt_mask);
            dpack[i >> 2] |= d << (8 * (i & 3));
            spack[i >> 1] |= slot << (16 * (i & 1));
            __syncwarp();
        }
        __syncthreads();  // (B)

        // ---- thread d owns digit d: records per digit in the tile, tile-local starts
        uint32_t tile_count = 0, incl = 0;
        if (tid < RADIX) {
#pragma unroll
            for (int w = 0; w < WARPS; w++) {
                const uint32_t c = wc[w][tid];
                wc[w][tid] = (uint16_t)tile_count;
                tile_count += c;
            }
            incl = tile_count;
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                const uint32_t o = __shfl_up_sync(0xffffffffu, incl, off);
                if (lane >= off) incl += o;
            }
            if (lane == 31) wtot[warp] = incl;
        }
        __syncthreads();  // (C)
        uint32_t tile_start = 0, published = 0;
        if (tid < RADIX) {
            uint32_t wprefix = 0;
#pragma unroll
            for (int w = 0; w < RADIX / 32; w++)
                if (w < warp) wprefix += wtot[w];
            tile_start = wprefix + incl - tile_count;
#pragma unroll
            for (int w = 0; w < WARPS; w++) wc[w][tid] = (uint16_t)(wc[w][tid] + tile_start);
            // the padding of a partial tile was counted under the largest digit
            published = tile_count - ((uint32_t)tid == dmask ? (uint32_t)TILE - count : 0u);
        }
        __syncthreads();  // (D) tile-local starts final

        // ---- exchange through shared memory so that the global writes are digit-contiguous
#pragma unroll
        for (int i = 0; i < IPT; i++) {
            const uint32_t d = (dpack[i >> 2] >> (8 * (i & 3))) & 0xFFu;
            const uint32_t s = ((spack[i >> 1] >> (16 * (i & 1))) & 0xFFFFu) + wc[warp][d];
            exk[s] = key[i];
            exv[s] = val[i];
        }
        if (tid < RADIX) {
            goff[tid] = running[tid] - tile_start;
            running[tid] += published;
        }
        __syncthreads();  // (E) exchange buffer and offsets complete

        // ---- coalesced scatter
#pragma unroll
        for (int k = 0; k < IPT; k++) {
            const uint32_t s = k * BLOCK + tid;
            if (s < count) {
                const K kk = exk[s];
                const uint32_t dst = goff[digit_of(kk, shift, dmask)] + s;
                kout[dst] = kk;
                vout[dst] = exv[s];
            }
        }
        tile = next;
    }
}

}  // namespace osort
}  // namespace sufr
