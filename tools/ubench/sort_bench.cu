// Micro-benchmark of the radix-sort pass: the round-1 kernel (upsweep + scan + downsweep per digit) against
// block shapes of the count-matrix scatter kernel (sufr_b200/csrc/onesweep.cuh), on random (u64 key, u32 value)
// records, digits = key bits [32, 56) -- the three passes the fast path runs after the pass fused into key generation.
// Also checks every shape against the round-1 result (both are stable sorts: identical output) and, on a small input
// with a partial tile, skewed digits and a narrow last digit, against std::stable_sort.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo --expt-relaxed-constexpr \
//             -o tools/ubench/sort_bench tools/ubench/sort_bench.cu
// Run:   tools/ubench/sort_bench [records = 2^30]
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <vector>

#include "../../sufr_b200/csrc/onesweep.cuh"
#include "../../sufr_b200/csrc/radix_sort.cuh"
#include "radix_sort_r1.cuh"

using namespace sufr;

#define CK(x)                                                                                  \
    do {                                                                                       \
        cudaError_t e_ = (x);                                                                  \
        if (e_ != cudaSuccess) {                                                               \
            printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__);    \
            exit(1);                                                                           \
        }                                                                                      \
    } while (0)

__device__ __host__ inline uint64_t mix64(uint64_t z) {
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
__global__ void init_kernel(uint64_t* k, uint32_t* v, uint64_t n, int skew) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t z = mix64((i + 1) * 0x9E3779B97F4A7C15ull);
        if (skew == 1) z &= 0x0303FF0FFFFFFFFFull;  // few distinct digits
        if (skew >= 2) {  // every sorted digit takes one of (1 << (skew - 2)) values: 2 -> all records in one bin
            const uint64_t keep = (1ull << (skew - 2)) - 1;
            z &= ~0x00FFFFFF00000000ull | (keep << 32) | (keep << 40) | (keep << 48);
        }
        k[i] = z;
        v[i] = (uint32_t)i;
    }
}
__global__ void diff_kernel(const uint64_t* a, const uint64_t* b, const uint32_t* va, const uint32_t* vb, uint64_t n,
                            unsigned long long* bad) {
    unsigned long long c = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
        c += (a[i] != b[i] || va[i] != vb[i]) ? 1 : 0;
    if (c) atomicAdd(bad, c);
}

struct Bufs {
    uint64_t *ka, *kb, *kref;
    uint32_t *va, *vb, *vref;
    unsigned long long* bad;
    uint32_t* counts;
    uint64_t n;
};

static float elapsed(cudaEvent_t a, cudaEvent_t b) {
    float t;
    CK(cudaEventElapsedTime(&t, a, b));
    return t;
}

// counting pass + scan + the scatter kernel, every block owning a run of consecutive tiles
template <int BLOCK, int IPT, int CTAS>
void run_matrix(const char* name, Bufs& B, int begin_bit, int end_bit) {
    using Cfg = osort::PassConfig<uint64_t, uint32_t, BLOCK, IPT>;
    cudaFuncAttributes fa{};
    auto kern = osort::onesweep_kernel<uint64_t, uint32_t, BLOCK, IPT, CTAS>;
    CK(cudaFuncGetAttributes(&fa, kern));
    CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::dyn_smem));
    int occ = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, BLOCK, Cfg::dyn_smem));
    const int passes = (end_bit - begin_bit + 7) / 8;
    const uint64_t tiles = (B.n + Cfg::TILE - 1) / Cfg::TILE;
    uint32_t grid = 148 * CTAS;
    const uint32_t tpb = (uint32_t)((tiles + grid - 1) / grid);
    grid = (uint32_t)((tiles + tpb - 1) / tpb);
    float best_total = 1e30f, best_pass[8] = {}, best_up[8] = {};
    cudaEvent_t ev[20];
    for (auto& e : ev) CK(cudaEventCreate(&e));
    for (int rep = 0; rep < 3; rep++) {
        init_kernel<<<148 * 8, 256>>>(B.ka, B.va, B.n, 0);
        CK(cudaDeviceSynchronize());
        CK(cudaEventRecord(ev[0]));
        bool in_b = false;
        for (int p = 0; p < passes; p++) {
            const int bit = begin_bit + 8 * p, nb = std::min(8, end_bit - bit);
            const uint64_t* kin = in_b ? B.kb : B.ka;
            rsort_r1::upsweep_kernel<uint64_t, Cfg::TILE / 256><<<grid, 256>>>(kin, B.n, bit, (1u << nb) - 1u, B.counts, tpb);
            rsort_r1::scan_counts_kernel<<<1, 1024>>>(B.counts, 256u * grid);
            CK(cudaEventRecord(ev[1 + 2 * p]));
            kern<<<grid, BLOCK, Cfg::dyn_smem>>>(kin, in_b ? B.ka : B.kb, in_b ? B.vb : B.va, in_b ? B.va : B.vb, B.n, bit,
                                                 (1u << nb) - 1u, B.counts, tpb);
            CK(cudaEventRecord(ev[2 + 2 * p]));
            in_b = !in_b;
        }
        CK(cudaDeviceSynchronize());
        CK(cudaGetLastError());
        float tot = elapsed(ev[0], ev[2 * passes]);
        if (tot < best_total) {
            best_total = tot;
            for (int p = 0; p < passes; p++) {
                best_up[p] = elapsed(ev[2 * p], ev[1 + 2 * p]);
                best_pass[p] = elapsed(ev[1 + 2 * p], ev[2 + 2 * p]);
            }
        }
        if (rep == 0) {
            CK(cudaMemset(B.bad, 0, 8));
            diff_kernel<<<148 * 8, 256>>>(in_b ? B.kb : B.ka, B.kref, in_b ? B.vb : B.va, B.vref, B.n, B.bad);
            unsigned long long bad = 0;
            CK(cudaMemcpy(&bad, B.bad, 8, cudaMemcpyDeviceToHost));
            if (bad) printf("  !! %s: %llu records differ from the round-1 sort\n", name, bad);
        }
    }
    printf("%-30s MATRIX regs %3d smem %6zu occ %d | count+scan %6.3f | passes", name, fa.numRegs,
           Cfg::dyn_smem + fa.sharedSizeBytes, occ, best_up[passes - 1]);
    for (int p = 0; p < passes; p++) printf(" %7.3f", best_pass[p]);
    printf(" | total %7.3f ms | last pass %6.0f GB/s\n", best_total, (double)B.n * 24 / (best_pass[passes - 1] * 1e-3) / 1e9);
    for (auto& e : ev) cudaEventDestroy(e);
    fflush(stdout);
}

// How much of the scatter pass is the DRAM locality of its writes?  The same kernel on keys whose digits take 1, 4, 16,
// 64 or 256 values: the instruction count per record is the same, only the length of the per-digit output runs changes.
template <int BLOCK, int IPT, int CTAS>
void run_locality(Bufs& B) {
    using Cfg = osort::PassConfig<uint64_t, uint32_t, BLOCK, IPT>;
    auto kern = osort::onesweep_kernel<uint64_t, uint32_t, BLOCK, IPT, CTAS>;
    CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::dyn_smem));
    const uint64_t tiles = (B.n + Cfg::TILE - 1) / Cfg::TILE;
    uint32_t grid = 148 * CTAS;
    const uint32_t tpb = (uint32_t)((tiles + grid - 1) / grid);
    grid = (uint32_t)((tiles + tpb - 1) / tpb);
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    for (int bits : {0, 2, 4, 6, 8}) {
        float best = 1e30f;
        for (int rep = 0; rep < 3; rep++) {
            init_kernel<<<148 * 8, 256>>>(B.ka, B.va, B.n, bits == 8 ? 0 : 2 + bits);
            rsort_r1::upsweep_kernel<uint64_t, Cfg::TILE / 256><<<grid, 256>>>(B.ka, B.n, 32, 255u, B.counts, tpb);
            rsort_r1::scan_counts_kernel<<<1, 1024>>>(B.counts, 256u * grid);
            CK(cudaDeviceSynchronize());
            CK(cudaEventRecord(e0));
            kern<<<grid, BLOCK, Cfg::dyn_smem>>>(B.ka, B.kb, B.va, B.vb, B.n, 32, 255u, B.counts, tpb);
            CK(cudaEventRecord(e1));
            CK(cudaDeviceSynchronize());
            CK(cudaGetLastError());
            best = std::min(best, elapsed(e0, e1));
        }
        printf("locality <%d,%d,%d>: %3d distinct digits -> scatter pass %7.3f ms  %6.0f GB/s\n", BLOCK, IPT, CTAS, 1 << bits, best,
               (double)B.n * 24 / (best * 1e-3) / 1e9);
    }
    fflush(stdout);
}

// The same launches as run_matrix on a small input, against std::stable_sort
template <int BLOCK, int IPT, int CTAS>
bool small_check(const char* name, int skew) {
    using Cfg = osort::PassConfig<uint64_t, uint32_t, BLOCK, IPT>;
    auto kern = osort::onesweep_kernel<uint64_t, uint32_t, BLOCK, IPT, CTAS>;
    CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::dyn_smem));
    const uint64_t n = 1000003;  // partial last tile
    const uint64_t tiles = (n + Cfg::TILE - 1) / Cfg::TILE;
    uint32_t grid = 148 * CTAS;
    const uint32_t tpb = (uint32_t)((tiles + grid - 1) / grid);
    grid = (uint32_t)((tiles + tpb - 1) / tpb);
    uint64_t *ka, *kb;
    uint32_t *va, *vb, *counts;
    CK(cudaMalloc(&ka, n * 8 + 64));
    CK(cudaMalloc(&kb, n * 8 + 64));
    CK(cudaMalloc(&va, n * 4 + 64));
    CK(cudaMalloc(&vb, n * 4 + 64));
    CK(cudaMalloc(&counts, 256u * grid * 4));
    init_kernel<<<148, 256>>>(ka, va, n, skew);
    std::vector<uint64_t> hk(n);
    CK(cudaMemcpy(hk.data(), ka, n * 8, cudaMemcpyDeviceToHost));
    bool ok = true;
    for (int variant = 0; variant < 2 && ok; variant++) {
        const int begin_bit = variant ? 35 : 32, end_bit = variant ? 64 : 56;  // variant 1: narrow last digit
        const uint64_t mask = (end_bit == 64 ? ~0ull : ((1ull << end_bit) - 1)) & ~((1ull << begin_bit) - 1);
        std::vector<uint32_t> order(n);
        std::iota(order.begin(), order.end(), 0u);
        std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return (hk[a] & mask) < (hk[b] & mask); });
        init_kernel<<<148, 256>>>(ka, va, n, skew);
        const int passes = (end_bit - begin_bit + 7) / 8;
        bool in_b = false;
        for (int p = 0; p < passes; p++) {
            const int bit = begin_bit + 8 * p, nb = std::min(8, end_bit - bit);
            const uint64_t* kin = in_b ? kb : ka;
            rsort_r1::upsweep_kernel<uint64_t, Cfg::TILE / 256><<<grid, 256>>>(kin, n, bit, (1u << nb) - 1u, counts, tpb);
            rsort_r1::scan_counts_kernel<<<1, 1024>>>(counts, 256u * grid);
            kern<<<grid, BLOCK, Cfg::dyn_smem>>>(kin, in_b ? ka : kb, in_b ? vb : va, in_b ? va : vb, n, bit, (1u << nb) - 1u,
                                                 counts, tpb);
            in_b = !in_b;
        }
        CK(cudaDeviceSynchronize());
        CK(cudaGetLastError());
        std::vector<uint32_t> hv(n);
        std::vector<uint64_t> hks(n);
        CK(cudaMemcpy(hv.data(), in_b ? vb : va, n * 4, cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(hks.data(), in_b ? kb : ka, n * 8, cudaMemcpyDeviceToHost));
        uint64_t bad = 0;
        for (uint64_t i = 0; i < n; i++) bad += (hv[i] != order[i] || hks[i] != hk[order[i]]) ? 1 : 0;
        if (bad) {
            printf("  !! small check %s skew %d bits [%d,%d): %llu of %llu records wrong\n", name, skew, begin_bit, end_bit,
                   (unsigned long long)bad, (unsigned long long)n);
            ok = false;
        }
    }
    cudaFree(ka); cudaFree(kb); cudaFree(va); cudaFree(vb); cudaFree(counts);
    return ok;
}

// a shape's benchmark row is printed only when its small checks pass
#define MAT(B_, I_, C_)                                                                      \
    do {                                                                                     \
        const char* nm = "<" #B_ "," #I_ "," #C_ ">";                                        \
        if (small_check<B_, I_, C_>(nm, 0) && small_check<B_, I_, C_>(nm, 1))                \
            run_matrix<B_, I_, C_>(nm, B, 32, 56);                                           \
        else                                                                                 \
            failed++;                                                                        \
    } while (0)

int main(int argc, char** argv) {
    Bufs B{};
    B.n = argc > 1 ? strtoull(argv[1], nullptr, 10) : (1ull << 30);
    const uint64_t n = B.n;
    cudaDeviceProp prop{};
    CK(cudaGetDeviceProperties(&prop, 0));
    printf("%s, %d SMs, %llu records of (u64, u32), digits = key bits [32, 56)\n", prop.name, prop.multiProcessorCount,
           (unsigned long long)n);
    CK(cudaMalloc(&B.ka, n * 8 + 64));
    CK(cudaMalloc(&B.kb, n * 8 + 64));
    CK(cudaMalloc(&B.kref, n * 8 + 64));
    CK(cudaMalloc(&B.va, n * 4 + 64));
    CK(cudaMalloc(&B.vb, n * 4 + 64));
    CK(cudaMalloc(&B.vref, n * 4 + 64));
    CK(cudaMalloc(&B.bad, 8));
    CK(cudaMalloc(&B.counts, 256 * 148 * 16 * 4));

    // round-1 sort: upsweep + scan + downsweep per digit
    {
        float best = 1e30f;
        cudaEvent_t e0, e1;
        CK(cudaEventCreate(&e0));
        CK(cudaEventCreate(&e1));
        bool in_b = false;
        for (int rep = 0; rep < 3; rep++) {
            init_kernel<<<148 * 8, 256>>>(B.ka, B.va, n, 0);
            CK(cudaDeviceSynchronize());
            CK(cudaEventRecord(e0));
            in_b = rsort_r1::sort_pairs<uint64_t, uint32_t>(B.ka, B.kb, B.va, B.vb, n, 32, 56, B.counts, 0);
            CK(cudaEventRecord(e1));
            CK(cudaDeviceSynchronize());
            best = std::min(best, elapsed(e0, e1));
        }
        CK(cudaMemcpy(B.kref, in_b ? B.kb : B.ka, n * 8, cudaMemcpyDeviceToDevice));
        CK(cudaMemcpy(B.vref, in_b ? B.vb : B.va, n * 4, cudaMemcpyDeviceToDevice));
        printf("%-34s 3 x (upsweep + scan + downsweep)                       | total %7.3f ms | %6.0f GB/s per pass incl. upsweep\n",
               "round-1 rsort::sort_pairs", best, (double)n * 24 * 3 / (best * 1e-3) / 1e9);
        fflush(stdout);
    }

    {   // the sort the build uses: count + scan + scatter per digit (radix_sort.cuh)
        float best = 1e30f;
        cudaEvent_t e0, e1;
        CK(cudaEventCreate(&e0));
        CK(cudaEventCreate(&e1));
        bool in_b = false;
        for (int rep = 0; rep < 3; rep++) {
            init_kernel<<<148 * 8, 256>>>(B.ka, B.va, n, 0);
            CK(cudaDeviceSynchronize());
            CK(cudaEventRecord(e0));
            in_b = rsort::sort_pairs<uint64_t, uint32_t>(B.ka, B.kb, B.va, B.vb, n, 32, 56, B.counts, 0);
            CK(cudaEventRecord(e1));
            CK(cudaDeviceSynchronize());
            best = std::min(best, elapsed(e0, e1));
        }
        CK(cudaMemset(B.bad, 0, 8));
        diff_kernel<<<148 * 8, 256>>>(in_b ? B.kb : B.ka, B.kref, in_b ? B.vb : B.va, B.vref, n, B.bad);
        unsigned long long bad = 0;
        CK(cudaMemcpy(&bad, B.bad, 8, cudaMemcpyDeviceToHost));
        printf("%-34s 3 x (count + scan + scatter), 512 threads x 16, 1 CTA/SM     | total %7.3f ms | %6.0f GB/s per pass incl. count%s\n",
               "round-2 rsort::sort_pairs", best, (double)n * 24 * 3 / (best * 1e-3) / 1e9, bad ? "  !! DIFFERS" : "");
        fflush(stdout);
    }
    if (getenv("SORT_BENCH_LOCALITY")) {
        run_locality<512, 16, 1>(B);
        run_locality<256, 16, 2>(B);
        return 0;
    }
    int failed = 0;
    MAT(256, 16, 2);
    MAT(512, 8, 2);
    MAT(512, 16, 1);
    MAT(1024, 8, 1);
    MAT(256, 8, 4);
    printf("small checks against std::stable_sort: %s\n", failed ? "FAILED" : "all shapes pass");
    return failed ? 1 : 0;
}
