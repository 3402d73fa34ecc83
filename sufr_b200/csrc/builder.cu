// Build pipeline + the build side of the C ABI of libsufr_b200.so (the read side is index.cu).
//
// Replaces SufrBuilder::<T>::new up to write() (libsufr/src/sufr_builder.rs:143-217) on one B200:
//
//   encode   transform_kernel, pack_kernel            text transform, dense alphabet, packed text
//   keys     keygen_kernel (or shard compaction)      first key word of every suffix
//   sort     rsort::{upsweep,scan,downsweep}          stable LSD radix sort of (key word, position)
//   refine   resolve / active compaction / segmented  groups of equal key words: next key word, then
//            sort rounds, then prefix doubling        (full sort only) prefix doubling on ranks
//   lcp      resolve_kernel, lcp_complete_kernel      LCP from clz(x ^ y) of adjacent key words
//   finish   N-run tie rule, suffix filter, widen     sufr_builder.rs:305-307, :446-449
//
// The oracle (oracle/) is never linked or called from here.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstdlib>
#include <cstring>
#include <exception>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/sufr_b200.h"
#include "common.cuh"
#include "context.hpp"
#include "host_io.hpp"
#include "kernels.cuh"
#include "keys.cuh"
#include "pool.hpp"
#include "radix_sort.cuh"
#include "scan.cuh"
#include "stream_io.hpp"
#include "verify.cuh"

namespace sufr {

thread_local std::string g_last_error;

struct EventTimer {
    cudaStream_t stream;
    std::vector<cudaEvent_t> ev;
    explicit EventTimer(cudaStream_t s) : stream(s) {}
    ~EventTimer() {
        for (auto e : ev) cudaEventDestroy(e);
    }
    int mark() {
        cudaEvent_t e;
        SUFR_CUDA_CHECK(cudaEventCreate(&e));
        SUFR_CUDA_CHECK(cudaEventRecord(e, stream));
        ev.push_back(e);
        return (int)ev.size() - 1;
    }
    double ms(int a, int b) {
        float t = 0;
        SUFR_CUDA_CHECK(cudaEventElapsedTime(&t, ev[a], ev[b]));
        return t;
    }
};

// Thrown when prefix doubling is needed but this attempt sorts only a subset of the positions (suffix
// filter applied up front, or one key-range shard): the build is redone over all positions.
struct NeedFullSort {};

// Host side of the compact device->host transfer: widen a staged array into the result with a few threads.
// The destination is written once and not read back, so the AVX2 path uses streaming (non-temporal) stores:
// no read-for-ownership traffic on the host memory bus, which the incoming DMA writes share.
}  // namespace sufr
#include <immintrin.h>
namespace sufr {

template <typename Src, typename Dst>
static void widen_range_scalar(const Src* src, Dst* dst, uint64_t lo, uint64_t hi) {
    for (uint64_t i = lo; i < hi; i++) dst[i] = (Dst)src[i];
}
__attribute__((target("avx2"))) static void widen_range_avx2(const uint8_t* src, uint64_t* dst, uint64_t lo, uint64_t hi) {
    uint64_t i = lo;
    for (; i < hi && ((uintptr_t)(dst + i) & 31); i++) dst[i] = src[i];
    for (; i + 16 <= hi; i += 16) {
        __m128i b = _mm_loadu_si128((const __m128i*)(src + i));
        _mm256_stream_si256((__m256i*)(dst + i), _mm256_cvtepu8_epi64(b));
        _mm256_stream_si256((__m256i*)(dst + i + 4), _mm256_cvtepu8_epi64(_mm_srli_si128(b, 4)));
        _mm256_stream_si256((__m256i*)(dst + i + 8), _mm256_cvtepu8_epi64(_mm_srli_si128(b, 8)));
        _mm256_stream_si256((__m256i*)(dst + i + 12), _mm256_cvtepu8_epi64(_mm_srli_si128(b, 12)));
    }
    for (; i < hi; i++) dst[i] = src[i];
    _mm_sfence();
}
__attribute__((target("avx2"))) static void widen_range_avx2(const uint8_t* src, uint32_t* dst, uint64_t lo, uint64_t hi) {
    uint64_t i = lo;
    for (; i < hi && ((uintptr_t)(dst + i) & 31); i++) dst[i] = src[i];
    for (; i + 16 <= hi; i += 16) {
        __m128i b = _mm_loadu_si128((const __m128i*)(src + i));
        _mm256_stream_si256((__m256i*)(dst + i), _mm256_cvtepu8_epi32(b));
        _mm256_stream_si256((__m256i*)(dst + i + 8), _mm256_cvtepu8_epi32(_mm_srli_si128(b, 8)));
    }
    for (; i < hi; i++) dst[i] = src[i];
    _mm_sfence();
}
__attribute__((target("avx2"))) static void widen_range_avx2(const uint32_t* src, uint64_t* dst, uint64_t lo, uint64_t hi) {
    uint64_t i = lo;
    for (; i < hi && ((uintptr_t)(dst + i) & 31); i++) dst[i] = src[i];
    for (; i + 8 <= hi; i += 8) {
        __m256i a = _mm256_loadu_si256((const __m256i*)(src + i));
        _mm256_stream_si256((__m256i*)(dst + i), _mm256_cvtepu32_epi64(_mm256_castsi256_si128(a)));
        _mm256_stream_si256((__m256i*)(dst + i + 4), _mm256_cvtepu32_epi64(_mm256_extracti128_si256(a, 1)));
    }
    for (; i < hi; i++) dst[i] = src[i];
    _mm_sfence();
}

template <typename Src, typename Dst>
static void host_widen(const Src* src, Dst* dst, uint64_t count, int threads) {
    if (threads < 1) threads = 1;
    static const bool avx2 = __builtin_cpu_supports("avx2");
    std::vector<std::thread> pool;
    for (int t = 0; t < threads; t++) {
        pool.emplace_back([=]() {
            uint64_t lo = count * (uint64_t)t / threads, hi = count * (uint64_t)(t + 1) / threads;
            if (avx2) widen_range_avx2(src, dst, lo, hi);
            else widen_range_scalar(src, dst, lo, hi);
        });
    }
    for (auto& th : pool) th.join();
}

// ---------------------------------------------------------------------------------------------
// Position-dependent kernels and the build pipeline, once per position width (suffix_array.rs:460-470).
namespace p32 {
using pos_t = uint32_t;
#include "pos_kernels.inl"
#include "build_impl.inl"
}  // namespace p32
namespace p64 {
using pos_t = uint64_t;
#include "pos_kernels.inl"
#include "build_impl.inl"
}  // namespace p64

// the radix sort for the read side (approx.cuh): the instance the 32-bit build already uses, so no new kernel
bool sort_u64_u32_pairs(uint64_t* keys_a, uint64_t* keys_b, uint32_t* vals_a, uint32_t* vals_b, uint64_t n, int end_bit,
                        uint32_t* counts, cudaStream_t stream) {
    return rsort::sort_pairs<uint64_t, uint32_t>(keys_a, keys_b, vals_a, vals_b, n, 0, end_bit, counts, stream);
}
size_t sort_counts_words() { return rsort::counts_words(); }

// texts of u32::MAX bytes and more need 64-bit positions; SUFR_B200_DEBUG_POS64 forces them (tests)
static void run_build(Ctx& ctx, const SufrB200Args& args, uint32_t index_bits, int text_memory, int result_memory,
                      SufrB200Result* out) {
    if (args.text_len >= 0xFFFFFFFFull || getenv("SUFR_B200_DEBUG_POS64")) {
        p64::Build b(ctx, args, index_bits, text_memory, result_memory);
        b.run(out);
    } else {
        p32::Build b(ctx, args, index_bits, text_memory, result_memory);
        b.run(out);
    }
}
void free_owner(ResultOwner* o) {
    if (!o) return;
    if (o->memory == SUFR_B200_MEM_DEVICE) {
        if (o->ctx) {
            std::lock_guard<std::mutex> lock(o->ctx->mu);
            if (o->text) o->ctx->pool.free(o->text);
            if (o->sa) o->ctx->pool.free(o->sa);
            if (o->lcp) o->ctx->pool.free(o->lcp);
        }
    } else if (o->ctx) {
        std::lock_guard<std::mutex> lock(o->ctx->mu);
        if (o->text) o->ctx->pinned.put(o->text);
        if (o->sa) o->ctx->pinned.put(o->sa);
        if (o->lcp) o->ctx->pinned.put(o->lcp);
    } else {
        if (o->text && o->text_malloc) free(o->text);
        else if (o->text) cudaFreeHost(o->text);
        if (o->sa) cudaFreeHost(o->sa);
        if (o->lcp) cudaFreeHost(o->lcp);
    }
    free(o->n_ranges);
    delete o;
}

Ctx* make_ctx(int device) {
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        cudaGetLastError();
        throw Error(SUFR_B200_ERR_CUDA, "no CUDA device available: the sufr_b200 build path has no CPU fallback");
    }
    if (device < 0 || device >= count) throw Error(SUFR_B200_ERR_ARGUMENT, "invalid CUDA device ordinal");
    SUFR_CUDA_CHECK(cudaSetDevice(device));
    auto c = std::make_unique<Ctx>();
    c->device = device;
    SUFR_CUDA_CHECK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    return c.release();
}

void release_ctx(Ctx& ctx) {
    cudaStreamSynchronize(ctx.stream);
    ctx.pinned.release();
    ctx.pool.release_all();
    cudaStreamDestroy(ctx.stream);
}

// The host result of sufr_b200_create / _create_multi (what SufrBuilder holds after `new`): the counts of the device
// result `dev`, the transformed text the writer returned (malloc, owned by the result from here on) and a copy of the
// N runs.  The suffix and LCP arrays are in the file only, like the reference's builder struct (sufr_builder.rs:38-89).
static void host_result(const SufrB200Result& dev, uint8_t* host_text, SufrB200Result* res) {
    auto owner = std::make_unique<ResultOwner>();
    owner->memory = SUFR_B200_MEM_HOST;
    owner->text = host_text;
    owner->text_malloc = true;
    if (dev.num_n_ranges) {
        owner->n_ranges = (uint64_t*)malloc(dev.num_n_ranges * 16);
        memcpy(owner->n_ranges, dev.n_ranges, dev.num_n_ranges * 16);
    }
    *res = dev;
    res->memory = SUFR_B200_MEM_HOST;
    res->text = host_text;
    res->sa = nullptr;
    res->lcp = nullptr;
    res->n_ranges = owner->n_ranges;
    res->owner = owner.release();
}
}  // namespace sufr

using namespace sufr;

extern "C" {

int sufr_b200_abi_version(void) { return SUFR_B200_ABI_VERSION; }

const char* sufr_b200_last_error(void) { return g_last_error.c_str(); }

int sufr_b200_device_count(void) {
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return count;
}

int sufr_b200_ctx_create(int device, SufrB200Ctx** out) {
    return guarded([&] {
        if (!out) throw Error(SUFR_B200_ERR_ARGUMENT, "out is NULL");
        *out = reinterpret_cast<SufrB200Ctx*>(make_ctx(device));
    });
}

void sufr_b200_ctx_destroy(SufrB200Ctx* c) {
    if (!c) return;
    Ctx* ctx = reinterpret_cast<Ctx*>(c);
    cudaSetDevice(ctx->device);
    release_ctx(*ctx);
    delete ctx;
}

int sufr_b200_ctx_reserve(SufrB200Ctx* c, uint64_t text_len, uint32_t index_bits) {
    return guarded([&] {
        Ctx* ctx = reinterpret_cast<Ctx*>(c);
        if (!ctx) throw Error(SUFR_B200_ERR_ARGUMENT, "ctx is NULL");
        CtxLock lock(*ctx);
        uint64_t per = 32;
        (void)index_bits;
        ctx->pool.reserve((size_t)(per * text_len + (64ull << 20)));
    });
}

void sufr_b200_ctx_trim(SufrB200Ctx* c) {
    Ctx* ctx = reinterpret_cast<Ctx*>(c);
    if (!ctx) return;
    // not CtxLock: this call reports no error
    std::lock_guard<std::mutex> lock(ctx->mu);
    cudaSetDevice(ctx->device);
    ctx->pool.trim();
    ctx->pinned.release();
}

int sufr_b200_build(SufrB200Ctx* c, const SufrB200Args* args, uint32_t index_bits, int text_memory, int result_memory,
                    SufrB200Result* out) {
    return guarded([&] {
        Ctx* ctx = reinterpret_cast<Ctx*>(c);
        if (!ctx || !args || !out) throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
        if (args->text_len && !args->text) throw Error(SUFR_B200_ERR_ARGUMENT, "text is NULL");
        std::lock_guard<std::mutex> lock(ctx->mu);
        try {
            run_build(*ctx, *args, index_bits, text_memory, result_memory, out);
        } catch (...) {
            cudaStreamSynchronize(ctx->stream);
            throw;
        }
    });
}

void sufr_b200_result_free(SufrB200Ctx*, SufrB200Result* r) {
    if (!r) return;
    free_owner(static_cast<ResultOwner*>(r->owner));
    memset(r, 0, sizeof(*r));
}

int sufr_b200_patch_seam(SufrB200Ctx* c, const SufrB200Args* args, SufrB200Result* r, uint64_t prev_last_suffix) {
    return guarded([&] {
        Ctx* ctx = reinterpret_cast<Ctx*>(c);
        if (!ctx || !args || !r) throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
        if (r->num_suffixes == 0) return;
        // The seam needs the text only: recompute the pair LCP on the host from the transformed text
        // when the result is on the host, on the device otherwise.
        SeedMaskInfo mask;
        bool has_mask = args->seed_mask && parse_seed_mask(args->seed_mask, mask);
        uint64_t q = (!has_mask && args->has_max_query_len) ? args->max_query_len : 0;
        CtxLock lock(*ctx);
        const uint64_t a = prev_last_suffix, b = r->first_suffix, n = r->text_len;
        if (a >= n || b >= n) throw Error(SUFR_B200_ERR_ARGUMENT, "suffix out of range");
        uint64_t l = 0;
        // Windows of the two suffixes in TRANSFORMED form, from wherever the text is at hand: the host result,
        // the device result, or (host results of ranks > 0 carry no text) the caller's raw text + the transform.
        auto fetch = [&](uint64_t p, uint64_t len, uint8_t* dst) {
            if (r->text && r->memory == SUFR_B200_MEM_HOST) {
                memcpy(dst, r->text + p, len);
            } else if (r->text) {
                SUFR_CUDA_CHECK(cudaMemcpyAsync(dst, r->text + p, len, cudaMemcpyDeviceToHost, ctx->stream));
                SUFR_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
            } else {
                // raw text of the caller (host or device memory, as it was passed to the build) + the transform
                if (!args->text) throw Error(SUFR_B200_ERR_ARGUMENT, "patch_seam needs the text (result or args)");
                cudaPointerAttributes attr{};
                bool on_device = cudaPointerGetAttributes(&attr, args->text) == cudaSuccess &&
                                 (attr.type == cudaMemoryTypeDevice || attr.type == cudaMemoryTypeManaged);
                cudaGetLastError();
                if (on_device) {
                    SUFR_CUDA_CHECK(cudaMemcpyAsync(dst, args->text + p, len, cudaMemcpyDeviceToHost, ctx->stream));
                    SUFR_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
                } else {
                    memcpy(dst, args->text + p, len);
                }
                for (uint64_t i = 0; i < len; i++) {  // sufr_builder.rs:149-156
                    uint8_t c = dst[i];
                    if (c >= 97 && c <= 122) c = args->ignore_softmask ? (uint8_t)'N' : (uint8_t)(c & 0x5F);
                    dst[i] = c;
                }
            }
        };
        auto in_run = [&](uint64_t p, uint64_t& end) {
            uint64_t lo = 0, hi = r->num_n_ranges;
            while (lo < hi) {
                uint64_t mid = (lo + hi) / 2;
                if (r->n_ranges[2 * mid] <= p && p < r->n_ranges[2 * mid + 1]) { end = r->n_ranges[2 * mid + 1]; return true; }
                if (r->n_ranges[2 * mid] < p) lo = mid + 1; else hi = mid;
            }
            return false;
        };
        uint64_t ea = 0, eb = 0;
        if (!has_mask && r->num_n_ranges && in_run(a, ea) && in_run(b, eb)) {
            l = std::min(ea - a, eb - b);  // sufr_builder.rs:305-307
        } else {
            // the two suffixes come from different key ranges, so they differ within the first few symbols;
            // the window grows if they do not
            uint64_t win = has_mask ? mask.bytes.size() + 64 : 4096;
            while (true) {
                uint64_t la = std::min(win, n - a), lb = std::min(win, n - b);
                std::vector<uint8_t> buf(la + lb);
                fetch(a, la, buf.data());
                fetch(b, lb, buf.data() + la);
                if (has_mask) {
                    l = 0;
                    for (uint64_t k = 0; k < mask.positions.size(); k++) {
                        uint64_t o = mask.positions[k];
                        if (a + o >= n || b + o >= n || buf[o] != buf[la + o]) break;
                        l++;
                    }
                    break;
                }
                uint64_t lim = std::min(la, lb);
                if (q && q < lim) lim = q;
                l = 0;
                while (l < lim && buf[l] == buf[la + l]) l++;
                bool hit_window = (l == lim) && !(q && lim == q) && lim < std::min(n - a, n - b);
                if (!hit_window) break;
                win *= 16;
            }
        }
        if (r->memory == SUFR_B200_MEM_DEVICE) {
            if (r->index_bits == 32) {
                uint32_t v = (uint32_t)l;
                SUFR_CUDA_CHECK(cudaMemcpyAsync(r->lcp, &v, 4, cudaMemcpyHostToDevice, ctx->stream));
            } else {
                SUFR_CUDA_CHECK(cudaMemcpyAsync(r->lcp, &l, 8, cudaMemcpyHostToDevice, ctx->stream));
            }
            SUFR_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
        } else {
            if (r->index_bits == 32) ((uint32_t*)r->lcp)[0] = (uint32_t)l;
            else ((uint64_t*)r->lcp)[0] = l;
        }
    });
}

int sufr_b200_verify(SufrB200Ctx* c, const SufrB200Args* args, const SufrB200Result* r, int has_prev,
                     uint64_t prev_last_suffix, SufrB200VerifyReport* out) {
    return guarded([&] {
        Ctx* ctx = reinterpret_cast<Ctx*>(c);
        if (!ctx || !args || !r || !out) throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
        if (r->memory != SUFR_B200_MEM_DEVICE || !r->text)
            throw Error(SUFR_B200_ERR_ARGUMENT, "sufr_b200_verify needs a device result (with its transformed text)");
        SeedMaskInfo mask;
        const bool has_mask = args->seed_mask && parse_seed_mask(args->seed_mask, mask);
        CtxLock lock(*ctx);
        cudaStream_t st = ctx->stream;
        const uint64_t n = r->text_len, s = r->num_suffixes;
        verify::Params P{};
        P.text = r->text;
        P.n = n;
        P.sa = r->sa;
        P.lcp = r->lcp;
        P.s = s;
        P.wide = r->index_bits == 64;
        P.filter = args->is_dna && !args->allow_ambiguity;
        P.mode = has_mask ? 2 : (args->has_max_query_len && args->max_query_len > 0 ? 1 : 0);
        P.q = args->max_query_len;
        P.has_prev = has_prev ? 1 : 0;
        P.prev_last = prev_last_suffix;
        DevBuf<uint32_t> d_maskpos;
        if (has_mask) {
            std::vector<uint32_t> mp(mask.positions.begin(), mask.positions.end());
            d_maskpos = DevBuf<uint32_t>(ctx->pool, mp.size());
            SUFR_CUDA_CHECK(cudaMemcpyAsync(d_maskpos.get(), mp.data(), mp.size() * 4, cudaMemcpyHostToDevice, st));
            SUFR_CUDA_CHECK(cudaStreamSynchronize(st));
            P.mask_pos = d_maskpos.get();
            P.weight = (uint32_t)mask.weight;
        }
        DevBuf<uint64_t> d_ns, d_ne;
        if (!has_mask && r->num_n_ranges) {  // find_lcp consults the runs only outside mask mode (sufr_builder.rs:301-307)
            std::vector<uint64_t> hs(r->num_n_ranges), he(r->num_n_ranges);
            for (uint64_t i = 0; i < r->num_n_ranges; i++) { hs[i] = r->n_ranges[2 * i]; he[i] = r->n_ranges[2 * i + 1]; }
            d_ns = DevBuf<uint64_t>(ctx->pool, hs.size());
            d_ne = DevBuf<uint64_t>(ctx->pool, he.size());
            SUFR_CUDA_CHECK(cudaMemcpyAsync(d_ns.get(), hs.data(), hs.size() * 8, cudaMemcpyHostToDevice, st));
            SUFR_CUDA_CHECK(cudaMemcpyAsync(d_ne.get(), he.data(), he.size() * 8, cudaMemcpyHostToDevice, st));
            SUFR_CUDA_CHECK(cudaStreamSynchronize(st));
            P.n_starts = d_ns.get();
            P.n_ends = d_ne.get();
            P.num_n_ranges = (uint32_t)r->num_n_ranges;
        }
        DevBuf<uint32_t> bitmap(ctx->pool, n / 32 + 2);
        DevBuf<verify::Report> d_rep(ctx->pool, 1);
        DevBuf<unsigned long long> d_cnt(ctx->pool, 1);
        verify::Report init{};
        init.first_bad_rank = ~0ull;
        SUFR_CUDA_CHECK(cudaMemsetAsync(bitmap.get(), 0, (n / 32 + 2) * 4, st));
        SUFR_CUDA_CHECK(cudaMemsetAsync(d_cnt.get(), 0, 8, st));
        SUFR_CUDA_CHECK(cudaMemcpyAsync(d_rep.get(), &init, sizeof(init), cudaMemcpyHostToDevice, st));
        EventTimer timer(st);
        const int t0 = timer.mark();
        const uint32_t grid = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(1, div_up(s, 256)), (uint64_t)num_sms() * 16);
        DevBuf<uint32_t> defer_bits(ctx->pool, s / 32 + 2);
        SUFR_CUDA_CHECK(cudaMemsetAsync(defer_bits.get(), 0, (s / 32 + 2) * 4, st));
        int method = 0;
        if (s) {
            verify::positions_kernel<<<grid, 256, 0, st>>>(P, bitmap.get(), d_rep.get());
            SUFR_KERNEL_CHECK();
            verify::pairs_kernel<<<grid, 256, 0, st>>>(P, d_rep.get(), defer_bits.get(), 0);
            SUFR_KERNEL_CHECK();
            verify::Report mid{};
            SUFR_CUDA_CHECK(cudaMemcpyAsync(&mid, d_rep.get(), sizeof(mid), cudaMemcpyDeviceToHost, st));
            SUFR_CUDA_CHECK(cudaStreamSynchronize(st));
            if (mid.deferred) {
                // deep repeats.  Full sort with every position present in this array: linear-time proof through the
                // inverse suffix array; otherwise (filtered / sharded / capped keys) the deferred pairs directly.
                const bool linear = P.mode == 0 && s == n && !has_prev && mid.duplicates == 0 && mid.out_of_range == 0 &&
                                    n <= 0xFFFFFFFFull;
                if (linear) {
                    method = 2;
                    DevBuf<uint32_t> isa(ctx->pool, n + 1);
                    verify::isa_kernel<<<grid, 256, 0, st>>>(P, isa.get());
                    SUFR_KERNEL_CHECK();
                    verify::order_by_rank_kernel<<<grid, 256, 0, st>>>(P, isa.get(), defer_bits.get(), d_rep.get());
                    SUFR_KERNEL_CHECK();
                    const uint64_t chunks = div_up(n, verify::kKasaiChunk);
                    verify::kasai_kernel<<<(uint32_t)std::max<uint64_t>(1, div_up(chunks, 256)), 256, 0, st>>>(
                        P, isa.get(), defer_bits.get(), d_rep.get());
                    SUFR_KERNEL_CHECK();
                    SUFR_CUDA_CHECK(cudaStreamSynchronize(st));
                } else {
                    method = 1;
                    verify::pairs_kernel<<<grid, 256, 0, st>>>(P, d_rep.get(), defer_bits.get(), 1);
                    SUFR_KERNEL_CHECK();
                }
            }
        }
        if (P.filter && n) {
            verify::count_indexed_kernel<<<(uint32_t)std::min<uint64_t>(div_up(n, 256 * 16), (uint64_t)num_sms() * 16), 256, 0, st>>>(
                r->text, n, d_cnt.get());
            SUFR_KERNEL_CHECK();
        }
        const int t1 = timer.mark();
        verify::Report rep{};
        unsigned long long cnt = 0;
        SUFR_CUDA_CHECK(cudaMemcpyAsync(&rep, d_rep.get(), sizeof(rep), cudaMemcpyDeviceToHost, st));
        SUFR_CUDA_CHECK(cudaMemcpyAsync(&cnt, d_cnt.get(), 8, cudaMemcpyDeviceToHost, st));
        SUFR_CUDA_CHECK(cudaStreamSynchronize(st));
        memset(out, 0, sizeof(*out));
        out->pairs_checked = rep.pairs_checked;
        out->order_errors = rep.order_errors;
        out->lcp_errors = rep.lcp_errors;
        out->out_of_range = rep.out_of_range;
        out->not_indexed = rep.not_indexed;
        out->duplicates = rep.duplicates;
        out->first_bad_rank = rep.first_bad_rank;
        out->max_lcp = rep.max_lcp;
        out->lcp_sum = rep.lcp_sum;
        out->expected_suffixes = P.filter ? cnt : n;
        out->deferred_pairs = rep.deferred;
        out->method = (uint32_t)method;
        out->ms = timer.ms(t0, t1);
    });
}

int sufr_b200_write(const SufrB200Args* args, const SufrB200Result* r) {
    return guarded([&] {
        if (!args || !r) throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
        if (r->memory != SUFR_B200_MEM_HOST) throw Error(SUFR_B200_ERR_ARGUMENT, "sufr_b200_write needs a host result");
        write_sufr_file(*args, *r);
    });
}

int sufr_b200_create(const SufrB200Args* args, int device, SufrB200Result* out) {
    SufrB200Result local;
    SufrB200Result* res = out ? out : &local;
    int rc = guarded([&] {
        if (!args) throw Error(SUFR_B200_ERR_ARGUMENT, "args is NULL");
        if (args->world_size > 1)
            throw Error(SUFR_B200_ERR_ARGUMENT,
                        "sufr_b200_create is the single-process path; a sharded build exchanges (count, first, last) "
                        "between sufr_b200_build and sufr_b200_write");
        std::unique_ptr<Ctx> ctx(make_ctx(device));
        SufrB200Result dev;
        memset(&dev, 0, sizeof(dev));
        auto teardown = [&] {
            if (dev.owner) free_owner(static_cast<ResultOwner*>(dev.owner));
            dev.owner = nullptr;
            ctx->pinned.sizes.clear();
            release_ctx(*ctx);
        };
        try {
            {
                std::lock_guard<std::mutex> lock(ctx->mu);
                run_build(*ctx, *args, 0, SUFR_B200_MEM_HOST, SUFR_B200_MEM_DEVICE, &dev);
            }
            // the suffix and LCP arrays go straight from device memory into the file
            uint8_t* host_text = nullptr;
            const auto w0 = std::chrono::steady_clock::now();
            stream_result_to_file(ctx->device, ctx->stream, *args, dev, &host_text);
            const double write_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - w0).count();
            host_result(dev, host_text, res);
            res->timings.d2h_ms = write_ms;  // device -> host -> file, overlapped
            res->d2h_bytes = (host_text ? dev.text_len : 0) + 2 * dev.num_suffixes * (dev.index_bits / 8);
        } catch (...) {
            teardown();
            throw;
        }
        teardown();
    });
    if (rc == SUFR_B200_OK && !out) sufr_b200_result_free(nullptr, &local);
    return rc;
}

// One call, several GPUs of one box: a host thread per device builds key-range shard r of `num_devices`, the raw text
// is uploaded once and replicated over NVLink (peer copies from the first device), the threads exchange
// (count, first, last) in host memory, every shard repairs its seam LCP and streams its slice of the suffix / LCP
// arrays into the file at its offset (sufr_builder.rs:817-918 writes the same sections serially).
int sufr_b200_create_multi(const SufrB200Args* args, const int* devices, int num_devices, uint32_t index_bits,
                           SufrB200Result* out) {
    SufrB200Result local;
    SufrB200Result* res = out ? out : &local;
    int rc = guarded([&] {
        if (!args || !devices) throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
        if (num_devices < 1 || num_devices > 64) throw Error(SUFR_B200_ERR_ARGUMENT, "num_devices must be 1..64");
        if (args->world_size > 1)
            throw Error(SUFR_B200_ERR_ARGUMENT, "sufr_b200_create_multi shards the build itself: pass world_size <= 1");
        if (args->text_len && !args->text) throw Error(SUFR_B200_ERR_ARGUMENT, "text is NULL");
        for (int i = 0; i < num_devices; i++)
            for (int k = 0; k < i; k++)
                if (devices[i] == devices[k]) throw Error(SUFR_B200_ERR_ARGUMENT, "a device is listed twice");
        const int W = num_devices;
        const uint64_t n = args->text_len;

        struct Shard {
            std::unique_ptr<Ctx> ctx;
            SufrB200Args a;
            SufrB200Result dev;
            uint8_t* host_text = nullptr;
            double write_ms = 0, h2d_ms = 0;
            std::exception_ptr err;
        };
        std::vector<Shard> sh(W);
        for (auto& x : sh) memset(&x.dev, 0, sizeof(x.dev));
        std::atomic<bool> failed{false};
        struct Barrier {
            std::mutex mu;
            std::condition_variable cv;
            int waiting = 0, generation = 0, parties;
            explicit Barrier(int p) : parties(p) {}
            void wait() {
                std::unique_lock<std::mutex> lock(mu);
                const int gen = generation;
                if (++waiting == parties) { waiting = 0; generation++; cv.notify_all(); }
                else cv.wait(lock, [&] { return gen != generation; });
            }
        } bar(W);
        uint8_t* raw0 = nullptr;  // raw text on the first device

        auto worker = [&](int r) {
            Shard& me = sh[r];
            auto step = [&](auto&& f) {
                if (failed.load()) return;
                try { f(); } catch (...) { me.err = std::current_exception(); failed.store(true); }
            };
            DevBuf<uint8_t> raw;
            step([&] {
                me.ctx.reset(make_ctx(devices[r]));
                me.a = *args;
                me.a.rank = r;
                me.a.world_size = W;
                raw = DevBuf<uint8_t>(me.ctx->pool, n + 16);
                if (r == 0) {
                    const auto t0 = std::chrono::steady_clock::now();
                    if (n) SUFR_CUDA_CHECK(cudaMemcpyAsync(raw.get(), args->text, n, cudaMemcpyHostToDevice, me.ctx->stream));
                    SUFR_CUDA_CHECK(cudaStreamSynchronize(me.ctx->stream));
                    me.h2d_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
                    raw0 = raw.get();
                } else {
                    cudaDeviceEnablePeerAccess(devices[0], 0);  // direct NVLink copies when the pair allows it
                    cudaGetLastError();
                }
            });
            bar.wait();
            step([&] {
                if (r > 0 && n) {
                    SUFR_CUDA_CHECK(cudaMemcpyPeerAsync(raw.get(), devices[r], raw0, devices[0], n, me.ctx->stream));
                    SUFR_CUDA_CHECK(cudaStreamSynchronize(me.ctx->stream));
                }
            });
            bar.wait();  // the first device keeps its copy alive until every peer has read it
            step([&] {
                me.a.text = raw.get();
                std::lock_guard<std::mutex> lock(me.ctx->mu);
                run_build(*me.ctx, me.a, index_bits, SUFR_B200_MEM_DEVICE, SUFR_B200_MEM_DEVICE, &me.dev);
            });
            raw.reset();
            bar.wait();
            step([&] {
                // (count, first, last) of every shard are final: offsets, total, previous non-empty shard
                uint64_t off = 0, total = 0;
                bool have_prev = false;
                uint64_t prev_last = 0;
                for (int k = 0; k < W; k++) {
                    if (k < r) {
                        off += sh[k].dev.num_suffixes;
                        if (sh[k].dev.num_suffixes) { have_prev = true; prev_last = sh[k].dev.last_suffix; }
                    }
                    total += sh[k].dev.num_suffixes;
                }
                me.dev.shard_offset = off;
                me.dev.total_suffixes = total;
                if (have_prev && me.dev.num_suffixes) {
                    if (sufr_b200_patch_seam(reinterpret_cast<SufrB200Ctx*>(me.ctx.get()), &me.a, &me.dev, prev_last) != SUFR_B200_OK)
                        throw Error(SUFR_B200_ERR_INTERNAL, "seam repair failed: " + g_last_error);
                }
                me.a.text = args->text;  // host text again (unused by the writer)
                const auto w0 = std::chrono::steady_clock::now();
                stream_result_to_file(me.ctx->device, me.ctx->stream, me.a, me.dev, r == 0 ? &me.host_text : nullptr);
                me.write_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - w0).count();
            });
        };
        std::vector<std::thread> threads;
        for (int r = 1; r < W; r++) threads.emplace_back(worker, r);
        worker(0);
        for (auto& t : threads) t.join();

        // result of the whole build: counts, transformed text, n_ranges
        std::exception_ptr first_err;
        for (auto& x : sh)
            if (x.err && !first_err) first_err = x.err;
        if (!first_err) {
            host_result(sh[0].dev, sh[0].host_text, res);
            sh[0].host_text = nullptr;
            res->num_suffixes = sh[0].dev.total_suffixes;
            res->shard_offset = 0;
            res->timings.h2d_ms = sh[0].h2d_ms;
            res->kernel_launches = 0;
            res->peak_device_bytes = 0;
            res->d2h_bytes = n;
            res->h2d_bytes = n;
            for (auto& x : sh) {
                res->timings.total_ms = std::max(res->timings.total_ms, x.dev.timings.total_ms);
                res->timings.d2h_ms = std::max(res->timings.d2h_ms, x.write_ms);
                res->kernel_launches += x.dev.kernel_launches;
                res->peak_device_bytes = std::max(res->peak_device_bytes, x.dev.peak_device_bytes);
                res->d2h_bytes += 2 * x.dev.num_suffixes * (x.dev.index_bits / 8);
                res->refine_rounds = std::max(res->refine_rounds, x.dev.refine_rounds);
                res->doubling_rounds = std::max(res->doubling_rounds, x.dev.doubling_rounds);
            }
        }
        for (auto& x : sh) {  // tear the per-device state down on its device
            if (!x.ctx) continue;
            cudaSetDevice(x.ctx->device);
            if (x.dev.owner) free_owner(static_cast<ResultOwner*>(x.dev.owner));
            x.dev.owner = nullptr;
            x.ctx->pinned.sizes.clear();
            release_ctx(*x.ctx);
            free(x.host_text);
        }
        if (first_err) std::rethrow_exception(first_err);
    });
    if (rc == SUFR_B200_OK && !out) sufr_b200_result_free(nullptr, &local);
    return rc;
}

int64_t sufr_b200_seed_mask(const char* mask, uint8_t* bytes, uint64_t* positions, uint64_t* differences) {
    SeedMaskInfo m;
    if (!mask || !parse_seed_mask(mask, m)) return -1;
    for (size_t i = 0; i < m.bytes.size(); i++)
        if (bytes) bytes[i] = m.bytes[i];
    for (size_t i = 0; i < m.positions.size(); i++) {
        if (positions) positions[i] = m.positions[i];
        if (differences) differences[i] = m.positions[i] - i;
    }
    return (int64_t)m.weight;
}

uint64_t sufr_b200_find_lcp_full_offset(uint64_t lcp, const char* mask) {
    if (!mask) return lcp;
    SeedMaskInfo m;
    if (!parse_seed_mask(mask, m)) return (uint64_t)-1;
    return lcp_full_offset(lcp, m);
}

int sufr_b200_read_sequence_file(const char* path, uint8_t delim, SufrB200Sequences* out) {
    return guarded([&] {
        if (!path || !out) throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
        read_sequence_file(path, delim, out);
    });
}

void sufr_b200_sequences_free(SufrB200Sequences* s) { free_sequences(s); }

int sufr_b200_synth_dna(SufrB200Ctx* c, uint8_t* device_text, uint64_t text_len, uint64_t seed,
                        const uint64_t* record_starts, uint64_t num_records, uint8_t delimiter) {
    return guarded([&] {
        Ctx* ctx = reinterpret_cast<Ctx*>(c);
        if (!ctx || !device_text) throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
        CtxLock lock(*ctx);
        if (text_len == 0) return;
        synth_dna_kernel<<<grid_for(text_len, 4), kBlock, 0, ctx->stream>>>(device_text, text_len, seed);
        SUFR_KERNEL_CHECK();
        DevBuf<uint64_t> d_starts(ctx->pool, num_records ? num_records : 1);
        if (num_records)
            SUFR_CUDA_CHECK(cudaMemcpyAsync(d_starts.get(), record_starts, num_records * 8, cudaMemcpyHostToDevice,
                                            ctx->stream));
        uint64_t threads = num_records ? num_records : 1;
        synth_marks_kernel<<<(unsigned)div_up(threads, 256), 256, 0, ctx->stream>>>(device_text, text_len, d_starts.get(),
                                                                                   num_records, delimiter);
        SUFR_KERNEL_CHECK();
        SUFR_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
    });
}

}  // extern "C"
