// Build pipeline + C ABI of libsufr_b200.so.
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
#include <fcntl.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <cerrno>
#include <chrono>
#include <condition_variable>
#include <cstdlib>
#include <deque>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/sufr_b200.h"
#include "common.cuh"
#include "host_io.hpp"
#include "kernels.cuh"
#include "keys.cuh"
#include "pool.hpp"
#include "radix_sort.cuh"
#include "scan.cuh"
#include "search.cuh"
#include "verify.cuh"

namespace sufr {

thread_local std::string g_last_error;

// Pinned host buffers are expensive to allocate (page-locking tens of GB takes seconds), so host results
// hand their buffers back to the context for the next build.
struct PinnedCache {
    std::vector<std::pair<void*, size_t>> free_list;
    void* get(size_t bytes) {
        if (bytes == 0) bytes = 1;
        size_t best = (size_t)-1;
        for (size_t i = 0; i < free_list.size(); i++)
            if (free_list[i].second >= bytes && (best == (size_t)-1 || free_list[i].second < free_list[best].second)) best = i;
        if (best != (size_t)-1 && free_list[best].second <= 2 * bytes + (1u << 20)) {
            void* p = free_list[best].first;
            sizes[p] = free_list[best].second;
            free_list.erase(free_list.begin() + best);
            return p;
        }
        void* p = nullptr;
        cudaError_t e = cudaMallocHost(&p, bytes);
        if (e != cudaSuccess) {
            cudaGetLastError();
            release();
            e = cudaMallocHost(&p, bytes);
            if (e != cudaSuccess) {
                cudaGetLastError();
                throw Error(SUFR_B200_ERR_OUT_OF_MEMORY, "cudaMallocHost(" + std::to_string(bytes) + " bytes) failed");
            }
        }
        sizes[p] = bytes;
        return p;
    }
    void put(void* p) {
        auto it = sizes.find(p);
        if (it == sizes.end()) { cudaFreeHost(p); return; }
        free_list.push_back({p, it->second});
        sizes.erase(it);
        while (free_list.size() > 6) {  // keep a couple of builds' worth
            cudaFreeHost(free_list.front().first);
            free_list.erase(free_list.begin());
        }
    }
    void release() {
        for (auto& f : free_list) cudaFreeHost(f.first);
        free_list.clear();
    }
    std::map<void*, size_t> sizes;  // buffers currently lent out
};

struct Ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    DevicePool pool;
    PinnedCache pinned;
    uint64_t launches = 0;
    std::mutex mu;
};

// Holds everything a returned result owns.
struct ResultOwner {
    Ctx* ctx = nullptr;          // device buffers go back to this pool
    bool owns_ctx = false;       // sufr_b200_create made a private context
    bool text_malloc = false;    // host text from malloc (sufr_b200_create), not from the pinned cache
    int memory = SUFR_B200_MEM_HOST;
    void* text = nullptr;
    void* sa = nullptr;
    void* lcp = nullptr;
    uint64_t* n_ranges = nullptr;
    // kept for sufr_b200_patch_seam on device results
};

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
static void free_owner(ResultOwner* o) {
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
    if (o->owns_ctx && o->ctx) {
        cudaStreamDestroy(o->ctx->stream);
        delete o->ctx;
    }
    delete o;
}

// Every entry point leaves the calling thread's current CUDA device as it found it (the library switches to the
// device of the context / of each shard inside; frameworks such as torch cache the current device per thread).
struct DeviceRestore {
    int prev = -1;
    DeviceRestore() { if (cudaGetDevice(&prev) != cudaSuccess) { cudaGetLastError(); prev = -1; } }
    ~DeviceRestore() { if (prev >= 0) cudaSetDevice(prev); }
};

template <typename F>
static int guarded(F&& f) {
    DeviceRestore restore;
    try {
        f();
        return SUFR_B200_OK;
    } catch (const Error& e) {
        g_last_error = e.what();
        return e.code;
    } catch (const std::bad_alloc&) {
        g_last_error = "host allocation failed";
        return SUFR_B200_ERR_OUT_OF_MEMORY;
    } catch (const std::exception& e) {
        g_last_error = e.what();
        return SUFR_B200_ERR_INTERNAL;
    }
}

// A ring of pinned host buffers, each with an event that marks the end of the last copy that used it.  Shared by the
// two directions of the file path: StreamWriter (device -> slot -> file) and upload_file_sections (file -> slot ->
// device).  acquire() blocks until a slot is free and returns -1 once abort() has been called.
class PinnedSlots {
   public:
    PinnedSlots(size_t slot_bytes, int nslots) : slot_bytes_(slot_bytes) {
        try {
            for (int i = 0; i < nslots; i++) {
                slots_.push_back(Slot{nullptr, nullptr});
                SUFR_CUDA_CHECK(cudaMallocHost(&slots_.back().buf, slot_bytes_));
                SUFR_CUDA_CHECK(cudaEventCreateWithFlags(&slots_.back().ev, cudaEventDisableTiming));
                free_.push_back(i);
            }
        } catch (...) {  // a constructor that throws runs no destructor: release what was allocated
            release();
            throw;
        }
    }
    ~PinnedSlots() { release(); }
    PinnedSlots(const PinnedSlots&) = delete;
    PinnedSlots& operator=(const PinnedSlots&) = delete;
    size_t slot_bytes() const { return slot_bytes_; }
    void* buf(int i) const { return slots_[i].buf; }
    cudaEvent_t event(int i) const { return slots_[i].ev; }
    int acquire() {
        std::unique_lock<std::mutex> lock(mu_);
        cv_.wait(lock, [&] { return !free_.empty() || aborted_; });
        if (aborted_) return -1;
        const int i = free_.front();
        free_.pop_front();
        return i;
    }
    void put(int i) {
        {
            std::lock_guard<std::mutex> lock(mu_);
            free_.push_back(i);
        }
        cv_.notify_one();
    }
    void abort() {
        {
            std::lock_guard<std::mutex> lock(mu_);
            aborted_ = true;
        }
        cv_.notify_all();
    }

   private:
    struct Slot { void* buf; cudaEvent_t ev; };
    void release() {
        for (auto& sl : slots_) {
            if (sl.buf) cudaFreeHost(sl.buf);
            if (sl.ev) cudaEventDestroy(sl.ev);
        }
        slots_.clear();
    }
    size_t slot_bytes_;
    std::vector<Slot> slots_;
    std::deque<int> free_;
    std::mutex mu_;
    std::condition_variable cv_;
    bool aborted_ = false;
};

// sufr_b200_create: the sections of the file go from device memory to the file through a small ring of pinned
// buffers -- the device->host copy of one chunk overlaps the pwrite of the previous ones, and no host copy of the
// suffix / LCP arrays is ever allocated (page-locking 2 * s * sizeof(T) bytes costs seconds by itself).
class StreamWriter {
   public:
    StreamWriter(OutputFile& file, int device, cudaStream_t stream, size_t slot_bytes = 64u << 20, int nslots = 6,
                 int nworkers = 4)
        : file_(file), device_(device), stream_(stream), slots_(slot_bytes, nslots) {
        for (int i = 0; i < nworkers; i++) workers_.emplace_back([this] { work(); });
    }
    ~StreamWriter() {
        try { finish(); } catch (...) {}
    }
    // Queue `len` bytes of device memory for file offset `off`; `host_copy` (optional) also receives them.
    void submit(const void* dev, size_t len, uint64_t off, uint8_t* host_copy = nullptr) {
        const char* p = (const char*)dev;
        while (len) {
            const size_t chunk = std::min(len, slots_.slot_bytes());
            const int slot = slots_.acquire();
            if (slot < 0) {
                std::lock_guard<std::mutex> lock(mu_);
                std::rethrow_exception(err_);
            }
            SUFR_CUDA_CHECK(cudaMemcpyAsync(slots_.buf(slot), p, chunk, cudaMemcpyDeviceToHost, stream_));
            SUFR_CUDA_CHECK(cudaEventRecord(slots_.event(slot), stream_));
            {
                std::lock_guard<std::mutex> lock(mu_);
                jobs_.push_back({slot, chunk, off, host_copy});
            }
            cv_work_.notify_one();
            p += chunk;
            off += chunk;
            if (host_copy) host_copy += chunk;
            len -= chunk;
            bytes_ += chunk;
        }
    }
    void finish() {
        {
            std::lock_guard<std::mutex> lock(mu_);
            if (done_) return;
            done_ = true;
        }
        cv_work_.notify_all();
        for (auto& t : workers_) t.join();
        workers_.clear();
        if (err_) std::rethrow_exception(err_);
    }
    uint64_t bytes() const { return bytes_; }

   private:
    struct Job { int slot; size_t len; uint64_t off; uint8_t* host_copy; };
    void work() {
        cudaSetDevice(device_);
        for (;;) {
            Job j;
            {
                std::unique_lock<std::mutex> lock(mu_);
                cv_work_.wait(lock, [&] { return !jobs_.empty() || done_; });
                if (jobs_.empty()) return;
                j = jobs_.front();
                jobs_.pop_front();
            }
            try {
                cudaError_t e = cudaEventSynchronize(slots_.event(j.slot));
                if (e != cudaSuccess) throw Error(100 + (int)e, std::string("CUDA error in the file writer: ") + cudaGetErrorString(e));
                if (j.host_copy) memcpy(j.host_copy, slots_.buf(j.slot), j.len);
                file_.write(j.off, slots_.buf(j.slot), j.len);
            } catch (...) {
                {
                    std::lock_guard<std::mutex> lock(mu_);
                    if (!err_) err_ = std::current_exception();
                }
                slots_.abort();
            }
            slots_.put(j.slot);
        }
    }
    OutputFile& file_;
    int device_;
    cudaStream_t stream_;
    PinnedSlots slots_;
    std::deque<Job> jobs_;
    std::vector<std::thread> workers_;
    std::mutex mu_;
    std::condition_variable cv_work_;
    bool done_ = false;
    std::exception_ptr err_;
    uint64_t bytes_ = 0;
};

// sufr_b200_index_open, the mirror of StreamWriter: host threads pread chunks of the file into the pinned slots and
// queue each slot's host->device copy on the context's stream.  A slot is refilled once the event recorded behind its
// last copy has completed, so reads, copies and the other threads' reads overlap.  Returns after a synchronise.
struct FileSection {
    uint64_t file_off;
    uint64_t len;
    void* dev;
};
static void upload_file_sections(int fd, const std::string& path, int device, cudaStream_t stream,
                                 const std::vector<FileSection>& sections) {
    const size_t slot_bytes = 32u << 20;
    struct Chunk { uint64_t file_off; size_t len; char* dev; };
    std::vector<Chunk> chunks;
    for (const auto& s : sections)
        for (uint64_t o = 0; o < s.len; o += slot_bytes)
            chunks.push_back({s.file_off + o, (size_t)std::min<uint64_t>(slot_bytes, s.len - o), (char*)s.dev + o});
    if (chunks.empty()) return;
    const int hw = std::max(2, (int)std::thread::hardware_concurrency());
    const int readers = std::min<int>(std::min(16, hw), (int)chunks.size());
    PinnedSlots slots(slot_bytes, readers + 4);
    std::atomic<size_t> next{0};
    std::mutex err_mu;
    std::exception_ptr err;
    auto work = [&]() {
        try {
            SUFR_CUDA_CHECK(cudaSetDevice(device));
            for (;;) {
                const size_t c = next.fetch_add(1);
                if (c >= chunks.size()) return;
                const int slot = slots.acquire();
                if (slot < 0) return;
                try {
                    SUFR_CUDA_CHECK(cudaEventSynchronize(slots.event(slot)));  // the slot's previous copy is done
                    pread_all(fd, slots.buf(slot), chunks[c].len, chunks[c].file_off, path);
                    SUFR_CUDA_CHECK(cudaMemcpyAsync(chunks[c].dev, slots.buf(slot), chunks[c].len, cudaMemcpyHostToDevice, stream));
                    SUFR_CUDA_CHECK(cudaEventRecord(slots.event(slot), stream));
                } catch (...) {
                    slots.put(slot);
                    throw;
                }
                slots.put(slot);
            }
        } catch (...) {
            {
                std::lock_guard<std::mutex> lock(err_mu);
                if (!err) err = std::current_exception();
            }
            slots.abort();
        }
    };
    std::vector<std::thread> pool;
    for (int t = 1; t < readers; t++) pool.emplace_back(work);
    work();
    for (auto& th : pool) th.join();
    const cudaError_t e = cudaStreamSynchronize(stream);  // before the slots are released
    if (err) std::rethrow_exception(err);
    SUFR_CUDA_CHECK(e);
}

// Writes the file of a DEVICE result (sufr_builder.rs:817-918) and returns the transformed text in `host_text`
// (malloc; what SufrBuilder.text holds after `new`).
static void stream_result_to_file(Ctx& ctx, const SufrB200Args& args, const SufrB200Result& r, uint8_t** host_text) {
    const std::string path = args.path ? args.path : "out.sufr";  // sufr_builder.rs:215
    const size_t w = r.index_bits / 8;
    const SufrFrame f = make_sufr_frame(args, r.index_bits, r.text_len, r.total_suffixes);
    const bool sharded = args.world_size > 1;
    const bool leader = !sharded || args.rank == 0;
    OutputFile out(path, f.names_pos + f.tail.size(), !sharded);
    uint8_t* text = nullptr;
    try {
        if (leader) {  // ranks > 0 of a sharded build neither write nor return the text
            text = (uint8_t*)malloc(std::max<uint64_t>(1, r.text_len));
            if (!text) throw Error(SUFR_B200_ERR_OUT_OF_MEMORY, "out of host memory for the transformed text");
        }
        {
            // page-cache / tmpfs writes are CPU bound (page allocation + copy): many writers on many small slots,
            // shared fairly between the ranks of a multi-GPU build
            const int hw = (int)std::thread::hardware_concurrency();
            const int share = std::max(1, (int)args.world_size);
            int workers = std::max(2, std::min(24, (hw - 2) / share));
            if (const char* dbg = getenv("SUFR_B200_WRITER_THREADS")) workers = std::max(1, atoi(dbg));
            StreamWriter sw(out, ctx.device, ctx.stream, 16u << 20, workers + 4, workers);
            if (leader) {
                out.write(0, f.head.data(), f.head.size());
                out.write(f.names_pos, f.tail.data(), f.tail.size());
                sw.submit(r.text, r.text_len, f.text_pos, text);
            }
            sw.submit(r.sa, r.num_suffixes * w, f.sa_pos + r.shard_offset * w);
            sw.submit(r.lcp, r.num_suffixes * w, f.lcp_pos + r.shard_offset * w);
            sw.finish();
        }
        out.close();
    } catch (...) {
        free(text);
        throw;
    }
    if (host_text) *host_text = text; else free(text);
}

static Ctx* make_ctx(int device) {
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

// Rebuilds the KeySpec of a finished result far enough to compute one pair LCP (seam repair).
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
    cudaStreamSynchronize(ctx->stream);
    ctx->pool.release_all();
    ctx->pinned.release();
    cudaStreamDestroy(ctx->stream);
    delete ctx;
}

int sufr_b200_ctx_reserve(SufrB200Ctx* c, uint64_t text_len, uint32_t index_bits) {
    return guarded([&] {
        Ctx* ctx = reinterpret_cast<Ctx*>(c);
        if (!ctx) throw Error(SUFR_B200_ERR_ARGUMENT, "ctx is NULL");
        std::lock_guard<std::mutex> lock(ctx->mu);
        SUFR_CUDA_CHECK(cudaSetDevice(ctx->device));
        uint64_t per = 32;
        (void)index_bits;
        ctx->pool.reserve((size_t)(per * text_len + (64ull << 20)));
    });
}

void sufr_b200_ctx_trim(SufrB200Ctx* c) {
    Ctx* ctx = reinterpret_cast<Ctx*>(c);
    if (!ctx) return;
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
        std::lock_guard<std::mutex> lock(ctx->mu);
        SUFR_CUDA_CHECK(cudaSetDevice(ctx->device));
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
        std::lock_guard<std::mutex> lock(ctx->mu);
        SUFR_CUDA_CHECK(cudaSetDevice(ctx->device));
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

// ---------------------------------------------------------------------------------------------
// LCP-subsampled suffix array + batched search (search.cuh)
struct SufrB200Index {
    Ctx* ctx = nullptr;
    const uint8_t* text = nullptr;
    const void* sa = nullptr;
    const void* lcp = nullptr;
    uint64_t n = 0, s = 0;
    // bytes from `text` on that may be read with 16-byte loads: n + 16 for an index that owns its (padded) text, n for
    // one that borrows a build result's (gather_regions_kernel reads the last chunk byte by byte then)
    uint64_t text_readable = 0;
    int wide = 0;
    bool is_mask = false;
    uint64_t build_mql = 0;
    uint32_t weight = 0, mask_len = 0;
    DevBuf<uint32_t> maskpos;
    DevBuf<unsigned char> sub_sa, sub_rank;
    uint64_t sub_len = 0, sub_mql = 0;
    bool has_sub = false;
    // an index opened from a file owns its arrays (text / sa / lcp above point into these)
    DevBuf<unsigned char> own_text, own_sa, own_lcp;
    // sequence starts (u64) for locate; num_starts == 0: none
    DevBuf<unsigned long long> starts;
    uint64_t num_starts = 0;
    // the last sufr_b200_index_locate: rank ranges and hit offsets of its queries, for sufr_b200_index_hits
    DevBuf<unsigned long long> loc_begin, loc_end, loc_offsets;
    uint64_t loc_queries = 0, loc_hits = 0;
    bool has_loc = false;
    // max_query_len the index was built with, as sufr_file.rs:521-528 defines it: the mask weight, else the build's
    // max_query_len, else the text length
    uint64_t built_mql() const { return is_mask ? weight : (build_mql ? build_mql : n); }
};

static void index_set_mask(SufrB200Index& idx, Ctx& ctx, const char* seed_mask, bool has_mql, uint64_t mql) {
    SeedMaskInfo mask;
    if (seed_mask && parse_seed_mask(seed_mask, mask)) {
        idx.is_mask = true;
        idx.weight = (uint32_t)mask.weight;
        idx.mask_len = (uint32_t)mask.bytes.size();
        std::vector<uint32_t> mp(mask.positions.begin(), mask.positions.end());
        idx.maskpos = DevBuf<uint32_t>(ctx.pool, mp.size());
        SUFR_CUDA_CHECK(cudaMemcpyAsync(idx.maskpos.get(), mp.data(), mp.size() * 4, cudaMemcpyHostToDevice, ctx.stream));
        SUFR_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
    } else {
        idx.build_mql = has_mql ? mql : 0;
    }
}

static void index_set_starts(SufrB200Index& idx, Ctx& ctx, const uint64_t* starts, uint64_t count) {
    idx.num_starts = count;
    if (!count) return;
    idx.starts = DevBuf<unsigned long long>(ctx.pool, count);
    SUFR_CUDA_CHECK(cudaMemcpyAsync(idx.starts.get(), starts, count * 8, cudaMemcpyHostToDevice, ctx.stream));
    SUFR_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
}

int sufr_b200_index_create(SufrB200Ctx* c, const SufrB200Args* args, const SufrB200Result* r, SufrB200Index** out) {
    return guarded([&] {
        Ctx* ctx = reinterpret_cast<Ctx*>(c);
        if (!ctx || !args || !r || !out) throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
        if (r->memory != SUFR_B200_MEM_DEVICE || !r->text)
            throw Error(SUFR_B200_ERR_ARGUMENT, "sufr_b200_index_create needs a device result (with its transformed text)");
        if (args->world_size > 1) throw Error(SUFR_B200_ERR_ARGUMENT, "an index needs the whole suffix array (world_size <= 1)");
        auto idx = std::make_unique<SufrB200Index>();
        idx->ctx = ctx;
        idx->text = r->text;
        idx->sa = r->sa;
        idx->lcp = r->lcp;
        idx->n = r->text_len;
        idx->text_readable = r->text_len;
        idx->s = r->num_suffixes;
        idx->wide = r->index_bits == 64;
        if (args->num_sequences && !args->sequence_starts) throw Error(SUFR_B200_ERR_ARGUMENT, "sequence_starts is NULL");
        std::lock_guard<std::mutex> lock(ctx->mu);
        SUFR_CUDA_CHECK(cudaSetDevice(ctx->device));
        index_set_mask(*idx, *ctx, args->seed_mask, args->has_max_query_len, args->max_query_len);
        index_set_starts(*idx, *ctx, args->sequence_starts, args->num_sequences);
        *out = idx.release();
    });
}

void sufr_b200_index_free(SufrB200Index* idx) {
    if (!idx) return;
    DeviceRestore restore;
    {
        std::lock_guard<std::mutex> lock(idx->ctx->mu);
        cudaSetDevice(idx->ctx->device);
        cudaStreamSynchronize(idx->ctx->stream);
        idx->maskpos.reset();
        idx->sub_sa.reset();
        idx->sub_rank.reset();
        idx->own_text.reset();
        idx->own_sa.reset();
        idx->own_lcp.reset();
        idx->starts.reset();
        idx->loc_begin.reset();
        idx->loc_end.reset();
        idx->loc_offsets.reset();
    }
    delete idx;
}

// with the context's lock held
static uint64_t index_subsample_locked(SufrB200Index* idx, uint64_t max_query_len) {
        Ctx& ctx = *idx->ctx;
        idx->sub_sa.reset();
        idx->sub_rank.reset();
        idx->has_sub = false;
        idx->sub_len = 0;
        const size_t w = idx->wide ? 8 : 4;
        search::SubsampleIn in{idx->lcp, idx->wide, max_query_len};
        DevBuf<uint32_t> partials(ctx.pool, scan::partials_count(idx->s));
        uint32_t total = 0;
        if (idx->s) {
            scan::scan_reduce(idx->s, in, scan::SumU32{}, partials.get(), ctx.stream);
            SUFR_CUDA_CHECK(cudaMemcpyAsync(&total, partials.get() + div_up(idx->s, scan::CHUNK), 4, cudaMemcpyDeviceToHost, ctx.stream));
            SUFR_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
        }
        idx->sub_sa = DevBuf<unsigned char>(ctx.pool, (size_t)total * w + 8);
        idx->sub_rank = DevBuf<unsigned char>(ctx.pool, (size_t)total * w + 8);
        if (idx->s) {
            scan::scan_apply(idx->s, in, scan::SumU32{}, search::SubsampleOut{idx->sa, idx->wide, idx->sub_sa.get(), idx->sub_rank.get()},
                             partials.get(), ctx.stream);
            SUFR_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
        }
        idx->sub_len = total;
        idx->sub_mql = max_query_len;
        idx->has_sub = true;
        return total;
}

int sufr_b200_index_subsample(SufrB200Index* idx, uint64_t max_query_len, uint64_t* kept) {
    return guarded([&] {
        if (!idx) throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
        std::lock_guard<std::mutex> lock(idx->ctx->mu);
        SUFR_CUDA_CHECK(cudaSetDevice(idx->ctx->device));
        const uint64_t total = index_subsample_locked(idx, max_query_len);
        if (kept) *kept = total;
    });
}

static void launch_search(SufrB200Index* idx, const uint8_t* d_q, const uint64_t* d_off, uint64_t nq, int has_mql,
                          uint64_t mql, int use_subsample, unsigned long long* d_b, unsigned long long* d_e) {
    search::Params P{};
    P.text = idx->text;
    P.n = idx->n;
    P.sa = use_subsample ? (const void*)idx->sub_sa.get() : idx->sa;
    P.rank = use_subsample ? (const void*)idx->sub_rank.get() : nullptr;
    P.len = use_subsample ? idx->sub_len : idx->s;
    P.wide = idx->wide;
    P.is_mask = idx->is_mask;
    P.build_mql = idx->build_mql;
    P.has_run_mql = has_mql ? 1 : 0;
    P.run_mql = mql;
    P.mask_pos = idx->maskpos.get();
    P.weight = idx->weight;
    P.mask_len = idx->mask_len;
    search::search_kernel<<<(unsigned)div_up(nq, 128), 128, 0, idx->ctx->stream>>>(P, d_q, d_off, nq, d_b, d_e);
    SUFR_KERNEL_CHECK();
}

int sufr_b200_index_search(SufrB200Index* idx, const uint8_t* queries, const uint64_t* offsets, uint64_t nq, int has_mql,
                           uint64_t mql, int use_subsample, uint64_t* rank_begin, uint64_t* rank_end) {
    return guarded([&] {
        if (!idx || !offsets || !rank_begin || !rank_end || (nq && !queries && offsets[nq])) throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
        if (use_subsample && !idx->has_sub) throw Error(SUFR_B200_ERR_ARGUMENT, "sufr_b200_index_subsample has not been called");
        if (nq == 0) return;
        Ctx& ctx = *idx->ctx;
        std::lock_guard<std::mutex> lock(ctx.mu);
        SUFR_CUDA_CHECK(cudaSetDevice(ctx.device));
        const uint64_t bytes = offsets[nq];
        DevBuf<uint8_t> d_q(ctx.pool, bytes + 8);
        DevBuf<uint64_t> d_off(ctx.pool, nq + 1);
        DevBuf<unsigned long long> d_b(ctx.pool, nq), d_e(ctx.pool, nq);
        if (bytes) SUFR_CUDA_CHECK(cudaMemcpyAsync(d_q.get(), queries, bytes, cudaMemcpyHostToDevice, ctx.stream));
        SUFR_CUDA_CHECK(cudaMemcpyAsync(d_off.get(), offsets, (nq + 1) * 8, cudaMemcpyHostToDevice, ctx.stream));
        launch_search(idx, d_q.get(), d_off.get(), nq, has_mql, mql, use_subsample, d_b.get(), d_e.get());
        SUFR_CUDA_CHECK(cudaMemcpyAsync(rank_begin, d_b.get(), nq * 8, cudaMemcpyDeviceToHost, ctx.stream));
        SUFR_CUDA_CHECK(cudaMemcpyAsync(rank_end, d_e.get(), nq * 8, cudaMemcpyDeviceToHost, ctx.stream));
        SUFR_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
    });
}

int sufr_b200_index_suffixes(SufrB200Index* idx, uint64_t rank_begin, uint64_t count, uint64_t* out) {
    return guarded([&] {
        if (!idx || (count && !out)) throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
        if (rank_begin > idx->s || count > idx->s - rank_begin) throw Error(SUFR_B200_ERR_ARGUMENT, "rank range out of bounds");
        if (count == 0) return;
        Ctx& ctx = *idx->ctx;
        std::lock_guard<std::mutex> lock(ctx.mu);
        SUFR_CUDA_CHECK(cudaSetDevice(ctx.device));
        if (idx->wide) {
            SUFR_CUDA_CHECK(cudaMemcpyAsync(out, (const uint64_t*)idx->sa + rank_begin, count * 8, cudaMemcpyDeviceToHost, ctx.stream));
            SUFR_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
        } else {
            std::vector<uint32_t> tmp(count);
            SUFR_CUDA_CHECK(cudaMemcpyAsync(tmp.data(), (const uint32_t*)idx->sa + rank_begin, count * 4, cudaMemcpyDeviceToHost, ctx.stream));
            SUFR_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
            for (uint64_t i = 0; i < count; i++) out[i] = tmp[i];
        }
    });
}

static char* dup_cstr(const std::string& s) {
    char* p = (char*)malloc(s.size() + 1);
    if (!p) throw std::bad_alloc();
    memcpy(p, s.data(), s.size());
    p[s.size()] = 0;
    return p;
}

int sufr_b200_file_info(const char* path, SufrB200FileInfo* out) {
    return guarded([&] {
        if (!path || !out) throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
        memset(out, 0, sizeof(*out));
        SufrFileInfo fi;
        read_sufr_info(path, fi);
        SufrB200FileInfo r;
        memset(&r, 0, sizeof(r));
        r.version = fi.version;
        r.index_bits = fi.index_bits;
        r.is_dna = fi.is_dna;
        r.allow_ambiguity = fi.allow_ambiguity;
        r.ignore_softmask = fi.ignore_softmask;
        r.text_len = fi.text_len;
        r.num_suffixes = fi.num_suffixes;
        r.max_query_len = fi.max_query_len;
        r.num_sequences = fi.sequence_starts.size();
        r.text_pos = fi.text_pos;
        r.sa_pos = fi.sa_pos;
        r.lcp_pos = fi.lcp_pos;
        r.file_bytes = fi.file_bytes;
        try {
            if (!fi.seed_mask.empty()) r.seed_mask = dup_cstr(fi.seed_mask);
            r.sequence_starts = (uint64_t*)calloc(std::max<size_t>(1, fi.sequence_starts.size()), 8);
            r.sequence_names = (char**)calloc(std::max<size_t>(1, fi.sequence_names.size()), sizeof(char*));
            if (!r.sequence_starts || !r.sequence_names) throw std::bad_alloc();
            for (size_t i = 0; i < fi.sequence_starts.size(); i++) {
                r.sequence_starts[i] = fi.sequence_starts[i];
                r.sequence_names[i] = dup_cstr(fi.sequence_names[i]);
            }
        } catch (...) {
            sufr_b200_file_info_free(&r);
            throw;
        }
        *out = r;
    });
}

void sufr_b200_file_info_free(SufrB200FileInfo* info) {
    if (!info) return;
    free(info->seed_mask);
    if (info->sequence_names)
        for (uint64_t i = 0; i < info->num_sequences; i++) free(info->sequence_names[i]);
    free(info->sequence_names);
    free(info->sequence_starts);
    memset(info, 0, sizeof(*info));
}

int sufr_b200_index_open(SufrB200Ctx* c, const char* path, SufrB200Index** out) {
    return guarded([&] {
        Ctx* ctx = reinterpret_cast<Ctx*>(c);
        if (!ctx || !path || !out) throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
        SufrFileInfo fi;
        read_sufr_info(path, fi);
        const int fd = open(path, O_RDONLY);
        if (fd < 0) throw Error(SUFR_B200_ERR_IO, std::string(path) + ": " + strerror(errno));
        struct FdCloser { int fd; ~FdCloser() { close(fd); } } closer{fd};
        std::lock_guard<std::mutex> lock(ctx->mu);
        SUFR_CUDA_CHECK(cudaSetDevice(ctx->device));
        auto idx = std::make_unique<SufrB200Index>();  // (on failure freed before the lock is released)
        idx->ctx = ctx;
        idx->n = fi.text_len;
        idx->s = fi.num_suffixes;
        idx->wide = fi.index_bits == 64;
        const size_t w = fi.index_bits / 8;
        idx->own_text = DevBuf<unsigned char>(ctx->pool, fi.text_len + 16);
        idx->text_readable = fi.text_len + 16;
        idx->own_sa = DevBuf<unsigned char>(ctx->pool, fi.num_suffixes * w + 16);
        idx->own_lcp = DevBuf<unsigned char>(ctx->pool, fi.num_suffixes * w + 16);
        idx->text = idx->own_text.get();
        idx->sa = idx->own_sa.get();
        idx->lcp = idx->own_lcp.get();
        upload_file_sections(fd, path, ctx->device, ctx->stream,
                             {{fi.text_pos, fi.text_len, idx->own_text.get()},
                              {fi.sa_pos, fi.num_suffixes * w, idx->own_sa.get()},
                              {fi.lcp_pos, fi.num_suffixes * w, idx->own_lcp.get()}});
        // a corrupt suffix array would send the searches outside the text: refused here, before any search runs
        if (fi.num_suffixes) {
            DevBuf<unsigned long long> d_max(ctx->pool, 1);
            SUFR_CUDA_CHECK(cudaMemsetAsync(d_max.get(), 0, 8, ctx->stream));
            const uint32_t grid = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(1, div_up(fi.num_suffixes, 256 * 8)),
                                                               (uint64_t)num_sms() * 8);
            search::max_entry_kernel<<<grid, 256, 0, ctx->stream>>>(idx->sa, fi.num_suffixes, idx->wide, d_max.get());
            SUFR_KERNEL_CHECK();
            unsigned long long mx = 0;
            SUFR_CUDA_CHECK(cudaMemcpyAsync(&mx, d_max.get(), 8, cudaMemcpyDeviceToHost, ctx->stream));
            SUFR_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
            if (mx >= fi.text_len)
                throw Error(SUFR_B200_ERR_IO, std::string(path) + ": invalid .sufr file: suffix array entry " + std::to_string(mx) +
                                                  " is not below the text length " + std::to_string(fi.text_len));
        }
        index_set_mask(*idx, *ctx, fi.seed_mask.empty() ? nullptr : fi.seed_mask.c_str(), fi.max_query_len > 0,
                       fi.max_query_len);
        index_set_starts(*idx, *ctx, fi.sequence_starts.data(), fi.sequence_starts.size());
        *out = idx.release();
    });
}

int sufr_b200_index_locate(SufrB200Index* idx, const uint8_t* queries, const uint64_t* offsets, uint64_t nq, int has_mql,
                           uint64_t mql, int low_memory, uint64_t* rank_begin, uint64_t* rank_end, uint64_t* hit_offsets) {
    return guarded([&] {
        if (!idx || !offsets || (nq && (!rank_begin || !rank_end)) || !hit_offsets || (nq && !queries && offsets[nq]))
            throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
        for (uint64_t i = 0; i < nq; i++)
            if (offsets[i + 1] < offsets[i]) throw Error(SUFR_B200_ERR_ARGUMENT, "query offsets are not ascending");
        Ctx& ctx = *idx->ctx;
        std::lock_guard<std::mutex> lock(ctx.mu);
        SUFR_CUDA_CHECK(cudaSetDevice(ctx.device));
        idx->has_loc = false;
        idx->loc_begin.reset();
        idx->loc_end.reset();
        idx->loc_offsets.reset();
        // sufr_file.rs:514-560: the in-memory mode searches the LCP-subsampled array when the effective max_query_len
        // is shorter than the build's
        int use_sub = 0;
        if (!low_memory) {
            const uint64_t built = idx->built_mql();
            const uint64_t eff = (has_mql && mql > 0) ? std::min(mql, built) : built;
            if (eff != built) {
                if (!idx->has_sub || idx->sub_mql != eff) index_subsample_locked(idx, eff);
                use_sub = 1;
            }
        }
        idx->loc_begin = DevBuf<unsigned long long>(ctx.pool, nq + 1);
        idx->loc_end = DevBuf<unsigned long long>(ctx.pool, nq + 1);
        idx->loc_offsets = DevBuf<unsigned long long>(ctx.pool, nq + 1);
        SUFR_CUDA_CHECK(cudaMemsetAsync(idx->loc_offsets.get(), 0, 8, ctx.stream));
        if (nq) {
            const uint64_t bytes = offsets[nq];
            DevBuf<uint8_t> d_q(ctx.pool, bytes + 8);
            DevBuf<uint64_t> d_off(ctx.pool, nq + 1);
            if (bytes) SUFR_CUDA_CHECK(cudaMemcpyAsync(d_q.get(), queries, bytes, cudaMemcpyHostToDevice, ctx.stream));
            SUFR_CUDA_CHECK(cudaMemcpyAsync(d_off.get(), offsets, (nq + 1) * 8, cudaMemcpyHostToDevice, ctx.stream));
            launch_search(idx, d_q.get(), d_off.get(), nq, has_mql, mql, use_sub, idx->loc_begin.get(), idx->loc_end.get());
            DevBuf<unsigned long long> partials(ctx.pool, scan::partials_count(nq));
            scan::inclusive_scan(nq, search::HitCountIn{idx->loc_begin.get(), idx->loc_end.get()}, scan::SumU64{},
                                 search::HitOffsetOut{idx->loc_offsets.get()}, partials.get(), ctx.stream);
            SUFR_CUDA_CHECK(cudaMemcpyAsync(rank_begin, idx->loc_begin.get(), nq * 8, cudaMemcpyDeviceToHost, ctx.stream));
            SUFR_CUDA_CHECK(cudaMemcpyAsync(rank_end, idx->loc_end.get(), nq * 8, cudaMemcpyDeviceToHost, ctx.stream));
        }
        SUFR_CUDA_CHECK(cudaMemcpyAsync(hit_offsets, idx->loc_offsets.get(), (nq + 1) * 8, cudaMemcpyDeviceToHost, ctx.stream));
        SUFR_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
        idx->loc_queries = nq;
        idx->loc_hits = hit_offsets[nq];
        idx->has_loc = true;
    });
}

int sufr_b200_index_hits(SufrB200Index* idx, uint64_t first, uint64_t count, uint64_t* suffix, uint64_t* sequence,
                         uint64_t* sequence_pos) {
    return guarded([&] {
        if (!idx) throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
        Ctx& ctx = *idx->ctx;
        std::lock_guard<std::mutex> lock(ctx.mu);  // (the state of the last locate is read under the lock it is written under)
        if (!idx->has_loc) throw Error(SUFR_B200_ERR_ARGUMENT, "sufr_b200_index_locate has not been called");
        if (first > idx->loc_hits || count > idx->loc_hits - first)
            throw Error(SUFR_B200_ERR_ARGUMENT, "hit window [" + std::to_string(first) + ", +" + std::to_string(count) +
                                                    ") is beyond the " + std::to_string(idx->loc_hits) + " hits of the last locate");
        if (count == 0) return;
        SUFR_CUDA_CHECK(cudaSetDevice(ctx.device));
        DevBuf<unsigned long long> d_out(ctx.pool, 3 * count);
        unsigned long long* d_suf = d_out.get();
        search::hits_kernel<<<(unsigned)div_up(count, 256), 256, 0, ctx.stream>>>(
            idx->sa, idx->wide, idx->loc_begin.get(), idx->loc_offsets.get(), idx->loc_queries, idx->starts.get(),
            idx->num_starts, first, count, d_suf, d_suf + count, d_suf + 2 * count);
        SUFR_KERNEL_CHECK();
        uint64_t* outs[3] = {suffix, sequence, sequence_pos};
        for (int k = 0; k < 3; k++)
            if (outs[k]) SUFR_CUDA_CHECK(cudaMemcpyAsync(outs[k], d_suf + k * count, count * 8, cudaMemcpyDeviceToHost, ctx.stream));
        SUFR_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
    });
}

// extract / list, with the context's lock held, after the window's kernel left the regions of its m entries in
// d_src / d_len: scans the lengths into byte offsets (copied to byte_offsets[0..m]), takes the longest leading run of
// entries whose bytes fit in max_bytes, gathers that run's bytes into `bytes` and returns its length.  The copies to
// the caller's other outputs are queued by the caller, which then synchronises.
static uint64_t index_gather(SufrB200Index* idx, uint64_t m, const unsigned long long* d_src, const unsigned long long* d_len,
                             uint64_t max_bytes, uint64_t* byte_offsets, uint8_t* bytes, DevBuf<uint8_t>& d_bytes) {
    Ctx& ctx = *idx->ctx;
    DevBuf<unsigned long long> d_off(ctx.pool, m + 1);
    DevBuf<unsigned long long> partials(ctx.pool, scan::partials_count(m));
    SUFR_CUDA_CHECK(cudaMemsetAsync(d_off.get(), 0, 8, ctx.stream));
    scan::inclusive_scan(m, search::ArrayIn{d_len}, scan::SumU64{}, search::HitOffsetOut{d_off.get()}, partials.get(),
                         ctx.stream);
    SUFR_CUDA_CHECK(cudaMemcpyAsync(byte_offsets, d_off.get(), (m + 1) * 8, cudaMemcpyDeviceToHost, ctx.stream));
    SUFR_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
    const uint64_t k = (uint64_t)(std::upper_bound(byte_offsets, byte_offsets + m + 1, max_bytes) - byte_offsets) - 1;
    const uint64_t total = byte_offsets[k];
    if (total) {
        d_bytes = DevBuf<uint8_t>(ctx.pool, div_up(total, 16) * 16);
        const uint64_t chunks = div_up(total, 16);
        search::gather_regions_kernel<<<(unsigned)div_up(chunks, 256), 256, 0, ctx.stream>>>(
            idx->text, idx->n, idx->text_readable, d_src, d_off.get(), k, total, d_bytes.get());
        SUFR_KERNEL_CHECK();
        SUFR_CUDA_CHECK(cudaMemcpyAsync(bytes, d_bytes.get(), total, cudaMemcpyDeviceToHost, ctx.stream));
    }
    return k;
}

int sufr_b200_index_extract(SufrB200Index* idx, uint64_t first, uint64_t max_hits, uint64_t prefix_len,
                            uint64_t suffix_len, uint64_t max_bytes, uint64_t* num_hits, uint64_t* suffix,
                            uint64_t* sequence, uint64_t* region_start, uint64_t* region_end, uint64_t* byte_offsets,
                            uint8_t* bytes) {
    return guarded([&] {
        if (!idx || !num_hits || !byte_offsets || !bytes) throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
        Ctx& ctx = *idx->ctx;
        std::lock_guard<std::mutex> lock(ctx.mu);  // (the state of the last locate is read under the lock it is written under)
        if (!idx->has_loc) throw Error(SUFR_B200_ERR_ARGUMENT, "sufr_b200_index_locate has not been called");
        if (first > idx->loc_hits || max_hits > idx->loc_hits - first)
            throw Error(SUFR_B200_ERR_ARGUMENT, "hit window [" + std::to_string(first) + ", +" + std::to_string(max_hits) +
                                                    ") is beyond the " + std::to_string(idx->loc_hits) + " hits of the last locate");
        *num_hits = 0;
        byte_offsets[0] = 0;
        if (max_hits == 0) return;
        SUFR_CUDA_CHECK(cudaSetDevice(ctx.device));
        const uint64_t m = max_hits;
        DevBuf<unsigned long long> d_out(ctx.pool, 6 * m);
        unsigned long long* d = d_out.get();
        search::extract_regions_kernel<<<(unsigned)div_up(m, 256), 256, 0, ctx.stream>>>(
            idx->sa, idx->wide, idx->loc_begin.get(), idx->loc_offsets.get(), idx->loc_queries, idx->starts.get(),
            idx->num_starts, idx->n, first, m, prefix_len, suffix_len, d, d + m, d + 2 * m, d + 3 * m, d + 4 * m, d + 5 * m);
        SUFR_KERNEL_CHECK();
        DevBuf<uint8_t> d_bytes;
        const uint64_t k = index_gather(idx, m, d + 4 * m, d + 5 * m, max_bytes, byte_offsets, bytes, d_bytes);
        uint64_t* outs[4] = {suffix, sequence, region_start, region_end};
        for (int o = 0; o < 4; o++)
            if (outs[o] && k) SUFR_CUDA_CHECK(cudaMemcpyAsync(outs[o], d + o * m, k * 8, cudaMemcpyDeviceToHost, ctx.stream));
        SUFR_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
        *num_hits = k;
    });
}

int sufr_b200_index_list(SufrB200Index* idx, uint64_t first, uint64_t max_rows, uint64_t len, uint64_t max_bytes,
                         uint64_t* num_rows, uint64_t* suffix, uint64_t* lcp, uint64_t* byte_offsets, uint8_t* bytes) {
    return guarded([&] {
        if (!idx || !num_rows || !byte_offsets || !bytes) throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
        if (first > idx->s || max_rows > idx->s - first)
            throw Error(SUFR_B200_ERR_ARGUMENT, "rank window [" + std::to_string(first) + ", +" + std::to_string(max_rows) +
                                                    ") is beyond the " + std::to_string(idx->s) + " suffixes");
        *num_rows = 0;
        byte_offsets[0] = 0;
        if (max_rows == 0) return;
        Ctx& ctx = *idx->ctx;
        std::lock_guard<std::mutex> lock(ctx.mu);
        SUFR_CUDA_CHECK(cudaSetDevice(ctx.device));
        const uint64_t m = max_rows;
        DevBuf<unsigned long long> d_out(ctx.pool, 4 * m);
        unsigned long long* d = d_out.get();
        search::list_rows_kernel<<<(unsigned)div_up(m, 256), 256, 0, ctx.stream>>>(idx->sa, idx->lcp, idx->wide, idx->n, first,
                                                                                   m, len, d, d + m, d + 2 * m, d + 3 * m);
        SUFR_KERNEL_CHECK();
        DevBuf<uint8_t> d_bytes;
        const uint64_t k = index_gather(idx, m, d + 2 * m, d + 3 * m, max_bytes, byte_offsets, bytes, d_bytes);
        if (suffix && k) SUFR_CUDA_CHECK(cudaMemcpyAsync(suffix, d, k * 8, cudaMemcpyDeviceToHost, ctx.stream));
        if (lcp && k) SUFR_CUDA_CHECK(cudaMemcpyAsync(lcp, d + m, k * 8, cudaMemcpyDeviceToHost, ctx.stream));
        SUFR_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
        *num_rows = k;
    });
}

int sufr_b200_index_string_at(SufrB200Index* idx, uint64_t pos, uint64_t len, uint8_t* out, uint64_t* out_len) {
    return guarded([&] {
        if (!idx || !out_len) throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
        if (pos > idx->n)
            throw Error(SUFR_B200_ERR_ARGUMENT, "position " + std::to_string(pos) + " is beyond the text length " +
                                                    std::to_string(idx->n));
        const uint64_t k = std::min(len, idx->n - pos);
        if (k && !out) throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
        *out_len = 0;
        if (k) {
            Ctx& ctx = *idx->ctx;
            std::lock_guard<std::mutex> lock(ctx.mu);
            SUFR_CUDA_CHECK(cudaSetDevice(ctx.device));
            SUFR_CUDA_CHECK(cudaMemcpyAsync(out, idx->text + pos, k, cudaMemcpyDeviceToHost, ctx.stream));
            SUFR_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
        }
        *out_len = k;
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
            cudaStreamSynchronize(ctx->stream);
            ctx->pinned.sizes.clear();
            ctx->pinned.release();
            ctx->pool.release_all();
            cudaStreamDestroy(ctx->stream);
        };
        try {
            {
                std::lock_guard<std::mutex> lock(ctx->mu);
                run_build(*ctx, *args, 0, SUFR_B200_MEM_HOST, SUFR_B200_MEM_DEVICE, &dev);
            }
            // the suffix and LCP arrays go straight from device memory into the file
            uint8_t* host_text = nullptr;
            const auto w0 = std::chrono::steady_clock::now();
            stream_result_to_file(*ctx, *args, dev, &host_text);
            const double write_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - w0).count();
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
            res->sa = nullptr;   // in the file, like the reference's builder struct (sufr_builder.rs:38-89)
            res->lcp = nullptr;
            res->n_ranges = owner->n_ranges;
            res->timings.d2h_ms = write_ms;  // device -> host -> file, overlapped
            res->d2h_bytes = (host_text ? dev.text_len : 0) + 2 * dev.num_suffixes * (dev.index_bits / 8);
            res->owner = owner.release();
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
                stream_result_to_file(*me.ctx, me.a, me.dev, r == 0 ? &me.host_text : nullptr);
                me.write_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - w0).count();
            });
        };
        std::vector<std::thread> threads;
        for (int r = 1; r < W; r++) threads.emplace_back(worker, r);
        worker(0);
        for (auto& t : threads) t.join();

        // result of the whole build (what SufrBuilder holds after `new`): counts, transformed text, n_ranges
        auto owner = std::make_unique<ResultOwner>();
        std::exception_ptr first_err;
        for (auto& x : sh)
            if (x.err && !first_err) first_err = x.err;
        if (!first_err) {
            owner->memory = SUFR_B200_MEM_HOST;
            owner->text = sh[0].host_text;
            owner->text_malloc = true;
            sh[0].host_text = nullptr;
            if (sh[0].dev.num_n_ranges) {
                owner->n_ranges = (uint64_t*)malloc(sh[0].dev.num_n_ranges * 16);
                memcpy(owner->n_ranges, sh[0].dev.n_ranges, sh[0].dev.num_n_ranges * 16);
            }
            *res = sh[0].dev;
            res->memory = SUFR_B200_MEM_HOST;
            res->text = (uint8_t*)owner->text;
            res->sa = nullptr;
            res->lcp = nullptr;
            res->n_ranges = owner->n_ranges;
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
            cudaStreamSynchronize(x.ctx->stream);
            x.ctx->pinned.sizes.clear();
            x.ctx->pinned.release();
            x.ctx->pool.release_all();
            cudaStreamDestroy(x.ctx->stream);
            free(x.host_text);
        }
        if (first_err) std::rethrow_exception(first_err);
        res->owner = owner.release();
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
        std::lock_guard<std::mutex> lock(ctx->mu);
        SUFR_CUDA_CHECK(cudaSetDevice(ctx->device));
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
