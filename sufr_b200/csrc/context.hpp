// Host-side state shared by the build (builder.cu) and the read side (index.cu): the per-device context, the owner
// of a returned result, and the guard every C entry point runs in.
#pragma once
#include <map>
#include <mutex>
#include <new>
#include <string>
#include <utility>
#include <vector>

#include "../../include/sufr_b200.h"
#include "common.cuh"
#include "pool.hpp"

namespace sufr {

extern thread_local std::string g_last_error;

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
    bool text_malloc = false;    // host text from malloc (sufr_b200_create), not from the pinned cache
    int memory = SUFR_B200_MEM_HOST;
    void* text = nullptr;
    void* sa = nullptr;
    void* lcp = nullptr;
    uint64_t* n_ranges = nullptr;
    // kept for sufr_b200_patch_seam on device results
};

Ctx* make_ctx(int device);
// Waits for the context's stream, then frees its pinned buffers, its device pool and the stream.
void release_ctx(Ctx& ctx);
void free_owner(ResultOwner* o);

// Holds the context's lock with the context's device current on the calling thread.
class CtxLock {
   public:
    explicit CtxLock(Ctx& ctx) : lock_(ctx.mu) { SUFR_CUDA_CHECK(cudaSetDevice(ctx.device)); }

   private:
    std::lock_guard<std::mutex> lock_;
};

// Every entry point leaves the calling thread's current CUDA device as it found it (the library switches to the
// device of the context / of each shard inside; frameworks such as torch cache the current device per thread).
struct DeviceRestore {
    int prev = -1;
    DeviceRestore() { if (cudaGetDevice(&prev) != cudaSuccess) { cudaGetLastError(); prev = -1; } }
    ~DeviceRestore() { if (prev >= 0) cudaSetDevice(prev); }
};

template <typename F>
int guarded(F&& f) {
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

}  // namespace sufr
