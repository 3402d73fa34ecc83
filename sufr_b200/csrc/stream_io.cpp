// The file path of libsufr_b200.so: a ring of pinned host buffers between a `.sufr` file and device memory, in both
// directions (stream_io.hpp).
#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <exception>
#include <mutex>
#include <thread>
#include <vector>

#include "common.cuh"
#include "host_io.hpp"
#include "stream_io.hpp"

namespace sufr {
namespace {

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
};

}  // namespace

// sufr_b200_index_open, the mirror of StreamWriter: host threads pread chunks of the file into the pinned slots and
// queue each slot's host->device copy on the context's stream.  A slot is refilled once the event recorded behind its
// last copy has completed, so reads, copies and the other threads' reads overlap.  Returns after a synchronise.
void upload_file_sections(int fd, const std::string& path, int device, cudaStream_t stream,
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
void stream_result_to_file(int device, cudaStream_t stream, const SufrB200Args& args, const SufrB200Result& r,
                           uint8_t** host_text) {
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
            StreamWriter sw(out, device, stream, 16u << 20, workers + 4, workers);
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

}  // namespace sufr
