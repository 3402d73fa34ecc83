// Read side of libsufr_b200.so: a device index over a build result or a `.sufr` file, batched search and locate,
// extract / list / string_at, and the `.sufr` header reader of the C ABI.
#include <fcntl.h>
#include <unistd.h>

#include <algorithm>
#include <cerrno>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "../../include/sufr_b200.h"
#include "approx.cuh"
#include "context.hpp"
#include "host_io.hpp"
#include "kmers.cuh"
#include "pool.hpp"
#include "scan.cuh"
#include "search.cuh"
#include "stream_io.hpp"

using namespace sufr;

// Refuses a batch of nq queries (blob + offsets[0..nq]) before any lock is taken or state is dropped.
static void check_queries(const uint8_t* queries, const uint64_t* offsets, uint64_t nq) {
    if (!offsets || (!queries && offsets[nq])) throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
    for (uint64_t i = 0; i < nq; i++)
        if (offsets[i + 1] < offsets[i]) throw Error(SUFR_B200_ERR_ARGUMENT, "query offsets are not ascending");
}

// With the context's lock held: the grand total a scan over n elements left in `partials`, once the stream is done.
template <typename T>
static T read_total(Ctx& ctx, T* partials, uint64_t n) {
    T total = 0;
    SUFR_CUDA_CHECK(cudaMemcpyAsync(&total, scan::total_ptr(partials, n), sizeof(T), cudaMemcpyDeviceToHost, ctx.stream));
    SUFR_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
    return total;
}

// With the context's lock held: d_off[0] = 0 and d_off[1..m] = the inclusive sums of `in` over m entries, queued.
template <typename In>
static void exclusive_offsets(Ctx& ctx, uint64_t m, In in, unsigned long long* d_off) {
    SUFR_CUDA_CHECK(cudaMemsetAsync(d_off, 0, 8, ctx.stream));
    if (!m) return;
    DevBuf<unsigned long long> partials(ctx.pool, scan::partials_count(m));
    scan::inclusive_scan(m, in, scan::SumU64{}, search::HitOffsetOut{d_off}, partials.get(), ctx.stream);
}

// With the context's lock held: the total of one reduce of `in` over n >= 1 elements.
template <typename Op, typename In>
static typename Op::T kmer_reduce(Ctx& ctx, uint64_t n, In in, Op op) {
    DevBuf<typename Op::T> partials(ctx.pool, scan::partials_count(n));
    scan::scan_reduce(n, in, op, partials.get(), ctx.stream);
    return read_total(ctx, partials.get(), n);
}

// The last sufr_b200_index_locate, _mems or _approx (`source`): rank ranges and hit offsets of its `entries` queries
// (or MEMs, or matches), for sufr_b200_index_hits and _extract, and after _approx the mismatches of its matches, for
// sufr_b200_index_approx_matches.
struct LocateState {
    DevBuf<unsigned long long> begin, end, offsets, mismatches;
    uint64_t entries = 0, hits = 0;
    enum Source { NONE, LOCATE, MEMS, APPROX } source = NONE;

    // With the context's lock held, once the call that replaces the state has queued the rank ranges of its m entries
    // into begin / end: queues their hit offsets (the exclusive scan of their occurrence counts) and passes them, on the
    // device, to copy_out, which queues the call's copies, synchronises and returns the total of the hits.  Only then
    // is the state recorded as `from`'s.
    template <typename CopyOut>
    void set(Ctx& ctx, uint64_t m, Source from, CopyOut copy_out) {
        offsets = DevBuf<unsigned long long>(ctx.pool, m + 1);
        exclusive_offsets(ctx, m, search::HitCountIn{begin.get(), end.get()}, offsets.get());
        hits = copy_out(offsets.get());
        entries = m;
        source = from;
    }
};

extern "C" {

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
    LocateState loc;
    // the separator bytes of index_approx (a 256-bit mask, made by its first call), and the nodes and binary-search
    // steps per depth of its last call
    DevBuf<uint32_t> sep;
    std::vector<unsigned long long> approx_levels;
    // DNA index: k-mers are made of ACGT only
    bool is_dna = false;
    // the k-mer occurrence bitmap of the last k-mer call (kmer_occ_k == 0: none), so that the windows of one
    // enumeration or multiplicity track do not each pass over the text again
    DevBuf<uint32_t> kmer_occ;
    uint64_t kmer_occ_k = 0;
    // each group's count at its last rank (u32 per rank) for kmer_occ_k, made by the first multiplicity window and kept
    // for the next ones; released with the bitmap when another k comes
    DevBuf<uint32_t> kmer_tail;
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
        idx->is_dna = args->is_dna;
        if (args->num_sequences && !args->sequence_starts) throw Error(SUFR_B200_ERR_ARGUMENT, "sequence_starts is NULL");
        CtxLock lock(*ctx);
        index_set_mask(*idx, *ctx, args->seed_mask, args->has_max_query_len, args->max_query_len);
        index_set_starts(*idx, *ctx, args->sequence_starts, args->num_sequences);
        *out = idx.release();
    });
}

void sufr_b200_index_free(SufrB200Index* idx) {
    if (!idx) return;
    DeviceRestore restore;
    Ctx& ctx = *idx->ctx;
    // not CtxLock: this call reports no error, and the buffers go back to the pool whatever cudaSetDevice returns
    std::lock_guard<std::mutex> lock(ctx.mu);
    cudaSetDevice(ctx.device);
    cudaStreamSynchronize(ctx.stream);
    delete idx;  // (its device buffers go back to the pool under the lock)
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
        total = read_total(ctx, partials.get(), idx->s);
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
        CtxLock lock(*idx->ctx);
        const uint64_t total = index_subsample_locked(idx, max_query_len);
        if (kept) *kept = total;
    });
}

// With the context's lock held: a batch of nq queries (blob + offsets) queued for upload to the device.
struct DeviceQueries {
    DevBuf<uint8_t> q;
    DevBuf<uint64_t> off;
    DeviceQueries(Ctx& ctx, const uint8_t* queries, const uint64_t* offsets, uint64_t nq)
        : q(ctx.pool, offsets[nq] + 8), off(ctx.pool, nq + 1) {
        if (offsets[nq]) SUFR_CUDA_CHECK(cudaMemcpyAsync(q.get(), queries, offsets[nq], cudaMemcpyHostToDevice, ctx.stream));
        SUFR_CUDA_CHECK(cudaMemcpyAsync(off.get(), offsets, (nq + 1) * 8, cudaMemcpyHostToDevice, ctx.stream));
    }
};

// The search parameters that come from the index: its full suffix array, without a run-time cap.
static search::Params search_params(const SufrB200Index* idx) {
    search::Params P{};
    P.text = idx->text;
    P.n = idx->n;
    P.sa = idx->sa;
    P.len = idx->s;
    P.num_suffixes = idx->s;
    P.wide = idx->wide;
    P.is_mask = idx->is_mask;
    P.build_mql = idx->build_mql;
    P.mask_pos = idx->maskpos.get();
    P.weight = idx->weight;
    P.mask_len = idx->mask_len;
    return P;
}

// With the context's lock held: uploads nq >= 1 queries (blob + offsets) and queues their search, whose rank ranges go
// to d_b / d_e.
static void launch_search(SufrB200Index* idx, const uint8_t* queries, const uint64_t* offsets, uint64_t nq, int has_mql,
                          uint64_t mql, int use_subsample, unsigned long long* d_b, unsigned long long* d_e) {
    Ctx& ctx = *idx->ctx;
    DeviceQueries dq(ctx, queries, offsets, nq);
    search::Params P = search_params(idx);
    if (use_subsample) {
        P.sa = idx->sub_sa.get();
        P.rank = idx->sub_rank.get();
        P.len = idx->sub_len;
    }
    P.has_run_mql = has_mql && mql > 0;  // a run-time max_query_len of 0 is no cap, on a capped index too
    P.run_mql = mql;
    search::search_kernel<<<(unsigned)div_up(nq, 128), 128, 0, ctx.stream>>>(P, dq.q.get(), dq.off.get(), nq, d_b, d_e);
    SUFR_KERNEL_CHECK();
}

int sufr_b200_index_search(SufrB200Index* idx, const uint8_t* queries, const uint64_t* offsets, uint64_t nq, int has_mql,
                           uint64_t mql, int use_subsample, uint64_t* rank_begin, uint64_t* rank_end) {
    return guarded([&] {
        if (!idx || !rank_begin || !rank_end) throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
        check_queries(queries, offsets, nq);
        if (use_subsample && !idx->has_sub) throw Error(SUFR_B200_ERR_ARGUMENT, "sufr_b200_index_subsample has not been called");
        if (nq == 0) return;
        Ctx& ctx = *idx->ctx;
        CtxLock lock(ctx);
        DevBuf<unsigned long long> d_b(ctx.pool, nq), d_e(ctx.pool, nq);
        launch_search(idx, queries, offsets, nq, has_mql, mql, use_subsample, d_b.get(), d_e.get());
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
        CtxLock lock(ctx);
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
        CtxLock lock(*ctx);
        auto idx = std::make_unique<SufrB200Index>();  // (on failure freed before the lock is released)
        idx->ctx = ctx;
        idx->n = fi.text_len;
        idx->s = fi.num_suffixes;
        idx->wide = fi.index_bits == 64;
        idx->is_dna = fi.is_dna;
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
        if (!idx || (nq && (!rank_begin || !rank_end)) || !hit_offsets) throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
        check_queries(queries, offsets, nq);
        Ctx& ctx = *idx->ctx;
        CtxLock lock(ctx);
        idx->loc = LocateState{};
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
        LocateState& loc = idx->loc;
        loc.begin = DevBuf<unsigned long long>(ctx.pool, nq + 1);
        loc.end = DevBuf<unsigned long long>(ctx.pool, nq + 1);
        if (nq) launch_search(idx, queries, offsets, nq, has_mql, mql, use_sub, loc.begin.get(), loc.end.get());
        loc.set(ctx, nq, LocateState::LOCATE, [&](const unsigned long long* d_hit_offsets) {
            if (nq) {
                SUFR_CUDA_CHECK(cudaMemcpyAsync(rank_begin, loc.begin.get(), nq * 8, cudaMemcpyDeviceToHost, ctx.stream));
                SUFR_CUDA_CHECK(cudaMemcpyAsync(rank_end, loc.end.get(), nq * 8, cudaMemcpyDeviceToHost, ctx.stream));
            }
            SUFR_CUDA_CHECK(cudaMemcpyAsync(hit_offsets, d_hit_offsets, (nq + 1) * 8, cudaMemcpyDeviceToHost, ctx.stream));
            SUFR_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
            return hit_offsets[nq];
        });
    });
}

// The refusal shared by index_matching_stats and index_mems, before any device work.
static void check_matching_args(const SufrB200Index* idx) {
    if (idx->is_mask)
        throw Error(SUFR_B200_ERR_UNSUPPORTED, "matching statistics and MEMs need an index without a seed mask: a seed-mask "
                                               "order does not sort contiguous bytes, so it has no longest match");
}

// With the context's lock held: queues matching_stats_kernel over the `total` bytes of the uploaded batch.
static void launch_matching_stats(SufrB200Index* idx, const DeviceQueries& dq, uint64_t nq, uint64_t total,
                                  unsigned long long* d_ms, unsigned long long* d_b, unsigned long long* d_e) {
    Ctx& ctx = *idx->ctx;
    search::matching_stats_kernel<<<(unsigned)div_up(total, 128), 128, 0, ctx.stream>>>(
        search_params(idx), dq.q.get(), reinterpret_cast<const unsigned long long*>(dq.off.get()), nq, total, d_ms, d_b, d_e);
    SUFR_KERNEL_CHECK();
}

int sufr_b200_index_matching_stats(SufrB200Index* idx, const uint8_t* queries, const uint64_t* offsets, uint64_t nq,
                                   uint64_t* match_len, uint64_t* rank_begin, uint64_t* rank_end) {
    return guarded([&] {
        if (!idx) throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
        check_queries(queries, offsets, nq);
        if (offsets[nq] && (!match_len || !rank_begin || !rank_end)) throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
        check_matching_args(idx);
        const uint64_t total = offsets[nq];
        if (total == 0) return;
        Ctx& ctx = *idx->ctx;
        CtxLock lock(ctx);
        DeviceQueries dq(ctx, queries, offsets, nq);
        DevBuf<unsigned long long> d_out(ctx.pool, 3 * total);
        unsigned long long* d = d_out.get();
        launch_matching_stats(idx, dq, nq, total, d, d + total, d + 2 * total);
        uint64_t* outs[3] = {match_len, rank_begin, rank_end};
        for (int k = 0; k < 3; k++)
            SUFR_CUDA_CHECK(cudaMemcpyAsync(outs[k], d + k * total, total * 8, cudaMemcpyDeviceToHost, ctx.stream));
        SUFR_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
    });
}

int sufr_b200_index_mems(SufrB200Index* idx, const uint8_t* queries, const uint64_t* offsets, uint64_t nq,
                         uint64_t min_len, uint64_t* num_mems, uint64_t* mem_query, uint64_t* mem_pos, uint64_t* mem_len,
                         uint64_t* rank_begin, uint64_t* rank_end, uint64_t* hit_offsets) {
    return guarded([&] {
        if (!idx || !num_mems || !hit_offsets) throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
        check_queries(queries, offsets, nq);
        if (offsets[nq] && (!mem_query || !mem_pos || !mem_len || !rank_begin || !rank_end))
            throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
        if (min_len == 0) throw Error(SUFR_B200_ERR_ARGUMENT, "min_len must be at least 1");
        check_matching_args(idx);
        const uint64_t total = offsets[nq];
        Ctx& ctx = *idx->ctx;
        CtxLock lock(ctx);
        idx->loc = LocateState{};
        LocateState& loc = idx->loc;
        // matching statistics of every byte, then the MEMs compacted by one scan of their flags
        uint64_t mems = 0;
        DevBuf<unsigned long long> d_ms, d_mem;
        if (total) {
            DeviceQueries dq(ctx, queries, offsets, nq);
            d_ms = DevBuf<unsigned long long>(ctx.pool, 3 * total);
            unsigned long long* ms = d_ms.get();
            launch_matching_stats(idx, dq, nq, total, ms, ms + total, ms + 2 * total);
            const auto* d_off = reinterpret_cast<const unsigned long long*>(dq.off.get());
            const search::MemFlagIn in{ms, d_off, nq, min_len};
            DevBuf<unsigned long long> partials(ctx.pool, scan::partials_count(total));
            scan::scan_reduce(total, in, scan::SumU64{}, partials.get(), ctx.stream);
            mems = read_total(ctx, partials.get(), total);
            loc.begin = DevBuf<unsigned long long>(ctx.pool, mems + 1);
            loc.end = DevBuf<unsigned long long>(ctx.pool, mems + 1);
            // (query, position, length) of every MEM, then the byte each one starts at
            d_mem = DevBuf<unsigned long long>(ctx.pool, 4 * mems + 1);
            unsigned long long* m = d_mem.get();
            scan::scan_apply(total, in, scan::SumU64{}, search::MemOut{m + 3 * mems}, partials.get(), ctx.stream);
            if (mems) {
                search::mem_fill_kernel<<<(unsigned)div_up(mems, 256), 256, 0, ctx.stream>>>(
                    m + 3 * mems, mems, ms, ms + total, ms + 2 * total, d_off, nq, m, m + mems, m + 2 * mems,
                    loc.begin.get(), loc.end.get());
                SUFR_KERNEL_CHECK();
            }
        } else {
            loc.begin = DevBuf<unsigned long long>(ctx.pool, 1);
            loc.end = DevBuf<unsigned long long>(ctx.pool, 1);
        }
        // the MEMs take the place of locate's queries
        loc.set(ctx, mems, LocateState::MEMS, [&](const unsigned long long* d_hit_offsets) {
            if (mems) {
                uint64_t* outs[5] = {mem_query, mem_pos, mem_len, rank_begin, rank_end};
                const unsigned long long* srcs[5] = {d_mem.get(), d_mem.get() + mems, d_mem.get() + 2 * mems,
                                                     loc.begin.get(), loc.end.get()};
                for (int k = 0; k < 5; k++)
                    SUFR_CUDA_CHECK(cudaMemcpyAsync(outs[k], srcs[k], mems * 8, cudaMemcpyDeviceToHost, ctx.stream));
            }
            SUFR_CUDA_CHECK(cudaMemcpyAsync(hit_offsets, d_hit_offsets, (mems + 1) * 8, cudaMemcpyDeviceToHost, ctx.stream));
            SUFR_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
            *num_mems = mems;
            return hit_offsets[mems];
        });
    });
}

// With the context's lock held, under which the last locate, mems or approx wrote the state read here: refuses a window of hits
// that is not inside that call's.
static void check_hit_window(const SufrB200Index* idx, uint64_t first, uint64_t count) {
    if (idx->loc.source == LocateState::NONE)
        throw Error(SUFR_B200_ERR_ARGUMENT, "none of sufr_b200_index_locate, _mems and _approx has been called");
    if (first > idx->loc.hits || count > idx->loc.hits - first)
        throw Error(SUFR_B200_ERR_ARGUMENT, "hit window [" + std::to_string(first) + ", +" + std::to_string(count) +
                                                ") is beyond the " + std::to_string(idx->loc.hits) +
                                                " hits of the last locate, mems or approx");
}

int sufr_b200_index_hits(SufrB200Index* idx, uint64_t first, uint64_t count, uint64_t* suffix, uint64_t* sequence,
                         uint64_t* sequence_pos) {
    return guarded([&] {
        if (!idx) throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
        Ctx& ctx = *idx->ctx;
        CtxLock lock(ctx);
        check_hit_window(idx, first, count);
        if (count == 0) return;
        DevBuf<unsigned long long> d_out(ctx.pool, 3 * count);
        unsigned long long* d_suf = d_out.get();
        search::hits_kernel<<<(unsigned)div_up(count, 256), 256, 0, ctx.stream>>>(
            idx->sa, idx->wide, idx->loc.begin.get(), idx->loc.offsets.get(), idx->loc.entries, idx->starts.get(),
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
    exclusive_offsets(ctx, m, search::ArrayIn{d_len}, d_off.get());
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
        CtxLock lock(ctx);
        check_hit_window(idx, first, max_hits);
        *num_hits = 0;
        byte_offsets[0] = 0;
        if (max_hits == 0) return;
        const uint64_t m = max_hits;
        DevBuf<unsigned long long> d_out(ctx.pool, 6 * m);
        unsigned long long* d = d_out.get();
        search::extract_regions_kernel<<<(unsigned)div_up(m, 256), 256, 0, ctx.stream>>>(
            idx->sa, idx->wide, idx->loc.begin.get(), idx->loc.offsets.get(), idx->loc.entries, idx->starts.get(),
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
        CtxLock lock(ctx);
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
            CtxLock lock(ctx);
            SUFR_CUDA_CHECK(cudaMemcpyAsync(out, idx->text + pos, k, cudaMemcpyDeviceToHost, ctx.stream));
            SUFR_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
        }
        *out_len = k;
    });
}

// ---- search with mismatches (approx.cuh)

// bits that hold v (at least 1)
static int bits_for(uint64_t v) {
    int b = 1;
    while (b < 64 && (v >> b)) b++;
    return b;
}

// Children one slice of a level may hold.  A level that has more is expanded in slices, each taken to completion
// before the next, so the search keeps at most one sliced level per depth: the budget is set so that max_depth + 2
// levels (nodes, 32 bytes, and their packed offsets, 8 bytes, each) fit in half the memory the pool and the device
// have free.  Below 2^24 (the packed counts of a level stay under 2^32).  SUFR_B200_DEBUG_APPROX_NODES=<n> sets it,
// so that tests reach the sliced path on small inputs.
static uint64_t approx_node_budget(Ctx& ctx, uint64_t max_depth) {
    if (const char* dbg = getenv("SUFR_B200_DEBUG_APPROX_NODES"))
        return std::min<uint64_t>(1ull << 22, std::max<uint64_t>(1, strtoull(dbg, nullptr, 10)));
    size_t free_b = 0, total_b = 0;
    SUFR_CUDA_CHECK(cudaMemGetInfo(&free_b, &total_b));
    const uint64_t avail = free_b + (ctx.pool.capacity() - ctx.pool.in_use());
    const uint64_t per = (sizeof(approx::Node) + 8) * (max_depth + 2);
    return std::max<uint64_t>(1024, std::min<uint64_t>(1ull << 22, avail / 2 / per));
}

// One level of the search: its nodes (all at one depth), the exclusive scan of their packed counts, and the slices
// [cuts[j], cuts[j + 1]) it is expanded in, with the scan's value at each cut.
struct ApproxLevel {
    DevBuf<approx::Node> nodes;
    uint64_t count = 0;
    uint32_t depth = 0;
    DevBuf<unsigned long long> excl;
    std::vector<uint64_t> cuts;
    std::vector<unsigned long long> at;
    size_t next = 0;
};

// With the context's lock held: every match of the queries whose offsets are d_off, unsorted, into `finals` (grown as
// needed); returns their number.  d_stats[2 d], [2 d + 1] += the nodes and search steps at depth d.
static uint64_t approx_search(SufrB200Index* idx, const approx::Params& P, const unsigned long long* d_off, uint64_t nq,
                              uint64_t max_depth, DevBuf<approx::Final>& finals, unsigned long long* d_stats) {
    Ctx& ctx = *idx->ctx;
    const uint64_t budget = approx_node_budget(ctx, max_depth);
    const uint64_t cap = idx->build_mql;
    uint64_t num_finals = 0;
    std::vector<ApproxLevel> stack;
    for (uint64_t q0 = 0; q0 < nq; q0 += budget) {  // roots: the queries, `budget` at a time
        ApproxLevel root;
        root.count = std::min(budget, nq - q0);
        root.nodes = DevBuf<approx::Node>(ctx.pool, root.count);
        approx::root_kernel<<<(unsigned)div_up(root.count, 256), 256, 0, ctx.stream>>>(d_off, q0, root.count, cap, idx->n,
                                                                                      idx->s, root.nodes.get());
        SUFR_KERNEL_CHECK();
        stack.push_back(std::move(root));
        while (!stack.empty()) {
            ApproxLevel& L = stack.back();
            if (L.cuts.empty()) {  // count the level's children, and cut it into slices of at most `budget` of them
                DevBuf<unsigned long long> counts(ctx.pool, L.count), partials(ctx.pool, scan::partials_count(L.count));
                approx::count_kernel<<<(unsigned)div_up(L.count, approx::BLOCK), approx::BLOCK, 0, ctx.stream>>>(
                    P, L.nodes.get(), L.count, counts.get(), d_stats + 2 * L.depth);
                SUFR_KERNEL_CHECK();
                L.excl = DevBuf<unsigned long long>(ctx.pool, L.count);
                scan::inclusive_scan(L.count, search::ArrayIn{counts.get()}, scan::SumU64{}, approx::ExclOut{L.excl.get()},
                                     partials.get(), ctx.stream);
                const unsigned long long total = read_total(ctx, partials.get(), L.count);
                L.cuts = {0};
                L.at = {0};
                if ((uint32_t)total > budget) {
                    std::vector<unsigned long long> h(L.count + 1);
                    SUFR_CUDA_CHECK(cudaMemcpyAsync(h.data(), L.excl.get(), L.count * 8, cudaMemcpyDeviceToHost, ctx.stream));
                    SUFR_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
                    h[L.count] = total;
                    for (uint64_t i = 1; i < L.count; i++)  // (a slice holds one node at least)
                        if ((uint32_t)h[i + 1] - (uint32_t)L.at.back() > budget) {
                            L.cuts.push_back(i);
                            L.at.push_back(h[i]);
                        }
                }
                L.cuts.push_back(L.count);
                L.at.push_back(total);
            }
            const uint64_t a = L.cuts[L.next], b = L.cuts[L.next + 1];
            const unsigned long long span = L.at[L.next + 1] - L.at[L.next];
            const uint64_t children = (uint32_t)span, matches = span >> 32;
            L.next++;
            ApproxLevel child;
            child.count = children;
            child.depth = L.depth + 1;
            if (children) child.nodes = DevBuf<approx::Node>(ctx.pool, children);
            if (num_finals + matches > finals.size()) {
                DevBuf<approx::Final> bigger(ctx.pool, std::max<uint64_t>(num_finals + matches, 2 * finals.size()));
                if (num_finals)
                    SUFR_CUDA_CHECK(cudaMemcpyAsync(bigger.get(), finals.get(), num_finals * sizeof(approx::Final),
                                                    cudaMemcpyDeviceToDevice, ctx.stream));
                finals = std::move(bigger);
            }
            if (span) {
                approx::expand_kernel<<<(unsigned)div_up(b - a, approx::BLOCK), approx::BLOCK, 0, ctx.stream>>>(
                    P, L.nodes.get(), L.excl.get(), a, b, child.nodes.get(), finals.get(), num_finals);
                SUFR_KERNEL_CHECK();
            }
            num_finals += matches;
            if (L.next + 1 == L.cuts.size()) stack.pop_back();  // (its buffers go back to the pool in stream order)
            if (children) stack.push_back(std::move(child));
        }
    }
    return num_finals;
}

int sufr_b200_index_approx(SufrB200Index* idx, const uint8_t* queries, const uint64_t* offsets, uint64_t nq,
                           uint64_t max_mismatches, uint64_t* match_offsets, uint64_t* num_hits) {
    return guarded([&] {
        if (!idx || !match_offsets || !num_hits) throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
        check_queries(queries, offsets, nq);
        if (max_mismatches > 16)
            throw Error(SUFR_B200_ERR_ARGUMENT, "max_mismatches = " + std::to_string(max_mismatches) + " is above 16");
        if (idx->is_mask)
            throw Error(SUFR_B200_ERR_UNSUPPORTED, "search with mismatches needs an index without a seed mask: a seed-mask "
                                                   "order does not sort contiguous bytes");
        const int rank_bits = bits_for(idx->s ? idx->s - 1 : 0), query_bits = bits_for(nq ? nq - 1 : 0);
        if (rank_bits + query_bits > 64)
            throw Error(SUFR_B200_ERR_ARGUMENT, std::to_string(nq) + " queries are too many for one call on " +
                                                    std::to_string(idx->s) + " suffixes: split the batch");
        uint64_t max_depth = 0;  // the longest m' that can match
        for (uint64_t i = 0; i < nq; i++) {
            uint64_t m = offsets[i + 1] - offsets[i];
            if (idx->build_mql && m > idx->build_mql) m = idx->build_mql;
            if (m <= idx->n && m > max_depth) max_depth = m;
        }
        if (max_depth > 0xFFFFFFFFull) throw Error(SUFR_B200_ERR_ARGUMENT, "a query is longer than 2^32 - 1 bytes");
        Ctx& ctx = *idx->ctx;
        CtxLock lock(ctx);
        idx->loc = LocateState{};
        LocateState& loc = idx->loc;
        idx->approx_levels.assign(2 * max_depth, 0);
        approx::Params P{};
        P.text = idx->text;
        P.n = idx->n;
        P.sa = idx->sa;
        P.wide = idx->wide;
        P.k = (uint32_t)max_mismatches;
        if (!idx->sep) {
            idx->sep = DevBuf<uint32_t>(ctx.pool, 8);
            SUFR_CUDA_CHECK(cudaMemsetAsync(idx->sep.get(), 0, 32, ctx.stream));
            approx::separators_kernel<<<(unsigned)div_up(idx->num_starts + 1, 256), 256, 0, ctx.stream>>>(
                idx->text, idx->n, idx->starts.get(), idx->num_starts, idx->sep.get());
            SUFR_KERNEL_CHECK();
        }
        P.sep = idx->sep.get();
        uint64_t matches = 0;
        DevBuf<uint64_t> keys_a, keys_b;
        DevBuf<uint32_t> vals_a, vals_b;
        bool sorted_in_b = false;
        loc.begin = DevBuf<unsigned long long>(ctx.pool, 1);  // (replaced below when there are matches)
        loc.end = DevBuf<unsigned long long>(ctx.pool, 1);
        loc.mismatches = DevBuf<unsigned long long>(ctx.pool, 1);
        if (max_depth && idx->s) {
            DeviceQueries dq(ctx, queries, offsets, nq);
            const auto* d_off = reinterpret_cast<const unsigned long long*>(dq.off.get());
            P.queries = dq.q.get();
            P.offsets = d_off;
            DevBuf<unsigned long long> d_stats(ctx.pool, 2 * max_depth);
            SUFR_CUDA_CHECK(cudaMemsetAsync(d_stats.get(), 0, 2 * max_depth * 8, ctx.stream));
            DevBuf<approx::Final> finals;
            matches = approx_search(idx, P, d_off, nq, max_depth, finals, d_stats.get());
            SUFR_CUDA_CHECK(cudaMemcpyAsync(idx->approx_levels.data(), d_stats.get(), 2 * max_depth * 8,
                                            cudaMemcpyDeviceToHost, ctx.stream));
            if (matches > 0xFFFFFFFFull)
                throw Error(SUFR_B200_ERR_UNSUPPORTED, std::to_string(matches) + " matches: more than 2^32 - 1 in one "
                                                                                 "call, split the batch");
            if (matches) {  // (query, rank_begin) order: one radix sort of the packed pair
                keys_a = DevBuf<uint64_t>(ctx.pool, matches);
                keys_b = DevBuf<uint64_t>(ctx.pool, matches);
                vals_a = DevBuf<uint32_t>(ctx.pool, matches);
                vals_b = DevBuf<uint32_t>(ctx.pool, matches);
                DevBuf<uint32_t> counts(ctx.pool, sort_counts_words());
                approx::final_keys_kernel<<<(unsigned)div_up(matches, 256), 256, 0, ctx.stream>>>(
                    finals.get(), matches, rank_bits, keys_a.get(), vals_a.get());
                SUFR_KERNEL_CHECK();
                sorted_in_b = sort_u64_u32_pairs(keys_a.get(), keys_b.get(), vals_a.get(), vals_b.get(), matches,
                                                 rank_bits + query_bits, counts.get(), ctx.stream);
                loc.begin = DevBuf<unsigned long long>(ctx.pool, matches);
                loc.end = DevBuf<unsigned long long>(ctx.pool, matches);
                loc.mismatches = DevBuf<unsigned long long>(ctx.pool, matches);
                approx::final_gather_kernel<<<(unsigned)div_up(matches, 256), 256, 0, ctx.stream>>>(
                    finals.get(), (sorted_in_b ? vals_b : vals_a).get(), matches, loc.begin.get(), loc.end.get(),
                    loc.mismatches.get());
                SUFR_KERNEL_CHECK();
            }
        }
        DevBuf<unsigned long long> d_mo(ctx.pool, nq + 1);
        approx::match_offsets_kernel<<<(unsigned)div_up(nq + 1, 256), 256, 0, ctx.stream>>>(
            (sorted_in_b ? keys_b : keys_a).get(), matches, rank_bits, nq, d_mo.get());
        SUFR_KERNEL_CHECK();
        SUFR_CUDA_CHECK(cudaMemcpyAsync(match_offsets, d_mo.get(), (nq + 1) * 8, cudaMemcpyDeviceToHost, ctx.stream));
        // the matches take the place of locate's queries
        loc.set(ctx, matches, LocateState::APPROX, [&](const unsigned long long* d_hit_offsets) {
            SUFR_CUDA_CHECK(cudaMemcpyAsync(num_hits, d_hit_offsets + matches, 8, cudaMemcpyDeviceToHost, ctx.stream));
            SUFR_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
            return *num_hits;
        });
    });
}

int sufr_b200_index_approx_matches(SufrB200Index* idx, uint64_t first, uint64_t count, uint64_t* mismatches,
                                   uint64_t* rank_begin, uint64_t* rank_end, uint64_t* hit_offsets) {
    return guarded([&] {
        if (!idx) throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
        Ctx& ctx = *idx->ctx;
        CtxLock lock(ctx);
        const LocateState& loc = idx->loc;
        if (loc.source != LocateState::APPROX)
            throw Error(SUFR_B200_ERR_ARGUMENT, "the last call that set the locate state was not sufr_b200_index_approx");
        if (first > loc.entries || count > loc.entries - first)
            throw Error(SUFR_B200_ERR_ARGUMENT, "match window [" + std::to_string(first) + ", +" + std::to_string(count) +
                                                    ") is beyond the " + std::to_string(loc.entries) + " matches");
        const std::pair<uint64_t*, const unsigned long long*> outs[3] = {
            {mismatches, loc.mismatches.get()}, {rank_begin, loc.begin.get()}, {rank_end, loc.end.get()}};
        for (const auto& o : outs)
            if (o.first && count)
                SUFR_CUDA_CHECK(cudaMemcpyAsync(o.first, o.second + first, count * 8, cudaMemcpyDeviceToHost, ctx.stream));
        if (hit_offsets)
            SUFR_CUDA_CHECK(cudaMemcpyAsync(hit_offsets, loc.offsets.get() + first, (count + 1) * 8,
                                            cudaMemcpyDeviceToHost, ctx.stream));
        SUFR_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
    });
}

int sufr_b200_index_approx_levels(SufrB200Index* idx, uint64_t max_levels, uint64_t* num_levels, uint64_t* nodes,
                                  uint64_t* steps) {
    return guarded([&] {
        if (!idx || !num_levels) throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
        CtxLock lock(*idx->ctx);
        const uint64_t levels = idx->approx_levels.size() / 2;
        for (uint64_t d = 0; d < std::min(levels, max_levels); d++) {
            if (nodes) nodes[d] = idx->approx_levels[2 * d];
            if (steps) steps[d] = idx->approx_levels[2 * d + 1];
        }
        *num_levels = levels;
    });
}

// ---- k-mers (kmers.cuh)

// Checks shared by the three k-mer calls, before any device work.
static void check_kmer_args(const SufrB200Index* idx, uint64_t k) {
    if (idx->is_mask)
        throw Error(SUFR_B200_ERR_UNSUPPORTED, "k-mers need an index without a seed mask: a seed-mask order does not "
                                               "sort contiguous bytes, so equal k-mers are not adjacent in it");
    if (k == 0) throw Error(SUFR_B200_ERR_ARGUMENT, "k must be at least 1");
    if (idx->build_mql && k > idx->build_mql)
        throw Error(SUFR_B200_ERR_ARGUMENT, "k = " + std::to_string(k) + " is above the max_query_len " +
                                                std::to_string(idx->build_mql) +
                                                " the index was built with: LCP values above it are not exact");
}

// With the context's lock held: the occurrence bitmap of k (bit p of word p / 32: position p is a k-mer occurrence),
// made by a pass over the text unless the last k-mer call left it for the same k.
static const uint32_t* kmer_occurrences(SufrB200Index* idx, uint64_t k) {
    if (idx->kmer_occ_k == k) return idx->kmer_occ.get();
    Ctx& ctx = *idx->ctx;
    idx->kmer_occ.reset();
    idx->kmer_tail.reset();
    idx->kmer_occ_k = 0;
    const uint64_t P = div_up(idx->n, 32) * 32;
    DevBuf<uint32_t> excl(ctx.pool, P / 32 + 1), occ(ctx.pool, P / 32 + 1);
    if (P) {
        kmers::excluded_kernel<<<(unsigned)div_up(P, 256), 256, 0, ctx.stream>>>(idx->text, idx->n, P, idx->is_dna,
                                                                                  excl.get());
        SUFR_KERNEL_CHECK();
        if (idx->num_starts) {
            kmers::record_ends_kernel<<<(unsigned)div_up(idx->num_starts, 256), 256, 0, ctx.stream>>>(
                idx->starts.get(), idx->num_starts, excl.get());
            SUFR_KERNEL_CHECK();
        }
        DevBuf<unsigned long long> partials(ctx.pool, scan::partials_count(P));
        scan::inclusive_scan(P, kmers::NextExcludedIn{excl.get(), P}, kmers::MinU64{},
                             kmers::OccurrenceOut{occ.get(), P, k}, partials.get(), ctx.stream);
    }
    idx->kmer_occ = std::move(occ);
    idx->kmer_occ_k = k;
    return idx->kmer_occ.get();
}

static kmers::Ranks kmer_ranks(SufrB200Index* idx, uint64_t k) {
    return kmers::Ranks{idx->sa, idx->lcp, idx->wide, kmer_occurrences(idx, k), idx->s, k};
}

int sufr_b200_index_kmer_spectrum(SufrB200Index* idx, uint64_t k, uint64_t num_bins, uint64_t* histogram,
                                  uint64_t* distinct, uint64_t* occurrences, uint64_t* max_count) {
    return guarded([&] {
        if (!idx || !histogram) throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
        check_kmer_args(idx, k);
        if (num_bins < 1 || num_bins > 65536)
            throw Error(SUFR_B200_ERR_ARGUMENT, "num_bins = " + std::to_string(num_bins) + " is not in [1, 65536]");
        Ctx& ctx = *idx->ctx;
        CtxLock lock(ctx);
        DevBuf<unsigned long long> d_out(ctx.pool, num_bins + 2);  // histogram, then occurrences and the maximum
        unsigned long long* d = d_out.get();
        SUFR_CUDA_CHECK(cudaMemsetAsync(d, 0, (num_bins + 2) * 8, ctx.stream));
        if (idx->s) {
            const kmers::Ranks R = kmer_ranks(idx, k);
            const uint64_t rows = div_up(idx->s, 32) * 32;  // (whole rows: SpectrumOut votes per row)
            DevBuf<unsigned long long> partials(ctx.pool, scan::partials_count(rows));
            scan::inclusive_scan(rows, kmers::GroupIn<62>{R, 0}, kmers::SpanOp{},
                                 kmers::SpectrumOut{num_bins, d, d + num_bins}, partials.get(), ctx.stream);
        }
        std::vector<uint64_t> totals(2);
        SUFR_CUDA_CHECK(cudaMemcpyAsync(histogram, d, num_bins * 8, cudaMemcpyDeviceToHost, ctx.stream));
        SUFR_CUDA_CHECK(cudaMemcpyAsync(totals.data(), d + num_bins, 16, cudaMemcpyDeviceToHost, ctx.stream));
        SUFR_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
        uint64_t sum = 0;
        for (uint64_t i = 0; i < num_bins; i++) sum += histogram[i];
        if (distinct) *distinct = sum;
        if (occurrences) *occurrences = totals[0];
        if (max_count) *max_count = totals[1];
    });
}

// With the context's lock held: the group that starts at rank lo and runs at least to rank a - 1 (longer than an
// enumeration chunk).  Its end is the first rank at or after a that starts a group, or s, found in windows that double
// from a - lo ranks, so the search costs time in proportion to the group; its count is one sum over its ranks.
static void kmer_long_group(SufrB200Index* idx, const kmers::Ranks& R, uint64_t lo, uint64_t a, uint64_t& end,
                            uint64_t& count) {
    Ctx& ctx = *idx->ctx;
    end = idx->s;
    for (uint64_t w = a - lo; a < idx->s; a += w, w *= 2) {
        w = std::min(w, idx->s - a);
        const unsigned long long e = kmer_reduce(ctx, w, kmers::BoundaryIn{R, a}, kmers::MinU64{});
        if (e != kmers::NONE) {
            end = e;
            break;
        }
    }
    count = kmer_reduce(ctx, end - lo, kmers::OccIn{R, lo}, scan::SumU64{});
}

int sufr_b200_index_kmers(SufrB200Index* idx, uint64_t k, uint64_t min_count, uint64_t max_count, uint64_t first_rank,
                          uint64_t max_kmers, uint64_t* num_kmers, uint64_t* next_rank, uint64_t* rank_begin,
                          uint64_t* rank_end, uint64_t* count, uint8_t* bytes) {
    return guarded([&] {
        if (!idx || !num_kmers || !next_rank || (max_kmers && (!rank_begin || !rank_end || !count)))
            throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
        check_kmer_args(idx, k);
        if (min_count > max_count)
            throw Error(SUFR_B200_ERR_ARGUMENT, "min_count " + std::to_string(min_count) + " is above max_count " +
                                                    std::to_string(max_count));
        const uint64_t s = idx->s;
        if (first_rank > s)
            throw Error(SUFR_B200_ERR_ARGUMENT, "first_rank " + std::to_string(first_rank) + " is beyond the " +
                                                    std::to_string(s) + " suffixes");
        *num_kmers = 0;
        *next_rank = first_rank;
        if (first_rank == s || max_kmers == 0) return;
        Ctx& ctx = *idx->ctx;
        CtxLock lock(ctx);
        const kmers::Ranks R = kmer_ranks(idx, k);
        const uint64_t lo = first_rank, lo_count = min_count ? min_count : 1;  // (a group without occurrences is no k-mer)
        // a chunk of ranks from lo, cut after its last complete group: twice max_kmers ranks hold max_kmers groups or
        // cover twice the ranks the window lists, so a window costs time in proportion to the ranks it covers
        const uint64_t L = std::min({s - lo, std::max<uint64_t>(max_kmers < s ? 2 * max_kmers : s, 1u << 16),
                                     kmers::CHUNK_MAX});
        DevBuf<unsigned long long> d_listed(ctx.pool, L), partials(ctx.pool, scan::partials_count(L));
        DevBuf<uint32_t> listed_partials(ctx.pool, scan::partials_count(L));
        scan::inclusive_scan(L, kmers::GroupIn<31>{R, lo}, kmers::ChunkOp{},
                             kmers::KmerChunkOut{d_listed.get()},
                             partials.get(), ctx.stream);
        const kmers::ListedIn listed_in{d_listed.get(), lo_count, max_count};
        scan::scan_reduce(L, listed_in, scan::SumU32{}, listed_partials.get(), ctx.stream);
        uint32_t listed = 0;
        uint64_t tail_next = 0;
        SUFR_CUDA_CHECK(cudaMemcpyAsync(&listed, scan::total_ptr(listed_partials.get(), L), 4, cudaMemcpyDeviceToHost,
                                        ctx.stream));
        unsigned long long last = 0;
        SUFR_CUDA_CHECK(cudaMemcpyAsync(&last, d_listed.get() + L - 1, 8, cudaMemcpyDeviceToHost, ctx.stream));
        SUFR_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
        // where the next window starts if every group of the chunk is listed: lo + L when the chunk ends at a group
        // boundary or holds no group start, else the start of the group it cuts
        tail_next = ((last & kmers::TAIL) || !(last & kmers::HEAD)) ? lo + L : lo + ((last >> 31) & kmers::ChunkOp::COUNT);
        uint64_t m = 0, next = tail_next;
        DevBuf<unsigned long long> d_out;
        if (tail_next == lo) {  // the group that starts at lo runs past the chunk (lo + L < s: rank s - 1 ends a group)
            uint64_t e, c;
            kmer_long_group(idx, R, lo, lo + L, e, c);
            next = e;
            if (c >= lo_count && c <= max_count) {
                m = 1;
                rank_begin[0] = lo;
                rank_end[0] = e;
                count[0] = c;
                d_out = DevBuf<unsigned long long>(ctx.pool, 1);
                SUFR_CUDA_CHECK(cudaMemcpyAsync(d_out.get(), rank_begin, 8, cudaMemcpyHostToDevice, ctx.stream));
            }
        } else if (listed) {
            m = std::min<uint64_t>(listed, max_kmers);
            d_out = DevBuf<unsigned long long>(ctx.pool, 3 * m);
            unsigned long long* o = d_out.get();
            scan::scan_apply(L, listed_in, scan::SumU32{}, kmers::ListedOut{d_listed.get(), lo, m, o, o + m, o + 2 * m},
                             listed_partials.get(), ctx.stream);
            uint64_t* outs[3] = {rank_begin, rank_end, count};
            for (int j = 0; j < 3; j++)
                SUFR_CUDA_CHECK(cudaMemcpyAsync(outs[j], o + j * m, m * 8, cudaMemcpyDeviceToHost, ctx.stream));
        }
        DevBuf<unsigned long long> d_pos;
        DevBuf<uint8_t> d_bytes;
        if (m && bytes) {  // d_out starts with the groups' first ranks
            d_pos = DevBuf<unsigned long long>(ctx.pool, m);
            kmers::kmer_positions_kernel<<<(unsigned)div_up(m, 256), 256, 0, ctx.stream>>>(R, d_out.get(), m, d_pos.get());
            SUFR_KERNEL_CHECK();
            const uint64_t total = m * k;
            d_bytes = DevBuf<uint8_t>(ctx.pool, total);
            kmers::kmer_bytes_kernel<<<(unsigned)div_up(total, 256), 256, 0, ctx.stream>>>(idx->text, d_pos.get(), k,
                                                                                            total, d_bytes.get());
            SUFR_KERNEL_CHECK();
            SUFR_CUDA_CHECK(cudaMemcpyAsync(bytes, d_bytes.get(), total, cudaMemcpyDeviceToHost, ctx.stream));
        }
        SUFR_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
        if (listed > max_kmers && tail_next != lo) next = rank_end[m - 1];
        *num_kmers = m;
        *next_rank = next;
    });
}

int sufr_b200_index_kmer_multiplicity(SufrB200Index* idx, uint64_t k, uint64_t first_pos, uint64_t num_positions,
                                      uint32_t* out) {
    return guarded([&] {
        if (!idx || (num_positions && !out)) throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
        check_kmer_args(idx, k);
        if (first_pos > idx->n || num_positions > idx->n - first_pos)
            throw Error(SUFR_B200_ERR_ARGUMENT, "position window [" + std::to_string(first_pos) + ", +" +
                                                    std::to_string(num_positions) + ") is beyond the text length " +
                                                    std::to_string(idx->n));
        if (num_positions == 0) return;
        Ctx& ctx = *idx->ctx;
        CtxLock lock(ctx);
        DevBuf<uint32_t> d_out(ctx.pool, num_positions);
        SUFR_CUDA_CHECK(cudaMemsetAsync(d_out.get(), 0, num_positions * 4, ctx.stream));
        if (idx->s) {
            const kmers::Ranks R = kmer_ranks(idx, k);
            DevBuf<unsigned long long> partials(ctx.pool, scan::partials_count(idx->s));
            // each group's count at its last rank, once per k (the windows of a track share it) ...
            if (!idx->kmer_tail.get()) {
                DevBuf<uint32_t> at_tail(ctx.pool, idx->s);
                scan::inclusive_scan(idx->s, kmers::GroupIn<62>{R, 0}, kmers::SpanOp{}, kmers::GroupCountOut{at_tail.get()},
                                     partials.get(), ctx.stream);
                idx->kmer_tail = std::move(at_tail);
            }
            // ... then back over the group and out to the text positions in the window
            scan::inclusive_scan(idx->s, kmers::GroupCountIn{R, idx->kmer_tail.get()}, kmers::SpanOp{},
                                 kmers::MultiplicityOut{R, first_pos, num_positions, d_out.get()}, partials.get(),
                                 ctx.stream);
        }
        SUFR_CUDA_CHECK(cudaMemcpyAsync(out, d_out.get(), num_positions * 4, cudaMemcpyDeviceToHost, ctx.stream));
        SUFR_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
    });
}

}  // extern "C"
