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
#include "context.hpp"
#include "host_io.hpp"
#include "pool.hpp"
#include "scan.cuh"
#include "search.cuh"
#include "stream_io.hpp"

using namespace sufr;

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
    // the last sufr_b200_index_locate or _mems: rank ranges and hit offsets of its queries (or MEMs), for
    // sufr_b200_index_hits and sufr_b200_index_extract
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

// With the context's lock held: uploads nq >= 1 queries (blob + offsets) and queues their search, whose rank ranges go
// to d_b / d_e.
static void launch_search(SufrB200Index* idx, const uint8_t* queries, const uint64_t* offsets, uint64_t nq, int has_mql,
                          uint64_t mql, int use_subsample, unsigned long long* d_b, unsigned long long* d_e) {
    Ctx& ctx = *idx->ctx;
    DeviceQueries dq(ctx, queries, offsets, nq);
    search::Params P{};
    P.text = idx->text;
    P.n = idx->n;
    P.sa = use_subsample ? (const void*)idx->sub_sa.get() : idx->sa;
    P.rank = use_subsample ? (const void*)idx->sub_rank.get() : nullptr;
    P.len = use_subsample ? idx->sub_len : idx->s;
    P.num_suffixes = idx->s;
    P.wide = idx->wide;
    P.is_mask = idx->is_mask;
    P.build_mql = idx->build_mql;
    P.has_run_mql = has_mql && mql > 0;  // a run-time max_query_len of 0 is no cap, on a capped index too
    P.run_mql = mql;
    P.mask_pos = idx->maskpos.get();
    P.weight = idx->weight;
    P.mask_len = idx->mask_len;
    search::search_kernel<<<(unsigned)div_up(nq, 128), 128, 0, ctx.stream>>>(P, dq.q.get(), dq.off.get(), nq, d_b, d_e);
    SUFR_KERNEL_CHECK();
}

int sufr_b200_index_search(SufrB200Index* idx, const uint8_t* queries, const uint64_t* offsets, uint64_t nq, int has_mql,
                           uint64_t mql, int use_subsample, uint64_t* rank_begin, uint64_t* rank_end) {
    return guarded([&] {
        if (!idx || !offsets || !rank_begin || !rank_end || (nq && !queries && offsets[nq])) throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
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
        CtxLock lock(ctx);
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
            launch_search(idx, queries, offsets, nq, has_mql, mql, use_sub, idx->loc_begin.get(), idx->loc_end.get());
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

// Argument checks shared by index_matching_stats and index_mems, before any device work.
static void check_matching_args(const SufrB200Index* idx, const uint8_t* queries, const uint64_t* offsets, uint64_t nq) {
    if (nq && !queries && offsets[nq]) throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
    for (uint64_t i = 0; i < nq; i++)
        if (offsets[i + 1] < offsets[i]) throw Error(SUFR_B200_ERR_ARGUMENT, "query offsets are not ascending");
    if (idx->is_mask)
        throw Error(SUFR_B200_ERR_UNSUPPORTED, "matching statistics and MEMs need an index without a seed mask: a seed-mask "
                                               "order does not sort contiguous bytes, so it has no longest match");
}

// With the context's lock held: queues matching_stats_kernel over the `total` bytes of the uploaded batch.
static void launch_matching_stats(SufrB200Index* idx, const DeviceQueries& dq, uint64_t nq, uint64_t total,
                                  unsigned long long* d_ms, unsigned long long* d_b, unsigned long long* d_e) {
    Ctx& ctx = *idx->ctx;
    search::Params P{};
    P.text = idx->text;
    P.n = idx->n;
    P.sa = idx->sa;
    P.len = idx->s;
    P.num_suffixes = idx->s;
    P.wide = idx->wide;
    P.build_mql = idx->build_mql;
    search::matching_stats_kernel<<<(unsigned)div_up(total, 128), 128, 0, ctx.stream>>>(
        P, dq.q.get(), reinterpret_cast<const unsigned long long*>(dq.off.get()), nq, total, d_ms, d_b, d_e);
    SUFR_KERNEL_CHECK();
}

int sufr_b200_index_matching_stats(SufrB200Index* idx, const uint8_t* queries, const uint64_t* offsets, uint64_t nq,
                                   uint64_t* match_len, uint64_t* rank_begin, uint64_t* rank_end) {
    return guarded([&] {
        if (!idx || !offsets) throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
        if (offsets[nq] && (!match_len || !rank_begin || !rank_end)) throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
        check_matching_args(idx, queries, offsets, nq);
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
        if (!idx || !offsets || !num_mems || !hit_offsets) throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
        if (offsets[nq] && (!mem_query || !mem_pos || !mem_len || !rank_begin || !rank_end))
            throw Error(SUFR_B200_ERR_ARGUMENT, "NULL argument");
        if (min_len == 0) throw Error(SUFR_B200_ERR_ARGUMENT, "min_len must be at least 1");
        check_matching_args(idx, queries, offsets, nq);
        const uint64_t total = offsets[nq];
        Ctx& ctx = *idx->ctx;
        CtxLock lock(ctx);
        idx->has_loc = false;
        idx->loc_begin.reset();
        idx->loc_end.reset();
        idx->loc_offsets.reset();
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
            unsigned long long count = 0;
            SUFR_CUDA_CHECK(cudaMemcpyAsync(&count, partials.get() + div_up(total, scan::CHUNK), 8, cudaMemcpyDeviceToHost,
                                            ctx.stream));
            SUFR_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
            mems = count;
            idx->loc_begin = DevBuf<unsigned long long>(ctx.pool, mems + 1);
            idx->loc_end = DevBuf<unsigned long long>(ctx.pool, mems + 1);
            // (query, position, length) of every MEM, then the byte each one starts at
            d_mem = DevBuf<unsigned long long>(ctx.pool, 4 * mems + 1);
            unsigned long long* m = d_mem.get();
            scan::scan_apply(total, in, scan::SumU64{}, search::MemOut{m + 3 * mems}, partials.get(), ctx.stream);
            if (mems) {
                search::mem_fill_kernel<<<(unsigned)div_up(mems, 256), 256, 0, ctx.stream>>>(
                    m + 3 * mems, mems, ms, ms + total, ms + 2 * total, d_off, nq, m, m + mems, m + 2 * mems,
                    idx->loc_begin.get(), idx->loc_end.get());
                SUFR_KERNEL_CHECK();
            }
        } else {
            idx->loc_begin = DevBuf<unsigned long long>(ctx.pool, 1);
            idx->loc_end = DevBuf<unsigned long long>(ctx.pool, 1);
        }
        // the MEMs take the place of locate's queries: hit offsets = exclusive scan of their occurrence counts
        idx->loc_offsets = DevBuf<unsigned long long>(ctx.pool, mems + 1);
        SUFR_CUDA_CHECK(cudaMemsetAsync(idx->loc_offsets.get(), 0, 8, ctx.stream));
        if (mems) {
            DevBuf<unsigned long long> partials(ctx.pool, scan::partials_count(mems));
            scan::inclusive_scan(mems, search::HitCountIn{idx->loc_begin.get(), idx->loc_end.get()}, scan::SumU64{},
                                 search::HitOffsetOut{idx->loc_offsets.get()}, partials.get(), ctx.stream);
            uint64_t* outs[5] = {mem_query, mem_pos, mem_len, rank_begin, rank_end};
            const unsigned long long* srcs[5] = {d_mem.get(), d_mem.get() + mems, d_mem.get() + 2 * mems,
                                                 idx->loc_begin.get(), idx->loc_end.get()};
            for (int k = 0; k < 5; k++)
                SUFR_CUDA_CHECK(cudaMemcpyAsync(outs[k], srcs[k], mems * 8, cudaMemcpyDeviceToHost, ctx.stream));
        }
        SUFR_CUDA_CHECK(cudaMemcpyAsync(hit_offsets, idx->loc_offsets.get(), (mems + 1) * 8, cudaMemcpyDeviceToHost, ctx.stream));
        SUFR_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
        *num_mems = mems;
        idx->loc_queries = mems;
        idx->loc_hits = hit_offsets[mems];
        idx->has_loc = true;
    });
}

// With the context's lock held, under which the last locate or mems wrote the state read here: refuses a window of hits
// that is not inside that call's.
static void check_hit_window(const SufrB200Index* idx, uint64_t first, uint64_t count) {
    if (!idx->has_loc)
        throw Error(SUFR_B200_ERR_ARGUMENT, "neither sufr_b200_index_locate nor sufr_b200_index_mems has been called");
    if (first > idx->loc_hits || count > idx->loc_hits - first)
        throw Error(SUFR_B200_ERR_ARGUMENT, "hit window [" + std::to_string(first) + ", +" + std::to_string(count) +
                                                ") is beyond the " + std::to_string(idx->loc_hits) + " hits of the last locate or mems");
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
        CtxLock lock(ctx);
        check_hit_window(idx, first, max_hits);
        *num_hits = 0;
        byte_offsets[0] = 0;
        if (max_hits == 0) return;
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

}  // extern "C"
