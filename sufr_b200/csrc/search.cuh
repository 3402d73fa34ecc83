// The consumer of the LCP array (SURVEY 8(f) rank 4): LCP-subsampled suffix array and batched search over a
// device-resident index.  Mirrors, for one batch of queries at a time,
//   SufrFile::subsample_suffix_array   libsufr/src/sufr_file.rs:429-456   keep (suffix, rank) where lcp < max_query_len
//   SufrSearch::search                 libsufr/src/sufr_search.rs:104-176 first / last occurrence, rank mapping
//   suffix_search_first / _last        :179-249                          binary search with LCP skipping
//   compare                            :261-350                          full / max-query-len / seed-mask comparison
// One thread per query; the reference runs one rayon task per query (sufr_file.rs:816-826).
#pragma once
#include "common.cuh"

namespace sufr {
namespace search {

struct Params {
    const uint8_t* text;
    uint64_t n;               // text length
    const void* sa;           // the array that is searched: full suffix array, or the subsampled one
    const void* rank;         // ranks of the subsampled entries in the full array (NULL: searching the full array)
    uint64_t len;             // entries of `sa`
    int wide;                 // entries are u64 (else u32)
    int is_mask;              // SuffixSortType::Mask (else MaxQueryLen(build_mql))
    uint64_t build_mql;       // max_query_len the index was built with (0 = none)
    int has_run_mql;          // a max_query_len was given at search time
    uint64_t run_mql;
    const uint32_t* mask_pos; // seed mask: offsets of the care positions
    uint32_t weight;
    uint32_t mask_len;
};

struct Comparison {
    uint64_t lcp;
    int cmp;  // query vs suffix: -1 Less, 0 Equal, 1 Greater
};

__device__ __forceinline__ uint64_t entry(const void* a, uint64_t i, int wide) {
    return wide ? reinterpret_cast<const unsigned long long*>(a)[i] : (uint64_t) reinterpret_cast<const uint32_t*>(a)[i];
}

// util.rs:19-37
__device__ __forceinline__ uint64_t full_offset(const Params& P, uint64_t lcp) {
    if (!P.is_mask || lcp == 0 || lcp > P.mask_len) return lcp;
    const uint64_t offset = P.mask_pos[lcp - 1];
    const uint64_t next_offset = lcp < P.weight ? P.mask_pos[lcp] : 0;
    if (next_offset > offset && next_offset - offset > 1) return next_offset;
    return offset + 1;
}

// sufr_search.rs:261-350
__device__ Comparison compare(const Params& P, const uint8_t* q, uint64_t qlen, uint64_t suffix_pos, uint64_t skip) {
    uint64_t lcp, mql;
    if (!P.is_mask) {
        if (P.build_mql > 0 && P.has_run_mql) mql = P.build_mql < P.run_mql ? P.build_mql : P.run_mql;
        else if (P.has_run_mql) mql = P.run_mql;
        else mql = P.build_mql;
        if (mql > 0 && skip >= mql) {
            lcp = skip;
        } else {
            const uint64_t text_start = suffix_pos + skip;
            uint64_t text_end = mql > 0 ? text_start + mql : text_start + qlen;
            if (text_end > P.n) text_end = P.n;
            uint64_t c = 0;
            while (skip + c < qlen && text_start + c < text_end && q[skip + c] == P.text[text_start + c]) c++;
            lcp = c + skip;
        }
    } else {
        mql = P.has_run_mql ? P.run_mql : 0;
        if (skip >= P.weight || (mql > 0 && skip >= mql)) {
            lcp = skip;
        } else {
            const uint64_t end = mql > 0 ? (mql < P.weight ? mql : P.weight) : P.weight;
            uint64_t query_len = 0, suffix_len = 0;
            for (uint64_t k = skip; k < end; k++) {
                if (P.mask_pos[k] < qlen) query_len++;
                if (suffix_pos + P.mask_pos[k] < P.n) suffix_len++;
            }
            const uint64_t len = query_len < suffix_len ? query_len : suffix_len;
            uint64_t c = 0;
            while (c < len) {
                const uint64_t off = P.mask_pos[skip + c];
                if (suffix_pos + off >= P.n || q[off] != P.text[suffix_pos + off]) break;
                c++;
            }
            lcp = skip + c;
        }
    }
    Comparison r;
    r.lcp = lcp;
    if (mql > 0 && lcp >= mql) {
        r.cmp = 0;  // seen enough
    } else {
        const uint64_t fo = full_offset(P, lcp);
        if (fo >= qlen) r.cmp = 0;                        // the entire query matched
        else if (suffix_pos + fo >= P.n) r.cmp = 1;       // (the reference panics here; the end of the text sorts first)
        else r.cmp = q[fo] < P.text[suffix_pos + fo] ? -1 : (q[fo] > P.text[suffix_pos + fo] ? 1 : 0);
    }
    return r;
}

// sufr_search.rs:179-213
__device__ long long search_first(const Params& P, const uint8_t* q, uint64_t qlen) {
    long long low = 0, high = (long long)P.len - 1;
    uint64_t left_lcp = 0, right_lcp = 0;
    while (high >= low) {
        const long long mid = low + (high - low) / 2;
        const uint64_t mid_val = entry(P.sa, mid, P.wide);
        const Comparison c = compare(P, q, qlen, mid_val, left_lcp < right_lcp ? left_lcp : right_lcp);
        const uint64_t before = mid > 0 ? entry(P.sa, mid - 1, P.wide) : mid_val;
        if (c.cmp == 0 && (mid == 0 || compare(P, q, qlen, before, 0).cmp == 1)) return mid;
        if (c.cmp == 1) { low = mid + 1; left_lcp = c.lcp; }
        else { high = mid - 1; right_lcp = c.lcp; }
    }
    return -1;
}

// sufr_search.rs:216-249
__device__ long long search_last(const Params& P, const uint8_t* q, uint64_t qlen, long long low) {
    const long long n = (long long)P.len;
    long long high = n - 1;
    uint64_t left_lcp = 0, right_lcp = 0;
    while (high >= low) {
        const long long mid = low + (high - low) / 2;
        const uint64_t mid_val = entry(P.sa, mid, P.wide);
        const Comparison c = compare(P, q, qlen, mid_val, left_lcp < right_lcp ? left_lcp : right_lcp);
        const uint64_t after = mid < n - 1 ? entry(P.sa, mid + 1, P.wide) : mid_val;
        if (c.cmp == 0 && (mid == n - 1 || compare(P, q, qlen, after, 0).cmp == -1)) return mid;
        if (c.cmp == -1) { high = mid - 1; right_lcp = c.lcp; }
        else { low = mid + 1; left_lcp = c.lcp; }
    }
    return -1;
}

// One thread per query.  rank_begin / rank_end = the half-open range of ranks in the FULL suffix array
// (SearchResultLocations::ranks), both ~0 when the query does not occur.
__global__ void __launch_bounds__(128) search_kernel(Params P, const uint8_t* __restrict__ queries,
                                                     const uint64_t* __restrict__ offsets, uint64_t num_queries,
                                                     unsigned long long* __restrict__ rank_begin,
                                                     unsigned long long* __restrict__ rank_end) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= num_queries) return;
    const uint8_t* q = queries + offsets[i];
    const uint64_t qlen = offsets[i + 1] - offsets[i];
    rank_begin[i] = ~0ull;
    rank_end[i] = ~0ull;
    if (P.len == 0) return;
    const long long start = search_first(P, q, qlen);
    if (start < 0) return;
    long long end = search_last(P, q, qlen, start);
    if (end < 0) end = start;
    if (!P.rank) {
        rank_begin[i] = (unsigned long long)start;
        rank_end[i] = (unsigned long long)end + 1;
    } else {  // compressed suffix array: sufr_search.rs:121-139
        rank_begin[i] = entry(P.rank, start, P.wide);
        if (start == end) rank_end[i] = (uint64_t)start == P.len - 1 ? P.len : entry(P.rank, start + 1, P.wide);
        else rank_end[i] = entry(P.rank, end, P.wide) + 1;
    }
}

// sufr_file.rs:443-453: the entries with lcp < max_query_len, and their ranks
struct SubsampleIn {
    static constexpr bool kFlags = true;  // scan.cuh: scanned with warp votes
    const void* lcp;
    int wide;
    uint64_t mql;
    __device__ uint32_t operator()(uint64_t i) const { return entry(lcp, i, wide) < mql ? 1u : 0u; }
};
struct SubsampleOut {
    const void* sa;
    int wide;
    void* out_sa;
    void* out_rank;
    __device__ void operator()(uint64_t i, uint32_t v, uint32_t incl) const {
        if (!v) return;
        if (wide) {
            reinterpret_cast<unsigned long long*>(out_sa)[incl - 1] = reinterpret_cast<const unsigned long long*>(sa)[i];
            reinterpret_cast<unsigned long long*>(out_rank)[incl - 1] = i;
        } else {
            reinterpret_cast<uint32_t*>(out_sa)[incl - 1] = reinterpret_cast<const uint32_t*>(sa)[i];
            reinterpret_cast<uint32_t*>(out_rank)[incl - 1] = (uint32_t)i;
        }
    }
};

// ---- locate (SufrFile::locate, sufr_file.rs:1132-1169) on the device: the search above, an exclusive scan of the
// per-query hit counts (hit_offsets[num_queries + 1]), then one thread per hit of a window of the total.
struct HitCountIn {
    const unsigned long long* begin;
    const unsigned long long* end;
    __device__ unsigned long long operator()(uint64_t i) const {
        return begin[i] == ~0ull || end[i] <= begin[i] ? 0ull : end[i] - begin[i];  // (ranks stay below num_suffixes)
    }
};
struct HitOffsetOut {  // offsets[0] = 0 is set by the caller
    unsigned long long* offsets;
    __device__ void operator()(uint64_t i, unsigned long long, unsigned long long incl) const { offsets[i + 1] = incl; }
};

// last index i in [0, n) with a[i] <= v, or -1 (upper_bound - 1)
__device__ __forceinline__ long long last_at_or_below(const unsigned long long* a, uint64_t n, uint64_t v) {
    uint64_t lo = 0, hi = n;
    while (lo < hi) {
        const uint64_t mid = lo + (hi - lo) / 2;
        if (a[mid] <= v) lo = mid + 1; else hi = mid;
    }
    return (long long)lo - 1;
}

// Hit h of [first, first + count): its query q (hit_offsets[q] <= h < hit_offsets[q + 1]), its rank in the full suffix
// array, the suffix, and the record holding it (sequence starts ascend; none = UINT64_MAX and the suffix itself).
// Consecutive hits of a query read consecutive suffix array entries.
__global__ void __launch_bounds__(256) hits_kernel(const void* sa, int wide, const unsigned long long* __restrict__ rank_begin,
                                                   const unsigned long long* __restrict__ hit_offsets, uint64_t num_queries,
                                                   const unsigned long long* __restrict__ starts, uint64_t num_starts,
                                                   uint64_t first, uint64_t count, unsigned long long* __restrict__ suffix,
                                                   unsigned long long* __restrict__ sequence,
                                                   unsigned long long* __restrict__ sequence_pos) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= count) return;
    const uint64_t h = first + t;
    const long long q = last_at_or_below(hit_offsets, num_queries + 1, h);
    const uint64_t rank = rank_begin[q] + (h - hit_offsets[q]);
    const uint64_t suf = entry(sa, rank, wide);
    const long long seq = num_starts ? last_at_or_below(starts, num_starts, suf) : -1;
    suffix[t] = suf;
    sequence[t] = seq < 0 ? ~0ull : (unsigned long long)seq;
    sequence_pos[t] = seq < 0 ? suf : suf - starts[seq];
}

// max over the entries of a suffix array read from a file (checked against the text length before any search):
// 16-byte loads (`a` is 16-byte aligned), the last few entries one by one
__global__ void __launch_bounds__(256) max_entry_kernel(const void* a, uint64_t len, int wide, unsigned long long* out) {
    unsigned long long m = 0;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t per = wide ? 2 : 4;  // entries per 16 bytes
    const uint4* v = reinterpret_cast<const uint4*>(a);
    for (uint64_t i = t; i < len / per; i += stride) {
        const uint4 x = v[i];
        if (wide) {
            m = max(m, ((unsigned long long)x.y << 32) | x.x);
            m = max(m, ((unsigned long long)x.w << 32) | x.z);
        } else {
            m = max(m, (unsigned long long)max(max(x.x, x.y), max(x.z, x.w)));
        }
    }
    for (uint64_t i = len / per * per + t; i < len; i += stride) m = max(m, (unsigned long long)entry(a, i, wide));
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) m = max(m, __shfl_down_sync(0xffffffffu, m, off));
    if ((threadIdx.x & 31) == 0) atomicMax(out, m);
}

}  // namespace search
}  // namespace sufr
