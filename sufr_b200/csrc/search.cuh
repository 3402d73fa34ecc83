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
    uint64_t num_suffixes;    // entries of the full suffix array
    int wide;                 // entries are u64 (else u32)
    int is_mask;              // SuffixSortType::Mask (else MaxQueryLen(build_mql))
    uint64_t build_mql;       // max_query_len the index was built with (0 = none)
    int has_run_mql;          // a max_query_len > 0 was given at search time (0 = none, as for the subsample choice)
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
        // one sampled entry matches: the range runs to the next sampled rank, or to the end of the FULL array
        rank_begin[i] = entry(P.rank, start, P.wide);
        if (start == end) rank_end[i] = (uint64_t)start == P.len - 1 ? P.num_suffixes : entry(P.rank, start + 1, P.wide);
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

// Hit h of the last locate: its query q (hit_offsets[q] <= h < hit_offsets[q + 1]), its rank in the full suffix array,
// the suffix, and the record holding it (sequence starts ascend; -1 = none).  Consecutive hits of a query read
// consecutive suffix array entries.
struct HitLocation {
    uint64_t suffix;
    long long sequence;
};
__device__ __forceinline__ HitLocation locate_hit(const void* sa, int wide, const unsigned long long* rank_begin,
                                                  const unsigned long long* hit_offsets, uint64_t num_queries,
                                                  const unsigned long long* starts, uint64_t num_starts, uint64_t h) {
    const long long q = last_at_or_below(hit_offsets, num_queries + 1, h);
    const uint64_t rank = rank_begin[q] + (h - hit_offsets[q]);
    HitLocation r;
    r.suffix = entry(sa, rank, wide);
    r.sequence = num_starts ? last_at_or_below(starts, num_starts, r.suffix) : -1;
    return r;
}

// Hit first + t for t < count: suffix, record (none = UINT64_MAX) and position in the record (none: the suffix itself).
__global__ void __launch_bounds__(256) hits_kernel(const void* sa, int wide, const unsigned long long* __restrict__ rank_begin,
                                                   const unsigned long long* __restrict__ hit_offsets, uint64_t num_queries,
                                                   const unsigned long long* __restrict__ starts, uint64_t num_starts,
                                                   uint64_t first, uint64_t count, unsigned long long* __restrict__ suffix,
                                                   unsigned long long* __restrict__ sequence,
                                                   unsigned long long* __restrict__ sequence_pos) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= count) return;
    const HitLocation l = locate_hit(sa, wide, rank_begin, hit_offsets, num_queries, starts, num_starts, first + t);
    suffix[t] = l.suffix;
    sequence[t] = l.sequence < 0 ? ~0ull : (unsigned long long)l.sequence;
    sequence_pos[t] = l.sequence < 0 ? l.suffix : l.suffix - starts[l.sequence];
}

// ---- matching statistics and MEMs (include/sufr_b200.h gives the definitions) over the full suffix array of an index
// without a seed mask: ms[i] = the longest l <= min(m - i, cap) such that q[i, i+l) starts an indexed suffix, and the
// rank range of the suffixes it starts.

// The insertion rank of q: the first rank whose suffix does not sort before q.  search_first's binary search with LCP
// skipping, without its stop at the first equal suffix.
__device__ uint64_t search_insert(const Params& P, const uint8_t* q, uint64_t qlen) {
    long long low = 0, high = (long long)P.len - 1;
    uint64_t left_lcp = 0, right_lcp = 0;
    while (high >= low) {
        const long long mid = low + (high - low) / 2;
        const Comparison c = compare(P, q, qlen, entry(P.sa, mid, P.wide), left_lcp < right_lcp ? left_lcp : right_lcp);
        if (c.cmp == 1) { low = mid + 1; left_lcp = c.lcp; }
        else { high = mid - 1; right_lcp = c.lcp; }
    }
    return (uint64_t)low;
}

// bytes q[0, qlen) shares with the suffix at p
__device__ __forceinline__ uint64_t common_prefix(const Params& P, const uint8_t* q, uint64_t qlen, uint64_t p) {
    const uint64_t limit = qlen < P.n - p ? qlen : P.n - p;
    uint64_t c = 0;
    while (c < limit && q[c] == P.text[p + c]) c++;
    return c;
}

// One thread per byte j of the batch (total = offsets[num_queries]); its query is the last one starting at or before
// j.  The suffix sharing the longest prefix with q[i..] is a neighbour of its insertion rank r, so
// ms = max(lcp(q[i..], SA[r-1]), lcp(q[i..], SA[r])), then the range of q[i, i+ms) by search_first / search_last.
// P searches the full array (rank == NULL) with no run-time cap; P.build_mql caps the query as it caps the order.
__global__ void __launch_bounds__(128) matching_stats_kernel(Params P, const uint8_t* __restrict__ queries,
                                                             const unsigned long long* __restrict__ offsets,
                                                             uint64_t num_queries, uint64_t total,
                                                             unsigned long long* __restrict__ match_len,
                                                             unsigned long long* __restrict__ rank_begin,
                                                             unsigned long long* __restrict__ rank_end) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= total) return;
    const long long qi = last_at_or_below(offsets, num_queries + 1, j);
    const uint8_t* q = queries + j;
    uint64_t len = offsets[qi + 1] - j;
    if (P.build_mql > 0 && len > P.build_mql) len = P.build_mql;
    uint64_t ms = 0;
    if (P.len) {
        const uint64_t r = search_insert(P, q, len);
        if (r > 0) ms = common_prefix(P, q, len, entry(P.sa, r - 1, P.wide));
        if (r < P.len) {
            const uint64_t next = common_prefix(P, q, len, entry(P.sa, r, P.wide));
            if (next > ms) ms = next;
        }
    }
    match_len[j] = ms;
    rank_begin[j] = ~0ull;
    rank_end[j] = ~0ull;
    if (ms == 0) return;
    const long long first = search_first(P, q, ms);  // (>= 0: a suffix starts with q[0, ms))
    long long last = search_last(P, q, ms, first);
    if (last < 0) last = first;
    rank_begin[j] = (unsigned long long)first;
    rank_end[j] = (unsigned long long)last + 1;
}

// Byte j starts a MEM iff ms[j] >= min_len and (it starts its query or ms[j-1] <= ms[j]).
struct MemFlagIn {
    const unsigned long long* ms;
    const unsigned long long* offsets;
    uint64_t num_queries;
    uint64_t min_len;
    __device__ unsigned long long operator()(uint64_t j) const {
        if (ms[j] < min_len) return 0ull;
        if (j == 0 || ms[j - 1] <= ms[j]) return 1ull;
        return offsets[last_at_or_below(offsets, num_queries + 1, j)] == j ? 1ull : 0ull;
    }
};
// The compaction stores only where MEM incl - 1 starts (no loads between its stores, scan.cuh); mem_fill_kernel
// gathers the rest.
struct MemOut {
    unsigned long long* at;
    __device__ void operator()(uint64_t j, unsigned long long v, unsigned long long incl) const {
        if (v) at[incl - 1] = j;
    }
};

// One thread per MEM k starting at byte at[k] of the batch: its query, position in the query, length and rank range.
__global__ void __launch_bounds__(256) mem_fill_kernel(const unsigned long long* __restrict__ at, uint64_t mems,
                                                       const unsigned long long* __restrict__ ms,
                                                       const unsigned long long* __restrict__ rb,
                                                       const unsigned long long* __restrict__ re,
                                                       const unsigned long long* __restrict__ offsets,
                                                       uint64_t num_queries, unsigned long long* __restrict__ mem_query,
                                                       unsigned long long* __restrict__ mem_pos,
                                                       unsigned long long* __restrict__ mem_len,
                                                       unsigned long long* __restrict__ begin,
                                                       unsigned long long* __restrict__ end) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= mems) return;
    const uint64_t j = at[k];
    const long long q = last_at_or_below(offsets, num_queries + 1, j);
    mem_query[k] = (unsigned long long)q;
    mem_pos[k] = j - offsets[q];
    mem_len[k] = ms[j];
    begin[k] = rb[j];
    end[k] = re[j];
}

// ---- extract / list (SufrFile::extract, SufrFile::list): one thread per hit or rank computes the text region
// [src, src + len) of its entry; an inclusive scan of the lengths (ArrayIn + HitOffsetOut) gives the byte offsets of
// the entries in the output, and gather_regions_kernel copies the regions there.

// Hit first + t: the region around its suffix p in record [a, e) (include/sufr_b200.h): rel = p - a,
// start = rel - min(rel, prefix_len), end = min(rel + suffix_len, e - a); src = a + start, len = end - start.
// A suffix outside every record belongs to [0, s_0), or to [0, n) without sequence starts.
__global__ void __launch_bounds__(256) extract_regions_kernel(
    const void* sa, int wide, const unsigned long long* __restrict__ rank_begin,
    const unsigned long long* __restrict__ hit_offsets, uint64_t num_queries, const unsigned long long* __restrict__ starts,
    uint64_t num_starts, uint64_t n, uint64_t first, uint64_t count, uint64_t prefix_len, uint64_t suffix_len,
    unsigned long long* __restrict__ suffix, unsigned long long* __restrict__ sequence,
    unsigned long long* __restrict__ region_start, unsigned long long* __restrict__ region_end,
    unsigned long long* __restrict__ src, unsigned long long* __restrict__ len) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= count) return;
    const HitLocation l = locate_hit(sa, wide, rank_begin, hit_offsets, num_queries, starts, num_starts, first + t);
    const uint64_t a = l.sequence < 0 ? 0 : starts[l.sequence];
    const uint64_t e = l.sequence < 0 ? (num_starts ? starts[0] : n)
                                      : ((uint64_t)l.sequence + 1 < num_starts ? starts[l.sequence + 1] : n);
    const uint64_t rel = l.suffix - a, span = e - a;
    const uint64_t start = rel - (prefix_len < rel ? prefix_len : rel);
    const uint64_t end = suffix_len >= span - rel ? span : rel + suffix_len;  // (p < e: no overflow)
    suffix[t] = l.suffix;
    sequence[t] = l.sequence < 0 ? ~0ull : (unsigned long long)l.sequence;
    region_start[t] = start;
    region_end[t] = end;
    src[t] = a + start;
    len[t] = end - start;
}

// Rank first + t: SA[r], LCP[r] as stored, and the first min(max_len, n - SA[r]) bytes of the suffix.
__global__ void __launch_bounds__(256) list_rows_kernel(const void* sa, const void* lcp, int wide, uint64_t n, uint64_t first,
                                                        uint64_t count, uint64_t max_len,
                                                        unsigned long long* __restrict__ suffix,
                                                        unsigned long long* __restrict__ lcp_out,
                                                        unsigned long long* __restrict__ src,
                                                        unsigned long long* __restrict__ len) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= count) return;
    const uint64_t suf = entry(sa, first + t, wide);
    const uint64_t rest = n - suf;
    suffix[t] = suf;
    lcp_out[t] = entry(lcp, first + t, wide);
    src[t] = suf;
    len[t] = max_len < rest ? max_len : rest;
}

struct ArrayIn {
    const unsigned long long* a;
    __device__ unsigned long long operator()(uint64_t i) const { return a[i]; }
};

// The 16 text bytes at the 16-byte aligned address `al`.  Vector load when the whole chunk lies in
// [text, text + readable) (the text plus the padding its allocation is known to have), else byte by byte with the
// bytes outside [text, text + n) read as 0: no load leaves the text allocation, whatever its padding and alignment.
__device__ __forceinline__ unsigned __int128 load_chunk(const uint8_t* text, uint64_t n, uint64_t readable, uintptr_t al) {
    const uintptr_t base = (uintptr_t)text;
    if (al >= base && al + 16 <= base + readable) {
        const uint4 v = __ldg(reinterpret_cast<const uint4*>(al));
        return ((unsigned __int128)(((unsigned long long)v.w << 32) | v.z) << 64) | (((unsigned long long)v.y << 32) | v.x);
    }
    unsigned __int128 r = 0;
    for (int k = 0; k < 16; k++)
        if (al + k >= base && al + k < base + n) r |= (unsigned __int128)text[al + k - base] << (8 * k);
    return r;
}

// Copies t[src_i, src_i + len_i) to out + off_i for the m entries (off[0] = 0, off[i + 1] = off[i] + len_i,
// total = off[m]).  Parallel over OUTPUT bytes, so one region of tens of MB spreads over the whole GPU like millions
// of short ones: thread c owns output bytes [16c, 16c + 16) and writes them with one 16-byte store (out is 16-byte
// aligned and holds total rounded up to 16 bytes; the bytes past total are written as 0).  Its entries come from a
// binary search over the offsets, narrowed to the warp's range by two searches per warp; each run of bytes from one
// entry is two aligned 16-byte loads and a shift.
__global__ void __launch_bounds__(256) gather_regions_kernel(const uint8_t* __restrict__ text, uint64_t n, uint64_t readable,
                                                             const unsigned long long* __restrict__ src,
                                                             const unsigned long long* __restrict__ off, uint64_t m,
                                                             uint64_t total, uint8_t* __restrict__ out) {
    const uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    const uint64_t warp_first = (c - lane) * 16;
    if (warp_first >= total) return;  // (warp-uniform)
    const uint64_t warp_last = ((c - lane) + 32) * 16 < total ? ((c - lane) + 32) * 16 - 1 : total - 1;
    long long lo = 0, hi = 0;
    if (lane == 0) lo = last_at_or_below(off, m, warp_first);
    if (lane == 31) hi = last_at_or_below(off, m, warp_last);
    lo = __shfl_sync(0xffffffffu, lo, 0);
    hi = __shfl_sync(0xffffffffu, hi, 31);
    const uint64_t j0 = c * 16;
    if (j0 >= total) return;
    const uint64_t jend = j0 + 16 < total ? j0 + 16 : total;
    uint64_t i = (uint64_t)lo + (uint64_t)last_at_or_below(off + lo, (uint64_t)(hi - lo) + 1, j0);
    unsigned __int128 acc = 0;
    for (uint64_t j = j0; j < jend; i++) {
        const uint64_t o = off[i], seg_end = off[i + 1] < jend ? off[i + 1] : jend;
        if (seg_end <= j) continue;  // an empty entry
        const uint64_t s = src[i] + (j - o), seg = seg_end - j;
        const uintptr_t addr = (uintptr_t)(text + s), al = addr & ~(uintptr_t)15;
        const int sh = (int)(addr & 15);
        unsigned __int128 v = load_chunk(text, n, readable, al);
        if (sh) {
            v >>= 8 * sh;
            if (sh + seg > 16) v |= load_chunk(text, n, readable, al + 16) << (8 * (16 - sh));
        }
        if (seg < 16) v &= ((unsigned __int128)1 << (8 * seg)) - 1;
        acc |= v << (8 * (j - j0));
        j = seg_end;
    }
    uint4 w;
    w.x = (uint32_t)acc;
    w.y = (uint32_t)(acc >> 32);
    w.z = (uint32_t)(acc >> 64);
    w.w = (uint32_t)(acc >> 96);
    reinterpret_cast<uint4*>(out)[c] = w;
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
