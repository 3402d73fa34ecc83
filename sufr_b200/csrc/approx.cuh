// Search with mismatches (include/sufr_b200.h gives the definition): every string w of length m' = min(m, cap) that
// starts an indexed suffix and lies within k substitutions of q[0, m'), none of them onto a separator byte.
//
// Backtracking over the full suffix array, one level of depth at a time.  A node (q, d, e, [lo, hi)) is a candidate
// w[0, d) with e mismatches whose suffixes are the ranks [lo, hi).  Inside such a range the byte at offset d does not
// decrease with the rank, except that the one suffix of exactly d bytes (if any) sorts first, so each child is one run
// of equal bytes, found by a binary search over the range.  Per level:
//   count_kernel    one thread per node: its children that go on (packed low 32 bits) and that end here (high 32)
//   scan            exclusive offsets of the packed counts (scan.cuh)
//   expand_kernel   one thread per node of a slice: recomputes the children and writes them to the next level, in
//                   (query, rank) order, and the ones that end here to the finals
// A child ends here when it reaches depth m', or when its range holds a single suffix: that one is compared to the
// rest of the query at once.  The finals are put in (query, rank) order afterwards by one radix sort.
#pragma once
#include "common.cuh"
#include "search.cuh"

namespace sufr {

// The stable radix sort of (u64 key, u32 value) pairs on key bits [0, end_bit) (rsort::sort_pairs); defined in
// builder.cu, the unit that holds the sort's kernels.  Returns true when the result is in (keys_b, vals_b).
bool sort_u64_u32_pairs(uint64_t* keys_a, uint64_t* keys_b, uint32_t* vals_a, uint32_t* vals_b,
                        uint64_t n, int end_bit, uint32_t* counts, cudaStream_t stream);
size_t sort_counts_words();

namespace approx {

constexpr int BLOCK = 128;

struct Node {
    unsigned long long lo, hi;  // the ranks whose suffixes start with the candidate
    uint32_t q, d, e, m;        // query, depth, mismatches so far, m' of the query
};

struct Final {
    unsigned long long lo, hi;
    uint32_t q, e;
};

struct Params {
    const uint8_t* text;
    uint64_t n;
    const void* sa;
    int wide;
    const uint8_t* queries;
    const unsigned long long* offsets;
    uint32_t k;
    const uint32_t* sep;  // separator bytes: bit b & 31 of sep[b >> 5] (device memory: a kernel parameter indexed
                          // with a variable would be copied to the stack)
};

__device__ __forceinline__ bool is_sep(const Params& P, uint32_t b) { return (__ldg(P.sep + (b >> 5)) >> (b & 31)) & 1u; }

__device__ __forceinline__ uint32_t byte_at(const Params& P, uint64_t r, uint32_t d) {
    return P.text[search::entry(P.sa, r, P.wide) + d];
}

// The first rank in [lo, hi) whose byte at d is above b (upper) or not below b, or hi.
__device__ __forceinline__ uint64_t bound(const Params& P, uint64_t lo, uint64_t hi, uint32_t d, uint32_t b, bool upper,
                                          uint32_t& steps) {
    while (lo < hi) {
        const uint64_t mid = lo + (hi - lo) / 2;
        const uint32_t c = byte_at(P, mid, d);
        if (upper ? c <= b : c < b) lo = mid + 1;
        else hi = mid;
        steps++;
    }
    return lo;
}

// w[0, m') of the single suffix at rank r, which matches the candidate on [0, d) with e mismatches: its mismatches
// on all m' bytes, or -1 when it is no match.
__device__ __forceinline__ int finish_single(const Params& P, const uint8_t* q, uint32_t d, uint32_t e, uint32_t m,
                                             uint64_t r) {
    const uint64_t p = search::entry(P.sa, r, P.wide);
    if (p + m > P.n) return -1;
    for (uint32_t j = d; j < m; j++) {
        const uint32_t c = P.text[p + j];
        if (c != q[j] && (is_sep(P, c) || ++e > P.k)) return -1;
    }
    return (int)e;
}

// Calls next(lo, hi, e) for every child of the node that goes on to depth d + 1, and fin(lo, hi, e) for every child
// that is a match.  `steps` counts the binary-search steps.
template <typename Next, typename Fin>
__device__ __forceinline__ void visit_children(const Params& P, const Node& nd, uint32_t& steps, Next next, Fin fin) {
    uint64_t lo = nd.lo;
    const uint64_t hi = nd.hi;
    if (lo >= hi) return;
    if (search::entry(P.sa, lo, P.wide) + nd.d == P.n) lo++;  // the suffix of exactly d bytes
    const uint8_t* q = P.queries + P.offsets[nd.q];
    const uint32_t qb = q[nd.d], d1 = nd.d + 1;
    auto child = [&](uint64_t a, uint64_t b, uint32_t e) {
        if (d1 == nd.m) {
            fin(a, b, e);
        } else if (b - a == 1) {
            const int f = finish_single(P, q, d1, e, nd.m, a);
            if (f >= 0) fin(a, b, (uint32_t)f);
        } else {
            next(a, b, e);
        }
    };
    if (nd.e == P.k) {  // no mismatch left: the query's byte only
        const uint64_t a = bound(P, lo, hi, nd.d, qb, false, steps);
        const uint64_t b = bound(P, a, hi, nd.d, qb, true, steps);
        if (a < b) child(a, b, nd.e);
        return;
    }
    for (uint64_t r = lo; r < hi;) {  // one run per byte present
        const uint32_t c = byte_at(P, r, nd.d);
        const uint64_t end = bound(P, r + 1, hi, nd.d, c, true, steps);
        if (c == qb) child(r, end, nd.e);
        else if (!is_sep(P, c)) child(r, end, nd.e + 1);
        r = end;
    }
}

// Roots: the queries [first, first + count), each the node (q, 0, 0, [0, s)); an empty range for a query with m' = 0
// or m' > n.
__global__ void __launch_bounds__(256) root_kernel(const unsigned long long* __restrict__ offsets, uint64_t first,
                                                   uint64_t count, uint64_t cap, uint64_t n, uint64_t s,
                                                   Node* __restrict__ out) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const uint64_t q = first + i;
    uint64_t m = offsets[q + 1] - offsets[q];
    if (cap && m > cap) m = cap;
    Node nd;
    nd.lo = 0;
    nd.hi = (m == 0 || m > n) ? 0 : s;
    nd.q = (uint32_t)q;
    nd.d = 0;
    nd.e = 0;
    nd.m = (uint32_t)m;
    out[i] = nd;
}

// One thread per node: counts[i] = its children that go on | (its matches << 32).  stats[0] / stats[1] += the nodes
// and the binary-search steps of the level.
__global__ void __launch_bounds__(BLOCK) count_kernel(Params P, const Node* __restrict__ nodes, uint64_t count,
                                                      unsigned long long* __restrict__ counts,
                                                      unsigned long long* __restrict__ stats) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t steps = 0;
    if (i < count) {
        unsigned long long v = 0;
        visit_children(
            P, nodes[i], steps, [&](uint64_t, uint64_t, uint32_t) { v += 1; },
            [&](uint64_t, uint64_t, uint32_t) { v += 1ull << 32; });
        counts[i] = v;
    }
    const uint32_t live = __popc(__ballot_sync(0xffffffffu, i < count));
    steps = __reduce_add_sync(0xffffffffu, steps);
    if ((threadIdx.x & 31) == 0 && live) {
        atomicAdd(stats, (unsigned long long)live);
        atomicAdd(stats + 1, (unsigned long long)steps);
    }
}

// The exclusive scan of the packed counts (no carry crosses bit 32: a level holds fewer than 2^24 nodes).
struct ExclOut {
    unsigned long long* excl;
    __device__ void operator()(uint64_t i, unsigned long long v, unsigned long long incl) const { excl[i] = incl - v; }
};

// One thread per node of the slice [a, b): its children go to next + (their offset from node a), its matches to
// finals + finals_base + (their offset from node a).
__global__ void __launch_bounds__(BLOCK) expand_kernel(Params P, const Node* __restrict__ nodes,
                                                       const unsigned long long* __restrict__ excl, uint64_t a,
                                                       uint64_t b, Node* __restrict__ next, Final* __restrict__ finals,
                                                       uint64_t finals_base) {
    const uint64_t i = a + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= b) return;
    const Node nd = nodes[i];
    const unsigned long long o = excl[i], o0 = excl[a];
    uint64_t c = (uint32_t)o - (uint32_t)o0, f = finals_base + (o >> 32) - (o0 >> 32);
    uint32_t steps = 0;
    visit_children(
        P, nd, steps,
        [&](uint64_t lo, uint64_t hi, uint32_t e) {
            Node ch;
            ch.lo = lo;
            ch.hi = hi;
            ch.q = nd.q;
            ch.d = nd.d + 1;
            ch.e = e;
            ch.m = nd.m;
            next[c++] = ch;
        },
        [&](uint64_t lo, uint64_t hi, uint32_t e) {
            Final r;
            r.lo = lo;
            r.hi = hi;
            r.q = nd.q;
            r.e = e;
            finals[f++] = r;
        });
}

// Sort keys: (query << rank_bits) | rank_begin, and the index of the final.
__global__ void __launch_bounds__(256) final_keys_kernel(const Final* __restrict__ finals, uint64_t count, int rank_bits,
                                                         uint64_t* __restrict__ keys, uint32_t* __restrict__ vals) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    keys[i] = ((uint64_t)finals[i].q << rank_bits) | finals[i].lo;
    vals[i] = (uint32_t)i;
}

// The finals in sorted order: rank ranges and mismatches.
__global__ void __launch_bounds__(256) final_gather_kernel(const Final* __restrict__ finals,
                                                           const uint32_t* __restrict__ order, uint64_t count,
                                                           unsigned long long* __restrict__ begin,
                                                           unsigned long long* __restrict__ end,
                                                           unsigned long long* __restrict__ mismatches) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= count) return;
    const Final f = finals[order[j]];
    begin[j] = f.lo;
    end[j] = f.hi;
    mismatches[j] = f.e;
}

// match_offsets[q] for q <= num_queries: the sorted matches of the queries before q.
__global__ void __launch_bounds__(256) match_offsets_kernel(const uint64_t* __restrict__ keys, uint64_t count,
                                                            int rank_bits, uint64_t num_queries,
                                                            unsigned long long* __restrict__ match_offsets) {
    const uint64_t q = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q > num_queries) return;
    uint64_t lo = 0, hi = count;
    while (lo < hi) {
        const uint64_t mid = lo + (hi - lo) / 2;
        if ((keys[mid] >> rank_bits) < q) lo = mid + 1;
        else hi = mid;
    }
    match_offsets[q] = lo;
}

// The separator bytes: t[n - 1] and t[c - 1] for every sequence start c > 0, as a 256-bit mask.
__global__ void __launch_bounds__(256) separators_kernel(const uint8_t* __restrict__ text, uint64_t n,
                                                         const unsigned long long* __restrict__ starts,
                                                         uint64_t num_starts, uint32_t* __restrict__ mask) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i > num_starts) return;
    const uint64_t c = i < num_starts ? starts[i] : n;
    if (c == 0 || c > n) return;
    const uint32_t b = text[c - 1];
    atomicOr(mask + (b >> 5), 1u << (b & 31));
}

}  // namespace approx
}  // namespace sufr
