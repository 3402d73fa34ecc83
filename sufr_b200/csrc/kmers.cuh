// k-mer counting over a device index (include/sufr_b200.h gives the definitions): the count spectrum, the distinct
// k-mers with their counts, and the count of the k-mer at every text position.
//
// Two passes.  In text order, a reverse min-scan over an "excluded byte" bitmap (record last bytes, and bytes outside
// ACGT in a DNA index) gives the next excluded byte at or after every position; a position is an occurrence when that
// byte is at least k bytes away, kept as a bitmap of n bits.  In rank order, a group starts at every rank with
// LCP[r] < k (and at rank 0); a segmented scan (GroupOp) carries the group's occurrence count, and for enumeration its
// first rank, to the group's last rank, where the three calls emit what they need.
#pragma once
#include "scan.cuh"
#include "search.cuh"

namespace sufr {
namespace kmers {

constexpr unsigned long long NONE = ~0ull;

__device__ __forceinline__ uint32_t bit(const uint32_t* words, uint64_t p) { return (words[p >> 5] >> (p & 31)) & 1u; }

// ---- text order

// Excluded-byte bitmap over P = n rounded up to 32 positions: bit p is set for p >= n - 1 (the last byte of the last
// record, and the padding) and, in a DNA index, for bytes other than ACGT.  One thread per position, one ballot per
// word; the grid covers P exactly, so every warp is whole.
__global__ void __launch_bounds__(256) excluded_kernel(const uint8_t* __restrict__ text, uint64_t n, uint64_t P, int dna,
                                                       uint32_t* __restrict__ excl) {
    const uint64_t p = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p - (threadIdx.x & 31) >= P) return;  // (warp-uniform: P is a multiple of 32)
    bool ex = p + 1 >= n;
    if (!ex && dna) {
        const uint8_t c = text[p];
        ex = !(c == 'A' || c == 'C' || c == 'G' || c == 'T');
    }
    const uint32_t w = __ballot_sync(0xffffffffu, ex);
    if ((threadIdx.x & 31) == 0) excl[p >> 5] = w;
}

// The byte before every sequence start is the last byte of a record (of [0, c_0) for the first start).
__global__ void __launch_bounds__(256) record_ends_kernel(const unsigned long long* __restrict__ starts, uint64_t num_starts,
                                                          uint32_t* __restrict__ excl) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= num_starts || starts[i] == 0) return;
    const uint64_t p = starts[i] - 1;
    atomicOr(&excl[p >> 5], 1u << (p & 31));
}

struct MinU64 {
    using T = unsigned long long;
    __host__ __device__ static T identity() { return NONE; }
    __device__ T operator()(T a, T b) const { return a < b ? a : b; }
};

// element i of the reverse scan is position p = P - 1 - i: the inclusive min is the next excluded byte at or after p
struct NextExcludedIn {
    const uint32_t* excl;
    uint64_t P;
    __device__ unsigned long long operator()(uint64_t i) const {
        const uint64_t p = P - 1 - i;
        return bit(excl, p) ? p : NONE;
    }
};
// p is an occurrence iff [p, p + k) holds no excluded byte.  A row of 32 elements is one aligned word of positions in
// descending order, so its ballot, bit-reversed, is the word (the scan covers P elements: every row is whole).
struct OccurrenceOut {
    uint32_t* occ;
    uint64_t P, k;
    __device__ void operator()(uint64_t i, unsigned long long, unsigned long long next) const {
        const uint64_t p = P - 1 - i;
        const uint32_t b = __ballot_sync(0xffffffffu, next - p >= k);  // (next >= p: every p >= n - 1 is excluded)
        if ((i & 31) == 0) occ[p >> 5] = __brev(b);
    }
};

// ---- rank order

// A segmented sum in one 64-bit word, so that the scan keeps one register pair per row and moves it with one shuffle:
//   HEAD   the scanned range holds a group start;
//   TAIL   the element (the right end of the range) is the last rank of its group;
//   count  the low CB bits: occurrences from the latest group start (or the range start) to the element;
//   start  with CB = 31 only (enumeration of a chunk of at most 2^30 ranks), bits [31, 62): the offset of the latest
//          group start from the chunk's first rank.
// A combination keeps the right operand when it holds a group start; otherwise it keeps HEAD and start from the left,
// adds the counts and takes TAIL from the right.  TAIL is meaningful only in the inclusive value of an element (a chunk
// total's right end may be padding), which is the only place it is read.
constexpr unsigned long long HEAD = 1ull << 63, TAIL = 1ull << 62;
template <int CB>
struct GroupOp {
    using T = unsigned long long;
    static constexpr T COUNT = (1ull << CB) - 1;
    static constexpr T KEEP = ~(COUNT | TAIL);  // HEAD, and the start offset when CB = 31
    __host__ __device__ static T identity() { return 0; }
    __device__ T operator()(T a, T b) const { return (b & HEAD) ? b : ((a & KEEP) | ((a & COUNT) + (b & COUNT)) | (b & TAIL)); }
};
using SpanOp = GroupOp<62>;   // spectrum and multiplicity: the count only
using ChunkOp = GroupOp<31>;  // enumeration: the count and the start offset

struct Ranks {
    const void* sa;
    const void* lcp;
    int wide;
    const uint32_t* occ;
    uint64_t s, k;
    __device__ bool head(uint64_t r) const { return r == 0 || search::entry(lcp, r, wide) < k; }
    // r is the last rank of its group
    __device__ bool tail(uint64_t r) const { return r + 1 >= s || search::entry(lcp, r + 1, wide) < k; }
    __device__ bool is_occ(uint64_t r) const { return bit(occ, search::entry(sa, r, wide)); }
};

// element i is rank lo + i; ranks at or past s (the padding of a scan rounded up to whole rows) are the identity
template <int CB>
struct GroupIn {
    Ranks R;
    uint64_t lo;
    __device__ unsigned long long operator()(uint64_t i) const {
        const uint64_t r = lo + i;
        if (r >= R.s) return 0;
        unsigned long long v = (unsigned long long)R.is_occ(r) | (R.tail(r) ? TAIL : 0ull);
        if (R.head(r)) v |= HEAD | (CB == 31 ? (unsigned long long)i << 31 : 0ull);
        return v;
    }
};

// Spectrum: at the last rank of each group with a count c >= 1, bin min(c, num_bins) - 1.  Count 1 dominates, so its
// tally is one ballot and one shared-memory atomic per row; the other counts go to a block histogram in shared memory
// for bins below SMALL_BINS, straight to `hist` above.  finish() flushes the block's nonzero entries to `hist` and adds
// the block's occurrences and maximum to `totals` = {occurrences, max}.  The scan covers s rounded up to 32 ranks, so
// every row calls the ballot whole.
constexpr int SMALL_BINS = 256;
struct SpectrumOut {
    static constexpr bool kBlockHooks = true;
    uint64_t num_bins;
    unsigned long long* hist;
    unsigned long long* totals;
    // per block: the bins of the counts >= 2 and the count-1 tally (at most one per rank of the block's 4096: u32), then
    // the occurrences and the maximum of the counts >= 2
    struct State {
        uint32_t bins[SMALL_BINS];
        uint32_t ones;
        unsigned long long occ, max;
    };
    __device__ static State& block_state() {
        __shared__ State state;
        return state;
    }
    __device__ void begin() const {
        State& st = block_state();
        for (int i = threadIdx.x; i < SMALL_BINS; i += blockDim.x) st.bins[i] = 0;
        if (threadIdx.x == 0) {
            st.ones = 0;
            st.occ = st.max = 0;
        }
        // (apply_kernel synchronises the block before its first store)
    }
    __device__ void operator()(uint64_t, unsigned long long, unsigned long long incl) const {
        State& st = block_state();
        const unsigned long long c = (incl & TAIL) ? incl & SpanOp::COUNT : 0;
        const uint32_t ones = __ballot_sync(0xffffffffu, c == 1);
        if ((threadIdx.x & 31) == 0 && ones) atomicAdd(&st.ones, (uint32_t)__popc(ones));
        if (c >= 2) {
            const uint64_t bin = (c < num_bins ? c : num_bins) - 1;
            if (bin < SMALL_BINS) atomicAdd(&st.bins[bin], 1u);
            else atomicAdd(&hist[bin], 1ull);
            atomicAdd(&st.occ, c);
            atomicMax(&st.max, c);
        }
    }
    __device__ void finish() const {
        __syncthreads();
        const State& st = block_state();
        const int bins = num_bins < SMALL_BINS ? (int)num_bins : SMALL_BINS;
        for (int i = threadIdx.x; i < bins; i += blockDim.x) {
            const unsigned long long v = (unsigned long long)st.bins[i] + (i == 0 ? st.ones : 0u);  // (count 1: bin 0)
            if (v) atomicAdd(&hist[i], v);
        }
        if (threadIdx.x == 0) {
            const unsigned long long mx = st.max ? st.max : (st.ones ? 1ull : 0ull);
            atomicAdd(&totals[0], st.ones + st.occ);
            if (mx) atomicMax(&totals[1], mx);
        }
    }
};

// Enumeration over the chunk [lo, lo + L), L <= CHUNK_MAX: incl[i] = the inclusive value of rank lo + i (at the last
// rank of a group that starts in the chunk: TAIL, HEAD, its start offset and its count).  The host takes where the
// next window starts from incl[L - 1].
constexpr uint64_t CHUNK_MAX = 1ull << 30;
struct KmerChunkOut {
    unsigned long long* incl;
    __device__ void operator()(uint64_t i, unsigned long long, unsigned long long v) const { incl[i] = v; }
};
// the complete groups of the chunk whose count lies in [min_count, max_count]
struct ListedIn {
    static constexpr bool kFlags = true;  // scan.cuh: scanned with warp votes (a chunk holds at most 2^30 ranks)
    const unsigned long long* incl;
    uint64_t min_count, max_count;
    __device__ uint32_t operator()(uint64_t i) const {
        const unsigned long long v = incl[i], c = v & ChunkOp::COUNT;
        return (v & TAIL) && (v & HEAD) && c >= min_count && c <= max_count ? 1u : 0u;
    }
};
// the first max_kmers listed groups, in rank order
struct ListedOut {
    const unsigned long long* group;  // KmerChunkOut's incl
    uint64_t lo, max_kmers;
    unsigned long long* out_begin;
    unsigned long long* out_end;
    unsigned long long* out_count;
    __device__ void operator()(uint64_t i, uint32_t v, uint32_t nth) const {
        if (!v || nth > max_kmers) return;
        const unsigned long long g = group[i];
        out_begin[nth - 1] = lo + ((g >> 31) & ChunkOp::COUNT);
        out_end[nth - 1] = lo + i + 1;
        out_count[nth - 1] = g & ChunkOp::COUNT;
    }
};

// A group longer than a chunk, starting at rank lo: its end is the first rank r > lo with LCP[r] < k (min-scan of
// BoundaryIn over a window of ranks from a), its count the occurrences among its ranks (sum of OccIn from lo).
struct BoundaryIn {
    Ranks R;
    uint64_t a;
    __device__ unsigned long long operator()(uint64_t i) const { return R.head(a + i) ? a + i : NONE; }
};
struct OccIn {
    Ranks R;
    uint64_t a;
    __device__ unsigned long long operator()(uint64_t i) const { return R.is_occ(a + i); }
};

// One thread per listed k-mer: the text position of its group's first occurrence (the group's first rank in a DNA
// index; further only past ranks whose suffix is no occurrence, in a plain index whose delimiter occurs in a record).
__global__ void __launch_bounds__(256) kmer_positions_kernel(Ranks R, const unsigned long long* __restrict__ begin,
                                                             uint64_t m, unsigned long long* __restrict__ pos) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    uint64_t r = begin[j];
    while (!R.is_occ(r)) r++;
    pos[j] = search::entry(R.sa, r, R.wide);
}

// out[j * k + o] = t[pos[j] + o]: one thread per output byte
__global__ void __launch_bounds__(256) kmer_bytes_kernel(const uint8_t* __restrict__ text,
                                                         const unsigned long long* __restrict__ pos, uint64_t k,
                                                         uint64_t total, uint8_t* __restrict__ out) {
    const uint64_t b = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= total) return;
    const uint64_t j = b / k;
    out[b] = text[pos[j] + (b - j * k)];
}

// Multiplicity, forward pass: the count of every group at its last rank, saturated to u32.
struct GroupCountOut {
    uint32_t* at_tail;
    __device__ void operator()(uint64_t r, unsigned long long, unsigned long long incl) const {
        const unsigned long long c = incl & SpanOp::COUNT;
        if (incl & TAIL) at_tail[r] = c < 0xffffffffull ? (uint32_t)c : 0xffffffffu;
    }
};
// Reverse pass: element i is rank r = s - 1 - i; a group's last rank starts a segment (HEAD) whose count is the
// group's, and the other ranks add 0, so the inclusive count at every rank of the group is the group's.
struct GroupCountIn {
    Ranks R;
    const uint32_t* at_tail;
    __device__ unsigned long long operator()(uint64_t i) const {
        const uint64_t r = R.s - 1 - i;
        return R.tail(r) ? HEAD | at_tail[r] : 0ull;
    }
};
// out[SA[r] - first] = the count, for the occurrences inside the window [first, first + num)
struct MultiplicityOut {
    Ranks R;
    uint64_t first, num;
    uint32_t* out;
    __device__ unsigned long long load(uint64_t i, unsigned long long, unsigned long long) const {
        const uint64_t r = R.s - 1 - i;
        const uint64_t p = search::entry(R.sa, r, R.wide);
        return p - first < num && bit(R.occ, p) ? p - first : NONE;
    }
    __device__ void store(uint64_t, unsigned long long, unsigned long long incl, unsigned long long at) const {
        if (at != NONE) out[at] = (uint32_t)(incl & SpanOp::COUNT);
    }
};

}  // namespace kmers
}  // namespace sufr
