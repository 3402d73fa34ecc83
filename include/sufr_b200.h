/*
 * sufr_b200.h -- C ABI of the B200-native suffix-array / LCP-array constructor.
 *
 * Drop-in boundary for ONE path of TravisWheelerLab/sufr (v0.7.12): libsufr's `create`
 * (`SufrBuilder::<T>::new`, libsufr/src/sufr_builder.rs:143-220, called from
 * `SuffixArray::write`, libsufr/src/suffix_array.rs:460-470, and `sufr::create`,
 * sufr/src/lib.rs:321-371).  Everything here is plain C: pointers, sizes, no CUDA or torch types.
 * A Rust host binds these symbols from an `extern "C"` block (INTEGRATION.md shows the shim).
 *
 * Results are bit-exact with the reference for the SA and LCP arrays, u32 and u64 index widths
 * (see DESIGN.md for the two cases where the reference itself is not a function of its input).
 * There is no CPU fallback: every entry point that computes fails with an error when no CUDA
 * device is available.
 */
#ifndef SUFR_B200_H
#define SUFR_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SUFR_B200_ABI_VERSION 2

/* Return codes. */
#define SUFR_B200_OK 0
#define SUFR_B200_ERR_ARGUMENT 1      /* the reference's `bail!` argument errors, same message text */
#define SUFR_B200_ERR_OUT_OF_MEMORY 2
#define SUFR_B200_ERR_INTERNAL 3
#define SUFR_B200_ERR_IO 4            /* "{filename}: {io error}" (sufr_builder.rs:820) */
#define SUFR_B200_ERR_UNSUPPORTED 5
#define SUFR_B200_ERR_CUDA 100        /* 100 + cudaError_t */

/* Where a buffer lives. */
#define SUFR_B200_MEM_HOST 0
#define SUFR_B200_MEM_DEVICE 1

/* Per-device context: one CUDA stream and one device memory pool.  One context per GPU per process. */
typedef struct SufrB200Ctx SufrB200Ctx;

/*
 * Mirrors `SufrBuilderArgs` (libsufr/src/types.rs:527-582) field by field.  Options become a
 * presence flag + value (max_query_len) or a nullable pointer (path, seed_mask).
 */
typedef struct SufrB200Args {
    const uint8_t* text;          /* types.rs:530  raw text bytes; borrowed for the call */
    uint64_t text_len;
    const char* path;             /* types.rs:533  NULL = None ("out.sufr" when a file is written) */
    uint8_t low_memory;           /* types.rs:536  accepted and ignored, like the reference builder */
    uint8_t has_max_query_len;    /* types.rs:540  Option tag */
    uint8_t is_dna;               /* types.rs:546 */
    uint8_t allow_ambiguity;      /* types.rs:550 */
    uint8_t ignore_softmask;      /* types.rs:554 */
    uint8_t reserved[3];
    uint64_t max_query_len;
    const uint64_t* sequence_starts;   /* types.rs:558 */
    const char* const* sequence_names; /* types.rs:562  num_sequences NUL-terminated UTF-8 strings */
    uint64_t num_sequences;
    uint64_t num_partitions;      /* types.rs:573  accepted; does not change the result (DESIGN.md) */
    const char* seed_mask;        /* types.rs:577  NULL = None, else "1101..." */
    uint64_t random_seed;         /* types.rs:581  accepted; does not change the result */
    /* Sharding, one process per GPU: this call builds key-range shard `rank` of `world_size`.
     * Single GPU: rank 0, world_size 1. */
    int32_t rank;
    int32_t world_size;
} SufrB200Args;

/* Phase timings measured with CUDA events on the context's stream (milliseconds). */
typedef struct SufrB200Timings {
    double h2d_ms;        /* host -> device copy of the text (0 when the text was already resident) */
    double encode_ms;     /* text transform, alphabet, packing, N-run scan   (sufr_builder.rs:144-195) */
    double keys_ms;       /* first key word of every suffix + shard selection (partition assignment, :404-487) */
    double sort_ms;       /* radix sort of (key, position)                    (sort, :495-598) */
    double refine_ms;     /* equal-key groups: next-word / prefix-doubling refinement (merge compares, :634-767) */
    double lcp_ms;        /* LCP values not already produced by the sort      (find_lcp, :268-334) */
    double finish_ms;     /* N-run tie rule, suffix filter, widening          (:446-449, :305-307) */
    double d2h_ms;        /* device -> host copy of text / SA / LCP (0 for device results) */
    double total_ms;      /* first kernel to last kernel, excluding h2d/d2h */
    /* The dominant kernel (radix-sort downsweep of the main sort), timed per launch with CUDA events: */
    double dominant_kernel_ms;        /* sum over its launches in this build */
    uint64_t dominant_kernel_launches;
    uint64_t dominant_kernel_bytes;   /* algorithmic bytes of ONE launch: elements x 2 x (8 B key + 4 B position) */
} SufrB200Timings;

typedef struct SufrB200Result {
    uint32_t index_bits;      /* 32 or 64: width of the SA / LCP elements */
    uint32_t memory;          /* SUFR_B200_MEM_HOST (pinned) or SUFR_B200_MEM_DEVICE */
    uint64_t text_len;
    uint64_t num_suffixes;    /* suffixes in THIS shard (== total_suffixes when world_size == 1) */
    uint64_t total_suffixes;  /* SufrBuilder.num_suffixes over all shards.  Sharded full sorts balance the shards on a */
    uint64_t shard_offset;    /*   sampled histogram: then these two are (num_suffixes, 0) and the CALLER overwrites them with */
                              /*   the sum / prefix sum of the ranks' num_suffixes (the same exchange the seam repair needs) */
    uint64_t first_suffix;    /* SA[0] / SA[num_suffixes-1] of this shard: inputs of the seam repair */
    uint64_t last_suffix;     /*   (sufr_builder.rs:893-902); undefined when num_suffixes == 0 */
    uint8_t* text;            /* transformed text (SufrBuilder.text), text_len bytes; NULL in HOST results of ranks > 0 */
    void* sa;                 /* num_suffixes elements of index_bits */
    void* lcp;                /* num_suffixes elements; lcp[0] of shard > 0 needs sufr_b200_patch_seam */
    uint64_t* n_ranges;       /* host: num_n_ranges pairs [start, end) (SufrBuilder.n_ranges) */
    uint64_t num_n_ranges;
    SufrB200Timings timings;
    uint64_t kernel_launches; /* kernels launched by this build */
    uint64_t peak_device_bytes;
    uint32_t alphabet_size;   /* distinct bytes in the transformed text */
    uint32_t bits_per_symbol;
    uint32_t refine_rounds;   /* next-word refinement rounds */
    uint32_t doubling_rounds; /* prefix-doubling rounds (0 unless the text has deep repeats) */
    uint64_t h2d_bytes;       /* bytes this build copied host -> device (0 for a device-resident text) */
    uint64_t d2h_bytes;       /* bytes it copied device -> host: large host results travel compactly (LCP as */
                              /*   bytes + exceptions, 64-bit SA as u32) and are widened by host threads */
    uint32_t position_bits;   /* width of text positions INSIDE the build: 32, or 64 for texts of u32::MAX bytes and */
    uint32_t reserved2;       /*   more (suffix_array.rs:460-470; SUFR_B200_DEBUG_POS64 forces 64 on short texts) */
    void* owner;              /* internal */
} SufrB200Result;

/* -- context ------------------------------------------------------------------------------- */
int sufr_b200_ctx_create(int device, SufrB200Ctx** out);
void sufr_b200_ctx_destroy(SufrB200Ctx* ctx);
/* Pre-size the device memory pool for texts of up to `text_len` bytes (optional). */
int sufr_b200_ctx_reserve(SufrB200Ctx* ctx, uint64_t text_len, uint32_t index_bits);
/* Give pooled device memory that holds no live result back to the driver. */
void sufr_b200_ctx_trim(SufrB200Ctx* ctx);

/* -- build: replaces SufrBuilder::<u32>::new / SufrBuilder::<u64>::new up to (not including) write()
 *    (sufr_builder.rs:143-217).  `text_memory` says where args->text lives, `result_memory` where the
 *    outputs should be left.  index_bits: 32, 64, or 0 = the reference's dispatch
 *    (u32 iff text_len < u32::MAX, suffix_array.rs:460-470). */
int sufr_b200_build(SufrB200Ctx* ctx, const SufrB200Args* args, uint32_t index_bits, int text_memory,
                    int result_memory, SufrB200Result* out);
void sufr_b200_result_free(SufrB200Ctx* ctx, SufrB200Result* result);

/* Seam repair between shards (sufr_builder.rs:893-902): sets lcp[0] of this shard to the LCP of
 * (`prev_last_suffix`, first_suffix).  No-op for an empty shard. */
int sufr_b200_patch_seam(SufrB200Ctx* ctx, const SufrB200Args* args, SufrB200Result* result,
                         uint64_t prev_last_suffix);

/* -- verify: full check of a finished DEVICE result against the transformed text, independent of the data
 *    structures of the build (sufr_b200/csrc/verify.cuh): every SA entry is an indexed position
 *    (sufr_builder.rs:446-449) and none occurs twice; EVERY adjacent pair is in the order the mode defines and
 *    every LCP value is the mode's value (full sort; N-run rule :305-307, :701-712; --max-query-len; seed mask).
 *    Sharded builds: every rank verifies its shard, `has_prev` / `prev_last_suffix` add the seam pair.
 *    The result is correct iff all error counters are 0 and the ranks' num_suffixes sum to expected_suffixes. */
typedef struct SufrB200VerifyReport {
    uint64_t pairs_checked;     /* adjacent pairs compared (num_suffixes - 1, + 1 with has_prev) */
    uint64_t order_errors;
    uint64_t lcp_errors;
    uint64_t out_of_range;      /* SA entries >= text_len */
    uint64_t not_indexed;       /* SA entries the reference would not index */
    uint64_t duplicates;        /* positions that occur more than once in this array */
    uint64_t first_bad_rank;    /* smallest rank with an order / LCP error, UINT64_MAX if none */
    uint64_t max_lcp;
    uint64_t lcp_sum;
    uint64_t expected_suffixes; /* positions of the text the reference indexes */
    uint64_t deferred_pairs;    /* pairs sharing >= 2048 bytes: settled by a second pass, see method */
    uint32_t method;            /* 0 direct comparison only; 1 deferred pairs compared directly without a bound;
                                   2 deferred pairs by successor ranks (inverse suffix array) + Kasai LCP in text order */
    uint32_t reserved;
    double ms;                  /* device time of the check */
} SufrB200VerifyReport;
int sufr_b200_verify(SufrB200Ctx* ctx, const SufrB200Args* args, const SufrB200Result* result, int has_prev,
                     uint64_t prev_last_suffix, SufrB200VerifyReport* out);

/* -- the consumer of the LCP array (SURVEY 8(f) rank 4): LCP-subsampled suffix array + batched search over a
 *    device-resident index.  An index made by index_create borrows text / SA / LCP of a DEVICE result, which must
 *    outlive it; one made by index_open (below) owns copies read from a `.sufr` file.
 *      subsample  SufrFile::subsample_suffix_array (sufr_file.rs:429-456): the entries with lcp < max_query_len and
 *                 their ranks ("compressed" in-memory suffix array)
 *      search     SufrSearch::search (sufr_search.rs:104-350) for a batch of queries, one GPU thread per query:
 *                 queries = concatenated bytes, offsets[num_queries + 1], ascending (SUFR_B200_ERR_ARGUMENT "query
 *                 offsets are not ascending" otherwise, as in every call that takes a batch);
 *                 has/max_query_len = the run-time `-m` (a max_query_len of 0 is no run-time cap, also on an index
 *                 built with one);
 *                 use_subsample != 0 searches the subsampled array and maps the hits back through the ranks.
 *                 rank_begin / rank_end (host, num_queries each) = half-open rank range in the full suffix array
 *                 (SearchResultLocations::ranks), both UINT64_MAX when the query does not occur; count = end - begin.
 *      suffixes   SA[rank_begin .. rank_begin + count) as u64 (what `locate` reports), host output. */
typedef struct SufrB200Index SufrB200Index;
int sufr_b200_index_create(SufrB200Ctx* ctx, const SufrB200Args* args, const SufrB200Result* device_result,
                           SufrB200Index** out);
int sufr_b200_index_subsample(SufrB200Index* index, uint64_t max_query_len, uint64_t* kept);
int sufr_b200_index_search(SufrB200Index* index, const uint8_t* queries, const uint64_t* offsets, uint64_t num_queries,
                           int has_max_query_len, uint64_t max_query_len, int use_subsample, uint64_t* rank_begin,
                           uint64_t* rank_end);
int sufr_b200_index_suffixes(SufrB200Index* index, uint64_t rank_begin, uint64_t count, uint64_t* out);
void sufr_b200_index_free(SufrB200Index* index);

/* -- the read side of a `.sufr` file (SufrFile::read, sufr_file.rs:145-275), version 6 only.
 *    file_info  header, sequence starts, seed mask and names, validated (host only, no device needed): the sections
 *               must follow each other without gaps up to exactly the end of the file, element width 4 or 8
 *               ((lcp_pos - sa_pos) / num_suffixes), num_suffixes <= text_len, sequence starts strictly increasing
 *               and below text_len, mask bytes 0 / 1 forming a valid mask.  A file that fails a check gives
 *               SUFR_B200_ERR_IO ("{path}: invalid .sufr file: ..."); a version other than 6 SUFR_B200_ERR_UNSUPPORTED.
 *    index_open an index that OWNS device copies of text, suffix array, LCP array and sequence starts (host threads
 *               pread the file into pinned buffers that are copied to the device as they fill).  Every suffix array
 *               entry is checked to be below text_len on the device before the index is returned.
 *    index_locate  index_search + per-query hit offsets: hit_offsets[num_queries + 1] (exclusive scan of the counts).
 *               low_memory == 0 searches the LCP-subsampled array when the effective max_query_len is shorter than
 *               the build's (sufr_file.rs:514-560; the subsample is made and kept as needed, replacing one of
 *               another max_query_len that index_subsample made), low_memory != 0 the full array.  Ranges and offsets stay on the device for index_hits.
 *    index_hits hits [first_hit, first_hit + count) of the last index_locate or index_mems (below), in query order and
 *               rank order within a query (after index_mems, MEM order and rank order within a MEM): suffix = SA[rank], sequence = index of the record holding it, sequence_pos = suffix - its
 *               start.  An index without sequence starts gives sequence = UINT64_MAX and sequence_pos = suffix.
 *               Any of the three outputs may be NULL.  A window beyond the total is SUFR_B200_ERR_ARGUMENT.
 *    An index made by index_create takes its sequence starts from args (none when args->num_sequences == 0).
 *
 * -- extract, list, string_at (SufrFile::extract, SufrFile::list, SuffixArray::string_at) on the device, on an index
 *    from index_open or index_create.  t = the text, n = its length, SA / LCP = the full arrays (s entries), sequence
 *    starts s_0 < ... < s_{k-1} (k may be 0).
 *      records    record i owns [s_i, e_i) with e_i = s_{i+1}, e_{k-1} = n (the rule of index_hits: a record's region
 *                 can include its delimiter or the final '$').  A position outside every record (k = 0 or p < s_0)
 *                 belongs to [0, s_0), or to [0, n) when k = 0; its sequence is UINT64_MAX.
 *    index_extract  hits [first_hit, first_hit + max_hits) of the last index_locate or index_mems, in its order (query
 *               order, then rank order; the MEMs are the queries after index_mems).  For a hit at suffix p in record [a, e): rel = p - a, start = rel - min(rel, prefix_len),
 *               end = min(rel + suffix_len, e - a) (suffix_len UINT64_MAX = to the end of the record);
 *               region_start / region_end = start / end, relative to the record start, and the bytes are
 *               t[a + start, a + end).  The offset of the suffix in its region is rel - start = p - a - start.
 *    index_list rows [first_rank, first_rank + max_rows): suffix = SA[r], lcp = LCP[r] as stored, bytes =
 *               t[SA[r], min(SA[r] + len, n)) (len UINT64_MAX = the whole suffix).
 *    byte budget  both calls take the longest leading run of their window whose bytes fit in max_bytes: its length
 *               goes to *num_hits / *num_rows, its bytes to bytes[0 .. byte_offsets[num]), and byte_offsets[0 .. num]
 *               are the entries' exclusive offsets into `bytes`.  byte_offsets needs max_hits / max_rows + 1 entries
 *               and receives the offsets of the WHOLE window, so byte_offsets[i + 1] - byte_offsets[i] is the size of
 *               entry i also where it did not fit.  When the first entry alone does not fit, the call returns OK with
 *               num = 0 and byte_offsets[1] = that entry's size: retry with a buffer of at least that many bytes.
 *               suffix, sequence, region_start, region_end and lcp may be NULL (their first num entries are written);
 *               byte_offsets and bytes may not.
 *    index_string_at  t[pos, min(pos + len, n)) to out, its length to *out_len (pos = n: empty).
 *    SUFR_B200_ERR_ARGUMENT, before any device work: extract without a prior index_locate, a hit window beyond the
 *    last locate's hits, a rank window beyond s, pos > n, NULL required pointers. */
typedef struct SufrB200FileInfo {
    uint32_t version;
    uint32_t index_bits;          /* 32 or 64: width of SA / LCP entries and sequence starts in the file */
    uint8_t is_dna;
    uint8_t allow_ambiguity;
    uint8_t ignore_softmask;
    uint8_t reserved[5];
    uint64_t text_len;
    uint64_t num_suffixes;
    uint64_t max_query_len;       /* of the build; 0 = none (always 0 with a seed mask) */
    uint64_t num_sequences;
    uint64_t text_pos;
    uint64_t sa_pos;
    uint64_t lcp_pos;
    uint64_t file_bytes;
    char* seed_mask;              /* NULL = none, else "1101..." */
    uint64_t* sequence_starts;    /* num_sequences entries */
    char** sequence_names;        /* num_sequences NUL-terminated strings */
} SufrB200FileInfo;
int sufr_b200_file_info(const char* path, SufrB200FileInfo* out);
void sufr_b200_file_info_free(SufrB200FileInfo* info);
int sufr_b200_index_open(SufrB200Ctx* ctx, const char* path, SufrB200Index** out);
int sufr_b200_index_locate(SufrB200Index* index, const uint8_t* queries, const uint64_t* offsets, uint64_t num_queries,
                           int has_max_query_len, uint64_t max_query_len, int low_memory, uint64_t* rank_begin,
                           uint64_t* rank_end, uint64_t* hit_offsets);
int sufr_b200_index_hits(SufrB200Index* index, uint64_t first_hit, uint64_t count, uint64_t* suffix, uint64_t* sequence,
                         uint64_t* sequence_pos);
int sufr_b200_index_extract(SufrB200Index* index, uint64_t first_hit, uint64_t max_hits, uint64_t prefix_len,
                            uint64_t suffix_len /* UINT64_MAX = to the end of the record */, uint64_t max_bytes,
                            uint64_t* num_hits, uint64_t* suffix, uint64_t* sequence, uint64_t* region_start,
                            uint64_t* region_end, uint64_t* byte_offsets /* max_hits + 1 */, uint8_t* bytes);
int sufr_b200_index_list(SufrB200Index* index, uint64_t first_rank, uint64_t max_rows,
                         uint64_t len /* UINT64_MAX = whole suffix */, uint64_t max_bytes, uint64_t* num_rows,
                         uint64_t* suffix, uint64_t* lcp, uint64_t* byte_offsets /* max_rows + 1 */, uint8_t* bytes);
int sufr_b200_index_string_at(SufrB200Index* index, uint64_t pos, uint64_t len, uint8_t* out, uint64_t* out_len);

/* -- matching statistics and maximal exact matches (MEMs) of long queries, on the device, on an index from index_open
 *    or index_create.  t = the text, n its length, SA the full suffix array (s entries; the LCP array and its
 *    subsample play no part).  Only indexed suffixes count: the positions SA holds (in DNA mode, positions the build
 *    does not index are no matches).  A query q of length m is compared byte for byte, as index_search compares it:
 *    no transformation, and the end of the text sorts first.  cap = the build's max_query_len, or none; there is no
 *    run-time cap here.  Queries and offsets are those of index_search; the outputs are per byte of the batch.
 *      matching statistics  for each 0 <= i < m, ms[i] = the largest l <= min(m - i, cap) such that q[i, i+l) is a
 *               prefix of some indexed suffix, and [rank_begin[i], rank_end[i]) the half-open rank range of all indexed
 *               suffixes with that prefix (contiguous in SA).  ms[i] = 0: both are UINT64_MAX.
 *      MEMs with minimum length L >= 1  the pairs (i, ms[i]) with ms[i] >= L and (i == 0 or ms[i-1] <= ms[i]); their
 *               occurrences are the ranks [rank_begin[i], rank_end[i]).  Without a cap every such occurrence is maximal
 *               both ways: it cannot extend right, as ms[i] is the longest match, and it cannot extend left, as
 *               q[i-1, i+ms[i]) occurs nowhere or ms[i-1] would be larger.  Shorter MEMs at other occurrences are not
 *               listed (the extra matches of MUMmer's -maxmatch): for each query position only its longest match is.
 *               With a cap, lengths stop at cap: a match of length cap is "at least cap" long, and the maximality
 *               above holds only for matches shorter than cap.
 *    index_matching_stats  match_len / rank_begin / rank_end: offsets[num_queries] entries each (ms of byte
 *               offsets[k] + i of the batch is ms[i] of query k).
 *    index_mems  the MEMs of every query, in query order and position order: *num_mems of them (at most one per byte,
 *               so offsets[num_queries] entries suffice for mem_query, mem_pos, mem_len, rank_begin, rank_end);
 *               hit_offsets[0 .. num_mems] = exclusive scan of their occurrence counts (offsets[num_queries] + 1
 *               entries).  The MEMs then take the place of locate's queries: index_hits and index_extract return their
 *               occurrences, windowed and byte-budgeted, until the next index_locate or index_mems.
 *    A batch of empty queries gives no entries.  SUFR_B200_ERR_ARGUMENT, before any device work: NULL required
 *    pointers, offsets not ascending, min_len == 0.  SUFR_B200_ERR_UNSUPPORTED: an index built with a seed mask (its
 *    order is not a lexicographic order of contiguous bytes, so "longest match" has no meaning the array can answer). */
int sufr_b200_index_matching_stats(SufrB200Index* index, const uint8_t* queries, const uint64_t* offsets,
                                   uint64_t num_queries, uint64_t* match_len /* offsets[num_queries] */,
                                   uint64_t* rank_begin, uint64_t* rank_end);
int sufr_b200_index_mems(SufrB200Index* index, const uint8_t* queries, const uint64_t* offsets, uint64_t num_queries,
                         uint64_t min_len, uint64_t* num_mems, uint64_t* mem_query, uint64_t* mem_pos,
                         uint64_t* mem_len, uint64_t* rank_begin, uint64_t* rank_end,
                         uint64_t* hit_offsets /* offsets[num_queries] + 1 */);

/* -- search with mismatches, on the device, on an index from index_open or index_create without a seed mask.  t = the
 *    text, n its length, SA the full suffix array (the LCP array and its subsample play no part).
 *      separators  Z = the byte t[n - 1] and the byte t[c_i - 1] of every sequence start c_i > 0 ('$' and '%' with the
 *               default delimiter), as byte values.  Computed once per index and kept with it.
 *      match    of a query q of length m with budget k (max_mismatches): let m' = min(m, cap), cap = the build's
 *               max_query_len, or m without one (index_locate compares the same first cap bytes).  A match is a string
 *               w of m' bytes such that (a) w = t[p, p + m') for an indexed position p (an entry of SA) with
 *               p + m' <= n; (b) w differs from q[0, m') in at most k positions, bytes compared as they are (as
 *               index_search compares them); (c) no position where they differ holds a byte of Z in w: a substitution
 *               never puts a record separator into a match, while an equal separator byte still matches.  So k = 0
 *               gives the range index_locate gives (full array, no run-time cap) for every non-empty query.  An empty
 *               query, or one with m' > n, has no match.
 *    index_approx  the matches of every query, one per distinct w: [rank_begin, rank_end) = the half-open rank range of
 *               the suffixes that start with w (contiguous in SA; for a cap index the order is exact on the first cap
 *               bytes, DESIGN.md §3 item 4), and mismatches = the Hamming distance of w to q[0, m').  In query order,
 *               then rank order (the byte order of the w).  match_offsets[q] .. match_offsets[q + 1] are the matches
 *               of query q (num_queries + 1 entries); *num_hits = their occurrences in all.  The matches take the
 *               place of locate's queries: index_hits and index_extract return their occurrences, windowed and
 *               byte-budgeted, until the next index_locate, index_mems or index_approx (the k-mer calls leave them).
 *               Device memory is bounded whatever the batch: a level of the search with more nodes than fit is
 *               expanded in slices (DESIGN.md §7b).
 *    index_approx_matches  matches [first, first + count) of the last index_approx: mismatches, rank_begin, rank_end
 *               (count entries each) and hit_offsets (count + 1 entries, global indices into the hits).  Any output
 *               may be NULL.
 *    index_approx_levels  the profile of the last index_approx: nodes[d] / steps[d] = the search nodes at depth d and
 *               the binary-search steps that counted their children (the expansion repeats them), for
 *               d < min(max_levels, *num_levels); *num_levels = the longest m' of the batch.  nodes / steps may be NULL.
 *    SUFR_B200_ERR_ARGUMENT, before any device work: NULL required pointers, offsets not ascending,
 *    max_mismatches > 16; for index_approx_matches, a window beyond the matches, or a locate state that the last
 *    index_locate / index_mems set.  SUFR_B200_ERR_UNSUPPORTED: an index built with a seed mask (its order is not
 *    over contiguous bytes), with the locate state left as it was. */
int sufr_b200_index_approx(SufrB200Index* index, const uint8_t* queries, const uint64_t* offsets, uint64_t num_queries,
                           uint64_t max_mismatches, uint64_t* match_offsets /* num_queries + 1 */, uint64_t* num_hits);
int sufr_b200_index_approx_matches(SufrB200Index* index, uint64_t first, uint64_t count, uint64_t* mismatches,
                                   uint64_t* rank_begin, uint64_t* rank_end, uint64_t* hit_offsets /* count + 1 */);
int sufr_b200_index_approx_levels(SufrB200Index* index, uint64_t max_levels, uint64_t* num_levels, uint64_t* nodes,
                                  uint64_t* steps);

/* -- k-mer counting on the device, on an index from index_open or index_create without a seed mask.  t = the text,
 *    n its length, SA / LCP the full arrays (s entries), sequence starts c_0 < ... < c_{R-1}.  Records follow
 *    index_extract: record i owns [c_i, c_{i+1}), the last one [c_{R-1}, n), positions before c_0 belong to [0, c_0);
 *    an index without starts is one record [0, n).
 *      occurrence  a position p of record [a, e) with p + k <= e - 1: the k bytes lie inside the record and never
 *               include its last byte (the delimiter, or the final '$').  In a DNA index (is_dna) all k bytes are also
 *               A, C, G or T, so k-mers with N are not counted.  Every occurrence is an indexed position.
 *      group    the maximal rank run [b, e) with b == 0 || LCP[b] < k and LCP[r] >= k for b < r < e: the rank range
 *               index_search returns for its first k bytes.  A group with at least one occurrence is one distinct
 *               k-mer; its count is the number of its ranks that are occurrences (e - b in a DNA index; smaller in a
 *               plain index only where a delimiter byte also appears inside a record).
 *      k        1 <= k, and k <= the build's max_query_len when it has one (LCP values below it are exact, DESIGN.md
 *               §3 item 4); a k above n gives no k-mers.
 *    index_kmer_spectrum  histogram[i] = distinct k-mers with count i + 1 for i < num_bins - 1; histogram[num_bins - 1]
 *               = those with count >= num_bins.  1 <= num_bins <= 65536.  distinct / occurrences / max_count may be
 *               NULL.
 *    index_kmers  the groups with b >= first_rank whose count lies in [max(min_count, 1), max_count] (UINT64_MAX = no
 *               upper bound), in rank order (the byte order of the k-mers), at most max_kmers of them: rank_begin /
 *               rank_end = [b, e), count, and the k bytes t[SA[b'], +k) at bytes[j * k ..], where b' is the group's
 *               first occurrence (bytes may be NULL; it needs max_kmers * k bytes).  *next_rank = where the next window
 *               starts: every group with first_rank <= b < *next_rank has been considered, and *next_rank == s at the
 *               end.  A group that starts before first_rank is not listed.  A window costs time in proportion to the
 *               ranks it covers, so an enumeration in windows is one pass over the arrays in total.
 *    index_kmer_multiplicity  out[i] = the count of the k-mer at position first_pos + i if that position is an
 *               occurrence, else 0; saturated at UINT32_MAX.  first_pos + num_positions <= n.  Each call is one pass
 *               over the ranks, whatever the window (the first call for a k one more, whose per-rank counts, 4 s bytes,
 *               are kept for the next windows).
 *    Each call leaves the locate state of index_locate / index_mems as it was; the occurrence bitmap of the last k
 *    (n / 8 bytes) is kept with the index for the next call with the same k, and released with the per-rank counts
 *    when a call with another k comes.  SUFR_B200_ERR_ARGUMENT, before any
 *    device work: NULL required pointers, k == 0, k above the build's max_query_len, num_bins out of range,
 *    min_count > max_count, first_rank > s, a position window beyond n.  SUFR_B200_ERR_UNSUPPORTED: an index built
 *    with a seed mask. */
int sufr_b200_index_kmer_spectrum(SufrB200Index* index, uint64_t k, uint64_t num_bins, uint64_t* histogram,
                                  uint64_t* distinct, uint64_t* occurrences, uint64_t* max_count);
int sufr_b200_index_kmers(SufrB200Index* index, uint64_t k, uint64_t min_count, uint64_t max_count,
                          uint64_t first_rank, uint64_t max_kmers, uint64_t* num_kmers, uint64_t* next_rank,
                          uint64_t* rank_begin, uint64_t* rank_end, uint64_t* count, uint8_t* bytes);
int sufr_b200_index_kmer_multiplicity(SufrB200Index* index, uint64_t k, uint64_t first_pos, uint64_t num_positions,
                                      uint32_t* out);

/* -- write: replaces SufrBuilder::write (sufr_builder.rs:817-918), version-6 `.sufr` layout.
 *    Single shard: writes the whole file.  Sharded: every rank calls it with the same path; rank 0
 *    writes header, text and the names tail, every rank pwrites its SA / LCP slice at its offset.
 *    `result` must be a HOST result. */
int sufr_b200_write(const SufrB200Args* args, const SufrB200Result* result);

/* -- create: SufrBuilder::new as a single call (build on `device`, then write args->path or
 *    "out.sufr").  The suffix and LCP arrays stream from device memory into the file through a ring
 *    of pinned buffers (copy and pwrite overlap; no host copy of them is allocated), so the result is
 *    what the reference's builder struct holds after `new` (sufr_builder.rs:38-89): counts, the
 *    transformed text, n_ranges -- `sa` and `lcp` are NULL, they are in the file.  timings.d2h_ms is
 *    the wall time of that streaming write.  Free with sufr_b200_result_free(NULL, out).
 *    `out` may be NULL.  Single process only (world_size <= 1): sharded builds go through
 *    sufr_b200_build / sufr_b200_patch_seam / sufr_b200_write. */
int sufr_b200_create(const SufrB200Args* args, int device, SufrB200Result* out);

/* -- create on several GPUs of one box in ONE call (sufr::create is one call too, sufr/src/lib.rs:321-371): a host
 *    thread per device builds key-range shard r of num_devices; the text is uploaded once and replicated over NVLink
 *    (peer copies), seams are repaired from the shards' (count, first, last), and every device streams its slice of
 *    the suffix / LCP arrays into args->path at its offset.  index_bits: 32, 64 or 0 = the reference's dispatch
 *    (suffix_array.rs:460-470).  args->rank / world_size must be 0 / <= 1.  The result is that of sufr_b200_create
 *    (counts over all shards; timings: the slowest shard).  num_devices == 1 is a plain single-GPU create. */
int sufr_b200_create_multi(const SufrB200Args* args, const int* devices, int num_devices, uint32_t index_bits,
                           SufrB200Result* out);

/* -- helpers shared with the host-side mirror ---------------------------------------------- */
/* SeedMask::new (types.rs:80-97): returns the weight, or -1 if the mask is invalid.
 * bytes/positions/differences may be NULL; otherwise they need strlen(mask) entries. */
int64_t sufr_b200_seed_mask(const char* mask, uint8_t* bytes, uint64_t* positions, uint64_t* differences);
/* find_lcp_full_offset (util.rs:19-37); mask == NULL means "not a mask sort". */
uint64_t sufr_b200_find_lcp_full_offset(uint64_t lcp, const char* mask);

/* read_sequence_file (util.rs:51-89): FASTA / FASTQ -> text with delimiters and trailing '$'. */
typedef struct SufrB200Sequences {
    uint8_t* seq;
    uint64_t seq_len;
    uint64_t* start_positions;
    char** sequence_names;
    uint64_t num_sequences;
} SufrB200Sequences;
int sufr_b200_read_sequence_file(const char* path, uint8_t sequence_delimiter, SufrB200Sequences* out);
void sufr_b200_sequences_free(SufrB200Sequences* seqs);

/* Synthetic workload generators used by bench.py (device buffers, deterministic in `seed`). */
int sufr_b200_synth_dna(SufrB200Ctx* ctx, uint8_t* device_text, uint64_t text_len, uint64_t seed,
                        const uint64_t* record_starts, uint64_t num_records, uint8_t delimiter);

/* Message of the last error on the calling thread. */
const char* sufr_b200_last_error(void);
int sufr_b200_abi_version(void);
/* Number of CUDA devices visible (0 when there is none or the driver is missing). */
int sufr_b200_device_count(void);

#ifdef __cplusplus
}
#endif
#endif /* SUFR_B200_H */
