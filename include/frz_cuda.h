/*
 * frz_cuda.h — C ABI of the B200-native `match_list` path of saghen/frizbee.
 *
 * This header is the drop-in boundary (SURVEY.md §8(b)).  Every entry point
 * names the reference interface it replaces (paths relative to the reference
 * crate root).  Plain pointers and sizes only: no torch, no C++ types.
 *
 * Reference interfaces replaced:
 *   trait Specialized::match_list            src/matcher/algo.rs:14-22
 *   Matcher::{new,from_patterns,from_query}  src/matcher/mod.rs:90-136
 *   Matcher::match_list                      src/matcher/mod.rs:212-222
 *   Matcher::match_list_parallel             src/matcher/parallel.rs:18-89
 *   Pattern::{parse,parse_query}             src/pattern.rs:100-222
 *   radix_sort_matches                       src/sort.rs:6-40
 *   Match / Config / Scoring / enums         src/lib.rs:141-153,236-271,313-323,439-478
 *
 * There is NO CPU fallback behind this ABI: every compute entry point fails
 * with FRZ_ERR_NO_DEVICE / FRZ_ERR_CUDA when no sm_100 device is usable.
 */
#ifndef FRZ_CUDA_H
#define FRZ_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FRZ_ABI_VERSION 2
#if defined(__GNUC__)
#define FRZ_API __attribute__((visibility("default")))
#else
#define FRZ_API
#endif

/* ------------------------------------------------------------------ status */

typedef enum frz_status {
    FRZ_OK = 0,
    FRZ_ERR_INVALID_ARG = 1,
    /* reference panics: "needle too long and could overflow the u16 score" (src/lib.rs:524-527) */
    FRZ_ERR_NEEDLE_TOO_LONG = 2,
    /* reference panics: "gap penalties too large" (src/lib.rs:532-536) */
    FRZ_ERR_GAP_OVERFLOW = 3,
    /* reference panics: "too many items in haystack, will overflow the u32 index" (src/matcher/mod.rs:438-446) */
    FRZ_ERR_TOO_MANY_ITEMS = 4,
    /* reference panics: "threads must be positive" (src/matcher/parallel.rs:24) */
    FRZ_ERR_THREADS_ZERO = 5,
    /* caller-provided output buffer too small; *n_out holds the required count */
    FRZ_ERR_CAPACITY = 6,
    FRZ_ERR_CUDA = 7,
    FRZ_ERR_NO_DEVICE = 8,
    /* feature of the reference not built on the GPU path yet (never a silent CPU fallback) */
    FRZ_ERR_UNSUPPORTED = 9,
    FRZ_ERR_OOM = 10,
    /* NCCL missing / failed, or a peer rank did not answer (multi-GPU entry points only) */
    FRZ_ERR_NCCL = 11
} frz_status;

/* thread-local, human-readable detail for the last non-OK status */
FRZ_API const char* frz_last_error(void);
FRZ_API const char* frz_status_str(frz_status s);
FRZ_API int frz_abi_version(void);

/* ------------------------------------------------------------------- types */

/* `Match` (src/lib.rs:141-153).  The reference struct is default-repr Rust; the shim converts. */
typedef struct frz_match {
    uint32_t index; /* index in the original haystack list (+ index_offset) */
    uint16_t score;
    uint8_t exact;  /* 0/1 */
    uint8_t _pad;   /* always 0 */
} frz_match;

/* `Scoring` (src/lib.rs:439-478), defaults from src/const.rs:1-10 */
typedef struct frz_scoring {
    uint16_t match_score;          /* 12 */
    uint16_t mismatch_penalty;     /*  6 */
    uint16_t gap_open_penalty;     /*  5 */
    uint16_t gap_extend_penalty;   /*  1 */
    uint16_t prefix_bonus;         /* 12 */
    uint16_t capitalization_bonus; /*  4 */
    uint16_t matching_case_bonus;  /*  4 */
    uint16_t exact_match_bonus;    /*  8 */
    uint16_t delimiter_bonus;      /*  4 */
} frz_scoring;

/* `CaseMatching` (src/lib.rs:353-377) */
enum { FRZ_CASE_IGNORE = 0, FRZ_CASE_SMART = 1, FRZ_CASE_RESPECT = 2 };
/* `UnicodeMatching` (src/lib.rs:379-402) */
enum { FRZ_UNICODE_IGNORE = 0, FRZ_UNICODE_SMART = 1, FRZ_UNICODE_ALWAYS = 2 };
/* `Matching` (src/lib.rs:413-436) */
enum { FRZ_MATCHING_FUZZY = 0, FRZ_MATCHING_EXACT = 1, FRZ_MATCHING_PREFIX = 2,
       FRZ_MATCHING_SUFFIX = 3, FRZ_MATCHING_SUBSTRING = 4 };
/* `SortStrategy` (src/lib.rs:311-351) */
enum { FRZ_SORT_SCORE_THEN_INDEX_ASC = 0, FRZ_SORT_SCORE_THEN_INDEX_DESC = 1,
       FRZ_SORT_INDEX_ASC = 2, FRZ_SORT_INDEX_DESC = 3 };

#define FRZ_MAX_TYPOS_NONE (-1)

/* `Config` (src/lib.rs:236-271) */
typedef struct frz_config {
    int32_t max_typos;     /* FRZ_MAX_TYPOS_NONE (= Rust `None`) or 0..65535; default 0 */
    uint8_t casing;        /* FRZ_CASE_*;     default SMART */
    uint8_t unicode;       /* FRZ_UNICODE_*;  default SMART */
    uint8_t matching;      /* FRZ_MATCHING_*; default FUZZY */
    uint8_t sort;          /* FRZ_SORT_*;     default SCORE_THEN_INDEX_ASC */
    frz_scoring scoring;
    /* Which reference SIMD backend the integer results are bit-exact with
     * (SURVEY.md §8 finding 1: scores depend on the lane count).
     * 0 = auto: the backend `Matcher::get_backend` (src/matcher/mod.rs:448-498)
     * would select on THIS host's CPU; else 16 (SSE/NEON/scalar), 32 (AVX2),
     * 64 (AVX-512+VBMI) = lane count of the u8 family; the u16 family
     * (needle too long for u8 scores) uses half of it. */
    uint8_t emulate_lanes;
    uint8_t _pad;
} frz_config;

/* `Pattern` + `PatternConfig` (src/pattern.rs:9-18, 230-246).  Overrides use -1 = inherit. */
typedef struct frz_pattern {
    const uint8_t* needle;
    size_t needle_len;
    uint8_t negated;
    uint8_t has_scoring;       /* 1 → `scoring` overrides Config::scoring */
    int8_t casing;             /* -1 inherit, else FRZ_CASE_* */
    int8_t unicode;            /* -1 inherit, else FRZ_UNICODE_* */
    int8_t matching;           /* -1 inherit, else FRZ_MATCHING_* */
    int8_t _pad[3];
    int32_t max_typos;         /* -1 inherit (PatternConfig cannot express "unlimited"), else 0..65535 */
    frz_scoring scoring;
} frz_pattern;

FRZ_API void frz_config_default(frz_config* out);   /* Config::default()  src/lib.rs:260-271 */
FRZ_API void frz_scoring_default(frz_scoring* out); /* Scoring::default() src/lib.rs:461-478 */

/* ------------------------------------------------------- query-atom parser */

/* Owned parse result of Pattern::parse_query (src/pattern.rs:190-222). */
typedef struct frz_query frz_query;
FRZ_API frz_status frz_parse_query(const uint8_t* query, size_t len, frz_query** out);
/* Pattern::parse (src/pattern.rs:100-165) on one atom; result holds exactly one pattern
 * (even when its needle is empty, as in the reference). */
FRZ_API frz_status frz_parse_atom(const uint8_t* atom, size_t len, frz_query** out);
FRZ_API size_t frz_query_len(const frz_query* q);
/* The returned pattern's `needle` points into `q`; valid until frz_query_destroy. */
FRZ_API frz_status frz_query_get(const frz_query* q, size_t i, frz_pattern* out);
FRZ_API void frz_query_destroy(frz_query* q);

/* ----------------------------------------------------------------- corpus */

/* A haystack list, packed and resident in HBM on one device.  Read-only for matchers (only frz_corpus_append mutates it),
 * reusable across matchers/needles (the interactive use: haystacks fixed, needle changes).
 * Replaces the `&[S: AsRef<str>]` argument of Matcher::match_list (src/matcher/mod.rs:212).
 * Input is Arrow-style: `bytes` = concatenated UTF-8, `offsets[n+1]` monotone byte offsets. */
typedef struct frz_corpus frz_corpus;

FRZ_API frz_status frz_corpus_create(const uint8_t* bytes, const uint64_t* offsets, uint64_t n,
                             int device, frz_corpus** out);
/* same, for either Arrow offset width (Utf8 = 4-byte, LargeUtf8 = 8-byte offsets); a sliced array may start at
 * offsets[0] != 0.  The value bytes are streamed host->device in tile-aligned chunks on a copy stream while
 * the bucketing kernels run (SURVEY.md §8(f) rank 1: the step before Matcher::match_list, src/matcher/mod.rs:212). */
FRZ_API frz_status frz_corpus_create_arrow(const uint8_t* bytes, const void* offsets, int offset_width, uint64_t n,
                                   int device, frz_corpus** out);
/* Incremental ingestion: appends n_new haystacks (host Arrow buffers, either offset width); they take the indices
 * [frz_corpus_len, frz_corpus_len + n_new).  Only the partial last tile is re-bucketed.  Synchronous; the caller
 * must not run it concurrently with a match on the same corpus.  (Reference side: the caller pushing onto the
 * Vec<String> it later passes to Matcher::match_list, src/matcher/mod.rs:212.) */
FRZ_API frz_status frz_corpus_append(frz_corpus* c, const uint8_t* bytes, const void* offsets, int offset_width,
                             uint64_t n_new);
/* same, from a pointer array + lengths (the layout a Rust `&[&str]` has) */
FRZ_API frz_status frz_corpus_create_ptrs(const uint8_t* const* ptrs, const uint32_t* lens, uint64_t n,
                                  int device, frz_corpus** out);
/* same, but `d_bytes`/`d_offsets` are already device pointers on `device` */
FRZ_API frz_status frz_corpus_create_device(const uint8_t* d_bytes, const uint64_t* d_offsets, uint64_t n,
                                    uint64_t total_bytes, int device, void* stream, frz_corpus** out);
FRZ_API uint64_t frz_corpus_len(const frz_corpus* c);
FRZ_API uint64_t frz_corpus_total_bytes(const frz_corpus* c);   /* sum of haystack lengths */
FRZ_API uint64_t frz_corpus_device_bytes(const frz_corpus* c);  /* HBM footprint of the packed form */
FRZ_API int frz_corpus_device(const frz_corpus* c);
FRZ_API void frz_corpus_destroy(frz_corpus* c);

/* ---------------------------------------------------------------- matcher */

/* `Matcher` (src/matcher/mod.rs:76-188). */
typedef struct frz_matcher frz_matcher;

/* Matcher::from_patterns (src/matcher/mod.rs:105-111); n_patterns == 1 ⇔ Matcher::new */
FRZ_API frz_status frz_matcher_create(const frz_pattern* patterns, size_t n_patterns,
                              const frz_config* config, frz_matcher** out);
/* Matcher::from_query (src/matcher/mod.rs:136-138) */
FRZ_API frz_status frz_matcher_from_query(const uint8_t* query, size_t len, const frz_config* config,
                                  frz_matcher** out);
/* Matcher::set_config (src/matcher/mod.rs:154-160) */
FRZ_API frz_status frz_matcher_set_config(frz_matcher* m, const frz_config* config);
/* `impl Clone for Matcher` (src/matcher/mod.rs:76): same patterns and config, its own device scratch */
FRZ_API frz_status frz_matcher_clone(const frz_matcher* m, frz_matcher** out);
FRZ_API void frz_matcher_destroy(frz_matcher* m);

/* Introspection of what `get_backend` selected for pattern i (src/matcher/mod.rs:448-498):
 * lanes ∈ {8,16,32,64}; score_bits ∈ {8,16}; prefilter_lanes ∈ {16,32,64}; is_literal 0/1. */
FRZ_API frz_status frz_matcher_backend_info(const frz_matcher* m, size_t i, int* lanes, int* score_bits,
                                    int* prefilter_lanes, int* is_literal);
FRZ_API size_t frz_matcher_num_patterns(const frz_matcher* m); /* compiled (non-empty-needle) patterns */

/* Matcher::match_list (src/matcher/mod.rs:212-222): all patterns, ordered per config.sort.
 * `out` is HOST memory with room for `cap` matches.  On FRZ_ERR_CAPACITY *n_out = needed. */
FRZ_API frz_status frz_match_list(frz_matcher* m, const frz_corpus* corpus,
                          frz_match* out, uint64_t cap, uint64_t* n_out);

/* Specialized::match_list / Matcher::match_list_into (src/matcher/algo.rs:17-22,
 * src/matcher/mod.rs:373-392): matches appended in input (index-ascending) order,
 * indices offset by `index_offset`, no sort. */
FRZ_API frz_status frz_match_list_into(frz_matcher* m, const frz_corpus* corpus, uint32_t index_offset,
                               frz_match* out, uint64_t cap, uint64_t* n_out);

/* End-to-end convenience: Matcher::match_list on HOST Arrow buffers (pack + H2D + match + D2H
 * in one call; nothing stays resident). */
FRZ_API frz_status frz_match_list_host(frz_matcher* m, const uint8_t* bytes, const uint64_t* offsets,
                               uint64_t n, int device, frz_match* out, uint64_t cap, uint64_t* n_out);
/* same, for either Arrow offset width (4 or 8 bytes); H2D chunks overlap the pack kernels */
FRZ_API frz_status frz_match_list_host_arrow(frz_matcher* m, const uint8_t* bytes, const void* offsets, int offset_width,
                                     uint64_t n, int device, frz_match* out, uint64_t cap, uint64_t* n_out);

/* Matcher::match_list_indices (src/matcher/mod.rs:234-262) for CHOSEN haystacks — the rows a UI is about to display:
 * for haystack which[j] (corpus-relative index) writes its Match to out_matches[j] and the byte offsets of the
 * matched characters, in the reference's descending order, to out_indices[j * stride ...]; out_counts[j] = how many
 * the haystack has (UNtruncated: when it exceeds `stride` only the first `stride` offsets were stored — call again with
 * a larger stride), or UINT32_MAX when that haystack does not match.  Host pointers.  Multi-pattern matchers pool
 * the atoms' indices like match_one_indices_multi (src/matcher/multi.rs:56-79).  Like the reference's, not a tuned path. */
FRZ_API frz_status frz_match_indices(frz_matcher* m, const frz_corpus* corpus, const uint32_t* which, uint64_t n,
                             frz_match* out_matches, uint32_t* out_indices, uint32_t stride, uint32_t* out_counts);

/* ------------------------------------------------ multi-GPU: match_list_parallel
 *
 * Matcher::match_list_parallel (src/matcher/parallel.rs:18-89) with GPUs in place of worker threads: the haystack list
 * is sharded by contiguous index range (shard g = [g*ceil(N/G), ...), SURVEY.md §8(e)), every GPU runs the whole local
 * pipeline on its shard with its own clone of the matcher (parallel.rs:46) and leaves a locally ordered run in HBM
 * (parallel.rs:67-73), ONE ncclAllGather moves the runs (padded to the longest) over NVLink, every GPU merges them
 * (k_merge_matches_by, src/k_merge.rs:90-131) and copies ITS slice of the merged list to the host buffer, so the
 * device->host copy runs over all PCIe links in parallel.  The match counts (the Vec lengths the k-merge reads) travel
 * through a small pinned host block shared by the ranks, published by each GPU as soon as its prefilter has run —
 * no second collective, and the exchange overlaps the scoring kernels.
 *
 * NCCL is loaded at run time (dlopen "libnccl.so.2", so a process that already carries PyTorch's NCCL shares it);
 * a communicator over ONE GPU never touches NCCL. */
typedef struct frz_comm frz_comm;
#define FRZ_UNIQUE_ID_BYTES 128

/* Single-process form — what a Rust caller of match_list_parallel uses: one communicator over `n_gpus` devices of this
 * process (`devices` NULL = 0..n_gpus-1), ncclCommInitAll, one worker thread per GPU inside the library (the
 * std::thread::scope pool of parallel.rs:39-66). */
FRZ_API frz_status frz_comm_create_local(int n_gpus, const int* devices, frz_comm** out);
/* Multi-process form (one rank per process: torchrun, MPI): rank 0 gets an id, the host program ships those 128 bytes
 * to every rank, every rank joins.  Collective: all ranks must call frz_comm_create_rank. */
FRZ_API frz_status frz_comm_unique_id(uint8_t id[FRZ_UNIQUE_ID_BYTES]);
FRZ_API frz_status frz_comm_create_rank(const uint8_t id[FRZ_UNIQUE_ID_BYTES], int world, int rank, int device, frz_comm** out);
FRZ_API void frz_comm_destroy(frz_comm* c);
FRZ_API int frz_comm_world(const frz_comm* c);
FRZ_API int frz_comm_rank(const frz_comm* c);      /* rank of this process (multi-process form), 0 for the local form */
FRZ_API int frz_comm_device(const frz_comm* c, int local_index);
/* Host buffer every rank's GPU can write: pinned; in the multi-process form ONE shared-memory segment mapped and pinned
 * by every rank (collective: every rank calls it with the same size and gets its own mapping of the same memory). */
FRZ_API frz_status frz_comm_host_alloc(frz_comm* c, uint64_t bytes, void** out);
FRZ_API frz_status frz_comm_host_free(frz_comm* c, void* p);
/* host-side barrier over the ranks of the communicator (no-op for the local form) */
FRZ_API frz_status frz_comm_barrier(frz_comm* c);

/* Contiguous index-range shards of one host Arrow list, shard g resident on the communicator's g-th GPU (local form).
 * `shards_out` receives frz_comm_world(c) corpora (empty shards are valid). */
FRZ_API frz_status frz_corpus_create_sharded(const uint8_t* bytes, const void* offsets, int offset_width, uint64_t n,
                                     frz_comm* c, frz_corpus** shards_out);

/* Matcher::match_list_parallel (src/matcher/parallel.rs:18-89), local form: shards[g] lives on the communicator's g-th
 * GPU and covers the indices after shards[0..g).  Blocking; `out` is host memory (frz_comm_host_alloc memory lets all
 * GPUs copy concurrently; any other memory works).  On FRZ_ERR_CAPACITY *n_out = needed. */
FRZ_API frz_status frz_match_list_parallel(frz_matcher* m, const frz_corpus* const* shards, int n_shards, frz_comm* c,
                                   frz_match* out, uint64_t cap, uint64_t* n_out);
/* One rank of the multi-process form.  Collective: every rank calls it with its shard and the index of its first
 * haystack.  `out` must be the buffer returned by frz_comm_host_alloc (every rank writes its slice of the merged list
 * into the shared segment; on return the WHOLE list is there) — or NULL with cap 0 to skip the host copy.
 * *d_out (optional) receives this rank's device copy of the merged list, valid until the next call on `c`. */
FRZ_API frz_status frz_match_list_parallel_rank(frz_matcher* m, const frz_corpus* shard, uint32_t index_offset, frz_comm* c,
                                        frz_match* out, uint64_t cap, uint64_t* n_out, const frz_match** d_out);
/* same, end to end: this rank's shard arrives as HOST Arrow buffers (streamed H2D + pack, as frz_match_list_host_arrow) */
FRZ_API frz_status frz_match_list_parallel_rank_host(frz_matcher* m, const uint8_t* bytes, const void* offsets, int offset_width,
                                             uint64_t n, uint32_t index_offset, frz_comm* c, frz_match* out, uint64_t cap,
                                             uint64_t* n_out);
/* How host-out calls move the matches on this communicator: 2 = P2P placement (every GPU stores its matches at their
 * merged positions in the peers' slice buffers over NVLink — peer access in the local form, cudaIpc in the multi-process
 * form — then every GPU copies its slice out), 0 = ncclAllGather of whole runs + merge.  Chosen at creation (default 2 on
 * more than one GPU; FRZ_PARALLEL_EXCHANGE=allgather selects 0); 2 is downgraded to 0 by the first call when peer memory
 * cannot be mapped.  1 and 3 are no longer returned.  Device-out calls always use the all-gather. */
FRZ_API int frz_comm_exchange_mode(const frz_comm* c);

/* Device timings (ms) of the last parallel call on local rank `local_index`: [0] local pipeline (prefilter, scoring,
 * sort) [1] all-gather + merge [2] device->host slice [3] total; and the matcher clone that ran it (for
 * frz_matcher_last_timings).  Blocks until that rank's stream is idle. */
FRZ_API frz_status frz_comm_last_timings(frz_comm* c, int local_index, float* ms4, const frz_matcher** clone);

/* Device-resident variant used by the multi-GPU path (Matcher::match_list_parallel,
 * src/matcher/parallel.rs:18-89): this rank's shard → a locally ordered run left in HBM.
 * `d_out` (cap matches) and `d_count` (one uint64) are device pointers; `stream` is a
 * cudaStream_t (NULL = default stream).  Asynchronous: returns after enqueueing. */
FRZ_API frz_status frz_match_shard_device(frz_matcher* m, const frz_corpus* shard, uint32_t index_offset,
                                  frz_match* d_out, uint64_t cap, uint64_t* d_count, void* stream);
/* The count of a shard call is known before its scores (it is the prefilter's survivor count): this makes
 * `stream` (a second cudaStream_t) wait only until d_count has been written, so the count exchange of
 * match_list_parallel (the `Vec` lengths the reference's k-merge reads, src/k_merge.rs:96-104) overlaps scoring. */
FRZ_API frz_status frz_matcher_wait_count(frz_matcher* m, void* stream);

/* k_merge_matches_by (src/k_merge.rs:90-131) on device: `d_runs` holds `n_runs` runs, run r at
 * d_runs + r*run_stride with run_counts_host[r] valid entries, each already ordered per `sort`.
 * `score_bound`: upper bound of the scores in the runs (frz_matcher_score_bound), 0 = unknown.
 * Writes the merged sequence to d_out (may not alias d_runs).  Asynchronous on `stream`.  Uses one grow-only scratch
 * per device for the life of the process: calls for the same device must not overlap (one stream, or serialise). */
FRZ_API frz_status frz_merge_runs_device(const frz_match* d_runs, uint64_t run_stride,
                                 const uint64_t* run_counts_host, int n_runs, uint8_t sort,
                                 uint32_t score_bound, frz_match* d_out, int device, void* stream);
/* Upper bound of any score this matcher can emit (sum over its non-negated patterns, saturating at
 * 65535); lets the device sort / merge use a single counting pass.  0 for an empty matcher. */
FRZ_API uint32_t frz_matcher_score_bound(const frz_matcher* m);

/* Test aid: copies the compiled device pattern (frizbee_b200/csrc/frz_device.cuh: FrzPatternDev) of pattern i; out_size
 * must equal its size.  Lets host builds of the kernel cores run with exactly the constants the GPU receives. */
FRZ_API frz_status frz_matcher_debug_pattern(const frz_matcher* m, size_t i, void* out, size_t out_size);

/* radix_sort_matches (src/sort.rs:6-40): stable, descending score; `matches` is host memory. */
FRZ_API frz_status frz_radix_sort_matches(frz_match* matches, uint64_t n, int device);

/* Per-stage device timings (ms) of the most recent frz_match_list* call on this matcher:
 * [0]=prefilter [1]=smith-waterman [2]=sort/emit [3]=total device; bytes = algorithmic bytes. */
FRZ_API frz_status frz_matcher_last_timings(const frz_matcher* m, float* ms4, uint64_t* launches);

#ifdef __cplusplus
}
#endif
#endif /* FRZ_CUDA_H */
