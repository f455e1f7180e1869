/*
 * cco_b200.h -- C ABI of the Blackwell-native Correlated Cross-Occurrence (CCO) model builder.
 *
 * This is the drop-in boundary for the train hot path of actionml/universal-recommender.
 * It replaces the two calls the reference makes into Apache Mahout 0.13.0:
 *
 *   SimilarityAnalysis.cooccurrencesIDSs(Array[IndexedDataset], randomSeed,
 *       maxInterestingItemsPerThing, maxNumInteractions)       src/main/scala/URAlgorithm.scala:323-329
 *   SimilarityAnalysis.crossOccurrenceDownsampled(
 *       List[DownsamplableCrossOccurrenceDataset], randomSeed) src/main/scala/URAlgorithm.scala:343-346
 *
 * A Scala object with those two signatures marshals each IndexedDataset's matrix into CSR and
 * calls cco_train() over JNI (INTEGRATION.md has the stub); everything else in the reference
 * (engine.json, DataSource, Preparator, URModel, EsClient) is untouched.
 *
 * Plain C: pointers and sizes only, no CUDA/torch types.  All functions return 0 on success or
 * a negative cco_status_t; cco_last_error() gives the message (thread-local).  There is no CPU
 * fallback: every entry point that computes fails with CCO_E_CUDA when no sm_100 device exists.
 */
#ifndef CCO_B200_H
#define CCO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CCO_ABI_VERSION 2

typedef enum {
  CCO_OK = 0,
  CCO_E_INVALID_ARG = -1,    /* mirrors IllegalArgumentException / Preconditions.checkArgument in Mahout */
  CCO_E_CUDA = -2,           /* CUDA runtime / no usable device */
  CCO_E_NCCL = -3,
  CCO_E_OOM = -4,
  CCO_E_SHAPE_MISMATCH = -5, /* matrices do not share the user (row) space -- Preparator.scala:47-77 */
  CCO_E_UNSUPPORTED = -6
} cco_status_t;

/*
 * Input: one binary user x item matrix per event type, exactly what Preparator builds as
 * IndexedDatasetSpark (src/main/scala/Preparator.scala:160-214): every stored value is 1.0
 * (RandomAccessSparseVector.setQuick(col, 1.0), :201-208) so there is no values array;
 * n_rows is the size of the shared user dictionary (newRowCardinality, :213), including users
 * with no interaction in this event type.  Column indices may come in any order inside a row
 * and duplicates collapse (setQuick semantics).  The library never keeps host pointers.
 */
typedef struct {
  int64_t n_rows;         /* U, must be equal for all matrices of one call, < 2^31 (Mahout keys are Int) */
  int32_t n_cols;         /* I of this event type, < 2^31 - 1 */
  const int64_t *row_ptr; /* [n_rows + 1], row_ptr[0] == 0, monotone */
  const int32_t *col_idx; /* [row_ptr[n_rows]], each in [0, n_cols) */
} cco_csr_t;

/*
 * Per-matrix parameters = DownsamplableCrossOccurrenceDataset(iD, maxElementsPerRow,
 * maxInterestingElements, minLLROpt) as built at src/main/scala/URAlgorithm.scala:336-340.
 * Defaults in the reference: 500 / 50 / None (URAlgorithm.scala:54,56,338-340).
 */
typedef struct {
  int32_t max_interactions; /* m >= 1: maxItemsPerUser | maxEventsPerEventType */
  int32_t top_k;            /* k in [1, CCO_MAX_TOP_K]: maxCorrelatorsPerItem | maxCorrelatorsPerEventType */
  int32_t has_min_llr;      /* Option[Double].isDefined */
  double min_llr;           /* keep a cell only if llr >= min_llr */
} cco_indicator_params_t;

#define CCO_MAX_TOP_K 2048

/*
 * Limits (each one is a clean CCO_E_UNSUPPORTED with a message, never a wrong result):
 *  - top_k <= CCO_MAX_TOP_K;  stored entries per matrix < 2^32;  n_rows < 2^31 - 1 (Mahout row keys are Int).
 *  - packed accumulator word: a row's co-occurrence counts live in shared memory as (column << count_bits | count) in
 *    32 bits.  count <= min(largest primary-item marginal, largest column marginal of this event type) must fit next to
 *    the column id: bitlen(n_cols + 1) + bitlen(max count) <= 32.  After the reference's default downsampling (500) every
 *    marginal is <= ~560, i.e. 10 bits: item spaces up to 4M columns.  Without downsampling (m huge) a 1M-column space
 *    allows counts < 4096.
 */

/* cco_train flags */
enum {
  /* Row sample rate of sampleDownAndBinarize: 0 = real min(m,d)/d (default); 1 = literal
   * Int/Int division recalled from Mahout 0.13.0 (1 if d <= m else 0).  DESIGN.md "Downsampling". */
  CCO_FLAG_ROWRATE_INTDIV = 1,
  /* LogLikelihood.entropy evaluation order: 0 = left-to-right subtraction (default);
   * 2 = varargs form xLogX(sum) - (sum of xLogX).  Last-bit difference only. */
  CCO_FLAG_ENTROPY_VARARGS = 2,
  /* inputs are already canonical (columns strictly ascending inside each row): skip the check */
  CCO_FLAG_ASSUME_CANONICAL = 4,
  /* measurement only: leave the packed indicator arrays in HBM (col/llr/count host arrays are not
   * filled; row_ptr is).  Used for the device-resident throughput number of bench.py. */
  CCO_FLAG_RESULT_ON_DEVICE = 8,
  /* result contents.  The reference consumer keeps only the ordered column ids of each row (package.scala:100-108
   * drops the LLR values, nothing reads k11): NO_COUNT skips the count array (cco_result_matrix returns NULL for it),
   * NO_LLR skips the LLR array too -- 80 instead of 321 MB come back per train at C3. */
  CCO_FLAG_RESULT_NO_COUNT = 16,
  CCO_FLAG_RESULT_NO_LLR = 32,
  /* tests only, not for production (cco_ingest_strings): the id hash keeps 2 bits, so nearly every pair of distinct ids
   * collides and the exact byte-comparison pass does the grouping.  The output is the same, only slower. */
  CCO_FLAG_INGEST_SHORT_HASH = 64
};

/*
 * Sampler (the repo's definition; Mahout's java.util.Random-per-Spark-block stream is not
 * reproducible by construction, SURVEY.md A.1).  For a stored (user u, item j) of a matrix with
 * raw row count d_u and raw column count c_j:
 *   mix64(z): z ^= z>>30; z *= 0xbf58476d1ce4e5b9; z ^= z>>27; z *= 0x94d049bb133111eb; z ^= z>>31
 *   h    = mix64( mix64(((uint64)(uint32)seed << 32) | (uint32)u) + (uint64)(uint32)j * 0x9e3779b97f4a7c15 )
 *   u01  = (double)(h >> 11) * 2^-53
 *   keep = u01 <= min( min(m,d_u)/d_u , min(m,c_j)/c_j )          (fp64, IEEE division)
 * Identity whenever every d_u <= m and c_j <= m -- the regime where parity with Mahout is exact.
 */

typedef struct {
  int32_t device;     /* CUDA device ordinal for this context */
  int32_t rank;       /* rank of this context in a multi-GPU job, 0 if world_size == 1 */
  int32_t world_size; /* number of cooperating contexts (one process per GPU) */
  int32_t reserved;
  /* world_size > 1: 128-byte NCCL unique id obtained from cco_nccl_unique_id() on rank 0 and
   * distributed by the host (any transport); ignored when world_size == 1 */
  const unsigned char *nccl_unique_id;
  /* optional (NULL / 0 = library-owned pinned memory): host memory the result arrays are placed in, e.g. a shared
   * segment another process maps, so that this rank's indicator slice reaches its reader without a copy.  The library
   * page-locks it (cudaHostRegister) for the life of the context; it is reused once every result has been freed. */
  void *result_arena;
  size_t result_arena_bytes;
} cco_config_t;

typedef struct cco_ctx cco_ctx_t;
typedef struct cco_result cco_result_t;
typedef struct cco_dataset cco_dataset_t;

/* Per-call statistics (the metrics/logging hook; replaces the logger.info dimension lines of
 * Preparator.scala:60,66,74 and feeds bench.py's roofline arithmetic). */
typedef struct {
  int64_t n_users;
  int64_t nnz_in_total;         /* stored entries handed in, all matrices */
  int64_t nnz_downsampled[16];  /* per matrix (first 16), after canonicalise + downsample */
  int64_t products[16];         /* per indicator: P(A',B') = sum_u degA'(u) * degB'(u), this rank's rows */
  int64_t distinct_cells[16];   /* per indicator: nnz(A'^T B') visited, this rank's rows */
  int64_t out_nnz[16];          /* per indicator: kept cells, this rank's rows */
  int64_t llr_evaluated[16];    /* per indicator: cells whose fp64 LLR was evaluated (rest: dominance-filtered) */
  /* CUDA-event times of this call.  ms_h2d: host->device copies (copy stream; overlaps ms_prepare in cco_train);
   * ms_prepare: histogram + allreduce + sampleDownAndBinarize + transpose; ms_cooccurrence: all indicators incl.
   * scheduling and result packing; ms_d2h: always 0 (the result copies overlap the next indicator on the copy
   * stream and are inside ms_cooccurrence / ms_total); ms_total: the whole call on the launch stream. */
  float ms_h2d, ms_prepare, ms_cooccurrence, ms_d2h, ms_total;
  float ms_indicator[16];       /* per indicator: row kernels only */
  int32_t n_kernel_launches;    /* kernels of this library launched by the call */
  int32_t n_mats;
  /* breakdown of ms_prepare: [0] input check + raw column histogram  [1] all-reduce of the raw counts (multi-GPU)
   * [2] sampleDownAndBinarize pass 1 (keep decisions, kept counts, marginals)  [3] kept-count all-gather + marginal
   * all-reduce (multi-GPU) + row_ptr scans  [4] pass 2 (ordered write)  [5] column-block all-gather + pack (multi-GPU)
   * [6] transpose of A' + largest marginals */
  float ms_prep_stage[8];
} cco_stats_t;

int cco_abi_version(void);
const char *cco_last_error(void);
const char *cco_status_string(int status);

/* number of sm_100 (B200) devices visible; <0 on CUDA failure */
int cco_device_count(void);

/* world_size > 1 only: fill 128 bytes on rank 0, hand them to every rank's cco_create */
int cco_nccl_unique_id(unsigned char out[128]);

int cco_create(const cco_config_t *cfg, cco_ctx_t **out);
/*
 * Group context: ONE context over several B200s of this process -- what the single Spark-driver thread of the reference
 * (URAlgorithm.scala:292-307) can drive through JNI.  cco_train / cco_cooccurrences_idss on it run one host thread per
 * GPU inside the library (NCCL communicator from ncclCommInitAll): each GPU uploads its block of user rows from the SAME
 * host matrices, computes a work-balanced range of primary-item rows, and copies its slice into ONE merged result (full
 * row range, one set of host arrays).  Resident datasets (cco_dataset_upload / cco_ingest) stay per-GPU APIs.
 */
int cco_create_group(int32_t n_devices, const int32_t *devices, cco_ctx_t **out);
int cco_destroy(cco_ctx_t *ctx);

/* Pinned host memory the caller can fill directly (e.g. wrapped as a direct ByteBuffer by the
 * JNI shim) so cco_train's host->device copies run at PCIe speed.  Optional. */
int cco_host_alloc(cco_ctx_t *ctx, size_t bytes, void **out);
int cco_host_free(cco_ctx_t *ctx, void *p);

/*
 * The whole hot path, mats[0] = primary (A):
 *   A' = sampleDownAndBinarize(A, seed, params[0].m); N = n_rows; colA = nnzPerColumn(A')
 *   out[0] = top-k_0 by LLR of A'^T A' (diagonal excluded), out[i] = top-k_i by LLR of A'^T B'_i
 * In a multi-GPU job every rank passes the same matrices; rank r computes a work-balanced range
 * of primary-item rows and its result holds only those rows (cco_result_row_range).
 * One call at a time per context.
 */
int cco_train(cco_ctx_t *ctx, int32_t n_mats, const cco_csr_t *mats, const cco_indicator_params_t *params,
              int32_t seed, uint32_t flags, cco_result_t **out);

/*
 * Split form of cco_train for callers that keep the matrices resident in HBM across trains
 * (the `drmA.checkpoint()` / cache() role in Mahout): upload once (host->device copy, validation,
 * canonicalisation), train any number of times with different parameters / seeds.
 * cco_train(...) == cco_dataset_upload + cco_train_dataset + cco_dataset_free.
 */
int cco_dataset_upload(cco_ctx_t *ctx, int32_t n_mats, const cco_csr_t *mats, uint32_t flags, cco_dataset_t **out);
int cco_train_dataset(cco_ctx_t *ctx, const cco_dataset_t *ds, const cco_indicator_params_t *params, int32_t seed,
                      uint32_t flags, cco_result_t **out);
int cco_dataset_free(cco_dataset_t *ds);

/*
 * Pure host helper (no GPU needed): the rank partition cco_train uses.  work_prefix[i] = products of primary items
 * [0, i) (exclusive prefix, n_items + 1 entries); bounds[r]..bounds[r+1] is rank r's contiguous item range, cut so
 * that every rank gets an equal share of (products + 1 per row).  Identical on every rank by construction.
 */
int cco_partition_rows(const int64_t *work_prefix, int32_t n_items, int32_t world_size, int32_t *bounds);

/*
 * Next row (SURVEY.md 8f-1), the ingest right before the boundary: Preparator.prepare + IndexedDatasetSpark.apply
 * (src/main/scala/Preparator.scala:44-87, 100-216) on integer-tokenised events.  Type 0 is the primary event: the
 * user dictionary = users with at least min_events_per_user primary events (duplicates counted, :129-132; 0/1 = any
 * primary event); every type is restricted to those users (:175-178); each type's item dictionary holds the items that
 * still have an event (:184); duplicates collapse (:201-208).  Dictionaries are in ascending raw-id order.
 * user_map [n_users_raw] and item_maps[t] [n_items_raw of t] are host arrays filled with the new id or -1.
 * The resulting dataset is resident in HBM and goes straight into cco_train_dataset.
 */
typedef struct {
  int64_t n_events;
  const int64_t *user; /* raw user id in [0, n_users_raw) */
  const int32_t *item; /* raw item id in [0, n_items_raw) */
  int32_t n_items_raw;
} cco_events_t;
int cco_ingest(cco_ctx_t *ctx, int32_t n_types, const cco_events_t *events, int64_t n_users_raw, int32_t min_events_per_user,
               int32_t *user_map, int32_t *const *item_maps, cco_dataset_t **out);
/*
 * Bench/test utility: the synthetic Zipf event streams of SURVEY.md 8(d) generated straight into HBM (no host event
 * arrays), then the same ingest as cco_ingest.  Stream of one event type, bit-identical to synth.py's numpy twin:
 *   h1 = mix64(mix64(seed) + (e + 1) * 0x9e3779b97f4a7c15), h2 = mix64(h1 ^ 0x6a09e667f3bcc909)      e = 0 .. n_events-1
 *   user = user_perm[upper_bound(user_cdf, (h1 >> 11) * 2^-53)], item = item_perm[upper_bound(item_cdf, (h2 >> 11) * 2^-53)]
 * cdf = inclusive, normalised cumulative weights over ranks; perm maps rank -> id.  All arrays are host pointers.
 * keep_item_space != 0: the item dictionary of every type is its raw id space (identity), not only the ids with an event.
 */
typedef struct {
  int64_t n_events;
  uint64_t seed;
  int32_t n_items;
  int32_t reserved;
  const double *item_cdf;   /* [n_items] */
  const int32_t *item_perm; /* [n_items] */
} cco_synth_type_t;
int cco_synth_ingest(cco_ctx_t *ctx, int32_t n_types, const cco_synth_type_t *types, int64_t n_users_raw, const double *user_cdf,
                     const int32_t *user_perm, int32_t min_events_per_user, int32_t keep_item_space, cco_dataset_t **out);
/* copy matrix i of a resident dataset into caller-provided host arrays ([n_rows + 1] and [nnz], see cco_dataset_shape) */
int cco_dataset_copy_to_host(const cco_dataset_t *ds, int32_t i, int64_t *row_ptr, int32_t *col_idx);
int cco_dataset_shape(const cco_dataset_t *ds, int32_t i, int64_t *n_rows, int32_t *n_cols, int64_t *nnz);
/* test helper: copy matrix i of a resident dataset back to the host (malloc'ed; free with cco_free) */
int cco_dataset_download(const cco_dataset_t *ds, int32_t i, int64_t **row_ptr, int32_t **col_idx);

/* CUDA-event stopwatch on the context's launch stream (what bench.py brackets its timed region with) */
int cco_timer_start(cco_ctx_t *ctx);
int cco_timer_stop(cco_ctx_t *ctx, float *ms);

/* SimilarityAnalysis.cooccurrencesIDSs convenience: one global (k, m) for every matrix */
int cco_cooccurrences_idss(cco_ctx_t *ctx, int32_t n_mats, const cco_csr_t *mats, int32_t seed,
                           int32_t max_interesting_items_per_thing, int32_t max_num_interactions,
                           uint32_t flags, cco_result_t **out);

/*
 * Result = List[IndexedDataset]; element i has rowIDs = A.columnIDs, columnIDs = B_i.columnIDs.
 * Indicator i as CSR over primary items: rows sorted by (llr desc, col asc), so the consumer's
 * sortBy(-llr) in package.scala:100-108 is a no-op.  count = k11 of each kept cell.
 * Pointers are owned by the result (pinned host memory) and live until cco_result_free.
 * row_ptr has (row_end - row_begin + 1) entries, relative to this rank's first row.
 */
int cco_result_num_matrices(const cco_result_t *r);
int cco_result_row_range(const cco_result_t *r, int32_t i, int64_t *row_begin, int64_t *row_end);
int cco_result_matrix(const cco_result_t *r, int32_t i, int64_t *n_rows, int32_t *n_cols,
                      const int64_t **row_ptr, const int32_t **col_idx, const double **llr,
                      const int32_t **count);
int cco_result_stats(const cco_result_t *r, cco_stats_t *out);
int cco_result_free(cco_result_t *r);

/*
 * Next row (SURVEY.md 8f-2): the model as the Elasticsearch bulk body, assembled on the device.  Replaces, per primary item,
 * IndexedDatasetConversions.toStringMapRDD (src/main/scala/package.scala:82-110: non-zeros ordered by -LLR, mapped to
 * column id strings, LLR dropped, empty rows -> empty array), URModel.save's groupAll + ("id" -> item)
 * (src/main/scala/URModel.scala:47-102) and the bulk serialisation of saveToEs with es.mapping.id = id
 * (src/main/scala/EsClient.scala:300-313).  One document per row of the result (a rank's slice or a merged model):
 *     {"index":{"_id":"<item>"}}\n{"id":"<item>","<names[0]>":["<col>",...],"<names[1]>":[...]}\n
 * Strings are JSON-escaped here ('"' and '\\' get a backslash, bytes < 0x20 become \u00xx, the rest passes through).
 * dictionaries: id i = bytes[offsets[i] .. offsets[i + 1]) (UTF-8); row_ids covers the primary item space, col_ids[i]
 * the item space of event i.  *out_bytes is pinned memory owned by the context: release it with cco_host_free.
 */
typedef struct {
  int64_t n;
  const int64_t *offsets; /* [n + 1] */
  const char *bytes;
} cco_dictionary_t;
int cco_format_es_bulk(cco_ctx_t *ctx, const cco_result_t *res, int32_t n_names, const char *const *names,
                       const cco_dictionary_t *row_ids, const cco_dictionary_t *col_ids, char **out_bytes, int64_t *out_len);

/*
 * Preparator.prepare from raw id strings (src/main/scala/Preparator.scala:111-126, 170-190), on the device.  Event type t
 * is two columns of strings: the user and the item id of event e are user.bytes / item.bytes [offsets[e] .. offsets[e + 1]).
 * Two ids are equal iff their bytes are equal (no normalisation; NUL, the empty id and non-ASCII bytes are ordinary ids).
 *  - user_dict: users of type 0 with at least min_events_per_user type-0 events (duplicates count; 0 or 1 = any), in order
 *    of first appearance among the type-0 events.  Users seen only in other types are dropped.
 *  - item_dicts[t]: the items of the type-t events whose user is in user_dict, in order of first appearance among those
 *    events.  Every type has its own id space.
 *  - *out: the same resident dataset cco_ingest builds from the same tokens (n_rows = user_dict.n for every type, columns
 *    ascending within a row, duplicates collapsed), ready for cco_train_dataset.
 * Every offsets / bytes pointer written into user_dict and item_dicts is pinned memory owned by the context: release each
 * with cco_host_free.  On error nothing is written and nothing is kept.
 * Errors: CCO_E_INVALID_ARG for null pointers, n_types < 1, user.n != item.n, n >= 2^32 events in a type, offsets[0] != 0
 * or decreasing offsets (all checked before the id bytes are read); CCO_E_UNSUPPORTED for a group context and for more
 * than 2^31 - 2 distinct type-0 users or distinct items in one item dictionary.
 */
typedef struct {
  cco_dictionary_t user; /* user.n == item.n == number of events */
  cco_dictionary_t item;
} cco_string_events_t;
int cco_ingest_strings(cco_ctx_t *ctx, int32_t n_types, const cco_string_events_t *events, int32_t min_events_per_user,
                       uint32_t flags, cco_dictionary_t *user_dict, cco_dictionary_t *item_dicts /* [n_types] */,
                       cco_dataset_t **out);

/*
 * Next row (SURVEY.md 8f-3): the backfill ranks of PopModel (src/main/scala/PopModel.scala:113-182) as per-item event
 * histograms over 1 / 2 / 3 time buckets of [start_ms, end_ms) -- what URAlgorithm.getRanksRDD (URAlgorithm.scala:537-560)
 * joins into the model.  events: (item index, event time in epoch milliseconds), already restricted to the ranking's event
 * names.  score[j] is meaningful iff present[j] != 0: `popular` lists the items with an event in the interval, `trending`
 * the items seen in both halves (newer - older), `hot` the items seen in all three thirds ((newer - middle) - (middle -
 * older)); `trending` / `hot` are empty when the older (or middle) bucket has no event at all, as in the reference.
 * RankingType.Random / UserDefined are not histograms and stay with the caller.
 */
enum { CCO_POP_POPULAR = 0, CCO_POP_TRENDING = 1, CCO_POP_HOT = 2 };
int cco_pop_model(cco_ctx_t *ctx, int32_t mode, int64_t n_events, const int32_t *item, const int64_t *time_ms, int32_t n_items,
                  int64_t start_ms, int64_t end_ms, double *score, unsigned char *present);

/*
 * The whole model document as URModel.save writes it with recsModel "all" (src/main/scala/URAlgorithm.scala:351-367,
 * 537-560; URModel.scala:57-102): groupAll(correlators ++ propertiesRDD), where propertiesRDD is the item properties
 * full-outer-joined with one rank field per ranking.  Rankings and property ids join the model rows by their id strings.
 *  - Documents: one per model row, in row order, then one per extra id in order of first appearance in the sequence
 *    (ranking 0's events, ranking 1's, ..., property ids).  An extra id is not a row and has a present rank in at least one
 *    ranking or a property entry.  An id seen only in rankings where it is not present (trending / hot inner joins, the
 *    empty-bucket rules) gets no document.
 *  - Fields, in this order: "id"; for rows only, the indicator arrays exactly as cco_format_es_bulk writes them;
 *    ,"<ranking name>":<score> for each ranking in which the id is present; ,<fragment> if the id's property fragment is
 *    not empty.  The action line is {"index":{"_id":"<id>"}} as in cco_format_es_bulk.
 *  - A property fragment is JSON object members without braces ("categories":["Phones"],"available":"2017-..."),
 *    serialised by the caller and spliced in verbatim: $set properties, userDefined ranks, random ranks.
 *  - Scores are the histograms of cco_pop_model (same bucket edges, same empty-bucket rules): integral doubles written as
 *    Java's Double.toString writes them: "<int>.0" when |v| < 10^7, otherwise d.dddE<n> with the trailing zeros of the
 *    fraction stripped and at least one fractional digit (1.0E7, 1.2345678E7, -8.589934592E9).
 *  - Ids are equal iff their bytes are equal.  With n_rankings == 0 and no properties the output is byte-identical to
 *    cco_format_es_bulk.
 * ranking.item holds the item id of every event of the ranking's event names (any user, any time); time_ms[e] is event
 * e's time in epoch milliseconds.  prop_ids and prop_json are both NULL or both given with the same n.  flags accepts
 * CCO_FLAG_INGEST_SHORT_HASH (tests only).  A group context formats on its first GPU.  *out_bytes is pinned memory owned by
 * the context: release it with cco_host_free.
 * Errors: CCO_E_INVALID_ARG for null pointers, only one of prop_ids / prop_json, row_ids.n != the model's row count, bad
 * offsets in any dictionary (checked before any id byte is read), end_ms < start_ms, a bad mode, a ranking name that is
 * null, repeated, "id" or an indicator name, two equal ids in row_ids, two equal ids in prop_ids.  CCO_E_UNSUPPORTED for a
 * result that is one rank's row slice (extra documents would repeat across ranks), more than 3 rankings, 2^31 or more
 * events in a ranking, 2^32 or more ids in all, or 2^31 or more distinct ids.
 */
typedef struct {
  const char *name;         /* ES field, e.g. "popRank" */
  int32_t mode;             /* CCO_POP_POPULAR / _TRENDING / _HOT */
  int32_t reserved;
  int64_t start_ms, end_ms; /* [end - duration, end), as cco_pop_model */
  cco_dictionary_t item;    /* the item id of every event of the ranking's event names */
  const int64_t *time_ms;   /* [item.n] event times */
} cco_ranking_t;
int cco_format_model_bulk(cco_ctx_t *ctx, const cco_result_t *res, int32_t n_names, const char *const *names,
                          const cco_dictionary_t *row_ids, const cco_dictionary_t *col_ids, int32_t n_rankings,
                          const cco_ranking_t *rankings, const cco_dictionary_t *prop_ids, const cco_dictionary_t *prop_json,
                          uint32_t flags, char **out_bytes, int64_t *out_len);

/*
 * Debug/parity entry (tests only): full integer co-occurrence matrix A^T B of two canonical
 * binary matrices computed by the same accumulation kernel as cco_train, no LLR, no top-k.
 * Output CSR over the columns of A with ascending column ids, malloc'ed; free with cco_free.
 */
int cco_debug_cooccurrence(cco_ctx_t *ctx, const cco_csr_t *a, const cco_csr_t *b, int64_t **row_ptr,
                           int32_t **col_idx, int32_t **count);
/* Debug/parity entry (tests only): sampleDownAndBinarize of one matrix on the device. */
int cco_debug_downsample(cco_ctx_t *ctx, const cco_csr_t *m, int32_t max_interactions, int32_t seed,
                         uint32_t flags, int64_t **row_ptr, int32_t **col_idx, int32_t *raw_col_counts,
                         int32_t *new_col_counts);
/* Debug/parity entry (tests only): the device LLR of n cells. */
int cco_debug_llr(cco_ctx_t *ctx, int64_t n, const int64_t *k11, const int64_t *k12, const int64_t *k21,
                  const int64_t *k22, uint32_t flags, double *out);
void cco_free(void *p);

#ifdef __cplusplus
}
#endif
#endif /* CCO_B200_H */
