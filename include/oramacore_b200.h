/*
 * oramacore_b200.h — C ABI of the B200-native OramaCore search hot path.
 *
 * The reference (oramasearch/oramacore @ 666ab48) has no plugin / FFI boundary for this
 * path: the seam is Rust-to-Rust (SURVEY.md §8b).  Each entry point below names the
 * reference interface it replaces (file:line relative to the reference root).  Plain
 * pointers and sizes only; all `out_*` buffers are caller-allocated HOST memory; the
 * library owns every device allocation behind the opaque handles.  The shared library
 * (liboramacore_b200.so) is CUDA-only: there is no CPU fallback, every call fails with
 * OC_ERR_CUDA when no sm_100-class device is usable.
 *
 * Status: 0 = OC_OK, <0 = error; text via oc_last_error() (thread-local, valid until the
 * next call on that thread).  Handles are Send+Sync: calls on one ctx are serialised
 * internally (one stream per ctx); different ctxs run concurrently.
 */
#ifndef ORAMACORE_B200_H
#define ORAMACORE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OC_OK 0
#define OC_ERR_INVALID (-1)     /* bad argument / shape                                   */
#define OC_ERR_CUDA (-2)        /* CUDA runtime failure (incl. "no device")               */
#define OC_ERR_OOM (-3)         /* device or host allocation failed                       */
#define OC_ERR_UNSUPPORTED (-4) /* e.g. limit+offset > OC_MAX_TOPK                        */
#define OC_ERR_COMM (-5)        /* NCCL failure / libnccl not loadable                    */

#define OC_MAX_TOPK 1024u       /* max limit+offset handled on device                     */
#define OC_MAX_TOKENS 32u       /* u32 token bitmask, token_score.rs:293                  */

#define OC_MODE_FULLTEXT 0      /* ScoreMode::FullText | Default, token_score.rs:472-484  */
#define OC_MODE_VECTOR 1        /* ScoreMode::Vector,             token_score.rs:485-494  */
#define OC_MODE_HYBRID 2        /* ScoreMode::Hybrid,             token_score.rs:495-503  */

#define OC_DTYPE_F32 0
#define OC_DTYPE_BF16 1         /* storage extension (reference stores f32, embedding_field.rs:232) */

typedef struct oc_ctx oc_ctx;   /* one device + stream + workspace (one per process/GPU)  */
typedef struct oc_emb oc_emb;   /* == one EmbeddingFieldStorage (embedding_field.rs:29-34) */
typedef struct oc_str oc_str;   /* == the StringFieldStorage set of one Index (string_field.rs:32-36) */
typedef struct oc_filter oc_filter; /* == a FilterResult<DocumentId> evaluated to a bitmap on the device (filter.rs:344-392) */

const char *oc_last_error(void);
int oc_version(void);
/* sizeof of {oc_search_params, oc_timing, oc_emb_info_t, oc_str_info_t} as compiled: lets a
 * binding (Rust repr(C), ctypes) verify its mirror of the structs at load time. */
void oc_abi_sizes(size_t out[4]);

/* ---- context ------------------------------------------------------------------------ */
/* Replaces nothing in the reference (it has no device); one ctx per GPU, one process per GPU. */
int oc_init(int device_id, oc_ctx **out);
void oc_shutdown(oc_ctx *ctx);
/* Number of SMs / device name, for bench reporting. */
int oc_device_info(oc_ctx *ctx, int *sm_count, size_t *hbm_bytes, char *name, size_t name_cap);

/* Document-sharded multi-GPU (SURVEY.md §8e; no reference analogue — the reference is
 * single-node).  Rank 0 creates the id, the host runtime broadcasts it, every rank joins.
 * After oc_comm_init, oc_search with params.sharded=1 all-gathers per-shard top-k over
 * NCCL/NVLink and merges on device; every rank receives the global answer.  When corpus df has
 * to be counted (a filter, multi-term tokens, tombstones: token_score.rs:262-275) the per-token
 * counters are summed across ranks with one ncclAllReduce before the idf is derived.  Every rank
 * must issue the same batch with the same flags: OC_SHARD_TOMBSTONES is set on ALL ranks while
 * ANY rank's string store holds uncommitted deletes (the host runtime routes deletes, so it knows). */
#define OC_SHARDED 1
#define OC_SHARD_TOMBSTONES 2
#define OC_SHARD_COUNT_DF 4      /* count corpus df across ranks (one ncclAllReduce) instead of using the per-term
                                    global_df tables: required, on EVERY rank, while any rank's string store lacks
                                    them (an oc_str_commit on a shard drops its table) */
#define OC_COMM_ID_BYTES 128
int oc_comm_unique_id(uint8_t out_id[OC_COMM_ID_BYTES]);
int oc_comm_init(oc_ctx *ctx, int world_size, int rank, const uint8_t id[OC_COMM_ID_BYTES]);
/* Optional: direct NVLink exchange of the per-shard top-k records instead of the NCCL all-gather.  After
 * oc_comm_init every rank exports the CUDA-IPC handle of its receive window, the host runtime all-gathers the
 * blobs (world x OC_P2P_HANDLE_BYTES, rank order) and every rank imports them.  From then on the pack kernel of a
 * sharded oc_search stores each query's record straight into all ranks' windows (peer memory over NVLink /
 * NVSwitch) and bumps a per-query arrival counter; the merge kernel waits on the counters: no library collective
 * on the data path.  Batches whose records exceed the 1 MiB window fall back to ncclAllGather. */
#define OC_P2P_HANDLE_BYTES 128
int oc_comm_p2p_export(oc_ctx *ctx, uint8_t out_handle[OC_P2P_HANDLE_BYTES]);
int oc_comm_p2p_import(oc_ctx *ctx, const uint8_t *handles);

/* ---- embedding store ------------------------------------------------------------------
 * EmbeddingFieldStorage::new (embedding_field.rs:64-78): metric fixed = cosine;
 * rescale_e5 = Model::rescale_score for the E5 family (python/embeddings.rs:71-92). */
int oc_emb_create(oc_ctx *ctx, uint32_t dim, int dtype, int rescale_e5, oc_emb **out);
void oc_emb_destroy(oc_emb *emb);
int oc_emb_reserve(oc_emb *emb, uint64_t n_rows);
/* EmbeddingFieldStorage::insert(DocumentId, Vec<Vec<f32>>) (embedding_field.rs:232-237),
 * batched: n vectors, doc_ids[i] may repeat (several chunks per document). rows = n x dim
 * row-major in the store's dtype, host memory. */
int oc_emb_insert(oc_emb *emb, const uint64_t *doc_ids, const void *rows, uint64_t n);
/* EmbeddingFieldStorage::delete (embedding_field.rs:240-242). */
int oc_emb_delete(oc_emb *emb, const uint64_t *doc_ids, uint64_t n);

typedef struct {
    uint64_t num_embeddings;  /* live vectors,   info().num_embeddings (embedding_field.rs:303-310) */
    uint64_t num_rows;        /* incl. tombstones */
    uint32_t dimensions;
    int dtype;
    uint64_t device_bytes;
} oc_emb_info_t;
int oc_emb_info(oc_emb *emb, oc_emb_info_t *out);

/* EmbeddingFieldStorage::search (embedding_field.rs:250-278) for B targets at once:
 * exact top-`limit` by cosine distance (== storage.search(target, limit, None) :255-266),
 * then similarity = 1 - distance, rescale, keep score >= similarity (:268-276).
 * filter_bits: NULL or a bitmap over DocumentId (FilterResult::contains, :54-61).
 * out_doc_ids/out_scores: B x limit, best first; out_counts[b] = hits kept (<= limit). */
int oc_emb_search(oc_emb *emb, const float *queries, uint32_t B, uint32_t limit, float similarity,
                  const uint64_t *filter_bits, uint64_t filter_nbits, uint64_t *out_doc_ids,
                  float *out_scores, uint32_t *out_counts);

/* ---- string (BM25F) store --------------------------------------------------------------
 * One oc_str holds all string fields of an Index over a shared row space
 * (row -> DocumentId).  Committed postings are handed over in CSR per field — what
 * StringFieldStorage::insert(DocumentId, IndexedValue{field_length:u16, terms}) accumulates
 * and compact() lays out (string_field.rs:155-177, 186-191). */
int oc_str_create(oc_ctx *ctx, uint32_t n_fields, oc_str **out);
void oc_str_destroy(oc_str *s);
/* row_doc_ids: NULL => DocumentId == row; must be ascending. document_count = N for idf
 * (Index::document_count, token_score.rs:221) — GLOBAL when sharded. */
int oc_str_set_rows(oc_str *s, uint64_t n_rows, const uint64_t *row_doc_ids, uint64_t document_count);
/* Postings of one field: term t owns [term_offsets[t], term_offsets[t+1]); rows ascending,
 * unique per term. avg_field_len = info().avg_field_length (string_field.rs:228-235),
 * global when sharded. global_df: NULL, or per-term corpus df across all shards. */
int oc_str_load_field(oc_str *s, uint32_t field, float avg_field_len, uint32_t n_terms,
                      const uint64_t *term_offsets, const uint32_t *post_row, const uint16_t *post_tf,
                      const uint16_t *post_len, const uint32_t *global_df);
/* StringFieldStorage::insert(DocumentId, IndexedValue{field_length:u16, terms}) (string_field.rs:155-177),
 * with terms already resolved to the field's term ids by the host dictionary: buffered on the host,
 * visible to searches after oc_str_commit. Re-inserting a document (before or after a commit) replaces its
 * postings in that field: the last insert wins.  A term id may appear once per call. */
int oc_str_insert(oc_str *s, uint32_t field, uint64_t doc_id, uint16_t field_len, uint32_t n_terms,
                  const uint32_t *term_ids, const uint16_t *tfs);
/* == compact(version) (string_field.rs:186-191): merges pending inserts / deletes into the NEXT snapshot of the
 * device-resident layout (rows = ascending doc ids; avg_field_len and document_count refreshed unless the caller
 * owns the corpus-wide values, see oc_str_set_global) and publishes it with a pointer swap — the reference's
 * CURRENT + versions/<n> scheme (embedding_field.rs:91-95).  The build runs WITHOUT the context lock on the
 * store's own stream: oc_search keeps serving the previous version meanwhile.  A failed commit changes nothing
 * (the pending ops stay queued).  One commit at a time per store. */
int oc_str_commit(oc_str *s);
/* StringFieldStorage::delete (string_field.rs:180-182).  Ops apply in call order like the reference's compact:
 * the committed rows of the document are tombstoned at once and its still-pending inserts are cancelled; an
 * insert after the delete is a new document. */
int oc_str_delete(oc_str *s, const uint64_t *doc_ids, uint64_t n);
/* The caller owns document_count (N of the idf = Index::document_count, token_score.rs:221 — it also counts
 * documents that have no string field, index/mod.rs:1460) and, when avg_field_len[n_fields] is given, the
 * corpus-wide average field lengths (this store is one shard of a larger index): oc_str_commit keeps the
 * caller's values instead of recomputing local ones (avg_field_len == NULL: averages stay locally computed).
 * Call again after commits to refresh them. */
int oc_str_set_global(oc_str *s, uint64_t document_count, const float *avg_field_len);

typedef struct {
    uint64_t total_documents;  /* rows                              */
    uint64_t total_postings;
    uint64_t unique_terms_count;
    uint32_t n_fields;
    uint64_t device_bytes;
    uint64_t version;          /* published snapshot, bumped by every load / commit (== CURRENT)  */
    uint64_t pending_postings; /* inserted, not yet committed (cf. pending_ops, embedding_field.rs:303-310) */
} oc_str_info_t;
int oc_str_info(oc_str *s, oc_str_info_t *out);

/* ---- search() ---------------------------------------------------------------------------
 * TokenScoreContext::execute (token_score.rs:460-509) + apply_omc_multipliers
 * (search.rs:39-48) + count (search.rs:482) + sort_token_scores/top_n (sort.rs:17-46,
 * 260-279) + skip(offset).take(limit) (search.rs:494-498), for a batch of B queries.
 *
 * Query text is resolved to index terms on the host (tokenise+stem token_score.rs:196-209;
 * prefix/Levenshtein expansion inside StringStorage); the ABI takes, per query, its tokens,
 * and per token the expanded (field, term id, weight) list, weight = field boost x
 * exact-match factor (the "ntf already includes boost" contract, token_score.rs:180-185). */
typedef struct {
    int mode;                          /* OC_MODE_*                                         */
    uint32_t n_queries;                /* B                                                  */
    uint32_t limit, offset;            /* Limit / SearchOffset (types.rs:747-756)            */
    float similarity;                  /* Similarity (types.rs:878-901); vector & hybrid     */
    float threshold;                   /* Threshold (types.rs:859-876); < 0 => None          */
    float bm25_k, bm25_b;              /* 1.2 / 0.75 (token_score.rs:283; bm25.rs:56-63)     */
    const float *q_vecs;               /* B x dim fp32 (vector, hybrid) or NULL              */
    const uint32_t *q_token_offsets;   /* B+1 (fulltext, hybrid) or NULL                     */
    const uint32_t *token_term_offsets;/* n_tokens+1                                         */
    const uint32_t *term_field;        /* per expanded term                                  */
    const uint32_t *term_id;
    const float *term_weight;
    const uint64_t *filter_bits;       /* NULL or bitmap over DocumentId                     */
    uint64_t filter_nbits;
    const uint64_t *omc_doc_ids;       /* OMC multipliers sorted by doc id (index/mod.rs:1720-1739) */
    const float *omc_mult;
    uint64_t n_omc;
    int sharded;                       /* OC_SHARDED [| OC_SHARD_TOMBSTONES | OC_SHARD_COUNT_DF] => merge across oc_comm ranks */
    uint32_t vector_limit;             /* 0 => limit.  Candidate depth of the vector stage = limit_hint, which the
                                          reference keeps at `limit` while top_n takes limit+offset (search.rs:330-336):
                                          a caller that needs the rows [0, limit+offset) of one index (multi-index
                                          union, oc_merge_results) asks for limit' = limit+offset, vector_limit = limit */
    const struct oc_filter *filter;    /* NULL, or a device-resident DocumentId bitmap (oc_filter_*): takes precedence
                                          over filter_bits and is not re-uploaded per call                           */
} oc_search_params;

/* out_doc_ids/out_scores: B x limit (best first, after offset); out_n[b] hits written;
 * out_count[b] = all matching documents. emb may be NULL for fulltext, str NULL for vector. */
int oc_search(oc_ctx *ctx, oc_emb *emb, oc_str *str, const oc_search_params *p,
              uint64_t *out_doc_ids, float *out_scores, uint32_t *out_n, uint64_t *out_count);

/* ---- filters on the device -------------------------------------------------------------------------
 * FilterContext::execute_filter (read/index/filter.rs:344-392) yields a FilterResult tree: And / Or / Not over
 * plain DocumentId sets (:351-362, 378-389), consulted by the scorers through contains(doc)
 * (embedding_field.rs:54-61, string_field.rs:66-69).  Here a FilterResult is a bitmap over DocumentId
 * [0, nbits) that lives on the device: build the leaves from id lists, combine with And / Or / Not (word-wise
 * kernels), hand the handle to any number of oc_search / oc_search_facets calls (no per-call upload).
 * execute_filter's own rule — AND the where-filter with NOT(uncommitted deletes) — is oc_filter_and +
 * oc_filter_not over an id leaf of the deleted documents. */
int oc_filter_from_ids(oc_ctx *ctx, const uint64_t *doc_ids, uint64_t n, uint64_t nbits, oc_filter **out);  /* PlainFilterResult::from_iter; ids >= nbits ignored */
int oc_filter_from_bits(oc_ctx *ctx, const uint64_t *bits, uint64_t nbits, oc_filter **out);
int oc_filter_and(const oc_filter *a, const oc_filter *b, oc_filter **out);   /* FilterResult::And */
int oc_filter_or(const oc_filter *a, const oc_filter *b, oc_filter **out);    /* FilterResult::Or  */
int oc_filter_not(const oc_filter *a, oc_filter **out);                       /* FilterResult::Not (within [0, nbits)) */
int oc_filter_count(const oc_filter *f, uint64_t *out);                       /* documents that pass */
int oc_filter_read(const oc_filter *f, uint64_t *out_bits /* (nbits+63)/64 words */);
void oc_filter_destroy(oc_filter *f);

/* ---- facets over the score set ------------------------------------------------------------------
 * FacetContext::execute (read/index/facet.rs:147-209): for each requested variant of a filter field — bool
 * true / false (bool_field.rs:182-208), a number range [from, to], both ends inclusive (number_field.rs:368-387,
 * NumberFilter::Between), a string_filter key (string_filter_field.rs:175-193) — the number of the variant's
 * documents that are keys of the score map.  The store keeps, per field, the variants' document lists on the
 * device (number fields: documents sorted by value, so a range is a slice); a search in facet mode makes the tile
 * scorer emit the bitmap of matched documents (+ the vector hits) and one kernel counts every (query, variant).
 * As in the reference (search.rs:361-396) the score map is computed WITHOUT the where-filter (uncommitted deletes
 * stay excluded), so p->filter_bits / p->filter are ignored here: hits come from oc_search, facets from this call.
 * A document may be listed under several variants (array values).  nbits: DocumentId space [0, nbits). */
typedef struct oc_facets oc_facets;
typedef struct {
    uint32_t field;     /* id returned by oc_facets_add_*                                     */
    uint32_t variant;   /* bool / string fields: variant index                                */
    double from, to;    /* number fields: inclusive range                                     */
} oc_facet_req;
int oc_facets_create(oc_ctx *ctx, uint64_t nbits, oc_facets **out);
void oc_facets_destroy(oc_facets *f);
int oc_facets_add_field(oc_facets *f, uint32_t n_variants, const uint64_t *variant_offsets /* n+1 */, const uint64_t *doc_ids,
                        uint32_t *out_field);
int oc_facets_add_number_field(oc_facets *f, uint64_t n, const double *values_sorted, const uint64_t *doc_ids, uint32_t *out_field);
/* out_counts: n_queries x n_reqs.  emb / str as for oc_search (the mode decides which are needed). */
int oc_search_facets(oc_ctx *ctx, oc_emb *emb, oc_str *str, oc_facets *facets, const oc_search_params *p,
                     const oc_facet_req *reqs, uint32_t n_reqs, uint64_t *out_counts);

/* ---- sortBy over the score map -----------------------------------------------------------------------
 * sort_token_scores with Some(sort_by) (read/sort.rs:17-98, 236-257): instead of the relevance top-n, the score map's
 * keys in the order of a number, date or bool field — value groups in the requested order (IndexSortContext::execute,
 * read/index/sort.rs:186-264), ascending DocumentId inside a group — then skip(offset).take(limit).  Each hit carries
 * its score-map value.  The score map is exactly oc_search's: where-filter, uncommitted deletes, threshold, OMC and
 * hybrid fusion apply, and out_count is oc_search's count.  A document without a value in the field is never emitted
 * but still counts.  Number values compare as f64 (NaN rejected), dates as exact i64, bools false < true.  A document
 * may hold one value per field (listing it twice is OC_ERR_INVALID).  A store is immutable once built: to refresh it,
 * build a new one.  nbits: DocumentId space [0, nbits), at most 2^32. */
typedef struct oc_sort oc_sort;            /* == the bool / number / date field storages IndexSortContext reads */
int oc_sort_create(oc_ctx *ctx, uint64_t nbits, oc_sort **out);
void oc_sort_destroy(oc_sort *s);
int oc_sort_add_number_field(oc_sort *s, uint64_t n, const uint64_t *doc_ids, const double *values, uint32_t *out_field);
int oc_sort_add_date_field(oc_sort *s, uint64_t n, const uint64_t *doc_ids, const int64_t *ts, uint32_t *out_field);
int oc_sort_add_bool_field(oc_sort *s, uint64_t n_true, const uint64_t *true_docs, uint64_t n_false, const uint64_t *false_docs,
                           uint32_t *out_field);
/* Outputs as oc_search; out_keys: NULL or B x limit, the sort value of each hit (bool: 0 / 1, date: the timestamp as
 * f64).  An unknown field is OC_ERR_INVALID (SortFieldNotFound); p->sharded is OC_ERR_UNSUPPORTED.  OC_SORT_FORM=walk |
 * gather forces one of the two device selection forms (otherwise each query picks one from its count). */
int oc_search_sorted(oc_ctx *ctx, oc_emb *emb, oc_str *str, oc_sort *s, uint32_t field, int descending,
                     const oc_search_params *p, uint64_t *out_doc_ids, float *out_scores, uint32_t *out_n,
                     uint64_t *out_count, double *out_keys);
/* The selection form (0 = walk, 1 = gather) each query of the last oc_search_sorted on ctx took; n_queries <= its B. */
int oc_sort_last_forms(oc_ctx *ctx, uint32_t n_queries, uint8_t *out);
/* Multi-index union in field order (MergeSortedIterator, read/sort.rs:491-560), host only, like oc_merge_results:
 * per index the rows of oc_search_sorted with limit' = limit+offset, offset' = 0, vector_limit = limit and their
 * out_keys.  Equal keys: the lower index first.  Keys compare exactly (the reference clamps date keys to i32). */
int oc_merge_sorted_results(uint32_t n_indexes, uint32_t n_queries, uint32_t limit, uint32_t offset, uint32_t in_stride,
                            int descending, const uint64_t *const *doc_ids, const float *const *scores,
                            const double *const *keys, const uint32_t *const *n, const uint64_t *const *counts,
                            uint64_t *out_doc_ids, float *out_scores, uint32_t *out_n, uint64_t *out_count);

/* ---- multi-index collections ---------------------------------------------------------------------
 * search_on_indexes runs every index of a collection into ONE score map (read/search.rs:304-338,
 * token_score.rs:472-499): document ids are unique per collection, so the per-index maps are disjoint; hybrid
 * normalisation is per index; count = sum of the per-index counts; then one top_n(limit+offset) and
 * skip(offset).take(limit) (search.rs:482-498).  The caller runs oc_search once per index with
 * limit' = limit+offset, offset' = 0, vector_limit = limit and merges here (host; k sorted lists of <= limit'
 * entries).  in_stride = limit' (row stride of the per-index arrays).  Ties: ascending document id. */
int oc_merge_results(uint32_t n_indexes, uint32_t n_queries, uint32_t limit, uint32_t offset, uint32_t in_stride,
                     const uint64_t *const *doc_ids, const float *const *scores, const uint32_t *const *n,
                     const uint64_t *const *counts, uint64_t *out_doc_ids /* B x limit */, float *out_scores,
                     uint32_t *out_n, uint64_t *out_count);

/* ---- term dictionary and query-term resolution (host only; no device needed) ------------------------
 * The step the reference performs before the posting walk: TextParser::tokenize_and_stem(term) —
 * originals, plus stems unless `exact`, [""] when nothing is left (token_score.rs:196-209) — and the
 * expansion of every token to index terms inside StringStorage's FST (string_field.rs:208-225): the exact
 * term when `exact` (tolerance Some(0), token_score.rs:240), terms within Levenshtein distance t for
 * tolerance = Some(t) (tests/fulltext_search.rs:956-1018), prefix expansion otherwise (:633-644); an
 * exactly matching term carries exact_match_boost (tests/boost_integration.rs:449-490; the reference's
 * constant lives in oramacore_fields 0.2.0 and is not visible: 2.0 is this library's default).
 * Term ids are stable: the id a term gets from oc_dict_add_terms is the id oc_str_insert / the loaded
 * posting lists use for it.  Output = the CSR arrays of oc_search_params. */
typedef struct oc_dict oc_dict;
typedef struct oc_resolved oc_resolved;
/* writes the stem of tok[0..len) into out (cap bytes) and returns its length; 0 = no stem */
typedef size_t (*oc_stem_fn)(const char *tok, size_t len, char *out, size_t cap, void *user);
typedef struct {
    const char *const *texts;   /* n_queries NUL-terminated query strings ("term" of SearchParams)        */
    uint32_t n_queries;
    int exact;                  /* exact match (types.rs "exact")                                          */
    int tolerance;              /* < 0: None => prefix expansion; t >= 0: Levenshtein <= t (bytes)         */
    const float *field_boost;   /* n_fields, NULL = 1.0 (boost: field -> f32, token_score.rs:138-147)      */
    const uint8_t *field_mask;  /* n_fields, NULL = all string fields (properties, token_score.rs:159-178) */
    float exact_match_boost;    /* <= 0: default 2.0                                                       */
} oc_resolve_params;
int oc_dict_create(uint32_t n_fields, oc_dict **out);
void oc_dict_destroy(oc_dict *d);
int oc_dict_add_terms(oc_dict *d, uint32_t field, const char *const *terms, uint32_t n, uint32_t *out_ids);
int oc_dict_lookup(oc_dict *d, uint32_t field, const char *term, uint32_t *out_id);   /* 0xffffffff = absent */
uint32_t oc_dict_size(oc_dict *d, uint32_t field);
int oc_dict_set_stemmer(oc_dict *d, oc_stem_fn fn, void *user);
/* the Snowball English (Porter2) algorithm with the oc_stem_fn signature, from csrc/stem_en.h; pinned to its published
 * sample vocabulary: oc_dict_set_stemmer(d, oc_stem_english, NULL).  The reference's own stemmer lives in the
 * un-vendored oramacore_lib::nlp::TextParser; a host that links it passes its own function instead. */
size_t oc_stem_english(const char *tok, size_t len, char *out, size_t cap, void *user);
int oc_dict_resolve(oc_dict *d, const oc_resolve_params *p, oc_resolved **out);
void oc_resolved_arrays(const oc_resolved *r, const uint32_t **q_token_offsets, const uint32_t **token_term_offsets,
                        const uint32_t **term_field, const uint32_t **term_id, const float **term_weight,
                        uint32_t *n_tokens, uint32_t *n_terms);
/* points p's query arrays (and n_queries) at r; r must outlive the oc_search call */
void oc_resolved_fill(const oc_resolved *r, oc_search_params *p);
void oc_resolved_free(oc_resolved *r);

/* ---- micro-batching front --------------------------------------------------------------
 * The reference runs one search per request task, many at a time (bin/oramacore.rs:76-79,
 * SURVEY.md §8b "Threading"); the GPU path earns its throughput on batches.  A batcher coalesces
 * concurrent single-query oc_search calls: the first submitter of a group leads it, waits up to
 * max_wait_us (or until max_batch queries are in), runs ONE oc_search for the group and scatters
 * the per-query results to the blocked callers.  Coalesced: queries with the same (mode, limit,
 * offset, similarity, threshold, bm25_k, bm25_b), no filter, no OMC, not sharded; any other call
 * is passed straight to oc_search.  p->n_queries must be 1; outputs as for oc_search with B = 1. */
typedef struct oc_batcher oc_batcher;
int oc_batcher_create(oc_ctx *ctx, oc_emb *emb, oc_str *str, uint32_t max_batch, uint32_t max_wait_us, oc_batcher **out);
void oc_batcher_destroy(oc_batcher *b);
int oc_batcher_search(oc_batcher *b, const oc_search_params *p, uint64_t *out_doc_ids, float *out_scores,
                      uint32_t *out_n, uint64_t *out_count);
/* queries that went through a coalesced batch / number of batches / calls passed straight through */
int oc_batcher_stats(oc_batcher *b, uint64_t *n_queries, uint64_t *n_batches, uint64_t *n_direct);

/* ---- pinned host buffers (optional) ----------------------------------------------------------
 * Query vectors handed to oc_search from memory obtained here (or otherwise page-locked) are
 * DMA'd straight from the caller's buffer; pageable buffers are staged through a pinned blob. */
int oc_pinned_alloc(size_t bytes, void **out);
void oc_pinned_free(void *p);

/* ---- measurement ------------------------------------------------------------------------
 * CUDA-event timings (ms, on the ctx stream) of the last oc_search / oc_emb_search on this
 * ctx, and launch counts. */
typedef struct {
    float h2d_ms;        /* query / term / filter upload                                   */
    float device_ms;     /* all kernels of the call (inputs resident)                      */
    float d2h_ms;        /* result download                                                */
    float scan_ms;       /* embedding scan kernel(s) only                                  */
    float bm25_ms;       /* posting-list scorer kernel(s) only                             */
    float fuse_ms;       /* merge / fusion / top-k kernel(s)                               */
    float comm_ms;       /* all-gather + cross-shard merge                                 */
    uint32_t kernel_launches;
    uint32_t scan_launches;
    uint64_t scan_bytes;     /* algorithmic bytes swept by the scan kernels (rows x stride x elem) */
    uint64_t bm25_postings;  /* postings walked by the scorer (x8 B = algorithmic bytes)    */
    uint64_t h2d_bytes, d2h_bytes;
    uint32_t scan_tensor_core;   /* 1 => the batched tcgen05 (tf32 select + exact re-score) scan ran */
    uint32_t scan_unproven;      /* queries whose candidate buffers overflowed in the tensor-core scan and were
                                    re-run through the exact sweep (device_ms includes that re-run)     */
    uint32_t scan_variant;       /* OC_SCAN_*: which sweep kernel served the batch                      */
    float scan_sweep_ms;         /* device time of the sweep launch(es) alone (scan_ms also holds the threshold pass) */
    float rerun_ms;              /* device time of re-running flagged queries (exact sweep + second tail), in device_ms */
    uint32_t scan_rescored;      /* rows re-scored in exact fp32 per query (batch average) by the tensor-core scan */
} oc_timing;
#define OC_SCAN_EXACT 0          /* emb_scan_kernel: exact fp32 sweep (B < 8, limit > 32, tiny stores)          */
#define OC_SCAN_TC_TF32 1        /* emb_gemm_kernel: kind::tf32 on the fp32 rows, one CTA per SM               */
#define OC_SCAN_TC_TF32_PAIR 2   /* emb_gemm_pair_kernel: same, CTA pairs (cta_group::2)                       */
#define OC_SCAN_TC_CVT_PAIR 3    /* emb_gemm_cvt_kernel: fp32 rows rounded to bf16 in the SM, kind::f16, pairs */
#define OC_SCAN_TC_BF16 4        /* emb_gemm_kernel on a bf16 store (kind::f16)                                */
#define OC_SCAN_TC_BF16_PAIR 5   /* emb_gemm_pair_kernel on a bf16 store                                       */
int oc_last_timing(oc_ctx *ctx, oc_timing *out);
/* Total kernels this library has launched on ctx since oc_init. */
uint64_t oc_launch_count(oc_ctx *ctx);

#ifdef __cplusplus
}
#endif
#endif
