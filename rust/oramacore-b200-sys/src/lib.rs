//! Bindings for `include/oramacore_b200.h` (C ABI of the B200-native search hot path) and safe
//! wrappers shaped like the reference types they replace:
//!   * `EmbeddingField`  ~ `EmbeddingFieldStorage` (read/index/embedding_field.rs:29-34)
//!   * `StringFields`    ~ the `StringFieldStorage` set of an Index (read/index/string_field.rs:32-36)
//!   * `Ctx::search`     ~ `TokenScoreContext::execute` + OMC + count + top-N
//!                         (token_score.rs:460-509, search.rs:39-48, 482-498, sort.rs:260-279)
//! SOURCE ONLY: the build image has no Rust toolchain; the identical ABI is exercised by the
//! ctypes mirror (`oramacore_b200/_lib.py`) and the GPU parity tests.
use std::ffi::{c_char, c_int, c_void, CStr};

#[repr(C)] pub struct OcCtx { _p: [u8; 0] }
#[repr(C)] pub struct OcEmb { _p: [u8; 0] }
#[repr(C)] pub struct OcStr { _p: [u8; 0] }
#[repr(C)] pub struct OcBatcher { _p: [u8; 0] }
#[repr(C)] pub struct OcFilter { _p: [u8; 0] }
#[repr(C)] pub struct OcFacets { _p: [u8; 0] }
#[repr(C)] pub struct OcSort { _p: [u8; 0] }
#[repr(C)] pub struct OcDict { _p: [u8; 0] }
#[repr(C)] pub struct OcResolved { _p: [u8; 0] }

pub const OC_MODE_FULLTEXT: c_int = 0;
pub const OC_MODE_VECTOR: c_int = 1;
pub const OC_MODE_HYBRID: c_int = 2;
pub const OC_DTYPE_F32: c_int = 0;
pub const OC_DTYPE_BF16: c_int = 1;
/// `OcSearchParams::sharded`: merge across `oc_comm` ranks; add `OC_SHARD_TOMBSTONES` on every rank while
/// any rank's string store holds uncommitted deletes (the df all-reduce must be entered by all ranks).
pub const OC_SHARDED: c_int = 1;
pub const OC_SHARD_TOMBSTONES: c_int = 2;
/// count corpus df across ranks instead of using replicated tables (a commit on a shard drops them)
pub const OC_SHARD_COUNT_DF: c_int = 4;

#[repr(C)]
pub struct OcSearchParams {
    pub mode: c_int,
    pub n_queries: u32,
    pub limit: u32,
    pub offset: u32,
    pub similarity: f32,
    pub threshold: f32, // < 0 => None
    pub bm25_k: f32,
    pub bm25_b: f32,
    pub q_vecs: *const f32,
    pub q_token_offsets: *const u32,
    pub token_term_offsets: *const u32,
    pub term_field: *const u32,
    pub term_id: *const u32,
    pub term_weight: *const f32,
    pub filter_bits: *const u64,
    pub filter_nbits: u64,
    pub omc_doc_ids: *const u64,
    pub omc_mult: *const f32,
    pub n_omc: u64,
    pub sharded: c_int,
    pub vector_limit: u32,          // 0 => limit (limit_hint of the vector stage, search.rs:330-336)
    pub filter: *const OcFilter,    // device-resident FilterResult bitmap; wins over filter_bits
}

#[repr(C)]
pub struct OcFacetReq { pub field: u32, pub variant: u32, pub from: f64, pub to: f64 }

#[repr(C)]
pub struct OcResolveParams {
    pub texts: *const *const c_char,
    pub n_queries: u32,
    pub exact: c_int,
    pub tolerance: c_int,           // < 0 => None (prefix expansion)
    pub field_boost: *const f32,
    pub field_mask: *const u8,
    pub exact_match_boost: f32,
}
pub type OcStemFn = unsafe extern "C" fn(tok: *const c_char, len: usize, out: *mut c_char, cap: usize, user: *mut c_void) -> usize;

extern "C" {
    pub fn oc_last_error() -> *const c_char;
    pub fn oc_abi_sizes(out: *mut usize);
    pub fn oc_init(device_id: c_int, out: *mut *mut OcCtx) -> c_int;
    pub fn oc_shutdown(ctx: *mut OcCtx);
    pub fn oc_comm_unique_id(out_id: *mut u8) -> c_int;
    pub fn oc_comm_init(ctx: *mut OcCtx, world: c_int, rank: c_int, id: *const u8) -> c_int;
    pub fn oc_emb_create(ctx: *mut OcCtx, dim: u32, dtype: c_int, rescale_e5: c_int, out: *mut *mut OcEmb) -> c_int;
    pub fn oc_emb_destroy(emb: *mut OcEmb);
    pub fn oc_emb_insert(emb: *mut OcEmb, doc_ids: *const u64, rows: *const c_void, n: u64) -> c_int;
    pub fn oc_emb_delete(emb: *mut OcEmb, doc_ids: *const u64, n: u64) -> c_int;
    pub fn oc_emb_search(emb: *mut OcEmb, queries: *const f32, b: u32, limit: u32, similarity: f32,
                         filter_bits: *const u64, filter_nbits: u64, out_doc_ids: *mut u64,
                         out_scores: *mut f32, out_counts: *mut u32) -> c_int;
    pub fn oc_str_create(ctx: *mut OcCtx, n_fields: u32, out: *mut *mut OcStr) -> c_int;
    pub fn oc_str_destroy(s: *mut OcStr);
    pub fn oc_str_set_rows(s: *mut OcStr, n_rows: u64, row_doc_ids: *const u64, document_count: u64) -> c_int;
    pub fn oc_str_load_field(s: *mut OcStr, field: u32, avg_field_len: f32, n_terms: u32, term_offsets: *const u64,
                             post_row: *const u32, post_tf: *const u16, post_len: *const u16,
                             global_df: *const u32) -> c_int;
    pub fn oc_str_delete(s: *mut OcStr, doc_ids: *const u64, n: u64) -> c_int;
    /// StringFieldStorage::insert (string_field.rs:155-177): buffered until `oc_str_commit`
    pub fn oc_str_insert(s: *mut OcStr, field: u32, doc_id: u64, field_len: u16, n_terms: u32,
                         term_ids: *const u32, tfs: *const u16) -> c_int;
    /// compaction (string_field.rs:186-191): merges pending inserts / deletes into the device layout
    pub fn oc_str_commit(s: *mut OcStr) -> c_int;
    /// page-locked host buffers: query vectors placed here are DMA'd without staging
    pub fn oc_pinned_alloc(bytes: usize, out: *mut *mut c_void) -> c_int;
    /// micro-batching front: one query per call from many threads, coalesced into batched `oc_search`
    pub fn oc_batcher_create(ctx: *mut OcCtx, emb: *mut OcEmb, s: *mut OcStr, max_batch: u32, max_wait_us: u32,
                             out: *mut *mut OcBatcher) -> c_int;
    pub fn oc_batcher_destroy(b: *mut OcBatcher);
    pub fn oc_batcher_search(b: *mut OcBatcher, p: *const OcSearchParams, out_doc_ids: *mut u64, out_scores: *mut f32,
                             out_n: *mut u32, out_count: *mut u64) -> c_int;
    pub fn oc_batcher_stats(b: *mut OcBatcher, n_queries: *mut u64, n_batches: *mut u64, n_direct: *mut u64) -> c_int;
    pub fn oc_pinned_free(p: *mut c_void);
    pub fn oc_search(ctx: *mut OcCtx, emb: *mut OcEmb, s: *mut OcStr, p: *const OcSearchParams,
                     out_doc_ids: *mut u64, out_scores: *mut f32, out_n: *mut u32, out_count: *mut u64) -> c_int;
    /// caller-owned N / average field lengths (shards; Index::document_count), kept across commits
    pub fn oc_str_set_global(s: *mut OcStr, document_count: u64, avg_field_len: *const f32) -> c_int;
    // FilterResult (filter.rs:344-392) evaluated on the device
    pub fn oc_filter_from_ids(ctx: *mut OcCtx, doc_ids: *const u64, n: u64, nbits: u64, out: *mut *mut OcFilter) -> c_int;
    pub fn oc_filter_from_bits(ctx: *mut OcCtx, bits: *const u64, nbits: u64, out: *mut *mut OcFilter) -> c_int;
    pub fn oc_filter_and(a: *const OcFilter, b: *const OcFilter, out: *mut *mut OcFilter) -> c_int;
    pub fn oc_filter_or(a: *const OcFilter, b: *const OcFilter, out: *mut *mut OcFilter) -> c_int;
    pub fn oc_filter_not(a: *const OcFilter, out: *mut *mut OcFilter) -> c_int;
    pub fn oc_filter_count(f: *const OcFilter, out: *mut u64) -> c_int;
    pub fn oc_filter_read(f: *const OcFilter, out_bits: *mut u64) -> c_int;
    pub fn oc_filter_destroy(f: *mut OcFilter);
    // facets over the score set (facet.rs:147-209)
    pub fn oc_facets_create(ctx: *mut OcCtx, nbits: u64, out: *mut *mut OcFacets) -> c_int;
    pub fn oc_facets_destroy(f: *mut OcFacets);
    pub fn oc_facets_add_field(f: *mut OcFacets, n_variants: u32, variant_offsets: *const u64, doc_ids: *const u64, out_field: *mut u32) -> c_int;
    pub fn oc_facets_add_number_field(f: *mut OcFacets, n: u64, values_sorted: *const f64, doc_ids: *const u64, out_field: *mut u32) -> c_int;
    pub fn oc_search_facets(ctx: *mut OcCtx, emb: *mut OcEmb, s: *mut OcStr, f: *mut OcFacets, p: *const OcSearchParams,
                            reqs: *const OcFacetReq, n_reqs: u32, out_counts: *mut u64) -> c_int;
    /// search_on_indexes' union of the per-index maps (search.rs:304-338, 482-498), host side
    pub fn oc_merge_results(n_indexes: u32, n_queries: u32, limit: u32, offset: u32, in_stride: u32,
                            doc_ids: *const *const u64, scores: *const *const f32, n: *const *const u32,
                            counts: *const *const u64, out_doc_ids: *mut u64, out_scores: *mut f32,
                            out_n: *mut u32, out_count: *mut u64) -> c_int;
    // sortBy over the score map (read/sort.rs:17-98, index/sort.rs:186-264)
    pub fn oc_sort_create(ctx: *mut OcCtx, nbits: u64, out: *mut *mut OcSort) -> c_int;
    pub fn oc_sort_destroy(s: *mut OcSort);
    pub fn oc_sort_add_number_field(s: *mut OcSort, n: u64, doc_ids: *const u64, values: *const f64, out_field: *mut u32) -> c_int;
    pub fn oc_sort_add_date_field(s: *mut OcSort, n: u64, doc_ids: *const u64, ts: *const i64, out_field: *mut u32) -> c_int;
    pub fn oc_sort_add_bool_field(s: *mut OcSort, n_true: u64, true_docs: *const u64, n_false: u64, false_docs: *const u64,
                                  out_field: *mut u32) -> c_int;
    pub fn oc_search_sorted(ctx: *mut OcCtx, emb: *mut OcEmb, s: *mut OcStr, st: *mut OcSort, field: u32, descending: c_int,
                            p: *const OcSearchParams, out_doc_ids: *mut u64, out_scores: *mut f32, out_n: *mut u32,
                            out_count: *mut u64, out_keys: *mut f64) -> c_int;
    pub fn oc_sort_last_forms(ctx: *mut OcCtx, n_queries: u32, out: *mut u8) -> c_int;
    /// MergeSortedIterator (read/sort.rs:491-560) over per-index sorted rows, host side
    pub fn oc_merge_sorted_results(n_indexes: u32, n_queries: u32, limit: u32, offset: u32, in_stride: u32, descending: c_int,
                                   doc_ids: *const *const u64, scores: *const *const f32, keys: *const *const f64,
                                   n: *const *const u32, counts: *const *const u64, out_doc_ids: *mut u64, out_scores: *mut f32,
                                   out_n: *mut u32, out_count: *mut u64) -> c_int;
    // term dictionary + batch query resolution (tokenize_and_stem + FST expansion), host only
    pub fn oc_dict_create(n_fields: u32, out: *mut *mut OcDict) -> c_int;
    pub fn oc_dict_destroy(d: *mut OcDict);
    pub fn oc_dict_add_terms(d: *mut OcDict, field: u32, terms: *const *const c_char, n: u32, out_ids: *mut u32) -> c_int;
    pub fn oc_dict_lookup(d: *mut OcDict, field: u32, term: *const c_char, out_id: *mut u32) -> c_int;
    pub fn oc_dict_size(d: *mut OcDict, field: u32) -> u32;
    pub fn oc_dict_set_stemmer(d: *mut OcDict, f: Option<OcStemFn>, user: *mut c_void) -> c_int;
    pub fn oc_dict_resolve(d: *mut OcDict, p: *const OcResolveParams, out: *mut *mut OcResolved) -> c_int;
    pub fn oc_resolved_fill(r: *const OcResolved, p: *mut OcSearchParams);
    pub fn oc_resolved_free(r: *mut OcResolved);
}

fn check(rc: c_int) -> anyhow::Result<()> {
    if rc == 0 { return Ok(()); }
    let msg = unsafe { CStr::from_ptr(oc_last_error()) }.to_string_lossy().into_owned();
    anyhow::bail!("oramacore_b200 error {rc}: {msg}")
}

pub struct Ctx(*mut OcCtx);
unsafe impl Send for Ctx {}
unsafe impl Sync for Ctx {}
impl Ctx {
    pub fn new(device: i32) -> anyhow::Result<Self> {
        let mut sizes = [0usize; 4];
        unsafe { oc_abi_sizes(sizes.as_mut_ptr()) };
        assert_eq!(sizes[0], std::mem::size_of::<OcSearchParams>(), "oc_search_params layout drift");
        let mut p = std::ptr::null_mut();
        check(unsafe { oc_init(device, &mut p) })?;
        Ok(Ctx(p))
    }
}
impl Drop for Ctx { fn drop(&mut self) { unsafe { oc_shutdown(self.0) } } }

/// `EmbeddingFieldStorage` (embedding_field.rs): same method shapes.
pub struct EmbeddingField { h: *mut OcEmb, dim: usize }
unsafe impl Send for EmbeddingField {}
unsafe impl Sync for EmbeddingField {}
impl EmbeddingField {
    pub fn new(ctx: &Ctx, dimensions: usize, is_e5: bool) -> anyhow::Result<Self> {
        let mut h = std::ptr::null_mut();
        check(unsafe { oc_emb_create(ctx.0, dimensions as u32, 0, is_e5 as c_int, &mut h) })?;
        Ok(Self { h, dim: dimensions })
    }
    /// insert(DocumentId, Vec<Vec<f32>>)  (embedding_field.rs:232-237)
    pub fn insert(&self, doc_id: u64, vectors: &[Vec<f32>]) -> anyhow::Result<()> {
        let flat: Vec<f32> = vectors.iter().flat_map(|v| v.iter().copied()).collect();
        debug_assert_eq!(flat.len(), vectors.len() * self.dim);
        let ids = vec![doc_id; vectors.len()];
        check(unsafe { oc_emb_insert(self.h, ids.as_ptr(), flat.as_ptr() as *const c_void, ids.len() as u64) })
    }
    /// delete(DocumentId)  (embedding_field.rs:240-242)
    pub fn delete(&self, doc_id: u64) -> anyhow::Result<()> { check(unsafe { oc_emb_delete(self.h, &doc_id, 1) }) }
    /// search(&VectorSearchParams, &mut HashMap)  (embedding_field.rs:250-278): `output[doc] += score`
    pub fn search(&self, target: &[f32], similarity: f32, limit: usize, filter: Option<(&[u64], u64)>,
                  output: &mut std::collections::HashMap<u64, f32>) -> anyhow::Result<()> {
        let (mut docs, mut scores, mut n) = (vec![0u64; limit], vec![0f32; limit], 0u32);
        let (fb, nb) = filter.map(|(b, n)| (b.as_ptr(), n)).unwrap_or((std::ptr::null(), 0));
        check(unsafe { oc_emb_search(self.h, target.as_ptr(), 1, limit as u32, similarity, fb, nb,
                                     docs.as_mut_ptr(), scores.as_mut_ptr(), &mut n) })?;
        for i in 0..n as usize { *output.entry(docs[i]).or_insert(0.0) += scores[i]; }
        Ok(())
    }
}
impl Drop for EmbeddingField { fn drop(&mut self) { unsafe { oc_emb_destroy(self.h) } } }
