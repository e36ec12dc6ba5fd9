// sort.cuh — sortBy on the device: sort_token_scores_by_field + truncate (read/sort.rs:48-98, 236-257) over the
// orders IndexSortContext::execute yields for number, date and bool fields (read/index/sort.rs:186-264).
//
// The score map's key set arrives as a bitmap over DocumentId (the matched rows of the BM25 tile scorers + the
// vector hits, as for facets).  K6 (sort_select_kernel) finds, per query, the first n_keep = limit + offset keys in
// the field's walk order — value groups in the requested order, ascending DocumentId inside a group — in one of two
// forms chosen per query on the device:
//   walk   — stream the field's precomputed order permutation and test each document's bit; stops after n_keep hits
//            (cheap when the map is dense: a match-all query reads about n_keep entries);
//   gather — visit the set bits of the bitmap, form (rank' << 32 | id) keys and radix-select the n_keep smallest
//            (cheap when the map is sparse: one pass over the bitmap words).
// K7 (sort_score_kernel) then gives each picked document its score-map value with the rounded ops of K4 (fuse.cuh).
#pragma once
#include "fuse.cuh"

namespace oc {

constexpr uint32_t SORT_NONE = 0xffffffffu;        // rank of a document that has no value in the field
constexpr uint32_t SORT_THREADS = 256;
constexpr uint32_t SORT_WALK_PER_THREAD = 4;       // consecutive order entries per thread and step
constexpr uint32_t SORT_GATHER_STEP = SORT_THREADS * 32;           // keys one step of 256 bitmap words can add
constexpr uint32_t SORT_GATHER_CAP = SORT_GATHER_STEP + OC_MAX_TOPK; // buffered keys before a radix select
// Switch rule: walk when walk_cost x (order entries the walk is expected to read) <= (bitmap words + map keys) the
// gather reads.  The walk expects the map keys spread evenly over the DocumentIds.  Measured on the B200 (DESIGN §8).
constexpr float SORT_WALK_COST = 4.0f;
enum { SORT_FORM_AUTO = -1, SORT_FORM_WALK = 0, SORT_FORM_GATHER = 1 };

struct SortSelParams {
    const uint32_t *bits;               // [q][stride_words] score-map keys over DocumentId [0, cap_bits)
    uint64_t stride_words, cap_bits;
    const unsigned long long *count;    // [q] size of the score map (K4)
    const uint32_t *rank;               // [nbits] dense rank of the document's value, SORT_NONE = no value
    uint64_t nbits;
    const uint32_t *order;              // [n_pop] DocumentIds by (rank, id asc), rank ascending or descending
    uint64_t n_pop;
    uint32_t n_ranks;
    int descending;
    uint32_t n_keep;
    int form;                           // SORT_FORM_*
    uint64_t *pick;                     // [q][n_keep] picked DocumentIds in walk order
    uint32_t *n_pick;                   // [q]
    uint8_t *form_out;                  // [q] SORT_FORM_WALK / SORT_FORM_GATHER
};

__device__ __forceinline__ bool sort_in_map(const uint32_t *bq, uint64_t cap_bits, uint64_t d) {
    return d < cap_bits && ((__ldg(bq + (d >> 5)) >> (d & 31)) & 1u);
}

__device__ __forceinline__ bool sort_choose_walk(const SortSelParams &p, uint64_t cnt) {
    if (p.form != SORT_FORM_AUTO) return p.form == SORT_FORM_WALK;
    if (cnt == 0 || p.n_pop == 0) return false;
    const double hits = double(cnt) * double(p.n_pop) / double(p.nbits);   // map keys that have a value
    const double walk = hits >= double(p.n_keep) ? double(p.n_keep) * double(p.nbits) / double(cnt) : double(p.n_pop);
    const double gather = double(p.cap_bits) / 32.0 + double(cnt);
    return double(SORT_WALK_COST) * walk <= gather;
}

// one CTA per query; dynamic shared memory: SORT_GATHER_CAP + next_pow2(n_keep) u64 keys
__global__ void __launch_bounds__(SORT_THREADS) sort_select_kernel(const SortSelParams p) {
    extern __shared__ __align__(16) uint8_t smem[];
    const uint32_t q = blockIdx.x, tid = threadIdx.x, lane = tid & 31;
    const uint32_t *bq = p.bits + size_t(q) * p.stride_words;
    uint64_t *pick = p.pick + size_t(q) * p.n_keep;
    const bool walk = sort_choose_walk(p, p.count[q]);
    if (walk) {
        uint32_t found = 0;
        for (uint64_t base = 0; base < p.n_pop && found < p.n_keep; base += uint64_t(SORT_THREADS) * SORT_WALK_PER_THREAD) {
            uint32_t ids[SORT_WALK_PER_THREAD], m = 0;
#pragma unroll
            for (uint32_t u = 0; u < SORT_WALK_PER_THREAD; u++) {
                const uint64_t i = base + uint64_t(tid) * SORT_WALK_PER_THREAD + u;
                ids[u] = i < p.n_pop ? __ldg(p.order + i) : 0u;
                if (i < p.n_pop && sort_in_map(bq, p.cap_bits, ids[u])) m |= 1u << u;
            }
            uint32_t total;
            uint32_t pos = found + block_exclusive_scan(__popc(m), &total);   // order of the entries is kept
#pragma unroll
            for (uint32_t u = 0; u < SORT_WALK_PER_THREAD; u++)
                if ((m >> u) & 1u) { if (pos < p.n_keep) pick[pos] = ids[u]; pos++; }
            found += total;
        }
        if (tid == 0) { p.n_pick[q] = min(found, p.n_keep); p.form_out[q] = SORT_FORM_WALK; }
        return;
    }
    // gather: key K = ~(rank' << 32 | id) — the LARGEST K is the first document of the walk (rank' = rank, or
    // n_ranks - 1 - rank when descending); K is never 0 (KEY_NONE) since rank' < 0xffffffff
    uint64_t *buf = reinterpret_cast<uint64_t *>(smem);
    const uint32_t kp2 = max(32u, next_pow2(p.n_keep));
    uint64_t *sel = buf + SORT_GATHER_CAP;
    __shared__ uint32_t s_kept;
    __shared__ unsigned long long s_cut;
    if (tid == 0) { s_kept = 0; s_cut = 0ull; }
    __syncthreads();
    auto key_of = [&](uint64_t d) -> uint64_t {
        if (d >= p.nbits) return 0ull;
        const uint32_t r = __ldg(p.rank + d);
        if (r == SORT_NONE) return 0ull;
        const uint32_t rr = p.descending ? p.n_ranks - 1u - r : r;
        return ~((uint64_t(rr) << 32) | d);
    };
    auto flush = [&]() {   // keep the n_keep largest keys, raise the cut-off to the smallest of them
        const uint32_t nv = s_kept;
        __syncthreads();
        const uint32_t got = block_select_largest(buf, nv, p.n_keep, sel);
        for (uint32_t i = tid; i < got; i += blockDim.x) buf[i] = sel[i];
        if (tid == 0) { s_kept = got; if (got == p.n_keep) s_cut = ~0ull; }
        __syncthreads();
        if (got == p.n_keep) {
            unsigned long long mn = ~0ull;
            for (uint32_t i = tid; i < got; i += blockDim.x) mn = min(mn, (unsigned long long)buf[i]);
            atomicMin(&s_cut, mn);
        }
        __syncthreads();
    };
    const uint64_t words = (p.cap_bits + 31) / 32;
    for (uint64_t w0 = 0; w0 < words; w0 += SORT_THREADS) {
        const bool full = s_kept + SORT_GATHER_STEP > SORT_GATHER_CAP;
        __syncthreads();   // every thread has read s_kept before any adds to it
        if (full) flush();
        const unsigned long long cut = s_cut;
        const uint64_t w = w0 + tid;
        const uint32_t v = w < words ? __ldg(bq + w) : 0u;
        uint32_t n = 0;
        for (uint32_t b = v; b; b &= b - 1) n += key_of(w * 32 + (__ffs(b) - 1)) > cut ? 1u : 0u;
        uint32_t incl = n;   // warp-aggregated slot reservation
        for (uint32_t o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
        uint32_t base = 0;
        if (lane == 31 && incl) base = atomicAdd(&s_kept, incl);
        base = __shfl_sync(0xffffffffu, base, 31) + incl - n;
        for (uint32_t b = v; b; b &= b - 1) {
            const uint64_t k = key_of(w * 32 + (__ffs(b) - 1));
            if (k > cut) buf[base++] = k;
        }
        __syncthreads();
    }
    if (s_kept > p.n_keep) flush();
    const uint32_t got = s_kept;
    for (uint32_t i = tid; i < kp2; i += blockDim.x) sel[i] = i < got ? buf[i] : KEY_NONE;
    __syncthreads();
    group_bitonic_desc(sel, kp2, tid, blockDim.x, 0);
    for (uint32_t i = tid; i < got; i += blockDim.x) pick[i] = uint32_t(~sel[i]);
    if (tid == 0) { p.n_pick[q] = got; p.form_out[q] = SORT_FORM_GATHER; }
}

struct SortScoreParams {
    FuseParams fp;                      // mode, limit, offset, vector hits, OMC and the outputs of K4's layout
    uint32_t n_queries;
    const float *gmin, *gmax;           // [q] K4's global extrema (hybrid normalisation)
    const uint64_t *pick;               // [q][n_keep]
    const uint32_t *n_pick;
    const float *p_ft;                  // [q][n_keep] fulltext score of each pick (bm25_point_kernel)
    const uint8_t *p_present;
    const uint32_t *rank;               // [nbits]
    const double *rank_value;           // [n_ranks] the sort value of each rank
    double *out_key;                    // [q][limit]
};

// one thread per (query, output slot): the score-map value of the picked document with K4's ops in K4's order
__global__ void __launch_bounds__(256) sort_score_kernel(const SortScoreParams p) {
    const FuseParams &fp = p.fp;
    const uint32_t gid = blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= p.n_queries * fp.limit) return;
    const uint32_t q = gid / fp.limit, j = gid % fp.limit;
    const uint32_t np = p.n_pick[q];
    const uint32_t n_out = np > fp.offset ? min(fp.limit, np - fp.offset) : 0u;
    const size_t o = size_t(q) * fp.limit + j;
    if (j == 0) fp.out_n[q] = n_out;
    if (j >= n_out) { fp.out_doc[o] = 0; fp.out_score[o] = 0.f; p.out_key[o] = 0.0; return; }
    const uint32_t i = fp.offset + j;
    const size_t pi = size_t(q) * fp.n_keep + i;
    const uint64_t d = p.pick[pi];
    const bool has_ft = fp.mode != OC_MODE_VECTOR, has_v = fp.mode != OC_MODE_FULLTEXT;
    float vs = 0.f;
    bool vhit = false;
    if (has_v) {   // output[doc] += score over the vector hits in order (embedding_field.rs:273-274)
        const uint32_t vc = fp.v_count[q];
        const uint64_t *vdoc = fp.v_doc + size_t(q) * fp.v_stride;
        const float *vscore = fp.v_score + size_t(q) * fp.v_stride;
        for (uint32_t k = 0; k < vc; k++) if (vdoc[k] == d) { vs = __fadd_rn(vs, vscore[k]); vhit = true; }
    }
    float f;
    if (has_ft && has_v) {   // normalize_and_combine (token_score.rs:393-422)
        const float gmin = p.gmin[q], den = __fsub_rn(p.gmax[q], gmin);
        if (vhit) {
            const float vn = __fdiv_rn(__fsub_rn(vs, gmin), den);
            const float fn = p.p_present[pi] ? __fdiv_rn(__fsub_rn(p.p_ft[pi], gmin), den) : 0.0f;
            f = __fadd_rn(fn, vn);
        } else {
            f = __fdiv_rn(__fsub_rn(p.p_ft[pi], gmin), den);
        }
    } else {
        f = has_ft ? p.p_ft[pi] : vs;
    }
    if (fp.n_omc) {
        bool found;
        const float m = omc_lookup(fp, d, &found);
        if (found) f = __fmul_rn(f, m);
    }
    fp.out_doc[o] = d;
    fp.out_score[o] = f;
    p.out_key[o] = p.rank_value[p.rank[d]];
}

}  // namespace oc
