// fuse.cuh — K4: hybrid score fusion + OMC + global top-n + count, one CTA per query.
//
// Replaces normalize_and_combine (read/index/token_score.rs:393-422),
// apply_omc_multipliers (read/search.rs:39-48), `count = map.len()` (search.rs:482),
// sort_token_scores / top_n (read/sort.rs:17-46, 260-279) and skip(offset).take(limit)
// (search.rs:494-498).
//
// Inputs are the small per-(query, tile) products of the BM25 tile kernel (candidates,
// counts, extrema) and the <= limit vector hits of the scan merge.  Every arithmetic
// step uses explicit round-to-nearest ops in the reference's order so results equal the
// CPU restatement bit for bit given equal inputs.
#pragma once
#include "emb_scan.cuh"

namespace oc {

struct FuseParams {
    int mode;                     // OC_MODE_*
    uint32_t n_tiles, n_keep;     // n_keep = limit + offset
    uint32_t limit, offset;
    uint32_t capb;                // smem key buffer, pow2 >= 2*n_keep
    // fulltext side (NULL in vector mode)
    const uint64_t *cand_key;     // [q][tile][n_keep] (rank proxy | row)
    const float *cand_ft;         // raw bm25 score
    const uint32_t *cand_cnt;     // [q][tile]
    const uint32_t *tile_count;
    const float *tile_max, *tile_min;
    const uint64_t *str_row_doc_ids;  // NULL => doc == row
    // vector side (NULL in fulltext mode), stride = v_stride (= limit)
    const uint64_t *v_doc;
    const float *v_score;
    const uint32_t *v_count;
    const uint32_t *v_row;        // string row of each hit (hybrid) or NULL
    const float *v_ft;
    const uint8_t *v_present;
    uint32_t v_stride;
    // OMC by doc id, ascending
    const uint64_t *omc_doc;
    const float *omc_mult;
    uint32_t n_omc;
    // outputs
    uint64_t *out_doc;            // [q][limit]
    float *out_score;
    uint32_t *out_n;
    unsigned long long *out_count;
    float *out_min;               // actual global min (rank-proxy validation), may be NULL
    float *out_max;               // actual global max (sortBy re-scores picked documents with it), may be NULL
};

__device__ __forceinline__ float omc_lookup(const FuseParams &p, uint64_t doc, bool *found) {
    uint32_t lo = 0, hi = p.n_omc;
    while (lo < hi) {
        const uint32_t m = (lo + hi) >> 1;
        if (p.omc_doc[m] < doc) lo = m + 1; else hi = m;
    }
    *found = lo < p.n_omc && p.omc_doc[lo] == doc;
    return *found ? p.omc_mult[lo] : 1.0f;
}

constexpr uint32_t FUSE_MAX_V = OC_MAX_TOPK;

__global__ void __launch_bounds__(256) fuse_topk_kernel(const FuseParams p) {
    extern __shared__ __align__(16) uint8_t smem[];
    uint64_t *buf = reinterpret_cast<uint64_t *>(smem);               // [capb]
    uint64_t *sel = buf + p.capb;                                     // [next_pow2(n_keep)] selection scratch
    float *vsum = reinterpret_cast<float *>(sel + max(32u, next_pow2(p.n_keep)));   // [v_stride] merged vector score
    uint32_t *vfirst = reinterpret_cast<uint32_t *>(vsum + p.v_stride); // [v_stride] 1 = unique head
    __shared__ unsigned int s_maxo, s_mino;
    __shared__ unsigned long long s_count;
    const uint32_t q = blockIdx.x, tid = threadIdx.x;
    const bool has_ft = p.mode != OC_MODE_VECTOR;
    const bool has_v = p.mode != OC_MODE_FULLTEXT;
    const uint32_t vc = has_v ? p.v_count[q] : 0;
    const uint64_t *vdoc = has_v ? p.v_doc + size_t(q) * p.v_stride : nullptr;
    const float *vscore = has_v ? p.v_score + size_t(q) * p.v_stride : nullptr;

    if (tid == 0) { s_maxo = f32_ordered(0.f); s_mino = f32_ordered(0.f); s_count = 0; }
    // ---- merge duplicate docs among the vector hits: output[doc] += score (embedding_field.rs:273-274)
    for (uint32_t j = tid; j < vc; j += blockDim.x) {
        bool head = true;
        for (uint32_t i = 0; i < j; i++) if (vdoc[i] == vdoc[j]) { head = false; break; }
        float s = 0.f;
        if (head) for (uint32_t i = j; i < vc; i++) if (vdoc[i] == vdoc[j]) s = __fadd_rn(s, vscore[i]);
        vsum[j] = s;
        vfirst[j] = head ? 1u : 0u;
    }
    __syncthreads();

    // ---- count and extrema
    unsigned long long cnt = 0;
    float lmax = 0.f, lmin = 0.f;
    if (has_ft)
        for (uint32_t t = tid; t < p.n_tiles; t += blockDim.x) {
            const size_t s = size_t(q) * p.n_tiles + t;
            cnt += p.tile_count[s];
            lmax = fmaxf(lmax, p.tile_max[s]);
            lmin = fminf(lmin, p.tile_min[s]);
        }
    for (uint32_t j = tid; j < vc; j += blockDim.x)
        if (vfirst[j]) {
            lmax = fmaxf(lmax, vsum[j]);
            lmin = fminf(lmin, vsum[j]);
            const bool in_ft = has_ft && p.v_present[size_t(q) * p.v_stride + j];
            if (!in_ft) cnt++;
        }
    for (int o = 16; o > 0; o >>= 1) {
        lmax = fmaxf(lmax, __shfl_xor_sync(0xffffffffu, lmax, o));
        lmin = fminf(lmin, __shfl_xor_sync(0xffffffffu, lmin, o));
        cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    }
    if ((tid & 31) == 0) {
        atomicMax(&s_maxo, f32_ordered(lmax));
        atomicMin(&s_mino, f32_ordered(lmin));
        if (cnt) atomicAdd(&s_count, cnt);
    }
    __syncthreads();
    const float gmax = f32_unordered(s_maxo), gmin = f32_unordered(s_mino);
    const float den = __fsub_rn(gmax, gmin);   // (max - min), token_score.rs:406,412
    const bool hybrid = has_ft && has_v;

    // ---- candidate stream: tile candidates (minus vector-hit rows), then the vector hits
    const uint64_t n_ft_slots = has_ft ? uint64_t(p.n_tiles) * p.n_keep : 0;
    const uint64_t total = n_ft_slots + vc;
    auto load = [&](uint64_t i) -> uint64_t {
        if (i < n_ft_slots) {
            const uint32_t t = uint32_t(i / p.n_keep), k = uint32_t(i % p.n_keep);
            const size_t s = size_t(q) * p.n_tiles + t;
            if (k >= p.cand_cnt[s]) return KEY_NONE;
            const uint32_t row = key_idx(p.cand_key[s * p.n_keep + k]);
            if (hybrid)
                for (uint32_t j = 0; j < vc; j++)
                    if (p.v_row[size_t(q) * p.v_stride + j] == row) return KEY_NONE;  // scored below
            float f = p.cand_ft[s * p.n_keep + k];
            if (hybrid) f = __fdiv_rn(__fsub_rn(f, gmin), den);       // (v - min) / (max - min)
            if (p.n_omc) {
                bool found;
                const uint64_t doc = p.str_row_doc_ids ? p.str_row_doc_ids[row] : uint64_t(row);
                const float m = omc_lookup(p, doc, &found);
                if (found) f = __fmul_rn(f, m);
            }
            return f == f ? make_key(f, row) : KEY_NONE;              // NaN dropped (sort.rs:264-267)
        }
        const uint32_t j = uint32_t(i - n_ft_slots);
        if (!vfirst[j]) return KEY_NONE;
        float f;
        uint32_t idx;
        if (hybrid) {
            const size_t vs = size_t(q) * p.v_stride + j;
            const float vn = __fdiv_rn(__fsub_rn(vsum[j], gmin), den);
            const float fn = p.v_present[vs] ? __fdiv_rn(__fsub_rn(p.v_ft[vs], gmin), den) : 0.0f;
            f = __fadd_rn(fn, vn);                                    // entry(k).or_default() += v
            idx = p.v_row[vs] != 0xffffffffu ? p.v_row[vs] : (0xfffffffeu - j);
        } else {
            f = vsum[j];
            idx = j;
        }
        if (p.n_omc) {
            bool found;
            const float m = omc_lookup(p, vdoc[j], &found);
            if (found) f = __fmul_rn(f, m);
        }
        return f == f ? make_key(f, idx) : KEY_NONE;
    };
    // Most tiles emit no candidate once the query's threshold has warmed up: compact the valid
    // slots first (per-thread counts + block exclusive scan) and sort only those; fall back to
    // the streaming top-n when they do not fit the key buffer.
    uint32_t got;
    {
        uint32_t mine = 0;
        if (has_ft)
            for (uint32_t t = tid; t < p.n_tiles; t += blockDim.x) mine += min(p.cand_cnt[size_t(q) * p.n_tiles + t], p.n_keep);
        uint32_t n_valid_ft;
        const uint32_t my_pos = block_exclusive_scan(mine, &n_valid_ft);
        const uint32_t n_all = n_valid_ft + vc;
        if (n_all <= p.capb) {
            uint32_t pos = my_pos;
            if (has_ft)
                for (uint32_t t = tid; t < p.n_tiles; t += blockDim.x) {
                    const uint32_t c = min(p.cand_cnt[size_t(q) * p.n_tiles + t], p.n_keep);
                    for (uint32_t k = 0; k < c; k++) buf[pos++] = load(uint64_t(t) * p.n_keep + k);
                }
            for (uint32_t j = tid; j < vc; j += blockDim.x) buf[n_valid_ft + j] = load(n_ft_slots + j);
            const uint32_t np2 = max(32u, next_pow2(n_all));
            const uint32_t kp2 = max(32u, next_pow2(p.n_keep));
            if (np2 > 2 * kp2) {
                // many more candidates than needed: radix-select the n_keep best, sort only those
                for (uint32_t i = tid; i < kp2; i += blockDim.x) sel[i] = KEY_NONE;
                __syncthreads();
                block_select_largest(buf, n_all, p.n_keep, sel);
                group_bitonic_desc(sel, kp2, tid, blockDim.x, 0);
                for (uint32_t i = tid; i < kp2; i += blockDim.x) buf[i] = sel[i];
                __syncthreads();
            } else {
                for (uint32_t i = n_all + tid; i < np2; i += blockDim.x) buf[i] = KEY_NONE;
                group_bitonic_desc(buf, np2, tid, blockDim.x, 0);
            }
            uint32_t real = min(n_all, p.n_keep);
            __shared__ uint32_t s_real2;
            if (tid == 0) { while (real > 0 && buf[real - 1] == KEY_NONE) real--; s_real2 = real; }
            __syncthreads();
            got = s_real2;
        } else {
            got = block_topn_stream(buf, p.capb, p.n_keep, total, load);
        }
    }

    // ---- skip(offset).take(limit)
    const uint32_t n_out = got > p.offset ? min(p.limit, got - p.offset) : 0;
    for (uint32_t i = tid; i < p.limit; i += blockDim.x) {
        uint64_t doc = 0; float sc = 0.f;
        if (i < n_out) {
            const uint64_t k = buf[p.offset + i];
            const uint32_t idx = key_idx(k);
            sc = key_score(k);
            if (p.mode == OC_MODE_VECTOR) doc = vdoc[idx];
            else if (hybrid && idx >= 0xfffffffeu - FUSE_MAX_V) doc = vdoc[0xfffffffeu - idx];
            else doc = p.str_row_doc_ids ? p.str_row_doc_ids[idx] : uint64_t(idx);
        }
        p.out_doc[size_t(q) * p.limit + i] = doc;
        p.out_score[size_t(q) * p.limit + i] = sc;
    }
    if (tid == 0) {
        p.out_n[q] = n_out;
        p.out_count[q] = s_count;
        if (p.out_min) p.out_min[q] = gmin;
        if (p.out_max) p.out_max[q] = gmax;
    }
}

// map vector hits (doc ids) to string-store rows by binary search over ascending row_doc_ids
__global__ void map_docs_to_rows_kernel(const uint64_t *docs, const uint32_t *counts, uint32_t stride,
                                        uint32_t n_queries, const uint64_t *row_doc_ids, uint64_t n_rows,
                                        uint32_t *out_rows) {
    const uint32_t gid = blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= n_queries * stride) return;
    const uint32_t q = gid / stride, j = gid % stride;
    uint32_t r = 0xffffffffu;
    if (j < counts[q]) {
        const uint64_t d = docs[gid];
        if (!row_doc_ids) {
            if (d < n_rows) r = uint32_t(d);
        } else {
            uint64_t lo = 0, hi = n_rows;
            while (lo < hi) { const uint64_t m = (lo + hi) >> 1; if (row_doc_ids[m] < d) lo = m + 1; else hi = m; }
            if (lo < n_rows && row_doc_ids[lo] == d) r = uint32_t(lo);
        }
    }
    out_rows[gid] = r;
}

// DocumentId bitmap -> row bitmap (alive AND filter); one thread per 32 rows.
__global__ void rows_ok_kernel(const uint64_t *row_doc_ids, uint64_t n_rows, const uint32_t *alive_bits,
                               const uint64_t *filter_bits, uint64_t filter_nbits, uint32_t *out_bits,
                               uint64_t n_words) {
    const uint64_t w = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (w >= n_words) return;
    uint32_t bits = 0;
    for (uint32_t b = 0; b < 32; b++) {
        const uint64_t r = w * 32 + b;
        if (r >= n_rows) break;
        bool ok = alive_bits ? ((alive_bits[w] >> b) & 1u) : true;
        if (ok && filter_bits) {
            const uint64_t d = row_doc_ids ? row_doc_ids[r] : r;
            ok = d < filter_nbits && ((filter_bits[d >> 6] >> (d & 63)) & 1ull);
        }
        bits |= (ok ? 1u : 0u) << b;
    }
    out_bits[w] = bits;
}

}  // namespace oc
