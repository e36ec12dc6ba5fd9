// capi.cu — host side of liboramacore_b200.so: the C ABI declared in
// include/oramacore_b200.h over the sm_100a kernels (emb_scan.cuh, bm25.cuh, fuse.cuh).
// No torch, no CPU fallback: every entry point needs a live CUDA device.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <utility>
#include <string>
#include <unordered_map>
#include <vector>

#include "bm25.cuh"
#include "comm.h"
#include "dict.h"
#include "stem_en.h"
#include "emb_gemm.cuh"
#include "emb_scan.cuh"
#include "fuse.cuh"
#include "sort.cuh"
#include "oramacore_b200.h"

using namespace oc;

// ------------------------------------------------------------------------------------ errors
static thread_local char g_err[512] = "";
static int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
#define CU(x)                                                                                   \
    do {                                                                                        \
        cudaError_t _e = (x);                                                                   \
        if (_e != cudaSuccess)                                                                  \
            return fail(_e == cudaErrorMemoryAllocation ? OC_ERR_OOM : OC_ERR_CUDA, "%s: %s (%s:%d)", #x, \
                        cudaGetErrorString(_e), __FILE__, __LINE__);                            \
    } while (0)
#define OCTRY(x)                \
    do {                        \
        int _r = (x);           \
        if (_r != OC_OK) return _r; \
    } while (0)

extern "C" const char *oc_last_error(void) { return g_err; }
extern "C" int oc_version(void) { return 100; }
extern "C" void oc_abi_sizes(size_t out[4]) {
    out[0] = sizeof(oc_search_params); out[1] = sizeof(oc_timing); out[2] = sizeof(oc_emb_info_t); out[3] = sizeof(oc_str_info_t);
}

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is per (device, function): remember what was configured
// per device so several contexts on different GPUs in one process each get their kernels configured
static bool smem_cfg_needed(int device, const void *fn, size_t smem) {
    static std::mutex mu;
    static std::map<std::pair<int, const void *>, size_t> done;
    std::lock_guard<std::mutex> g(mu);
    size_t &v = done[std::make_pair(device, fn)];
    if (smem <= v) return false;
    v = smem;
    return true;
}

// ------------------------------------------------------------------------------------ buffers
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return OC_OK;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 4 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) { e = cudaMalloc(&p, bytes); want = bytes; }
        if (e != cudaSuccess) return fail(OC_ERR_OOM, "cudaMalloc(%zu): %s", bytes, cudaGetErrorString(e));
        cap = want;
        return OC_OK;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <typename T> T *as() { return reinterpret_cast<T *>(p); }
};
struct HostBuf {  // pinned staging
    void *p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return OC_OK;
        if (p) cudaFreeHost(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 4 + 256;
        cudaError_t e = cudaMallocHost(&p, want);
        if (e != cudaSuccess) return fail(OC_ERR_OOM, "cudaMallocHost(%zu): %s", want, cudaGetErrorString(e));
        cap = want;
        return OC_OK;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
    template <typename T> T *as() { return reinterpret_cast<T *>(p); }
};

// lays several host arrays out in one pinned blob -> one H2D copy (sources are copied once,
// straight into the pinned staging buffer)
struct Packer {
    struct Seg { const void *src; size_t off, bytes; bool direct; };
    std::vector<Seg> segs;
    size_t total = 0;
    // direct = the source already lives in pinned host memory (oc_pinned_alloc / cudaHostRegister):
    // it is DMA'd straight from the caller's buffer instead of being staged
    size_t add(const void *src, size_t bytes, bool direct = false) {
        const size_t off = (total + 255) & ~size_t(255);
        segs.push_back({src, off, bytes, direct});
        total = off + bytes;
        return off;
    }
    void fill(void *dst) const {
        for (const Seg &g : segs) if (g.bytes && g.src && !g.direct) memcpy(static_cast<uint8_t *>(dst) + g.off, g.src, g.bytes);
    }
};
static bool is_pinned_host(const void *p) {
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}

enum { EV_START, EV_H2D, EV_DEV, EV_D2H, EV_SCAN0, EV_SCAN1, EV_BM0, EV_BM1, EV_FUSE0, EV_FUSE1, EV_COMM0, EV_COMM1, EV_SWEEP0, EV_SWEEP1, EV_RR0, EV_RR1, EV_SORT0, EV_SORT1, EV_N };

constexpr size_t P2P_WIN_BYTES = size_t(1) << 20;   // per (parity, source rank): a batch's records must fit (256 queries x 520 B = 133 KB)
constexpr uint32_t P2P_MAX_Q = 4096;
constexpr size_t P2P_FLAG_BYTES = size_t(2) * P2P_MAX_Q * 4;
constexpr uint32_t P2P_MAX_WORLD = 16;

struct oc_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t side = nullptr;      // descriptor upload + BM25 plan/precompute while the main stream sweeps the matrix
    cudaEvent_t ev_side = nullptr;
    bool sweep_timed = false;         // EV_SWEEP0/1 recorded in this call (tensor-core path)
    uint32_t cvt_stages_default = 5;  // run_vector_stage: ring depth of the converting sweep when the caller has no preference
    bool rerun_timed = false;         // EV_RR0/1 recorded: flagged queries were re-run through the exact sweep
    bool side_dirty = false;          // work was queued on the side stream and not yet joined (an error path returned early)
    cudaDeviceProp prop{};
    std::mutex mu;
    cudaEvent_t ev[EV_N]{};
    oc_timing timing{};
    uint64_t launches = 0;
    uint32_t call_launches = 0, call_scan_launches = 0;
    // workspaces
    DevBuf in_blob, in_blob0, q_pad, q_inv, eff_norm, filter_dev, scan_cand, v_doc, v_score, v_row, v_cnt, v_srow, v_ft, v_present, v_raw;
    DevBuf seg, df_dev, row_ok, tau, cand_key, cand_ft, cand_cnt, tile_cnt, tile_max, tile_min, min_hint;
    DevBuf out_blob, shard_send, shard_recv, work_ctr, flat_desc, mbits, dbits, facet_req, facet_out;
    DevBuf sort_pick, sort_npick, sort_form, sort_rows, sort_ft, sort_present, sort_max, sort_keys;
    std::vector<uint8_t> sort_forms;  // SORT_FORM_* of each query of the last oc_search_sorted
    bool gemm_pending = false; const float *gemm_inv_norm = nullptr;
    DevBuf q_bf16, q_rho, pre_post, dense_buf, g_thr, g_eps, g_ovf, g_ovfcnt, g_resc, g_cand, g_cnt, g_flag, g_max, r_qpad, r_qinv, r_map, r_doc, r_score, r_row, r_cnt, r_raw;

    HostBuf h_in, h_out, h_in0;   // h_in0 / in_blob0: query vectors + filter, uploaded before the descriptors
    OcComm comm;
    // direct NVLink exchange of the shard records (oc_comm_p2p_*): one IPC-shared window per rank —
    // [2 parities][P2P_MAX_Q] arrival counters, then [2 parities][world source ranks][P2P_WIN_BYTES] records
    struct P2P {
        bool ready = false;
        uint8_t *local = nullptr;
        uint8_t *peer[16] = {};      // peer[rank] == local
        uint64_t seq = 0;            // exchanges done (all ranks run the same batches): parity = seq & 1
    } p2p;
};

static inline void launched(oc_ctx *c, bool scan = false) {
    c->launches++; c->call_launches++;
    if (scan) c->call_scan_launches++;
}

extern "C" int oc_init(int device_id, oc_ctx **out) {
    if (!out) return fail(OC_ERR_INVALID, "oc_init: out is NULL");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(OC_ERR_CUDA, "no CUDA device: %s (this library has no CPU fallback)", cudaGetErrorString(e));
    if (device_id < 0 || device_id >= n) return fail(OC_ERR_INVALID, "device %d out of range (%d devices)", device_id, n);
    CU(cudaSetDevice(device_id));
    oc_ctx *c = new oc_ctx();
    c->device = device_id;
    CU(cudaGetDeviceProperties(&c->prop, device_id));
    if (c->prop.major < 10) {
        int mj = c->prop.major, mn = c->prop.minor;
        delete c;
        return fail(OC_ERR_CUDA, "device sm_%d%d is not sm_100-class; kernels are built for sm_100a only", mj, mn);
    }
    CU(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&c->side, cudaStreamNonBlocking));
    CU(cudaEventCreateWithFlags(&c->ev_side, cudaEventDisableTiming));
    for (int i = 0; i < EV_N; i++) CU(cudaEventCreate(&c->ev[i]));
    *out = c;
    return OC_OK;
}

extern "C" void oc_shutdown(oc_ctx *c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    for (int r = 0; r < 16; r++) if (c->p2p.ready && c->p2p.peer[r] && c->p2p.peer[r] != c->p2p.local) cudaIpcCloseMemHandle(c->p2p.peer[r]);
    if (c->p2p.local) cudaFree(c->p2p.local);
    c->comm.destroy();
    DevBuf *bufs[] = {&c->in_blob, &c->q_pad, &c->q_inv, &c->eff_norm, &c->filter_dev, &c->scan_cand, &c->v_doc,
                      &c->v_score, &c->v_row, &c->v_cnt, &c->v_srow, &c->v_ft, &c->v_present, &c->v_raw, &c->seg, &c->df_dev,
                      &c->row_ok, &c->tau, &c->cand_key, &c->cand_ft, &c->cand_cnt, &c->tile_cnt, &c->tile_max,
                      &c->tile_min, &c->min_hint, &c->out_blob, &c->shard_send, &c->shard_recv, &c->work_ctr, &c->flat_desc, &c->mbits, &c->dbits, &c->facet_req, &c->facet_out, &c->q_bf16, &c->q_rho, &c->pre_post, &c->dense_buf, &c->g_thr, &c->g_eps, &c->g_ovf, &c->g_ovfcnt, &c->g_resc, &c->g_cand, &c->g_cnt, &c->g_max,
                      &c->g_flag, &c->r_qpad, &c->r_qinv, &c->r_map, &c->r_doc, &c->r_score, &c->r_row, &c->r_cnt, &c->r_raw,
                      &c->sort_pick, &c->sort_npick, &c->sort_form, &c->sort_rows, &c->sort_ft, &c->sort_present, &c->sort_max, &c->sort_keys};
    for (DevBuf *b : bufs) b->release();
    c->h_in.release(); c->h_out.release();
    for (int i = 0; i < EV_N; i++) if (c->ev[i]) cudaEventDestroy(c->ev[i]);
    cudaStreamDestroy(c->stream);
    if (c->side) cudaStreamDestroy(c->side);
    if (c->ev_side) cudaEventDestroy(c->ev_side);
    delete c;
}

extern "C" int oc_device_info(oc_ctx *c, int *sm_count, size_t *hbm_bytes, char *name, size_t name_cap) {
    if (!c) return fail(OC_ERR_INVALID, "ctx is NULL");
    if (sm_count) *sm_count = c->prop.multiProcessorCount;
    if (hbm_bytes) *hbm_bytes = c->prop.totalGlobalMem;
    if (name && name_cap) { strncpy(name, c->prop.name, name_cap - 1); name[name_cap - 1] = 0; }
    return OC_OK;
}

extern "C" int oc_pinned_alloc(size_t bytes, void **out) {
    if (!out) return fail(OC_ERR_INVALID, "out is NULL");
    CU(cudaMallocHost(out, bytes ? bytes : 1));
    return OC_OK;
}
extern "C" void oc_pinned_free(void *p) { if (p) cudaFreeHost(p); }

extern "C" int oc_last_timing(oc_ctx *c, oc_timing *out) {
    if (!c || !out) return fail(OC_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> g(c->mu);
    *out = c->timing;
    return OC_OK;
}
extern "C" uint64_t oc_launch_count(oc_ctx *c) { return c ? c->launches : 0; }

extern "C" int oc_comm_unique_id(uint8_t out_id[OC_COMM_ID_BYTES]) {
    std::string err;
    if (!OcComm::unique_id(out_id, &err)) return fail(OC_ERR_COMM, "%s", err.c_str());
    return OC_OK;
}
extern "C" int oc_comm_init(oc_ctx *c, int world, int rank, const uint8_t id[OC_COMM_ID_BYTES]) {
    if (!c || world < 1 || rank < 0 || rank >= world) return fail(OC_ERR_INVALID, "bad comm arguments");
    std::lock_guard<std::mutex> g(c->mu);
    CU(cudaSetDevice(c->device));
    std::string err;
    if (!c->comm.init(world, rank, id, &err)) return fail(OC_ERR_COMM, "%s", err.c_str());
    return OC_OK;
}

// Direct NVLink exchange: rank r exports the IPC handle of its window, the host runtime all-gathers the blobs (like
// the NCCL unique id) and every rank maps all peers' windows.  Afterwards the sharded oc_search stores each query's
// shard record straight into every rank's window from the pack kernel and the merge kernel waits on arrival
// counters — no library collective on the data path (ncclAllGather stays the fallback for batches larger than a window).
extern "C" int oc_comm_p2p_export(oc_ctx *c, uint8_t out[OC_P2P_HANDLE_BYTES]) {
    if (!c || !out) return fail(OC_ERR_INVALID, "NULL argument");
    if (c->comm.world < 2 || c->comm.world > (int)P2P_MAX_WORLD) return fail(OC_ERR_INVALID, "oc_comm_init first (2..%u ranks)", P2P_MAX_WORLD);
    std::lock_guard<std::mutex> g(c->mu);
    CU(cudaSetDevice(c->device));
    if (!c->p2p.local) {
        const size_t bytes = P2P_FLAG_BYTES + size_t(2) * c->comm.world * P2P_WIN_BYTES;
        CU(cudaMalloc(&c->p2p.local, bytes));
        CU(cudaMemset(c->p2p.local, 0, bytes));
    }
    cudaIpcMemHandle_t h;
    CU(cudaIpcGetMemHandle(&h, c->p2p.local));
    static_assert(sizeof(h) <= OC_P2P_HANDLE_BYTES, "handle blob");
    memset(out, 0, OC_P2P_HANDLE_BYTES);
    memcpy(out, &h, sizeof(h));
    return OC_OK;
}
extern "C" int oc_comm_p2p_import(oc_ctx *c, const uint8_t *handles) {
    if (!c || !handles) return fail(OC_ERR_INVALID, "NULL argument");
    if (!c->p2p.local) return fail(OC_ERR_INVALID, "oc_comm_p2p_export first");
    std::lock_guard<std::mutex> g(c->mu);
    CU(cudaSetDevice(c->device));
    for (int r = 0; r < c->comm.world; r++) {
        if (r == c->comm.rank) { c->p2p.peer[r] = c->p2p.local; continue; }
        cudaIpcMemHandle_t h;
        memcpy(&h, handles + size_t(r) * OC_P2P_HANDLE_BYTES, sizeof(h));
        void *ptr = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) return fail(OC_ERR_COMM, "cudaIpcOpenMemHandle(rank %d): %s", r, cudaGetErrorString(e));
        c->p2p.peer[r] = static_cast<uint8_t *>(ptr);
    }
    c->p2p.seq = 0;
    c->p2p.ready = true;
    return OC_OK;
}

// ------------------------------------------------------------------------------------ embedding store
struct oc_emb {
    oc_ctx *ctx;
    uint32_t dim, stride;
    int dtype, e5;
    void *rows = nullptr;        // [cap][stride] fp32 or bf16
    uint32_t esz = 4;            // element bytes
    float *inv_norm = nullptr;   // [cap] (NaN = tombstone)
    uint64_t *row_doc = nullptr; // [cap]
    float *rho_x = nullptr;      // device scalar: max over rows of |x - bf16(x)| / |x| (fp32 stores; the sweep's error bound)
    uint64_t n_rows = 0, cap = 0, n_live = 0;
    std::unordered_multimap<uint64_t, uint64_t> doc_rows;  // doc -> rows (for delete)
};

extern "C" int oc_emb_create(oc_ctx *c, uint32_t dim, int dtype, int rescale_e5, oc_emb **out) {
    if (!c || !out) return fail(OC_ERR_INVALID, "NULL argument");
    if (dim == 0 || dim > 1024) return fail(OC_ERR_UNSUPPORTED, "dim %u unsupported (1..1024)", dim);
    if (dtype != OC_DTYPE_F32 && dtype != OC_DTYPE_BF16) return fail(OC_ERR_UNSUPPORTED, "dtype %d unknown", dtype);
    oc_emb *e = new oc_emb();
    e->ctx = c; e->dim = dim; e->dtype = dtype; e->e5 = rescale_e5 ? 1 : 0;
    e->esz = dtype == OC_DTYPE_BF16 ? 2 : 4;
    e->stride = ((dim + 127) / 128) * 128;
    if (e->stride / 128 == 5 || e->stride / 128 == 7) e->stride += 128;  // instantiated widths: 1,2,3,4,6,8
    {
        std::lock_guard<std::mutex> g(c->mu);
        if (cudaSetDevice(c->device) != cudaSuccess || cudaMalloc(&e->rho_x, 4) != cudaSuccess || cudaMemset(e->rho_x, 0, 4) != cudaSuccess) {
            delete e;
            return fail(OC_ERR_CUDA, "oc_emb_create: device allocation failed");
        }
    }
    *out = e;
    return OC_OK;
}

extern "C" void oc_emb_destroy(oc_emb *e) {
    if (!e) return;
    cudaSetDevice(e->ctx->device);
    cudaStreamSynchronize(e->ctx->stream);
    cudaFree(e->rows); cudaFree(e->inv_norm); cudaFree(e->row_doc); cudaFree(e->rho_x);
    delete e;
}

static int emb_grow(oc_emb *e, uint64_t want_rows) {
    if (want_rows <= e->cap) return OC_OK;
    oc_ctx *c = e->ctx;
    uint64_t ncap = std::max<uint64_t>(want_rows, e->cap + e->cap / 2);
    ncap = (ncap + 63) / 64 * 64;
    void *nr = nullptr; float *nn = nullptr; uint64_t *nd = nullptr;
    CU(cudaMalloc(&nr, ncap * e->stride * e->esz));
    CU(cudaMalloc(&nn, (ncap + 64) * sizeof(float)));
    CU(cudaMalloc(&nd, ncap * sizeof(uint64_t)));
    if (e->n_rows) {
        CU(cudaMemcpyAsync(nr, e->rows, e->n_rows * e->stride * e->esz, cudaMemcpyDeviceToDevice, c->stream));
        CU(cudaMemcpyAsync(nn, e->inv_norm, e->n_rows * sizeof(float), cudaMemcpyDeviceToDevice, c->stream));
        CU(cudaMemcpyAsync(nd, e->row_doc, e->n_rows * sizeof(uint64_t), cudaMemcpyDeviceToDevice, c->stream));
    }
    CU(cudaStreamSynchronize(c->stream));
    cudaFree(e->rows); cudaFree(e->inv_norm); cudaFree(e->row_doc);
    e->rows = nr; e->inv_norm = nn; e->row_doc = nd; e->cap = ncap;
    return OC_OK;
}

extern "C" int oc_emb_reserve(oc_emb *e, uint64_t n_rows) {
    if (!e) return fail(OC_ERR_INVALID, "emb is NULL");
    std::lock_guard<std::mutex> g(e->ctx->mu);
    CU(cudaSetDevice(e->ctx->device));
    return emb_grow(e, n_rows);
}

extern "C" int oc_emb_insert(oc_emb *e, const uint64_t *doc_ids, const void *rows, uint64_t n) {
    if (!e || (!doc_ids && n) || (!rows && n)) return fail(OC_ERR_INVALID, "NULL argument");
    if (n == 0) return OC_OK;
    oc_ctx *c = e->ctx;
    std::lock_guard<std::mutex> g(c->mu);
    CU(cudaSetDevice(c->device));
    if (e->n_rows + n > 0xfffffff0ull) return fail(OC_ERR_UNSUPPORTED, "more than 2^32 rows per store");
    OCTRY(emb_grow(e, e->n_rows + n));
    uint8_t *dst = static_cast<uint8_t *>(e->rows) + e->n_rows * e->stride * e->esz;
    if (e->stride != e->dim) CU(cudaMemsetAsync(dst, 0, n * e->stride * e->esz, c->stream));
    CU(cudaMemcpy2DAsync(dst, size_t(e->stride) * e->esz, rows, size_t(e->dim) * e->esz, size_t(e->dim) * e->esz, n,
                         cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(e->row_doc + e->n_rows, doc_ids, n * sizeof(uint64_t), cudaMemcpyHostToDevice, c->stream));
    const uint64_t warps_per_block = 8;
    const uint64_t blocks = (n + warps_per_block - 1) / warps_per_block;
    if (e->esz == 2) emb_inv_norm_kernel<bf16_t><<<(unsigned)blocks, 256, 0, c->stream>>>(e->rows, e->stride, e->n_rows, e->n_rows + n, e->inv_norm, nullptr);
    else emb_inv_norm_kernel<float><<<(unsigned)blocks, 256, 0, c->stream>>>(e->rows, e->stride, e->n_rows, e->n_rows + n, e->inv_norm,
                                                                             reinterpret_cast<unsigned int *>(e->rho_x));
    launched(c);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(c->stream));
    for (uint64_t i = 0; i < n; i++) e->doc_rows.emplace(doc_ids[i], e->n_rows + i);
    e->n_rows += n; e->n_live += n;
    return OC_OK;
}

__global__ void tombstone_rows_kernel(float *inv_norm, const uint64_t *rows, uint64_t n) {
    const uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n) inv_norm[rows[i]] = __int_as_float(0x7fc00000);
}

extern "C" int oc_emb_delete(oc_emb *e, const uint64_t *doc_ids, uint64_t n) {
    if (!e || (!doc_ids && n)) return fail(OC_ERR_INVALID, "NULL argument");
    oc_ctx *c = e->ctx;
    std::lock_guard<std::mutex> g(c->mu);
    CU(cudaSetDevice(c->device));
    std::vector<uint64_t> rows;
    for (uint64_t i = 0; i < n; i++) {
        auto range = e->doc_rows.equal_range(doc_ids[i]);
        for (auto it = range.first; it != range.second; ++it) rows.push_back(it->second);
        e->doc_rows.erase(range.first, range.second);
    }
    if (rows.empty()) return OC_OK;
    OCTRY(c->in_blob.ensure(rows.size() * 8));
    CU(cudaMemcpyAsync(c->in_blob.p, rows.data(), rows.size() * 8, cudaMemcpyHostToDevice, c->stream));
    tombstone_rows_kernel<<<(unsigned)((rows.size() + 255) / 256), 256, 0, c->stream>>>(e->inv_norm, c->in_blob.as<uint64_t>(), rows.size());
    launched(c);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(c->stream));
    e->n_live -= rows.size();
    return OC_OK;
}

extern "C" int oc_emb_info(oc_emb *e, oc_emb_info_t *out) {
    if (!e || !out) return fail(OC_ERR_INVALID, "NULL argument");
    out->num_embeddings = e->n_live; out->num_rows = e->n_rows; out->dimensions = e->dim; out->dtype = e->dtype;
    out->device_bytes = e->cap * (uint64_t(e->stride) * e->esz + 4 + 8);
    return OC_OK;
}

// ---- scan launch plumbing
template <int NCH, int QB, typename T>
static int launch_scan_t(oc_ctx *c, const ScanParams &sp, uint32_t grid, size_t smem) {
    if (smem_cfg_needed(c->device, (const void *)emb_scan_kernel<NCH, QB, T>, smem))
        CU(cudaFuncSetAttribute(emb_scan_kernel<NCH, QB, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    emb_scan_kernel<NCH, QB, T><<<grid, SCAN_THREADS, smem, c->stream>>>(sp);
    launched(c, true);
    CU(cudaGetLastError());
    return OC_OK;
}
template <int QB, typename T>
static int launch_scan_q(oc_ctx *c, const ScanParams &sp, uint32_t grid, size_t smem) {
    switch (sp.stride / 128) {
        case 1: return launch_scan_t<1, QB, T>(c, sp, grid, smem);
        case 2: return launch_scan_t<2, QB, T>(c, sp, grid, smem);
        case 3: return launch_scan_t<3, QB, T>(c, sp, grid, smem);
        case 4: return launch_scan_t<4, QB, T>(c, sp, grid, smem);
        case 6: return launch_scan_t<6, QB, T>(c, sp, grid, smem);
        case 8: return launch_scan_t<8, QB, T>(c, sp, grid, smem);
    }
    return fail(OC_ERR_UNSUPPORTED, "stride %u not instantiated", sp.stride);
}
template <int QB>
static int launch_scan_d(oc_ctx *c, const ScanParams &sp, uint32_t grid, size_t smem, uint32_t esz) {
    return esz == 2 ? launch_scan_q<QB, bf16_t>(c, sp, grid, smem) : launch_scan_q<QB, float>(c, sp, grid, smem);
}

struct ScanPlan {
    uint32_t rows_per_stage, n_stages, wcap, grid, qb_max;
};
static ScanPlan plan_scan(const oc_ctx *c, const oc_emb *e, uint32_t n_keep) {
    ScanPlan pl;
    uint32_t qb = 4;
    const uint32_t row_bytes = e->stride * e->esz;
    uint32_t R = (32768 / row_bytes) / 8 * 8;
    if (R < 8) R = 8;
    pl.rows_per_stage = R;
    pl.wcap = std::max<uint32_t>(32, next_pow2(2 * n_keep));
    const size_t budget = 227 * 1024 - 1024;
    while (qb > 1 && size_t(SCAN_CONSUMER_WARPS) * qb * pl.wcap * 8 > budget / 2) qb >>= 1;
    pl.qb_max = qb;
    const size_t fixed = size_t(SCAN_CONSUMER_WARPS) * qb * pl.wcap * 8 + 256;
    const size_t per_stage = size_t(R) * row_bytes + R * 4 + 16;
    uint32_t S = (uint32_t)std::min<size_t>(8, fixed < budget ? (budget - fixed) / per_stage : 0);
    pl.n_stages = S;
    const uint64_t tiles = (e->n_rows + R - 1) / R;
    pl.grid = (uint32_t)std::min<uint64_t>(c->prop.multiProcessorCount, std::max<uint64_t>(tiles, 1));
    return pl;
}

// ---- exact sweeps (K1) + merge for nq prepared queries; results into the given buffers
struct VecOut { uint64_t *doc; float *score; uint32_t *row; uint32_t *cnt; float *raw; };
static int run_exact_sweeps(oc_ctx *c, oc_emb *e, const float *inv_norm, const float *qpad, const float *qinv,
                            uint32_t nq, uint32_t limit, float similarity, const VecOut &o) {
    ScanPlan pl = plan_scan(c, e, limit);
    if (pl.n_stages < 2) return fail(OC_ERR_UNSUPPORTED, "limit %u leaves no shared memory for the scan ring", limit);
    OCTRY(c->scan_cand.ensure(size_t(nq) * pl.grid * limit * 8));
    uint32_t q0 = 0;
    while (q0 < nq) {
        const uint32_t rem = nq - q0;
        const uint32_t qb = std::min<uint32_t>(pl.qb_max, rem >= 4 ? 4 : (rem >= 2 ? 2 : 1));
        ScanParams sp{};
        sp.rows = e->rows; sp.inv_norm = inv_norm; sp.n_rows = e->n_rows; sp.stride = e->stride;
        sp.queries = qpad + size_t(q0) * e->stride;
        sp.inv_qnorm = qinv + q0;
        sp.n_keep = limit; sp.wcap = pl.wcap; sp.rows_per_stage = pl.rows_per_stage; sp.n_stages = pl.n_stages;
        sp.n_ctas_total = pl.grid;
        sp.cand = c->scan_cand.as<uint64_t>() + size_t(q0) * pl.grid * limit;
        const size_t smem = scan_smem_bytes(e->stride, pl.rows_per_stage, pl.n_stages, pl.wcap, qb, e->esz);
        if (qb == 4) OCTRY((launch_scan_d<4>(c, sp, pl.grid, smem, e->esz)));
        else if (qb == 2) OCTRY((launch_scan_d<2>(c, sp, pl.grid, smem, e->esz)));
        else OCTRY((launch_scan_d<1>(c, sp, pl.grid, smem, e->esz)));
        c->timing.scan_bytes += e->n_rows * (uint64_t(e->stride) * e->esz + 4);
        q0 += qb;
    }
    CU(cudaEventRecord(c->ev[EV_SCAN1], c->stream));
    ScanMergeParams mp{};
    mp.cand = c->scan_cand.as<uint64_t>(); mp.n_lists = pl.grid; mp.n_keep = limit; mp.limit = limit;
    mp.capb = std::max<uint32_t>(2048, next_pow2(2 * limit));
    mp.row_doc_ids = e->row_doc; mp.rescale_e5 = e->e5; mp.similarity = similarity;
    mp.out_doc = o.doc; mp.out_score = o.score; mp.out_row = o.row; mp.out_count = o.cnt; mp.out_raw = o.raw;
    if (smem_cfg_needed(c->device, (const void *)emb_scan_merge_kernel, size_t(mp.capb) * 8))
        CU(cudaFuncSetAttribute(emb_scan_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(mp.capb * 8)));
    emb_scan_merge_kernel<<<nq, 256, mp.capb * 8, c->stream>>>(mp);
    launched(c);
    CU(cudaGetLastError());
    return OC_OK;
}

// ---- TMA descriptors (driver entry point fetched through the runtime: no -lcuda link)
typedef CUresult (*EncodeTiled_t)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
// sw64: bf16 matrix, 32-element (64-byte) boxes in the SWIZZLE_64B layout (operand of the converting sweep)
static int make_tmap_2d(CUtensorMap *m, const void *base, uint64_t n_rows, uint32_t stride, uint32_t box_rows, bool bf16,
                        bool sw64 = false) {
    static EncodeTiled_t fn = nullptr;
    if (!fn) {
        void *f = nullptr;
        cudaDriverEntryPointQueryResult qr;
        CU(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &qr));
        if (!f || qr != cudaDriverEntryPointSuccess) return fail(OC_ERR_CUDA, "cuTensorMapEncodeTiled unavailable");
        fn = (EncodeTiled_t)f;
    }
    cuuint64_t dims[2] = {stride, n_rows};
    cuuint64_t strides[1] = {cuuint64_t(stride) * (bf16 ? 2 : 4)};
    cuuint32_t box[2] = {(bf16 && !sw64) ? 2 * GEMM_KB : GEMM_KB, box_rows};   // 128 bytes of K (64 when sw64)
    cuuint32_t estr[2] = {1, 1};
    // L2 promotion granule = the 128-byte box row: with 256 B every tile load also pulled the neighbouring
    // K-block into L2, and the converting sweep re-fetched 17 % of the matrix from DRAM (ncu: 3.59 GB read
    // vs 3.12 GB with 128 B; algorithmic 3.08 GB).  OC_TMA_PROMO=256|none: profiling switch.
    const char *penv = getenv("OC_TMA_PROMO");
    const CUtensorMapL2promotion promo = !penv ? CU_TENSOR_MAP_L2_PROMOTION_L2_128B
                                         : penv[0] == '2' ? CU_TENSOR_MAP_L2_PROMOTION_L2_256B
                                         : penv[0] == 'n' ? CU_TENSOR_MAP_L2_PROMOTION_NONE : CU_TENSOR_MAP_L2_PROMOTION_L2_128B;
    CUresult r = fn(m, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void *>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, sw64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B, promo,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(OC_ERR_CUDA, "cuTensorMapEncodeTiled failed: %d", (int)r);
    return OC_OK;
}

static bool g_disable_gemm = false;   // OC_DISABLE_GEMM=1: force the exact sweep path (A/B testing)

// Runs prep + (tensor-core batched scan | exact sweeps) + merge for B queries already in device
// memory (q_dev: B x dim).  Leaves hits in c->v_doc / v_score / v_row / v_cnt / v_raw ([B][limit]).
static int run_vector_stage(oc_ctx *c, oc_emb *e, const float *q_dev, uint32_t B, uint32_t limit, float similarity,
                            const uint64_t *filter_dev, uint64_t filter_nbits) {
    OCTRY(c->v_doc.ensure(size_t(B) * limit * 8));
    OCTRY(c->v_score.ensure(size_t(B) * limit * 4));
    OCTRY(c->v_row.ensure(size_t(B) * limit * 4));
    OCTRY(c->v_cnt.ensure(size_t(B) * 4));
    OCTRY(c->v_raw.ensure(size_t(B) * limit * 4));
    if (e->n_rows == 0) {
        CU(cudaMemsetAsync(c->v_cnt.p, 0, size_t(B) * 4, c->stream));
        CU(cudaMemsetAsync(c->v_doc.p, 0, size_t(B) * limit * 8, c->stream));
        CU(cudaMemsetAsync(c->v_score.p, 0, size_t(B) * limit * 4, c->stream));
        CU(cudaMemsetAsync(c->v_row.p, 0xff, size_t(B) * limit * 4, c->stream));
        return OC_OK;
    }
    const uint32_t n_qgroups = (B + GEMM_M - 1) / GEMM_M, Bpad = n_qgroups * GEMM_M;
    OCTRY(c->q_pad.ensure(size_t(Bpad) * e->stride * 4));
    OCTRY(c->q_inv.ensure(size_t(Bpad) * 4));
    OCTRY(c->q_rho.ensure(size_t(Bpad) * 4));
    const char *env = getenv("OC_DISABLE_GEMM");
    g_disable_gemm = env && env[0] == '1';
    // tensor-core scan: a batch (the distance is a true GEMM), a store large enough that the threshold pass sees
    // at least `limit` row groups of <= 256 rows with data (its seeds are the limit-th largest group maximum; with
    // fewer live groups the threshold degenerates to "gather everything" and the query falls back to the exact sweep)
    const bool use_gemm = !g_disable_gemm && B >= 8 && limit <= GEMM_MAX_LIMIT && e->n_rows >= std::max<uint64_t>(4096, uint64_t(limit) * 256);
    // (the prep kernel writes rows [0, B) whole, zero padded: only the rows of a partial last query group need clearing)
    if (use_gemm && Bpad != B) CU(cudaMemsetAsync(c->q_pad.as<float>() + size_t(B) * e->stride, 0, size_t(Bpad - B) * e->stride * 4, c->stream));
    emb_prep_queries_kernel<<<(B + 7) / 8, 256, 0, c->stream>>>(q_dev, e->dim, e->stride, B, c->q_pad.as<float>(), c->q_inv.as<float>(),
                                                                c->q_rho.as<float>());
    launched(c);
    const float *inv_norm = e->inv_norm;
    if (filter_dev) {
        OCTRY(c->eff_norm.ensure((e->n_rows + 64) * 4));
        emb_apply_filter_kernel<<<(unsigned)((e->n_rows + 255) / 256), 256, 0, c->stream>>>(
            e->inv_norm, e->row_doc, e->n_rows, filter_dev, filter_nbits, c->eff_norm.as<float>());
        launched(c);
        inv_norm = c->eff_norm.as<float>();
    }
    VecOut out{c->v_doc.as<uint64_t>(), c->v_score.as<float>(), c->v_row.as<uint32_t>(), c->v_cnt.as<uint32_t>(), c->v_raw.as<float>()};
    CU(cudaEventRecord(c->ev[EV_SCAN0], c->stream));
    if (!use_gemm) return run_exact_sweeps(c, e, inv_norm, c->q_pad.as<float>(), c->q_inv.as<float>(), B, limit, similarity, out);

    // ---------------- K2: tcgen05 batched scan ----------------
    const bool bf16 = e->esz == 2;
    // NG = 2: one CTA serves two query groups against each staged X tile (one copy of X per 256 queries)
    const int NG = n_qgroups >= 2 ? 2 : 1;
    const uint32_t n_super = NG == 1 ? n_qgroups : (n_qgroups + 1) / 2;
    // CTA pairs (cta_group::2): two SMs share one 256-query x 512-row tile (25 % less L2->SM traffic)
    const char *penv = getenv("OC_GEMM_PAIR");
    const uint32_t n_pairs = c->prop.multiProcessorCount / 2;
    // default: fp32 stores only (there the pair feeds the converting sweep); for bf16 stores the pair kernel
    // measured ~4 % slower than two groups per CTA on the tensor-bound 10M x 1024 workload (OC_GEMM_PAIR=1 forces it)
    const bool pair_wanted = penv ? penv[0] == '1' : e->esz == 4;
    const bool pair = NG == 2 && pair_wanted && !(penv && penv[0] == '0') && n_pairs >= n_super;
    const uint32_t cpg = pair ? std::max<uint32_t>(1, n_pairs / n_super)
                              : std::max<uint32_t>(1, c->prop.multiProcessorCount / n_super);
    const uint32_t grid = pair ? 2 * cpg * n_super : cpg * n_super;
    const uint32_t lists = (NG == 1 || pair) ? cpg * 2 : cpg;
    if (lists > 512) return fail(OC_ERR_UNSUPPORTED, "%u candidate lists per query (> 512)", lists);
    // fp32 store, pair path: convert the operands to bf16 inside the SM (kind::f16 at twice the tf32 rate)
    const char *cenv = getenv("OC_GEMM_CVT");
    const bool cvt = pair && !bf16 && !(cenv && cenv[0] == '0');
    const uint32_t cap = GEMM_LIST_CAP;
    const uint32_t Bpad2 = n_super * NG * GEMM_M;   // query rows the kernel may address (TMA zero-fills beyond the tensor)
    CUtensorMap tm_q, tm_x;
    const void *q_operand = c->q_pad.p;
    if (bf16 || cvt) {   // the sweep's query operand in the store's dtype (the exact re-score keeps the fp32 query)
        OCTRY(c->q_bf16.ensure(size_t(Bpad) * e->stride * 2));
        const size_t nq_el = size_t(Bpad) * e->stride;
        f32_to_bf16_kernel<<<(unsigned)((nq_el + 255) / 256), 256, 0, c->stream>>>(c->q_pad.as<float>(), c->q_bf16.as<uint16_t>(), nq_el);
        launched(c);
        q_operand = c->q_bf16.p;
    }
    OCTRY(make_tmap_2d(&tm_q, q_operand, Bpad, e->stride, GEMM_M, bf16 || cvt, cvt));
    OCTRY(make_tmap_2d(&tm_x, e->rows, e->n_rows, e->stride, pair ? 128 : GEMM_N, bf16));
    OCTRY(c->g_thr.ensure(size_t(B) * 4));
    OCTRY(c->g_eps.ensure(size_t(B) * 4));
    OCTRY(c->g_cand.ensure(size_t(Bpad2) * lists * cap * 8));
    OCTRY(c->g_cnt.ensure(size_t(Bpad2) * lists * 4));
    OCTRY(c->g_ovf.ensure(size_t(B) * GEMM_OVF_CAP * 8));
    OCTRY(c->g_ovfcnt.ensure(size_t(B) * 4));
    OCTRY(c->g_resc.ensure(size_t(B) * 4));
    OCTRY(c->g_flag.ensure(B));
    OCTRY(c->g_max.ensure(size_t(Bpad2) * lists * 4));
    GemmParams gp{};
    gp.n_rows = e->n_rows; gp.n_kblocks = e->stride / (bf16 ? 2 * GEMM_KB : GEMM_KB); gp.inv_norm = inv_norm; gp.n_queries = B;   // cvt: 32-element K-blocks too
    gp.n_qgroups = n_qgroups; gp.ctas_per_group = cpg; gp.cap = cap; gp.lists_per_query = lists;
    gp.thr = c->g_thr.as<unsigned int>(); gp.eps_v = c->g_eps.as<float>(); gp.limit = limit; gp.cand = c->g_cand.as<uint64_t>(); gp.cand_cnt = c->g_cnt.as<uint32_t>();
    gp.gmax = c->g_max.as<float>();
    gp.ovf = c->g_ovf.as<uint64_t>(); gp.ovf_cnt = c->g_ovfcnt.as<uint32_t>(); gp.ovf_cap = GEMM_OVF_CAP;
    // ring depth of the converting sweep: 5 stages alone on the SM; 4 stages (OC_CVT_STAGES=4) leave ~60 KB of shared
    // memory so one CTA of the BM25 tile scorer (side stream) can co-reside and use the issue slots the HBM-bound sweep leaves idle
    const char *stenv = getenv("OC_CVT_STAGES");
    const uint32_t cvt_stages = (stenv && stenv[0] == '4') ? 4 : (stenv && stenv[0] == '5') ? 5 : c->cvt_stages_default;
    if (smem_cfg_needed(c->device, (const void *)emb_gemm_cvt_kernel<5>, gemm_cvt_smem_bytes(5))) {   // all sweep variants at once
        CU(cudaFuncSetAttribute(emb_gemm_kernel<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gemm_smem_bytes(1)));
        CU(cudaFuncSetAttribute(emb_gemm_kernel<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gemm_smem_bytes(2)));
        CU(cudaFuncSetAttribute(emb_gemm_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gemm_smem_bytes(1)));
        CU(cudaFuncSetAttribute(emb_gemm_kernel<2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gemm_smem_bytes(2)));
        CU(cudaFuncSetAttribute(emb_gemm_pair_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gemm_pair_smem_bytes()));
        CU(cudaFuncSetAttribute(emb_gemm_pair_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gemm_pair_smem_bytes()));
        CU(cudaFuncSetAttribute(emb_gemm_cvt_kernel<5>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gemm_cvt_smem_bytes(5)));
        CU(cudaFuncSetAttribute(emb_gemm_cvt_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gemm_cvt_smem_bytes(4)));
        CU(cudaFuncSetAttribute(emb_gemm_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gemm_merge_smem_bytes()));
    }
    auto launch_gemm = [&]() -> int {
        if (cvt && cvt_stages == 4) emb_gemm_cvt_kernel<4><<<grid, CVT_THREADS, gemm_cvt_smem_bytes(4), c->stream>>>(tm_q, tm_x, gp);
        else if (cvt) emb_gemm_cvt_kernel<5><<<grid, CVT_THREADS, gemm_cvt_smem_bytes(5), c->stream>>>(tm_q, tm_x, gp);
        else if (pair && !bf16) emb_gemm_pair_kernel<false><<<grid, GEMM_THREADS, gemm_pair_smem_bytes(), c->stream>>>(tm_q, tm_x, gp);
        else if (pair) emb_gemm_pair_kernel<true><<<grid, GEMM_THREADS, gemm_pair_smem_bytes(), c->stream>>>(tm_q, tm_x, gp);
        else if (NG == 1 && !bf16) emb_gemm_kernel<1, false><<<grid, GEMM_THREADS, gemm_smem_bytes(1), c->stream>>>(tm_q, tm_x, gp);
        else if (NG == 1) emb_gemm_kernel<1, true><<<grid, GEMM_THREADS, gemm_smem_bytes(1), c->stream>>>(tm_q, tm_x, gp);
        else if (!bf16) emb_gemm_kernel<2, false><<<grid, GEMM_THREADS, gemm_smem_bytes(2), c->stream>>>(tm_q, tm_x, gp);
        else emb_gemm_kernel<2, true><<<grid, GEMM_THREADS, gemm_smem_bytes(2), c->stream>>>(tm_q, tm_x, gp);
        launched(c, gp.max_mode == 0);   // the one-tile threshold pass is not counted as a sweep
        CU(cudaGetLastError());
        return OC_OK;
    };
    // threshold pass: one row tile per CTA, record per-list maxima; thr = (limit-th largest maximum) - 2 eps
    gp.max_mode = 1; gp.tile_limit = 1;
    OCTRY(launch_gemm());
    GemmThrParams tp{};
    tp.gmax = c->g_max.as<float>(); tp.lists = lists; tp.limit = limit; tp.inv_qnorm = c->q_inv.as<float>();
    tp.eps_const = (bf16 || cvt) ? GEMM_EPS_ACC : GEMM_EPS_TF32;
    tp.rho_x = cvt ? e->rho_x : nullptr;                          // bf16 store: the rows are exact
    tp.rho_q = (bf16 || cvt) ? c->q_rho.as<float>() : nullptr;
    tp.thr = c->g_thr.as<unsigned int>(); tp.eps_v = c->g_eps.as<float>(); tp.ovf_cnt = c->g_ovfcnt.as<uint32_t>();
    gemm_thr_kernel<<<B, 256, 0, c->stream>>>(tp);
    launched(c);
    // the sweep
    gp.max_mode = 0; gp.tile_limit = 0;
    CU(cudaEventRecord(c->ev[EV_SWEEP0], c->stream));
    OCTRY(launch_gemm());
    CU(cudaEventRecord(c->ev[EV_SWEEP1], c->stream));
    c->sweep_timed = true;
    c->timing.scan_bytes += e->n_rows * (uint64_t(e->stride) * e->esz + 4);
    CU(cudaEventRecord(c->ev[EV_SCAN1], c->stream));
    GemmMergeParams mp{};
    mp.cand = gp.cand; mp.cand_cnt = gp.cand_cnt; mp.n_lists = lists; mp.cap = cap; mp.limit = limit;
    mp.ovf = gp.ovf; mp.ovf_cnt = gp.ovf_cnt; mp.ovf_cap = gp.ovf_cap; mp.eps_v = tp.eps_v;
    mp.rows = e->rows; mp.rows_bf16 = bf16 ? 1 : 0; mp.stride = e->stride; mp.inv_norm = inv_norm; mp.queries = c->q_pad.as<float>();
    mp.inv_qnorm = c->q_inv.as<float>(); mp.row_doc_ids = e->row_doc; mp.rescale_e5 = e->e5; mp.similarity = similarity;
    mp.out_doc = out.doc; mp.out_score = out.score; mp.out_row = out.row; mp.out_count = out.cnt; mp.out_raw = out.raw;
    mp.out_unproven = c->g_flag.as<uint8_t>(); mp.out_rescored = c->g_resc.as<uint32_t>();
    emb_gemm_merge_kernel<<<B, 512, gemm_merge_smem_bytes(), c->stream>>>(mp);
    launched(c);
    CU(cudaGetLastError());
    // the overflow flags travel back with the results; oc_*search re-runs flagged queries (fix_unproven)
    c->gemm_pending = true; c->gemm_inv_norm = inv_norm;
    c->timing.scan_tensor_core = 1;
    c->timing.scan_variant = cvt ? OC_SCAN_TC_CVT_PAIR : bf16 ? (pair ? OC_SCAN_TC_BF16_PAIR : OC_SCAN_TC_BF16) : (pair ? OC_SCAN_TC_TF32_PAIR : OC_SCAN_TC_TF32);
    return OC_OK;
}

// Re-runs the queries whose tensor-core result failed the exactness proof through the exact
// K1 sweep and patches their slots of c->v_* (rare).  flags: host copy of g_flag.
static int fix_unproven(oc_ctx *c, oc_emb *e, const uint8_t *flags, uint32_t B, uint32_t limit, float similarity,
                        uint32_t *n_redone) {
    std::vector<uint32_t> redo;
    for (uint32_t q = 0; q < B; q++) if (flags[q]) redo.push_back(q);
    *n_redone = (uint32_t)redo.size();
    c->timing.scan_unproven = *n_redone;
    if (redo.empty()) return OC_OK;
    const float *inv_norm = c->gemm_inv_norm;
    VecOut out{c->v_doc.as<uint64_t>(), c->v_score.as<float>(), c->v_row.as<uint32_t>(), c->v_cnt.as<uint32_t>(), c->v_raw.as<float>()};
    const uint32_t nr = (uint32_t)redo.size();
    OCTRY(c->r_qpad.ensure(size_t(nr) * e->stride * 4));
    OCTRY(c->r_qinv.ensure(size_t(nr) * 4));
    OCTRY(c->r_map.ensure(size_t(nr) * 4));
    OCTRY(c->r_doc.ensure(size_t(nr) * limit * 8));
    OCTRY(c->r_score.ensure(size_t(nr) * limit * 4));
    OCTRY(c->r_row.ensure(size_t(nr) * limit * 4));
    OCTRY(c->r_cnt.ensure(size_t(nr) * 4));
    OCTRY(c->r_raw.ensure(size_t(nr) * limit * 4));
    for (uint32_t i = 0; i < nr; i++) {
        CU(cudaMemcpyAsync(c->r_qpad.as<float>() + size_t(i) * e->stride, c->q_pad.as<float>() + size_t(redo[i]) * e->stride,
                           size_t(e->stride) * 4, cudaMemcpyDeviceToDevice, c->stream));
        CU(cudaMemcpyAsync(c->r_qinv.as<float>() + i, c->q_inv.as<float>() + redo[i], 4, cudaMemcpyDeviceToDevice, c->stream));
    }
    CU(cudaMemcpyAsync(c->r_map.p, redo.data(), size_t(nr) * 4, cudaMemcpyHostToDevice, c->stream));
    VecOut ro{c->r_doc.as<uint64_t>(), c->r_score.as<float>(), c->r_row.as<uint32_t>(), c->r_cnt.as<uint32_t>(), c->r_raw.as<float>()};
    OCTRY(run_exact_sweeps(c, e, inv_norm, c->r_qpad.as<float>(), c->r_qinv.as<float>(), nr, limit, similarity, ro));
    scatter_rows_kernel<<<nr, 64, 0, c->stream>>>(c->r_map.as<uint32_t>(), nr, limit, ro.doc, ro.score, ro.row, ro.cnt, ro.raw,
                                                   out.doc, out.score, out.row, out.cnt, out.raw);
    launched(c);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(c->stream));   // redo vector lives on the stack
    return OC_OK;
}

static void begin_call(oc_ctx *c) {
    c->call_launches = 0; c->call_scan_launches = 0; c->gemm_pending = false; c->sweep_timed = false; c->rerun_timed = false;
    memset(&c->timing, 0, sizeof(c->timing));
}
static int finish_timing(oc_ctx *c, bool scan, bool bm, bool fuse, bool comm) {
    auto el = [&](int a, int b) { float ms = 0; cudaEventElapsedTime(&ms, c->ev[a], c->ev[b]); return ms; };
    c->timing.h2d_ms = el(EV_START, EV_H2D);
    c->timing.rerun_ms = c->rerun_timed ? el(EV_RR0, EV_RR1) : 0.f;
    c->timing.device_ms = el(EV_H2D, EV_DEV) + c->timing.rerun_ms;   // a re-run is device work of this batch
    c->timing.d2h_ms = el(EV_DEV, EV_D2H);
    c->timing.scan_ms = scan ? el(EV_SCAN0, EV_SCAN1) : 0;
    c->timing.scan_sweep_ms = !scan ? 0 : (c->sweep_timed ? el(EV_SWEEP0, EV_SWEEP1) : c->timing.scan_ms);
    c->timing.bm25_ms = bm ? el(EV_BM0, EV_BM1) : 0;
    c->timing.fuse_ms = fuse ? el(EV_FUSE0, EV_FUSE1) : 0;
    c->timing.comm_ms = comm ? el(EV_COMM0, EV_COMM1) : 0;
    c->timing.kernel_launches = c->call_launches;
    c->timing.scan_launches = c->call_scan_launches;
    return OC_OK;
}

extern "C" int oc_emb_search(oc_emb *e, const float *queries, uint32_t B, uint32_t limit, float similarity,
                             const uint64_t *filter_bits, uint64_t filter_nbits, uint64_t *out_doc_ids,
                             float *out_scores, uint32_t *out_counts) {
    if (!e || !queries || !out_doc_ids || !out_scores || !out_counts) return fail(OC_ERR_INVALID, "NULL argument");
    if (B == 0) return OC_OK;
    if (limit == 0 || limit > OC_MAX_TOPK) return fail(OC_ERR_UNSUPPORTED, "limit %u outside 1..%u", limit, OC_MAX_TOPK);
    oc_ctx *c = e->ctx;
    std::lock_guard<std::mutex> g(c->mu);
    CU(cudaSetDevice(c->device));
    begin_call(c);
    const size_t qbytes = size_t(B) * e->dim * 4;
    const size_t fwords = filter_bits ? (filter_nbits + 63) / 64 : 0;
    OCTRY(c->in_blob.ensure(qbytes));
    CU(cudaEventRecord(c->ev[EV_START], c->stream));
    CU(cudaMemcpyAsync(c->in_blob.p, queries, qbytes, cudaMemcpyHostToDevice, c->stream));
    if (fwords) {
        OCTRY(c->filter_dev.ensure(fwords * 8));
        CU(cudaMemcpyAsync(c->filter_dev.p, filter_bits, fwords * 8, cudaMemcpyHostToDevice, c->stream));
    }
    c->timing.h2d_bytes = qbytes + fwords * 8;
    CU(cudaEventRecord(c->ev[EV_H2D], c->stream));
    OCTRY(run_vector_stage(c, e, c->in_blob.as<float>(), B, limit, similarity,
                           fwords ? c->filter_dev.as<uint64_t>() : nullptr, filter_nbits));
    CU(cudaEventRecord(c->ev[EV_DEV], c->stream));
    const size_t ob = size_t(B) * limit * 12 + size_t(B) * 4;
    const size_t o_resc = ob + ((size_t(B) + 3) & ~size_t(3));
    OCTRY(c->h_out.ensure(o_resc + size_t(B) * 4));
    uint8_t *h = c->h_out.as<uint8_t>();
    auto fetch = [&]() -> int {
        CU(cudaMemcpyAsync(h, c->v_doc.p, size_t(B) * limit * 8, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaMemcpyAsync(h + size_t(B) * limit * 8, c->v_score.p, size_t(B) * limit * 4, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaMemcpyAsync(h + size_t(B) * limit * 12, c->v_cnt.p, size_t(B) * 4, cudaMemcpyDeviceToHost, c->stream));
        if (c->gemm_pending) {
            CU(cudaMemcpyAsync(h + ob, c->g_flag.p, B, cudaMemcpyDeviceToHost, c->stream));
            CU(cudaMemcpyAsync(h + o_resc, c->g_resc.p, size_t(B) * 4, cudaMemcpyDeviceToHost, c->stream));
        }
        return OC_OK;
    };
    OCTRY(fetch());
    CU(cudaEventRecord(c->ev[EV_D2H], c->stream));
    CU(cudaStreamSynchronize(c->stream));
    if (c->gemm_pending) {
        uint64_t resc = 0;
        for (uint32_t q = 0; q < B; q++) resc += reinterpret_cast<const uint32_t *>(h + o_resc)[q];
        c->timing.scan_rescored = (uint32_t)(resc / B);
        uint32_t redone = 0;
        CU(cudaEventRecord(c->ev[EV_RR0], c->stream));
        OCTRY(fix_unproven(c, e, h + ob, B, limit, similarity, &redone));
        if (redone) {
            c->gemm_pending = false; OCTRY(fetch());
            CU(cudaEventRecord(c->ev[EV_RR1], c->stream));
            c->rerun_timed = true;
            CU(cudaStreamSynchronize(c->stream));
        }
    }
    c->timing.d2h_bytes = ob;
    memcpy(out_doc_ids, h, size_t(B) * limit * 8);
    memcpy(out_scores, h + size_t(B) * limit * 8, size_t(B) * limit * 4);
    memcpy(out_counts, h + size_t(B) * limit * 12, size_t(B) * 4);
    return finish_timing(c, e->n_rows > 0, false, false, false);
}

// ------------------------------------------------------------------------------------ string store
// Snapshot model (the reference keeps `CURRENT` + `versions/<n>` per field and swaps the pointer after
// compact(), embedding_field.rs:91-95 / string_field.rs:186-191): searches work on the published,
// immutable StrSnap they grabbed at call entry; oc_str_commit builds the next snapshot WITHOUT the
// ctx lock (host merge + upload on the store's own stream) and publishes it with a pointer swap, so
// searches keep running on the previous version while a commit is in flight.  Ops that arrive during
// a commit: inserts queue for the next one, deletes hit the old snapshot at once and are replayed on
// the new one before it is published.
struct StrField {
    float avg_len = 0;
    uint32_t n_terms = 0;
    std::vector<uint64_t> term_offsets;  // host copy (n_terms+1)
    std::vector<uint32_t> global_df;     // optional: per-term corpus df across all shards
    PostingRaw *raw = nullptr;           // device: (row, tf, field_len) as loaded
    Posting *post = nullptr;             // device: (row, tf') derived for b_cached
    float b_cached = -1.f;
    uint64_t n_post = 0;
    std::vector<PostingRaw> host_post;   // host copy of the committed postings (term-major), kept for oc_str_commit
};
struct StrSnap {
    int device = 0;
    uint64_t version = 0;
    std::vector<StrField> fields;
    uint64_t n_rows = 0, document_count = 0;
    std::vector<uint64_t> row_doc_host;  // empty => identity
    uint64_t *row_doc = nullptr;         // device or NULL
    uint32_t *alive = nullptr;           // device bitmap (allocated on first delete)
    std::vector<uint32_t> alive_host;
    uint64_t n_deleted = 0;
    ~StrSnap() {
        int dev = -1;
        cudaGetDevice(&dev);
        if (dev != device) cudaSetDevice(device);
        for (auto &f : fields) { cudaFree(f.post); cudaFree(f.raw); }
        cudaFree(row_doc); cudaFree(alive);
        if (dev >= 0 && dev != device) cudaSetDevice(dev);
    }
    // row of a DocumentId, or ~0ull
    uint64_t row_of(uint64_t doc) const {
        if (row_doc_host.empty()) return doc < n_rows ? doc : ~0ull;
        auto it = std::lower_bound(row_doc_host.begin(), row_doc_host.end(), doc);
        return (it == row_doc_host.end() || *it != doc) ? ~0ull : uint64_t(it - row_doc_host.begin());
    }
};
struct PendingPost { uint64_t doc, seq; uint32_t term; uint16_t tf, len; };   // term == ~0u: "document inserted with no term"
struct oc_str {
    oc_ctx *ctx = nullptr;
    std::mutex mu;                                   // cur / pending / logs (short critical sections; never held across device work of a search)
    std::shared_ptr<StrSnap> cur;                    // the published snapshot ("CURRENT")
    uint64_t version = 0;
    std::vector<std::vector<PendingPost>> pending;   // per field: StringFieldStorage::insert since the last commit
    uint64_t seq = 0;                                // op sequence: a delete only cancels inserts that came before it
    std::unordered_map<uint64_t, uint64_t> pending_deleted;   // doc -> seq of its latest delete
    bool committing = false;
    std::vector<uint64_t> deletes_during_commit;
    bool global_count = false, global_avg = false;   // document_count / avg_field_len are values owned by the caller (shard of a larger index; an
                                                     // Index whose document_count also counts documents without string fields): commit keeps them
    cudaStream_t load_stream = nullptr;
};
static std::shared_ptr<StrSnap> str_snapshot(oc_str *s) {
    std::lock_guard<std::mutex> g(s->mu);
    return s->cur;
}

extern "C" int oc_str_create(oc_ctx *c, uint32_t n_fields, oc_str **out) {
    if (!c || !out || n_fields == 0) return fail(OC_ERR_INVALID, "bad arguments");
    std::lock_guard<std::mutex> g(c->mu);
    CU(cudaSetDevice(c->device));
    oc_str *s = new oc_str();
    s->ctx = c;
    s->cur = std::make_shared<StrSnap>();
    s->cur->device = c->device;
    s->cur->fields.resize(n_fields);
    s->pending.resize(n_fields);
    CU(cudaStreamCreateWithFlags(&s->load_stream, cudaStreamNonBlocking));
    *out = s;
    return OC_OK;
}
extern "C" void oc_str_destroy(oc_str *s) {
    if (!s) return;
    cudaSetDevice(s->ctx->device);
    cudaStreamSynchronize(s->ctx->stream);
    if (s->load_stream) { cudaStreamSynchronize(s->load_stream); cudaStreamDestroy(s->load_stream); }
    s->cur.reset();
    delete s;
}

// Bulk load (oc_str_set_rows + oc_str_load_field per field) starts a fresh snapshot; both run under the
// ctx lock, i.e. never concurrently with a search on this ctx.
extern "C" int oc_str_set_rows(oc_str *s, uint64_t n_rows, const uint64_t *row_doc_ids, uint64_t document_count) {
    if (!s) return fail(OC_ERR_INVALID, "str is NULL");
    if (n_rows > 0xfffffff0ull) return fail(OC_ERR_UNSUPPORTED, "more than 2^32 rows per store");
    oc_ctx *c = s->ctx;
    std::lock_guard<std::mutex> g(c->mu);
    CU(cudaSetDevice(c->device));
    if (row_doc_ids)
        for (uint64_t i = 1; i < n_rows; i++)
            if (row_doc_ids[i] <= row_doc_ids[i - 1]) return fail(OC_ERR_INVALID, "row_doc_ids must be strictly ascending");
    auto ns = std::make_shared<StrSnap>();
    ns->device = c->device;
    ns->n_rows = n_rows; ns->document_count = document_count;
    if (row_doc_ids && n_rows) {
        ns->row_doc_host.assign(row_doc_ids, row_doc_ids + n_rows);
        CU(cudaMalloc(&ns->row_doc, n_rows * 8));
        CU(cudaMemcpy(ns->row_doc, row_doc_ids, n_rows * 8, cudaMemcpyHostToDevice));
    }
    std::lock_guard<std::mutex> g2(s->mu);
    if (s->committing) return fail(OC_ERR_INVALID, "oc_str_set_rows while a commit is in flight");
    ns->fields.resize(s->cur->fields.size());
    ns->version = ++s->version;
    s->cur = ns;
    // a document count that differs from the row count can only be a corpus-wide N (this store is a shard)
    s->global_count = s->global_avg = document_count != n_rows;
    for (auto &p : s->pending) p.clear();
    s->pending_deleted.clear();
    return OC_OK;
}

extern "C" int oc_str_set_global(oc_str *s, uint64_t document_count, const float *avg_field_len) {
    if (!s) return fail(OC_ERR_INVALID, "str is NULL");
    oc_ctx *c = s->ctx;
    std::lock_guard<std::mutex> g(c->mu);
    std::lock_guard<std::mutex> g2(s->mu);
    StrSnap &S = *s->cur;
    S.document_count = document_count;
    if (avg_field_len)
        for (size_t i = 0; i < S.fields.size(); i++)
            if (S.fields[i].avg_len != avg_field_len[i]) { S.fields[i].avg_len = avg_field_len[i]; S.fields[i].b_cached = -1.f; }
    s->global_count = true;
    s->global_avg = avg_field_len != nullptr;
    return OC_OK;
}

extern "C" int oc_str_load_field(oc_str *s, uint32_t field, float avg_field_len, uint32_t n_terms,
                                 const uint64_t *term_offsets, const uint32_t *post_row, const uint16_t *post_tf,
                                 const uint16_t *post_len, const uint32_t *global_df) {
    if (!s || !term_offsets) return fail(OC_ERR_INVALID, "bad arguments");
    oc_ctx *c = s->ctx;
    std::lock_guard<std::mutex> g(c->mu);
    CU(cudaSetDevice(c->device));
    std::shared_ptr<StrSnap> snap = str_snapshot(s);
    StrSnap &S = *snap;
    if (field >= S.fields.size()) return fail(OC_ERR_INVALID, "field %u out of range", field);
    StrField &f = S.fields[field];
    cudaFree(f.post); f.post = nullptr; cudaFree(f.raw); f.raw = nullptr; f.b_cached = -1.f;
    const uint64_t np = term_offsets[n_terms];
    if (np && (!post_row || !post_tf || !post_len)) return fail(OC_ERR_INVALID, "posting arrays are NULL");
    for (uint32_t t = 0; t < n_terms; t++) {
        if (term_offsets[t + 1] < term_offsets[t]) return fail(OC_ERR_INVALID, "term_offsets not monotone");
        if (term_offsets[t + 1] - term_offsets[t] > 0xffffffffull) return fail(OC_ERR_UNSUPPORTED, "posting list too long");
    }
    f.avg_len = avg_field_len; f.n_terms = n_terms; f.n_post = np;
    f.host_post.resize(np);
    for (uint64_t i = 0; i < np; i++) {
        if (post_row[i] >= S.n_rows && S.n_rows) return fail(OC_ERR_INVALID, "posting row %u >= n_rows", post_row[i]);
        f.host_post[i].row = post_row[i]; f.host_post[i].tf = post_tf[i]; f.host_post[i].len = post_len[i];
    }
    f.term_offsets.assign(term_offsets, term_offsets + n_terms + 1);
    f.global_df.clear();
    if (global_df) f.global_df.assign(global_df, global_df + n_terms);
    if (np) {
        CU(cudaMalloc(&f.post, (np + 4) * sizeof(Posting)));
        CU(cudaMalloc(&f.raw, (np + 4) * sizeof(PostingRaw)));
        CU(cudaMemcpyAsync(f.raw, f.host_post.data(), np * sizeof(PostingRaw), cudaMemcpyHostToDevice, c->stream));
        CU(cudaStreamSynchronize(c->stream));
    }
    return OC_OK;
}

// tombstones `rows` of snapshot S (host bitmap + device copy on stream st)
static int snap_tombstone(StrSnap &S, const std::vector<uint64_t> &rows, cudaStream_t st) {
    if (rows.empty() || S.n_rows == 0) return OC_OK;
    const uint64_t words = (S.n_rows + BM25_TILE - 1) / BM25_TILE * (BM25_TILE / 32);
    if (S.alive_host.empty()) {
        S.alive_host.assign(words, 0xffffffffu);
        CU(cudaMalloc(&S.alive, words * 4));
    }
    for (uint64_t r : rows)
        if (S.alive_host[r >> 5] & (1u << (r & 31))) { S.alive_host[r >> 5] &= ~(1u << (r & 31)); S.n_deleted++; }
    CU(cudaMemcpyAsync(S.alive, S.alive_host.data(), words * 4, cudaMemcpyHostToDevice, st));
    CU(cudaStreamSynchronize(st));
    return OC_OK;
}

// StringFieldStorage::delete (string_field.rs:180-182).  Ops apply in order, as the reference's compact
// does: a delete tombstones the committed rows of the document now and cancels its inserts that are
// still pending (inserted before this call); an insert after the delete is a new document.
extern "C" int oc_str_delete(oc_str *s, const uint64_t *doc_ids, uint64_t n) {
    if (!s || (!doc_ids && n)) return fail(OC_ERR_INVALID, "NULL argument");
    oc_ctx *c = s->ctx;
    std::lock_guard<std::mutex> g(c->mu);      // the device bitmap is read by searches on the ctx stream
    CU(cudaSetDevice(c->device));
    std::lock_guard<std::mutex> g2(s->mu);
    StrSnap &S = *s->cur;
    std::vector<uint64_t> rows;
    for (uint64_t i = 0; i < n; i++) {
        s->pending_deleted[doc_ids[i]] = ++s->seq;
        if (s->committing) s->deletes_during_commit.push_back(doc_ids[i]);
        const uint64_t r = S.row_of(doc_ids[i]);
        if (r != ~0ull) rows.push_back(r);
    }
    return snap_tombstone(S, rows, c->stream);
}

// StringFieldStorage::insert(DocumentId, IndexedValue{field_length, terms}) (string_field.rs:155-177):
// buffered on the host; visible to searches after oc_str_commit (== compact, :186-191).  Inserting a
// document again (before or after a commit) replaces its postings in that field: last insert wins.
extern "C" int oc_str_insert(oc_str *s, uint32_t field, uint64_t doc_id, uint16_t field_len, uint32_t n_terms,
                             const uint32_t *term_ids, const uint16_t *tfs) {
    if (!s || (n_terms && (!term_ids || !tfs))) return fail(OC_ERR_INVALID, "bad arguments");
    std::lock_guard<std::mutex> g(s->mu);
    if (field >= s->pending.size()) return fail(OC_ERR_INVALID, "field %u out of range", field);
    for (uint32_t i = 0; i < n_terms; i++)
        if (term_ids[i] == 0xffffffffu) return fail(OC_ERR_INVALID, "term id 0xffffffff is reserved");
    const uint64_t q = ++s->seq;
    auto &pv = s->pending[field];
    if (n_terms == 0) pv.push_back({doc_id, q, 0xffffffffu, 0, field_len});
    for (uint32_t i = 0; i < n_terms; i++) pv.push_back({doc_id, q, term_ids[i], tfs[i], field_len});
    return OC_OK;
}

// Merges pending inserts and deletes into the next snapshot: rows are the ascending doc ids, postings
// term-major / row-ascending, avg_field_len and document_count refreshed (unless the caller owns the
// corpus-wide values), tombstones dropped.  Everything is built in temporaries; the published snapshot
// is replaced only after every field validated and uploaded, so a failed commit changes nothing.
extern "C" int oc_str_commit(oc_str *s) {
    if (!s) return fail(OC_ERR_INVALID, "str is NULL");
    oc_ctx *c = s->ctx;
    std::shared_ptr<StrSnap> base;
    std::vector<std::vector<PendingPost>> pend;
    std::unordered_map<uint64_t, uint64_t> pdel;
    std::vector<uint32_t> base_alive;
    bool global_count, global_avg;
    {
        std::lock_guard<std::mutex> g(s->mu);
        if (s->committing) return fail(OC_ERR_INVALID, "a commit of this store is already in flight");
        s->committing = true;
        s->deletes_during_commit.clear();
        base = s->cur;
        pend.resize(s->pending.size());
        for (size_t i = 0; i < pend.size(); i++) pend[i].swap(s->pending[i]);
        pdel.swap(s->pending_deleted);
        base_alive = base->alive_host;
        global_count = s->global_count; global_avg = s->global_avg;
    }
    // on failure: put the taken ops back (in front of whatever arrived meanwhile) and leave `cur` alone
    auto abort_commit = [&](int rc) {
        std::lock_guard<std::mutex> g(s->mu);
        for (size_t i = 0; i < pend.size(); i++) {
            pend[i].insert(pend[i].end(), s->pending[i].begin(), s->pending[i].end());
            s->pending[i].swap(pend[i]);
        }
        for (auto &kv : pdel) { auto it = s->pending_deleted.find(kv.first); if (it == s->pending_deleted.end() || it->second < kv.second) s->pending_deleted[kv.first] = kv.second; }
        s->committing = false;
        return rc;
    };
    if (cudaSetDevice(c->device) != cudaSuccess) return abort_commit(fail(OC_ERR_CUDA, "cudaSetDevice failed"));
    const StrSnap &B = *base;
    const size_t nf = B.fields.size();
    // ---- pending ops in order: drop inserts cancelled by a later delete, keep the last insert per (field, doc)
    for (size_t fi = 0; fi < nf; fi++) {
        auto &pv = pend[fi];
        std::unordered_map<uint64_t, uint64_t> last;   // doc -> seq of its last surviving insert in this field
        for (auto &pn : pv) {
            auto d = pdel.find(pn.doc);
            if (d != pdel.end() && pn.seq < d->second) continue;
            uint64_t &l = last[pn.doc];
            if (pn.seq > l) l = pn.seq;
        }
        size_t w = 0;
        for (auto &pn : pv) {
            auto it = last.find(pn.doc);
            if (it != last.end() && it->second == pn.seq) pv[w++] = pn;
        }
        pv.resize(w);
    }
    // ---- row space of the next snapshot
    std::vector<uint64_t> docs;
    std::vector<uint8_t> old_alive(B.n_rows, 1);
    for (uint64_t r = 0; r < B.n_rows; r++) {
        const bool alive = base_alive.empty() || ((base_alive[r >> 5] >> (r & 31)) & 1u);
        old_alive[r] = alive;
        if (alive) docs.push_back(B.row_doc_host.empty() ? r : B.row_doc_host[r]);
    }
    for (auto &pv : pend) for (auto &pn : pv) docs.push_back(pn.doc);
    std::sort(docs.begin(), docs.end());
    docs.erase(std::unique(docs.begin(), docs.end()), docs.end());
    if (docs.size() > 0xfffffff0ull) return abort_commit(fail(OC_ERR_UNSUPPORTED, "more than 2^32 rows per store"));
    auto row_of = [&](uint64_t d) { return (uint32_t)(std::lower_bound(docs.begin(), docs.end(), d) - docs.begin()); };
    std::vector<uint32_t> remap(B.n_rows, 0xffffffffu);
    for (uint64_t r = 0; r < B.n_rows; r++) if (old_alive[r]) remap[r] = row_of(B.row_doc_host.empty() ? r : B.row_doc_host[r]);
    auto ns = std::make_shared<StrSnap>();
    ns->device = c->device;
    ns->fields.resize(nf);
    struct Rec { uint32_t term, row; uint16_t tf, len; };
    for (size_t fi = 0; fi < nf; fi++) {
        const StrField &of = B.fields[fi];
        StrField &f = ns->fields[fi];
        // the committed postings are already term-major / row-ascending and the row remap is monotone, so only the
        // PENDING postings are sorted; the next CSR is a per-term linear merge of (surviving old list, new list):
        // O(P_old + p log p) instead of a sort of everything
        std::vector<uint8_t> replaced(docs.size(), 0);   // a re-inserted document replaces its old postings in this field
        for (auto &pn : pend[fi]) replaced[row_of(pn.doc)] = 1;
        std::vector<Rec> add;
        add.reserve(pend[fi].size());
        uint32_t max_term = of.n_terms;
        for (auto &pn : pend[fi]) {
            if (pn.term == 0xffffffffu) continue;
            add.push_back({pn.term, row_of(pn.doc), pn.tf, pn.len});
            max_term = std::max(max_term, pn.term + 1);
        }
        std::sort(add.begin(), add.end(), [](const Rec &a, const Rec &b) { return a.term != b.term ? a.term < b.term : a.row < b.row; });
        for (size_t i = 1; i < add.size(); i++)
            if (add[i].term == add[i - 1].term && add[i].row == add[i - 1].row)
                return abort_commit(fail(OC_ERR_INVALID, "field %zu: term %u listed twice in one insert of a document", fi, add[i].term));
        f.n_terms = max_term;
        f.term_offsets.assign(size_t(max_term) + 1, 0);
        f.host_post.clear();
        f.host_post.reserve(of.host_post.size() + add.size());
        std::vector<uint16_t> len_of_row(docs.size(), 0);
        size_t ai = 0;
        for (uint32_t t = 0; t < max_term; t++) {
            f.term_offsets[t] = f.host_post.size();
            uint64_t oi = t < of.n_terms ? of.term_offsets[t] : 0, oe = t < of.n_terms ? of.term_offsets[t + 1] : 0;
            auto old_next = [&]() -> bool {   // advances oi to the next surviving old posting of this term
                while (oi < oe) {
                    const uint32_t nr = remap[of.host_post[oi].row];
                    if (nr != 0xffffffffu && !replaced[nr]) return true;
                    oi++;
                }
                return false;
            };
            for (;;) {
                const bool ho = old_next(), hn = ai < add.size() && add[ai].term == t;
                if (!ho && !hn) break;
                PostingRaw pr;
                if (ho && (!hn || remap[of.host_post[oi].row] < add[ai].row)) {
                    pr.row = remap[of.host_post[oi].row]; pr.tf = of.host_post[oi].tf; pr.len = of.host_post[oi].len; oi++;
                } else {   // (equal rows cannot happen: a row with a pending insert is `replaced`)
                    pr.row = add[ai].row; pr.tf = add[ai].tf; pr.len = add[ai].len; ai++;
                }
                f.host_post.push_back(pr);
                len_of_row[pr.row] = pr.len;
            }
        }
        f.term_offsets[max_term] = f.host_post.size();
        const size_t n_recs = f.host_post.size();
        f.avg_len = of.avg_len;
        if (!global_avg) {
            double sum = 0; uint64_t cnt = 0;
            for (uint16_t l : len_of_row) if (l) { sum += l; cnt++; }
            if (cnt) f.avg_len = (float)(sum / (double)cnt);   // info().avg_field_length
        }
        f.n_post = n_recs;
        // per-term corpus df of a shard cannot be refreshed locally: sharded searches on this snapshot count
        // df across ranks (OC_SHARD_COUNT_DF) until the caller loads new global tables
    }
    const bool identity = !docs.empty() && docs.front() == 0 && docs.back() == docs.size() - 1;
    ns->n_rows = docs.size();
    ns->document_count = global_count ? B.document_count : docs.size();
    // ---- upload on the store's own stream (searches keep the ctx stream)
    auto upload = [&]() -> int {
        if (!identity && !docs.empty()) {
            ns->row_doc_host = docs;
            CU(cudaMalloc(&ns->row_doc, docs.size() * 8));
            CU(cudaMemcpyAsync(ns->row_doc, docs.data(), docs.size() * 8, cudaMemcpyHostToDevice, s->load_stream));
        }
        for (auto &f : ns->fields) {
            const uint64_t np = f.host_post.size();
            if (!np) continue;
            CU(cudaMalloc(&f.post, (np + 4) * sizeof(Posting)));
            CU(cudaMalloc(&f.raw, (np + 4) * sizeof(PostingRaw)));
            CU(cudaMemcpyAsync(f.raw, f.host_post.data(), np * sizeof(PostingRaw), cudaMemcpyHostToDevice, s->load_stream));
        }
        CU(cudaStreamSynchronize(s->load_stream));
        return OC_OK;
    };
    const int urc = upload();
    if (urc != OC_OK) return abort_commit(urc);
    // ---- publish: replay the deletes that arrived while we were building, then swap the pointer
    {
        std::lock_guard<std::mutex> g(s->mu);
        std::vector<uint64_t> rows;
        for (uint64_t d : s->deletes_during_commit) { const uint64_t r = ns->row_of(d); if (r != ~0ull) rows.push_back(r); }
        const int trc = snap_tombstone(*ns, rows, s->load_stream);
        if (trc != OC_OK) { s->committing = false; return trc; }   // (pending ops were consumed; the old snapshot stays published)
        ns->version = ++s->version;
        s->cur = ns;
        s->deletes_during_commit.clear();
        s->committing = false;
    }
    return OC_OK;
}

extern "C" int oc_str_info(oc_str *s, oc_str_info_t *out) {
    if (!s || !out) return fail(OC_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> g(s->mu);
    const StrSnap &S = *s->cur;
    out->total_documents = S.n_rows - S.n_deleted; out->n_fields = (uint32_t)S.fields.size();
    out->total_postings = 0; out->unique_terms_count = 0;
    for (auto &f : S.fields) { out->total_postings += f.n_post; out->unique_terms_count += f.n_terms; }
    out->device_bytes = out->total_postings * 16 + (S.row_doc ? S.n_rows * 8 : 0);
    out->version = S.version;
    out->pending_postings = 0;
    for (auto &p : s->pending) out->pending_postings += p.size();
    return OC_OK;
}

// ------------------------------------------------------------------------------------ device-resident filters
struct oc_facets;
struct oc_sort;
struct oc_filter {
    oc_ctx *ctx;
    uint64_t nbits, words;
    uint64_t *bits = nullptr;   // device
};
__global__ void filter_scatter_ids_kernel(const uint64_t *ids, uint64_t n, uint64_t nbits, unsigned long long *bits) {
    const uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t d = ids[i];
    if (d < nbits) atomicOr(bits + (d >> 6), 1ull << (d & 63));
}
// op: 0 and, 1 or, 2 not(a); the padding bits of the last word stay clear
__global__ void filter_combine_kernel(const uint64_t *a, const uint64_t *b, uint64_t words, uint64_t nbits, int op, uint64_t *out) {
    const uint64_t w = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (w >= words) return;
    uint64_t v = op == 0 ? (a[w] & b[w]) : op == 1 ? (a[w] | b[w]) : ~a[w];
    if (w == words - 1 && (nbits & 63)) v &= (1ull << (nbits & 63)) - 1;
    out[w] = v;
}
__global__ void filter_popcount_kernel(const uint64_t *a, uint64_t words, unsigned long long *out) {
    uint64_t c = 0;
    for (uint64_t w = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x; w < words; w += uint64_t(gridDim.x) * blockDim.x) c += __popcll(a[w]);
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(out, (unsigned long long)c);
}
static int filter_alloc(oc_ctx *c, uint64_t nbits, oc_filter **out) {
    oc_filter *f = new oc_filter();
    f->ctx = c; f->nbits = nbits; f->words = (nbits + 63) / 64;
    cudaError_t e = cudaMalloc(&f->bits, std::max<uint64_t>(f->words, 1) * 8);
    if (e != cudaSuccess) { delete f; return fail(OC_ERR_OOM, "cudaMalloc(filter): %s", cudaGetErrorString(e)); }
    *out = f;
    return OC_OK;
}
extern "C" void oc_filter_destroy(oc_filter *f) {
    if (!f) return;
    std::lock_guard<std::mutex> g(f->ctx->mu);
    cudaSetDevice(f->ctx->device);
    cudaStreamSynchronize(f->ctx->stream);
    cudaFree(f->bits);
    delete f;
}
extern "C" int oc_filter_from_ids(oc_ctx *c, const uint64_t *doc_ids, uint64_t n, uint64_t nbits, oc_filter **out) {
    if (!c || !out || (n && !doc_ids)) return fail(OC_ERR_INVALID, "bad arguments");
    std::lock_guard<std::mutex> g(c->mu);
    CU(cudaSetDevice(c->device));
    oc_filter *f = nullptr;
    OCTRY(filter_alloc(c, nbits, &f));
    CU(cudaMemsetAsync(f->bits, 0, std::max<uint64_t>(f->words, 1) * 8, c->stream));
    if (n) {
        OCTRY(c->in_blob.ensure(n * 8));
        CU(cudaMemcpyAsync(c->in_blob.p, doc_ids, n * 8, cudaMemcpyHostToDevice, c->stream));
        filter_scatter_ids_kernel<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(c->in_blob.as<uint64_t>(), n, nbits,
                                                                                    reinterpret_cast<unsigned long long *>(f->bits));
        launched(c);
        CU(cudaGetLastError());
    }
    CU(cudaStreamSynchronize(c->stream));
    *out = f;
    return OC_OK;
}
extern "C" int oc_filter_from_bits(oc_ctx *c, const uint64_t *bits, uint64_t nbits, oc_filter **out) {
    if (!c || !out || (nbits && !bits)) return fail(OC_ERR_INVALID, "bad arguments");
    std::lock_guard<std::mutex> g(c->mu);
    CU(cudaSetDevice(c->device));
    oc_filter *f = nullptr;
    OCTRY(filter_alloc(c, nbits, &f));
    if (f->words) CU(cudaMemcpy(f->bits, bits, f->words * 8, cudaMemcpyHostToDevice));
    *out = f;
    return OC_OK;
}
static int filter_combine(const oc_filter *a, const oc_filter *b, int op, oc_filter **out) {
    if (!a || !out || (op != 2 && !b)) return fail(OC_ERR_INVALID, "NULL argument");
    if (b && (b->ctx != a->ctx || b->nbits != a->nbits)) return fail(OC_ERR_INVALID, "filters of different contexts / sizes");
    oc_ctx *c = a->ctx;
    std::lock_guard<std::mutex> g(c->mu);
    CU(cudaSetDevice(c->device));
    oc_filter *f = nullptr;
    OCTRY(filter_alloc(c, a->nbits, &f));
    if (f->words) {
        filter_combine_kernel<<<(unsigned)((f->words + 255) / 256), 256, 0, c->stream>>>(a->bits, b ? b->bits : nullptr, f->words, f->nbits, op, f->bits);
        launched(c);
        CU(cudaGetLastError());
        CU(cudaStreamSynchronize(c->stream));
    }
    *out = f;
    return OC_OK;
}
extern "C" int oc_filter_and(const oc_filter *a, const oc_filter *b, oc_filter **out) { return filter_combine(a, b, 0, out); }
extern "C" int oc_filter_or(const oc_filter *a, const oc_filter *b, oc_filter **out) { return filter_combine(a, b, 1, out); }
extern "C" int oc_filter_not(const oc_filter *a, oc_filter **out) { return filter_combine(a, nullptr, 2, out); }
extern "C" int oc_filter_count(const oc_filter *f, uint64_t *out) {
    if (!f || !out) return fail(OC_ERR_INVALID, "NULL argument");
    oc_ctx *c = f->ctx;
    std::lock_guard<std::mutex> g(c->mu);
    CU(cudaSetDevice(c->device));
    OCTRY(c->work_ctr.ensure(8));
    CU(cudaMemsetAsync(c->work_ctr.p, 0, 8, c->stream));
    if (f->words) {
        filter_popcount_kernel<<<(unsigned)std::min<uint64_t>((f->words + 255) / 256, 1184), 256, 0, c->stream>>>(
            f->bits, f->words, c->work_ctr.as<unsigned long long>());
        launched(c);
    }
    unsigned long long v = 0;
    CU(cudaMemcpyAsync(&v, c->work_ctr.p, 8, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    *out = v;
    return OC_OK;
}
extern "C" int oc_filter_read(const oc_filter *f, uint64_t *out_bits) {
    if (!f || !out_bits) return fail(OC_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> g(f->ctx->mu);
    CU(cudaSetDevice(f->ctx->device));
    CU(cudaStreamSynchronize(f->ctx->stream));
    if (f->words) CU(cudaMemcpy(out_bits, f->bits, f->words * 8, cudaMemcpyDeviceToHost));
    return OC_OK;
}

// ------------------------------------------------------------------------------------ multi-index union (host)
extern "C" int oc_merge_results(uint32_t n_indexes, uint32_t B, uint32_t limit, uint32_t offset, uint32_t in_stride,
                                const uint64_t *const *doc_ids, const float *const *scores, const uint32_t *const *n,
                                const uint64_t *const *counts, uint64_t *out_doc_ids, float *out_scores, uint32_t *out_n,
                                uint64_t *out_count) {
    if (!doc_ids || !scores || !n || !counts || !out_doc_ids || !out_scores || !out_n || !out_count) return fail(OC_ERR_INVALID, "NULL argument");
    if (limit == 0) return fail(OC_ERR_INVALID, "limit must be >= 1");
    std::vector<uint32_t> head(n_indexes);
    for (uint32_t q = 0; q < B; q++) {
        std::fill(head.begin(), head.end(), 0u);
        uint64_t cnt = 0;
        for (uint32_t i = 0; i < n_indexes; i++) {
            if (n[i][q] > in_stride) return fail(OC_ERR_INVALID, "index %u query %u: n > in_stride", i, q);
            cnt += counts[i][q];
        }
        uint32_t taken = 0, written = 0;
        while (written < limit) {   // k-way merge of lists already sorted by (score desc, doc asc); NaN never reaches a list
            int best = -1;
            for (uint32_t i = 0; i < n_indexes; i++) {
                if (head[i] >= n[i][q]) continue;
                if (best < 0) { best = (int)i; continue; }
                const float sa = scores[i][size_t(q) * in_stride + head[i]], sb = scores[best][size_t(q) * in_stride + head[best]];
                const uint64_t da = doc_ids[i][size_t(q) * in_stride + head[i]], db = doc_ids[best][size_t(q) * in_stride + head[best]];
                if (sa > sb || (sa == sb && da < db)) best = (int)i;
            }
            if (best < 0) break;
            if (taken >= offset) {
                out_doc_ids[size_t(q) * limit + written] = doc_ids[best][size_t(q) * in_stride + head[best]];
                out_scores[size_t(q) * limit + written] = scores[best][size_t(q) * in_stride + head[best]];
                written++;
            }
            taken++; head[best]++;
        }
        for (uint32_t k = written; k < limit; k++) { out_doc_ids[size_t(q) * limit + k] = 0; out_scores[size_t(q) * limit + k] = 0.f; }
        out_n[q] = written;
        out_count[q] = cnt;
    }
    return OC_OK;
}

// ------------------------------------------------------------------------------------ search()
// bm25.rs:78-82, evaluated on the host with libm (the same log1pf the oracle uses)
static inline float host_idf(float total_documents, uint64_t corpus_df) {
    const float df = (float)corpus_df;
    const float ratio = (total_documents - df + 0.5f) / (df + 0.5f);
    return log1pf(ratio);
}

template <bool MULTI, bool THRESH, bool OMC>
static int launch_tile_t(oc_ctx *c, const Bm25Params &bp, uint32_t grid, size_t smem, cudaStream_t st) {
    // (static smem counts against the 227 KB cap)
    if (smem_cfg_needed(c->device, (const void *)bm25_tile_kernel<MULTI, THRESH, OMC>, smem))
        CU(cudaFuncSetAttribute(bm25_tile_kernel<MULTI, THRESH, OMC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    bm25_tile_kernel<MULTI, THRESH, OMC><<<grid, BM25_THREADS, smem, st>>>(bp);
    launched(c);
    CU(cudaGetLastError());
    return OC_OK;
}
template <bool THRESH, bool OMC>
static int launch_tile2_t(oc_ctx *c, const Bm25Params &bp, size_t smem, cudaStream_t st, const ItemTok *flat, unsigned int *counter) {
    if (smem_cfg_needed(c->device, (const void *)bm25_tile2_kernel<THRESH, OMC>, smem))
        CU(cudaFuncSetAttribute(bm25_tile2_kernel<THRESH, OMC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    static std::mutex occ_mu;                         // occupancy per (device, shared-memory size): queried once
    static std::map<std::pair<int, size_t>, int> occ;
    int per_sm = 1;
    {
        std::lock_guard<std::mutex> g(occ_mu);
        auto it = occ.find(std::make_pair(c->device, smem));
        if (it == occ.end()) {
            CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, bm25_tile2_kernel<THRESH, OMC>, BM25_THREADS, smem));
            occ[std::make_pair(c->device, smem)] = per_sm;
        } else per_sm = it->second;
    }
    const uint64_t items = uint64_t(bp.n_tiles) * bp.n_queries;
    const uint32_t grid = (uint32_t)std::min<uint64_t>(items, uint64_t(std::max(per_sm, 1)) * c->prop.multiProcessorCount);
    bm25_tile2_kernel<THRESH, OMC><<<grid, BM25_THREADS, smem, st>>>(bp, flat, counter);
    launched(c);
    CU(cudaGetLastError());
    return OC_OK;
}
// multi == false (every token resolves to <= 1 term): the posting-centred persistent kernel; else the slot-scan kernel
static int launch_tile(oc_ctx *c, const Bm25Params &bp_in, uint32_t grid, bool multi, bool thr, bool omc, cudaStream_t st,
                       uint32_t max_tokens, unsigned int *counter /* zeroed by the caller */, bool counted_df) {
    const char *env = getenv("OC_BM25_TILE2");
    if (!multi && !(env && env[0] == '0')) {
        // one level of descriptors per (tile, query) item, prefetched by the kernel during the previous item
        const ItemTok *flat = nullptr;
        const char *fenv = getenv("OC_BM25_FLAT");
        const char *t3e = getenv("OC_BM25_TILE3");
        const bool can_flat = max_tokens <= BM25_FLAT_TOK && !(fenv && fenv[0] == '0');
        // counted_df (filter / tombstones / OC_SHARD_COUNT_DF): no token has a host-known idf, so nothing is shared or dense
        // and every hot term arrives as a long posting list — the accumulator kernel walks those at ~10 instructions per
        // posting, the register-folded scorers would fold each posting's row separately
        const bool use3 = can_flat && !thr && !omc && !counted_df && !bp_in.matched_bits && !(t3e && t3e[0] == '0');
        Bm25Params bp = bp_in;
        // OC_BM25_ORDER=1: deal the items of the dense-token queries first and the list-only queries last (a lighter
        // ragged end of the persistent schedule); measured 1-2 % SLOWER on both bench shapes (the tile-major order of
        // ALL queries keeps the posting ranges of a tile together in L2), so the natural order is the default
        const char *oenv = getenv("OC_BM25_ORDER");
        if (!use3 || !(oenv && oenv[0] == '1')) bp.perm = nullptr;
        if (can_flat) {
            const uint64_t n_it = uint64_t(bp.n_tiles) * bp.n_queries * BM25_FLAT_TOK;
            OCTRY(c->flat_desc.ensure(n_it * sizeof(ItemTok)));
            bm25_flatten_kernel<<<(unsigned)((n_it + 255) / 256), 256, 0, st>>>(bp, c->flat_desc.as<ItemTok>());
            launched(c);
            CU(cudaGetLastError());
            flat = c->flat_desc.as<ItemTok>();
        }
        if (use3) {
            // plain queries: the register-folded scorer (no accumulator arrays)
            const size_t smem3 = bm25_tile3_smem_bytes(bp.cap);
            if (smem_cfg_needed(c->device, (const void *)bm25_tile3_kernel, smem3))
                CU(cudaFuncSetAttribute(bm25_tile3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem3));
            static std::mutex occ3_mu;
            static std::map<std::pair<int, size_t>, int> occ3;
            int per_sm = 1;
            {
                std::lock_guard<std::mutex> g(occ3_mu);
                auto it = occ3.find(std::make_pair(c->device, smem3));
                if (it == occ3.end()) {
                    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, bm25_tile3_kernel, BM25_THREADS, smem3));
                    occ3[std::make_pair(c->device, smem3)] = per_sm;
                } else per_sm = it->second;
            }
            const uint64_t items = uint64_t(bp.n_tiles) * bp.n_queries;
            const uint32_t g3 = (uint32_t)std::min<uint64_t>(items, uint64_t(std::max(per_sm, 1)) * c->prop.multiProcessorCount);
            const char *seed_env = getenv("OC_BM25_SEED");
            if (bp.n_keep <= 32 && bp.n_tiles > 1 && !(seed_env && seed_env[0] == '0')) {   // warm start of the candidate thresholds
                bm25_seed_kernel<<<(bp.n_queries * 32 + 255) / 256, 256, 0, st>>>(bp);
                launched(c);
            }
            const char *wenv = getenv("OC_BM25_WARP");
            if (bp.n_keep <= 32 && !(wenv && wenv[0] == '0')) {   // a warp per item: no block barriers
                const size_t smemw = size_t(BW_WARPS) * sizeof(WarpScratch);
                if (smem_cfg_needed(c->device, (const void *)bm25_warp_kernel, smemw))
                    CU(cudaFuncSetAttribute(bm25_warp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemw));
                static std::mutex occw_mu;
                static std::map<int, int> occw;
                int pw = 1;
                {
                    std::lock_guard<std::mutex> g(occw_mu);
                    auto it = occw.find(c->device);
                    if (it == occw.end()) {
                        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&pw, bm25_warp_kernel, BW_WARPS * 32, smemw));
                        occw[c->device] = pw;
                    } else pw = it->second;
                }
                const uint32_t gw = (uint32_t)std::min<uint64_t>((items + BW_WARPS - 1) / BW_WARPS, uint64_t(std::max(pw, 1)) * c->prop.multiProcessorCount);
                bm25_warp_kernel<<<gw, BW_WARPS * 32, smemw, st>>>(bp, flat, counter);
                launched(c);
                CU(cudaGetLastError());
                return OC_OK;
            }
            bm25_tile3_kernel<<<g3, BM25_THREADS, smem3, st>>>(bp, flat, counter);
            launched(c);
            CU(cudaGetLastError());
            return OC_OK;
        }
        const size_t smem = bm25_tile2_smem_bytes(thr, omc, bp.cap);
        const int sel = (thr ? 2 : 0) | (omc ? 1 : 0);
        switch (sel) {
            case 0: return launch_tile2_t<false, false>(c, bp, smem, st, flat, counter);
            case 1: return launch_tile2_t<false, true>(c, bp, smem, st, flat, counter);
            case 2: return launch_tile2_t<true, false>(c, bp, smem, st, flat, counter);
            default: return launch_tile2_t<true, true>(c, bp, smem, st, flat, counter);
        }
    }
    Bm25Params bp = bp_in;
    bp.perm = nullptr;
    const size_t smem = bm25_smem_bytes(multi, thr, omc, bp.cap);
    const int sel = (multi ? 4 : 0) | (thr ? 2 : 0) | (omc ? 1 : 0);
    switch (sel) {
        case 0: return launch_tile_t<false, false, false>(c, bp, grid, smem, st);
        case 1: return launch_tile_t<false, false, true>(c, bp, grid, smem, st);
        case 2: return launch_tile_t<false, true, false>(c, bp, grid, smem, st);
        case 3: return launch_tile_t<false, true, true>(c, bp, grid, smem, st);
        case 4: return launch_tile_t<true, false, false>(c, bp, grid, smem, st);
        case 5: return launch_tile_t<true, false, true>(c, bp, grid, smem, st);
        case 6: return launch_tile_t<true, true, false>(c, bp, grid, smem, st);
        default: return launch_tile_t<true, true, true>(c, bp, grid, smem, st);
    }
}

#include "shard.cuh"
#include "batcher.h"

struct FacetJob {   // oc_search_facets: count, per query, the matched documents of each requested variant
    oc_facets *fc;
    const oc_facet_req *reqs;
    uint32_t n_reqs;
    uint64_t *out_counts;   // [B][n_reqs]
};
static int run_facets(oc_ctx *c, const FacetJob &fj, uint32_t B, bool has_ft, bool has_v, const StrSnap *S, uint32_t n_tiles,
                      uint32_t vlimit);
struct SortJob {    // oc_search_sorted: replace the top-n by the first limit+offset score-map keys in a field's order
    oc_sort *st;
    uint32_t field;
    bool descending;
    int form;           // SORT_FORM_* (OC_SORT_FORM)
    double *out_keys;   // NULL or [B][limit]
};
static int run_sort(oc_ctx *c, const SortJob &sj, const oc_search_params *p, uint32_t B, bool has_ft, bool has_v, const StrSnap *S,
                    uint32_t n_tiles, uint32_t vlimit, uint32_t n_keep, const FuseParams &fp, const Bm25Params &bp, const uint32_t *row_ok);

static int search_impl(oc_ctx *c, oc_emb *emb, oc_str *str, const oc_search_params *p, uint64_t *out_doc_ids,
                       float *out_scores, uint32_t *out_n, uint64_t *out_count, const FacetJob *fj, const SortJob *sj) {
    if (!c || !p || !out_doc_ids || !out_scores || !out_n || !out_count) return fail(OC_ERR_INVALID, "NULL argument");
    const uint32_t B = p->n_queries;
    if (B == 0) return OC_OK;
    const bool has_v = p->mode == OC_MODE_VECTOR || p->mode == OC_MODE_HYBRID;
    const bool has_ft = p->mode == OC_MODE_FULLTEXT || p->mode == OC_MODE_HYBRID;
    if (!has_v && !has_ft) return fail(OC_ERR_INVALID, "unknown mode %d", p->mode);
    if (has_v && (!emb || !p->q_vecs)) return fail(OC_ERR_INVALID, "vector/hybrid mode needs emb and q_vecs");
    if (has_ft && (!str || !p->q_token_offsets)) return fail(OC_ERR_INVALID, "fulltext/hybrid mode needs str and tokens");
    if (emb && emb->ctx != c) return fail(OC_ERR_INVALID, "emb belongs to another ctx");
    if (str && str->ctx != c) return fail(OC_ERR_INVALID, "str belongs to another ctx");
    if (p->limit == 0) return fail(OC_ERR_INVALID, "limit must be >= 1");
    const uint64_t n_keep64 = uint64_t(p->limit) + p->offset;
    if (n_keep64 > OC_MAX_TOPK) return fail(OC_ERR_UNSUPPORTED, "limit+offset %llu > %u", (unsigned long long)n_keep64, OC_MAX_TOPK);
    const uint32_t n_keep = (uint32_t)n_keep64;
    // limit_hint = limit, NOT limit+offset (search.rs:330-336); vector_limit lets a multi-index caller keep that depth
    const uint32_t vlimit = p->vector_limit ? p->vector_limit : p->limit;
    if (vlimit > OC_MAX_TOPK) return fail(OC_ERR_UNSUPPORTED, "vector_limit %u > %u", vlimit, OC_MAX_TOPK);
    if (p->sharded && !c->comm.ready()) return fail(OC_ERR_COMM, "sharded search without oc_comm_init");

    // the published snapshot of the string store: grabbed once, immutable for the whole call (a commit may
    // publish the next version meanwhile); declared before the lock so a last reference dies outside it
    std::shared_ptr<StrSnap> snap = str ? str_snapshot(str) : nullptr;
    StrSnap *S = snap.get();
    std::lock_guard<std::mutex> g(c->mu);
    CU(cudaSetDevice(c->device));
    begin_call(c);

    // staged segments go in one copy per contiguous run; pinned caller buffers are DMA'd directly
    auto upload = [&](const Packer &pk, HostBuf &hb, DevBuf &db, cudaStream_t st) -> int {
        OCTRY(hb.ensure(pk.total + 256));
        OCTRY(db.ensure(pk.total + 256));
        pk.fill(hb.p);
        size_t run0 = 0;
        for (size_t i = 0; i <= pk.segs.size(); i++) {
            const bool brk = i == pk.segs.size() || pk.segs[i].direct;
            if (brk) {
                const size_t end = i == pk.segs.size() ? pk.total : pk.segs[i].off;
                if (end > run0) CU(cudaMemcpyAsync(db.as<uint8_t>() + run0, hb.as<uint8_t>() + run0, end - run0, cudaMemcpyHostToDevice, st));
                if (i < pk.segs.size()) {
                    CU(cudaMemcpyAsync(db.as<uint8_t>() + pk.segs[i].off, pk.segs[i].src, pk.segs[i].bytes, cudaMemcpyHostToDevice, st));
                    run0 = pk.segs[i].off + pk.segs[i].bytes;
                }
            }
        }
        return OC_OK;
    };
    // ------------------------------------------------------------ vector stage first: the query vectors
    // (+ filter) go up alone and the matrix sweep starts; the host-side descriptor work below overlaps it
    if (p->filter && p->filter->ctx != c) return fail(OC_ERR_INVALID, "filter belongs to another ctx");
    const bool filter_h = !p->filter && p->filter_bits != nullptr;        // host bitmap: uploaded with this call
    const bool filter = filter_h || p->filter != nullptr;
    const uint64_t filter_nbits = p->filter ? p->filter->nbits : p->filter_nbits;
    const size_t fwords = filter_h ? (p->filter_nbits + 63) / 64 : 0;
    const uint64_t *filter_dev = p->filter ? p->filter->bits : nullptr;
    size_t h2d_early = 0;
    if (has_v) {
        Packer pk0;
        const size_t o_qv = pk0.add(p->q_vecs, size_t(B) * emb->dim * 4, is_pinned_host(p->q_vecs));
        const size_t o_flt = filter_h ? pk0.add(p->filter_bits, fwords * 8) : 0;
        CU(cudaEventRecord(c->ev[EV_START], c->stream));
        OCTRY(upload(pk0, c->h_in0, c->in_blob0, c->stream));
        CU(cudaEventRecord(c->ev[EV_H2D], c->stream));
        h2d_early = pk0.total;
        if (filter_h) filter_dev = reinterpret_cast<const uint64_t *>(c->in_blob0.as<uint8_t>() + o_flt);
        OCTRY(run_vector_stage(c, emb, reinterpret_cast<const float *>(c->in_blob0.as<uint8_t>() + o_qv), B, vlimit, p->similarity,
                               filter_dev, filter_nbits));
    }

    // ------------------------------------------------------------ host: descriptors
    const bool multi_rank = p->sharded && c->comm.world > 1;
    // sharded: every rank must take the same df decisions (they drive a collective), so the
    // tombstone state is the caller's global flag (OC_SHARD_TOMBSTONES), not this shard's
    const bool tombs_local = has_ft && S->n_deleted > 0;
    if (multi_rank && tombs_local && !(p->sharded & OC_SHARD_TOMBSTONES))
        return fail(OC_ERR_INVALID, "sharded search: this shard holds tombstones, set OC_SHARD_TOMBSTONES on every rank");
    const bool tombs = has_ft && (multi_rank ? (p->sharded & OC_SHARD_TOMBSTONES) != 0 : tombs_local);
    const uint32_t n_tiles = has_ft ? (uint32_t)((S->n_rows + BM25_TILE - 1) / BM25_TILE) : 0;
    std::vector<TermDesc> terms;
    std::vector<uint32_t> term_token;
    std::vector<uint64_t> term_key;     // (field << 32 | term id) of each expanded term
    std::vector<TokenDesc> tokens;
    std::vector<QueryDesc> queries;
    std::vector<uint8_t> tok_need_df;
    std::vector<PreDesc> pre_descs;
    std::vector<uint2> pre_items;
    bool any_multi = false, need_df = false, derived_now = false;
    uint32_t max_tokens = 0;    // tokens of the longest query of the batch
    uint64_t dense_bytes = 0;   // dense contribution arrays of this batch (zeroed before the precompute kernel fills them)
    // sharded: df comes from the replicated per-term table, or — OC_SHARD_COUNT_DF on every rank, e.g. after a
    // commit dropped the table — from counting + all-reduce.  A shard-local list length is never a corpus df.
    const bool count_df = multi_rank && (p->sharded & OC_SHARD_COUNT_DF) != 0;
    bool df_local_only = false;
    uint64_t postings_walked = 0;
    const bool thr = p->threshold >= 0.0f;
    if (has_ft) {
        for (auto &f : S->fields)   // streamed posting format depends on (avg_field_len, b): derive once
            if (f.n_post && f.b_cached != p->bm25_b) {
                bm25_derive_postings_kernel<<<(unsigned)((f.n_post + 255) / 256), 256, 0, c->stream>>>(f.raw, f.n_post, f.avg_len, p->bm25_b, f.post);
                launched(c);
                CU(cudaGetLastError());
                f.b_cached = p->bm25_b;
                derived_now = true;   // queued on the main stream: this call keeps the BM25 prologue there too
            }
        const float N = (float)S->document_count;  // token_score.rs:221
        queries.resize(B);
        for (uint32_t q = 0; q < B; q++) {
            const uint32_t t0 = p->q_token_offsets[q], t1 = p->q_token_offsets[q + 1];
            QueryDesc qd{};
            qd.token_begin = (uint32_t)tokens.size();
            const uint32_t ntok = t1 - t0;
            max_tokens = std::max(max_tokens, ntok);
            qd.required = thr ? (uint32_t)floorf((float)ntok * p->threshold) : 0;  // token_score.rs:211-218
            qd.flags = thr ? QF_THRESHOLD : 0;
            for (uint32_t t = t0; t < t1; t++) {
                TokenDesc tk{};
                tk.term_begin = (uint32_t)terms.size();
                tk.bit = 1u << ((t - t0) & 31u);
                uint64_t df_known = 0;
                for (uint32_t e = p->token_term_offsets[t]; e < p->token_term_offsets[t + 1]; e++) {
                    const uint32_t fi = p->term_field[e], ti = p->term_id[e];
                    if (fi >= S->fields.size()) return fail(OC_ERR_INVALID, "term field %u out of range", fi);
                    const StrField &f = S->fields[fi];
                    if (ti >= f.n_terms) continue;  // unknown term: no postings
                    TermDesc td{};
                    td.ptr = f.post + f.term_offsets[ti];
                    td.len = (uint32_t)(f.term_offsets[ti + 1] - f.term_offsets[ti]);
                    td.weight = p->term_weight ? p->term_weight[e] : 1.0f;
                    td.avg_len = f.avg_len;
                    df_known = f.global_df.empty() ? td.len : f.global_df[ti];
                    if (multi_rank && f.global_df.empty()) df_local_only = true;
                    postings_walked += td.len;
                    term_key.push_back((uint64_t(fi) << 32) | ti);
                    terms.push_back(td);
                    term_token.push_back((uint32_t)tokens.size());
                }
                tk.term_end = (uint32_t)terms.size();
                const uint32_t nt = tk.term_end - tk.term_begin;
                uint8_t need = 0;
                if (nt == 1 && !filter && !tombs && !count_df) tk.idf = host_idf(N, std::max<uint64_t>(1, df_known));
                else if (nt == 0) tk.idf = host_idf(N, 1);
                else { need = 1; need_df = true; tk.idf = 0.f; }
                if (nt != 1) { any_multi = any_multi || nt > 1; }
                tokens.push_back(tk);
                tok_need_df.push_back(need);
            }
            qd.token_end = (uint32_t)tokens.size();
            queries[q] = qd;
        }
        if (df_local_only && !count_df)
            return fail(OC_ERR_INVALID, "sharded search: a field of this shard has no corpus-wide df table (dropped by a commit?): "
                                        "reload it or pass OC_SHARD_COUNT_DF on every rank");
        // ---- batch-level sharing of per-posting contributions (single-term tokens with a host-known idf)
        {
            struct U { uint32_t first_e; uint32_t uses; };
            struct K128 { uint64_t a, b; };            // (field, term) | (weight bits, idf bits)
            size_t cap_t = 64;
            while (cap_t < tokens.size() * 2) cap_t <<= 1;
            std::vector<K128> tab_k(cap_t);
            std::vector<uint32_t> tab_v(cap_t, 0xffffffffu);   // open addressing, linear probing
            std::vector<U> uniq;
            std::vector<uint32_t> e_to_u(terms.size(), 0xffffffffu);
            uint64_t walked = 0, distinct = 0;
            for (size_t t = 0; t < tokens.size(); t++) {
                const TokenDesc &tk = tokens[t];
                if (tk.term_end - tk.term_begin != 1 || tok_need_df[t]) continue;
                const uint32_t e = tk.term_begin;
                if (terms[e].len < 64) continue;
                uint32_t wb, ib;
                memcpy(&wb, &terms[e].weight, 4); memcpy(&ib, &tk.idf, 4);
                const K128 key{term_key[e], (uint64_t(wb) << 32) | ib};
                uint64_t h = (key.a * 0x9E3779B97F4A7C15ull) ^ (key.b * 0xC2B2AE3D27D4EB4Full);
                size_t slot = (h ^ (h >> 29)) & (cap_t - 1);
                while (tab_v[slot] != 0xffffffffu && !(tab_k[slot].a == key.a && tab_k[slot].b == key.b)) slot = (slot + 1) & (cap_t - 1);
                if (tab_v[slot] == 0xffffffffu) {
                    tab_k[slot] = key; tab_v[slot] = (uint32_t)uniq.size();
                    uniq.push_back({e, 0}); distinct += terms[e].len;
                }
                uniq[tab_v[slot]].uses++;
                e_to_u[e] = tab_v[slot];
                walked += terms[e].len;
            }
            const char *share_env = getenv("OC_BM25_SHARE");   // "off" / "force": A/B testing of the sharing pass
            const bool share_off = share_env && !strcmp(share_env, "off"), share_force = share_env && !strcmp(share_env, "force");
            // hot terms (a posting in at least every 16th row) go DENSE: their contributions are scattered once per batch
            // into a float[rows] array and every (query, tile) item adds 8192 floats with 128-bit loads instead of
            // walking ~thousands of postings (posting-centred kernel only: every token of the batch has <= 1 term)
            const char *dense_env = getenv("OC_BM25_DENSE");
            const char *t2_env = getenv("OC_BM25_TILE2");
            const bool dense_on = !any_multi && !(dense_env && dense_env[0] == '0') && !share_off && !(t2_env && t2_env[0] == '0');
            const uint64_t rows_pad = uint64_t(n_tiles) * BM25_TILE;
            const uint64_t dense_min = std::max<uint64_t>(512, S->n_rows / 16);
            std::vector<uint8_t> u_dense(uniq.size(), 0);
            uint64_t n_dense = 0;
            if (dense_on)
                for (size_t u = 0; u < uniq.size(); u++)
                    if (terms[uniq[u].first_e].len >= dense_min && (n_dense + 1) * rows_pad * 4 <= (size_t(8) << 30)) { u_dense[u] = 1; n_dense++; }
            uint64_t walked_l = 0, distinct_l = 0;   // what is left for the list form
            for (size_t e = 0; e < terms.size(); e++)
                if (e_to_u[e] != 0xffffffffu && !u_dense[e_to_u[e]]) walked_l += terms[e].len;
            for (size_t u = 0; u < uniq.size(); u++) if (!u_dense[u]) distinct_l += terms[uniq[u].first_e].len;
            const bool lists = distinct_l && !share_off && (share_force || (walked_l >= 2 * distinct_l && walked_l >= (64u << 20))) &&
                               distinct_l * 8 <= (size_t(6) << 30);
            if (lists || n_dense) {
                if (lists) OCTRY(c->pre_post.ensure(distinct_l * 8 + 64));
                if (n_dense) OCTRY(c->dense_buf.ensure(n_dense * rows_pad * 4));
                dense_bytes = n_dense * rows_pad * 4;
                uint64_t off = 0, doff = 0;
                std::vector<uint64_t> u_off(uniq.size());
                std::vector<uint8_t> u_used(uniq.size(), 0);
                for (size_t u = 0; u < uniq.size(); u++) {
                    if (!u_dense[u] && !lists) continue;
                    u_used[u] = 1;
                    const TermDesc &td = terms[uniq[u].first_e];
                    PreDesc pd{};
                    pd.src = td.ptr; pd.len = td.len; pd.weight = td.weight;
                    pd.idf = tokens[term_token[uniq[u].first_e]].idf;
                    if (u_dense[u]) { u_off[u] = doff; pd.dense = c->dense_buf.as<float>() + doff; doff += rows_pad; }
                    else { u_off[u] = off; pd.dst = c->pre_post.as<Posting>() + off; off += td.len; }
                    const uint32_t pi = (uint32_t)pre_descs.size();
                    pre_descs.push_back(pd);
                    for (uint32_t ch = 0; ch * PRE_CHUNK < td.len; ch++) pre_items.push_back(make_uint2(pi, ch));
                }
                for (size_t e = 0; e < terms.size(); e++) {
                    const uint32_t u = e_to_u[e];
                    if (u == 0xffffffffu || !u_used[u]) continue;
                    if (u_dense[u]) { terms[e].ptr = reinterpret_cast<const Posting *>(c->dense_buf.as<float>() + u_off[u]); terms[e].flags |= TD_DENSE; }
                    else { terms[e].ptr = c->pre_post.as<Posting>() + u_off[u]; terms[e].flags |= TD_PRE; }
                }
            }
        }
    }
    // OMC rows for the tile kernel (string rows, ascending)
    std::vector<uint32_t> omc_rows; std::vector<float> omc_row_mult;
    const uint32_t n_omc = (uint32_t)p->n_omc;
    if (n_omc && (!p->omc_doc_ids || !p->omc_mult)) return fail(OC_ERR_INVALID, "omc arrays are NULL");
    if (n_omc && has_ft) {
        for (uint32_t i = 0; i < n_omc; i++) {
            if (i && p->omc_doc_ids[i] <= p->omc_doc_ids[i - 1]) return fail(OC_ERR_INVALID, "omc_doc_ids must be ascending");
            uint64_t r;
            if (S->row_doc_host.empty()) { r = p->omc_doc_ids[i]; if (r >= S->n_rows) continue; }
            else {
                auto it = std::lower_bound(S->row_doc_host.begin(), S->row_doc_host.end(), p->omc_doc_ids[i]);
                if (it == S->row_doc_host.end() || *it != p->omc_doc_ids[i]) continue;
                r = uint64_t(it - S->row_doc_host.begin());
            }
            omc_rows.push_back((uint32_t)r); omc_row_mult.push_back(p->omc_mult[i]);
        }
    }
    const bool omc_tile = !omc_rows.empty();

    // ------------------------------------------------------------ H2D: descriptors in one packed blob
    Packer pk;
    const size_t o_flt = (filter_h && !has_v) ? pk.add(p->filter_bits, fwords * 8) : 0;
    const size_t o_terms = has_ft ? pk.add(terms.data(), terms.size() * sizeof(TermDesc)) : 0;
    const size_t o_tokens = has_ft ? pk.add(tokens.data(), tokens.size() * sizeof(TokenDesc)) : 0;
    const size_t o_ttok = has_ft ? pk.add(term_token.data(), term_token.size() * 4) : 0;
    const size_t o_pre = pre_descs.empty() ? 0 : pk.add(pre_descs.data(), pre_descs.size() * sizeof(PreDesc));
    const size_t o_pitems = pre_items.empty() ? 0 : pk.add(pre_items.data(), pre_items.size() * sizeof(uint2));
    const size_t o_queries = has_ft ? pk.add(queries.data(), queries.size() * sizeof(QueryDesc)) : 0;
    const size_t o_omcd = n_omc ? pk.add(p->omc_doc_ids, size_t(n_omc) * 8) : 0;
    const size_t o_omcm = n_omc ? pk.add(p->omc_mult, size_t(n_omc) * 4) : 0;
    const size_t o_omcr = omc_tile ? pk.add(omc_rows.data(), omc_rows.size() * 4) : 0;
    const size_t o_omcrm = omc_tile ? pk.add(omc_row_mult.data(), omc_row_mult.size() * 4) : 0;
    // item order of the register-folded scorers (Bm25Params::perm): queries by their number of dense tokens, descending
    std::vector<uint32_t> q_perm;
    uint32_t cls_nq[BM25_CLASSES] = {0, 0, 0, 0, 0};
    if (has_ft && !any_multi && max_tokens <= BM25_FLAT_TOK) {
        std::vector<uint8_t> nd_q(B, 0);
        for (uint32_t q = 0; q < B; q++) {
            uint32_t nd = 0;
            for (uint32_t t = queries[q].token_begin; t < queries[q].token_end; t++)
                if (tokens[t].term_end > tokens[t].term_begin && (terms[tokens[t].term_begin].flags & TD_DENSE) && terms[tokens[t].term_begin].len) nd++;
            nd_q[q] = (uint8_t)std::min<uint32_t>(nd, BM25_CLASSES - 1);
        }
        // (used with OC_BM25_ORDER=1 only.)  TWO classes: every query with a dense token (one tile-major pass over the dense
        // arrays: one class per dense-token count re-streamed those arrays once per class and cost the 10M-document
        // workload 20 %), then the list-only queries, whose items are cheap and touch no dense array.  Inside the first
        // class the queries are sorted by their number of dense tokens, descending.
        auto cls_of = [&](uint32_t q) { return nd_q[q] ? 0u : BM25_CLASSES - 1; };
        for (uint32_t q = 0; q < B; q++) cls_nq[cls_of(q)]++;
        q_perm.resize(B);
        uint32_t at[BM25_CLASSES], acc = 0;
        for (uint32_t g = 0; g < BM25_CLASSES; g++) { at[g] = acc; acc += cls_nq[g]; }
        for (int nd = BM25_CLASSES - 1; nd >= 0; nd--)
            for (uint32_t q = 0; q < B; q++) if (nd_q[q] == nd) q_perm[at[cls_of(q)]++] = q;
    }
    const size_t o_perm = q_perm.empty() ? 0 : pk.add(q_perm.data(), q_perm.size() * 4);
    // hybrid: the descriptors, the shared-contribution precompute, the filter bitmap and the (term, tile) plan do
    // not depend on the vector results: they run on the side stream while the main stream sweeps the matrix
    // (OC_SIDE_STREAM=0 disables it: the step gets ~2.5 % longer, the sweep itself ~4 % shorter — A/B switch)
    const char *senv = getenv("OC_SIDE_STREAM");
    // (single-GPU only for now: the sharded path was measured and validated without it)
    const bool side = !(senv && senv[0] == '0') && has_v && has_ft && !need_df && !derived_now;
    if (!has_v) CU(cudaEventRecord(c->ev[EV_START], c->stream));
    if (c->side_dirty) { CU(cudaStreamSynchronize(c->side)); c->side_dirty = false; }   // leftover of a failed call
    if (side) { CU(cudaStreamWaitEvent(c->side, c->ev[EV_H2D], 0)); c->side_dirty = true; }   // the filter bitmap went up with the query vectors
    OCTRY(upload(pk, c->h_in, c->in_blob, side ? c->side : c->stream));
    if (!has_v) CU(cudaEventRecord(c->ev[EV_H2D], c->stream));   // hybrid/vector: this copy rides inside the device window
    c->timing.h2d_bytes = h2d_early + pk.total;
    uint8_t *din = c->in_blob.as<uint8_t>();
    if (filter_h && !has_v) filter_dev = reinterpret_cast<const uint64_t *>(din + o_flt);

    // ------------------------------------------------------------ fulltext stage + fusion (re-runnable)
    // arg-max selection (n_keep <= 32) needs no power-of-two buffer; the bitonic fallback does
    // (also >= BM25_SPARSE_MAX: the sparse finish of the posting-centred kernel pushes at most that many candidates)
    const uint32_t cap = n_keep <= 32 ? std::max<uint32_t>(n_keep + BM25_CHUNK, BM25_SPARSE_MAX) : next_pow2(std::max<uint32_t>(n_keep + BM25_CHUNK, BM25_SPARSE_MAX));
    Bm25Params bp{};
    float *min_hint_dev = nullptr;
    unsigned int *tile_counter = nullptr;
    const size_t o_doc = 0, o_sc = size_t(B) * p->limit * 8, o_n = o_sc + size_t(B) * p->limit * 4;
    const size_t o_cnt = (o_n + size_t(B) * 4 + 7) & ~size_t(7), o_min = o_cnt + size_t(B) * 8;
    const size_t o_gflag = o_min + size_t(B) * 4;                       // sharded: OR over the ranks of the per-query overflow flags
    const size_t out_bytes = o_gflag + ((size_t(B) + 3) & ~size_t(3));
    const size_t o_resc = out_bytes + ((size_t(B) + 3) & ~size_t(3));
    OCTRY(c->out_blob.ensure(out_bytes));
    OCTRY(c->h_out.ensure(o_resc + size_t(B) * 4));
    uint8_t *dout = c->out_blob.as<uint8_t>();
    FuseParams fp{};
    size_t fuse_smem = 0;
    bool did_comm = false;
    // The fulltext stage does not depend on the vector stage (the vector hits' fulltext scores are point lookups
    // afterwards): in hybrid mode it runs on the side stream, concurrently with the matrix sweep, and is joined
    // before the lookups and the fusion.  It runs ONCE per call; device_tail (lookups + fusion) is re-runnable.
    const uint32_t *row_ok = nullptr;
    auto bm25_stage = [&]() -> int {
        cudaStream_t ps = side ? c->side : c->stream;
        CU(cudaEventRecord(c->ev[EV_BM0], ps));
        const uint64_t ok_words = uint64_t(n_tiles) * (BM25_TILE / 32);
        if (filter || tombs) {
            OCTRY(c->row_ok.ensure(ok_words * 4));
            rows_ok_kernel<<<(unsigned)((ok_words + 255) / 256), 256, 0, ps>>>(
                S->row_doc, S->n_rows, tombs ? S->alive : nullptr, filter_dev, filter_nbits,
                c->row_ok.as<uint32_t>(), ok_words);
            launched(c);
            row_ok = c->row_ok.as<uint32_t>();
        }
        if (!pre_items.empty()) {
            if (dense_bytes) CU(cudaMemsetAsync(c->dense_buf.p, 0, dense_bytes, ps));
            bm25_precompute_kernel<<<(unsigned)pre_items.size(), 256, 0, ps>>>(
                reinterpret_cast<const PreDesc *>(din + o_pre), reinterpret_cast<const uint2 *>(din + o_pitems), p->bm25_k, row_ok);
            launched(c);
            CU(cudaGetLastError());
        }
        const size_t n_td = terms.size();
        OCTRY(c->seg.ensure((n_td * (size_t(n_tiles) + 1) + 1) * 4));
        if (n_td) {
            const uint64_t work = uint64_t(n_td) * (n_tiles + 1);
            bm25_plan_kernel<<<(unsigned)((work + 255) / 256), 256, 0, ps>>>(
                reinterpret_cast<const TermDesc *>(din + o_terms), (uint32_t)n_td, n_tiles, c->seg.as<uint32_t>());
            launched(c);
        }
        if (need_df) {   // (never on the side stream)
            // corpus_df by counting (token_score.rs:262-275), then idf on the host
            const size_t ntok = tokens.size();
            OCTRY(c->df_dev.ensure(ntok * 4));
            CU(cudaMemsetAsync(c->df_dev.p, 0, ntok * 4, c->stream));
            DfParams dp{};
            dp.terms = reinterpret_cast<const TermDesc *>(din + o_terms);
            dp.tokens = reinterpret_cast<const TokenDesc *>(din + o_tokens);
            dp.n_tokens = (uint32_t)ntok; dp.n_tiles = n_tiles; dp.seg = c->seg.as<uint32_t>();
            dp.row_ok_bits = row_ok; dp.df = c->df_dev.as<unsigned int>();
            if (n_tiles) {
                bm25_df_kernel<<<(unsigned)(uint64_t(n_tiles) * ntok), BM25_THREADS, 0, c->stream>>>(dp);
                launched(c);
            }
            if (multi_rank) {   // corpus df = sum of the shards' counts (disjoint documents)
                std::string err;
                if (!c->comm.all_reduce_sum_u32(c->df_dev.p, c->df_dev.p, ntok, c->stream, &err)) return fail(OC_ERR_COMM, "%s", err.c_str());
            }
            std::vector<uint32_t> dfh(ntok);
            CU(cudaMemcpyAsync(dfh.data(), c->df_dev.p, ntok * 4, cudaMemcpyDeviceToHost, c->stream));
            CU(cudaStreamSynchronize(c->stream));
            const float N = (float)S->document_count;
            for (size_t t = 0; t < ntok; t++)
                if (tok_need_df[t]) tokens[t].idf = host_idf(N, std::max<uint32_t>(1u, dfh[t]));
            CU(cudaMemcpyAsync(din + o_tokens, tokens.data(), ntok * sizeof(TokenDesc), cudaMemcpyHostToDevice, c->stream));
        }
        const size_t slots = size_t(B) * std::max<uint32_t>(n_tiles, 1);
        OCTRY(c->tau.ensure(size_t(B) * 16 + 16));   // [tau B x 8][min_hint B x 8][work counter]: one memset
        OCTRY(c->cand_key.ensure(slots * n_keep * 8));
        OCTRY(c->cand_ft.ensure(slots * n_keep * 4));
        OCTRY(c->cand_cnt.ensure(slots * 4));
        OCTRY(c->tile_cnt.ensure(slots * 4));
        OCTRY(c->tile_max.ensure(slots * 4));
        OCTRY(c->tile_min.ensure(slots * 4));
        min_hint_dev = reinterpret_cast<float *>(c->tau.as<uint8_t>() + size_t(B) * 8);
        tile_counter = reinterpret_cast<unsigned int *>(c->tau.as<uint8_t>() + size_t(B) * 16);
        CU(cudaMemsetAsync(c->tau.p, 0, size_t(B) * 16 + 16, ps));
        bp.terms = reinterpret_cast<const TermDesc *>(din + o_terms);
        bp.tokens = reinterpret_cast<const TokenDesc *>(din + o_tokens);
        bp.queries = reinterpret_cast<const QueryDesc *>(din + o_queries);
        bp.term_token = reinterpret_cast<const uint32_t *>(din + o_ttok);
        bp.seg = c->seg.as<uint32_t>();
        bp.n_queries = B; bp.n_tiles = n_tiles; bp.n_rows = S->n_rows;
        bp.k = p->bm25_k; bp.b = p->bm25_b;
        bp.row_ok_bits = row_ok;
        bp.omc_row = omc_tile ? reinterpret_cast<const uint32_t *>(din + o_omcr) : nullptr;
        bp.omc_mult = omc_tile ? reinterpret_cast<const float *>(din + o_omcrm) : nullptr;
        bp.n_omc = (uint32_t)omc_rows.size();
        bp.v_row = nullptr;            // the hybrid lookups are point lookups (bm25_point_kernel)
        bp.v_stride = vlimit;
        bp.v_ft = nullptr; bp.v_present = nullptr;
        bp.min_hint = min_hint_dev;
        bp.n_keep = n_keep; bp.cap = cap;
        bp.tau = c->tau.as<unsigned long long>();
        bp.cand_key = c->cand_key.as<uint64_t>(); bp.cand_ft = c->cand_ft.as<float>();
        bp.cand_cnt = c->cand_cnt.as<uint32_t>(); bp.tile_count = c->tile_cnt.as<uint32_t>();
        bp.tile_max = c->tile_max.as<float>(); bp.tile_min = c->tile_min.as<float>();
        bp.tile_first = 0;
        if (!q_perm.empty()) {
            bp.perm = reinterpret_cast<const uint32_t *>(din + o_perm);
            uint32_t off = 0, q0 = 0;
            for (uint32_t g = 0; g < BM25_CLASSES; g++) {
                bp.cls_off[g] = off; bp.cls_nq[g] = cls_nq[g]; bp.cls_q0[g] = q0;
                off += cls_nq[g] * n_tiles; q0 += cls_nq[g];
            }
        }
        if (fj || sj) {   // facets / sortBy: the tile kernels also emit the bitmap of matched rows (every (query, tile) item writes its 256 words)
            OCTRY(c->mbits.ensure(size_t(B) * std::max<uint32_t>(n_tiles, 1) * (BM25_TILE / 32) * 4));
            bp.matched_bits = c->mbits.as<uint32_t>();
        }
        if (n_tiles) OCTRY(launch_tile(c, bp, n_tiles * B, any_multi, thr, omc_tile, ps, max_tokens, tile_counter, need_df));
        CU(cudaEventRecord(c->ev[EV_BM1], ps));
        c->timing.bm25_postings = postings_walked;
        if (side) {   // join: the lookups and the fusion need the vector hits (main stream) and the tiles (side stream)
            CU(cudaEventRecord(c->ev_side, c->side));
            CU(cudaStreamWaitEvent(c->stream, c->ev_side, 0));
            c->side_dirty = false;
        }
        return OC_OK;
    };
    if (has_ft) OCTRY(bm25_stage());

    auto device_tail = [&]() -> int {
    if (has_ft && has_v) {
        // hybrid: vector hits -> string rows -> their fulltext scores (point lookups)
        OCTRY(c->v_srow.ensure(size_t(B) * vlimit * 4));
        OCTRY(c->v_ft.ensure(size_t(B) * vlimit * 4));
        OCTRY(c->v_present.ensure(size_t(B) * vlimit));
        map_docs_to_rows_kernel<<<(B * vlimit + 255) / 256, 256, 0, c->stream>>>(
            c->v_doc.as<uint64_t>(), c->v_cnt.as<uint32_t>(), vlimit, B, S->row_doc, S->n_rows, c->v_srow.as<uint32_t>());
        launched(c);
        PointParams pp{};
        pp.terms = bp.terms; pp.tokens = bp.tokens; pp.queries = bp.queries;
        pp.n_queries = B; pp.v_stride = vlimit; pp.v_row = c->v_srow.as<uint32_t>(); pp.row_ok_bits = row_ok;
        pp.k = p->bm25_k; pp.threshold = thr ? 1 : 0;
        pp.v_ft = c->v_ft.as<float>(); pp.v_present = c->v_present.as<uint8_t>();
        bm25_point_kernel<<<(B * vlimit * 32 + 255) / 256, 256, 0, c->stream>>>(pp);
        launched(c);
        CU(cudaGetLastError());
    }

    // ------------------------------------------------------------ fusion + top-n (+ shard exchange)
    fp = FuseParams{};
    fp.mode = p->mode; fp.n_tiles = n_tiles; fp.n_keep = n_keep; fp.limit = p->limit; fp.offset = p->offset;
    {   // smallest power-of-two key buffer that takes the candidates in one round (sort cost ~ capb log^2 capb)
        const uint64_t total = (has_ft ? uint64_t(n_tiles) * n_keep : 0) + (has_v ? vlimit : 0);
        // up to 16 K keys (128 KB) stay in shared memory and go through one radix select; the streaming bitonic path behind
        // it cost 0.44 ms per batch on the 10M-document fulltext workload (1221 tiles x 10 candidate slots per query:
        // profiles/r02_ncu_fuse_t1.md)
        fp.capb = next_pow2((uint32_t)std::min<uint64_t>(16384, std::max<uint64_t>(total, 2 * n_keep)));
        fp.capb = std::max<uint32_t>(fp.capb, std::max<uint32_t>(64, next_pow2(2 * n_keep)));
    }
    if (has_ft) {
        fp.cand_key = bp.cand_key; fp.cand_ft = bp.cand_ft; fp.cand_cnt = bp.cand_cnt; fp.tile_count = bp.tile_count;
        fp.tile_max = bp.tile_max; fp.tile_min = bp.tile_min; fp.str_row_doc_ids = S->row_doc;
    }
    if (has_v) {
        fp.v_doc = c->v_doc.as<uint64_t>(); fp.v_score = c->v_score.as<float>(); fp.v_count = c->v_cnt.as<uint32_t>();
        fp.v_row = has_ft ? c->v_srow.as<uint32_t>() : nullptr;
        fp.v_ft = c->v_ft.as<float>(); fp.v_present = c->v_present.as<uint8_t>();
    }
    fp.v_stride = vlimit;
    fp.omc_doc = n_omc ? reinterpret_cast<const uint64_t *>(din + o_omcd) : nullptr;
    fp.omc_mult = n_omc ? reinterpret_cast<const float *>(din + o_omcm) : nullptr;
    fp.n_omc = n_omc;
    fp.out_doc = reinterpret_cast<uint64_t *>(dout + o_doc); fp.out_score = reinterpret_cast<float *>(dout + o_sc);
    fp.out_n = reinterpret_cast<uint32_t *>(dout + o_n); fp.out_count = reinterpret_cast<unsigned long long *>(dout + o_cnt);
    fp.out_min = reinterpret_cast<float *>(dout + o_min);
    if (sj) {
        OCTRY(c->sort_max.ensure(size_t(B) * 4));
        fp.out_max = c->sort_max.as<float>();
    }
    fuse_smem = size_t(fp.capb) * 8 + size_t(std::max<uint32_t>(32, next_pow2(n_keep))) * 8 + size_t(vlimit) * 8 + 64;
    if (smem_cfg_needed(c->device, (const void *)fuse_topk_kernel, fuse_smem))
        CU(cudaFuncSetAttribute(fuse_topk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fuse_smem));

    if (p->sharded && c->comm.world > 1) {
        CU(cudaEventRecord(c->ev[EV_FUSE0], c->stream));
        OCTRY(run_sharded_merge(c, p, fp, has_ft ? (uint32_t)S->n_rows : 0, has_v ? (uint32_t)emb->n_rows : 0, B,
                                (has_v && c->gemm_pending) ? c->g_flag.as<uint8_t>() : nullptr, dout + o_gflag));
        CU(cudaEventRecord(c->ev[EV_FUSE1], c->stream));
        did_comm = true;
    } else {
        CU(cudaEventRecord(c->ev[EV_FUSE0], c->stream));
        fuse_topk_kernel<<<B, 256, fuse_smem, c->stream>>>(fp);
        launched(c);
        CU(cudaGetLastError());
        CU(cudaEventRecord(c->ev[EV_FUSE1], c->stream));
    }
    return OC_OK;
    };   // device_tail
    OCTRY(device_tail());
    CU(cudaEventRecord(c->ev[EV_DEV], c->stream));
    uint8_t *h = c->h_out.as<uint8_t>();
    CU(cudaMemcpyAsync(h, dout, out_bytes, cudaMemcpyDeviceToHost, c->stream));
    if (c->gemm_pending) {
        CU(cudaMemcpyAsync(h + out_bytes, c->g_flag.p, B, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaMemcpyAsync(h + o_resc, c->g_resc.p, size_t(B) * 4, cudaMemcpyDeviceToHost, c->stream));
    }
    CU(cudaEventRecord(c->ev[EV_D2H], c->stream));
    CU(cudaStreamSynchronize(c->stream));
    {   // tensor-core scan: re-run the (rare) queries whose candidate buffers overflowed
        // sharded: every rank must enter the collective the same number of times, so the decision to re-run is
        // taken on the flags all ranks exchanged inside the shard records (no host sync before the collective),
        // by every rank — also one whose own shard was served by the exact sweep
        bool rerun = false;
        if (did_comm && has_v) for (uint32_t q = 0; q < B; q++) rerun = rerun || h[o_gflag + q] != 0;
        uint32_t redone = 0;
        if (c->gemm_pending || rerun) CU(cudaEventRecord(c->ev[EV_RR0], c->stream));
        if (c->gemm_pending) {
            uint64_t resc = 0;
            for (uint32_t q = 0; q < B; q++) resc += reinterpret_cast<const uint32_t *>(h + o_resc)[q];
            c->timing.scan_rescored = (uint32_t)(resc / B);
            OCTRY(fix_unproven(c, emb, h + out_bytes, B, vlimit, p->similarity, &redone));
        }
        if (redone || rerun) {
            c->gemm_pending = false;
            OCTRY(device_tail());
            CU(cudaMemcpyAsync(h, dout, out_bytes, cudaMemcpyDeviceToHost, c->stream));
            CU(cudaEventRecord(c->ev[EV_RR1], c->stream));
            c->rerun_timed = true;
            CU(cudaStreamSynchronize(c->stream));
        }
    }

    // rank-proxy validation: with OMC multipliers the tile ranking assumed min == min_hint (0);
    // a negative global min changes the order of (ft - min) * omc -> rerun with the real min.
    if (!did_comm && p->mode == OC_MODE_HYBRID && omc_tile && n_tiles) {
        const float *mins = reinterpret_cast<const float *>(h + o_min);
        bool redo = false;
        for (uint32_t q = 0; q < B; q++) redo = redo || mins[q] < 0.f;
        if (redo) {
            CU(cudaMemcpyAsync(min_hint_dev, mins, size_t(B) * 4, cudaMemcpyHostToDevice, c->stream));
            CU(cudaMemsetAsync(c->tau.p, 0, size_t(B) * 8, c->stream));
            CU(cudaMemsetAsync(tile_counter, 0, 8, c->stream));
            OCTRY(launch_tile(c, bp, n_tiles * B, any_multi, thr, omc_tile, c->stream, max_tokens, tile_counter, need_df));
            fuse_topk_kernel<<<B, 256, fuse_smem, c->stream>>>(fp);
            launched(c);
            CU(cudaMemcpyAsync(c->h_out.p, dout, out_bytes, cudaMemcpyDeviceToHost, c->stream));
            CU(cudaStreamSynchronize(c->stream));
        }
    }
    if (fj) OCTRY(run_facets(c, *fj, B, has_ft, has_v, S, n_tiles, vlimit));
    float sort_ms = 0.f;
    if (sj) {   // after every re-run: the bitmap, the count and K4's extrema are final
        CU(cudaEventRecord(c->ev[EV_SORT0], c->stream));
        OCTRY(run_sort(c, *sj, p, B, has_ft, has_v, S, n_tiles, vlimit, n_keep, fp, bp, row_ok));
        CU(cudaEventRecord(c->ev[EV_SORT1], c->stream));
        CU(cudaMemcpyAsync(h, dout, out_bytes, cudaMemcpyDeviceToHost, c->stream));
        if (sj->out_keys) CU(cudaMemcpyAsync(sj->out_keys, c->sort_keys.p, size_t(B) * p->limit * 8, cudaMemcpyDeviceToHost, c->stream));
        c->sort_forms.resize(B);
        CU(cudaMemcpyAsync(c->sort_forms.data(), c->sort_form.p, B, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        CU(cudaEventElapsedTime(&sort_ms, c->ev[EV_SORT0], c->ev[EV_SORT1]));
    }
    c->timing.d2h_bytes = out_bytes;
    memcpy(out_doc_ids, h + o_doc, size_t(B) * p->limit * 8);
    memcpy(out_scores, h + o_sc, size_t(B) * p->limit * 4);
    memcpy(out_n, h + o_n, size_t(B) * 4);
    memcpy(out_count, h + o_cnt, size_t(B) * 8);
    OCTRY(finish_timing(c, has_v && emb->n_rows > 0, has_ft, true, did_comm));
    c->timing.device_ms += sort_ms;   // the sortBy kernels run after the plain tail's events
    c->timing.fuse_ms += sort_ms;
    return OC_OK;
}

extern "C" int oc_search(oc_ctx *c, oc_emb *emb, oc_str *str, const oc_search_params *p, uint64_t *out_doc_ids,
                         float *out_scores, uint32_t *out_n, uint64_t *out_count) {
    return search_impl(c, emb, str, p, out_doc_ids, out_scores, out_n, out_count, nullptr, nullptr);
}

// ------------------------------------------------------------------------------------ facets
// FacetContext::execute (read/index/facet.rs:147-209): for every requested variant of a filter field — bool
// true/false (bool_field.rs:182-208), a number range [from, to] inclusive (number_field.rs:368-387), a
// string_filter key (string_filter_field.rs:175-193) — count the documents of the variant that are keys of the
// score map.  On the device the score map's key set is a bitmap over DocumentId: the matched rows of the BM25
// tile kernels (+ the vector hits), and a variant is a slice of a device-resident document array.
struct FacetField {
    bool number = false;
    uint64_t n_docs = 0;
    uint64_t *docs = nullptr;              // device: variant-major (CSR) or value-sorted (number field)
    std::vector<uint64_t> offsets;         // host: n_variants + 1
    std::vector<double> values;            // host: ascending (number field)
};
struct oc_facets {
    oc_ctx *ctx;
    uint64_t nbits;                        // DocumentId space [0, nbits)
    std::vector<FacetField> fields;
};
struct FacetReqDev { const uint64_t *docs; uint64_t n; };

extern "C" int oc_facets_create(oc_ctx *c, uint64_t nbits, oc_facets **out) {
    if (!c || !out || nbits == 0) return fail(OC_ERR_INVALID, "bad arguments");
    oc_facets *f = new oc_facets();
    f->ctx = c; f->nbits = nbits;
    *out = f;
    return OC_OK;
}
extern "C" void oc_facets_destroy(oc_facets *f) {
    if (!f) return;
    {
        std::lock_guard<std::mutex> g(f->ctx->mu);
        cudaSetDevice(f->ctx->device);
        cudaStreamSynchronize(f->ctx->stream);
        for (auto &fl : f->fields) cudaFree(fl.docs);
    }
    delete f;
}
static int facets_add(oc_facets *f, FacetField &&fl, const uint64_t *doc_ids, uint32_t *out_field) {
    oc_ctx *c = f->ctx;
    std::lock_guard<std::mutex> g(c->mu);
    CU(cudaSetDevice(c->device));
    if (fl.n_docs) {
        CU(cudaMalloc(&fl.docs, fl.n_docs * 8));
        CU(cudaMemcpy(fl.docs, doc_ids, fl.n_docs * 8, cudaMemcpyHostToDevice));
    }
    f->fields.push_back(std::move(fl));
    if (out_field) *out_field = (uint32_t)f->fields.size() - 1;
    return OC_OK;
}
extern "C" int oc_facets_add_field(oc_facets *f, uint32_t n_variants, const uint64_t *variant_offsets, const uint64_t *doc_ids,
                                   uint32_t *out_field) {
    if (!f || !variant_offsets || n_variants == 0) return fail(OC_ERR_INVALID, "bad arguments");
    for (uint32_t v = 0; v < n_variants; v++)
        if (variant_offsets[v + 1] < variant_offsets[v]) return fail(OC_ERR_INVALID, "variant_offsets not monotone");
    if (variant_offsets[n_variants] && !doc_ids) return fail(OC_ERR_INVALID, "doc_ids is NULL");
    FacetField fl;
    fl.n_docs = variant_offsets[n_variants];
    fl.offsets.assign(variant_offsets, variant_offsets + n_variants + 1);
    return facets_add(f, std::move(fl), doc_ids, out_field);
}
extern "C" int oc_facets_add_number_field(oc_facets *f, uint64_t n, const double *values_sorted, const uint64_t *doc_ids,
                                          uint32_t *out_field) {
    if (!f || (n && (!values_sorted || !doc_ids))) return fail(OC_ERR_INVALID, "bad arguments");
    for (uint64_t i = 1; i < n; i++)
        if (!(values_sorted[i] >= values_sorted[i - 1])) return fail(OC_ERR_INVALID, "values must be ascending (no NaN)");
    FacetField fl;
    fl.number = true; fl.n_docs = n;
    fl.values.assign(values_sorted, values_sorted + n);
    return facets_add(f, std::move(fl), doc_ids, out_field);
}

// row bitmap -> DocumentId bitmap when rows are not document ids
__global__ void facet_rows_to_docs_kernel(const uint32_t *row_bits, uint64_t row_stride_words, const uint64_t *row_doc, uint64_t n_rows,
                                          uint32_t *doc_bits, uint64_t doc_stride_words, uint64_t nbits) {
    const uint32_t q = blockIdx.y;
    const uint64_t w = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (w * 32 >= n_rows) return;
    uint32_t v = row_bits[size_t(q) * row_stride_words + w];
    while (v) {
        const uint32_t b = __ffs(v) - 1;
        v &= v - 1;
        const uint64_t r = w * 32 + b;
        if (r < n_rows) { const uint64_t d = row_doc[r]; if (d < nbits) atomicOr(&doc_bits[size_t(q) * doc_stride_words + (d >> 5)], 1u << (d & 31)); }
    }
}
// the vector hits are keys of the score map too (token_score.rs:340-351, 416-419)
__global__ void facet_mark_hits_kernel(const uint64_t *v_doc, const uint32_t *v_cnt, uint32_t v_stride, uint32_t B, uint32_t *doc_bits,
                                       uint64_t doc_stride_words, uint64_t nbits_cap) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * v_stride) return;
    const uint32_t q = i / v_stride, j = i % v_stride;
    if (j >= v_cnt[q]) return;
    const uint64_t d = v_doc[i];
    if (d < nbits_cap) atomicOr(&doc_bits[size_t(q) * doc_stride_words + (d >> 5)], 1u << (d & 31));
}
// one block = 1024 documents of one variant, counted against every query's bitmap (the slice is read once)
__global__ void __launch_bounds__(256) facet_count_kernel(const FacetReqDev *reqs, uint32_t n_reqs, const uint32_t *bits,
                                                          uint64_t stride_words, uint64_t nbits_cap, uint32_t B,
                                                          unsigned long long *out) {
    const uint32_t r = blockIdx.y;
    const FacetReqDev rq = reqs[r];
    const uint64_t base = uint64_t(blockIdx.x) * 1024;
    if (base >= rq.n) return;
    uint64_t d[4];
#pragma unroll
    for (int u = 0; u < 4; u++) {
        const uint64_t i = base + threadIdx.x + u * 256;
        const uint64_t v = i < rq.n ? rq.docs[i] : ~0ull;
        d[u] = v < nbits_cap ? v : ~0ull;
    }
    __shared__ uint32_t s_c[8];
    for (uint32_t q = 0; q < B; q++) {
        const uint32_t *bq = bits + size_t(q) * stride_words;
        uint32_t c = 0;
#pragma unroll
        for (int u = 0; u < 4; u++)
            if (d[u] != ~0ull) c += (bq[d[u] >> 5] >> (d[u] & 31)) & 1u;
        c = __reduce_add_sync(0xffffffffu, c);
        if ((threadIdx.x & 31) == 0) s_c[threadIdx.x >> 5] = c;
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t t = 0;
            for (int w = 0; w < 8; w++) t += s_c[w];
            if (t) atomicAdd(out + size_t(q) * n_reqs + r, (unsigned long long)t);
        }
        __syncthreads();
    }
}

// the key set of each query's score map as a DocumentId bitmap over [0, *cap_bits): the tile scorers' matched rows
// (c->mbits) + the vector hits; *stride in u32 words
static int score_map_bits(oc_ctx *c, uint32_t B, bool has_ft, bool has_v, const StrSnap *S, uint32_t n_tiles, uint32_t vlimit,
                          uint64_t nbits, const uint32_t **bits, uint64_t *stride, uint64_t *cap_bits) {
    const uint64_t row_words = uint64_t(n_tiles) * (BM25_TILE / 32);
    const uint64_t doc_words = (nbits + 31) / 32;
    const bool identity = has_ft && S->row_doc == nullptr;
    if (identity && !has_v) {   // the row bitmap is the document bitmap
        *bits = c->mbits.as<uint32_t>(); *stride = row_words; *cap_bits = S->n_rows;
        return OC_OK;
    }
    OCTRY(c->dbits.ensure(size_t(B) * doc_words * 4));
    CU(cudaMemsetAsync(c->dbits.p, 0, size_t(B) * doc_words * 4, c->stream));
    if (has_ft && n_tiles) {
        if (identity) {
            const uint64_t wcopy = std::min(row_words, doc_words);
            CU(cudaMemcpy2DAsync(c->dbits.p, doc_words * 4, c->mbits.p, row_words * 4, wcopy * 4, B, cudaMemcpyDeviceToDevice, c->stream));
        } else {
            dim3 grid((unsigned)((row_words + 255) / 256), B);
            facet_rows_to_docs_kernel<<<grid, 256, 0, c->stream>>>(c->mbits.as<uint32_t>(), row_words, S->row_doc, S->n_rows,
                                                                  c->dbits.as<uint32_t>(), doc_words, nbits);
            launched(c);
        }
    }
    if (has_v) {
        facet_mark_hits_kernel<<<(B * vlimit + 255) / 256, 256, 0, c->stream>>>(c->v_doc.as<uint64_t>(), c->v_cnt.as<uint32_t>(), vlimit, B,
                                                                              c->dbits.as<uint32_t>(), doc_words, nbits);
        launched(c);
    }
    *bits = c->dbits.as<uint32_t>(); *stride = doc_words; *cap_bits = nbits;
    return OC_OK;
}

static int run_facets(oc_ctx *c, const FacetJob &fj, uint32_t B, bool has_ft, bool has_v, const StrSnap *S, uint32_t n_tiles,
                      uint32_t vlimit) {
    oc_facets *fc = fj.fc;
    // resolve the requests to device slices
    std::vector<FacetReqDev> rd(fj.n_reqs);
    uint64_t max_n = 0;
    for (uint32_t i = 0; i < fj.n_reqs; i++) {
        const oc_facet_req &rq = fj.reqs[i];
        if (rq.field >= fc->fields.size()) return fail(OC_ERR_INVALID, "facet request %u: unknown field %u", i, rq.field);
        const FacetField &fl = fc->fields[rq.field];
        uint64_t lo, hi;
        if (fl.number) {   // NumberFilter::Between = inclusive on both ends (number_field.rs:376, 604-631)
            lo = uint64_t(std::lower_bound(fl.values.begin(), fl.values.end(), rq.from) - fl.values.begin());
            hi = uint64_t(std::upper_bound(fl.values.begin(), fl.values.end(), rq.to) - fl.values.begin());
            if (hi < lo) hi = lo;
        } else {
            if (rq.variant + 1 >= fl.offsets.size()) return fail(OC_ERR_INVALID, "facet request %u: unknown variant %u", i, rq.variant);
            lo = fl.offsets[rq.variant]; hi = fl.offsets[rq.variant + 1];
        }
        rd[i].docs = fl.docs + lo; rd[i].n = hi - lo;
        max_n = std::max(max_n, rd[i].n);
    }
    const uint32_t *bits = nullptr; uint64_t stride = 0, cap_bits = 0;
    OCTRY(score_map_bits(c, B, has_ft, has_v, S, n_tiles, vlimit, fc->nbits, &bits, &stride, &cap_bits));
    OCTRY(c->facet_req.ensure(size_t(fj.n_reqs) * sizeof(FacetReqDev)));
    OCTRY(c->facet_out.ensure(size_t(B) * fj.n_reqs * 8));
    CU(cudaMemcpyAsync(c->facet_req.p, rd.data(), size_t(fj.n_reqs) * sizeof(FacetReqDev), cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemsetAsync(c->facet_out.p, 0, size_t(B) * fj.n_reqs * 8, c->stream));
    if (max_n) {
        dim3 grid((unsigned)((max_n + 1023) / 1024), fj.n_reqs);
        facet_count_kernel<<<grid, 256, 0, c->stream>>>(c->facet_req.as<FacetReqDev>(), fj.n_reqs, bits, stride, cap_bits, B,
                                                       c->facet_out.as<unsigned long long>());
        launched(c);
        CU(cudaGetLastError());
    }
    CU(cudaMemcpyAsync(fj.out_counts, c->facet_out.p, size_t(B) * fj.n_reqs * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));   // rd lives on this stack
    return OC_OK;
}

extern "C" int oc_search_facets(oc_ctx *c, oc_emb *emb, oc_str *str, oc_facets *facets, const oc_search_params *p,
                                const oc_facet_req *reqs, uint32_t n_reqs, uint64_t *out_counts) {
    if (!c || !p || !facets || !out_counts || (n_reqs && !reqs)) return fail(OC_ERR_INVALID, "NULL argument");
    if (facets->ctx != c) return fail(OC_ERR_INVALID, "facets belong to another ctx");
    if (p->sharded) return fail(OC_ERR_UNSUPPORTED, "facets over a sharded search: count per shard and add the counts");
    if (n_reqs == 0) return OC_OK;
    // the reference computes facets on the score map re-scored WITHOUT the where-filter (search.rs:361-396: only the
    // uncommitted deletes stay excluded), so that the counts do not collapse onto the selected category
    oc_search_params q = *p;
    q.filter_bits = nullptr; q.filter_nbits = 0; q.filter = nullptr;
    const uint32_t B = p->n_queries;
    std::vector<uint64_t> docs(size_t(B) * p->limit), cnt(B);
    std::vector<float> scores(size_t(B) * p->limit);
    std::vector<uint32_t> n(B);
    FacetJob fj{facets, reqs, n_reqs, out_counts};
    return search_impl(c, emb, str, &q, docs.data(), scores.data(), n.data(), cnt.data(), &fj, nullptr);
}

// ------------------------------------------------------------------------------------ sortBy
// sort_token_scores with Some(sort_by) (read/sort.rs:17-98, 236-257): the first limit+offset keys of the score map in
// the order IndexSortContext::execute yields (read/index/sort.rs:186-264), each with its score-map value.  Per field
// the store keeps on the device a dense rank of every document's value (SORT_NONE = no value), the two walk orders
// (rank ascending / descending, DocumentId ascending inside a rank) and the value of each rank (out_keys).
struct SortField {
    uint32_t *rank = nullptr;                       // device [nbits]
    uint32_t *order_asc = nullptr, *order_desc = nullptr;   // device [n_pop] DocumentIds
    double *rank_value = nullptr;                   // device [n_ranks]
    uint64_t n_pop = 0;
    uint32_t n_ranks = 0;
};
struct oc_sort {
    oc_ctx *ctx;
    uint64_t nbits;                                 // DocumentId space [0, nbits)
    std::vector<SortField> fields;
};

extern "C" int oc_sort_create(oc_ctx *c, uint64_t nbits, oc_sort **out) {
    if (!c || !out || nbits == 0) return fail(OC_ERR_INVALID, "bad arguments");
    if (nbits > (uint64_t(1) << 32)) return fail(OC_ERR_UNSUPPORTED, "sort store: nbits %llu > 2^32", (unsigned long long)nbits);
    oc_sort *s = new oc_sort();
    s->ctx = c; s->nbits = nbits;
    *out = s;
    return OC_OK;
}
static void sort_field_free(SortField &f) {
    cudaFree(f.rank); cudaFree(f.order_asc); cudaFree(f.order_desc); cudaFree(f.rank_value);
    f = SortField{};
}
extern "C" void oc_sort_destroy(oc_sort *s) {
    if (!s) return;
    {
        std::lock_guard<std::mutex> g(s->ctx->mu);
        cudaSetDevice(s->ctx->device);
        cudaStreamSynchronize(s->ctx->stream);
        for (auto &f : s->fields) sort_field_free(f);
    }
    delete s;
}
// (doc, key) pairs -> ranks and walk orders.  Key: double (number), int64 (date, exact), uint8 (bool: false < true).
template <typename K>
static int sort_add(oc_sort *s, uint64_t n, const uint64_t *docs, const K *keys, uint32_t *out_field) {
    std::vector<uint64_t> idx(n);
    for (uint64_t i = 0; i < n; i++) {
        if (docs[i] >= s->nbits) return fail(OC_ERR_INVALID, "sort field: document %llu >= nbits", (unsigned long long)docs[i]);
        idx[i] = i;
    }
    std::sort(idx.begin(), idx.end(), [&](uint64_t a, uint64_t b) { return keys[a] < keys[b] || (keys[a] == keys[b] && docs[a] < docs[b]); });
    std::vector<uint32_t> rank(s->nbits, SORT_NONE), asc(n), desc(n);
    std::vector<double> value;
    std::vector<uint64_t> group;   // start of each rank's run in asc
    for (uint64_t j = 0; j < n; j++) {
        const uint64_t i = idx[j];
        if (j == 0 || keys[i] != keys[idx[j - 1]]) { value.push_back(double(keys[i])); group.push_back(j); }
        // the reference would emit such a document once per value (an array field): not representable in one rank
        if (rank[docs[i]] != SORT_NONE) return fail(OC_ERR_INVALID, "sort field: document %llu is listed twice", (unsigned long long)docs[i]);
        rank[docs[i]] = uint32_t(value.size() - 1);
        asc[j] = uint32_t(docs[i]);
    }
    group.push_back(n);
    for (size_t g = group.size() - 1, o = 0; g-- > 0;)   // ranks descending, DocumentId ascending inside a rank
        for (uint64_t j = group[g]; j < group[g + 1]; j++) desc[o++] = asc[j];
    oc_ctx *c = s->ctx;
    std::lock_guard<std::mutex> g(c->mu);
    CU(cudaSetDevice(c->device));
    SortField f;
    f.n_pop = n; f.n_ranks = uint32_t(value.size());
    auto up = [&](void **dst, const void *src, size_t bytes) -> int {
        cudaError_t e = cudaMalloc(dst, std::max<size_t>(bytes, 8));
        if (e != cudaSuccess) return fail(OC_ERR_OOM, "cudaMalloc(sort field): %s", cudaGetErrorString(e));
        if (bytes) CU(cudaMemcpy(*dst, src, bytes, cudaMemcpyHostToDevice));
        return OC_OK;
    };
    int rc = up(reinterpret_cast<void **>(&f.rank), rank.data(), rank.size() * 4);
    if (rc == OC_OK) rc = up(reinterpret_cast<void **>(&f.order_asc), asc.data(), n * 4);
    if (rc == OC_OK) rc = up(reinterpret_cast<void **>(&f.order_desc), desc.data(), n * 4);
    if (rc == OC_OK) rc = up(reinterpret_cast<void **>(&f.rank_value), value.data(), value.size() * 8);
    if (rc != OC_OK) { sort_field_free(f); return rc; }
    s->fields.push_back(f);
    if (out_field) *out_field = uint32_t(s->fields.size() - 1);
    return OC_OK;
}
extern "C" int oc_sort_add_number_field(oc_sort *s, uint64_t n, const uint64_t *doc_ids, const double *values, uint32_t *out_field) {
    if (!s || (n && (!doc_ids || !values))) return fail(OC_ERR_INVALID, "bad arguments");
    for (uint64_t i = 0; i < n; i++) if (values[i] != values[i]) return fail(OC_ERR_INVALID, "sort field: value %llu is NaN", (unsigned long long)i);
    return sort_add(s, n, doc_ids, values, out_field);
}
extern "C" int oc_sort_add_date_field(oc_sort *s, uint64_t n, const uint64_t *doc_ids, const int64_t *ts, uint32_t *out_field) {
    if (!s || (n && (!doc_ids || !ts))) return fail(OC_ERR_INVALID, "bad arguments");
    return sort_add(s, n, doc_ids, ts, out_field);
}
extern "C" int oc_sort_add_bool_field(oc_sort *s, uint64_t n_true, const uint64_t *true_docs, uint64_t n_false, const uint64_t *false_docs,
                                      uint32_t *out_field) {
    if (!s || (n_true && !true_docs) || (n_false && !false_docs)) return fail(OC_ERR_INVALID, "bad arguments");
    std::vector<uint64_t> docs(false_docs, false_docs + n_false);
    docs.insert(docs.end(), true_docs, true_docs + n_true);
    std::vector<uint8_t> keys(n_false, 0);
    keys.resize(n_false + n_true, 1);
    return sort_add(s, docs.size(), docs.data(), keys.data(), out_field);
}

static int run_sort(oc_ctx *c, const SortJob &sj, const oc_search_params *p, uint32_t B, bool has_ft, bool has_v, const StrSnap *S,
                    uint32_t n_tiles, uint32_t vlimit, uint32_t n_keep, const FuseParams &fp, const Bm25Params &bp, const uint32_t *row_ok) {
    const SortField &fl = sj.st->fields[sj.field];
    SortSelParams sp{};
    OCTRY(score_map_bits(c, B, has_ft, has_v, S, n_tiles, vlimit, sj.st->nbits, &sp.bits, &sp.stride_words, &sp.cap_bits));
    OCTRY(c->sort_pick.ensure(size_t(B) * n_keep * 8));
    OCTRY(c->sort_npick.ensure(size_t(B) * 4));
    OCTRY(c->sort_form.ensure(B));
    OCTRY(c->sort_keys.ensure(size_t(B) * p->limit * 8));
    sp.count = fp.out_count;
    sp.rank = fl.rank; sp.nbits = sj.st->nbits;
    sp.order = sj.descending ? fl.order_desc : fl.order_asc;
    sp.n_pop = fl.n_pop; sp.n_ranks = fl.n_ranks; sp.descending = sj.descending ? 1 : 0;
    sp.n_keep = n_keep; sp.form = sj.form;
    sp.pick = c->sort_pick.as<uint64_t>(); sp.n_pick = c->sort_npick.as<uint32_t>(); sp.form_out = c->sort_form.as<uint8_t>();
    const size_t smem = (size_t(SORT_GATHER_CAP) + std::max<uint32_t>(32, next_pow2(n_keep))) * 8;
    if (smem_cfg_needed(c->device, (const void *)sort_select_kernel, smem))
        CU(cudaFuncSetAttribute(sort_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    sort_select_kernel<<<B, SORT_THREADS, smem, c->stream>>>(sp);
    launched(c);
    CU(cudaGetLastError());
    SortScoreParams ss{};
    if (has_ft) {   // the fulltext score of every pick: the point lookups of the hybrid path (bm25_point_kernel)
        OCTRY(c->sort_rows.ensure(size_t(B) * n_keep * 4));
        OCTRY(c->sort_ft.ensure(size_t(B) * n_keep * 4));
        OCTRY(c->sort_present.ensure(size_t(B) * n_keep));
        map_docs_to_rows_kernel<<<(B * n_keep + 255) / 256, 256, 0, c->stream>>>(sp.pick, sp.n_pick, n_keep, B, S->row_doc, S->n_rows,
                                                                                c->sort_rows.as<uint32_t>());
        launched(c);
        PointParams pp{};
        pp.terms = bp.terms; pp.tokens = bp.tokens; pp.queries = bp.queries;
        pp.n_queries = B; pp.v_stride = n_keep; pp.v_row = c->sort_rows.as<uint32_t>(); pp.row_ok_bits = row_ok;
        pp.k = p->bm25_k; pp.threshold = p->threshold >= 0.0f ? 1 : 0;
        pp.v_ft = c->sort_ft.as<float>(); pp.v_present = c->sort_present.as<uint8_t>();
        bm25_point_kernel<<<(unsigned)((uint64_t(B) * n_keep * 32 + 255) / 256), 256, 0, c->stream>>>(pp);
        launched(c);
        CU(cudaGetLastError());
        ss.p_ft = pp.v_ft; ss.p_present = pp.v_present;
    }
    ss.fp = fp; ss.n_queries = B;
    ss.gmin = fp.out_min; ss.gmax = fp.out_max;
    ss.pick = sp.pick; ss.n_pick = sp.n_pick;
    ss.rank = fl.rank; ss.rank_value = fl.rank_value;
    ss.out_key = c->sort_keys.as<double>();
    sort_score_kernel<<<(unsigned)((uint64_t(B) * p->limit + 255) / 256), 256, 0, c->stream>>>(ss);
    launched(c);
    CU(cudaGetLastError());
    return OC_OK;
}

extern "C" int oc_search_sorted(oc_ctx *c, oc_emb *emb, oc_str *str, oc_sort *s, uint32_t field, int descending,
                                const oc_search_params *p, uint64_t *out_doc_ids, float *out_scores, uint32_t *out_n,
                                uint64_t *out_count, double *out_keys) {
    if (!c || !p || !s) return fail(OC_ERR_INVALID, "NULL argument");
    if (s->ctx != c) return fail(OC_ERR_INVALID, "sort store belongs to another ctx");
    if (p->sharded) return fail(OC_ERR_UNSUPPORTED, "sortBy over a sharded search: sort per shard and merge with oc_merge_sorted_results");
    if (field >= s->fields.size()) return fail(OC_ERR_INVALID, "unknown sort field %u", field);   // SortFieldNotFound
    const char *fe = getenv("OC_SORT_FORM");   // walk | gather: force one selection form (A/B runs, tests)
    const int form = (fe && !strcmp(fe, "walk")) ? SORT_FORM_WALK : (fe && !strcmp(fe, "gather")) ? SORT_FORM_GATHER : SORT_FORM_AUTO;
    SortJob sj{s, field, descending != 0, form, out_keys};
    return search_impl(c, emb, str, p, out_doc_ids, out_scores, out_n, out_count, nullptr, &sj);
}

extern "C" int oc_sort_last_forms(oc_ctx *c, uint32_t n_queries, uint8_t *out) {
    if (!c || (n_queries && !out)) return fail(OC_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> g(c->mu);
    if (n_queries > c->sort_forms.size()) return fail(OC_ERR_INVALID, "the last sorted search had %zu queries", c->sort_forms.size());
    if (n_queries) memcpy(out, c->sort_forms.data(), n_queries);
    return OC_OK;
}

// MergeSortedIterator (read/sort.rs:491-560) + truncate over per-index lists already in field order: the list whose head
// key comes first wins; on equal keys the lower index wins (its whole value group comes first, as the iterator's strict
// comparison yields it).  Keys are compared exactly (dates too: no i32 clamp).
extern "C" int oc_merge_sorted_results(uint32_t n_indexes, uint32_t B, uint32_t limit, uint32_t offset, uint32_t in_stride,
                                       int descending, const uint64_t *const *doc_ids, const float *const *scores,
                                       const double *const *keys, const uint32_t *const *n, const uint64_t *const *counts,
                                       uint64_t *out_doc_ids, float *out_scores, uint32_t *out_n, uint64_t *out_count) {
    if (!doc_ids || !scores || !keys || !n || !counts || !out_doc_ids || !out_scores || !out_n || !out_count)
        return fail(OC_ERR_INVALID, "NULL argument");
    if (limit == 0) return fail(OC_ERR_INVALID, "limit must be >= 1");
    std::vector<uint32_t> head(n_indexes);
    for (uint32_t q = 0; q < B; q++) {
        std::fill(head.begin(), head.end(), 0u);
        uint64_t cnt = 0;
        for (uint32_t i = 0; i < n_indexes; i++) {
            if (n[i][q] > in_stride) return fail(OC_ERR_INVALID, "index %u query %u: n > in_stride", i, q);
            cnt += counts[i][q];
        }
        uint32_t taken = 0, written = 0;
        while (written < limit) {
            int best = -1;
            for (uint32_t i = 0; i < n_indexes; i++) {
                if (head[i] >= n[i][q]) continue;
                if (best < 0) { best = (int)i; continue; }
                const double ka = keys[i][size_t(q) * in_stride + head[i]], kb = keys[best][size_t(q) * in_stride + head[best]];
                if (descending ? ka > kb : ka < kb) best = (int)i;
            }
            if (best < 0) break;
            if (taken >= offset) {
                out_doc_ids[size_t(q) * limit + written] = doc_ids[best][size_t(q) * in_stride + head[best]];
                out_scores[size_t(q) * limit + written] = scores[best][size_t(q) * in_stride + head[best]];
                written++;
            }
            taken++; head[best]++;
        }
        for (uint32_t k = written; k < limit; k++) { out_doc_ids[size_t(q) * limit + k] = 0; out_scores[size_t(q) * limit + k] = 0.f; }
        out_n[q] = written;
        out_count[q] = cnt;
    }
    return OC_OK;
}

// ------------------------------------------------------------------------------------ micro-batching front
struct OcSearchExec {
    oc_ctx *c; oc_emb *e; oc_str *s;
    int operator()(const oc_search_params *p, uint64_t *docs, float *scores, uint32_t *n, uint64_t *count) const {
        return oc_search(c, e, s, p, docs, scores, n, count);
    }
};
struct oc_batcher {
    ocb::Batcher<OcSearchExec> q;
    oc_batcher(OcSearchExec x, uint32_t dim, uint32_t mb, uint32_t mw) : q(x, dim, mb, mw, x.e != nullptr, x.s != nullptr) {}
};
extern "C" int oc_batcher_create(oc_ctx *c, oc_emb *emb, oc_str *str, uint32_t max_batch, uint32_t max_wait_us, oc_batcher **out) {
    if (!c || !out || (!emb && !str)) return fail(OC_ERR_INVALID, "bad arguments");
    if ((emb && emb->ctx != c) || (str && str->ctx != c)) return fail(OC_ERR_INVALID, "store belongs to another ctx");
    if (max_batch == 0 || max_batch > 4096) return fail(OC_ERR_INVALID, "max_batch %u outside 1..4096", max_batch);
    *out = new oc_batcher(OcSearchExec{c, emb, str}, emb ? emb->dim : 0, max_batch, max_wait_us);
    return OC_OK;
}
extern "C" void oc_batcher_destroy(oc_batcher *b) { delete b; }
extern "C" int oc_batcher_search(oc_batcher *b, const oc_search_params *p, uint64_t *out_doc_ids, float *out_scores,
                                 uint32_t *out_n, uint64_t *out_count) {
    if (!b || !p || !out_doc_ids || !out_scores || !out_n || !out_count) return fail(OC_ERR_INVALID, "NULL argument");
    if (p->n_queries != 1) return fail(OC_ERR_INVALID, "oc_batcher_search takes one query per call (n_queries = %u)", p->n_queries);
    g_err[0] = 0;
    const int rc = b->q.submit(p, out_doc_ids, out_scores, out_n, out_count);
    // the batch ran on its leader's thread: that is where oc_last_error() holds the detail
    if (rc != OC_OK && g_err[0] == 0) return fail(rc, "the coalesced oc_search of this query's batch failed (detail on the leading caller's thread)");
    return rc;
}
extern "C" int oc_batcher_stats(oc_batcher *b, uint64_t *n_queries, uint64_t *n_batches, uint64_t *n_direct) {
    if (!b) return fail(OC_ERR_INVALID, "NULL argument");
    b->q.stats(n_queries, n_batches, n_direct);
    return OC_OK;
}

// ------------------------------------------------------------------------------------ term dictionary / query resolution
// Host only (no device): the step the reference performs before the posting walk — tokenize_and_stem
// (token_score.rs:196-209) and the FST term expansion inside StringStorage (string_field.rs:208-225).
struct oc_dict { ocd::Dict d; explicit oc_dict(uint32_t n) : d(n) {} };
struct oc_resolved { ocd::Resolved r; };

extern "C" int oc_dict_create(uint32_t n_fields, oc_dict **out) {
    if (!out || n_fields == 0) return fail(OC_ERR_INVALID, "bad arguments");
    *out = new oc_dict(n_fields);
    return OC_OK;
}
extern "C" void oc_dict_destroy(oc_dict *d) { delete d; }
extern "C" int oc_dict_add_terms(oc_dict *d, uint32_t field, const char *const *terms, uint32_t n, uint32_t *out_ids) {
    if (!d || field >= d->d.n_fields() || (n && !terms)) return fail(OC_ERR_INVALID, "bad arguments");
    for (uint32_t i = 0; i < n; i++) if (!terms[i]) return fail(OC_ERR_INVALID, "term %u is NULL", i);
    d->d.add_terms(field, terms, n, out_ids);
    return OC_OK;
}
extern "C" int oc_dict_lookup(oc_dict *d, uint32_t field, const char *term, uint32_t *out_id) {
    if (!d || field >= d->d.n_fields() || !term || !out_id) return fail(OC_ERR_INVALID, "bad arguments");
    if (!d->d.lookup(field, term, out_id)) *out_id = 0xffffffffu;
    return OC_OK;
}
extern "C" uint32_t oc_dict_size(oc_dict *d, uint32_t field) { return (d && field < d->d.n_fields()) ? d->d.size(field) : 0; }
// Snowball English (Porter2), restated in csrc/stem_en.h: an oc_stem_fn a host without its own parser can install
extern "C" size_t oc_stem_english(const char *tok, size_t len, char *out, size_t cap, void *user) {
    (void)user;
    if (!tok || !out) return 0;
    const std::string st = ocs::stem_english(std::string(tok, len));
    if (st.size() > cap) return 0;
    memcpy(out, st.data(), st.size());
    return st.size();
}
extern "C" int oc_dict_set_stemmer(oc_dict *d, oc_stem_fn fn, void *user) {
    if (!d) return fail(OC_ERR_INVALID, "dict is NULL");
    d->d.set_stemmer(fn, user);
    return OC_OK;
}
extern "C" int oc_dict_resolve(oc_dict *d, const oc_resolve_params *p, oc_resolved **out) {
    if (!d || !p || !out || (p->n_queries && !p->texts)) return fail(OC_ERR_INVALID, "bad arguments");
    for (uint32_t i = 0; i < p->n_queries; i++) if (!p->texts[i]) return fail(OC_ERR_INVALID, "text %u is NULL", i);
    if (p->tolerance > 8) return fail(OC_ERR_UNSUPPORTED, "tolerance %d > 8", p->tolerance);
    ocd::ResolveOpts o;
    o.exact = p->exact != 0; o.tolerance = p->tolerance; o.field_boost = p->field_boost; o.field_mask = p->field_mask;
    o.exact_match_boost = p->exact_match_boost > 0.f ? p->exact_match_boost : 2.0f;
    oc_resolved *r = new oc_resolved();
    d->d.resolve(p->texts, p->n_queries, o, &r->r);
    *out = r;
    return OC_OK;
}
extern "C" void oc_resolved_arrays(const oc_resolved *r, const uint32_t **q_token_offsets, const uint32_t **token_term_offsets,
                                   const uint32_t **term_field, const uint32_t **term_id, const float **term_weight,
                                   uint32_t *n_tokens, uint32_t *n_terms) {
    if (!r) return;
    static const uint32_t zero_u = 0; static const float one_f = 1.0f;   // empty arrays still get valid pointers
    if (q_token_offsets) *q_token_offsets = r->r.q_token_offsets.data();
    if (token_term_offsets) *token_term_offsets = r->r.token_term_offsets.data();
    if (term_field) *term_field = r->r.term_field.empty() ? &zero_u : r->r.term_field.data();
    if (term_id) *term_id = r->r.term_id.empty() ? &zero_u : r->r.term_id.data();
    if (term_weight) *term_weight = r->r.term_weight.empty() ? &one_f : r->r.term_weight.data();
    if (n_tokens) *n_tokens = (uint32_t)r->r.token_term_offsets.size() - 1;
    if (n_terms) *n_terms = (uint32_t)r->r.term_id.size();
}
extern "C" void oc_resolved_fill(const oc_resolved *r, oc_search_params *p) {
    if (!r || !p) return;
    oc_resolved_arrays(r, &p->q_token_offsets, &p->token_term_offsets, &p->term_field, &p->term_id, &p->term_weight, nullptr, nullptr);
    p->n_queries = (uint32_t)r->r.q_token_offsets.size() - 1;
}
extern "C" void oc_resolved_free(oc_resolved *r) { delete r; }
