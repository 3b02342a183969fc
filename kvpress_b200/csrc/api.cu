// api.cu — the extern "C" surface declared in include/kvpress_b200.h.
// Validates the problem, carves the caller's workspace and enqueues the kernels on the caller's
// stream. Never allocates, never synchronises (except the *_host convenience call), never throws.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"

namespace kvp {

static thread_local char g_last_cuda_error[256] = "";

static int fail_cuda(cudaError_t e) {
    snprintf(g_last_cuda_error, sizeof(g_last_cuda_error), "%s: %s", cudaGetErrorName(e),
             cudaGetErrorString(e));
    // launch-configuration errors are not sticky: clear them, or the cudaPeekAtLastError() of every later call
    // (of this library or of torch) would report this failure again
    cudaGetLastError();
    return KVP_ERR_CUDA;
}

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Rows (B * Hkv) a call may have. The score kernels put the row on gridDim.y (<= 65535). The generic-score path
// (keys_from_scores + selection pass + compaction grid) decodes rows from a 1-D grid of rows x tiles, which only
// needs that product to fit an int; the row cap keeps the counter slots (3 R + 8) in range.
constexpr int64_t kMaxRowsGridY = 65535;
constexpr int64_t kMaxRowsGeneric = (int64_t)1 << 24;
static int64_t max_rows(int scorer) { return scorer == KVP_SCORER_GENERIC ? kMaxRowsGeneric : kMaxRowsGridY; }

static int validate(const kvp_problem* p, Dims* d, bool need_kv_strides = true, int64_t row_cap = kMaxRowsGridY) {
    if (p == nullptr) return KVP_ERR_NULL_POINTER;
    if (p->dtype != KVP_BF16 && p->dtype != KVP_F16) return KVP_ERR_UNSUPPORTED_DTYPE;
    if (p->B <= 0 || p->Hkv <= 0 || p->S <= 0 || p->D <= 0) return KVP_ERR_UNSUPPORTED_SHAPE;
    if (p->D % 8 != 0 || p->D > 256) return KVP_ERR_UNSUPPORTED_SHAPE;
    if (p->Hq <= 0 || p->Hq % p->Hkv != 0) return KVP_ERR_UNSUPPORTED_SHAPE;
    if (p->n_kept < 0 || p->n_kept > p->S) return KVP_ERR_BAD_ARGUMENT;
    if ((int64_t)p->B * p->Hkv > row_cap) return KVP_ERR_UNSUPPORTED_SHAPE;
    if ((int64_t)p->B * p->Hkv * ((p->S + kTile - 1) / kTile) > 0x7FFFFFFF) return KVP_ERR_UNSUPPORTED_SHAPE;  // 1-D grids
    if (need_kv_strides) {
        for (int i = 0; i < 3; ++i) {
            // rows must stay 16-byte aligned: every outer stride is a multiple of 8 elements
            if (p->k_stride[i] % 8 != 0 || p->v_stride[i] % 8 != 0) return KVP_ERR_BAD_STRIDE;
            if (p->k_stride[i] < 0 || p->v_stride[i] < 0) return KVP_ERR_BAD_STRIDE;
        }
        if (p->k_stride[2] < p->D || p->v_stride[2] < p->D) return KVP_ERR_BAD_STRIDE;
    }
    d->B = p->B;
    d->H = p->Hkv;
    d->Hq = p->Hq;
    d->S = p->S;
    d->D = p->D;
    d->n_kept = p->n_kept;
    d->R = p->B * p->Hkv;
    d->ks = {p->k_stride[0], p->k_stride[1], p->k_stride[2]};
    d->vs = {p->v_stride[0], p->v_stride[1], p->v_stride[2]};
    return KVP_OK;
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

struct WsLayout {
    size_t keys_off, hist_off, sfx_off, meta_off, prefix_off, scorer_off, total;
    int S_pad, n_tiles;
    size_t hist_bytes, scorer_bytes;
};

static WsLayout layout(const Dims& d, int scorer, int window) {
    WsLayout L;
    L.n_tiles = (d.S + kTile - 1) / kTile;
    L.S_pad = L.n_tiles * kTile;
    size_t off = 0;
    // one zeroed region (a single memset node per call): hist_hi, hist_lo, counters, tile_prefix
    L.hist_off = off;
    off = align_up(off + ((size_t)d.R * 256 * 2 + (size_t)d.R * 3 + 64) * sizeof(uint32_t), 256);
    L.prefix_off = off;
    off = align_up(off + (size_t)d.R * L.n_tiles * sizeof(uint2), 256);
    L.hist_bytes = off - L.hist_off;
    L.keys_off = off;
    off = align_up(off + (size_t)d.R * L.S_pad * sizeof(uint16_t), 256);
    L.sfx_off = off;
    off = align_up(off + (size_t)d.R * L.n_tiles * kSfxStride * sizeof(uint16_t), 256);
    L.meta_off = off;
    off = align_up(off + (size_t)d.R * sizeof(uint2), 256);
    L.scorer_off = off;
    L.scorer_bytes = 0;
    if (scorer == KVP_SCORER_SNAPKV) L.scorer_bytes = snapkv_scratch_bytes(d, window);
    if (scorer == KVP_SCORER_EXPECTED_ATTENTION) L.scorer_bytes = ea_scratch_bytes(d);
    if (scorer == KVP_SCORER_KEYDIFF) L.scorer_bytes = keydiff_scratch_bytes(d);
    off = align_up(off + L.scorer_bytes, 256);
    L.total = off;
    return L;
}

static int carve(const Dims& d, int scorer, int window, void* workspace, size_t bytes,
                 Workspace* ws, WsLayout* Lout) {
    const WsLayout L = layout(d, scorer, window);
    if (workspace == nullptr) return KVP_ERR_NULL_POINTER;
    if (!aligned16(workspace)) return KVP_ERR_BAD_STRIDE;
    if (bytes < L.total) return KVP_ERR_WORKSPACE_TOO_SMALL;
    char* base = static_cast<char*>(workspace);
    ws->hist_hi = reinterpret_cast<uint32_t*>(base + L.hist_off);
    ws->hist_lo = ws->hist_hi + (size_t)d.R * 256;
    ws->counters = ws->hist_lo + (size_t)d.R * 256;
    ws->keys = reinterpret_cast<uint16_t*>(base + L.keys_off);
    ws->tile_sfx = reinterpret_cast<uint16_t*>(base + L.sfx_off);
    ws->row_meta = reinterpret_cast<uint2*>(base + L.meta_off);
    ws->tile_prefix = reinterpret_cast<uint2*>(base + L.prefix_off);
    ws->R = d.R;
    ws->scorer = base + L.scorer_off;
    ws->scorer_bytes = L.scorer_bytes;
    ws->S_pad = L.S_pad;
    ws->n_tiles = L.n_tiles;
    *Lout = L;
    return KVP_OK;
}

static int check_io(const void* K, const void* V, const void* K_out, const void* V_out) {
    if (!K || !V || !K_out || !V_out) return KVP_ERR_NULL_POINTER;
    if (!aligned16(K) || !aligned16(V) || !aligned16(K_out) || !aligned16(V_out))
        return KVP_ERR_BAD_STRIDE;
    return KVP_OK;
}

}  // namespace kvp

using namespace kvp;

extern "C" {

int kvp_abi_version(void) { return KVP_ABI_VERSION; }

const char* kvp_status_string(int status) {
    switch (status) {
        case KVP_OK: return "ok";
        case KVP_ERR_NULL_POINTER: return "null pointer";
        case KVP_ERR_UNSUPPORTED_SHAPE: return "unsupported shape";
        case KVP_ERR_UNSUPPORTED_DTYPE: return "unsupported dtype (bf16 / fp16 only)";
        case KVP_ERR_BAD_STRIDE: return "bad stride or alignment (rows must be 16-byte aligned)";
        case KVP_ERR_WORKSPACE_TOO_SMALL: return "workspace too small";
        case KVP_ERR_CUDA: return "CUDA error (see kvp_last_cuda_error)";
        case KVP_ERR_BAD_ARGUMENT: return "bad argument";
        case KVP_ERR_KERNEL_TIMEOUT: return "a kernel abandoned a bounded wait (outputs invalid)";
        default: return "unknown status";
    }
}

const char* kvp_last_cuda_error(void) { return g_last_cuda_error; }

int kvp_workspace_bytes(const kvp_problem* p, int scorer, size_t* bytes_out) {
    Dims d;
    int rc = validate(p, &d, false, max_rows(scorer));
    if (rc) return rc;
    if (!bytes_out) return KVP_ERR_NULL_POINTER;
    // window only changes the SnapKV scratch; size for the largest supported window
    *bytes_out = layout(d, scorer, 256).total;
    return KVP_OK;
}

int kvp_workspace_check(const kvp_problem* p, int scorer, const void* workspace, size_t workspace_bytes,
                        kvp_stream_t stream) {
    Dims d;
    int rc = validate(p, &d, false, max_rows(scorer));
    if (rc) return rc;
    Workspace ws;
    WsLayout L;
    if ((rc = carve(d, scorer, 256, const_cast<void*>(workspace), workspace_bytes, &ws, &L))) return rc;
    uint32_t flag = 0;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    cudaError_t e = cudaMemcpyAsync(&flag, ws.counters + kCounterErrSlot(d.R), sizeof(flag),
                                    cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return fail_cuda(e);
    return flag ? KVP_ERR_KERNEL_TIMEOUT : KVP_OK;
}

int kvp_launches_per_compress(const kvp_problem* p, int scorer, int* launches_out) {
    if (!p || !launches_out) return KVP_ERR_NULL_POINTER;
    switch (scorer) {
        case KVP_SCORER_STREAMING: *launches_out = 1; break;
        // "select, compact" below: the selection pass and the compaction grid (select_compact.cu)
        case KVP_SCORER_GENERIC: *launches_out = 4; break;  // memset, keys, select, compact
        case KVP_SCORER_KNORM: {  // cluster kernel | memset + (fused | score, select, compact)
            Dims d;
            if (validate(p, &d, false) == KVP_OK && knorm_cluster_applicable(d)) *launches_out = 1;
            else *launches_out = ((size_t)p->B * p->Hkv * p->S * p->D * 2 <= ((size_t)32 << 20)) ? 2 : 4;
            break;
        }
        case KVP_SCORER_KEYDIFF: *launches_out = 6; break;  // memset, anchor partials, merge, score, select, compact
        case KVP_SCORER_SNAPKV: *launches_out = 7; break;  // memset, stats, memset, colsum, finalize, select, compact
        case KVP_SCORER_EXPECTED_ATTENTION: {
            // press defaults (use_covariance + use_vnorm): memset, logits (the tensor-core kernels stage the V tiles and
            // take the value norms themselves), finalize, select, compact; head dims outside 64 / 128 have no covariance
            // path here, and the covariance-free scan adds the value-norm kernel on the side stream
            *launches_out = (p->D == 64 || p->D == 128) ? 5 : 6;
            break;
        }
        default: return KVP_ERR_BAD_ARGUMENT;
    }
    return KVP_OK;
}

// ---- Knorm ---------------------------------------------------------------------------------------
int kvp_knorm_score(const kvp_problem* p, const void* K, void* scores_out, kvp_stream_t stream) {
    Dims d;
    int rc = validate(p, &d);
    if (rc) return rc;
    if (!K || !scores_out) return KVP_ERR_NULL_POINTER;
    if (!aligned16(K)) return KVP_ERR_BAD_STRIDE;
    Workspace ws = {};
    cudaError_t e = launch_knorm_score(d, p->dtype, K, ws, scores_out, false,
                                       static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? KVP_OK : fail_cuda(e);
}

static int select_and_compact(const Dims& d, const void* K, const void* V, void* K_out,
                              void* V_out, int32_t* idx_out, const Workspace& ws,
                              cudaStream_t st) {
    cudaError_t e = launch_select_compact(d, K, V, K_out, V_out, idx_out, ws, st);
    return e == cudaSuccess ? KVP_OK : fail_cuda(e);
}

int kvp_knorm_compress(const kvp_problem* p, const void* K, const void* V, void* K_out,
                       void* V_out, int32_t* idx_out, void* scores_out, void* workspace,
                       size_t workspace_bytes, kvp_stream_t stream) {
    Dims d;
    int rc = validate(p, &d);
    if (rc) return rc;
    if (d.n_kept == 0) return KVP_OK;
    if ((rc = check_io(K, V, K_out, V_out))) return rc;
    Workspace ws;
    WsLayout L;
    if ((rc = carve(d, KVP_SCORER_KNORM, 0, workspace, workspace_bytes, &ws, &L))) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    // DecodingPress-sized caches: one launch of the cluster kernel (knorm_cluster.cu), no memset, no scratch
    cudaError_t e = launch_knorm_cluster(d, p->dtype, K, V, K_out, V_out, idx_out, scores_out, st);
    if (e != cudaErrorNotSupported) return e == cudaSuccess ? KVP_OK : fail_cuda(e);
    e = cudaMemsetAsync(ws.hist_hi, 0, L.hist_bytes, st);
    if (e != cudaSuccess) return fail_cuda(e);
    // Small caches beyond the cluster path are launch-latency-bound: one persistent kernel does
    // score + select + compact. Large caches measured faster as two kernels (the fused kernel's mixed
    // read/write item stream costs more HBM efficiency than the saved launch; K re-reads miss L2 anyway).
    const size_t k_bytes = (size_t)d.R * d.S * d.D * 2;
    static const size_t fused_max_bytes = [] {  // A/B knob: KVP_KNORM_FUSED_MAX_MB (default 32)
        const char* v = getenv("KVP_KNORM_FUSED_MAX_MB");
        return (size_t)((v && *v) ? atoll(v) : 32) << 20;
    }();
    if (k_bytes <= fused_max_bytes) {
        e = launch_knorm_fused(d, p->dtype, K, V, K_out, V_out, idx_out, scores_out, ws, st);
        if (e != cudaErrorNotSupported) return e == cudaSuccess ? KVP_OK : fail_cuda(e);
    }
    e = launch_knorm_score(d, p->dtype, K, ws, scores_out, true, st);
    if (e != cudaSuccess) return fail_cuda(e);
    return select_and_compact(d, K, V, K_out, V_out, idx_out, ws, st);
}

// ---- KeyDiff -------------------------------------------------------------------------------------
int kvp_keydiff_score(const kvp_problem* p, const void* K, void* scores_out, void* workspace,
                      size_t workspace_bytes, kvp_stream_t stream) {
    Dims d;
    int rc = validate(p, &d);
    if (rc) return rc;
    if (!K || !scores_out) return KVP_ERR_NULL_POINTER;
    if (!aligned16(K)) return KVP_ERR_BAD_STRIDE;
    Workspace ws;
    WsLayout L;
    if ((rc = carve(d, KVP_SCORER_KEYDIFF, 0, workspace, workspace_bytes, &ws, &L))) return rc;
    cudaError_t e = launch_keydiff_score(d, p->dtype, K, ws, scores_out, false, static_cast<cudaStream_t>(stream));
    if (e == cudaErrorNotSupported) return KVP_ERR_UNSUPPORTED_SHAPE;
    return e == cudaSuccess ? KVP_OK : fail_cuda(e);
}

int kvp_keydiff_compress(const kvp_problem* p, const void* K, const void* V, void* K_out, void* V_out,
                         int32_t* idx_out, void* scores_out, void* workspace, size_t workspace_bytes,
                         kvp_stream_t stream) {
    Dims d;
    int rc = validate(p, &d);
    if (rc) return rc;
    if (d.n_kept == 0) return KVP_OK;
    if ((rc = check_io(K, V, K_out, V_out))) return rc;
    Workspace ws;
    WsLayout L;
    if ((rc = carve(d, KVP_SCORER_KEYDIFF, 0, workspace, workspace_bytes, &ws, &L))) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    cudaError_t e = cudaMemsetAsync(ws.hist_hi, 0, L.hist_bytes, st);
    if (e != cudaSuccess) return fail_cuda(e);
    e = launch_keydiff_score(d, p->dtype, K, ws, scores_out, true, st);
    if (e == cudaErrorNotSupported) return KVP_ERR_UNSUPPORTED_SHAPE;
    if (e != cudaSuccess) return fail_cuda(e);
    return select_and_compact(d, K, V, K_out, V_out, idx_out, ws, st);
}

// ---- StreamingLLM --------------------------------------------------------------------------------
int kvp_streaming_score(const kvp_problem* p, int32_t n_sink, void* scores_out,
                        kvp_stream_t stream) {
    Dims d;
    int rc = validate(p, &d, false);
    if (rc) return rc;
    if (!scores_out) return KVP_ERR_NULL_POINTER;
    if (n_sink < 0) return KVP_ERR_BAD_ARGUMENT;
    cudaError_t e = launch_streaming_score(d, p->dtype, n_sink, scores_out,
                                           static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? KVP_OK : fail_cuda(e);
}

int kvp_streaming_compress(const kvp_problem* p, int32_t n_sink, const void* K, const void* V,
                           void* K_out, void* V_out, int32_t* idx_out, kvp_stream_t stream) {
    Dims d;
    int rc = validate(p, &d);
    if (rc) return rc;
    if (n_sink < 0) return KVP_ERR_BAD_ARGUMENT;
    if (d.n_kept == 0) return KVP_OK;
    if ((rc = check_io(K, V, K_out, V_out))) return rc;
    cudaError_t e = launch_streaming_compress(d, n_sink, K, V, K_out, V_out, idx_out,
                                              static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? KVP_OK : fail_cuda(e);
}

// ---- SnapKV --------------------------------------------------------------------------------------
int kvp_snapkv_score(const kvp_problem* p, const void* K, const void* q_window, int32_t window,
                     int32_t kernel_size, void* scores_out, void* workspace,
                     size_t workspace_bytes, kvp_stream_t stream) {
    Dims d;
    int rc = validate(p, &d);
    if (rc) return rc;
    if (!K || !q_window || !scores_out) return KVP_ERR_NULL_POINTER;
    if (!aligned16(K) || !aligned16(q_window)) return KVP_ERR_BAD_STRIDE;
    if (window <= 0 || window >= d.S || kernel_size <= 0 || (kernel_size & 1) == 0)
        return KVP_ERR_BAD_ARGUMENT;
    Workspace ws;
    WsLayout L;
    if ((rc = carve(d, KVP_SCORER_SNAPKV, window, workspace, workspace_bytes, &ws, &L))) return rc;
    cudaError_t e = cudaMemsetAsync(ws.hist_hi, 0, L.hist_bytes, static_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return fail_cuda(e);
    e = launch_snapkv_score(d, p->dtype, K, q_window, window, kernel_size, ws, scores_out, false,
                            static_cast<cudaStream_t>(stream));
    if (e == cudaErrorNotSupported) return KVP_ERR_UNSUPPORTED_SHAPE;
    return e == cudaSuccess ? KVP_OK : fail_cuda(e);
}

int kvp_snapkv_compress(const kvp_problem* p, const void* K, const void* V,
                        const void* q_window, int32_t window, int32_t kernel_size, void* K_out,
                        void* V_out, int32_t* idx_out, void* scores_out, void* workspace,
                        size_t workspace_bytes, kvp_stream_t stream) {
    Dims d;
    int rc = validate(p, &d);
    if (rc) return rc;
    if (d.n_kept == 0) return KVP_OK;
    if ((rc = check_io(K, V, K_out, V_out))) return rc;
    if (!q_window) return KVP_ERR_NULL_POINTER;
    if (!aligned16(q_window)) return KVP_ERR_BAD_STRIDE;
    if (window <= 0 || window >= d.S || kernel_size <= 0 || (kernel_size & 1) == 0)
        return KVP_ERR_BAD_ARGUMENT;
    Workspace ws;
    WsLayout L;
    if ((rc = carve(d, KVP_SCORER_SNAPKV, window, workspace, workspace_bytes, &ws, &L))) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    cudaError_t e = cudaMemsetAsync(ws.hist_hi, 0, L.hist_bytes, st);
    if (e != cudaSuccess) return fail_cuda(e);
    e = launch_snapkv_score(d, p->dtype, K, q_window, window, kernel_size, ws, scores_out, true,
                            st);
    if (e == cudaErrorNotSupported) return KVP_ERR_UNSUPPORTED_SHAPE;
    if (e != cudaSuccess) return fail_cuda(e);
    return select_and_compact(d, K, V, K_out, V_out, idx_out, ws, st);
}

// ---- ExpectedAttention ---------------------------------------------------------------------------
int kvp_expected_attention_score(const kvp_problem* p, const void* K, const void* V,
                                 const void* mu, const void* cov, float epsilon, int32_t n_sink,
                                 int32_t use_vnorm, void* scores_out, void* workspace,
                                 size_t workspace_bytes, kvp_stream_t stream) {
    Dims d;
    int rc = validate(p, &d);
    if (rc) return rc;
    if (!K || !mu || !scores_out || (use_vnorm && !V)) return KVP_ERR_NULL_POINTER;
    if (!aligned16(K) || !aligned16(mu) || (cov && !aligned16(cov))) return KVP_ERR_BAD_STRIDE;
    if (n_sink < 0 || n_sink >= d.S) return KVP_ERR_BAD_ARGUMENT;
    Workspace ws;
    WsLayout L;
    if ((rc = carve(d, KVP_SCORER_EXPECTED_ATTENTION, 0, workspace, workspace_bytes, &ws, &L)))
        return rc;
    cudaError_t e = cudaMemsetAsync(ws.hist_hi, 0, L.hist_bytes, static_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return fail_cuda(e);
    e = launch_ea_score(d, p->dtype, K, V, mu, cov, epsilon, n_sink, use_vnorm, ws, scores_out, false,
                        static_cast<cudaStream_t>(stream));
    if (e == cudaErrorNotSupported) return KVP_ERR_UNSUPPORTED_SHAPE;
    return e == cudaSuccess ? KVP_OK : fail_cuda(e);
}

int kvp_expected_attention_compress(const kvp_problem* p, const void* K, const void* V,
                                    const void* mu, const void* cov, float epsilon,
                                    int32_t n_sink, int32_t use_vnorm, void* K_out, void* V_out,
                                    int32_t* idx_out, void* scores_out, void* workspace,
                                    size_t workspace_bytes, kvp_stream_t stream) {
    Dims d;
    int rc = validate(p, &d);
    if (rc) return rc;
    if (d.n_kept == 0) return KVP_OK;
    if ((rc = check_io(K, V, K_out, V_out))) return rc;
    if (!mu) return KVP_ERR_NULL_POINTER;
    if (!aligned16(mu) || (cov && !aligned16(cov))) return KVP_ERR_BAD_STRIDE;
    if (n_sink < 0 || n_sink >= d.S) return KVP_ERR_BAD_ARGUMENT;
    Workspace ws;
    WsLayout L;
    if ((rc = carve(d, KVP_SCORER_EXPECTED_ATTENTION, 0, workspace, workspace_bytes, &ws, &L)))
        return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    cudaError_t e = cudaMemsetAsync(ws.hist_hi, 0, L.hist_bytes, st);
    if (e != cudaSuccess) return fail_cuda(e);
    e = launch_ea_score(d, p->dtype, K, V, mu, cov, epsilon, n_sink, use_vnorm, ws, scores_out,
                        true, st);
    if (e == cudaErrorNotSupported) return KVP_ERR_UNSUPPORTED_SHAPE;
    if (e != cudaSuccess) return fail_cuda(e);
    return select_and_compact(d, K, V, K_out, V_out, idx_out, ws, st);
}

// ---- generic scores ------------------------------------------------------------------------------
int kvp_scores_compress(const kvp_problem* p, const void* scores, const int64_t* score_stride,
                        const void* K, const void* V, void* K_out, void* V_out,
                        int32_t* idx_out, void* workspace, size_t workspace_bytes,
                        kvp_stream_t stream) {
    Dims d;
    int rc = validate(p, &d, true, kMaxRowsGeneric);
    if (rc) return rc;
    if (d.n_kept == 0) return KVP_OK;
    if ((rc = check_io(K, V, K_out, V_out))) return rc;
    if (!scores || !score_stride) return KVP_ERR_NULL_POINTER;
    Workspace ws;
    WsLayout L;
    if ((rc = carve(d, KVP_SCORER_GENERIC, 0, workspace, workspace_bytes, &ws, &L))) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    cudaError_t e = cudaMemsetAsync(ws.hist_hi, 0, L.hist_bytes, st);
    if (e != cudaSuccess) return fail_cuda(e);
    e = launch_keys_from_scores(d, p->dtype, scores, score_stride[0], score_stride[1], ws, st);
    if (e != cudaSuccess) return fail_cuda(e);
    return select_and_compact(d, K, V, K_out, V_out, idx_out, ws, st);
}

int kvp_scores_select(const kvp_problem* p, const void* scores, const int64_t* score_stride,
                      int32_t* idx_out, void* workspace, size_t workspace_bytes, kvp_stream_t stream) {
    Dims d;
    int rc = validate(p, &d, false, kMaxRowsGeneric);
    if (rc) return rc;
    if (d.n_kept == 0) return KVP_OK;
    if (!scores || !score_stride || !idx_out) return KVP_ERR_NULL_POINTER;
    Workspace ws;
    WsLayout L;
    if ((rc = carve(d, KVP_SCORER_GENERIC, 0, workspace, workspace_bytes, &ws, &L))) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    cudaError_t e = cudaMemsetAsync(ws.hist_hi, 0, L.hist_bytes, st);
    if (e != cudaSuccess) return fail_cuda(e);
    e = launch_keys_from_scores(d, p->dtype, scores, score_stride[0], score_stride[1], ws, st);
    if (e != cudaSuccess) return fail_cuda(e);
    d.ks = d.vs = {0, 0, 0};
    return select_and_compact(d, nullptr, nullptr, nullptr, nullptr, idx_out, ws, st);
}

int kvp_scores_compress_rerotate(const kvp_problem* p, const void* scores, const int64_t* score_stride,
                                 const void* K, const void* V, const float* inv_freq, void* K_out,
                                 void* V_out, int32_t* idx_out, void* workspace,
                                 size_t workspace_bytes, kvp_stream_t stream) {
    Dims d;
    int rc = validate(p, &d, true, kMaxRowsGeneric);
    if (rc) return rc;
    if (d.D % 16 != 0) return KVP_ERR_UNSUPPORTED_SHAPE;  // rotate_half pairs d with d + D/2
    if (d.n_kept == 0) return KVP_OK;
    if ((rc = check_io(K, V, K_out, V_out))) return rc;
    if (!scores || !score_stride || !inv_freq) return KVP_ERR_NULL_POINTER;
    Workspace ws;
    WsLayout L;
    if ((rc = carve(d, KVP_SCORER_GENERIC, 0, workspace, workspace_bytes, &ws, &L))) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    cudaError_t e = cudaMemsetAsync(ws.hist_hi, 0, L.hist_bytes, st);
    if (e != cudaSuccess) return fail_cuda(e);
    e = launch_keys_from_scores(d, p->dtype, scores, score_stride[0], score_stride[1], ws, st);
    if (e != cudaSuccess) return fail_cuda(e);
    e = launch_select_compact_rerotate(d, p->dtype, K, V, K_out, V_out, idx_out, ws, inv_freq, st);
    return e == cudaSuccess ? KVP_OK : fail_cuda(e);
}

}  // extern "C"
