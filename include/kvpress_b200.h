/*
 * kvpress_b200.h — C ABI of the B200-native fused KV-cache compression path.
 *
 * The reference (NVIDIA/kvpress, pure Python/PyTorch) has no FFI: its hot path is the ATen
 * sequence inside ScorerPress.compress (kvpress/presses/scorer_press.py:76-102):
 *     scores = self.score(...)                     (:90)   per-scorer, see below
 *     n_kept = int(k_len * (1 - ratio))            (:93-94) computed by the HOST and passed in
 *     indices = scores.topk(n_kept).indices        (:95)
 *     keys/values.gather(2, indices).contiguous()  (:99-100)
 * Every entry point below replaces that sequence (or its score() part) for one scorer:
 *     kvp_knorm_*              <- kvpress/presses/knorm_press.py:29-38
 *     kvp_streaming_*          <- kvpress/presses/streaming_llm_press.py:38-54
 *     kvp_snapkv_*             <- kvpress/presses/snapkv_press.py:41-105
 *     kvp_expected_attention_* <- kvpress/presses/expected_attention_press.py:126-165
 *     kvp_keydiff_*            <- kvpress/presses/keydiff_press.py:36-46
 *     kvp_scores_compress      <- scorer_press.py:93-100 for an arbitrary score tensor
 *                                 (what wrapper presses / user ScorerPress subclasses need)
 *
 * Conventions
 *   - All pointers are DEVICE pointers unless a name ends in _host. Nothing here is a torch type.
 *   - K, V: [B, Hkv, S, D], 16-bit floats (bf16 or fp16), innermost dim contiguous, outer dims
 *     arbitrary element strides (kvp_problem.k_stride / v_stride), 16-byte aligned rows.
 *   - Outputs K_out, V_out: contiguous [B, Hkv, n_kept, D]; rows in ASCENDING POSITION order
 *     (the reference emits score-descending order; attention is permutation invariant over
 *     (K,V) rows — see DESIGN.md "row order").
 *   - idx_out (nullable): int32 [B, Hkv, n_kept], the kept positions, ascending.
 *   - scores_out (nullable): [B, Hkv, S] in the K dtype, same values the reference's score()
 *     returns (including the max+1 sentinel on forced-keep positions).
 *   - Selection rule: the n_kept largest scores per (b, h) row; ties at the threshold are
 *     resolved towards the LOWEST position (deterministic; torch.topk leaves it unspecified).
 *   - Caller owns all memory (outputs + workspace of kvp_workspace_bytes()). The library
 *     allocates no device memory and never synchronises the stream (kvp_workspace_check excepted). Process-wide state is limited to write-once caches of device
 *     properties (SM count, occupancy, function attributes) and, for the covariance-free ExpectedAttention
 *     scan with use_vnorm (the tensor-core kernels take the value norms themselves), ONE internal side
 *     stream + two events per device: the ||v|| kernel is forked onto it
 *     and joined back into the caller's stream before the call returns; host threads enqueueing
 *     ExpectedAttention calls on the same device serialise on a mutex for those few microseconds.
 *     Calls are re-entrant per (stream, workspace); every call is CUDA-graph capturable.
 *   - Return value: KVP_OK (0) or a negative kvp_status. No exceptions cross this boundary.
 */
#ifndef KVPRESS_B200_H
#define KVPRESS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KVP_ABI_VERSION 1

typedef void* kvp_stream_t; /* a cudaStream_t */

typedef enum kvp_status {
    KVP_OK = 0,
    KVP_ERR_NULL_POINTER = -1,
    KVP_ERR_UNSUPPORTED_SHAPE = -2,
    KVP_ERR_UNSUPPORTED_DTYPE = -3,
    KVP_ERR_BAD_STRIDE = -4,
    KVP_ERR_WORKSPACE_TOO_SMALL = -5,
    KVP_ERR_CUDA = -6,
    KVP_ERR_BAD_ARGUMENT = -7,
    KVP_ERR_KERNEL_TIMEOUT = -8 /* a kernel abandoned a bounded wait: outputs invalid (library bug) */
} kvp_status;

typedef enum kvp_dtype { KVP_BF16 = 0, KVP_F16 = 1 } kvp_dtype;

typedef enum kvp_scorer {
    KVP_SCORER_GENERIC = 0, /* scores supplied by the caller            */
    KVP_SCORER_KNORM = 1,
    KVP_SCORER_STREAMING = 2,
    KVP_SCORER_SNAPKV = 3,
    KVP_SCORER_EXPECTED_ATTENTION = 4,
    KVP_SCORER_KEYDIFF = 5
} kvp_scorer;

/* One ScorerPress.compress call on one layer's cache. */
typedef struct kvp_problem {
    int32_t B;      /* batch                                                         */
    int32_t Hkv;    /* key/value heads                                               */
    int32_t Hq;     /* query heads (multiple of Hkv; = Hkv when the scorer has no Q) */
    int32_t S;      /* k_len, cached positions                                       */
    int32_t D;      /* head_dim (multiple of 8, <= 256)                              */
    int32_t n_kept; /* int(S * (1 - compression_ratio)), computed by the host        */
    int32_t dtype;  /* kvp_dtype of K, V, scores, Q, mu, cov                         */
    int32_t reserved;
    int64_t k_stride[3]; /* element strides of K for (b, h, s); stride of d is 1 */
    int64_t v_stride[3]; /* element strides of V for (b, h, s)                   */
} kvp_problem;

/* ---- library info ---------------------------------------------------------------------- */
int kvp_abi_version(void);
const char* kvp_status_string(int status);
/* Last CUDA error string recorded on this host thread by a failed call (never NULL). */
const char* kvp_last_cuda_error(void);

/* Bytes of scratch a *_compress / *_score call of this scorer needs (256-byte aligned). */
int kvp_workspace_bytes(const kvp_problem* p, int scorer, size_t* bytes_out);

/* Debugging aid. The work items of the persistent Knorm kernel wait on each other with BOUNDED spins; a wait that
 * expires raises a flag in the workspace instead of trapping the CUDA context. This call synchronises
 * `stream`, reads the flag of the last call that used `workspace` and returns KVP_OK or
 * KVP_ERR_KERNEL_TIMEOUT. Never needed for correct operation. */
int kvp_workspace_check(const kvp_problem* p, int scorer, const void* workspace, size_t workspace_bytes,
                        kvp_stream_t stream);

/* Number of kernel launches (incl. memset nodes) one *_compress call enqueues; bench.py
 * reports it as gpu_launches. */
int kvp_launches_per_compress(const kvp_problem* p, int scorer, int* launches_out);

/* ---- KnormPress: score = -||k||_2 (fp32 accumulate, one rounding to the K dtype) ------- */
int kvp_knorm_score(const kvp_problem* p, const void* K, void* scores_out, kvp_stream_t stream);
int kvp_knorm_compress(const kvp_problem* p, const void* K, const void* V, void* K_out,
                       void* V_out, int32_t* idx_out, void* scores_out, void* workspace,
                       size_t workspace_bytes, kvp_stream_t stream);

/* ---- StreamingLLMPress: keep [0, n_sink) and the most recent positions ------------------ */
int kvp_streaming_score(const kvp_problem* p, int32_t n_sink, void* scores_out,
                        kvp_stream_t stream);
int kvp_streaming_compress(const kvp_problem* p, int32_t n_sink, const void* K, const void* V,
                           void* K_out, void* V_out, int32_t* idx_out, kvp_stream_t stream);

/* ---- SnapKVPress -------------------------------------------------------------------------
 * q_window: RoPE'd queries of the last `window` positions, contiguous [B, Hq, window, D]
 * (snapkv_press.py:53-58 — the 64-row q_proj GEMM + RoPE is the caller's prologue).
 * Scores: softmax over all S keys (causal inside the window) of q·k/sqrt(D), mean over the
 * window queries, avg_pool1d(kernel_size, pad=kernel_size/2, stride 1, divisor kernel_size),
 * mean over the Hq/Hkv group; the last `window` positions are always kept. */
int kvp_snapkv_score(const kvp_problem* p, const void* K, const void* q_window, int32_t window,
                     int32_t kernel_size, void* scores_out, void* workspace,
                     size_t workspace_bytes, kvp_stream_t stream);
int kvp_snapkv_compress(const kvp_problem* p, const void* K, const void* V,
                        const void* q_window, int32_t window, int32_t kernel_size, void* K_out,
                        void* V_out, int32_t* idx_out, void* scores_out, void* workspace,
                        size_t workspace_bytes, kvp_stream_t stream);

/* ---- ExpectedAttentionPress --------------------------------------------------------------
 * mu: [B, Hq, D], cov: [B, Hq, D, D] (nullable = use_covariance False), both already rotated
 * by the average RoPE matrix (expected_attention_press.py:62-124 — the query-statistics
 * prologue stays with the caller). Scores over positions [n_sink, S):
 *   softmax_s( mu·k/sqrt(D) + k^T cov k / (2 D) ), mean over the group, (+eps) * ||v||_2 when
 *   use_vnorm; the first n_sink positions are always kept. */
int kvp_expected_attention_score(const kvp_problem* p, const void* K, const void* V,
                                 const void* mu, const void* cov, float epsilon, int32_t n_sink,
                                 int32_t use_vnorm, void* scores_out, void* workspace,
                                 size_t workspace_bytes, kvp_stream_t stream);
int kvp_expected_attention_compress(const kvp_problem* p, const void* K, const void* V,
                                    const void* mu, const void* cov, float epsilon,
                                    int32_t n_sink, int32_t use_vnorm, void* K_out, void* V_out,
                                    int32_t* idx_out, void* scores_out, void* workspace,
                                    size_t workspace_bytes, kvp_stream_t stream);

/* ---- generic: top-k + compaction of caller-supplied scores ------------------------------
 * scores: [B, Hkv, S] in the K dtype with element strides score_stride (b, h; s contiguous). */
int kvp_scores_compress(const kvp_problem* p, const void* scores, const int64_t* score_stride,
                        const void* K, const void* V, void* K_out, void* V_out,
                        int32_t* idx_out, void* workspace, size_t workspace_bytes,
                        kvp_stream_t stream);

/* ---- KeyDiffPress (kvpress/presses/keydiff_press.py:36-46): score = -cos(k, anchor), anchor = mean over
 * positions of k / ||k||; fp32 evaluation, one rounding to the K dtype. Two streaming passes over K. */
int kvp_keydiff_score(const kvp_problem* p, const void* K, void* scores_out, void* workspace,
                      size_t workspace_bytes, kvp_stream_t stream);
int kvp_keydiff_compress(const kvp_problem* p, const void* K, const void* V, void* K_out, void* V_out,
                         int32_t* idx_out, void* scores_out, void* workspace, size_t workspace_bytes,
                         kvp_stream_t stream);

/* ---- selection only: the n_kept best positions of every [S] score row, ascending, into idx_out
 * [B, Hkv, n_kept]; no K/V are touched (p->D and the K/V strides are ignored). What head-wise presses need:
 * AdaKVPress (kvpress/presses/adakv_press.py:53-78) = this call on the [B, Hkv, S] scores with n_safe, then
 * on the negated, head-flattened [B, 1, Hkv*S] scores with the number of positions to prune. */
int kvp_scores_select(const kvp_problem* p, const void* scores, const int64_t* score_stride,
                      int32_t* idx_out, void* workspace, size_t workspace_bytes, kvp_stream_t stream);

/* ---- KeyRerotationPress (SURVEY §8f, first "next" row): same selection as kvp_scores_compress, but each
 * kept key is re-rotated from its original position s to its new position j (kvpress/presses/
 * key_rerotation_press.py:50-152): k * cos((j-s) inv_freq) + rotate_half(k) * sin((j-s) inv_freq).
 * inv_freq: fp32 [D/2] (module.rotary_emb.inv_freq); D must be a multiple of 16. Values are copied as is. */
int kvp_scores_compress_rerotate(const kvp_problem* p, const void* scores, const int64_t* score_stride,
                                 const void* K, const void* V, const float* inv_freq, void* K_out,
                                 void* V_out, int32_t* idx_out, void* workspace,
                                 size_t workspace_bytes, kvp_stream_t stream);

/* Host buffers: every entry point takes DEVICE pointers (V may be pinned host memory for the scorers that do not read V to
 * score: the compaction kernel then gathers the kept V rows over PCIe). Staging whole caches from host memory through
 * these calls — per-kv-head chunks on three streams — is the host side's job: kvpress_b200/host_staging.py. */

#ifdef __cplusplus
}
#endif
#endif /* KVPRESS_B200_H */
