// keydiff.cu — KeyDiffPress scores (SURVEY §8f row 3; reference kvpress/presses/keydiff_press.py:36-46):
//     anchor = mean_s( k_s / max(||k_s||, 1e-12) )                      (F.normalize, then mean over positions)
//     score_s = -cos(k_s, anchor) = -(k_s . anchor) / (max(||k_s||, 1e-8) * max(||anchor||, 1e-8))
// evaluated in fp32 and rounded ONCE to the cache dtype (the reference rounds to 16 bits after every ATen op).
//
// HBM-bound, two streaming passes over K (the anchor needs every key before any score exists):
//   pass 1  keydiff_anchor_kernel  grid (chunks, rows): 256 positions per CTA, a sub-warp of LPR lanes per row,
//           every lane owns 8 fixed head-dim elements -> register accumulators of k/||k||; deterministic tree
//           (shuffles, shared memory, one partial [D] per CTA in the workspace)
//   merge   keydiff_merge_kernel   grid (rows): fixed-order sum of the partials, 1/S, ||anchor||
//   pass 2  keydiff_score_kernel   grid (chunks, rows): dot + norm per position, one rounding, ordered keys +
//           histogram for the shared select+compact stage
// Algorithmic bytes per (b, kv-head): row * (2 S + 3 n_kept) — K is read twice by construction.
#include "common.cuh"
#include "knorm_chunk.cuh"

#ifndef KVP_KD_BUTTERFLY
#define KVP_KD_BUTTERFLY 0
#endif

namespace kvp {

struct KeyDiffScratch {
    float* partial;  // [R][n_chunks][D]
    float* anchor;   // [R][D]  mean of the normalised keys
    float* anorm;    // [R]     max(||anchor||, 1e-8)
};

static inline size_t kd_align256(size_t x) { return (x + 255) / 256 * 256; }

size_t keydiff_scratch_bytes(const Dims& d) {
    const size_t n_chunks = (size_t)((d.S + kScoreChunk - 1) / kScoreChunk);
    return kd_align256((size_t)d.R * n_chunks * d.D * 4) + kd_align256((size_t)d.R * d.D * 4) +
           kd_align256((size_t)d.R * 4);
}

static KeyDiffScratch carve_keydiff(const Dims& d, const Workspace& ws) {
    const size_t n_chunks = (size_t)((d.S + kScoreChunk - 1) / kScoreChunk);
    char* p = static_cast<char*>(ws.scorer);
    KeyDiffScratch s;
    s.partial = reinterpret_cast<float*>(p);
    p += kd_align256((size_t)d.R * n_chunks * d.D * 4);
    s.anchor = reinterpret_cast<float*>(p);
    p += kd_align256((size_t)d.R * d.D * 4);
    s.anorm = reinterpret_cast<float*>(p);
    return s;
}

// ---- pass 1: per-CTA partial sums of the normalised keys ------------------------------------------
template <typename T, int LPR>
__global__ void __launch_bounds__(kTileThreads)
keydiff_anchor_kernel(const T* __restrict__ K, Strides3 ks, int H, int S, int D, int n_chunks,
                      KeyDiffScratch sc) {
    __shared__ float s_part[kTileThreads / 32][LPR * 8];
    const int chunk = blockIdx.x, row = blockIdx.y;
    const int b = row / H, h = row % H;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    constexpr int RPW = 32 / LPR;
    constexpr int TOK_PER_WARP = kScoreChunk / (kTileThreads / 32);
    constexpr int ITERS = TOK_PER_WARP / RPW;
    constexpr int U = (ITERS < 4) ? ITERS : 4;
    static_assert(ITERS % U == 0, "unroll must divide the iteration count");
    const int sub = lane % LPR, rsel = lane / LPR;
    const int nvec = D >> 3;
    const T* base = K + (int64_t)b * ks.b + (int64_t)h * ks.h + (int64_t)sub * 8;
    const int s_warp = chunk * kScoreChunk + warp * TOK_PER_WARP;
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = 0.f;
#pragma unroll 1
    for (int it = 0; it < ITERS; it += U) {
        int4 v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int s = s_warp + (it + u) * RPW + rsel;
            v[u] = make_int4(0, 0, 0, 0);
            if (s < S && sub < nvec) v[u] = ldg_plain(base + (int64_t)s * ks.s);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint32_t w[4] = {(uint32_t)v[u].x, (uint32_t)v[u].y, (uint32_t)v[u].z, (uint32_t)v[u].w};
            float f[8];
            float ss = 0.f;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float2 p = F16Traits<T>::unpack2(w[j]);
                f[2 * j] = p.x;
                f[2 * j + 1] = p.y;
                ss = fmaf(p.x, p.x, ss);
                ss = fmaf(p.y, p.y, ss);
            }
#pragma unroll
            for (int off = LPR / 2; off >= 1; off >>= 1) ss += __shfl_xor_sync(0xFFFFFFFFu, ss, off);
            const float inv = 1.f / fmaxf(sqrtf(ss), 1e-12f);  // rows past S are all-zero: contribute 0
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[j] = fmaf(f[j], inv, acc[j]);
        }
    }
    // lanes with the same `sub` (different rows) meet: xor over the row-select bits
#pragma unroll
    for (int off = LPR; off < 32; off <<= 1)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] += __shfl_xor_sync(0xFFFFFFFFu, acc[j], off);
    if (rsel == 0)
#pragma unroll
        for (int j = 0; j < 8; ++j) s_part[warp][sub * 8 + j] = acc[j];
    __syncthreads();
    if (tid < D) {
        float t = 0.f;
#pragma unroll
        for (int w = 0; w < kTileThreads / 32; ++w) t += s_part[w][tid];
        sc.partial[((size_t)row * n_chunks + chunk) * D + tid] = t;
    }
}

// ---- merge: anchor = (sum of partials) / S, ||anchor|| --------------------------------------------
// One CTA of 1024 threads per row: G = 1024 / D_pad thread groups, group g sums the chunks c = g, g+G, ... in
// a fixed order (4 chains), the groups meet in shared memory in a fixed order -> deterministic, and the serial
// chain per thread is n_chunks / G long instead of n_chunks (26 us -> a few us at 128k).
constexpr int kKdMergeThreads = 1024;
__global__ void __launch_bounds__(kKdMergeThreads)
keydiff_merge_kernel(int S, int D, int n_chunks, KeyDiffScratch sc) {
    __shared__ float s_grp[kKdMergeThreads];
    __shared__ float s_sq[256];
    const int row = blockIdx.x, tid = threadIdx.x;
    const int d_pad = (D <= 32) ? 32 : (D <= 64) ? 64 : (D <= 128) ? 128 : 256;
    const int G = kKdMergeThreads / d_pad;
    const int g = tid / d_pad, dd = tid % d_pad;
    float t = 0.f;
    if (dd < D) {
        const float* p = sc.partial + (size_t)row * n_chunks * D + dd;
        float t0 = 0.f, t1 = 0.f, t2 = 0.f, t3 = 0.f;
        int c = g;
        for (; c + 3 * G < n_chunks; c += 4 * G) {
            t0 += p[(size_t)c * D];
            t1 += p[(size_t)(c + G) * D];
            t2 += p[(size_t)(c + 2 * G) * D];
            t3 += p[(size_t)(c + 3 * G) * D];
        }
        for (; c < n_chunks; c += G) t0 += p[(size_t)c * D];
        t = (t0 + t1) + (t2 + t3);
    }
    s_grp[tid] = t;
    __syncthreads();
    float a = 0.f;
    if (tid < D) {
        for (int gg = 0; gg < G; ++gg) a += s_grp[gg * d_pad + tid];
        a /= (float)S;
        sc.anchor[(size_t)row * D + tid] = a;
    }
    if (tid < 256) s_sq[tid] = a * a;
    __syncthreads();
    for (int off = 128; off >= 1; off >>= 1) {
        if (tid < off) s_sq[tid] += s_sq[tid + off];
        __syncthreads();
    }
    if (tid == 0) sc.anorm[row] = fmaxf(sqrtf(s_sq[0]), 1e-8f);
}

// ---- pass 2: scores, keys, histogram ---------------------------------------------------------------
template <typename T, int LPR>
__global__ void __launch_bounds__(kTileThreads)
keydiff_score_kernel(const T* __restrict__ K, Strides3 ks, int H, int S, int D, KeyDiffScratch sc,
                     Workspace ws, uint16_t* __restrict__ scores_out, int want_keys) {
    __shared__ uint16_t skeys[kScoreChunk];
    __shared__ uint16_t sscores[kScoreChunk];
    __shared__ uint32_t shist[256];
    const int chunk = blockIdx.x, row = blockIdx.y;
    const int b = row / H, h = row % H;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    shist[tid] = 0;
    pdl_launch_dependents();  // the selection pass behind this one may start to take residency
    constexpr int RPW = 32 / LPR;
    constexpr int TOK_PER_WARP = kScoreChunk / (kTileThreads / 32);
    constexpr int ITERS = TOK_PER_WARP / RPW;
    constexpr int U = (ITERS < 8) ? ITERS : 8;
    static_assert(ITERS % U == 0, "unroll must divide the iteration count");
    const int sub = lane % LPR, rsel = lane / LPR;
    const int nvec = D >> 3;
    const T* base = K + (int64_t)b * ks.b + (int64_t)h * ks.h + (int64_t)sub * 8;
    const int s_warp = chunk * kScoreChunk + warp * TOK_PER_WARP;
    float a[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) a[j] = (sub < nvec) ? __ldg(sc.anchor + (size_t)row * D + sub * 8 + j) : 0.f;
    const float inv_anorm = 1.f / __ldg(sc.anorm + row);
#pragma unroll 1
    for (int it = 0; it < ITERS; it += U) {
        int4 v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int s = s_warp + (it + u) * RPW + rsel;
            v[u] = make_int4(0, 0, 0, 0);
            if (s < S && sub < nvec) v[u] = ldg_plain(base + (int64_t)s * ks.s);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint32_t w[4] = {(uint32_t)v[u].x, (uint32_t)v[u].y, (uint32_t)v[u].z, (uint32_t)v[u].w};
            float ss = 0.f, dot = 0.f;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float2 p = F16Traits<T>::unpack2(w[j]);
                ss = fmaf(p.x, p.x, ss);
                ss = fmaf(p.y, p.y, ss);
                dot = fmaf(p.x, a[2 * j], dot);
                dot = fmaf(p.y, a[2 * j + 1], dot);
            }
#if KVP_KD_BUTTERFLY
            // prepared experiment (default off, see DESIGN §5.3): one butterfly for both sums — after the first
            // exchange the lower half of the sub-warp owns ss and the upper half owns dot; log2(LPR)+1 shuffles
            // instead of 2*log2(LPR)
            {
                constexpr int HALF = LPR / 2;
                const bool upper = (sub & HALF) != 0;
                float keep = upper ? dot : ss;
                keep += __shfl_xor_sync(0xFFFFFFFFu, upper ? ss : dot, HALF);
#pragma unroll
                for (int off = HALF / 2; off >= 1; off >>= 1) keep += __shfl_xor_sync(0xFFFFFFFFu, keep, off);
                const float other = __shfl_xor_sync(0xFFFFFFFFu, keep, HALF);
                ss = upper ? other : keep;
                dot = upper ? keep : other;
            }
#else
#pragma unroll
            for (int off = LPR / 2; off >= 1; off >>= 1) {
                ss += __shfl_xor_sync(0xFFFFFFFFu, ss, off);
                dot += __shfl_xor_sync(0xFFFFFFFFu, dot, off);
            }
#endif
            if (sub == 0) {
                const int sl = warp * TOK_PER_WARP + (it + u) * RPW + rsel;
                const float cosv = dot / fmaxf(sqrtf(ss), 1e-8f) * inv_anorm;
                const uint16_t bits = F16Traits<T>::from_float(-cosv);
                sscores[sl] = bits;
                skeys[sl] = ordered_key16(bits, F16Traits<T>::kInfBits);
            }
        }
    }
    __syncthreads();
    const int s_begin = chunk * kScoreChunk;
    if (want_keys) {
        flush_chunk_keys<1>(skeys, sscores, shist, row, s_begin, S, ws, scores_out);
    } else if (s_begin + tid < S) {
        scores_out[(size_t)row * S + s_begin + tid] = sscores[tid];
    }
}

template <typename T>
static cudaError_t launch_keydiff_t(const Dims& d, const void* K, const Workspace& ws, void* scores_out,
                                    bool want_keys, cudaStream_t st) {
    if (d.D > 256) return cudaErrorNotSupported;
    const KeyDiffScratch sc = carve_keydiff(d, ws);
    const int n_chunks = (d.S + kScoreChunk - 1) / kScoreChunk;
    dim3 grid(n_chunks, d.R);
    const int nvec = d.D / 8;
    const T* Kp = static_cast<const T*>(K);
    uint16_t* so = static_cast<uint16_t*>(scores_out);
#define KVP_KD_ANCHOR(LPR) \
    keydiff_anchor_kernel<T, LPR><<<grid, kTileThreads, 0, st>>>(Kp, d.ks, d.H, d.S, d.D, n_chunks, sc)
#define KVP_KD_SCORE(LPR) \
    keydiff_score_kernel<T, LPR><<<grid, kTileThreads, 0, st>>>(Kp, d.ks, d.H, d.S, d.D, sc, ws, so, want_keys ? 1 : 0)
    if (nvec <= 4) KVP_KD_ANCHOR(4);
    else if (nvec <= 8) KVP_KD_ANCHOR(8);
    else if (nvec <= 16) KVP_KD_ANCHOR(16);
    else KVP_KD_ANCHOR(32);
    cudaError_t e = cudaPeekAtLastError();
    if (e != cudaSuccess) return e;
    keydiff_merge_kernel<<<d.R, kKdMergeThreads, 0, st>>>(d.S, d.D, n_chunks, sc);
    if ((e = cudaPeekAtLastError()) != cudaSuccess) return e;
    if (nvec <= 4) KVP_KD_SCORE(4);
    else if (nvec <= 8) KVP_KD_SCORE(8);
    else if (nvec <= 16) KVP_KD_SCORE(16);
    else KVP_KD_SCORE(32);
#undef KVP_KD_ANCHOR
#undef KVP_KD_SCORE
    return cudaPeekAtLastError();
}

cudaError_t launch_keydiff_score(const Dims& d, int dtype, const void* K, const Workspace& ws,
                                 void* scores_out, bool want_keys, cudaStream_t st) {
    if (dtype == KVP_BF16) return launch_keydiff_t<__nv_bfloat16>(d, K, ws, scores_out, want_keys, st);
    return launch_keydiff_t<__half>(d, K, ws, scores_out, want_keys, st);
}

}  // namespace kvp
