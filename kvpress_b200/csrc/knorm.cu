// knorm.cu — stage S for KnormPress and for caller-supplied scores.
//
// Reference semantics (kvpress/presses/knorm_press.py:38): scores = -keys.norm(dim=-1)
//   = -sqrt(sum_d k_d^2), accumulated in fp32, rounded ONCE to the K dtype.
// One CTA scores one tile of kTile positions of one (b, h) row with 128-bit loads
// (a sub-warp of LPR lanes per 2*D-byte row, U independent loads in flight per lane), stages
// the 16-bit ordered keys in shared memory, writes them coalesced and adds the tile's
// histogram of (key >> 8) to the row histogram the select stage starts from.
#include <stdlib.h>

#include "common.cuh"
#include "knorm_chunk.cuh"

namespace kvp {

template <typename T, int LPR>
__global__ void __launch_bounds__(kTileThreads)
knorm_score_kernel(const T* __restrict__ K, Strides3 ks, int H, int S, int D, Workspace ws,
                   uint16_t* __restrict__ scores_out, int want_keys, int keep_from_row) {
    __shared__ uint16_t skeys[kScoreChunk];
    __shared__ uint16_t sscores[kScoreChunk];
    __shared__ uint32_t shist[256];
    const int chunk = blockIdx.x, row = blockIdx.y, tid = threadIdx.x;
    shist[tid] = 0;  // kTileThreads == 256
    pdl_launch_dependents();  // the selection pass behind this one may start to take residency
    // L2 plan of a compress call (keep_from_row >= 0): the compaction stage re-reads the kept K rows, last rows first.
    // The rows it reaches while they can still be in L2 are loaded evict_last, the earlier ones evict_first, so that
    // the stream of early rows does not push the late ones out (profiles/r02_ab_knorm_l2.txt).
    if (keep_from_row < 0) knorm_score_chunk<T, LPR>(K, ks, row / H, row % H, chunk, S, D, skeys, sscores);
    else if (row >= keep_from_row) knorm_score_chunk<T, LPR, 1>(K, ks, row / H, row % H, chunk, S, D, skeys, sscores);
    else knorm_score_chunk<T, LPR, 2>(K, ks, row / H, row % H, chunk, S, D, skeys, sscores);
    __syncthreads();
    const int s_begin = chunk * kScoreChunk;
    if (want_keys) {
        flush_chunk_keys<1>(skeys, sscores, shist, row, s_begin, S, ws, scores_out);
    } else if (s_begin + tid < S) {  // score-only call
        scores_out[(size_t)row * S + s_begin + tid] = sscores[tid];
    }
}

template <typename T>
static cudaError_t launch_knorm_t(const Dims& d, const void* K, const Workspace& ws,
                                  void* scores_out, bool want_keys, cudaStream_t st) {
    dim3 grid((d.S + kScoreChunk - 1) / kScoreChunk, d.R);
    const int nvec = d.D / 8;
    const T* Kp = static_cast<const T*>(K);
    uint16_t* so = static_cast<uint16_t*>(scores_out);
    // rows whose K (row_bytes each) fits kKeepBytes of L2 at the end of the pass are kept for the compaction stage
    static const long long keep_mb = [] {  // A/B knob: KVP_KNORM_L2_KEEP_MB (default 0 = no hints: measured no gain)
        const char* v = getenv("KVP_KNORM_L2_KEEP_MB");
        return (long long)((v && *v) ? atoll(v) : 0);
    }();
    int keep_from_row = -1;
    const long long row_bytes = (long long)d.S * d.D * 2;
    if (want_keys && keep_mb > 0 && (long long)d.R * row_bytes > (keep_mb << 20)) {
        const long long n_keep = (keep_mb << 20) / row_bytes;
        keep_from_row = d.R - (int)n_keep;  // n_keep == 0: everything evict_first except nothing kept
        if (n_keep == 0) keep_from_row = -1;
    }
#define KVP_LAUNCH_KNORM(LPR)                                                                   \
    knorm_score_kernel<T, LPR><<<grid, kTileThreads, 0, st>>>(Kp, d.ks, d.H, d.S, d.D, ws, so, \
                                                              want_keys ? 1 : 0, keep_from_row)
    if (nvec <= 4) KVP_LAUNCH_KNORM(4);
    else if (nvec <= 8) KVP_LAUNCH_KNORM(8);
    else if (nvec <= 16) KVP_LAUNCH_KNORM(16);
    else KVP_LAUNCH_KNORM(32);
#undef KVP_LAUNCH_KNORM
    return cudaPeekAtLastError();
}

cudaError_t launch_knorm_score(const Dims& d, int dtype, const void* K, const Workspace& ws,
                               void* scores_out, bool want_keys, cudaStream_t st) {
    if (dtype == KVP_BF16)
        return launch_knorm_t<__nv_bfloat16>(d, K, ws, scores_out, want_keys, st);
    return launch_knorm_t<__half>(d, K, ws, scores_out, want_keys, st);
}

// ---- caller-supplied scores -> keys + histogram ------------------------------------------------
__global__ void __launch_bounds__(kTileThreads)
keys_from_scores_kernel(const uint16_t* __restrict__ scores, int64_t sb, int64_t sh, int H, int S,
                        uint16_t inf_bits, Workspace ws) {
    __shared__ uint16_t skeys[kTile];
    __shared__ uint32_t shist[256];
    // 1-D grid of rows x tiles: the generic-score path accepts more than 65535 rows (gridDim.y)
    const int n_tiles = ws.n_tiles;
    const int tile = (int)(blockIdx.x % (unsigned)n_tiles), row = (int)(blockIdx.x / (unsigned)n_tiles);
    const int tid = threadIdx.x;
    const int b = row / H, h = row % H;
    shist[tid] = 0;
    pdl_launch_dependents();  // the selection pass behind this one may start to take residency
    const uint16_t* src = scores + (int64_t)b * sb + (int64_t)h * sh;
    const int s = tile * kTile + tid;
    skeys[tid] = (s < S) ? ordered_key16(src[s], inf_bits) : (uint16_t)0;
    __syncthreads();
    flush_chunk_keys<1>(skeys, nullptr, shist, row, tile * kTile, S, ws, nullptr);
}

cudaError_t launch_keys_from_scores(const Dims& d, int dtype, const void* scores, int64_t sb, int64_t sh,
                                    const Workspace& ws, cudaStream_t st) {
    const dim3 grid(d.R * ws.n_tiles);
    keys_from_scores_kernel<<<grid, kTileThreads, 0, st>>>(static_cast<const uint16_t*>(scores),
                                                           sb, sh, d.H, d.S,
                                                           dtype == KVP_BF16 ? 0x7F80u : 0x7C00u, ws);
    return cudaPeekAtLastError();
}

}  // namespace kvp
