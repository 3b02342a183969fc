// select_compact.cu — stages T (per-row top-k threshold) and G (stable compaction of K and V).
//
// Replaces scores.topk(n_kept).indices + keys.gather + values.gather
// (kvpress/presses/scorer_press.py:95-100) for 16-bit scores:
//   * the score stage left, per (b,h) row, the ordered keys and a 256-bin histogram of key>>8;
// Two kernels, chained by programmatic dependent launch (PDL):
//   * selection pass (select_kernel), one CTA per refine item (row, 16 tiles): finds the threshold
//                    bin b1 from that histogram, histograms the low byte of the keys that fall in b1
//                    (-> row hist_lo, one warp per tile) and records, per tile, the suffix counts of
//                    those low bytes + the count of keys above b1. The CTA that finishes a row's last
//                    item runs the row scan: exact 16-bit threshold T, number of ties to take, and
//                    per tile the kept / tied positions of the tiles before it. Nothing in it waits.
//   * compaction grid (compact_kernel), one CTA per (row, tile of 256 positions): loads its keys,
//                    its tile prefix and the row's threshold (all final once the selection pass has
//                    completed), ranks its positions with warp ballots and copies the kept K and V
//                    rows (16-byte vectors) to [B,H,n_kept,D] in ascending position order. Ties at T
//                    go to the lowest positions. No waits of any kind.
// Tiles are visited in REVERSE order of the score stage so the K rows touched last (still in the
// 126 MB L2) are re-read first.
#include <stdlib.h>
#include <type_traits>

#include "common.cuh"
#include "knorm_chunk.cuh"

namespace kvp {

constexpr int kTilesPerWarp = 2;                                  // refine: tiles per warp
constexpr int kGroupTiles = (kTileThreads / 32) * kTilesPerWarp;  // tiles per refine item (16)
constexpr int kScanTiles = 4;                                     // row scan: consecutive tiles per thread and pass

// Copies `count` rows of `nvec` 16-byte vectors of BOTH tensors: dst row j <- src row list[j].
// K rows are plain loads (they may still sit in L2 from the score stage), V rows and all stores are
// streamed (evict-first). The loads of two consecutive batches (2 x 2*U 16-byte loads per thread) are
// issued before the first store, so a typical tile (<= 128 kept rows of 256 B) is ONE memory round trip.
// Generic loads on purpose: host_staging's zero-copy mode gathers V rows from pinned host memory here.
template <int U>
__device__ __forceinline__ void copy_rows_kv(const char* __restrict__ srcK, int64_t k_row_bytes,
                                             const char* __restrict__ srcV, int64_t v_row_bytes,
                                             char* __restrict__ dstK, char* __restrict__ dstV,
                                             int64_t dst_row_bytes, const int* __restrict__ list,
                                             int count, int nvec) {
    constexpr int STEP = kTileThreads * U;
    const int total = count * nvec;
    const uint64_t pol_first = l2_policy_evict_first();
    auto load = [&](int4 (&vk)[U], int4 (&vv)[U], int base) {
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int i = base + u * kTileThreads;
            if (i < total) {
                const int r = i / nvec;
                const int cc = i - r * nvec;
                const int64_t src_row = list[r];
                vk[u] = ldg_plain(srcK + src_row * k_row_bytes + cc * 16);
                vv[u] = ldg_hint(srcV + src_row * v_row_bytes + cc * 16, pol_first);
            }
        }
    };
    auto store = [&](const int4 (&vk)[U], const int4 (&vv)[U], int base) {
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int i = base + u * kTileThreads;
            if (i < total) {
                const int r = i / nvec;
                const int64_t off = (int64_t)r * dst_row_bytes + (i - r * nvec) * 16;
                stg_hint(dstK + off, vk[u], pol_first);
                stg_hint(dstV + off, vv[u], pol_first);
            }
        }
    };
    for (int base = threadIdx.x; base < total; base += 2 * STEP) {
        int4 ak[U], av[U], bk[U], bv[U];
        load(ak, av, base);
        const bool second = (base + STEP) < total;
        if (second) load(bk, bv, base + STEP);
        store(ak, av, base);
        if (second) store(bk, bv, base + STEP);
    }
}

// KeyRerotationPress epilogue (reference kvpress/presses/key_rerotation_press.py:50-131): the kept key
// that lands at output position j came from position s; it is rotated by delta = j - s positions:
//     out = k * cos(delta * inv_freq) + rotate_half(k) * sin(delta * inv_freq)
// with the reference's rounding points: angle and cos/sin in fp32, cos/sin rounded to the cache dtype, each
// product and the sum rounded to the cache dtype. A thread handles the vector pair (d, d + D/2).
template <typename T>
__device__ __forceinline__ void copy_rows_k_rerotated(const char* __restrict__ srcK, int64_t k_row_bytes,
                                                      char* __restrict__ dstK, int64_t dst_row_bytes,
                                                      const int* __restrict__ list, int count, int D,
                                                      const float* __restrict__ inv_freq, int out_pos0) {
    const int half_vec = D >> 4;  // 16-byte vectors in half a row
    const int total = count * half_vec;
    const uint64_t pol_first = l2_policy_evict_first();
    for (int i = threadIdx.x; i < total; i += kTileThreads) {
        const int r = i / half_vec, cc = i - r * half_vec;
        const int s = list[r];
        const float delta = (float)(out_pos0 + r) - (float)s;
        const char* src = srcK + (int64_t)s * k_row_bytes;
        const int4 lo = ldg_plain(src + cc * 16);
        const int4 hi = ldg_plain(src + (cc + half_vec) * 16);
        const uint32_t wl[4] = {(uint32_t)lo.x, (uint32_t)lo.y, (uint32_t)lo.z, (uint32_t)lo.w};
        const uint32_t wh[4] = {(uint32_t)hi.x, (uint32_t)hi.y, (uint32_t)hi.z, (uint32_t)hi.w};
        uint32_t ol[4], oh[4];
#pragma unroll
        for (int w = 0; w < 4; ++w) {
            uint16_t rl[2], rh[2];
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const float f = delta * __ldg(inv_freq + cc * 8 + w * 2 + e);
                float sn, cs;
                sincosf(f, &sn, &cs);
                const float c16 = F16Traits<T>::to_float(F16Traits<T>::from_float(cs));
                const float s16 = F16Traits<T>::to_float(F16Traits<T>::from_float(sn));
                const float kl = F16Traits<T>::to_float((uint16_t)(wl[w] >> (16 * e)));
                const float kh = F16Traits<T>::to_float((uint16_t)(wh[w] >> (16 * e)));
                auto rn = [](float x) { return F16Traits<T>::to_float(F16Traits<T>::from_float(x)); };
                rl[e] = F16Traits<T>::from_float(rn(kl * c16) + rn(-kh * s16));
                rh[e] = F16Traits<T>::from_float(rn(kh * c16) + rn(kl * s16));
            }
            ol[w] = (uint32_t)rl[0] | ((uint32_t)rl[1] << 16);
            oh[w] = (uint32_t)rh[0] | ((uint32_t)rh[1] << 16);
        }
        char* dst = dstK + (int64_t)r * dst_row_bytes;
        stg_hint(dst + cc * 16, make_int4((int)ol[0], (int)ol[1], (int)ol[2], (int)ol[3]), pol_first);
        stg_hint(dst + (cc + half_vec) * 16, make_int4((int)oh[0], (int)oh[1], (int)oh[2], (int)oh[3]), pol_first);
    }
}

// Plain copy of one tensor's rows (the V half of a rerotating compaction).
__device__ __forceinline__ void copy_rows_single(const char* __restrict__ src, int64_t row_bytes_src,
                                                 char* __restrict__ dst, int64_t dst_row_bytes,
                                                 const int* __restrict__ list, int count, int nvec) {
    const int total = count * nvec;
    const uint64_t pol_first = l2_policy_evict_first();
    for (int i = threadIdx.x; i < total; i += kTileThreads) {
        const int r = i / nvec, cc = i - r * nvec;
        const int4 v = ldg_hint(src + (int64_t)list[r] * row_bytes_src + cc * 16, pol_first);
        stg_hint(dst + (int64_t)r * dst_row_bytes + cc * 16, v, pol_first);
    }
}

struct SelectSmem {
    uint32_t hist[256];                    // hist_hi of the current row
    uint32_t lo[kTileThreads / 32][256];   // refine: per-warp low-byte histograms; scan: lo[0] = hist_lo
    int list[kTile];
    uint32_t wsum[2][8];
    uint32_t thr[3];
    uint32_t meta[2];  // fused compact item: the row's threshold key and tie budget, fetched by the polling thread
    int item;
    int b1;
    int last;
    int abort;
};

// Row scan, executed by the CTA that finished the LAST refine item of a row: exact threshold T,
// number of ties to take, and for every tile the number of kept (> T) and tied (== T) positions in
// the tiles before it. Publishes row_meta / tile_prefix, then raises the row's ready flag.
__device__ __forceinline__ void scan_row(SelectSmem& sm, int row, int n_kept, const Workspace& ws) {
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    __syncthreads();
    sm.lo[0][tid] = __ldcg(&ws.hist_lo[(size_t)row * 256 + tid]);  // sm.hist still holds hist_hi
    __syncthreads();
    if (warp == 0) {
        int b1, lo1;
        uint32_t above1, above2;
        warp_suffix_find(sm.hist, (uint32_t)n_kept, lane, b1, above1);
        const uint32_t need1 = (uint32_t)n_kept - above1;  // >= 1
        warp_suffix_find(sm.lo[0], need1, lane, lo1, above2);
        if (lane == 0) {
            sm.thr[0] = ((uint32_t)b1 << 8) | (uint32_t)lo1;
            sm.thr[1] = need1 - above2;  // ties (key == T) to take, >= 1
            sm.thr[2] = (uint32_t)lo1;
        }
    }
    __syncthreads();
    const uint32_t lo1 = sm.thr[2];
    if (tid == 0) ws.row_meta[row] = make_uint2(sm.thr[0], sm.thr[1]);
    const uint16_t* recs = ws.tile_sfx + (size_t)row * ws.n_tiles * kSfxStride;
    uint2* prefix = ws.tile_prefix + (size_t)row * ws.n_tiles;
    uint32_t carry_gt = 0, carry_eq = 0;
    // a pass covers kScanTiles consecutive tiles per thread, so tile order == thread order and the records of a
    // pass are ONE round trip (S <= 256 k: one pass)
    for (int p0 = 0; p0 < ws.n_tiles; p0 += kScanTiles * kTileThreads) {
        const int t0 = p0 + tid * kScanTiles;
        uint32_t gt[kScanTiles], eq[kScanTiles], sum_gt = 0, sum_eq = 0;
#pragma unroll
        for (int c = 0; c < kScanTiles; ++c) {
            gt[c] = eq[c] = 0;
            if (t0 + c < ws.n_tiles) {
                const uint16_t* r = recs + (size_t)(t0 + c) * kSfxStride;
                const uint32_t ge = __ldcg(r + lo1), g2 = __ldcg(r + lo1 + 1);
                gt[c] = (uint32_t)__ldcg(r + 257) + g2;
                eq[c] = ge - g2;
            }
            sum_gt += gt[c];
            sum_eq += eq[c];
        }
        if (p0 == 0) __threadfence();  // row_meta is visible before any prefix (= readiness) is
        uint32_t igt = sum_gt, ieq = sum_eq;  // inclusive warp scans
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const uint32_t a = __shfl_up_sync(0xFFFFFFFFu, igt, off);
            const uint32_t b = __shfl_up_sync(0xFFFFFFFFu, ieq, off);
            if (lane >= off) {
                igt += a;
                ieq += b;
            }
        }
        __syncthreads();
        if (lane == 31) {
            sm.wsum[0][warp] = igt;
            sm.wsum[1][warp] = ieq;
        }
        __syncthreads();
        uint32_t pg = carry_gt + igt - sum_gt, pe = carry_eq + ieq - sum_eq, tg = 0, te = 0;
#pragma unroll
        for (int w = 0; w < 8; ++w) {
            pg += (w < warp) ? sm.wsum[0][w] : 0u;
            pe += (w < warp) ? sm.wsum[1][w] : 0u;
            tg += sm.wsum[0][w];
            te += sm.wsum[1][w];
        }
#pragma unroll
        for (int c = 0; c < kScanTiles; ++c) {
            if (t0 + c < ws.n_tiles) {
                // 8-byte store: both halves become visible together; +1: 0 means not ready
                *reinterpret_cast<volatile unsigned long long*>(prefix + t0 + c) =
                    (unsigned long long)(pg + 1u) | ((unsigned long long)(pe + 1u) << 32);
            }
            pg += gt[c];
            pe += eq[c];
        }
        carry_gt += tg;
        carry_eq += te;
    }
}

// ---- refine item: (row, group of kGroupTiles tiles); one warp per tile, no block barriers inside ----
__device__ __forceinline__ void refine_item(SelectSmem& sm, int row, int group, int n_groups, int S,
                                            int n_kept, const Workspace& ws) {
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // this warp's key tiles are requested first: their latency overlaps the histogram read + search
    int4 kv[kTilesPerWarp];
#pragma unroll
    for (int tw = 0; tw < kTilesPerWarp; ++tw) {
        const int tile = group * kGroupTiles + warp * kTilesPerWarp + tw;
        kv[tw] = make_int4(0, 0, 0, 0);
        if (tile < ws.n_tiles)
            kv[tw] = __ldcg(reinterpret_cast<const int4*>(ws.keys + (size_t)row * ws.S_pad +
                                                           (size_t)tile * kTile + lane * 8));
    }
    sm.hist[tid] = __ldcg(&ws.hist_hi[(size_t)row * 256 + tid]);  // written by other CTAs' atomics
    __syncthreads();
    if (warp == 0) {
        int b1;
        uint32_t above;
        warp_suffix_find(sm.hist, (uint32_t)n_kept, lane, b1, above);
        if (lane == 0) sm.b1 = b1;
    }
    __syncthreads();
    const unsigned b1 = (unsigned)sm.b1;
    uint32_t* lo = sm.lo[warp];
    uint32_t acc[8];  // group-level low-byte histogram, bins [8*lane, 8*lane+8) of this warp's tiles
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] = 0;
#pragma unroll
    for (int tw = 0; tw < kTilesPerWarp; ++tw) {
        const int tile = group * kGroupTiles + warp * kTilesPerWarp + tw;
        if (tile >= ws.n_tiles) break;
#pragma unroll
        for (int i = 0; i < 8; ++i) lo[lane * 8 + i] = 0;
        __syncwarp();
        const int4 v = kv[tw];
        const uint32_t w4[4] = {(uint32_t)v.x, (uint32_t)v.y, (uint32_t)v.z, (uint32_t)v.w};
        uint32_t n_gt = 0;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const unsigned k = (w4[q >> 1] >> ((q & 1) * 16)) & 0xFFFFu;
            const bool valid = (tile * kTile + lane * 8 + q) < S;
            const unsigned hi = k >> 8;
            n_gt += (valid && hi > b1) ? 1u : 0u;
            if (valid && hi == b1) atomicAdd(&lo[k & 0xFF], 1u);
        }
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) n_gt += __shfl_xor_sync(0xFFFFFFFFu, n_gt, off);
        __syncwarp();
        // suffix sums over the 256 bins: lane owns bins [8*lane, 8*lane+8)
        uint32_t c[8], lane_sum = 0;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            c[i] = lo[lane * 8 + i];
            lane_sum += c[i];
            acc[i] += c[i];
        }
        uint32_t sfx = lane_sum;  // inclusive suffix over lanes
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const uint32_t t = __shfl_down_sync(0xFFFFFFFFu, sfx, off);
            if (lane + off < 32) sfx += t;
        }
        uint32_t run = sfx - lane_sum;  // candidates in bins above this lane's
        uint32_t out[8];
#pragma unroll
        for (int i = 7; i >= 0; --i) {
            run += c[i];
            out[i] = run;
        }
        uint16_t* rec = ws.tile_sfx + ((size_t)row * ws.n_tiles + tile) * kSfxStride;
        uint4 pk;
        pk.x = out[0] | (out[1] << 16);
        pk.y = out[2] | (out[3] << 16);
        pk.z = out[4] | (out[5] << 16);
        pk.w = out[6] | (out[7] << 16);
        *reinterpret_cast<uint4*>(rec + lane * 8) = pk;
        if (lane == 0) {
            rec[256] = 0;
            rec[257] = (uint16_t)n_gt;
        }
        __syncwarp();
    }
    // the CTA's share of the row's low-byte histogram: warps summed in shared memory first, then one coalesced atomic
    // per bin (per-warp atomics put 8 x 32 scattered sector updates per warp on the row's 256 counters)
#pragma unroll
    for (int i = 0; i < 8; ++i) lo[lane * 8 + i] = acc[i];
    __syncthreads();
    uint32_t bin_sum = 0;
#pragma unroll
    for (int w = 0; w < kTileThreads / 32; ++w) bin_sum += sm.lo[w][tid];
    if (bin_sum) atomicAdd(&ws.hist_lo[(size_t)row * 256 + tid], bin_sum);
    __threadfence();
    __syncthreads();
    if (tid == 0) sm.last = (atomicAdd(&ws.counters[1 + row], 1u) == (uint32_t)(n_groups - 1));
    __syncthreads();
    if (sm.last) {
        __threadfence();
        scan_row(sm, row, n_kept, ws);
    }
}

// ---- rank + copy of one (row, tile of kTile == kTileThreads positions, one per thread) ------------------
// key: this thread's position's ordered key; T / n_take: the row's threshold key and ties to take (row scan);
// gt_before / eq_before: kept (> T) and tied (== T) positions in the row's tiles before this one.
// Shared by the compaction grid and the fused Knorm kernel's compact items.
template <typename TR, int U>  // TR = void: plain copy; TR = cache dtype: KeyRerotationPress epilogue
__device__ __forceinline__ void rank_and_copy(int* list, uint32_t (&wsum)[2][8], int row, int tile, uint32_t key,
                                              uint32_t T, uint32_t n_take, uint32_t gt_before, uint32_t eq_before,
                                              const char* K, const char* V, Strides3 ks, Strides3 vs, char* K_out,
                                              char* V_out, int32_t* idx_out, int H, int S, int D, int n_kept,
                                              const float* inv_freq) {
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int s = tile * kTile + tid;
    const bool valid = s < S;
    const bool is_gt = valid && key > T;
    const bool is_eq = valid && key == T;
    const unsigned m_gt = __ballot_sync(0xFFFFFFFFu, is_gt);
    const unsigned m_eq = __ballot_sync(0xFFFFFFFFu, is_eq);
    if (lane == 0) {
        wsum[0][warp] = __popc(m_gt);
        wsum[1][warp] = __popc(m_eq);
    }
    __syncthreads();
    uint32_t gt_rank = __popc(m_gt & ((1u << lane) - 1u));
    uint32_t eq_rank = __popc(m_eq & ((1u << lane) - 1u));
    uint32_t tot_gt = 0, tot_eq = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) {
        gt_rank += (w < warp) ? wsum[0][w] : 0u;
        eq_rank += (w < warp) ? wsum[1][w] : 0u;
        tot_gt += wsum[0][w];
        tot_eq += wsum[1][w];
    }
    // ties are taken in position order: this tile may take those with global tie rank < n_take
    const uint32_t tie_room = (n_take > eq_before) ? (n_take - eq_before) : 0u;
    const uint32_t out_base = gt_before + min(eq_before, n_take);
    if (is_gt || (is_eq && eq_rank < tie_room)) list[gt_rank + min(eq_rank, tie_room)] = s;
    const int count = (int)(tot_gt + min(tot_eq, tie_room));
    __syncthreads();
    if (count == 0) return;
    const int b = row / H, h = row % H;
    const int64_t out_row0 = (int64_t)row * n_kept + out_base;
    if (idx_out != nullptr && tid < count) idx_out[out_row0 + tid] = list[tid];
    const int64_t row_bytes = (int64_t)D * 2;
    const char* k_src = K + ((int64_t)b * ks.b + (int64_t)h * ks.h) * 2;
    const char* v_src = V + ((int64_t)b * vs.b + (int64_t)h * vs.h) * 2;
    if (K_out == nullptr) {
        // selection only (kvp_scores_select): the kept positions in idx_out are the whole result
    } else if constexpr (std::is_void<TR>::value) {
        copy_rows_kv<U>(k_src, ks.s * 2, v_src, vs.s * 2, K_out + out_row0 * row_bytes, V_out + out_row0 * row_bytes,
                        row_bytes, list, count, D >> 3);
    } else {
        copy_rows_k_rerotated<TR>(k_src, ks.s * 2, K_out + out_row0 * row_bytes, row_bytes, list, count, D, inv_freq,
                                  (int)out_base);
        copy_rows_single(v_src, vs.s * 2, V_out + out_row0 * row_bytes, row_bytes, list, count, D >> 3);
    }
}

// ---- selection pass: one CTA per refine item (row, group of kGroupTiles tiles) ----------------------------
// Nothing here waits on another CTA, so a plain grid of any size is safe. The CTA that completes a row's last
// item runs that row's scan. Dependents are released at once: the compaction grid can take residency while
// this pass runs and parks in its pdl_wait() until the pass has completed.
__global__ void __launch_bounds__(kTileThreads)
select_kernel(int S, int n_kept, Workspace ws) {
    __shared__ SelectSmem sm;
    pdl_launch_dependents();
    pdl_wait();  // keys + histograms of the score stage are complete and visible
    const int n_groups = (ws.n_tiles + kGroupTiles - 1) / kGroupTiles;
    refine_item(sm, blockIdx.x / n_groups, blockIdx.x % n_groups, n_groups, S, n_kept, ws);
}

// ---- compaction grid: one CTA per (row, tile), last rows / last tiles first ---------------------------------
// 1-D grid (gridDim.y would cap the row count at 65535). After pdl_wait() the keys, the tile prefix and the row's
// threshold are final, so the three loads are independent and the CTA never waits for another one.
// Register budget (ptxas -v, sm_100a): no spills at the bound below; A/B of the (U, CTAs/SM) settings in DESIGN.md §4.1.
constexpr int kCompactU = 2;
constexpr int kCompactCtas = 4;
constexpr int kRerotCtas = 4;  // re-rotating variant: issue-bound on sincosf (A/B 220 -> 207 us, profiles/r01_ab_rerot.txt)
template <typename TR>
__global__ void __launch_bounds__(kTileThreads, std::is_void<TR>::value ? kCompactCtas : kRerotCtas)
compact_kernel(const char* __restrict__ K, const char* __restrict__ V, Strides3 ks, Strides3 vs,
               char* __restrict__ K_out, char* __restrict__ V_out, int32_t* __restrict__ idx_out, int H, int S, int D,
               int n_kept, Workspace ws, const float* __restrict__ inv_freq) {
    __shared__ int list[kTile];
    __shared__ uint32_t wsum[2][8];
    const int n_tiles = ws.n_tiles;
    const int row = ws.R - 1 - (int)(blockIdx.x / (unsigned)n_tiles);
    const int tile = n_tiles - 1 - (int)(blockIdx.x % (unsigned)n_tiles);
    pdl_wait();  // the selection pass (and through it the score stage) has completed
    const uint32_t key = __ldcg(&ws.keys[(size_t)row * ws.S_pad + (size_t)tile * kTile + threadIdx.x]);
    const uint2 before = __ldcg(&ws.tile_prefix[(size_t)row * n_tiles + tile]);  // +1 encoded (scan_row)
    const uint2 meta = __ldcg(&ws.row_meta[row]);
    rank_and_copy<TR, kCompactU>(list, wsum, row, tile, key, meta.x, meta.y, before.x - 1u, before.y - 1u, K, V, ks,
                                 vs, K_out, V_out, idx_out, H, S, D, n_kept, inv_freq);
}

template <typename TR>
static cudaError_t launch_select_compact_t(const Dims& d, const void* K, const void* V, void* K_out,
                                           void* V_out, int32_t* idx_out, const Workspace& ws,
                                           const float* inv_freq, cudaStream_t st) {
    const int n_groups = (ws.n_tiles + kGroupTiles - 1) / kGroupTiles;
    const dim3 sel_grid(d.R * n_groups), cmp_grid(d.R * ws.n_tiles);
    auto cmp = compact_kernel<TR>;
#ifndef KVP_NO_PDL
    cudaError_t e = launch_pdl(select_kernel, sel_grid, dim3(kTileThreads), 0, st, d.S, d.n_kept, ws);
    if (e != cudaSuccess) return e;
    return launch_pdl(cmp, cmp_grid, dim3(kTileThreads), 0, st, static_cast<const char*>(K),
                      static_cast<const char*>(V), d.ks, d.vs, static_cast<char*>(K_out), static_cast<char*>(V_out),
                      idx_out, d.H, d.S, d.D, d.n_kept, ws, inv_freq);
#else
    select_kernel<<<sel_grid, kTileThreads, 0, st>>>(d.S, d.n_kept, ws);
    cmp<<<cmp_grid, kTileThreads, 0, st>>>(static_cast<const char*>(K), static_cast<const char*>(V), d.ks, d.vs,
                                           static_cast<char*>(K_out), static_cast<char*>(V_out), idx_out, d.H, d.S,
                                           d.D, d.n_kept, ws, inv_freq);
    return cudaPeekAtLastError();
#endif
}

cudaError_t launch_select_compact(const Dims& d, const void* K, const void* V, void* K_out,
                                  void* V_out, int32_t* idx_out, const Workspace& ws,
                                  cudaStream_t st) {
    return launch_select_compact_t<void>(d, K, V, K_out, V_out, idx_out, ws, nullptr, st);
}

// Same selection, keys re-rotated to their new positions (KeyRerotationPress); inv_freq: fp32 [D/2].
cudaError_t launch_select_compact_rerotate(const Dims& d, int dtype, const void* K, const void* V,
                                           void* K_out, void* V_out, int32_t* idx_out,
                                           const Workspace& ws, const float* inv_freq, cudaStream_t st) {
    if (dtype == KVP_BF16)
        return launch_select_compact_t<__nv_bfloat16>(d, K, V, K_out, V_out, idx_out, ws, inv_freq, st);
    return launch_select_compact_t<__half>(d, K, V, K_out, V_out, idx_out, ws, inv_freq, st);
}

// ---- KnormPress: score + select + compact in ONE persistent kernel ---------------------------------
// Work items of three kinds share one ticket queue: S(row, chunk) scores 256 positions and adds to the
// row histogram; A(row, group) is the refine item (waits until all S items of its row are done);
// B(row, tile) is the compact item (waits for the row's ready flag). The queue is laid out in blocks
//     block p = [ A(p-1) | S(p, 0..m-1) | S(p, m..) evenly interleaved with B(p-lag, .) ]
// so that while row p is being scored (pure HBM reads), row p-lag is compacted: its K rows were read `lag`
// blocks ago and are re-read from the 126 MB L2 instead of HBM (V reads and all stores are L2-evict-first).
// lag = 2, m = 0 (small caches): no compact item ever waits for a refine item of the same block.
// lag = 1, m > 0 (large caches, K rows of one head = tens of MB): only two rows of K are live in L2; the m score
// items in front of the first compact item give the row's refine items + scan time to finish.
// Every item only waits on items that precede it in the queue, and S items never wait, so the kernel cannot
// deadlock for any grid size.
struct FusedItem {
    int kind;  // 0 = score, 1 = refine, 2 = compact, -1 = done
    int row, idx;
};

struct FusedQueue {
    int R, nT, nA, lag, m_head;
};

__host__ __device__ __forceinline__ long long fused_total_items(const FusedQueue& q) {
    return (long long)q.R * (2ll * q.nT + q.nA);
}

__host__ __device__ __forceinline__ FusedItem decode_fused_item(long long item, const FusedQueue& q) {
    FusedItem it = {-1, 0, 0};
    const int R = q.R, nT = q.nT, nA = q.nA, lag = q.lag;
    for (int p = 0; p < R + lag; ++p) {
        // closed form over the identical full blocks p in [lag, R)
        if (p == lag && R > lag) {
            const long long full = (long long)nA + 2ll * nT;
            const long long n_full = R - lag;
            const long long skip = item / full < n_full ? item / full : n_full;
            item -= skip * full;
            p += (int)skip;
            if (p >= R + lag) break;
        }
        const int a = (p >= 1 && p <= R) ? nA : 0;
        const int s = (p < R) ? nT : 0;
        const int b = (p >= lag && p - lag < R) ? nT : 0;
        const long long size = (long long)a + s + b;
        if (item >= size) {
            item -= size;
            continue;
        }
        if (item < a) {
            it.kind = 1; it.row = p - 1; it.idx = (int)item;
            return it;
        }
        const int j = (int)(item - a);
        const int mh = (s && b) ? (q.m_head < s ? q.m_head : s) : 0;  // score items in front of the mixed tail
        if (j < mh || b == 0) {
            it.kind = 0; it.row = p; it.idx = j;
            return it;
        }
        // tail: (s - mh) score items and b compact items, evenly interleaved (Bresenham)
        const long long idx = j - mh, tail = (long long)(s - mh) + b;
        const long long b_before = idx * b / tail, b_after = (idx + 1) * b / tail;
        if (b_after != b_before) { it.kind = 2; it.row = p - lag; it.idx = (int)b_before; }
        else                     { it.kind = 0; it.row = p;       it.idx = mh + (int)(idx - b_before); }
        return it;
    }
    return it;
}

// Host-side view of the queue for the CPU tests (tests/test_abi_symbols.py): item -> (kind, row, idx).
extern "C" int kvp_debug_fused_queue_item(int R, int nT, int nA, int lag, int m_head, long long item, int* out3) {
    const FusedQueue q = {R, nT, nA, lag, m_head};
    if (item < 0 || item >= fused_total_items(q)) return -1;
    const FusedItem it = decode_fused_item(item, q);
    out3[0] = it.kind; out3[1] = it.row; out3[2] = it.idx;
    return 0;
}

// Returns false when the wait was abandoned (error flag raised): the caller skips its item.
__device__ __forceinline__ bool spin_until(const uint32_t* counter, uint32_t need, volatile uint32_t* err) {
    const volatile uint32_t* flag = counter;
    uint32_t spins = 0;
    while (*flag < need) {
        __nanosleep(64);
        if (++spins > kSpinLimit) *err = 1u;  // a bug must not hang the GPU (nor trap the context)
        if ((spins & 255u) == 0u && *err != 0u) return false;
    }
    __threadfence();
    return true;
}

// Compact item of the fused queue: (row, tile) polls its tile prefix, which the row scan publishes last (the table
// is zeroed by the per-call memset, so one polled load doubles as the readiness flag; bounded spin), and the polling
// thread fetches the row's threshold right behind it. The keys are loaded after the wait: the score items of the
// same launch write them.
__device__ __forceinline__ void fused_compact_item(SelectSmem& sm, int row, int tile, const char* K, const char* V,
                                                   Strides3 ks, Strides3 vs, char* K_out, char* V_out,
                                                   int32_t* idx_out, int H, int S, int D, int n_kept,
                                                   const Workspace& ws) {
    if (threadIdx.x == 0) {
        const volatile unsigned long long* slot =
            reinterpret_cast<const volatile unsigned long long*>(ws.tile_prefix + (size_t)row * ws.n_tiles + tile);
        volatile uint32_t* err = ws.counters + kCounterErrSlot(ws.R);
        uint32_t spins = 0;
        unsigned long long raw = *slot;
        sm.abort = 0;
        while ((uint32_t)raw == 0u || (uint32_t)(raw >> 32) == 0u) {
            __nanosleep(64);
            if (++spins > kSpinLimit) *err = 1u;          // raise: the host reports it, nobody traps
            if ((spins & 255u) == 0u && *err != 0u) {     // raised here or by another CTA: drain
                sm.abort = 1;
                break;
            }
            raw = *slot;
        }
        __threadfence();
        sm.thr[0] = (uint32_t)raw - 1u;
        sm.thr[1] = (uint32_t)(raw >> 32) - 1u;
        if (!sm.abort) {  // published before the prefix table (scan_row): valid once the flag is up
            const uint2 m = __ldcg(&ws.row_meta[row]);
            sm.meta[0] = m.x;
            sm.meta[1] = m.y;
        }
    }
    __syncthreads();
    if (sm.abort) return;
    const uint32_t key = __ldcg(&ws.keys[(size_t)row * ws.S_pad + (size_t)tile * kTile + threadIdx.x]);
    rank_and_copy<void, 3>(sm.list, sm.wsum, row, tile, key, sm.meta[0], sm.meta[1], sm.thr[0], sm.thr[1], K, V, ks,
                           vs, K_out, V_out, idx_out, H, S, D, n_kept, nullptr);
}

template <typename Kern>
static int persistent_grid(Kern kernel, int threads, int n_items, PerDeviceInt& occupancy) {
    const int grid = device_sm_count() * cached_ctas_per_sm(kernel, threads, occupancy);
    return n_items < grid ? n_items : grid;
}

template <typename T, int LPR>
__global__ void __launch_bounds__(kTileThreads, 3)
knorm_fused_kernel(const T* __restrict__ K, const T* __restrict__ V, Strides3 ks, Strides3 vs,
                   char* __restrict__ K_out, char* __restrict__ V_out, int32_t* __restrict__ idx_out,
                   uint16_t* __restrict__ scores_out, int H, int S, int D, int n_kept, Workspace ws,
                   FusedQueue fq, int k_evict_last) {
    __shared__ SelectSmem sm;
    const int R = ws.R, nT = ws.n_tiles;
    const int nA = fq.nA;
    const long long total = fused_total_items(fq);
    uint32_t* score_done = ws.counters + kCounterMaxSlot(R) + 1;  // [R]
    uint16_t* skeys = reinterpret_cast<uint16_t*>(sm.list);       // 2 x 256 u16 alias the 1 KB list
    uint16_t* sscores = skeys + kScoreChunk;
    const int tid = threadIdx.x;
    while (true) {
        __syncthreads();  // previous item's shared state is dead
        if (tid == 0) sm.item = (int)atomicAdd(&ws.counters[0], 1u);
        __syncthreads();
        const long long item = (long long)(uint32_t)sm.item;
        if (item >= total) break;
        const FusedItem it = decode_fused_item(item, fq);
        if (it.kind == 0) {
            sm.hist[tid] = 0;
            if (k_evict_last)
                knorm_score_chunk<T, LPR, 1>(K, ks, it.row / H, it.row % H, it.idx, S, D, skeys, sscores);
            else
                knorm_score_chunk<T, LPR>(K, ks, it.row / H, it.row % H, it.idx, S, D, skeys, sscores);
            __syncthreads();
            flush_chunk_keys<1>(skeys, sscores, sm.hist, it.row, it.idx * kScoreChunk, S, ws, scores_out);
            __threadfence();
            __syncthreads();
            if (tid == 0) atomicAdd(&score_done[it.row], 1u);
        } else if (it.kind == 1) {
            if (tid == 0)
                sm.abort = spin_until(&score_done[it.row], (uint32_t)nT, ws.counters + kCounterErrSlot(R)) ? 0 : 1;
            __syncthreads();
            if (sm.abort) continue;
            refine_item(sm, it.row, it.idx, nA, S, n_kept, ws);
        } else {
            fused_compact_item(sm, it.row, it.idx, reinterpret_cast<const char*>(K),
                               reinterpret_cast<const char*>(V), ks, vs, K_out, V_out, idx_out, H, S, D, n_kept,
                               ws);
        }
    }
}

// Debug / A-B knobs of the fused kernel's queue (read once): KVP_KNORM_FUSED_LAG = 1 | 2,
// KVP_KNORM_FUSED_HEAD = percent of a row's score items in front of the mixed tail (lag 1),
// KVP_KNORM_FUSED_KLAST = 1: score-stage K loads carry an L2 evict_last hint.
static int env_int(const char* name, int dflt) {
    const char* v = getenv(name);
    return (v && *v) ? atoi(v) : dflt;
}

template <typename T>
static cudaError_t launch_knorm_fused_t(const Dims& d, const void* K, const void* V, void* K_out,
                                        void* V_out, int32_t* idx_out, void* scores_out,
                                        const Workspace& ws, cudaStream_t st) {
    static const int knob_lag = env_int("KVP_KNORM_FUSED_LAG", 0);
    static const int knob_head = env_int("KVP_KNORM_FUSED_HEAD", 50);
    static const int knob_klast = env_int("KVP_KNORM_FUSED_KLAST", -1);
    FusedQueue fq;
    fq.R = d.R;
    fq.nT = ws.n_tiles;
    fq.nA = (ws.n_tiles + kGroupTiles - 1) / kGroupTiles;
    // one kv-head row of K larger than ~8 MB: keep only two rows live in L2 (lag 1), else the latency-optimal lag 2
    const bool big_rows = (size_t)d.S * d.D * 2 >= ((size_t)8 << 20);
    fq.lag = (knob_lag == 1 || knob_lag == 2) ? knob_lag : (big_rows ? 1 : 2);
    if (fq.lag > d.R) fq.lag = d.R;
    fq.m_head = fq.lag == 1 ? (int)((long long)fq.nT * knob_head / 100) : 0;
    const int k_last = knob_klast >= 0 ? knob_klast : (big_rows ? 1 : 0);
    const long long total = fused_total_items(fq);
    if (total > 0x7FFFFFFFll) return cudaErrorNotSupported;
    const int nvec = d.D / 8;
#define KVP_LAUNCH_FUSED(LPR)                                                                         \
    do {                                                                                              \
        auto kern = knorm_fused_kernel<T, LPR>;                                                       \
        static PerDeviceInt occupancy;                                                                \
        const int grid = persistent_grid(kern, kTileThreads, (int)total, occupancy);                  \
        kern<<<grid, kTileThreads, 0, st>>>(static_cast<const T*>(K), static_cast<const T*>(V), d.ks,  \
                                            d.vs, static_cast<char*>(K_out), static_cast<char*>(V_out), \
                                            idx_out, static_cast<uint16_t*>(scores_out), d.H, d.S, d.D, \
                                            d.n_kept, ws, fq, k_last);                                \
    } while (0)
    if (nvec <= 4) KVP_LAUNCH_FUSED(4);
    else if (nvec <= 8) KVP_LAUNCH_FUSED(8);
    else if (nvec <= 16) KVP_LAUNCH_FUSED(16);
    else KVP_LAUNCH_FUSED(32);
#undef KVP_LAUNCH_FUSED
    return cudaPeekAtLastError();
}

cudaError_t launch_knorm_fused(const Dims& d, int dtype, const void* K, const void* V, void* K_out,
                               void* V_out, int32_t* idx_out, void* scores_out, const Workspace& ws,
                               cudaStream_t st) {
    if (dtype == KVP_BF16)
        return launch_knorm_fused_t<__nv_bfloat16>(d, K, V, K_out, V_out, idx_out, scores_out, ws, st);
    return launch_knorm_fused_t<__half>(d, K, V, K_out, V_out, idx_out, scores_out, ws, st);
}

// ---- StreamingLLM: the answer is two ranges, no scores needed --------------------------------
// kvpress/presses/streaming_llm_press.py:50-52 + scorer_press.py:95: ones everywhere except zeros
// on [n_sink, n_sink + n_pruned) => kept = [0, head) U [S - (n_kept - head), S),
// head = min(n_sink, n_kept) (lowest-position tie rule when n_kept < n_sink).
__global__ void __launch_bounds__(kTileThreads)
streaming_compact_kernel(const char* __restrict__ K, const char* __restrict__ V, Strides3 ks,
                         Strides3 vs, char* __restrict__ K_out, char* __restrict__ V_out,
                         int32_t* __restrict__ idx_out, int H, int S, int D, int n_kept,
                         int head) {
    __shared__ int s_list[kTile];
    const int tile = blockIdx.x, row = blockIdx.y, tid = threadIdx.x;
    const int b = row / H, h = row % H;
    const int j0 = tile * kTile;
    const int count = min(kTile, n_kept - j0);
    const int shift = S - n_kept;
    for (int j = tid; j < count; j += kTileThreads) {
        const int o = j0 + j;
        s_list[j] = (o < head) ? o : o + shift;
    }
    __syncthreads();
    const int64_t out_row0 = (int64_t)row * n_kept + j0;
    if (idx_out != nullptr)
        for (int j = tid; j < count; j += kTileThreads) idx_out[out_row0 + j] = s_list[j];
    const int64_t row_bytes = (int64_t)D * 2;
    copy_rows_kv<4>(K + ((int64_t)b * ks.b + (int64_t)h * ks.h) * 2, ks.s * 2,
                    V + ((int64_t)b * vs.b + (int64_t)h * vs.h) * 2, vs.s * 2,
                    K_out + out_row0 * row_bytes, V_out + out_row0 * row_bytes, row_bytes, s_list, count,
                    D >> 3);
}

cudaError_t launch_streaming_compress(const Dims& d, int n_sink, const void* K, const void* V,
                                      void* K_out, void* V_out, int32_t* idx_out,
                                      cudaStream_t st) {
    const int head = n_sink < d.n_kept ? n_sink : d.n_kept;
    dim3 grid((d.n_kept + kTile - 1) / kTile, d.R);
    streaming_compact_kernel<<<grid, kTileThreads, 0, st>>>(
        static_cast<const char*>(K), static_cast<const char*>(V), d.ks, d.vs,
        static_cast<char*>(K_out), static_cast<char*>(V_out), idx_out, d.H, d.S, d.D, d.n_kept,
        head);
    return cudaPeekAtLastError();
}

template <typename T>
__global__ void streaming_score_kernel(uint16_t* __restrict__ out, int S, int lo, int hi,
                                       int64_t total) {
    const uint16_t one = F16Traits<T>::from_float(1.0f);
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
         i += (int64_t)gridDim.x * blockDim.x) {
        const int s = (int)(i % S);
        out[i] = (s >= lo && s < hi) ? (uint16_t)0 : one;
    }
}

cudaError_t launch_streaming_score(const Dims& d, int dtype, int n_sink, void* scores_out,
                                   cudaStream_t st) {
    const int n_pruned = d.S - d.n_kept;
    const int64_t total = (int64_t)d.R * d.S;
    const int lo = n_sink, hi = (n_sink + n_pruned < d.S) ? n_sink + n_pruned : d.S;
    int blocks = (int)((total + 255) / 256);
    if (blocks > 148 * 8) blocks = 148 * 8;
    if (dtype == KVP_BF16)
        streaming_score_kernel<__nv_bfloat16>
            <<<blocks, 256, 0, st>>>(static_cast<uint16_t*>(scores_out), d.S, lo, hi, total);
    else
        streaming_score_kernel<__half>
            <<<blocks, 256, 0, st>>>(static_cast<uint16_t*>(scores_out), d.S, lo, hi, total);
    return cudaPeekAtLastError();
}

}  // namespace kvp
