// snapkv.cu — stage S for SnapKVPress (sm_100a: TMA + tcgen05 + TMEM).
//
// Reference semantics (kvpress/presses/snapkv_press.py:41-105), per kv head h with its G = Hq/Hkv
// query heads and the w = window_size last (RoPE'd) queries of each:
//     logit[r, j] = q_r . k_j / sqrt(d)          r = g*w + i (NQ = G*w query rows), j in [0, S)   (:62)
//     masked where j > S - w + i                  (causal inside the window)                        (:63-65)
//     p[r, :]     = softmax_j(logit[r, :])        (normaliser over ALL S keys)                      (:66)
//     s[j]        = mean_i, then avg_pool1d(kernel, pad=kernel/2, stride 1, /kernel), then mean_g
//                   of p[:, j] for j < S - w                                                         (:95-100)
//   and the last w positions are forced to be kept (:103). mean/pool/mean are linear and commute.
// The reference materialises repeat_kv(K), a [B,Hq,w,S] logit tensor, a mask and an fp32 softmax copy.
// Here K is streamed twice through TMA (second time mostly from L2) and never expanded:
//   pass 1 (snap_stats_kernel)  D[qrow, key] = Q_half[128 x d] * K_tile^T : thread = query row keeps an
//          online (max, sum exp2) over its row -> per-CTA partials;
//   (each pass-2 CTA first merges the partials into the exact normalisers: bias_r = (-m_r - log2 Z_r) / c)
//   pass 2 (snap_colsum_kernel) D[key, qrow] = K_tile[128 x d] * Q^T + 1 * bias^T (bias enters the MMA
//          as an extra K=16 step, hi/lo split): thread = key sums exp2(c * D) over its NQ columns
//          = sum_r p[r, j] -> fp32 pre-pool scores;
//   finalize (snap_finalize_kernel): 1/(G w) scaling, the 1-D box filter, ONE rounding to the cache
//          dtype, keys + histogram for the select stage.
// Both MMA kernels are persistent (one CTA per SM), warp-specialised: TMA producer, MMA issuer, TMEM
// allocator, two epilogue warpgroups draining two TMEM accumulator buffers.
#include <type_traits>

#include "common.cuh"
#include "umma.cuh"

namespace kvp {

#ifdef KVP_SNAP_PROFILE
// role-level cycle counters of CTA 0 of snap_stats_kernel (tools/snap_profile.py)
__device__ long long g_snap_prof[16];
#define SN_T0() const long long _t0 = clock64()
#define SN_ACC(slot) do { if (blockIdx.x == 0) g_snap_prof[slot] += clock64() - _t0; } while (0)
extern "C" void kvp_debug_snap_profile(long long* out, int reset) {
    if (reset) {
        long long z[16] = {0};
        cudaMemcpyToSymbol(g_snap_prof, z, sizeof(z));
    } else {
        cudaMemcpyFromSymbol(out, g_snap_prof, 16 * sizeof(long long));
    }
}
#else
#define SN_T0() do {} while (0)
#define SN_ACC(slot) do {} while (0)
#endif

constexpr int kSnTile = 128;
constexpr int kSnThreads = 640;  // 20 warps: TMA, MMA, TMEM-alloc, spare, 4 x 4 epilogue (2 warpgroups per TMEM buffer)
constexpr int kSnMaxParts = 640;
constexpr float kLog2e = 1.4426950408889634f;

__device__ __forceinline__ float fast_exp2(float x) {  // MUFU.EX2, 2 ulp; exp2(-inf) = 0
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

struct SnapScratch {
    float2* partial;  // [R][NQ][n_parts]  (max, sum) in the log2 domain
    float* colsum;    // [R][S_pad]        sum_r p[r, j]
};

static inline size_t sn_align(size_t x) { return (x + 255) / 256 * 256; }

size_t snapkv_scratch_bytes(const Dims& d, int window) {
    const int G = d.Hq / d.H;
    const size_t NQ = (size_t)G * window;
    const size_t S_pad = (size_t)((d.S + kTile - 1) / kTile) * kTile;
    return sn_align((size_t)d.R * NQ * kSnMaxParts * sizeof(float2)) + sn_align((size_t)d.R * S_pad * 4);
}

static SnapScratch carve_snap(const Dims& d, int window, const Workspace& ws) {
    const int G = d.Hq / d.H;
    const size_t NQ = (size_t)G * window;
    char* p = static_cast<char*>(ws.scorer);
    SnapScratch s;
    s.partial = reinterpret_cast<float2*>(p);
    p += sn_align((size_t)d.R * NQ * kSnMaxParts * sizeof(float2));
    s.colsum = reinterpret_cast<float*>(p);
    return s;
}

// Shared-memory layout shared by both passes. Q is resident ([NQP rows x D], K-major SW128 panels),
// K tiles stream through a 2-stage ring.
template <int D, int NQP>
struct SnSmem {
    static constexpr int kPanels = D / 64;
    static constexpr int kQPanel = NQP * 128;             // bytes of one 64-column panel of Q
    static constexpr int kQBytes = kPanels * kQPanel;
    static constexpr int kStageBytes = kPanels * kSnTile * 128;
    static constexpr int kQOff = 0;
    static constexpr int kStageOff = kQBytes;
    static constexpr int kAxOff = kStageOff + 2 * kStageBytes;  // ones operand [128 x 16]
    static constexpr int kBxOff = kAxOff + kSnTile * 32;        // bias operand [NQP x 16]
    static constexpr int kBarOff = kBxOff + NQP * 32;
    static constexpr int kTotal = kBarOff + 256;
    static_assert(kTotal + 1024 <= 227 * 1024, "shared memory budget");
};

struct SnCtaRange {
    int group, part, n_groups;
};

// ---- pass 1: per-query-row softmax statistics ---------------------------------------------------------
template <typename T, int D, int NQP>
__global__ void __launch_bounds__(kSnThreads, 1)
snap_stats_kernel(const __grid_constant__ CUtensorMap mapK, const __grid_constant__ CUtensorMap mapQ, int H,
                  int G, int S, int window, int R, int n_tiles128, int ctas_per_row, int n_parts,
                  SnapScratch sc) {
    using L = SnSmem<D, NQP>;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>(
        (reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    unsigned char* s_q = smem + L::kQOff;
    unsigned char* s_stage = smem + L::kStageOff;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::kBarOff);
    uint64_t* k_full = bars;       // [2]
    uint64_t* k_empty = bars + 2;  // [2]
    uint64_t* t_full = bars + 4;   // [2]
    uint64_t* t_empty = bars + 6;  // [2]
    uint64_t* q_full = bars + 8;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 10);

    constexpr int kQHalves = NQP / 128;  // 128-row blocks of Q; block qh -> TMEM buffer (qh & 1)
    constexpr int kBufCols = 128;        // N = 128 keys per MMA
    const int NQ = G * window;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n_groups = gridDim.x / ctas_per_row;
    const int group = blockIdx.x / ctas_per_row;
    const int part = blockIdx.x % ctas_per_row;

    if (tid == 0) {
        umma::prefetch_tmap(&mapK);
        umma::prefetch_tmap(&mapQ);
        for (int i = 0; i < 2; ++i) {
            umma::mbar_init(&k_full[i], 1);
            umma::mbar_init(&k_empty[i], 1);  // MMA commit only: the epilogue never reads K from smem
            umma::mbar_init(&t_full[i], 1);
            umma::mbar_init(&t_empty[i], 8);  // two warpgroups (column halves) drain each buffer
        }
        umma::mbar_init(q_full, 1);
        umma::mbar_fence_init();
    }
    if (warp == 2) umma::tmem_alloc(tmem_slot, 256);
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = *tmem_slot;

    const int tiles_per_part = (n_tiles128 + ctas_per_row - 1) / ctas_per_row;
    const int t_begin = part * tiles_per_part;
    const int t_end = min(n_tiles128, t_begin + tiles_per_part);
    const float c = kLog2e * rsqrtf((float)D);  // logits -> log2 domain

    uint32_t k_it = 0, h_it = 0, q_it = 0;
    for (int row = group; row < R; row += n_groups) {
        const int b = row / H, h = row % H;
        const int q_row0 = (b * (H * G) + h * G) * window;  // first of this kv head's NQ rows in q_window
        __syncthreads();  // previous row fully drained: s_q reusable

        if (warp == 0) {
            if (lane == 0) {
                // all NQP resident rows are loaded (boxes of min(NQP, 256) rows): rows >= NQ belong to the next kv
                // head or lie past the tensor (zero fill); their outputs are never read
                umma::mbar_arrive_expect_tx(q_full, (uint32_t)(L::kPanels * NQP * 128));
                for (int kp = 0; kp < L::kPanels; ++kp)
                    for (int r0 = 0; r0 < NQP; r0 += 256)
                        umma::tma_load_3d(s_q + kp * L::kQPanel + r0 * 128, &mapQ, q_full, kp * 64,
                                          q_row0 + r0, 0);
                for (int t = t_begin; t < t_end; ++t, ++k_it) {
                    const int stage = k_it & 1;
                    { SN_T0(); umma::mbar_wait(&k_empty[stage], ((k_it >> 1) & 1) ^ 1); SN_ACC(0); }
                    umma::mbar_arrive_expect_tx(&k_full[stage], L::kStageBytes);
                    for (int kp = 0; kp < L::kPanels; ++kp)
                        umma::tma_load_4d(s_stage + stage * L::kStageBytes + kp * (kSnTile * 128), &mapK,
                                          &k_full[stage], kp * 64, t * kSnTile, h, b);
                }
            }
        } else if (warp == 1) {
            if (lane == 0) {
                const uint32_t idesc = umma::instr_desc_f16(128, kBufCols, F16Traits<T>::kMmaFormat);
                umma::mbar_wait(q_full, q_it & 1);
                for (int t = t_begin; t < t_end; ++t, ++k_it) {
                    const int stage = k_it & 1;
                    { SN_T0(); umma::mbar_wait(&k_full[stage], (k_it >> 1) & 1); SN_ACC(1); }
                    umma::fence_after_sync();
                    const uint32_t kb = umma::smem_u32(s_stage + stage * L::kStageBytes);
#pragma unroll 1
                    for (int qh = 0; qh < kQHalves; ++qh, ++h_it) {
                        const int buf = h_it & 1;
                        { SN_T0(); umma::mbar_wait(&t_empty[buf], ((h_it >> 1) & 1) ^ 1); SN_ACC(2); }
                        umma::fence_after_sync();
#pragma unroll
                        for (int k = 0; k < D / 16; ++k) {
                            const int kp = k >> 2, kk = k & 3;
                            const uint64_t da = umma::smem_desc_sw128(
                                umma::smem_u32(s_q + kp * L::kQPanel + qh * (128 * 128)) + kk * 32);
                            const uint64_t db = umma::smem_desc_sw128(kb + kp * (kSnTile * 128) + kk * 32);
                            umma::mma_f16_ss(tmem + buf * kBufCols, da, db, idesc, k > 0);
                        }
                        umma::mma_commit(&t_full[buf]);
                    }
                    umma::mma_commit(&k_empty[stage]);
                }
            }
            ++q_it;
        } else if (warp >= 4) {
            // ===== epilogue: four warpgroups; warpgroup (buf, ch) drains column half ch of TMEM buffer buf;
            // thread = query row of the 128-block =====
            const int wgi = (warp - 4) >> 2;
            const int wg = wgi & 1;   // TMEM buffer
            const int ch = wgi >> 1;  // column half of the 128-key tile
            const int ew = warp & 3;
            const uint32_t lane_base = (uint32_t)(ew * 32) << 16;
            constexpr int kHalfCols = kBufCols / 2;  // 64 keys per warpgroup
            // each warpgroup may serve several 128-row blocks of Q (NQP = 512 -> two each)
            float run_m[(kQHalves + 1) / 2], run_z[(kQHalves + 1) / 2];
#pragma unroll
            for (int i = 0; i < (kQHalves + 1) / 2; ++i) {
                run_m[i] = -INFINITY;
                run_z[i] = 0.f;
            }
            for (int t = t_begin; t < t_end; ++t) {
                const int key0 = t * kSnTile + ch * kHalfCols;
                const bool interior = (key0 + kHalfCols) <= (S - window);  // no masking, all keys valid
#pragma unroll
                for (int qh = 0; qh < kQHalves; ++qh, ++h_it) {
                    const int buf = h_it & 1;
                    if (buf != wg) continue;
                    const int slot = qh >> 1;
                    const int r = qh * 128 + ew * 32 + lane;       // query row
                    const int limit = (S - window) + (r % window);  // last visible key position
                    { SN_T0(); umma::mbar_wait(&t_full[buf], (h_it >> 1) & 1); if (warp == 4 && lane == 0) SN_ACC(3); }
                    SN_T0();
                    umma::fence_after_sync();
                    const uint32_t tbase = tmem + lane_base + buf * kBufCols + ch * kHalfCols;
                    uint32_t y[2][16];
                    umma::tmem_ld16(tbase, y[0]);
                    // running max is kept in RAW logit units (q.k); c > 0 so the order is the same and the
                    // scale folds into one FFMA per element: exp2(fma(y, c, -m*c))
                    float m = run_m[slot], z = run_z[slot];
                    auto chunk = [&](const uint32_t (&yy)[16], int cc, auto masked) {
                        float v[16];
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            v[j] = __uint_as_float(yy[j]);
                            if (decltype(masked)::value) {
                                const int pos = key0 + cc * 16 + j;
                                if (pos > limit || pos >= S) v[j] = -INFINITY;
                            }
                        }
                        // tree max (depth 4) instead of a 16-long dependent chain
                        float m8[8], m4[4];
#pragma unroll
                        for (int j = 0; j < 8; ++j) m8[j] = fmaxf(v[j], v[j + 8]);
#pragma unroll
                        for (int j = 0; j < 4; ++j) m4[j] = fmaxf(m8[j], m8[j + 4]);
                        const float cmax = fmaxf(fmaxf(m4[0], m4[2]), fmaxf(m4[1], m4[3]));
                        const float m_new = fmaxf(m, cmax);
                        if (m_new > -INFINITY) {
                            const float neg = -m_new * c;
                            float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;  // four independent sum chains
#pragma unroll
                            for (int j = 0; j < 16; j += 4) {
                                a0 += fast_exp2(fmaf(v[j], c, neg));
                                a1 += fast_exp2(fmaf(v[j + 1], c, neg));
                                a2 += fast_exp2(fmaf(v[j + 2], c, neg));
                                a3 += fast_exp2(fmaf(v[j + 3], c, neg));
                            }
                            z = z * fast_exp2((m - m_new) * c) + ((a0 + a1) + (a2 + a3));
                            m = m_new;
                        }
                    };
                    // warp-uniform split: interior tiles (all but the last one or two) carry no mask code
                    if (interior) {
#pragma unroll
                        for (int cc = 0; cc < kHalfCols / 16; ++cc) {
                            umma::tmem_ld_wait();
                            if (cc + 1 < kHalfCols / 16) umma::tmem_ld16(tbase + (cc + 1) * 16, y[(cc + 1) & 1]);
                            chunk(y[cc & 1], cc, std::false_type{});
                        }
                    } else {
#pragma unroll
                        for (int cc = 0; cc < kHalfCols / 16; ++cc) {
                            umma::tmem_ld_wait();
                            if (cc + 1 < kHalfCols / 16) umma::tmem_ld16(tbase + (cc + 1) * 16, y[(cc + 1) & 1]);
                            chunk(y[cc & 1], cc, std::true_type{});
                        }
                    }
                    run_m[slot] = m;
                    run_z[slot] = z;
                    if (warp == 4 && lane == 0) SN_ACC(4);
                    umma::fence_before_sync();
                    __syncwarp();
                    if (lane == 0) umma::mbar_arrive(&t_empty[buf]);
                }
            }
#pragma unroll
            for (int qh = 0; qh < kQHalves; ++qh) {
                if (kQHalves > 1 && (qh & 1) != wg) continue;
                const int r = qh * 128 + ew * 32 + lane;
                if (r < NQ) {
                    // one Q block: both buffers (alternate tiles) x both column halves hold partial stats;
                    // several Q blocks: the block's buffer is fixed, two column halves
                    const int p_idx = (kQHalves == 1) ? (part * 4 + wg * 2 + ch) : (part * 2 + ch);
                    sc.partial[((size_t)row * NQ + r) * n_parts + p_idx] =
                        make_float2(run_m[qh >> 1] * c, run_z[qh >> 1]);  // (max in log2 units, sum)
                }
            }
        }
    }
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 2) umma::tmem_dealloc(tmem, 256);
}

// ---- pass 2: normalised column sums --------------------------------------------------------------------
template <typename T, int D, int NQP>
__global__ void __launch_bounds__(kSnThreads, 1)
snap_colsum_kernel(const __grid_constant__ CUtensorMap mapK, const __grid_constant__ CUtensorMap mapQ, int H,
                   int G, int S, int window, int R, int n_tiles128, int ctas_per_row, int n_parts,
                   SnapScratch sc, int S_pad) {
    using L = SnSmem<D, NQP>;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>(
        (reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    unsigned char* s_q = smem + L::kQOff;
    unsigned char* s_stage = smem + L::kStageOff;
    unsigned char* s_ax = smem + L::kAxOff;
    unsigned char* s_bx = smem + L::kBxOff;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::kBarOff);
    uint64_t* k_full = bars;
    uint64_t* k_empty = bars + 2;
    uint64_t* t_full = bars + 4;
    uint64_t* t_empty = bars + 6;
    uint64_t* q_full = bars + 8;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 10);

    constexpr int kNChunks = (NQP + 255) / 256;        // MMAs of N <= 256 per tile
    constexpr int kNPer = NQP / kNChunks;              // N of each MMA (128 or 256)
    constexpr int kBufCols = 256;
    const int NQ = G * window;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n_groups = gridDim.x / ctas_per_row;
    const int group = blockIdx.x / ctas_per_row;
    const int part = blockIdx.x % ctas_per_row;

    if (tid == 0) {
        umma::prefetch_tmap(&mapK);
        umma::prefetch_tmap(&mapQ);
        for (int i = 0; i < 2; ++i) {
            umma::mbar_init(&k_full[i], 1);
            umma::mbar_init(&k_empty[i], 1);
            umma::mbar_init(&t_full[i], 1);
            umma::mbar_init(&t_empty[i], 8);
        }
        umma::mbar_init(q_full, 1);
        umma::mbar_fence_init();
    }
    if (warp == 2) umma::tmem_alloc(tmem_slot, 512);
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = *tmem_slot;

    // only positions < S - window receive a score: tiles beyond are skipped entirely
    const int n_tiles_scored = min(n_tiles128, (S - window + kSnTile - 1) / kSnTile);
    const int tiles_per_part = (n_tiles_scored + ctas_per_row - 1) / ctas_per_row;
    const int t_begin = part * tiles_per_part;
    const int t_end = min(n_tiles_scored, t_begin + tiles_per_part);
    const float c = kLog2e * rsqrtf((float)D);

    uint32_t k_it = 0, h_it = 0, q_it = 0;
    for (int row = group; row < R; row += n_groups) {
        const int b = row / H, h = row % H;
        const int q_row0 = (b * (H * G) + h * G) * window;
        __syncthreads();
        // bias operand (hi/lo split) and the ones operand, both in the no-swizzle K=16 layout
        for (int n = tid; n < NQP; n += kSnThreads) {
            // exact normaliser of query row n from the per-CTA partials of pass 1:
            // p[n, j] = exp2(c*y - m) / Z = exp2(c * (y + bias)),  bias = (-m - log2 Z) / c
            // padding rows (n >= NQ): a bias that drives exp2(c * (y + bias)) to exactly 0, so a 16-column chunk
            // that straddles NQ (windows that are not multiples of 16) adds nothing for them
            float bias = -60000.f;
            if (n < NQ) {
                float m = -INFINITY, z = 0.f;
                const float2* part_n = sc.partial + ((size_t)row * NQ + n) * n_parts;
                for (int pp = 0; pp < n_parts; ++pp) {
                    const float2 pz = part_n[pp];
                    const float mn = fmaxf(m, pz.x);
                    z = (mn == -INFINITY) ? 0.f : z * fast_exp2(m - mn) + pz.y * fast_exp2(pz.x - mn);
                    m = mn;
                }
                bias = (-m - log2f(z)) / c;
            }
            const uint16_t hi = F16Traits<T>::from_float(bias);
            const uint16_t lo = F16Traits<T>::from_float(bias - F16Traits<T>::to_float(hi));
            *reinterpret_cast<uint4*>(s_bx + umma::k16_noswizzle_offset(n, 0)) =
                make_uint4((uint32_t)hi | ((uint32_t)lo << 16), 0u, 0u, 0u);
            *reinterpret_cast<uint4*>(s_bx + umma::k16_noswizzle_offset(n, 1)) = make_uint4(0u, 0u, 0u, 0u);
        }
        if (tid < kSnTile) {
            const uint32_t one = (uint32_t)F16Traits<T>::from_float(1.0f);
            *reinterpret_cast<uint4*>(s_ax + umma::k16_noswizzle_offset(tid, 0)) =
                make_uint4(one | (one << 16), 0u, 0u, 0u);
            *reinterpret_cast<uint4*>(s_ax + umma::k16_noswizzle_offset(tid, 1)) = make_uint4(0u, 0u, 0u, 0u);
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncthreads();

        if (warp == 0) {
            if (lane == 0) {
                // all NQP resident rows are loaded (boxes of min(NQP, 256) rows): rows >= NQ belong to the next kv
                // head or lie past the tensor (zero fill); their outputs are never read
                umma::mbar_arrive_expect_tx(q_full, (uint32_t)(L::kPanels * NQP * 128));
                for (int kp = 0; kp < L::kPanels; ++kp)
                    for (int r0 = 0; r0 < NQP; r0 += 256)
                        umma::tma_load_3d(s_q + kp * L::kQPanel + r0 * 128, &mapQ, q_full, kp * 64,
                                          q_row0 + r0, 0);
                for (int t = t_begin; t < t_end; ++t, ++k_it) {
                    const int stage = k_it & 1;
                    umma::mbar_wait(&k_empty[stage], ((k_it >> 1) & 1) ^ 1);
                    umma::mbar_arrive_expect_tx(&k_full[stage], L::kStageBytes);
                    for (int kp = 0; kp < L::kPanels; ++kp)
                        umma::tma_load_4d(s_stage + stage * L::kStageBytes + kp * (kSnTile * 128), &mapK,
                                          &k_full[stage], kp * 64, t * kSnTile, h, b);
                }
            }
        } else if (warp == 1) {
            if (lane == 0) {
                const uint32_t idesc = umma::instr_desc_f16(kSnTile, kNPer, F16Traits<T>::kMmaFormat);
                umma::mbar_wait(q_full, q_it & 1);
                for (int t = t_begin; t < t_end; ++t, ++k_it) {
                    const int stage = k_it & 1;
                    umma::mbar_wait(&k_full[stage], (k_it >> 1) & 1);
                    umma::fence_after_sync();
                    const uint32_t kb = umma::smem_u32(s_stage + stage * L::kStageBytes);
#pragma unroll 1
                    for (int nc = 0; nc < kNChunks; ++nc, ++h_it) {
                        const int buf = h_it & 1;
                        umma::mbar_wait(&t_empty[buf], ((h_it >> 1) & 1) ^ 1);
                        umma::fence_after_sync();
#pragma unroll
                        for (int k = 0; k < D / 16; ++k) {
                            const int kp = k >> 2, kk = k & 3;
                            const uint64_t da = umma::smem_desc_sw128(kb + kp * (kSnTile * 128) + kk * 32);
                            const uint64_t db = umma::smem_desc_sw128(
                                umma::smem_u32(s_q + kp * L::kQPanel + nc * (kNPer * 128)) + kk * 32);
                            umma::mma_f16_ss(tmem + buf * kBufCols, da, db, idesc, k > 0);
                        }
                        umma::mma_f16_ss(tmem + buf * kBufCols,
                                         umma::smem_desc_k16_noswizzle(umma::smem_u32(s_ax)),
                                         umma::smem_desc_k16_noswizzle(umma::smem_u32(s_bx) +
                                                                       (nc * kNPer / 8) * 256),
                                         idesc, 1);
                        umma::mma_commit(&t_full[buf]);
                    }
                    umma::mma_commit(&k_empty[stage]);
                }
            }
            ++q_it;
        } else if (warp >= 4) {
            // ===== epilogue: thread = key; warpgroup (buf, ch) sums exp2(c * D[key, r]) over column half ch
            // (query rows) of TMEM buffer buf; the halves meet in global memory with one atomicAdd each =====
            const int wgi = (warp - 4) >> 2;
            const int wg = wgi & 1;
            const int ch = wgi >> 1;
            const int ew = warp & 3;
            const uint32_t lane_base = (uint32_t)(ew * 32) << 16;
            constexpr int kHalfCols = kNPer / 2;
            for (int t = t_begin; t < t_end; ++t) {
                const int pos = t * kSnTile + ew * 32 + lane;
                float total = 0.f;
                bool mine = false;
#pragma unroll 1
                for (int nc = 0; nc < kNChunks; ++nc, ++h_it) {
                    const int buf = h_it & 1;
                    if (buf != wg) continue;
                    mine = true;
                    umma::mbar_wait(&t_full[buf], (h_it >> 1) & 1);
                    umma::fence_after_sync();
                    const uint32_t tbase = tmem + lane_base + buf * kBufCols + ch * kHalfCols;
                    // real query rows in this warpgroup's column half
                    const int n_cols = max(0, min(kHalfCols, NQ - nc * kNPer - ch * kHalfCols));
                    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
                    if (n_cols > 0) {
                        uint32_t y0[16], y1[16];
                        umma::tmem_ld16(tbase, y0);
                        auto accumulate = [&](const uint32_t (&yy)[16]) {
#pragma unroll
                            for (int j = 0; j < 16; j += 4) {
                                a0 += fast_exp2(__uint_as_float(yy[j]) * c);
                                a1 += fast_exp2(__uint_as_float(yy[j + 1]) * c);
                                a2 += fast_exp2(__uint_as_float(yy[j + 2]) * c);
                                a3 += fast_exp2(__uint_as_float(yy[j + 3]) * c);
                            }
                        };
                        // two 16-column chunks per iteration so both register buffers are static
#pragma unroll 1
                        for (int c0 = 0; c0 < n_cols; c0 += 32) {
                            umma::tmem_ld_wait();
                            const bool more1 = (c0 + 16) < n_cols;
                            if (more1) umma::tmem_ld16(tbase + c0 + 16, y1);
                            accumulate(y0);
                            if (more1) {
                                umma::tmem_ld_wait();
                                if (c0 + 32 < n_cols) umma::tmem_ld16(tbase + c0 + 32, y0);
                                accumulate(y1);
                            }
                        }
                    }
                    total += (a0 + a1) + (a2 + a3);
                    umma::fence_before_sync();
                    __syncwarp();
                    if (lane == 0) umma::mbar_arrive(&t_empty[buf]);
                }
                if (mine && pos < S - window) atomicAdd(&sc.colsum[(size_t)row * S_pad + pos], total);
            }
        }
    }
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 2) umma::tmem_dealloc(tmem, 512);
}

// ---- finalize: scaling, box filter, ONE rounding, keys + histogram -------------------------------------
template <typename T>
__global__ void __launch_bounds__(kTileThreads)
snap_finalize_kernel(int S, int window, int kernel_size, float inv_gw, SnapScratch sc, Workspace ws,
                     uint16_t* __restrict__ scores_out) {
    __shared__ uint16_t skeys[kTile];
    __shared__ uint16_t sscores[kTile];
    __shared__ uint32_t shist[256];
    __shared__ float s_max[8];
    const int tile = blockIdx.x, row = blockIdx.y, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    shist[tid] = 0;
    pdl_launch_dependents();  // the selection pass behind this one may start to take residency
    const int n_scored = S - window;
    float fmax_valid = -INFINITY;
    for (int sub = 0; sub < kFinalizeTiles; ++sub) {
        const int t = tile * kFinalizeTiles + sub;
        if (t >= ws.n_tiles) break;
        const int s = t * kTile + tid;
        uint16_t bits = 0, key = 0;
        if (s < S) {
            if (s >= n_scored) {
                key = kForcedKey;
            } else {
                const int half = kernel_size >> 1;
                float acc = 0.f;
                for (int o = -half; o <= half; ++o) {
                    const int j = s + o;
                    if (j >= 0 && j < n_scored) acc += sc.colsum[(size_t)row * ws.S_pad + j];
                }
                const float score = acc * inv_gw / (float)kernel_size;  // count_include_pad: always / kernel
                bits = F16Traits<T>::from_float(score);
                key = ordered_key16(bits, F16Traits<T>::kInfBits);
                fmax_valid = fmaxf(fmax_valid, F16Traits<T>::to_float(bits));
            }
        }
        __syncthreads();
        skeys[tid] = key;
        sscores[tid] = bits;
        __syncthreads();
        flush_chunk_keys<1, false>(skeys, sscores, shist, row, t * kTile, S, ws, scores_out);
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1)
        fmax_valid = fmaxf(fmax_valid, __shfl_xor_sync(0xFFFFFFFFu, fmax_valid, off));
    if (lane == 0) s_max[warp] = fmax_valid;
    __syncthreads();
    if (tid == 0) {
        float m = s_max[0];
        for (int w = 1; w < 8; ++w) m = fmaxf(m, s_max[w]);
        if (m > -INFINITY) {
            const uint32_t u = __float_as_uint(m);
            atomicMax(&ws.counters[kCounterMaxSlot(ws.R)], (u & 0x80000000u) ? ~u : (u | 0x80000000u));
        }
    }
    flush_row_hist(shist, row, ws);
}

// ---- host launcher -----------------------------------------------------------------------------------------
template <typename T, int D, int NQP>
static cudaError_t launch_snap_t(const Dims& d, int dtype, const void* K, const void* q_window, int window,
                                 int kernel_size, const Workspace& ws, void* scores_out, cudaStream_t st) {
    using L = SnSmem<D, NQP>;
    const int sm_count = device_sm_count();
    const int G = d.Hq / d.H;
    const int NQ = G * window;
    const SnapScratch sc = carve_snap(d, window, ws);
    const int n_tiles128 = (d.S + kSnTile - 1) / kSnTile;
    int ctas_per_row = sm_count / d.R;
    if (ctas_per_row < 1) ctas_per_row = 1;
    if (ctas_per_row > n_tiles128) ctas_per_row = n_tiles128;
    if (ctas_per_row > kSnMaxParts / 4) ctas_per_row = kSnMaxParts / 4;
    int n_groups = sm_count / ctas_per_row;
    if (n_groups > d.R) n_groups = d.R;
    const int grid = n_groups * ctas_per_row;
    const int n_parts = (NQP == 128) ? ctas_per_row * 4 : ctas_per_row * 2;

    CUtensorMap mapK, mapQ;
    {
        const uint64_t row_b = (uint64_t)d.ks.s * 2;
        const uint64_t h_b = d.H > 1 ? (uint64_t)d.ks.h * 2 : row_b * (uint64_t)d.S;
        const uint64_t b_b = d.B > 1 ? (uint64_t)d.ks.b * 2 : h_b * (uint64_t)d.H;
        const uint64_t dims[4] = {(uint64_t)D, (uint64_t)d.S, (uint64_t)d.H, (uint64_t)d.B};
        const uint64_t str[4] = {0, row_b, h_b, b_b};
        const uint32_t box[4] = {64, (uint32_t)kSnTile, 1, 1};
        cudaError_t e = make_tmap_16bit(&mapK, K, 4, dims, str, box);
        if (e != cudaSuccess) return e;
    }
    {
        const uint64_t rows = (uint64_t)d.B * d.Hq * window;
        const uint64_t dims[3] = {(uint64_t)D, rows, 1};
        const uint64_t str[3] = {0, (uint64_t)D * 2, rows * D * 2};
        const uint32_t box[3] = {64, (uint32_t)(NQP < 256 ? NQP : 256), 1};
        cudaError_t e = make_tmap_16bit(&mapQ, q_window, 3, dims, str, box);
        if (e != cudaSuccess) return e;
    }
    const int smem = L::kTotal + 1024;
    auto k1 = snap_stats_kernel<T, D, NQP>;
    auto k2 = snap_colsum_kernel<T, D, NQP>;
    static PerDeviceOnce smem_set1, smem_set2;  // one pair per <T, D, NQP> instantiation of this launcher
    cudaError_t e = ensure_dynamic_smem(k1, smem, smem_set1);
    if (e != cudaSuccess) return e;
    e = ensure_dynamic_smem(k2, smem, smem_set2);
    if (e != cudaSuccess) return e;

    k1<<<grid, kSnThreads, smem, st>>>(mapK, mapQ, d.H, G, d.S, window, d.R, n_tiles128, ctas_per_row,
                                       n_parts, sc);
    if ((e = cudaPeekAtLastError()) != cudaSuccess) return e;
    e = cudaMemsetAsync(sc.colsum, 0, (size_t)d.R * ws.S_pad * 4, st);  // warpgroups add their halves
    if (e != cudaSuccess) return e;
    k2<<<grid, kSnThreads, smem, st>>>(mapK, mapQ, d.H, G, d.S, window, d.R, n_tiles128, ctas_per_row, n_parts,
                                       sc, ws.S_pad);
    if ((e = cudaPeekAtLastError()) != cudaSuccess) return e;
    dim3 grid3((ws.n_tiles + kFinalizeTiles - 1) / kFinalizeTiles, d.R);
    snap_finalize_kernel<T><<<grid3, kTileThreads, 0, st>>>(d.S, window, kernel_size, 1.0f / (float)NQ, sc, ws,
                                                            static_cast<uint16_t*>(scores_out));
    if ((e = cudaPeekAtLastError()) != cudaSuccess) return e;
    if (scores_out != nullptr)
        e = launch_fill_sentinel(dtype, scores_out, d.R, d.S, d.S - window, d.S, ws, st);
    return e;
}

template <typename T>
static cudaError_t launch_snap_d(const Dims& d, int dtype, const void* K, const void* q_window, int window,
                                 int kernel_size, const Workspace& ws, void* scores_out, cudaStream_t st) {
    const int G = d.Hq / d.H;
    const int NQ = G * window;
    // any group size / window with G * window <= 512 query rows per kv head: the resident Q block is padded to
    // 128 / 256 / 512 rows, padding rows are computed and ignored (Llama-3.2-3B: G = 3, Qwen2-7B: G = 7, ...)
    if (NQ < 1 || NQ > 512) return cudaErrorNotSupported;
    const int NQP = NQ <= 128 ? 128 : (NQ <= 256 ? 256 : 512);
#define KVP_SNAP(DD, NN) \
    if (d.D == DD && NQP == NN) return launch_snap_t<T, DD, NN>(d, dtype, K, q_window, window, kernel_size, ws, scores_out, st)
    KVP_SNAP(128, 128);
    KVP_SNAP(128, 256);
    KVP_SNAP(128, 512);
    KVP_SNAP(64, 128);
    KVP_SNAP(64, 256);
    KVP_SNAP(64, 512);
#undef KVP_SNAP
    return cudaErrorNotSupported;
}

cudaError_t launch_snapkv_score(const Dims& d, int dtype, const void* K, const void* q_window, int window,
                                int kernel_size, const Workspace& ws, void* scores_out, bool want_keys,
                                cudaStream_t st) {
    (void)want_keys;
    if (dtype == KVP_BF16)
        return launch_snap_d<__nv_bfloat16>(d, dtype, K, q_window, window, kernel_size, ws, scores_out, st);
    return launch_snap_d<__half>(d, dtype, K, q_window, window, kernel_size, ws, scores_out, st);
}

}  // namespace kvp
