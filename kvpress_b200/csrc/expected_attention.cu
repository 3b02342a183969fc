// expected_attention.cu — stage S for ExpectedAttentionPress (sm_100a: TMA + tcgen05 + TMEM).
//
// Reference semantics (kvpress/presses/expected_attention_press.py:136-165), per kv head h and each
// of its G = Hq/Hkv query heads g, over positions s in [n_sink, S):
//     logit_g(s) = mu_g . k_s / sqrt(d) + k_s^T Sigma_g k_s / (2 d)              (:149-151)
//     p_g        = softmax_s(logit_g)                                              (:152)
//     score(s)   = mean_g p_g(s)          [* ||v_s||_2 after adding epsilon]       (:155-160)
//   and the n_sink first positions are forced to be kept (:163).
// The reference materialises repeat_kv(K)^T twice and a [B,Hq,D,S] einsum intermediate; here
//   kernel 1 (ea_logits_kernel, persistent, one CTA per SM, warp-specialised):
//       TMA streams 128-position K tiles (SWIZZLE_128B) into a 2-stage ring; one thread issues
//       tcgen05.mma  Y = K_tile[128 x D] * Sigma_g^T  for two heads at a time (N = 2D <= 256) into one
//       of two TMEM accumulator buffers; four epilogue warps read Y back (tcgen05.ld, thread = key
//       row) and finish  logit = sum_n k_n (Y_n + 2 sqrt(d) mu_n) / (2d)  with the k row taken from
//       the same shared-memory tile, keep online softmax statistics and store fp32 logits; four
//       more warps stream the matching V rows and store ||v||. Sigma for the G heads (G*D*D*2 bytes)
//       stays resident in shared memory for the CTA's whole range.
//   kernel 2 (ea_finalize_kernel): combines the per-CTA softmax statistics, forms the final score in
//       fp32, rounds it ONCE to the cache dtype, and emits keys + histogram for the select stage.
// Covariance-free mode (use_covariance=False) is a plain streaming GEMV kernel.
#include <mutex>
#include <stdlib.h>

#include "common.cuh"
#include "knorm_chunk.cuh"
#include "umma.cuh"

// Triangular quadratic form — EXPERIMENT, default off (measured slower, profiles/r02_ab_ea_tri_hint.txt).
// k^T cov k = sum_n k_n (sum_{c<=n} T[n][c] k_c) with T[n][c] = cov[n][c] + cov[c][n] (c < n), cov[n][n] (c == n),
// 0 (c > n), built once per call by ea_cov_tri_kernel into the scratch (exact whenever cov is symmetric, <= 2^-9
// relative per entry otherwise). The B operand of K-step k (contraction columns c in [16k, 16k+16)) then has no
// non-zero rows n < 16k, so the MMA warp issues that step on rows [32*(k/2), D) only: per head 2*(128+96+64+32) = 640
// instead of 1024 N-units at head_dim 128 (-37.5 % tensor work on paper). On the B200 the 15 narrower MMAs per
// head pair (N = 256, 96, 64, 32) take LONGER than the 9 full-width ones: ea_logits_kernel 122 us vs 115 us, the
// whole call 251 us vs 226 us. Parity-tested (all ExpectedAttention GPU tests pass with it on).
#ifndef KVP_EA_TRI
#define KVP_EA_TRI 0
#endif

// TIMING-ONLY experiment knobs (wrong results; used by tools/ea_experiments.py to locate the limiter of the logits
// kernel): bit 0 = the epilogue does not read the k row from shared memory, bit 1 = no bias MMA step, bit 2 = the
// epilogue does not read the accumulator at all (waits and releases only).
#ifndef KVP_EA_EXP
#define KVP_EA_EXP 0
#endif
// CTA-pair kernel knob: KVP_EA_EXP2 = TIMING-ONLY
// (wrong results): bit 0 = the epilogue reads only the first head of each pair from tensor memory, bit 1 = no logits
// stores, bit 2 = no accumulator read-back / k-row reads / FMAs at all, bit 3 = no online-softmax exponentials, bit 4 = no bias MMA
#ifndef KVP_EA_EXP2
#define KVP_EA_EXP2 0
#endif
#ifndef KVP_EA_PAIR_BOUNDS
#define KVP_EA_PAIR_BOUNDS 384   // __launch_bounds__ of the pair kernel (384 threads): up to 168 registers (512 -> 128: +3.6 us, run17)
#endif

namespace kvp {

#ifdef KVP_EA_PROFILE
__device__ long long g_ea_prof[32];
#define EA_T0() const long long _t0 = clock64()
#define EA_ACC(slot) do { if (blockIdx.x == 0) g_ea_prof[slot] += clock64() - _t0; } while (0)
#define EA_T1() const long long _t1 = clock64()
#define EA_ACC1(slot) do { if (blockIdx.x == 0) g_ea_prof[slot] += clock64() - _t1; } while (0)
#else
#define EA_T0() do {} while (0)
#define EA_ACC(slot) do {} while (0)
#define EA_T1() do {} while (0)
#define EA_ACC1(slot) do {} while (0)
#endif

constexpr int kEaTile = 128;      // key rows per MMA tile (M)
constexpr int kEaThreads = 384;   // 12 warps: TMA, MMA, TMEM-alloc, spare, 2 x 4 epilogue
constexpr int kEaMaxParts = 160;  // upper bound on CTAs per (b,h) row (>= SM count)

struct EaScratch {
    float* logits;    // [R][G][S_pad]
    float* vnorm;     // [R][S_pad]
    float2* partial;  // [R][G][n_parts] (max, sum exp) per CTA part
#if KVP_EA_TRI
    uint16_t* cov_tri;  // [B*Hq][D][D] lower-triangular form of cov
#endif
};

static inline size_t align256(size_t x) { return (x + 255) / 256 * 256; }

size_t ea_scratch_bytes(const Dims& d) {
    const int G = d.Hq / d.H;
    const size_t S_pad = (size_t)((d.S + kTile - 1) / kTile) * kTile;
    const size_t n_parts = (size_t)((d.S + kScoreChunkGeneric - 1) / kScoreChunkGeneric);
    const size_t parts = n_parts > kEaMaxParts ? n_parts : kEaMaxParts;
    return align256((size_t)d.R * G * S_pad * 4) + align256((size_t)d.R * S_pad * 4) +
           align256((size_t)d.R * G * parts * sizeof(float2))
#if KVP_EA_TRI
           + align256((size_t)d.B * d.Hq * d.D * d.D * 2)
#endif
        ;
}

static EaScratch carve_ea(const Dims& d, const Workspace& ws) {
    const int G = d.Hq / d.H;
    const size_t S_pad = (size_t)ws.S_pad;
    char* p = static_cast<char*>(ws.scorer);
    EaScratch s;
    s.logits = reinterpret_cast<float*>(p);
    p += align256((size_t)d.R * G * S_pad * 4);
    s.vnorm = reinterpret_cast<float*>(p);
    p += align256((size_t)d.R * S_pad * 4);
    s.partial = reinterpret_cast<float2*>(p);
#if KVP_EA_TRI
    {
        const size_t n_parts = (size_t)((d.S + kScoreChunkGeneric - 1) / kScoreChunkGeneric);
        const size_t parts = n_parts > kEaMaxParts ? n_parts : kEaMaxParts;
        p += align256((size_t)d.R * G * parts * sizeof(float2));
        s.cov_tri = reinterpret_cast<uint16_t*>(p);
    }
#endif
    return s;
}

// ---- shared-memory carve-up of ea_logits_kernel ---------------------------------------------------
template <int D, int G>
struct EaSmem {
    static constexpr int kPanels = D / 64;                 // 64-element (128 B) K panels
    static constexpr int kCovHeadPanel = D * 128;          // bytes of one head's [D x 64] panel
    static constexpr int kCovBytes = G * kPanels * kCovHeadPanel;
    static constexpr int kStageBytes = kPanels * kEaTile * 128;
    // K-tile ring: as deep as shared memory allows (4 when at most two heads' covariance is resident). With two
    // stages a tile has ONE tile time to arrive after its slot is released; any extra HBM latency (the concurrent
    // value-norm kernel) then starves the MMA pipe (profiles/r02_ea_experiments.txt).
    // V tiles (value norms computed inside this kernel): with at most two resident heads every tile leaves one epilogue
    // warpgroup idle, and there is room for a 2-stage V ring staged by TMA next to the K ring
#ifndef KVP_EA_V_STAGES
#define KVP_EA_V_STAGES 1  // A/B knob: 0 = value norms by the side-stream kernel, 1 / 2 = V ring depth inside this kernel
#endif
    static constexpr int kVStages = (G <= 2) ? KVP_EA_V_STAGES : 0;
    static constexpr int kFixedBytes = kCovBytes + kEaTile * 32 + G * D * 32 + 512 + 1024 + kVStages * kStageBytes;
    // as many K stages as fit, at most 4 (two units per row halve the tile time of a CTA: run6 measured the two-head
    // layout at 154 us with 2 stages against 116 us with 4)
    static constexpr int kFit = (227 * 1024 - kFixedBytes) / kStageBytes;
    static constexpr int kStages = kFit >= 4 ? 4 : (kFit >= 2 ? kFit : 2);
    static constexpr int kCovOff = 0;
    static constexpr int kStageOff = kCovBytes;
    // extra K=16 step that adds 2 sqrt(d) mu_g[n] to Y_g[.,n] inside the MMA: A-extra = [128 x 16]
    // with columns 0,1 = 1.0; B-extra = [G*D x 16] with column 0/1 = hi/lo halves of the bias
    static constexpr int kVStageOff = kStageOff + kStages * kStageBytes;
    static constexpr int kAxOff = kVStageOff + kVStages * kStageBytes;  // 128 rows * 32 B
    static constexpr int kBxOff = kAxOff + kEaTile * 32;                // G*D rows * 32 B
    static constexpr int kBarOff = kBxOff + G * D * 32;
    static constexpr int kTotal = kBarOff + 512;
    static_assert(kTotal + 1024 <= 227 * 1024, "shared memory budget");
};

// __launch_bounds__(512): ptxas keeps the kernel at <= 128 registers/thread (it is launched with
// kEaThreads = 384), leaving 16 K registers per SM for a co-resident ea_vnorm_kernel CTA.
template <typename T, int D, int G>
__global__ void __launch_bounds__(512, 1)
ea_logits_kernel(const __grid_constant__ CUtensorMap mapK, const __grid_constant__ CUtensorMap mapCov,
                 const __grid_constant__ CUtensorMap mapV, const T* __restrict__ mu, int H, int Hq, int S, int n_sink,
                 int R, int n_tiles128, int ctas_per_row, int n_parts, EaScratch sc, int S_pad, int g_total,
                 int n_split, int do_vnorm) {
    using L = EaSmem<D, G>;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    // dynamic shared memory is only guaranteed 16-B aligned: round up to 1024 B for the swizzle
    unsigned char* smem = reinterpret_cast<unsigned char*>(
        (reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    unsigned char* s_cov = smem + L::kCovOff;
    unsigned char* s_stage = smem + L::kStageOff;
    unsigned char* s_vstage = smem + L::kVStageOff;
    unsigned char* s_ax = smem + L::kAxOff;
    unsigned char* s_bx = smem + L::kBxOff;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::kBarOff);
    constexpr int kStages = L::kStages;
    uint64_t* k_full = bars;          // [kStages <= 4]
    uint64_t* k_empty = bars + 4;     // [kStages]
    uint64_t* t_full = bars + 8;      // [2]
    uint64_t* t_empty = bars + 10;    // [2]
    uint64_t* cov_full = bars + 12;   // [1]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 13);
    uint64_t* v_full = bars + 14;     // [2]
    uint64_t* v_empty = bars + 16;    // [2]
    float* s_red = reinterpret_cast<float*>(bars + 18);  // [8 warps][2 heads][2], then [2 wg][2][2]
    constexpr bool kInKernelV = L::kVStages > 0;

    constexpr int kHalves = (G + 1) / 2;          // head pairs per tile
    constexpr int HPH = (G >= 2) ? 2 : 1;         // heads per half
    constexpr int kN = HPH * D;                   // MMA N
    constexpr int kBufCols = 256;
    constexpr int kChunks = D / 32;
    static_assert(kN <= 256, "two heads must fit one MMA");

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
#ifdef KVP_EA_PROFILE
    const long long t_entry = clock64();
#endif

    // ---- which (row, tile range) this CTA owns; rows are visited round-robin -----------------------
    const int n_groups = gridDim.x / ctas_per_row;  // concurrent rows
    const int group = blockIdx.x / ctas_per_row;
    const int part = blockIdx.x % ctas_per_row;

    if (tid == 0) {
        umma::prefetch_tmap(&mapK);
        umma::prefetch_tmap(&mapCov);
        if (kInKernelV && do_vnorm) umma::prefetch_tmap(&mapV);
        for (int i = 0; i < kStages; ++i) {
            umma::mbar_init(&k_full[i], 1);
            umma::mbar_init(&k_empty[i], 1 + 8);  // MMA commit + 8 epilogue warps
        }
        for (int i = 0; i < 2; ++i) {
            umma::mbar_init(&t_full[i], 1);
            umma::mbar_init(&t_empty[i], 4);      // the 4 warps of the warpgroup that drained it
            umma::mbar_init(&v_full[i], 1);
            umma::mbar_init(&v_empty[i], 4);      // the 4 warps of the warpgroup that took the norms
        }
        umma::mbar_init(cov_full, 1);
        umma::mbar_fence_init();
    }
    if (warp == 2) umma::tmem_alloc(tmem_slot, 512);
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = *tmem_slot;

    const int tiles_per_part = (n_tiles128 + ctas_per_row - 1) / ctas_per_row;
    const int t_begin = part * tiles_per_part;
    const int t_end = min(n_tiles128, t_begin + tiles_per_part);
    const float inv_2d = 1.0f / (2.0f * (float)D);
    const float bias_scale = 2.0f * sqrtf((float)D);

    // pipeline state carried across rows (barriers keep flipping)
    uint32_t k_it = 0;  // tiles seen by this role
    uint32_t h_it = 0;  // halves seen by this role
    uint32_t cov_it = 0;
    uint32_t v_it = 0;  // V tiles this CTA owns, seen by this role

    // work unit = (row, group of G query heads of that kv head): the n_split units of a row run on different CTAs at the
    // same time and stream the same K tiles (the second reader finds them in L2), each with only its own heads'
    // covariance resident — which is what leaves room for the deeper K ring
    const int n_units = R * n_split;
    for (int unit = group; unit < n_units; unit += n_groups) {
        const int row = unit / n_split, pair = unit % n_split, g_off = pair * G;
        const int b = row / H, h = row % H;
        // the units of a row see the same tiles: unit `pair` also stages V and takes the value norms of the tiles
        // t with t % n_split == pair
        const bool v_active = kInKernelV && do_vnorm != 0;
        // this unit covers query heads [g_off, g_off + G) of the kv head's g_total heads
        const int hq0 = b * Hq + h * g_total + g_off;  // first of them in [B*Hq]
        __syncthreads();  // previous row fully drained (s_bias, s_cov, s_red reusable)
        for (int n = tid; n < G * D; n += kEaThreads) {
            // resident slot n / D may be a padding head (g_total not a multiple of the template's G): no bias
            const float bias = (g_off + n / D < g_total)
                                   ? bias_scale * F16Traits<T>::to_float(
                                                      reinterpret_cast<const uint16_t*>(mu)[(size_t)hq0 * D + n])
                                   : 0.f;
            const uint16_t hi = F16Traits<T>::from_float(bias);
            const uint16_t lo = F16Traits<T>::from_float(bias - F16Traits<T>::to_float(hi));
            *reinterpret_cast<uint4*>(s_bx + umma::k16_noswizzle_offset(n, 0)) =
                make_uint4((uint32_t)hi | ((uint32_t)lo << 16), 0u, 0u, 0u);
            *reinterpret_cast<uint4*>(s_bx + umma::k16_noswizzle_offset(n, 1)) = make_uint4(0u, 0u, 0u, 0u);
        }
        if (tid < kEaTile) {
            const uint32_t one = (uint32_t)F16Traits<T>::from_float(1.0f);
            *reinterpret_cast<uint4*>(s_ax + umma::k16_noswizzle_offset(tid, 0)) =
                make_uint4(one | (one << 16), 0u, 0u, 0u);
            *reinterpret_cast<uint4*>(s_ax + umma::k16_noswizzle_offset(tid, 1)) = make_uint4(0u, 0u, 0u, 0u);
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic writes -> UMMA reads
        __syncthreads();

        if (warp == 0) {
            // ===== TMA producer =====
            if (lane == 0) {
                umma::mbar_arrive_expect_tx(cov_full, L::kCovBytes);
                for (int kp = 0; kp < L::kPanels; ++kp)
                    for (int g = 0; g < G; ++g)
                        umma::tma_load_3d(s_cov + (kp * G + g) * L::kCovHeadPanel, &mapCov, cov_full,
                                          kp * 64, 0, hq0 + g);
                for (int t = t_begin; t < t_end; ++t, ++k_it) {
                    const int stage = k_it % kStages;
                    { EA_T0(); umma::mbar_wait(&k_empty[stage], ((k_it / kStages) & 1) ^ 1); EA_ACC(0); }
                    umma::mbar_arrive_expect_tx(&k_full[stage], L::kStageBytes);
                    for (int kp = 0; kp < L::kPanels; ++kp)
                        umma::tma_load_4d(s_stage + stage * L::kStageBytes + kp * (kEaTile * 128),
                                          &mapK, &k_full[stage], kp * 64, t * kEaTile, h, b);
                }
            }
        } else if (warp == 3) {
            // ===== V producer (own thread: a full V ring must never hold back the K prefetch) =====
            if (lane == 0 && v_active) {
                constexpr int kVS = L::kVStages > 0 ? L::kVStages : 1;
                for (int t = t_begin; t < t_end; ++t) {
                    if ((t % n_split) != pair) continue;
                    const int vs_i = v_it % kVS;
                    umma::mbar_wait(&v_empty[vs_i], ((v_it / kVS) & 1) ^ 1);
                    umma::mbar_arrive_expect_tx(&v_full[vs_i], L::kStageBytes);
                    for (int kp = 0; kp < L::kPanels; ++kp)
                        umma::tma_load_4d(s_vstage + vs_i * L::kStageBytes + kp * (kEaTile * 128), &mapV,
                                          &v_full[vs_i], kp * 64, t * kEaTile, h, b);
                    ++v_it;
                }
            }
        } else if (warp == 1) {
            // ===== MMA issuer =====
            if (lane == 0) {
                const uint32_t idesc = umma::instr_desc_f16(kEaTile, kN, F16Traits<T>::kMmaFormat);
                umma::mbar_wait(cov_full, cov_it & 1);
                for (int t = t_begin; t < t_end; ++t, ++k_it) {
                    const int stage = k_it % kStages;
                    { EA_T0(); umma::mbar_wait(&k_full[stage], (k_it / kStages) & 1); EA_ACC(1); }
                    umma::fence_after_sync();
                    const uint32_t a_base = umma::smem_u32(s_stage + stage * L::kStageBytes);
#pragma unroll 1
                    for (int half = 0; half < kHalves; ++half, ++h_it) {
                        const int buf = h_it & 1;
                        { EA_T0(); umma::mbar_wait(&t_empty[buf], ((h_it >> 1) & 1) ^ 1); EA_ACC(2); }
                        umma::fence_after_sync();
#pragma unroll
                        for (int k = 0; k < D / 16; ++k) {
                            const int kp = k >> 2, kk = k & 3;
                            const uint64_t da =
                                umma::smem_desc_sw128(a_base + kp * (kEaTile * 128) + kk * 32);
#if KVP_EA_TRI
                            // rows n < row0 of T are zero in this K-step's columns: issue on rows [row0, D) of
                            // every head (B rows are 128 B apart, 32 rows = four 1024-B swizzle atoms; the
                            // accumulator columns shift by the same row0). k = 0 covers all columns, so every
                            // later step accumulates.
                            constexpr int kGran = 32;
                            const int row0 = (k * 16 / kGran) * kGran;
                            if (row0 > 0) {
                                const uint32_t idesc_n = umma::instr_desc_f16(kEaTile, D - row0, F16Traits<T>::kMmaFormat);
#pragma unroll
                                for (int q = 0; q < HPH; ++q) {
                                    const uint64_t dbq = umma::smem_desc_sw128(
                                        umma::smem_u32(s_cov + (kp * G + half * HPH + q) * L::kCovHeadPanel) +
                                        row0 * 128 + kk * 32);
                                    umma::mma_f16_ss(tmem + buf * kBufCols + q * D + row0, da, dbq, idesc_n, 1);
                                }
                                continue;
                            }
#endif
                            const uint64_t db = umma::smem_desc_sw128(
                                umma::smem_u32(s_cov + (kp * G + half * HPH) * L::kCovHeadPanel) + kk * 32);
                            umma::mma_f16_ss(tmem + buf * kBufCols, da, db, idesc, k > 0);
                        }
#if !(KVP_EA_EXP & 2)
                        umma::mma_f16_ss(tmem + buf * kBufCols,
                                         umma::smem_desc_k16_noswizzle(umma::smem_u32(s_ax)),
                                         umma::smem_desc_k16_noswizzle(
                                             umma::smem_u32(s_bx) + (half * HPH * D / 8) * 256),
                                         idesc, 1);
#endif
                        umma::mma_commit(&t_full[buf]);
                    }
                    umma::mma_commit(&k_empty[stage]);
                }
            }
            ++cov_it;
        } else if (warp >= 4 && warp < 12) {
            // ===== epilogue: two warpgroups, warpgroup wg drains TMEM buffer wg; thread = key row =====
            const int wg = (warp - 4) >> 2;
            const int ew = warp & 3;       // TMEM lane quarter this warp may access
            const int r = ew * 32 + lane;  // row in tile == TMEM lane
            const uint32_t lane_base = (uint32_t)(ew * 32) << 16;
            float run_m[HPH], run_z[HPH];
#pragma unroll
            for (int q = 0; q < HPH; ++q) {
                run_m[q] = -INFINITY;
                run_z[q] = 0.f;
            }
#ifdef KVP_EA_PROFILE
            if (blockIdx.x == 0 && warp == 4 && lane == 0) g_ea_prof[9] += clock64() - t_entry;
#endif
            for (int t = t_begin; t < t_end; ++t, ++k_it) {
                const int stage = k_it % kStages;
                const unsigned char* krow = s_stage + stage * L::kStageBytes;
                const int s = t * kEaTile + r;
                const bool valid = (s >= n_sink) && (s < S);
                bool waited_k = false, released_k = false;
                if (kInKernelV && v_active && (t % n_split) == pair) {
                    // kHalves == 1: exactly one warpgroup has no accumulator to drain for this tile — it takes ||v||.
                    // BOTH warpgroups wait for the V tile: a waiter that skipped a phase of v_full would test the
                    // wrong parity the next time it is the reader (with one V stage and n_split odd the reader
                    // alternates) and read a tile that has not landed.
                    constexpr int kVS = L::kVStages > 0 ? L::kVStages : 1;
                    const int vs_i = v_it % kVS;
                    umma::mbar_wait(&v_full[vs_i], (v_it / kVS) & 1);
                    if ((int)(h_it & 1) != wg) {
                        const unsigned char* vrow = s_vstage + vs_i * L::kStageBytes;
                        float ss0 = 0.f, ss1 = 0.f;
#pragma unroll
                        for (int c8 = 0; c8 < D / 8; ++c8) {
                            const uint4 v = *reinterpret_cast<const uint4*>(
                                vrow + (c8 >> 3) * (kEaTile * 128) + umma::sw128_offset(r, c8 & 7));
                            const float2 f0 = F16Traits<T>::unpack2(v.x), f1 = F16Traits<T>::unpack2(v.y);
                            const float2 f2 = F16Traits<T>::unpack2(v.z), f3 = F16Traits<T>::unpack2(v.w);
                            ss0 = fmaf(f0.x, f0.x, ss0); ss1 = fmaf(f0.y, f0.y, ss1);
                            ss0 = fmaf(f1.x, f1.x, ss0); ss1 = fmaf(f1.y, f1.y, ss1);
                            ss0 = fmaf(f2.x, f2.x, ss0); ss1 = fmaf(f2.y, f2.y, ss1);
                            ss0 = fmaf(f3.x, f3.x, ss0); ss1 = fmaf(f3.y, f3.y, ss1);
                        }
                        __syncwarp();
                        if (lane == 0) umma::mbar_arrive(&v_empty[vs_i]);
                        if (s < S) sc.vnorm[(size_t)row * S_pad + s] = sqrtf(ss0 + ss1);
                    }
                    ++v_it;
                }
#pragma unroll 1
                for (int half = 0; half < kHalves; ++half, ++h_it) {
                    const int buf = h_it & 1;
                    if (buf != wg) continue;
                    if (!waited_k) {
                        EA_T0();
                        umma::mbar_wait(&k_full[stage], (k_it / kStages) & 1);
                        if (warp == 4 && lane == 0) EA_ACC(3);
                        waited_k = true;
                    }
                    {
                        EA_T0();
                        umma::mbar_wait(&t_full[buf], (h_it >> 1) & 1);
                        if (warp == 4 && lane == 0) EA_ACC(4);
                    }
                    EA_T0();
                    umma::fence_after_sync();
                    const uint32_t tbase = tmem + lane_base + buf * kBufCols;
                    uint64_t acc2[HPH][4];  // 4 independent fp32x2 accumulators per head
#pragma unroll
                    for (int q = 0; q < HPH; ++q)
#pragma unroll
                        for (int j = 0; j < 4; ++j) acc2[q][j] = 0ull;
                    // software pipeline over steps (16-column chunk c, head q): the TMEM load of step i+1
                    // is in flight while step i is being reduced
                    constexpr int kC16 = D / 16;
                    uint32_t y[2][16];
#if !(KVP_EA_EXP & 4)
                    umma::tmem_ld16(tbase, y[0]);
#pragma unroll
                    for (int c = 0; c < kC16; ++c) {
                        // k values of this row for columns [16c, 16c+16) as 8 fp32 pairs
                        uint64_t k2[8];
                        {
                            const int c0 = c * 16;
                            const int kpanel = c0 >> 6;
#pragma unroll
                            for (int ch = 0; ch < 2; ++ch) {
#if KVP_EA_EXP & 1
                                const uint4 v = make_uint4(0x3F803F80u + (uint32_t)(kpanel + ch), 0x3F803F80u, 0x3F803F80u,
                                                           0x3F803F80u + (uint32_t)r);
#else
                                const uint4 v = *reinterpret_cast<const uint4*>(
                                    krow + kpanel * (kEaTile * 128) +
                                    umma::sw128_offset(r, ((c0 & 63) >> 3) + ch));
#endif
                                k2[ch * 4] = pack_f32x2(F16Traits<T>::unpack2(v.x));
                                k2[ch * 4 + 1] = pack_f32x2(F16Traits<T>::unpack2(v.y));
                                k2[ch * 4 + 2] = pack_f32x2(F16Traits<T>::unpack2(v.z));
                                k2[ch * 4 + 3] = pack_f32x2(F16Traits<T>::unpack2(v.w));
                            }
                        }
#pragma unroll
                        for (int q = 0; q < HPH; ++q) {
                            constexpr int kSteps = kC16 * HPH;
                            const int step = c * HPH + q;
                            umma::tmem_ld_wait();
                            if (step + 1 < kSteps) {
                                const int cn = (step + 1) / HPH, qn = (step + 1) % HPH;
                                umma::tmem_ld16(tbase + qn * D + cn * 16, y[(step + 1) & 1]);
                            }
                            const uint32_t* yy = y[step & 1];
#pragma unroll
                            for (int j = 0; j < 8; ++j)
                                acc2[q][j & 3] = fma_f32x2(k2[j], pack_u32x2(yy[2 * j], yy[2 * j + 1]), acc2[q][j & 3]);
                        }
                    }
#else
                    (void)y;
                    (void)krow;
#endif
                    float acc[HPH];
#pragma unroll
                    for (int q = 0; q < HPH; ++q) {
                        const float2 a0 = unpack_f32x2(acc2[q][0]), a1 = unpack_f32x2(acc2[q][1]);
                        const float2 a2 = unpack_f32x2(acc2[q][2]), a3 = unpack_f32x2(acc2[q][3]);
                        acc[q] = ((a0.x + a0.y) + (a1.x + a1.y)) + ((a2.x + a2.y) + (a3.x + a3.y));
                    }
                    if (warp == 4 && lane == 0) EA_ACC(5);
                    // accumulator buffer can be overwritten by the next MMA
                    umma::fence_before_sync();
                    __syncwarp();
                    // Release both resources BEFORE the global stores below: mbarrier.arrive has release
                    // semantics and would otherwise wait for those stores to complete (~1k cycles per tile).
                    // A warpgroup drains at most one half per tile, so it is also done with the K tile.
                    if (lane == 0) {
                        umma::mbar_arrive(&t_empty[buf]);
                        umma::mbar_arrive(&k_empty[stage]);
                    }
                    released_k = true;
#pragma unroll
                    for (int q = 0; q < HPH; ++q) {
                        const int g = half * HPH + q;
                        const float lg = acc[q] * inv_2d;
                        if (valid && g < G && g_off + g < g_total) {
                            sc.logits[((size_t)row * g_total + g_off + g) * S_pad + s] = lg;
                            const float m_new = fmaxf(run_m[q], lg);
                            run_z[q] = run_z[q] * __expf(run_m[q] - m_new) + __expf(lg - m_new);
                            run_m[q] = m_new;
                        }
                    }
                }
                __syncwarp();
                if (!released_k) {
                    // This warpgroup had nothing to drain for tile t, but it still owes the stage its release. It must
                    // not give it before the tile has LANDED: an early arrival would be counted in the phase of the
                    // stage's PREVIOUS tile (whose other consumers may still be reading it) and complete that phase
                    // too soon — the producer would then overwrite a tile in use. Seen as a sporadic launch failure
                    // once the idle warpgroup got other work (value norms) and tiles got short (G = 1).
                    umma::mbar_wait(&k_full[stage], (k_it / kStages) & 1);
                    if (lane == 0) umma::mbar_arrive(&k_empty[stage]);
                }
            }
            // ---- warp-level (max, sum-exp) per head slot -> shared ---------------------------------------
#pragma unroll
            for (int q = 0; q < HPH; ++q) {
                float m = run_m[q], z = run_z[q];
#pragma unroll
                for (int off = 16; off >= 1; off >>= 1) {
                    const float m2 = __shfl_xor_sync(0xFFFFFFFFu, m, off);
                    const float z2 = __shfl_xor_sync(0xFFFFFFFFu, z, off);
                    const float mn = fmaxf(m, m2);
                    z = (mn == -INFINITY) ? 0.f : z * __expf(m - mn) + z2 * __expf(m2 - mn);
                    m = mn;
                }
                if (lane == 0) {
                    s_red[((warp - 4) * 2 + q) * 2] = m;
                    s_red[((warp - 4) * 2 + q) * 2 + 1] = z;
                }
            }
        }
        // ---- CTA-level softmax statistics of this (row, part) -> partial[row][g][part] ---------------
        __syncthreads();
        if (tid < G && g_off + tid < g_total) {
            // head g was accumulated in slot q of the warps of: both warpgroups (one half per tile,
            // tiles alternate) or warpgroup g / HPH (two halves per tile)
            const int g = tid, q = g % HPH;
            float m = -INFINITY, z = 0.f;
            for (int w = 0; w < 8; ++w) {
                if (kHalves == 2 && (w >> 2) != g / HPH) continue;
                const float m2 = s_red[(w * 2 + q) * 2], z2 = s_red[(w * 2 + q) * 2 + 1];
                const float mn = fmaxf(m, m2);
                z = (mn == -INFINITY) ? 0.f : z * __expf(m - mn) + z2 * __expf(m2 - mn);
                m = mn;
            }
            sc.partial[((size_t)row * g_total + g_off + g) * n_parts + part] = make_float2(m, z);
        }
    }

#ifdef KVP_EA_PROFILE
    if (blockIdx.x == 0 && tid == 0) g_ea_prof[7] += clock64() - t_entry;
    if (blockIdx.x == 0 && tid == 128) g_ea_prof[8] += clock64() - t_entry;
#endif
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 2) umma::tmem_dealloc(tmem, 512);
}

// ======================================================================================================================
// CTA-PAIR variant (cta_group::2, thread-block cluster of two): the default for even group sizes.
//
// Why: with both operands in shared memory an M128 x N256 x K16 MMA reads (128 + 256) x 32 B = 12 KB per 128 nominal
// cycles; the one-CTA kernel above issues them at ~180 cycles each with or without epilogue work
// (profiles/r02_ea_experiments.txt, r02_ea_roles*.txt) — the operand fetch, not the tensor pipe, sets its pace. A CTA
// pair runs ONE MMA of M = 256 over two consecutive K tiles: each CTA feeds its own 128 rows of A and only ITS half of
// B (one head's covariance instead of two), 8 KB per MMA and SM. The freed shared memory holds the covariance of a
// second head pair, so a K tile is staged once for four heads (two MMA halves per tile) instead of once per head pair.
//
// Work: unit = (row, group of 2*NH heads); item = (unit, pair of consecutive 128-position tiles). The items are cut
// into equal contiguous ranges, one per CTA pair (any number of pairs; a range may cross a unit boundary). CTA `c` of
// the pair owns tile 2*tp + c of item tp: stages it (TMA on its own barrier; a forwarding thread tells the leader), holds
// the covariance of head 2*half + c of each half, reads its 128 x N accumulator rows from its own tensor memory and
// finishes them exactly like the one-CTA kernel. Only the leader issues MMAs; its commits arrive on the barriers of
// both CTAs; the peer's epilogue releases accumulator buffers on the leader's barrier.
template <int D, int NH>
struct Ea2Smem {
    static constexpr int kPanels = D / 64;
    static constexpr int kCovHeadPanel = D * 128;                 // one head's [D rows x 64 columns] panel
    static constexpr int kCovBytes = NH * kPanels * kCovHeadPanel;  // this CTA's share: one head per half
    static constexpr int kStageBytes = kPanels * kEaTile * 128;
    static constexpr int kVStages = 1;
    static constexpr int kAxBytes = kEaTile * 32;
    static constexpr int kBxBytes = NH * D * 32;                  // bias rows of this CTA's heads
    static constexpr int kFixedBytes = kCovBytes + kAxBytes + kBxBytes + 512 + kVStages * kStageBytes;
    static constexpr int kFit = (227 * 1024 - 1024 - kFixedBytes) / kStageBytes;
    static constexpr int kStages = kFit >= 4 ? 4 : kFit;
    static_assert(kStages >= 2, "K ring needs two stages");
    static constexpr int kCovOff = 0;
    static constexpr int kStageOff = kCovBytes;
    static constexpr int kVStageOff = kStageOff + kStages * kStageBytes;
    static constexpr int kAxOff = kVStageOff + kVStages * kStageBytes;
    static constexpr int kBxOff = kAxOff + kAxBytes;
    static constexpr int kBarOff = kBxOff + kBxBytes;
    static constexpr int kTotal = kBarOff + 512;
    static_assert(kTotal + 1024 <= 227 * 1024, "shared memory budget");
};

// contiguous, balanced item ranges: pair p owns [ea2_start(p), ea2_start(p + 1))
__host__ __device__ inline long long ea2_start(int p, long long total, int n_pairs) {
    return ((long long)p * total) / n_pairs;
}
// the pair whose (non-empty) range contains `item`
__host__ __device__ inline int ea2_pair_of(long long item, long long total, int n_pairs) {
    int p = (int)((item * n_pairs) / total);
    if (p >= n_pairs) p = n_pairs - 1;
    while (p + 1 < n_pairs && ea2_start(p + 1, total, n_pairs) <= item) ++p;
    while (p > 0 && ea2_start(p, total, n_pairs) > item) --p;
    return p;
}

// Host-callable view of the partition for the CPU test of the schedule (tests/test_abi_symbols.py): for `pair` of
// `n_pairs` over `n_units` units of `n_tp` items: out4 = {first item, one past the last item}; for `unit`:
// {first pair that touches it, number of pairs that touch it}. Returns -1 on bad arguments.
extern "C" int kvp_debug_ea_pair_partition(int n_units, int n_tp, int n_pairs, int pair, int unit, long long* out4) {
    if (n_units < 1 || n_tp < 1 || n_pairs < 1 || out4 == nullptr) return -1;
    const long long total = (long long)n_units * n_tp;
    if ((long long)n_pairs > total || pair < 0 || pair >= n_pairs || unit < 0 || unit >= n_units) return -1;
    out4[0] = ea2_start(pair, total, n_pairs);
    out4[1] = ea2_start(pair + 1, total, n_pairs);
    const int first = ea2_pair_of((long long)unit * n_tp, total, n_pairs);
    out4[2] = first;
    out4[3] = ea2_pair_of((long long)(unit + 1) * n_tp - 1, total, n_pairs) - first + 1;
    return 0;
}

template <typename T, int D, int NH>
__global__ void __launch_bounds__(KVP_EA_PAIR_BOUNDS, 1)
ea_logits_pair_kernel(const __grid_constant__ CUtensorMap mapK, const __grid_constant__ CUtensorMap mapCov,
                      const __grid_constant__ CUtensorMap mapV, const T* __restrict__ mu, int H, int Hq, int S,
                      int n_sink, int R, int n_tiles128, int n_tp, int n_pairs, int n_parts, EaScratch sc, int S_pad,
                      int g_total, int n_split, int do_vnorm) {
    using L = Ea2Smem<D, NH>;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>(
        (reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);  // same offset in both CTAs of the pair
    unsigned char* s_cov = smem + L::kCovOff;
    unsigned char* s_stage = smem + L::kStageOff;
    unsigned char* s_vstage = smem + L::kVStageOff;
    unsigned char* s_ax = smem + L::kAxOff;
    unsigned char* s_bx = smem + L::kBxOff;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::kBarOff);
    constexpr int kStages = L::kStages;
    uint64_t* k_full = bars;          // [kStages]  per CTA: THIS CTA's tile has landed (its epilogue reads the k rows)
    uint64_t* k_empty = bars + 4;     // [kStages]  per CTA: MMA commit + the warps that read this CTA's k rows
    uint64_t* t_full = bars + 8;      // [2]        per CTA: MMA commit (multicast)
    uint64_t* t_empty = bars + 10;    // [2]        used in the leader only: 4 warps of each CTA drained the buffer
    uint64_t* cov_full = bars + 12;   // [1]        used in the leader only
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 13);
    uint64_t* v_full = bars + 14;     // [1]        per CTA
    uint64_t* v_empty = bars + 16;    // [1]        per CTA
    float* s_red = reinterpret_cast<float*>(bars + 18);  // [8 warps][2 head slots][2]
    uint64_t* k_pair = bars + 40;     // [kStages]  used in the leader only: one arrival per CTA = both tiles have landed

    constexpr int HPH = 2;            // heads per half: head 2*half + c lives in CTA c
    constexpr int kN = HPH * D;       // MMA N (both CTAs together)
    constexpr int kBufCols = 256;
    constexpr int G = 2 * NH;         // heads of a unit
    static_assert(kN <= 256, "two heads must fit one MMA");

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int c = (int)umma::cluster_ctarank();
    const bool leader = c == 0;
    const int P = blockIdx.x >> 1;
#ifdef KVP_EA_PROFILE
    const long long t_entry = clock64();
#endif

    if (tid == 0) {
        umma::prefetch_tmap(&mapK);
        umma::prefetch_tmap(&mapCov);
        if (do_vnorm) umma::prefetch_tmap(&mapV);
        for (int i = 0; i < kStages; ++i) {
            umma::mbar_init(&k_full[i], 1);
            umma::mbar_init(&k_empty[i], 1 + 4 * NH);  // MMA commit + the epilogue warps that read the tile's k rows
            umma::mbar_init(&k_pair[i], 2);            // the forwarding thread of each CTA
        }
        for (int i = 0; i < 2; ++i) {
            umma::mbar_init(&t_full[i], 1);
            umma::mbar_init(&t_empty[i], 8);            // 4 warps of the draining warpgroup in EACH CTA
        }
        umma::mbar_init(&v_full[0], 1);
        umma::mbar_init(&v_empty[0], 4);
        umma::mbar_init(cov_full, 1);
        umma::mbar_fence_init();
    }
    if (warp == 2) umma::tmem_alloc_pair(tmem_slot, 512);
    umma::fence_before_sync();
    __syncthreads();
    umma::cluster_sync();  // both CTAs' barriers exist before any remote arrival / transaction
    umma::fence_after_sync();
    const uint32_t tmem = *tmem_slot;

    const float inv_2d = 1.0f / (2.0f * (float)D);
    const float bias_scale = 2.0f * sqrtf((float)D);
    const long long total = (long long)R * n_split * n_tp;
    const long long i_begin = ea2_start(P, total, n_pairs), i_end = ea2_start(P + 1, total, n_pairs);

    uint32_t k_it = 0, h_it = 0, cov_it = 0, v_it = 0;  // pipeline state of this role, carried across units

    for (long long it = i_begin; it < i_end;) {
        const int unit = (int)(it / n_tp);
        const int tp_begin = (int)(it - (long long)unit * n_tp);
        const int tp_end = (int)min((long long)n_tp, tp_begin + (i_end - it));
        it += tp_end - tp_begin;
        const int row = unit / n_split, hp = unit % n_split, g_off = hp * G;
        const int b = row / H, h = row % H;
        const int hq0 = b * Hq + h * g_total + g_off;  // first head of the unit in [B*Hq]
        const bool v_active = do_vnorm != 0;
        // this CTA's slot among the partial softmax statistics of the unit
        const long long unit_first = (long long)unit * n_tp;
        const int first_pair = ea2_pair_of(unit_first, total, n_pairs);
        const int part = 2 * (P - first_pair) + c;

        // ---- unit prologue: both CTAs are done with the previous unit (every MMA that read either CTA's shared
        // memory has completed: each epilogue waited for the accumulators of all its tiles) ---------------------------
        __syncthreads();
        umma::cluster_sync();
        for (int n = tid; n < NH * D; n += kEaThreads) {
            // bias row n of this CTA: half n / D, head 2 * half + c, element n % D
            const int g = 2 * (n / D) + c;
            const float bias = bias_scale * F16Traits<T>::to_float(
                                                reinterpret_cast<const uint16_t*>(mu)[(size_t)(hq0 + g) * D + (n % D)]);
            const uint16_t hi = F16Traits<T>::from_float(bias);
            const uint16_t lo = F16Traits<T>::from_float(bias - F16Traits<T>::to_float(hi));
            *reinterpret_cast<uint4*>(s_bx + umma::k16_noswizzle_offset(n, 0)) =
                make_uint4((uint32_t)hi | ((uint32_t)lo << 16), 0u, 0u, 0u);
            *reinterpret_cast<uint4*>(s_bx + umma::k16_noswizzle_offset(n, 1)) = make_uint4(0u, 0u, 0u, 0u);
        }
        if (tid < kEaTile) {
            const uint32_t one = (uint32_t)F16Traits<T>::from_float(1.0f);
            *reinterpret_cast<uint4*>(s_ax + umma::k16_noswizzle_offset(tid, 0)) =
                make_uint4(one | (one << 16), 0u, 0u, 0u);
            *reinterpret_cast<uint4*>(s_ax + umma::k16_noswizzle_offset(tid, 1)) = make_uint4(0u, 0u, 0u, 0u);
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic writes -> UMMA reads
        __syncthreads();
        umma::cluster_sync();  // the peer's bias / ones operands are in place before the leader issues

        if (warp == 0) {
            // ===== TMA producer (both CTAs, own tiles; bytes counted on the leader's barriers) =====
            if (lane == 0) {
                if (leader) umma::mbar_arrive_expect_tx(cov_full, 2 * L::kCovBytes);
                for (int kp = 0; kp < L::kPanels; ++kp)
                    for (int half = 0; half < NH; ++half)
                        umma::tma_load_3d_pair(s_cov + (kp * NH + half) * L::kCovHeadPanel, &mapCov, cov_full,
                                               kp * 64, 0, hq0 + 2 * half + c);
                for (int tp = tp_begin; tp < tp_end; ++tp, ++k_it) {
                    const int stage = k_it % kStages;
                    { EA_T0(); umma::mbar_wait(&k_empty[stage], ((k_it / kStages) & 1) ^ 1); EA_ACC(0); }
                    umma::mbar_arrive_expect_tx(&k_full[stage], L::kStageBytes);
                    for (int kp = 0; kp < L::kPanels; ++kp)
                        umma::tma_load_4d(s_stage + stage * L::kStageBytes + kp * (kEaTile * 128), &mapK,
                                          &k_full[stage], kp * 64, (2 * tp + c) * kEaTile, h, b);
                }
            }
        } else if (warp == 2) {
            // ===== forwarder (both CTAs): "my K tile has landed" -> the leader's pair barrier. Each CTA's tile completes
            // on its OWN barrier, so its epilogue (generic-proxy reads of the k rows) observes the completion itself; the
            // MMA issuer waits for one arrival per CTA (release at cluster scope -> its acquire) =====
            if (lane == 0) {
                for (int tp = tp_begin; tp < tp_end; ++tp, ++k_it) {
                    const int stage = k_it % kStages;
                    umma::mbar_wait(&k_full[stage], (k_it / kStages) & 1);
                    umma::mbar_arrive_leader(&k_pair[stage]);
                }
            }
        } else if (warp == 3) {
            // ===== V producer (own tile, CTA-local barriers) =====
            if (lane == 0 && v_active) {
                for (int tp = tp_begin; tp < tp_end; ++tp) {
                    if ((tp % n_split) != hp) continue;   // the units of a row take turns
                    umma::mbar_wait(&v_empty[0], (v_it & 1) ^ 1);
                    umma::mbar_arrive_expect_tx(&v_full[0], L::kStageBytes);
                    for (int kp = 0; kp < L::kPanels; ++kp)
                        umma::tma_load_4d(s_vstage + kp * (kEaTile * 128), &mapV, &v_full[0], kp * 64,
                                          (2 * tp + c) * kEaTile, h, b);
                    ++v_it;
                }
            }
        } else if (warp == 1) {
            // ===== MMA issuer (leader only) =====
            if (lane == 0 && leader) {
                const uint32_t idesc = umma::instr_desc_f16(2 * kEaTile, kN, F16Traits<T>::kMmaFormat);
                umma::mbar_wait(cov_full, cov_it & 1);
                for (int tp = tp_begin; tp < tp_end; ++tp, ++k_it) {
                    const int stage = k_it % kStages;
                    { EA_T0(); umma::mbar_wait(&k_pair[stage], (k_it / kStages) & 1); EA_ACC(1); }
                    umma::fence_after_sync();
                    const uint32_t a_base = umma::smem_u32(s_stage + stage * L::kStageBytes);
#pragma unroll 1
                    for (int half = 0; half < NH; ++half, ++h_it) {
                        const int buf = h_it & 1;
                        { EA_T0(); umma::mbar_wait(&t_empty[buf], ((h_it >> 1) & 1) ^ 1); EA_ACC(2); }
                        umma::fence_after_sync();
#pragma unroll
                        for (int k = 0; k < D / 16; ++k) {
                            const int kp = k >> 2, kk = k & 3;
                            const uint64_t da = umma::smem_desc_sw128(a_base + kp * (kEaTile * 128) + kk * 32);
                            const uint64_t db = umma::smem_desc_sw128(
                                umma::smem_u32(s_cov + (kp * NH + half) * L::kCovHeadPanel) + kk * 32);
                            umma::mma_f16_ss_pair(tmem + buf * kBufCols, da, db, idesc, k > 0);
                        }
#if !(KVP_EA_EXP2 & 16)
                        umma::mma_f16_ss_pair(tmem + buf * kBufCols,
                                              umma::smem_desc_k16_noswizzle(umma::smem_u32(s_ax)),
                                              umma::smem_desc_k16_noswizzle(umma::smem_u32(s_bx) + (half * D / 8) * 256),
                                              idesc, 1);
#endif
                        umma::mma_commit_pair(&t_full[buf]);
                    }
                    umma::mma_commit_pair(&k_empty[stage]);
                }
            }
            ++cov_it;
        } else if (warp >= 4 && warp < 12) {
            // ===== epilogue (both CTAs): warpgroup wg drains TMEM buffer wg; thread = key row of THIS CTA's tile =====
            const int wg = (warp - 4) >> 2;
            const int ew = warp & 3;
            const int r = ew * 32 + lane;
            const uint32_t lane_base = (uint32_t)(ew * 32) << 16;
            float run_m[HPH], run_z[HPH];
#pragma unroll
            for (int q = 0; q < HPH; ++q) {
                run_m[q] = -INFINITY;
                run_z[q] = 0.f;
            }
            for (int tp = tp_begin; tp < tp_end; ++tp, ++k_it) {
                const int stage = k_it % kStages;
                const unsigned char* krow = s_stage + stage * L::kStageBytes;
                const int s = (2 * tp + c) * kEaTile + r;
                const bool valid = (s >= n_sink) && (s < S);
                if (v_active && (tp % n_split) == hp) {
                    // value norms of this CTA's tile: both warpgroups observe every V phase (one V stage), one of them
                    // reads — the warpgroup without an accumulator for this tile (NH = 1), or alternately (NH = 2)
                    { EA_T0(); umma::mbar_wait(&v_full[0], v_it & 1); if (warp == 4 && lane == 0) EA_ACC(6); }
                    const bool reader = (NH == 1) ? ((int)(h_it & 1) != wg) : ((int)(v_it & 1) == wg);
                    if (reader) {
                        EA_T0();
                        float ss0 = 0.f, ss1 = 0.f;
#pragma unroll
                        for (int c8 = 0; c8 < D / 8; ++c8) {
                            const uint4 v = *reinterpret_cast<const uint4*>(
                                s_vstage + (c8 >> 3) * (kEaTile * 128) + umma::sw128_offset(r, c8 & 7));
                            const float2 f0 = F16Traits<T>::unpack2(v.x), f1 = F16Traits<T>::unpack2(v.y);
                            const float2 f2 = F16Traits<T>::unpack2(v.z), f3 = F16Traits<T>::unpack2(v.w);
                            ss0 = fmaf(f0.x, f0.x, ss0); ss1 = fmaf(f0.y, f0.y, ss1);
                            ss0 = fmaf(f1.x, f1.x, ss0); ss1 = fmaf(f1.y, f1.y, ss1);
                            ss0 = fmaf(f2.x, f2.x, ss0); ss1 = fmaf(f2.y, f2.y, ss1);
                            ss0 = fmaf(f3.x, f3.x, ss0); ss1 = fmaf(f3.y, f3.y, ss1);
                        }
                        __syncwarp();
                        if (lane == 0) umma::mbar_arrive(&v_empty[0]);
                        if (s < S) sc.vnorm[(size_t)row * S_pad + s] = sqrtf(ss0 + ss1);
                        if (warp == 4 && lane == 0) EA_ACC(10);
                    }
                    ++v_it;
                }
#pragma unroll 1
                for (int half = 0; half < NH; ++half, ++h_it) {
                    const int buf = h_it & 1;
                    if (buf != wg) continue;
                    umma::mbar_wait(&k_full[stage], (k_it / kStages) & 1);  // this CTA's k rows are visible to these threads
                    {
                        EA_T0();
                        umma::mbar_wait(&t_full[buf], (h_it >> 1) & 1);
                        if (warp == 4 && lane == 0) EA_ACC(4);
                    }
                    EA_T0();
                    umma::fence_after_sync();
                    const uint32_t tbase = tmem + lane_base + buf * kBufCols;
                    uint64_t acc2[HPH][4];
#pragma unroll
                    for (int q = 0; q < HPH; ++q)
#pragma unroll
                        for (int j = 0; j < 4; ++j) acc2[q][j] = 0ull;
#if !(KVP_EA_EXP2 & 4)
                    constexpr int kC16 = D / 16;
                    uint32_t y[2][16];
                    umma::tmem_ld16(tbase, y[0]);
#pragma unroll
                    for (int cc = 0; cc < kC16; ++cc) {
                        uint64_t k2[8];
                        {
                            const int c0 = cc * 16;
                            const int kpanel = c0 >> 6;
#pragma unroll
                            for (int ch = 0; ch < 2; ++ch) {
                                const uint4 v = *reinterpret_cast<const uint4*>(
                                    krow + kpanel * (kEaTile * 128) + umma::sw128_offset(r, ((c0 & 63) >> 3) + ch));
                                k2[ch * 4] = pack_f32x2(F16Traits<T>::unpack2(v.x));
                                k2[ch * 4 + 1] = pack_f32x2(F16Traits<T>::unpack2(v.y));
                                k2[ch * 4 + 2] = pack_f32x2(F16Traits<T>::unpack2(v.z));
                                k2[ch * 4 + 3] = pack_f32x2(F16Traits<T>::unpack2(v.w));
                            }
                        }
#pragma unroll
                        for (int q = 0; q < HPH; ++q) {
                            constexpr int kSteps = kC16 * HPH;
                            const int step = cc * HPH + q;
                            umma::tmem_ld_wait();
                            if (step + 1 < kSteps) {
                                const int cn = (step + 1) / HPH, qn = (step + 1) % HPH;
                                if (!((KVP_EA_EXP2 & 1) && qn == 1)) umma::tmem_ld16(tbase + qn * D + cn * 16, y[(step + 1) & 1]);
                            }
                            const uint32_t* yy = y[step & 1];
#pragma unroll
                            for (int j = 0; j < 8; ++j)
                                acc2[q][j & 3] = fma_f32x2(k2[j], pack_u32x2(yy[2 * j], yy[2 * j + 1]), acc2[q][j & 3]);
                        }
                    }
#else
                    (void)krow;
#endif
                    float acc[HPH];
#pragma unroll
                    for (int q = 0; q < HPH; ++q) {
                        const float2 a0 = unpack_f32x2(acc2[q][0]), a1 = unpack_f32x2(acc2[q][1]);
                        const float2 a2 = unpack_f32x2(acc2[q][2]), a3 = unpack_f32x2(acc2[q][3]);
                        acc[q] = ((a0.x + a0.y) + (a1.x + a1.y)) + ((a2.x + a2.y) + (a3.x + a3.y));
                    }
                    if (warp == 4 && lane == 0) EA_ACC(5);
                    umma::fence_before_sync();
                    __syncwarp();
                    // release before the global stores (an arrive has release semantics): the accumulator buffer on the
                    // LEADER's barrier, this CTA's K stage on its own
                    if (lane == 0) {
                        umma::mbar_arrive_leader(&t_empty[buf]);
                        umma::mbar_arrive(&k_empty[stage]);
                    }
                    EA_T1();
#pragma unroll
                    for (int q = 0; q < HPH; ++q) {
                        const int g = half * HPH + q;
                        const float lg = acc[q] * inv_2d;
                        if (valid) {
#if !(KVP_EA_EXP2 & 2)
                            sc.logits[((size_t)row * g_total + g_off + g) * S_pad + s] = lg;
#endif
#if !(KVP_EA_EXP2 & 8)
                            const float m_new = fmaxf(run_m[q], lg);
                            run_z[q] = run_z[q] * __expf(run_m[q] - m_new) + __expf(lg - m_new);
                            run_m[q] = m_new;
#else
                            run_m[q] = fmaxf(run_m[q], lg);
#endif
                        }
                    }
                    if (warp == 4 && lane == 0) EA_ACC1(11);
                }
                __syncwarp();
            }
#ifdef KVP_EA_PROFILE
            if (blockIdx.x == 0 && warp == 4 && lane == 0) g_ea_prof[12] += clock64() - t_entry;
            if (blockIdx.x == 0 && warp == 8 && lane == 0) g_ea_prof[13] += clock64() - t_entry;
#endif
            // ---- warp-level (max, sum-exp) per head slot -> shared ---------------------------------------------------
#pragma unroll
            for (int q = 0; q < HPH; ++q) {
                float m = run_m[q], z = run_z[q];
#pragma unroll
                for (int off = 16; off >= 1; off >>= 1) {
                    const float m2 = __shfl_xor_sync(0xFFFFFFFFu, m, off);
                    const float z2 = __shfl_xor_sync(0xFFFFFFFFu, z, off);
                    const float mn = fmaxf(m, m2);
                    z = (mn == -INFINITY) ? 0.f : z * __expf(m - mn) + z2 * __expf(m2 - mn);
                    m = mn;
                }
                if (lane == 0) {
                    s_red[((warp - 4) * 2 + q) * 2] = m;
                    s_red[((warp - 4) * 2 + q) * 2 + 1] = z;
                }
            }
        }
        // ---- CTA-level softmax statistics of this CTA's tiles -> partial[row][g][part] -------------------------------
        __syncthreads();
        if (tid < G) {
            // head g sat in slot g % 2 of: the warps of warpgroup g / 2 (NH = 2: one half per warpgroup) or of both
            // warpgroups (NH = 1: tiles alternate)
            const int g = tid, q = g % HPH;
            float m = -INFINITY, z = 0.f;
            for (int w = 0; w < 8; ++w) {
                if (NH == 2 && (w >> 2) != g / HPH) continue;
                const float m2 = s_red[(w * 2 + q) * 2], z2 = s_red[(w * 2 + q) * 2 + 1];
                const float mn = fmaxf(m, m2);
                z = (mn == -INFINITY) ? 0.f : z * __expf(m - mn) + z2 * __expf(m2 - mn);
                m = mn;
            }
            sc.partial[((size_t)row * g_total + g_off + g) * n_parts + part] = make_float2(m, z);
        }
        if (part == 0 && tid >= 32 && tid < 32 + G) {
            // the unit's first CTA neutralises the slots no CTA of this unit owns (units take a varying number of pairs)
            const long long unit_last = unit_first + n_tp - 1;
            const int used = 2 * (ea2_pair_of(unit_last, total, n_pairs) - first_pair + 1);
            for (int p = used; p < n_parts; ++p)
                sc.partial[((size_t)row * g_total + g_off + (tid - 32)) * n_parts + p] = make_float2(-INFINITY, 0.f);
        }
    }

#ifdef KVP_EA_PROFILE
    if (blockIdx.x == 0 && tid == 0) g_ea_prof[7] += clock64() - t_entry;
    if (blockIdx.x == 0 && tid == 32) g_ea_prof[14] = i_end - i_begin;
#endif
    umma::fence_before_sync();
    __syncthreads();
    umma::cluster_sync();  // the peer may still be reading its accumulators / this CTA's barriers
    if (warp == 2) umma::tmem_dealloc_pair(tmem, 512);
}

// ---- covariance-free logits: mu.k / sqrt(d) with plain streaming loads (use_covariance=False) -------
template <typename T, int LPR>
__global__ void __launch_bounds__(256)
ea_mu_logits_kernel(const T* __restrict__ K, Strides3 ks, const T* __restrict__ mu, int H, int Hq, int G,
                    int S, int D, int n_sink, int n_parts, EaScratch sc, int S_pad) {
    __shared__ float s_mu[8 * 256];
    __shared__ float s_red[8][8][2];
    const int chunk = blockIdx.x, row = blockIdx.y, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int b = row / H, h = row % H;
    const int hq0 = b * Hq + h * G;
    const float scale = 1.0f / sqrtf((float)D);
    for (int i = tid; i < G * D; i += 256)
        s_mu[i] = F16Traits<T>::to_float(reinterpret_cast<const uint16_t*>(mu)[(size_t)hq0 * D + i]);
    __syncthreads();
    constexpr int RPW = 32 / LPR;
    constexpr int TOK_PER_WARP = kScoreChunkGeneric / 8;
    constexpr int ITERS = TOK_PER_WARP / RPW;
    constexpr int U = (ITERS < 4) ? ITERS : 4;
    const int sub = lane % LPR, rsel = lane / LPR;
    const int nvec = D >> 3;
    const T* base = K + (int64_t)b * ks.b + (int64_t)h * ks.h + (int64_t)sub * 8;
    const int s_warp = chunk * kScoreChunkGeneric + warp * TOK_PER_WARP;
    float run_m[8], run_z[8];
#pragma unroll
    for (int g = 0; g < 8; ++g) {
        run_m[g] = -INFINITY;
        run_z[g] = 0.f;
    }
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
            const int s = s_warp + (it + u) * RPW + rsel;
            const uint32_t w4[4] = {(uint32_t)v[u].x, (uint32_t)v[u].y, (uint32_t)v[u].z, (uint32_t)v[u].w};
            float kf[8];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float2 f = F16Traits<T>::unpack2(w4[j]);
                kf[2 * j] = f.x;
                kf[2 * j + 1] = f.y;
            }
#pragma unroll
            for (int g = 0; g < 8; ++g) {
                if (g < G) {
                    float dot = 0.f;
                    if (sub < nvec) {
#pragma unroll
                        for (int j = 0; j < 8; ++j) dot = fmaf(kf[j], s_mu[g * D + sub * 8 + j], dot);
                    }
#pragma unroll
                    for (int off = LPR / 2; off >= 1; off >>= 1) dot += __shfl_xor_sync(0xFFFFFFFFu, dot, off);
                    const float lg = dot * scale;
                    if (sub == 0 && s >= n_sink && s < S) {
                        sc.logits[((size_t)row * G + g) * S_pad + s] = lg;
                        const float mn = fmaxf(run_m[g], lg);
                        run_z[g] = run_z[g] * __expf(run_m[g] - mn) + __expf(lg - mn);
                        run_m[g] = mn;
                    }
                }
            }
        }
    }
    // merge the per-lane statistics (only lanes with sub == 0 hold any)
#pragma unroll
    for (int g = 0; g < 8; ++g) {
        if (g < G) {
            float m = run_m[g], z = run_z[g];
#pragma unroll
            for (int off = 16; off >= 1; off >>= 1) {
                const float m2 = __shfl_xor_sync(0xFFFFFFFFu, m, off);
                const float z2 = __shfl_xor_sync(0xFFFFFFFFu, z, off);
                const float mn = fmaxf(m, m2);
                z = (mn == -INFINITY) ? 0.f : z * __expf(m - mn) + z2 * __expf(m2 - mn);
                m = mn;
            }
            if (lane == 0) {
                s_red[warp][g][0] = m;
                s_red[warp][g][1] = z;
            }
        }
    }
    __syncthreads();
    if (tid < G) {
        float m = -INFINITY, z = 0.f;
        for (int w = 0; w < 8; ++w) {
            const float m2 = s_red[w][tid][0], z2 = s_red[w][tid][1];
            const float mn = fmaxf(m, m2);
            z = (mn == -INFINITY) ? 0.f : z * __expf(m - mn) + z2 * __expf(m2 - mn);
            m = mn;
        }
        sc.partial[((size_t)row * G + tid) * n_parts + chunk] = make_float2(m, z);
    }
}

// ---- ||v_s||_2 for every position: plain streaming kernel, launched on a side stream so that it shares
// the SMs with the tensor-bound logits kernel (which leaves ~70 % of the HBM bandwidth idle) -----------
template <typename T, int LPR>
__global__ void __launch_bounds__(kTileThreads, 4)
ea_vnorm_kernel(const T* __restrict__ V, Strides3 vs, int H, int S, int D, float* __restrict__ vnorm,
                int S_pad) {
    __shared__ float s_norm[kTile];
    const int tile = blockIdx.x, row = blockIdx.y, tid = threadIdx.x;
    row_norm_chunk<T, LPR>(V, vs, row / H, row % H, tile, S, D, s_norm);
    __syncthreads();
    const int s = tile * kTile + tid;
    if (s < S) vnorm[(size_t)row * S_pad + s] = s_norm[tid];
}

// ---- finalize: softmax normalisation, group mean, * ||v||, ONE rounding, keys + histogram -----------
// One CTA = kEaFinalPos consecutive positions of one row, 4 per thread: the G logits and the value norm arrive as
// 128-bit loads (all independent, issued before anything else), 1024 CTAs cover a 128k x 8-head cache in one wave.
constexpr int kEaFinalKpt = 4;
constexpr int kEaFinalPos = kTileThreads * kEaFinalKpt;
template <typename T>
__global__ void __launch_bounds__(kTileThreads)
ea_finalize_kernel(int G, int S, int n_sink, int use_vnorm, float eps, int n_parts, EaScratch sc,
                   Workspace ws, uint16_t* __restrict__ scores_out) {
    constexpr int KPT = kEaFinalKpt;
    __shared__ uint16_t skeys[kEaFinalPos];
    __shared__ uint16_t sscores[kEaFinalPos];
    __shared__ uint32_t shist[256];
    __shared__ float s_m[8], s_iz[8];
    __shared__ float s_max[8];
    const int chunk = blockIdx.x, row = blockIdx.y, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    shist[tid] = 0;
    pdl_launch_dependents();  // the selection pass behind this one may start to take residency
    const int s0 = chunk * kEaFinalPos + tid * KPT;
    const bool in_pad = s0 < ws.S_pad;  // the padded scratch rows are readable up to S_pad (a multiple of 256)
    // 1. independent loads first: this thread's logits / norms and (warps < G) the per-CTA softmax partials
    float4 lg[8];
#pragma unroll
    for (int g = 0; g < 8; ++g)
        lg[g] = (g < G && in_pad)
                    ? __ldcg(reinterpret_cast<const float4*>(&sc.logits[((size_t)row * G + g) * ws.S_pad + s0]))
                    : make_float4(0.f, 0.f, 0.f, 0.f);
    const float4 vn4 = (use_vnorm && in_pad)
                           ? __ldcg(reinterpret_cast<const float4*>(&sc.vnorm[(size_t)row * ws.S_pad + s0]))
                           : make_float4(1.f, 1.f, 1.f, 1.f);
    float pm = -INFINITY, pz = 0.f;
    if (warp < G) {
        for (int p = lane; p < n_parts; p += 32) {
            const float2 q = sc.partial[((size_t)row * G + warp) * n_parts + p];
            const float mn = fmaxf(pm, q.x);
            pz = (mn == -INFINITY) ? 0.f : pz * __expf(pm - mn) + q.y * __expf(q.x - mn);
            pm = mn;
        }
        // 2. exact softmax normalisers of the G heads
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) {
            const float m2 = __shfl_xor_sync(0xFFFFFFFFu, pm, off);
            const float z2 = __shfl_xor_sync(0xFFFFFFFFu, pz, off);
            const float mn = fmaxf(pm, m2);
            pz = (mn == -INFINITY) ? 0.f : pz * __expf(pm - mn) + z2 * __expf(m2 - mn);
            pm = mn;
        }
        if (lane == 0) {
            s_m[warp] = pm;
            s_iz[warp] = 1.0f / pz;
        }
    }
    __syncthreads();
    float fmax_valid = -INFINITY;
    const float vn[4] = {vn4.x, vn4.y, vn4.z, vn4.w};
#pragma unroll
    for (int i = 0; i < KPT; ++i) {
        const int s = s0 + i;
        uint16_t bits = 0, key = 0;
        if (s < S) {
            if (s < n_sink) {
                key = kForcedKey;
            } else {
                float p = 0.f;
#pragma unroll
                for (int g = 0; g < 8; ++g) {
                    if (g < G) {
                        const float l = (i == 0) ? lg[g].x : (i == 1) ? lg[g].y : (i == 2) ? lg[g].z : lg[g].w;
                        p += __expf(l - s_m[g]) * s_iz[g];
                    }
                }
                p *= (1.0f / (float)G);
                const float score = use_vnorm ? (p + eps) * vn[i] : p;
                bits = F16Traits<T>::from_float(score);
                key = ordered_key16(bits, F16Traits<T>::kInfBits);
                fmax_valid = fmaxf(fmax_valid, F16Traits<T>::to_float(bits));
            }
        }
        skeys[tid * KPT + i] = key;
        sscores[tid * KPT + i] = bits;
    }
    __syncthreads();
    flush_chunk_keys<KPT, false>(skeys, sscores, shist, row, chunk * kEaFinalPos, S, ws, scores_out);
    // max over valid scores of the whole tensor (for the reference's max+1 sentinel)
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1)
        fmax_valid = fmaxf(fmax_valid, __shfl_xor_sync(0xFFFFFFFFu, fmax_valid, off));
    if (lane == 0) s_max[warp] = fmax_valid;
    __syncthreads();
    if (tid == 0) {
        float m = s_max[0];
        for (int w = 1; w < 8; ++w) m = fmaxf(m, s_max[w]);
        if (m > -INFINITY) {
            // order-preserving float -> uint so atomicMax works (counters are zero-initialised)
            const uint32_t u = __float_as_uint(m);
            const uint32_t ord = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
            atomicMax(&ws.counters[kCounterMaxSlot(ws.R)], ord);
        }
    }
    flush_row_hist(shist, row, ws);
}

// scores_out[..., lo:hi] = round(max_valid_score + 1) — the value the reference pads with
// (expected_attention_press.py:163, snapkv_press.py:103: `scores.max().item() + 1`).
template <typename T>
__global__ void fill_sentinel_kernel(uint16_t* __restrict__ scores_out, int R, int S, int lo, int hi,
                                     const uint32_t* __restrict__ max_slot) {
    const uint32_t ord = *max_slot;
    pdl_launch_dependents();  // the selection pass behind this one may start to take residency
    const uint32_t u = (ord & 0x80000000u) ? (ord & 0x7FFFFFFFu) : ~ord;
    const float sentinel = __uint_as_float(u) + 1.0f;
    const uint16_t bits = F16Traits<T>::from_float(sentinel);
    const int width = hi - lo;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < R * width; i += gridDim.x * blockDim.x)
        scores_out[(size_t)(i / width) * S + lo + (i % width)] = bits;
}

cudaError_t launch_fill_sentinel(int dtype, void* scores_out, int R, int S, int lo, int hi,
                                 const Workspace& ws, cudaStream_t st) {
    if (hi <= lo) return cudaSuccess;
    const uint32_t* slot = ws.counters + kCounterMaxSlot(R);
    int blocks = (R * (hi - lo) + 255) / 256;
    if (blocks > 1024) blocks = 1024;
    if (dtype == KVP_BF16)
        fill_sentinel_kernel<__nv_bfloat16><<<blocks, 256, 0, st>>>(static_cast<uint16_t*>(scores_out), R, S, lo, hi, slot);
    else
        fill_sentinel_kernel<__half><<<blocks, 256, 0, st>>>(static_cast<uint16_t*>(scores_out), R, S, lo, hi, slot);
    return cudaPeekAtLastError();
}

#if KVP_EA_TRI
// cov [heads][D][D] -> T[n][c] = cov[n][c] + cov[c][n] (c < n), cov[n][n] (c == n), 0 (c > n); one rounding.
template <typename T>
__global__ void __launch_bounds__(256)
ea_cov_tri_kernel(const uint16_t* __restrict__ cov, uint16_t* __restrict__ tri, int D) {
    // one thread per element (it sits on the critical path in front of the logits kernel: two dependent-free loads,
    // one store, thousands of CTAs instead of a per-head loop)
    const size_t base = (size_t)blockIdx.y * D * D;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= D * D) return;
    const int n = i / D, cidx = i - n * D;
    const uint16_t a = cov[base + i];
    const uint16_t b = cov[base + (size_t)cidx * D + n];
    uint16_t out = 0;
    if (cidx == n) out = a;
    else if (cidx < n) out = F16Traits<T>::from_float(F16Traits<T>::to_float(a) + F16Traits<T>::to_float(b));
    tri[base + i] = out;
}
#endif

// ---- host launcher -----------------------------------------------------------------------------------
template <typename T, int D, int G>
static cudaError_t launch_ea_logits_t(const Dims& d, const void* K, const void* V_or_null, const void* mu,
                                      const void* cov, int n_sink, const Workspace& ws, const EaScratch& sc,
                                      int* n_parts_out, cudaStream_t st) {
    using L = EaSmem<D, G>;
    const int sm_count = device_sm_count();
    const int n_tiles128 = (d.S + kEaTile - 1) / kEaTile;
    // work units = (row, group of G heads); the CTAs of a unit split the row's tiles
    const int g_total = d.Hq / d.H;
    const int n_split = (g_total + G - 1) / G;
    const int n_units = d.R * n_split;
    int ctas_per_row = sm_count / n_units;  // CTAs per unit
    if (ctas_per_row < 1) ctas_per_row = 1;
    if (ctas_per_row > n_tiles128) ctas_per_row = n_tiles128;
    if (ctas_per_row > kEaMaxParts) ctas_per_row = kEaMaxParts;
    int n_groups = sm_count / ctas_per_row;
    if (n_groups > n_units) n_groups = n_units;
    const int grid = n_groups * ctas_per_row;
    *n_parts_out = ctas_per_row;

    CUtensorMap mapK, mapCov, mapV;
    const bool in_kernel_v = L::kVStages > 0 && V_or_null != nullptr;
    {  // V tiles are staged exactly like K tiles (same box, same swizzle), from V's own strides
        const void* base = in_kernel_v ? V_or_null : K;
        const Strides3& xs = in_kernel_v ? d.vs : d.ks;
        const uint64_t row_b = (uint64_t)xs.s * 2;
        const uint64_t h_b = d.H > 1 ? (uint64_t)xs.h * 2 : row_b * (uint64_t)d.S;
        const uint64_t b_b = d.B > 1 ? (uint64_t)xs.b * 2 : h_b * (uint64_t)d.H;
        const uint64_t dims[4] = {(uint64_t)D, (uint64_t)d.S, (uint64_t)d.H, (uint64_t)d.B};
        const uint64_t str[4] = {0, row_b, h_b, b_b};
        const uint32_t box[4] = {64, (uint32_t)kEaTile, 1, 1};
        cudaError_t e = make_tmap_16bit(&mapV, base, 4, dims, str, box);
        if (e != cudaSuccess) return e;
    }
    {
        const uint64_t row_b = (uint64_t)d.ks.s * 2;
        const uint64_t h_b = d.H > 1 ? (uint64_t)d.ks.h * 2 : row_b * (uint64_t)d.S;
        const uint64_t b_b = d.B > 1 ? (uint64_t)d.ks.b * 2 : h_b * (uint64_t)d.H;
        const uint64_t dims[4] = {(uint64_t)D, (uint64_t)d.S, (uint64_t)d.H, (uint64_t)d.B};
        const uint64_t str[4] = {0, row_b, h_b, b_b};
        const uint32_t box[4] = {64, (uint32_t)kEaTile, 1, 1};
        cudaError_t e = make_tmap_16bit(&mapK, K, 4, dims, str, box);
        if (e != cudaSuccess) return e;
    }
    {
        const uint64_t dims[3] = {(uint64_t)D, (uint64_t)D, (uint64_t)d.B * d.Hq};
        const uint64_t str[3] = {0, (uint64_t)D * 2, (uint64_t)D * D * 2};
        const uint32_t box[3] = {64, (uint32_t)D, 1};
        const void* cov_src = cov;
#if KVP_EA_TRI
        ea_cov_tri_kernel<T><<<dim3((D * D + 255) / 256, d.B * d.Hq), 256, 0, st>>>(
            static_cast<const uint16_t*>(cov), sc.cov_tri, D);
        cudaError_t pe = cudaPeekAtLastError();
        if (pe != cudaSuccess) return pe;
        cov_src = sc.cov_tri;
#endif
        cudaError_t e = make_tmap_16bit(&mapCov, cov_src, 3, dims, str, box);
        if (e != cudaSuccess) return e;
    }
    const int smem = L::kTotal + 1024;
    auto kern = ea_logits_kernel<T, D, G>;
    static PerDeviceOnce smem_set;  // one per <T, D, G> instantiation of this launcher
    cudaError_t e = ensure_dynamic_smem(kern, smem, smem_set);
    if (e != cudaSuccess) return e;
    kern<<<grid, kEaThreads, smem, st>>>(mapK, mapCov, mapV, static_cast<const T*>(mu), d.H, d.Hq, d.S, n_sink, d.R,
                                         n_tiles128, ctas_per_row, ctas_per_row, sc, ws.S_pad, g_total, n_split,
                                         in_kernel_v ? 1 : 0);
    return cudaPeekAtLastError();
}

// ---- host launcher of the CTA-pair kernel ---------------------------------------------------------------------------
template <typename T, int D, int NH>
static cudaError_t launch_ea_logits_pair_t(const Dims& d, const void* K, const void* V_or_null, const void* mu,
                                           const void* cov, int n_sink, const Workspace& ws, const EaScratch& sc,
                                           int* n_parts_out, cudaStream_t st) {
    using L = Ea2Smem<D, NH>;
    const int n_tiles128 = (d.S + kEaTile - 1) / kEaTile;
    const int n_tp = (n_tiles128 + 1) / 2;
    const int g_total = d.Hq / d.H;
    const int n_split = g_total / (2 * NH);
    const long long total = (long long)d.R * n_split * n_tp;

    const int smem = L::kTotal + 1024;
    auto kern = ea_logits_pair_kernel<T, D, NH>;
    static PerDeviceOnce smem_set;  // one per <T, D, NH> instantiation of this launcher
    cudaError_t e = ensure_dynamic_smem(kern, smem, smem_set);
    if (e != cudaSuccess) return e;

    cudaLaunchConfig_t cfg = {};
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cfg.blockDim = dim3(kEaThreads, 1, 1);
    cfg.dynamicSmemBytes = (size_t)smem;
    cfg.stream = st;
    // co-resident CTA pairs (a GPC with an odd SM count leaves one SM unpaired): queried once per device
    static PerDeviceInt max_pairs;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) dev = 0;
    if (max_pairs.v[dev] == 0) {
        cfg.gridDim = dim3(2 * (device_sm_count() / 2), 1, 1);
        int n = 0;
        if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess || n < 1) {
            (void)cudaGetLastError();
            n = device_sm_count() / 2;
        }
        max_pairs.v[dev] = n;
    }
    int n_pairs = max_pairs.v[dev];
    if (n_pairs > kEaMaxParts / 2) n_pairs = kEaMaxParts / 2;
    if ((long long)n_pairs > total) n_pairs = (int)total;  // every pair owns at least one item
    // slots of the per-CTA softmax partials of a unit: two per pair that touches it
    int max_count = 1;
    for (int u = 0; u < d.R * n_split; ++u) {
        const int first = ea2_pair_of((long long)u * n_tp, total, n_pairs);
        const int last = ea2_pair_of((long long)(u + 1) * n_tp - 1, total, n_pairs);
        if (last - first + 1 > max_count) max_count = last - first + 1;
    }
    const int n_parts = 2 * max_count;
    *n_parts_out = n_parts;

    CUtensorMap mapK, mapCov, mapV;
    const bool in_kernel_v = V_or_null != nullptr;
    {  // V tiles are staged exactly like K tiles (same box, same swizzle), from V's own strides
        const void* base = in_kernel_v ? V_or_null : K;
        const Strides3& xs = in_kernel_v ? d.vs : d.ks;
        const uint64_t row_b = (uint64_t)xs.s * 2;
        const uint64_t h_b = d.H > 1 ? (uint64_t)xs.h * 2 : row_b * (uint64_t)d.S;
        const uint64_t b_b = d.B > 1 ? (uint64_t)xs.b * 2 : h_b * (uint64_t)d.H;
        const uint64_t dims[4] = {(uint64_t)D, (uint64_t)d.S, (uint64_t)d.H, (uint64_t)d.B};
        const uint64_t str[4] = {0, row_b, h_b, b_b};
        const uint32_t box[4] = {64, (uint32_t)kEaTile, 1, 1};
        if ((e = make_tmap_16bit(&mapV, base, 4, dims, str, box)) != cudaSuccess) return e;
    }
    {
        const uint64_t row_b = (uint64_t)d.ks.s * 2;
        const uint64_t h_b = d.H > 1 ? (uint64_t)d.ks.h * 2 : row_b * (uint64_t)d.S;
        const uint64_t b_b = d.B > 1 ? (uint64_t)d.ks.b * 2 : h_b * (uint64_t)d.H;
        const uint64_t dims[4] = {(uint64_t)D, (uint64_t)d.S, (uint64_t)d.H, (uint64_t)d.B};
        const uint64_t str[4] = {0, row_b, h_b, b_b};
        const uint32_t box[4] = {64, (uint32_t)kEaTile, 1, 1};
        if ((e = make_tmap_16bit(&mapK, K, 4, dims, str, box)) != cudaSuccess) return e;
    }
    {
        const uint64_t dims[3] = {(uint64_t)D, (uint64_t)D, (uint64_t)d.B * d.Hq};
        const uint64_t str[3] = {0, (uint64_t)D * 2, (uint64_t)D * D * 2};
        const uint32_t box[3] = {64, (uint32_t)D, 1};
        if ((e = make_tmap_16bit(&mapCov, cov, 3, dims, str, box)) != cudaSuccess) return e;
    }
    cfg.gridDim = dim3(2 * n_pairs, 1, 1);
    return cudaLaunchKernelEx(&cfg, kern, mapK, mapCov, mapV, static_cast<const T*>(mu), d.H, d.Hq, d.S, n_sink, d.R,
                              n_tiles128, n_tp, n_pairs, n_parts, sc, (int)ws.S_pad, g_total, n_split,
                              in_kernel_v ? 1 : 0);
}

// Side stream + fork/join events for the concurrent V-norm kernel: created once per device, never
// modified afterwards (the only process-wide state of the library besides cached device properties).
struct EaSideStream {
    cudaStream_t stream = nullptr;
    cudaEvent_t fork = nullptr, join = nullptr;
    bool ok = false;
};
static std::mutex g_ea_enqueue_mu;  // serialises fork..join enqueues that share the side stream / events
static EaSideStream* ea_side_stream() {
    static EaSideStream per_device[64];
    static std::mutex mu;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    std::lock_guard<std::mutex> lock(mu);
    EaSideStream& s = per_device[dev];
    if (!s.ok) {
        if (cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
        if (cudaEventCreateWithFlags(&s.fork, cudaEventDisableTiming) != cudaSuccess) return nullptr;
        if (cudaEventCreateWithFlags(&s.join, cudaEventDisableTiming) != cudaSuccess) return nullptr;
        s.ok = true;
    }
    return &s;
}

template <typename T>
static cudaError_t launch_ea_vnorm_t(const Dims& d, const void* V, const Workspace& ws, const EaScratch& sc,
                                     cudaStream_t st) {
    dim3 grid(ws.n_tiles, d.R);
    const int nvec = d.D / 8;
#define KVP_EA_VN(LPR)                                                                               \
    ea_vnorm_kernel<T, LPR><<<grid, kTileThreads, 0, st>>>(static_cast<const T*>(V), d.vs, d.H, d.S, d.D, \
                                                           sc.vnorm, ws.S_pad)
    if (nvec <= 4) KVP_EA_VN(4);
    else if (nvec <= 8) KVP_EA_VN(8);
    else if (nvec <= 16) KVP_EA_VN(16);
    else KVP_EA_VN(32);
#undef KVP_EA_VN
    return cudaPeekAtLastError();
}

template <typename T>
static cudaError_t launch_ea_t(const Dims& d, int dtype, const void* K, const void* V, const void* mu,
                               const void* cov, float eps, int n_sink, int use_vnorm,
                               const Workspace& ws, void* scores_out, cudaStream_t st) {
    const int G = d.Hq / d.H;
    if (G > 8) return cudaErrorNotSupported;
    const int nvec = d.D / 8;
    const EaScratch sc = carve_ea(d, ws);
    int n_parts = 0;
    cudaError_t e = cudaSuccess;
    // Value norms: with covariance and at most two resident heads per CTA (the default layout) the logits kernel stages
    // the V tiles itself and an idle epilogue warpgroup takes the norms — no second kernel. Otherwise (covariance-free
    // scan, or the four-head A/B layout) ea_vnorm_kernel runs on an internal side stream next to the score kernel:
    // fork here, join before the finalize kernel.
#ifndef KVP_EA_RESIDENT_HEADS
#define KVP_EA_RESIDENT_HEADS 2  // A/B knob: 4 = round-1 layout (all four heads of a Llama-3.1-8B group in one CTA)
#endif
    const bool tc_path = cov != nullptr && (d.D == 128 || d.D == 64);
    // CTA-pair kernel (cta_group::2) for even group sizes; KVP_EA_PAIR=0 keeps the one-CTA kernel (A/B, odd groups)
    static const bool pair_knob = [] {
        const char* v = getenv("KVP_EA_PAIR");
        return !(v && *v) || atoi(v) != 0;
    }();
    const bool pair_path = pair_knob && tc_path && G % 2 == 0;
    const bool in_kernel_v = use_vnorm && tc_path &&
                             (pair_path || (KVP_EA_V_STAGES > 0 && (G <= 2 || KVP_EA_RESIDENT_HEADS == 2)));
    const void* v_for_logits = in_kernel_v ? V : nullptr;
    EaSideStream* side = (use_vnorm && !in_kernel_v) ? ea_side_stream() : nullptr;
    // host threads enqueueing on different streams of one device share the side stream and its two
    // events: hold the lock for the (host-only, microseconds) fork..join enqueue sequence
    std::unique_lock<std::mutex> enqueue_lock(g_ea_enqueue_mu, std::defer_lock);
    if (side != nullptr) enqueue_lock.lock();
    if (side != nullptr) {
        if ((e = cudaEventRecord(side->fork, st)) != cudaSuccess) return e;
        if ((e = cudaStreamWaitEvent(side->stream, side->fork, 0)) != cudaSuccess) return e;
    }
    if (cov != nullptr) {
        // tensor-core path: head_dim 64 or 128; the G query heads of a kv head are cut into groups of two (one for
        // G = 1), each group is a work unit with its own covariance resident in shared memory; an odd G pads its last
        // group with a head that has no bias and stores nothing (Llama-3.2-3B: 3, Qwen2-7B: 7, Llama-3.1-70B: 8).
        if (d.D != 128 && d.D != 64) return cudaErrorNotSupported;
        const bool d128 = d.D == 128;
        if (pair_path) {
            if (G % 4 == 0)
                e = d128 ? launch_ea_logits_pair_t<T, 128, 2>(d, K, v_for_logits, mu, cov, n_sink, ws, sc, &n_parts, st)
                         : launch_ea_logits_pair_t<T, 64, 2>(d, K, v_for_logits, mu, cov, n_sink, ws, sc, &n_parts, st);
            else
                e = d128 ? launch_ea_logits_pair_t<T, 128, 1>(d, K, v_for_logits, mu, cov, n_sink, ws, sc, &n_parts, st)
                         : launch_ea_logits_pair_t<T, 64, 1>(d, K, v_for_logits, mu, cov, n_sink, ws, sc, &n_parts, st);
        } else if (G == 1)
            e = d128 ? launch_ea_logits_t<T, 128, 1>(d, K, v_for_logits, mu, cov, n_sink, ws, sc, &n_parts, st)
                     : launch_ea_logits_t<T, 64, 1>(d, K, v_for_logits, mu, cov, n_sink, ws, sc, &n_parts, st);
        else if (G == 2 || KVP_EA_RESIDENT_HEADS == 2)
            // two resident heads per CTA, ceil(G / 2) CTAs share a row's K tiles
            e = d128 ? launch_ea_logits_t<T, 128, 2>(d, K, v_for_logits, mu, cov, n_sink, ws, sc, &n_parts, st)
                     : launch_ea_logits_t<T, 64, 2>(d, K, v_for_logits, mu, cov, n_sink, ws, sc, &n_parts, st);
        else
            e = d128 ? launch_ea_logits_t<T, 128, 4>(d, K, nullptr, mu, cov, n_sink, ws, sc, &n_parts, st)
                     : launch_ea_logits_t<T, 64, 4>(d, K, nullptr, mu, cov, n_sink, ws, sc, &n_parts, st);
    } else {
        n_parts = (d.S + kScoreChunkGeneric - 1) / kScoreChunkGeneric;
        dim3 grid(n_parts, d.R);
#define KVP_EA_MU(LPR)                                                                                   \
    ea_mu_logits_kernel<T, LPR><<<grid, 256, 0, st>>>(static_cast<const T*>(K), d.ks,                     \
                                                      static_cast<const T*>(mu), d.H, d.Hq, G, d.S, d.D, \
                                                      n_sink, n_parts, sc, ws.S_pad)
        if (nvec <= 4) KVP_EA_MU(4);
        else if (nvec <= 8) KVP_EA_MU(8);
        else if (nvec <= 16) KVP_EA_MU(16);
        else KVP_EA_MU(32);
#undef KVP_EA_MU
        e = cudaPeekAtLastError();
    }
    if (e != cudaSuccess) return e;
    if (use_vnorm && !in_kernel_v) {
        // launched AFTER the logits kernel so that its CTAs fill the resources the logits CTAs leave free
        cudaStream_t vst = side != nullptr ? side->stream : st;
        if ((e = launch_ea_vnorm_t<T>(d, V, ws, sc, vst)) != cudaSuccess) return e;
        if (side != nullptr) {  // join
            if ((e = cudaEventRecord(side->join, side->stream)) != cudaSuccess) return e;
            if ((e = cudaStreamWaitEvent(st, side->join, 0)) != cudaSuccess) return e;
        }
    }
    dim3 grid2((d.S + kEaFinalPos - 1) / kEaFinalPos, d.R);
    ea_finalize_kernel<T><<<grid2, kTileThreads, 0, st>>>(G, d.S, n_sink, use_vnorm, eps, n_parts, sc, ws,
                                                          static_cast<uint16_t*>(scores_out));
    e = cudaPeekAtLastError();
    if (e != cudaSuccess) return e;
    if (scores_out != nullptr) e = launch_fill_sentinel(dtype, scores_out, d.R, d.S, 0, n_sink, ws, st);
    return e;
}

#ifdef KVP_EA_PROFILE
extern "C" void kvp_debug_ea_profile(long long* out, int reset) {
    if (reset) {
        long long z[32] = {0};
        cudaMemcpyToSymbol(g_ea_prof, z, sizeof(z));
    } else {
        cudaMemcpyFromSymbol(out, g_ea_prof, 32 * sizeof(long long));
    }
}
#endif

cudaError_t launch_ea_score(const Dims& d, int dtype, const void* K, const void* V, const void* mu,
                            const void* cov, float eps, int n_sink, int use_vnorm,
                            const Workspace& ws, void* scores_out, bool want_keys,
                            cudaStream_t st) {
    (void)want_keys;  // keys + histogram are always produced; the select stage is skipped by the caller
    if (dtype == KVP_BF16)
        return launch_ea_t<__nv_bfloat16>(d, dtype, K, V, mu, cov, eps, n_sink, use_vnorm, ws, scores_out, st);
    return launch_ea_t<__half>(d, dtype, K, V, mu, cov, eps, n_sink, use_vnorm, ws, scores_out, st);
}

}  // namespace kvp
