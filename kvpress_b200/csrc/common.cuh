// common.cuh — shared device helpers and the internal (C++) launcher interface.
// sm_100a only. No torch types anywhere in csrc/.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/kvpress_b200.h"

namespace kvp {

// ---- tiling of the sequence axis for the select / compact stages --------------------------
constexpr int kTile = 256;          // positions per select/compact tile (one per thread)
constexpr int kTileThreads = 256;
constexpr int kSfxStride = 264;     // u16 per tile record: sfx[0..256], gt_hi at [257], padding
constexpr uint16_t kForcedKey = 0xFFFFu;  // ordered key of a forced-keep position
constexpr int kFinalizeTiles = 1;          // 256-position tiles per CTA of the finalize kernels (1: >5 waves at 128k, no tail)
constexpr int kScoreChunkGeneric = 256;   // positions per CTA of the plain streaming score kernels
// counters[] layout: [0] ticket (fused Knorm kernel), [1, 1+R) refine done, [1+R, 1+2R) row ready, then the slot below:
// order-preserving uint image of the largest valid score (for the reference's max+1 sentinel);
// [2+2R, 2+3R) score items done per row (fused Knorm kernel)
__host__ __device__ constexpr int kCounterMaxSlot(int R) { return 1 + 2 * R; }
// [3R + 8]: error flag. A bounded spin-wait that expires (a lost work item: library bug, or a device that
// cannot co-schedule the persistent grid) raises it instead of trapping the whole CUDA context; every CTA
// polls it with its ticket and drains. The host reads it back with kvp_workspace_check().
__host__ __device__ constexpr int kCounterErrSlot(int R) { return 3 * R + 8; }
constexpr uint32_t kSpinLimit = 1u << 22;  // x 64 ns nanosleep ~ 0.3 s

struct Strides3 {
    int64_t b, h, s;
};

// Device view of the scratch area (carved by carve_workspace in api.cu).
struct Workspace {
    uint16_t* keys;      // [R][S_pad] ordered 16-bit keys of the scores
    uint32_t* hist_hi;   // [R][256]   histogram of key >> 8
    uint32_t* hist_lo;   // [R][256]   histogram of key & 255 among keys with hi == threshold bin
    uint16_t* tile_sfx;  // [R][n_tiles][kSfxStride]
    uint32_t* counters;  // [0] work-queue ticket, [1 + row] refine items done, [1 + R + row] row ready;
                         // zeroed together with the histograms
    uint2* row_meta;     // [R] {threshold key T, ties to take}
    uint2* tile_prefix;  // [R][n_tiles] {kept (> T) + 1, tied (== T) + 1} positions in the tiles before;
                         // zero = row not scanned yet
    int R;
    void* scorer;        // scorer-specific scratch (SnapKV / ExpectedAttention)
    size_t scorer_bytes;
    int S_pad;
    int n_tiles;
};

struct Dims {
    int B, H, Hq, S, D, n_kept;
    int R;  // B * H rows
    Strides3 ks, vs;
};

// ---- 16-bit float -> ordered unsigned key (same for bf16 and fp16: sign-magnitude) --------
// inf_bits = 0x7F80 for bf16, 0x7C00 for fp16: anything above it (either sign) is a NaN, which
// torch.topk ranks above every number -> largest key.
__host__ __device__ __forceinline__ uint16_t ordered_key16(uint16_t bits, uint16_t inf_bits) {
    if ((bits & 0x7FFFu) > inf_bits) return 0xFFFFu;  // NaN
    if (bits == 0x8000u) bits = 0;                    // -0 == +0 (torch.topk compares by value)
    return (bits & 0x8000u) ? (uint16_t)(~bits) : (uint16_t)(bits | 0x8000u);
}
__host__ __device__ __forceinline__ uint16_t key16_to_bits(uint16_t key) {
    return (key & 0x8000u) ? (uint16_t)(key & 0x7FFFu) : (uint16_t)(~key);
}

template <typename T>
struct F16Traits;
template <>
struct F16Traits<__nv_bfloat16> {
    static __device__ __forceinline__ float2 unpack2(uint32_t w) {
        return make_float2(__uint_as_float(w << 16), __uint_as_float(w & 0xFFFF0000u));
    }
    static __device__ __forceinline__ uint16_t from_float(float f) {
        return __bfloat16_as_ushort(__float2bfloat16_rn(f));
    }
    static __device__ __forceinline__ float to_float(uint16_t b) {
        return __uint_as_float(((uint32_t)b) << 16);
    }
    static constexpr uint16_t kInfBits = 0x7F80u;
    static constexpr int kMmaFormat = 1;  // tcgen05 kind::f16 operand format: BF16
};
template <>
struct F16Traits<__half> {
    static __device__ __forceinline__ float2 unpack2(uint32_t w) {
        __half2 h = *reinterpret_cast<__half2*>(&w);
        return __half22float2(h);
    }
    static __device__ __forceinline__ uint16_t from_float(float f) {
        return __half_as_ushort(__float2half_rn(f));
    }
    static __device__ __forceinline__ float to_float(uint16_t b) {
        return __half2float(__ushort_as_half(b));
    }
    static constexpr uint16_t kInfBits = 0x7C00u;
    static constexpr int kMmaFormat = 0;  // F16
};

// ---- cache-hinted 128-bit global accesses ---------------------------------------------------
// sm_100a only accepts the bare .L2::evict_* qualifiers on 256-bit accesses; 128-bit accesses take
// an explicit createpolicy handle through .L2::cache_hint.
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ int4 ldg_hint(const void* p, uint64_t pol) {
    int4 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.s32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ int4 ldg_plain(const void* p) {
    int4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ void stg_hint(void* p, const int4& v, uint64_t pol) {
    asm volatile("st.global.L1::no_allocate.L2::cache_hint.v4.s32 [%0], {%1,%2,%3,%4}, %5;" ::"l"(p),
                 "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w), "l"(pol)
                 : "memory");
}

// ---- programmatic dependent launch (PDL) ------------------------------------------------------------------
// The selection pass and the compaction grid are launched with cudaLaunchAttributeProgrammaticStreamSerialization:
// their CTAs may become resident while the LAST wave of the kernel in front of them is still draining (that kernel
// calls pdl_launch_dependents() at its start) and park in pdl_wait() until that grid has completed and flushed, so
// the launch latency and the ramp of each grid are off the critical path. Both are no-ops for a plain launch.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                     Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

// ---- 256-bin suffix search, executed by ONE full warp ----------------------------------------
// Finds the largest bin b with sum_{i>=b} hist[i] >= need (need >= 1) and returns
// above = sum_{i>b} hist[i]. hist lives in shared memory. All 32 lanes get the result.
__device__ __forceinline__ void warp_suffix_find(const uint32_t* hist, uint32_t need, int lane,
                                                 int& bin, uint32_t& above) {
    const int top = 255 - 8 * lane;  // this lane owns bins top, top-1, ..., top-7
    uint32_t h[8];
    uint32_t lane_sum = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        h[i] = hist[top - i];
        lane_sum += h[i];
    }
    uint32_t incl = lane_sum;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, off);
        if (lane >= off) incl += t;
    }
    const unsigned crossed = __ballot_sync(0xFFFFFFFFu, incl >= need);
    int my_bin = 0;
    uint32_t my_above = 0;
    const int first = crossed ? (__ffs(crossed) - 1) : 31;
    if (lane == first) {
        uint32_t run = incl - lane_sum;
        my_bin = top - 7;
        my_above = incl - h[7];
        bool found = false;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            if (!found && run + h[i] >= need) {
                my_bin = top - i;
                my_above = run;
                found = true;
            }
            run += h[i];
        }
    }
    bin = __shfl_sync(0xFFFFFFFFu, my_bin, first);
    above = __shfl_sync(0xFFFFFFFFu, my_above, first);
}

// Adds a CTA's shared-memory histogram to the row histogram (call after a __syncthreads()).
__device__ __forceinline__ void flush_row_hist(const uint32_t* shist, int row, const Workspace& ws) {
    const int tid = threadIdx.x;
    if (tid < 256) {
        const uint32_t c = shist[tid];
        if (c) atomicAdd(&ws.hist_hi[(size_t)row * 256 + tid], c);
    }
}

// Common tail of every score kernel: KPT keys (and optionally scores) per thread staged in shared
// memory for a chunk of KPT*blockDim positions starting at s_begin -> coalesced global writes + row
// histogram of (key >> 8). Shared-memory atomics are warp-aggregated with match.any so heavily tied
// scores (bf16 norms take ~100 distinct values) do not serialise on one address.
// Call with all threads of a 256-thread CTA after a __syncthreads(); shist must be zeroed.
template <int KPT, bool kFlushHist = true>
__device__ __forceinline__ void flush_chunk_keys(const uint16_t* skeys, const uint16_t* sscores,
                                                 uint32_t* shist, int row, int s_begin, int S,
                                                 const Workspace& ws, uint16_t* scores_out) {
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int s0 = s_begin + tid * KPT;
    uint16_t k[KPT];
#pragma unroll
    for (int i = 0; i < KPT; ++i) k[i] = ((s0 + i) < S) ? skeys[tid * KPT + i] : (uint16_t)0;
    // the keys buffer is padded to a multiple of kTile per row: unconditional vector store
    uint16_t* kdst = ws.keys + (size_t)row * ws.S_pad + s0;
    if (KPT == 4) {
        // a KPT*256-position chunk may reach past the row's padding (S_pad is a multiple of 256 only)
        if (s0 < ws.S_pad) {
            uint2 pk;
            pk.x = (uint32_t)k[0] | ((uint32_t)k[1 % KPT] << 16);
            pk.y = (uint32_t)k[2 % KPT] | ((uint32_t)k[3 % KPT] << 16);
            *reinterpret_cast<uint2*>(kdst) = pk;
        }
    } else {
#pragma unroll
        for (int i = 0; i < KPT; ++i) kdst[i] = k[i];
    }
    if (scores_out != nullptr) {
        uint16_t* dst = scores_out + (size_t)row * S + s0;
#pragma unroll
        for (int i = 0; i < KPT; ++i)
            if (s0 + i < S) dst[i] = sscores[tid * KPT + i];
    }
#pragma unroll
    for (int i = 0; i < KPT; ++i) {
        const unsigned bin = ((s0 + i) < S) ? (unsigned)(k[i] >> 8) : 256u;
        const unsigned peers = __match_any_sync(0xFFFFFFFFu, bin);
        if (bin < 256u && lane == (__ffs(peers) - 1)) atomicAdd(&shist[bin], __popc(peers));
    }
    if (kFlushHist) {
        __syncthreads();
        flush_row_hist(shist, row, ws);
    }
}

// ---- host: per-device launch properties, resolved once per (device, kernel) and cached (tmap.cu) ----
// Nothing below is re-queried on the launch path: the C-ABI calls are host-latency sensitive
// (DecodingPress compactions, per-layer prefill hooks).
int device_sm_count();                         // SM count of the CURRENT device
constexpr int kMaxDevices = 64;
// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) once per (kernel, device). `done` is the CALLER's function-local
// static (one per launcher instantiation): kernels that differ only in non-type template arguments share one function
// POINTER TYPE, so a cache keyed on the template type of this helper would be shared between them.
struct PerDeviceOnce {
    unsigned long long mask = 0;  // bit per device; a lost race only repeats the idempotent call
};
template <typename Kern>
static inline cudaError_t ensure_dynamic_smem(Kern kern, int bytes, PerDeviceOnce& done) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev >= 0 && dev < kMaxDevices && ((done.mask >> dev) & 1ull)) return cudaSuccess;
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e == cudaSuccess && dev >= 0 && dev < kMaxDevices) done.mask |= 1ull << dev;
    return e;
}
// resident CTAs per SM of a kernel (occupancy query) once per (kernel, device); `cache` as above
struct PerDeviceInt {
    int v[kMaxDevices] = {0};
};
template <typename Kern>
static inline int cached_ctas_per_sm(Kern kern, int threads, PerDeviceInt& cache, int dyn_smem = 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) dev = 0;
    if (cache.v[dev] == 0) {
        int per_sm = 0;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, dyn_smem);
        cache.v[dev] = per_sm > 0 ? per_sm : 1;
    }
    return cache.v[dev];
}

// ---- launchers implemented in the .cu files (host, C++ linkage) -------------------------------
cudaError_t launch_knorm_score(const Dims& d, int dtype, const void* K, const Workspace& ws,
                               void* scores_out, bool want_keys, cudaStream_t st);
cudaError_t launch_knorm_fused(const Dims& d, int dtype, const void* K, const void* V, void* K_out,
                               void* V_out, int32_t* idx_out, void* scores_out, const Workspace& ws,
                               cudaStream_t st);
bool knorm_cluster_applicable(const Dims& d);
cudaError_t launch_knorm_cluster(const Dims& d, int dtype, const void* K, const void* V, void* K_out, void* V_out,
                                 int32_t* idx_out, void* scores_out, cudaStream_t st);
cudaError_t launch_keys_from_scores(const Dims& d, int dtype, const void* scores, int64_t sb, int64_t sh,
                                    const Workspace& ws, cudaStream_t st);
cudaError_t launch_select_compact(const Dims& d, const void* K, const void* V, void* K_out,
                                  void* V_out, int32_t* idx_out, const Workspace& ws,
                                  cudaStream_t st);
cudaError_t launch_select_compact_rerotate(const Dims& d, int dtype, const void* K, const void* V,
                                           void* K_out, void* V_out, int32_t* idx_out,
                                           const Workspace& ws, const float* inv_freq, cudaStream_t st);
cudaError_t launch_streaming_score(const Dims& d, int dtype, int n_sink, void* scores_out,
                                   cudaStream_t st);
cudaError_t launch_streaming_compress(const Dims& d, int n_sink, const void* K, const void* V,
                                      void* K_out, void* V_out, int32_t* idx_out,
                                      cudaStream_t st);

size_t snapkv_scratch_bytes(const Dims& d, int window);
cudaError_t launch_snapkv_score(const Dims& d, int dtype, const void* K, const void* q_window,
                                int window, int kernel_size, const Workspace& ws,
                                void* scores_out, bool want_keys, cudaStream_t st);
size_t keydiff_scratch_bytes(const Dims& d);
cudaError_t launch_keydiff_score(const Dims& d, int dtype, const void* K, const Workspace& ws,
                                 void* scores_out, bool want_keys, cudaStream_t st);
size_t ea_scratch_bytes(const Dims& d);
cudaError_t launch_fill_sentinel(int dtype, void* scores_out, int R, int S, int lo, int hi,
                                 const Workspace& ws, cudaStream_t st);
cudaError_t launch_ea_score(const Dims& d, int dtype, const void* K, const void* V, const void* mu,
                            const void* cov, float eps, int n_sink, int use_vnorm,
                            const Workspace& ws, void* scores_out, bool want_keys,
                            cudaStream_t st);

}  // namespace kvp
