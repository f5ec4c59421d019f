// Shared device/host helpers for libnpi (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/npi.h"

namespace npi {

constexpr int H = 128;          // hidden width of every SAGEConv / TopKPooling in Net_1 (src/classes.py:48-53)
constexpr int WARP = 32;

void set_error(const char* fmt, ...);
int grid_for(int ctas_per_sm);          // #SMs * ctas_per_sm (148 * k on B200)
int num_sms();
// out[K,128] = sum_g part[g][...] (+ row0 partials on row 0), fixed order (gemm.cu)
int launch_gemm_tn_reduce(const float* part, int G, int ktiles, int K, const float* row0, int R, float* out, cudaStream_t st);

// out[i] = sum of in[0..i), *total (nullable) = sum of all n; tile_sums: >= ceil(n / 4096) ints of scratch (sort.cu)
int launch_excl_scan_i32(const int32_t* in, int64_t n, int32_t* out, int32_t* total, int32_t* tile_sums, cudaStream_t st);

// Key bits of a radix sort by group id: ceil(log2 num_groups), at least 1 (topk.cu, grouprank.cu).
inline int group_bits(int32_t num_groups) {
    int b = 1;
    while (((int64_t)1 << b) < num_groups) ++b;
    return b;
}
// gptr[g] = first of the n group-sorted keys >= g, for g = 0 .. num_groups (one launch); *status = OR of the ntiles
// per-tile status bits 0..2 (topk.cu)
int launch_group_bounds(const uint32_t* keys, int64_t n, int32_t num_groups, const int32_t* tile_status, int ntiles,
                        int32_t* gptr, int32_t* status, cudaStream_t st);

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is a PER-DEVICE attribute: "configured once" flags are
// kept per device (a process that drives a second GPU configures the kernels there too).
struct OncePerDevice {
    bool done[64] = {};
    bool need() {
        int d = 0;
        if (cudaGetDevice(&d) != cudaSuccess) return true;
        d &= 63;
        if (done[d]) return false;
        done[d] = true;
        return true;
    }
};
struct MaxPerDevice {          // for kernels whose opt-in size grows with the problem
    size_t cur[64] = {};
    bool need(size_t v) {
        int d = 0;
        if (cudaGetDevice(&d) != cudaSuccess) return true;
        d &= 63;
        if (v <= cur[d]) return false;
        cur[d] = v;
        return true;
    }
};

#define NPI_CHECK_CUDA(expr)                                                              \
    do {                                                                                  \
        cudaError_t _e = (expr);                                                          \
        if (_e != cudaSuccess) {                                                          \
            npi::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
            return NPI_ERR_CUDA;                                                          \
        }                                                                                 \
    } while (0)

#define NPI_CHECK_LAUNCH()  NPI_CHECK_CUDA(cudaGetLastError())

#define NPI_REQUIRE(cond, ...)                                                            \
    do {                                                                                  \
        if (!(cond)) {                                                                    \
            npi::set_error(__VA_ARGS__);                                                  \
            return NPI_ERR_INVALID;                                                       \
        }                                                                                 \
    } while (0)

// ---------------------------------------------------------------- programmatic dependent launch
// The training step is a chain of ~30 dependent kernels of 5-40 us each; between two of them the GPU drains, the next
// grid is launched, its CTAs are scheduled and run their prologue -- a few microseconds every time, a fifth of the
// step in total.  Kernels of the chain are launched with the programmatic-stream-serialization attribute
// (launch_dep) and open with pdl_trigger() + pdl_wait(): the NEXT kernel of the stream may be scheduled as soon as
// every CTA of this one has started, and each kernel blocks in pdl_wait() until its predecessor has completed and
// flushed -- memory ordering is that of plain stream order, only launch latency, CTA scheduling and the
// parameter-only prologues overlap the predecessor's tail.  Only data written by kernels of EARLIER steps (weights) or
// by kernels that finished before the predecessor started may be touched before pdl_wait().  A kernel launched without
// the attribute (NPI_PDL=0, or by <<< >>>) executes both instructions as no-ops.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
#ifndef NPI_PDL_EARLY
#define NPI_PDL_EARLY 0
#endif
// Early trigger (at the top of a kernel) lets the successor's CTAs become resident -- and sit in pdl_wait() holding
// registers and shared memory -- for the whole run of this kernel: measured, that starves the auxiliary and extraction
// streams and costs 60 us per step (gpurun_out/r3d).  Default: no explicit trigger, the dependents are released when the
// CTAs of this kernel exit; what remains overlapped is the launch itself.
__device__ __forceinline__ void pdl_trigger() {
#if NPI_PDL_EARLY
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
#endif
}
bool pdl_enabled();      // api.cu: environment NPI_PDL != "0"

template <typename... KArgs, typename... Args>
inline cudaError_t launch_dep(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// Data-dependent size read on the device, clamped to the host bound the buffers were sized for: a
// count that exceeds the caller's capacity must never turn into an out-of-bounds access.
__device__ __forceinline__ int dev_size(const int32_t* n_dev, int n_host) {
    if (!n_dev) return n_host;
    const int n = *n_dev;
    return n < n_host ? n : n_host;
}

// ---------------------------------------------------------------- warp / block primitives
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ int warp_sum_i(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ int warp_incl_scan_i(int v, int lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int t = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += t;
    }
    return v;
}

// Exclusive block scan of one int per thread.  `sh` holds >= NT/32 + 1 ints.  Every thread
// of the block must call it.  Returns the exclusive prefix; *total receives the block sum.
template <int NT>
__device__ __forceinline__ int block_excl_scan(int v, int* sh, int* total) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int inc = warp_incl_scan_i(v, lane);
    __syncthreads();                       // protect sh from the previous call's readers
    if (lane == 31) sh[w] = inc;
    __syncthreads();
    if (w == 0) {
        int t = (lane < NT / 32) ? sh[lane] : 0;
        int ti = warp_incl_scan_i(t, lane);
        if (lane < NT / 32) sh[lane] = ti - t;
        if (lane == NT / 32 - 1) sh[NT / 32] = ti;
    }
    __syncthreads();
    *total = sh[NT / 32];
    return inc - v + sh[w];
}

// Orderable key of a score for the ranking entry points (rank.cu, topk.cu, grouprank.cu): ascending key = descending
// score, -0.0 and +0.0 one key, +-inf ordinary scores.
__device__ __forceinline__ uint32_t rank_key(float s) {
    uint32_t u = __float_as_uint(s);
    if (s == 0.0f) u = 0u;                                   // -0.0 and +0.0 are one threshold
    u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);          // order-preserving map to uint32
    return ~u;                                               // ascending key = descending score
}

// Workspace carver of the ranking entry points: consecutive regions, each rounded up to 256 bytes.  A null base carves
// nothing and only counts the bytes (the *_workspace_bytes query); `off` is the total.
struct WsCarver {
    char* base;
    int64_t off = 0;
    template <typename T>
    T* take(int64_t bytes) {
        char* p = base ? base + off : nullptr;
        off += (bytes + 255) / 256 * 256;
        return (T*)p;
    }
};

// Block sum of one value per thread in a fixed order (warp butterflies, then the warp partials in warp order):
// bit-reproducible for fp64.  `sh` holds NT / 32 values; every thread of the NT-thread block must call it.
template <int NT, typename T>
__device__ __forceinline__ T block_sum(T v, T* sh) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    __syncthreads();                                         // protect sh from the previous call's readers
    if (lane == 0) sh[w] = v;
    __syncthreads();
    T s = sh[0];
    for (int k = 1; k < NT / 32; ++k) s += sh[k];
    return s;
}

// True in the last CTA of the grid to arrive here, false in every other one (block-uniform).  Every thread calls it
// after its CTA has written its per-CTA partials; the last CTA then reads all partials with __ldcg.  The ticket counts
// the arrivals and is reset by the last CTA, so it is zero again for the next launch.
__device__ __forceinline__ bool last_cta(unsigned int* ticket) {
    __threadfence();
    __syncthreads();
    if (!__syncthreads_or(threadIdx.x == 0 && atomicAdd(ticket, 1u) == gridDim.x - 1u)) return false;
    __threadfence();
    if (threadIdx.x == 0) *ticket = 0u;
    return true;
}

// OR of a status word over the block, bits 0 .. NBITS - 1.  Every thread of the block must call it.
template <int NBITS>
__device__ __forceinline__ int block_or_bits(int st) {
    int r = 0;
#pragma unroll
    for (int b = 0; b < NBITS; ++b) r |= __syncthreads_or(st & (1 << b)) ? 1 << b : 0;
    return r;
}

// npi_sort_pairs_u32 of (keys_a, vals_a) by `bits` key bits with (keys_b, vals_b) as the other buffer pair.  On return
// (keys, vals) is the pair holding the sorted result and (free_keys, free_vals) the other one.
struct SortedPairs {
    uint32_t* keys; int32_t* vals;
    uint32_t* free_keys; int32_t* free_vals;
};
inline int sort_pairs(uint32_t* keys_a, int32_t* vals_a, uint32_t* keys_b, int32_t* vals_b, int64_t n, int bits, void* ws,
                      int64_t ws_bytes, cudaStream_t st, SortedPairs* out) {
    const int rc = npi_sort_pairs_u32(keys_a, vals_a, keys_b, vals_b, n, bits, ws, ws_bytes, st);
    if (npi_sort_passes(bits) & 1) *out = {keys_b, vals_b, keys_a, vals_a};
    else *out = {keys_a, vals_a, keys_b, vals_b};
    return rc;
}

__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ float4 add4(float4 a, float4 b) { return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }
__device__ __forceinline__ float4 mul4(float4 a, float s) { return make_float4(a.x * s, a.y * s, a.z * s, a.w * s); }
__device__ __forceinline__ float dot4(float4 a, float4 b) { return a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w; }

// ---------------------------------------------------------------- Philox4x32-10 (dropout)
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
        uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
        ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
        key.x += W0; key.y += W1;
    }
    return ctr;
}

}  // namespace npi
