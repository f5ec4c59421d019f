// Dense projections of the SAGEConv layers on the 5th-generation tensor cores (tcgen05, sm_100a).
//
//   C[M,128] = A[M,K] . B        K in {32,64,96,128};  B is [K,128] (transB = 0) or [128,K] (transB = 1)
//
// Same contract as gemm_nn (gemm.cu; reference src/classes.py:62,66,70 `@ weight` of PyG SAGEConv and
// its input gradient), computed with tcgen05.mma kind::tf32 and fp32 accumulators in TMEM.  fp32
// accuracy is kept by the error-compensated split  x = hi + lo  (hi = x rounded to the 11 significant
// bits of tf32, lo = x - hi rounded likewise):  A.B ~= lo_A.hi_B + hi_A.lo_B + hi_A.hi_B  -- three MMAs per
// K step, all accumulated in TMEM (the dropped lo.lo term is < 2^-22 relative).
//
// Layout: operands live in shared memory as K-major SWIZZLE_128B tiles ([128 rows][32 floats], row
// = 128 B, 16-byte chunk c of row r stored at chunk c ^ (r & 7), 8-row groups 1024 B apart); the
// whole B operand (hi and lo, K/32 tiles each) stays resident for the lifetime of the CTA, the A
// operand streams through in 32-column slices.  One CTA per SM, persistent over 128-row tiles.
#include <cuda.h>

#include "common.cuh"

namespace npi {
namespace tc {

constexpr uint32_t TILE_BYTES = 128 * 128;      // [128][32] fp32
constexpr uint32_t TMEM_COLS = 128;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// UMMA shared-memory descriptor, K-major, SWIZZLE_128B (cute::UMMA::SmemDescriptor bit layout)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);      // [0,14)  start address >> 4
    d |= (uint64_t)1 << 16;                        // [16,30) leading byte offset (unused for swizzled K-major)
    d |= (uint64_t)(1024u >> 4) << 32;             // [32,46) stride byte offset: 8-row groups are 1024 B apart
    d |= (uint64_t)1 << 46;                        // [46,48) descriptor version 1 (sm_100)
    d |= (uint64_t)2 << 61;                        // [61,64) SWIZZLE_128B
    return d;
}
// instruction descriptor: D = f32, A = B = tf32, both K-major, N = 128, M = 128
constexpr uint32_t IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((128u >> 3) << 17) | ((128u >> 4) << 24);

__device__ __forceinline__ void mma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t phase) {
    asm volatile(
        "{\n\t"
        ".reg .pred P1;\n\t"
        "LAB_WAIT:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
        "@P1 bra DONE;\n\t"
        "bra LAB_WAIT;\n\t"
        "DONE:\n\t"
        "}\n" ::"r"(bar), "r"(phase)
        : "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Split x = hi + lo with ROUND-TO-NEAREST parts (ties away, like cvt.rna.tf32.f32): both hi and lo carry
// 11 significant bits exactly as the tensor core reads them, lo is signed, and the dropped lo.lo term has
// a random sign.  A truncating split (mask the 13 low bits) leaves every dropped term with the sign of its
// product -- a bias of ~2^-22 . sum|a.b| that shows as 2e-3 relative error in weight gradients whose terms
// cancel (conv3.weight at random initialisation, tests/test_gpu_synth_parity.py *_init cases).
__device__ __forceinline__ float tf32_hi(float x) { return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xFFFFE000u); }
__device__ __forceinline__ float tf32_lo(float x, float h) { return tf32_hi(x - h); }

struct Args {
    const float* A; int lda; const int32_t* m_dev; int m_host; int K;
    const float* B; int transB; float* C; int single_pass;
};
int make_tmap_rows(CUtensorMap* tmap, const float* A, int lda, int rows, int cols);


// ------------------------------------------------------------------------------------------------
// TMA-fed version with the WEIGHTS RESIDENT IN TENSOR MEMORY (the product path).
//
// The product is computed transposed:  D[n, m] = sum_k Wt[n, k] . X[m, k]  (= C[m, n]).  The tensor
// core's "A" operand is Wt and comes from TMEM (tcgen05.mma accepts A from tensor memory, K-major):
// hi and lo parts of the 128 x K weight matrix take 2 x K of the 512 TMEM columns for the lifetime of
// the CTA (K <= 128: two 128-column accumulators take the other 256; 128 < K <= 192, the 178-column
// feature table of layer 1: one accumulator) -- so NO shared memory is spent on the
// weights (a register-staged design that kept 128 KB of W in smem had room for only three 32 KB
// operand stages, and was measured slower) and the MMA reads half as many operand bytes from shared memory.  The "B"
// operand is the streamed X tile [128 rows m][32 k], K-major SWIZZLE_128B -- exactly what a TMA box
// load of the raw fp32 rows produces.
//   warp 5 (one lane)  TMA producer: cp.async.bulk.tensor.2d of a 128 x 32 fp32 box (16 KB, rows beyond the
//                      tensor are zero-filled by the hardware) into a ring of TM_RAW landing slots -- the
//                      loads in flight do not depend on how far the tensor core has got
//   warps 6-13         splitters: landing slot -> registers -> (hi, lo) -> operand slot (ring of TM_OPS);
//                      element positions do not move, so the TMA's swizzle is preserved without any
//                      index arithmetic; the landing slot is handed back to the TMA right away
//   warp 4 (one lane)  MMA issuer: three kind::tf32 MMAs per K step (lo.hi, hi.lo, hi.hi), tcgen05.commit
//                      releases the stage to the TMA producer
//   warps 0-3          epilogue: tcgen05.ld hands lane l of warp w the values C[m0 .. m0+31][32w + l]; a
//                      store instruction of the warp therefore writes 32 CONSECUTIVE floats of one row of
//                      C (128 B coalesced) with no register transpose (with C untransposed in TMEM, lane = row,
//                      160 shuffles per 32 x 32 block are needed for the same effect)
#ifndef NPI_TM_RAW
#define NPI_TM_RAW 6
#endif
#ifndef NPI_TM_OPS
#define NPI_TM_OPS 3
#endif
constexpr int TM_RAW = NPI_TM_RAW;          // landing slots of the TMA (16 KB each): the bytes in flight per SM
constexpr int TM_OPS = NPI_TM_OPS;          // operand slots (hi tile | lo tile, 32 KB each) between splitters and MMA
constexpr int TM_SPLIT_WARPS = 8;
constexpr int TM_THREADS = 32 * (4 + 1 + 1 + TM_SPLIT_WARPS);        // 448
constexpr uint32_t TM_TMEM_COLS = 512;                                // W_hi | W_lo | acc0 | acc1

__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const void* tmap, int c0, int c1, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(dst), "l"(tmap), "r"(c0), "r"(c1), "r"(bar)
        : "memory");
}
// D[tmem] (+)= A[tmem] . B[smem]
__device__ __forceinline__ void mma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(IDESC), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t* r) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};\n" ::"r"(taddr),
        "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]),
        "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]),
        "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
        : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

#ifdef NPI_TM_TRACE      // tuning builds only: time stamps of CTA 0 (ns since kernel entry), printed at exit
#define TM_STAMP(i) do { if (blockIdx.x == 0) { unsigned long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); tm_trace[i] = t_; } } while (0)
#else
#define TM_STAMP(i) do { } while (0)
#endif

__global__ void __launch_bounds__(TM_THREADS, 1) gemm_tc_tma_kernel(Args a, const __grid_constant__ CUtensorMap tmap) {
    extern __shared__ uint8_t smem_raw[];
#ifdef NPI_TM_TRACE
    __shared__ unsigned long long tm_trace[12];
    if (threadIdx.x == 0) TM_STAMP(0);
#endif
    __shared__ __align__(8) uint64_t bar_raw[TM_RAW], bar_rawfree[TM_RAW], bar_full[TM_OPS], bar_empty[TM_OPS], bar_tfull[2], bar_tempty[2], bar_w;
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int M = dev_size(a.m_dev, a.m_host);
    const int KB = (a.K + 31) / 32;                    // up to 6 K blocks (K <= 192: the 178-column feature table)
    const uint32_t col_wlo = (uint32_t)KB * 32u, col_acc = 2u * col_wlo;
    const int nacc = KB <= 4 ? 2 : 1;                 // 2 * 32 KB of weights + accumulators must fit the 512 TMEM columns
    const int ntiles = (M + 127) / 128;
    // programmatic dependent launch (common.cuh): tensor-memory allocation, barrier set-up and the staging of the weights
    // (written in an earlier step) run while the kernel that produces A is still finishing; only the TMA producer touches
    // A, and it waits for that kernel first -- everything downstream (split, MMA, epilogue stores) follows its loads
    pdl_trigger();
    if ((int)blockIdx.x >= ntiles) { pdl_wait(); return; }            // uniform: nothing allocated yet

    uint8_t* sA = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);      // TM_OPS x (hi tile | lo tile)
    uint8_t* sR = sA + TM_OPS * 2 * TILE_BYTES;                                     // TM_RAW landing tiles

    if (warp == 4) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"(TM_TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid == 0) {
        for (int i = 0; i < TM_RAW; ++i) { mbar_init(smem_u32(&bar_raw[i]), 1); mbar_init(smem_u32(&bar_rawfree[i]), 32 * TM_SPLIT_WARPS); }
        for (int i = 0; i < TM_OPS; ++i) { mbar_init(smem_u32(&bar_full[i]), 32 * TM_SPLIT_WARPS); mbar_init(smem_u32(&bar_empty[i]), 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(smem_u32(&bar_tfull[i]), 1); mbar_init(smem_u32(&bar_tempty[i]), 128); }
        mbar_init(smem_u32(&bar_w), 128 + 32 * TM_SPLIT_WARPS);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    const int my_tiles = (ntiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
    if (tid == 0) TM_STAMP(1);

    // ---- weights -> tensor memory: lane n of TMEM holds Wt[n][0..K), hi at columns 0.., lo at columns 128..
    // A warp reaches only the 32 TMEM lanes of its quadrant (warp % 4).  Twelve warps share the K blocks so that
    // every thread has ONE round of loads in flight (the first version staged all of W from the four epilogue
    // warps, K block after K block: 5-7 us before the first MMA could issue, tm_trace): epilogue warps 0-3 take
    // K blocks 0 and 3 (both loaded before either is converted), splitter warps 8-11 block 1, 12,13,6,7 block 2.
    auto load_w = [&](int kb, int n, float* raw) {
        if (a.transB) {
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const float4 v = ldg4(a.B + (int64_t)n * a.K + kb * 32 + q * 4);
                raw[q * 4 + 0] = v.x; raw[q * 4 + 1] = v.y; raw[q * 4 + 2] = v.z; raw[q * 4 + 3] = v.w;
            }
        } else {
#pragma unroll
            for (int i = 0; i < 32; ++i) raw[i] = (kb * 32 + i < a.K) ? __ldg(a.B + (int64_t)(kb * 32 + i) * 128 + n) : 0.f;
        }
    };
    auto store_w = [&](int kb, int quad, const float* raw) {
        uint32_t hi[32], lo[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) {
            const float h = tf32_hi(raw[i]);
            hi[i] = __float_as_uint(h); lo[i] = __float_as_uint(tf32_lo(raw[i], h));
        }
        const uint32_t t = tmem + ((uint32_t)(quad * 32) << 16) + kb * 32;
        tmem_st32(t, hi);
        tmem_st32(t + col_wlo, lo);
    };
    if (warp >= 6) {
        const int quad = warp & 3;
        for (int kb = (warp >= 8 && warp < 12) ? 1 : 2; kb < KB; kb += 3) {
            float raw[32];
            load_w(kb, quad * 32 + lane, raw);
            store_w(kb, quad, raw);
        }
        tmem_st_wait();
        tc_fence_before();
        mbar_arrive(smem_u32(&bar_w));
    }
    if (warp < 4) {
        {
            float raw0[32], raw3[32];
            load_w(0, warp * 32 + lane, raw0);
            if (KB > 3) load_w(3, warp * 32 + lane, raw3);
            store_w(0, warp, raw0);
            if (KB > 3) store_w(3, warp, raw3);
        }
        tmem_st_wait();
        tc_fence_before();
        mbar_arrive(smem_u32(&bar_w));
        if (tid == 0) TM_STAMP(2);
        // ================= epilogue =================
        for (int it = 0; it < my_tiles; ++it) {
            const int row0 = ((int)blockIdx.x + it * (int)gridDim.x) * 128;
            const int acc = it % nacc;
            mbar_wait(smem_u32(&bar_tfull[acc]), (uint32_t)((it / nacc) & 1));
            tc_fence_after();
            if (tid == 0 && it == 0) TM_STAMP(5);
#pragma unroll
            for (int cb = 0; cb < 4; ++cb) {
                uint32_t r[32];
                tmem_ld32(tmem + ((uint32_t)(warp * 32) << 16) + col_acc + acc * 128 + cb * 32, r);
                tmem_ld_wait();
                // r[j] = C[row0 + cb*32 + j][warp*32 + lane]
                const int rbase = row0 + cb * 32;
                float* dst = a.C + (int64_t)rbase * 128 + warp * 32 + lane;
#pragma unroll
                for (int j = 0; j < 32; ++j)
                    if (rbase + j < M) dst[(int64_t)j * 128] = __uint_as_float(r[j]);
            }
            tc_fence_before();
            mbar_arrive(smem_u32(&bar_tempty[acc]));
            if (tid == 0 && it == 0) TM_STAMP(6);
        }
    } else if (warp == 4) {
        // ================= MMA issuer =================
        if (lane == 0) {
            int s = 0;
            mbar_wait(smem_u32(&bar_w), 0u);                      // the weights are in tensor memory
            tc_fence_after();
            for (int it = 0; it < my_tiles; ++it) {
                const int acc = it % nacc;
                mbar_wait(smem_u32(&bar_tempty[acc]), (uint32_t)(((it / nacc) & 1) ^ 1));
                tc_fence_after();
                const uint32_t d = tmem + col_acc + acc * 128;
                for (int kb = 0; kb < KB; ++kb, ++s) {
                    const int st = s % TM_OPS;
                    mbar_wait(smem_u32(&bar_full[st]), (uint32_t)((s / TM_OPS) & 1));
                    tc_fence_after();
                    const uint32_t xh = smem_u32(sA) + st * 2 * TILE_BYTES, xl = xh + TILE_BYTES;
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks) {
                        const uint32_t ko = ks * 32;
                        const uint32_t wh = tmem + kb * 32 + ks * 8, wl = wh + col_wlo;
                        const uint32_t accum = (kb | ks) ? 1u : 0u;
                        if (a.single_pass) {
                            mma_tf32_ts(d, wh, make_desc(xh + ko), accum);
                        } else {
                            mma_tf32_ts(d, wl, make_desc(xh + ko), accum);
                            mma_tf32_ts(d, wh, make_desc(xl + ko), 1u);
                            mma_tf32_ts(d, wh, make_desc(xh + ko), 1u);
                        }
                    }
                    mma_commit(smem_u32(&bar_empty[st]));       // stage reusable once these MMAs have read it
                }
                mma_commit(smem_u32(&bar_tfull[acc]));          // accumulator complete
            }
        }
        __syncwarp();
    } else if (warp == 5) {
        // ================= TMA producer =================
        if (lane == 0) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap) : "memory");
            pdl_wait();
            const int total = my_tiles * KB;
            for (int s = 0; s < total; ++s) {
                const int st = s % TM_RAW, it = s / KB, kb = s % KB;
                const int row0 = ((int)blockIdx.x + it * (int)gridDim.x) * 128;
                mbar_wait(smem_u32(&bar_rawfree[st]), (uint32_t)(((s / TM_RAW) & 1) ^ 1));
                mbar_expect_tx(smem_u32(&bar_raw[st]), TILE_BYTES);
                tma_load_2d(smem_u32(sR) + st * TILE_BYTES, &tmap, kb * 32, row0, smem_u32(&bar_raw[st]));
            }
        }
        __syncwarp();
    } else {
        // ================= splitters =================
        const int t = tid - 32 * 6;                                   // 0..255
        const int total = my_tiles * KB;
        for (int s = 0; s < total; ++s) {
            const int rs = s % TM_RAW, st = s % TM_OPS;
            const uint8_t* raw = sR + rs * TILE_BYTES;
            uint8_t* hi = sA + st * 2 * TILE_BYTES;
            uint8_t* lo = hi + TILE_BYTES;
            mbar_wait(smem_u32(&bar_raw[rs]), (uint32_t)((s / TM_RAW) & 1));
            if (t == 0 && s == 0) TM_STAMP(3);
            float4 v[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) v[q] = *reinterpret_cast<const float4*>(raw + (uint32_t)(t + q * 256) * 16u);
            mbar_arrive(smem_u32(&bar_rawfree[rs]));                   // the landing slot can be refilled
            mbar_wait(smem_u32(&bar_empty[st]), (uint32_t)(((s / TM_OPS) & 1) ^ 1));
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const uint32_t off = (uint32_t)(t + q * 256) * 16u;
                const float4 h = make_float4(tf32_hi(v[q].x), tf32_hi(v[q].y), tf32_hi(v[q].z), tf32_hi(v[q].w));
                const float4 l = make_float4(tf32_lo(v[q].x, h.x), tf32_lo(v[q].y, h.y), tf32_lo(v[q].z, h.z), tf32_lo(v[q].w, h.w));
                *reinterpret_cast<float4*>(hi + off) = h;
                *reinterpret_cast<float4*>(lo + off) = l;
            }
            fence_async_smem();
            mbar_arrive(smem_u32(&bar_full[st]));
            if (t == 0 && s == 0) TM_STAMP(4);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 4)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(TM_TMEM_COLS) : "memory");
#ifdef NPI_TM_TRACE
    if (tid == 0 && blockIdx.x == 0) {
        TM_STAMP(7);
        printf("tm_trace M=%d tiles/cta=%d: init %llu  W-in-tmem %llu  first-raw %llu  first-split %llu  first-acc %llu  first-epilogue-done %llu  exit %llu ns\n",
               M, my_tiles, tm_trace[1] - tm_trace[0], tm_trace[2] - tm_trace[0], tm_trace[3] - tm_trace[0], tm_trace[4] - tm_trace[0],
               tm_trace[5] - tm_trace[0], tm_trace[6] - tm_trace[0], tm_trace[7] - tm_trace[0]);
    }
#endif
}



// ------------------------------------------------------------------------------------------------
// Weight gradient  out[128,128] = A[M,128]^T . D[M,128]  (dW = X^T . DXA of reference SAGEConv backward,
// SURVEY Appendix A.2) on tcgen05: the reduction runs over the ROWS, so both operands are "MN-major"
// for the tensor core -- a row of A (resp. D) holds the 128 values of the UMMA M (resp. N) dimension
// for one reduction index.  MN-major tf32 operands have exactly one legal shared-memory layout,
// SWIZZLE_128B_BASE32B (cute Layout_MN_SW128_32B_Atom: 32 floats x 4 rows, the 32-byte chunk index
// XORed with row & 3).  Slab of 32 rows: [4 column blocks of 32 floats][32 rows][128 B]; descriptor
// LBO = 4096 B (between column blocks), SBO = 512 B (between 4-row atoms); one UMMA_K step = 8 rows.  Persistent CTAs take slabs round-robin (split over rows),
// accumulate everything in ONE 128x128 fp32 TMEM tile and write it out once; the per-CTA partials
// are summed in a fixed order by gemm_tn_reduce_kernel.  Same 3xTF32 split as the projection above.
// Warp roles inside one CTA (1 CTA per SM):
//   warps 0-3    epilogue: TMEM -> registers -> global (warp w owns TMEM lanes 32w..32w+31)
//   warp  4      MMA issuer (one elected lane) + TMEM allocation
//   warps 5-16   three producer groups of 4 warps; group g fills smem stage g with the slabs s = g, g+3, g+6, ...
//                (global -> registers -> hi/lo split -> swizzled smem), so three slabs are in flight per SM
//                while the tensor core works on a fourth; tcgen05.commit frees a stage when its MMAs have read it
constexpr int WS_STAGES = 3;
constexpr int WS_EPI_WARPS = 4;
constexpr int WS_PROD_WARPS = 4 * WS_STAGES;
constexpr int WS_THREADS = 32 * (WS_EPI_WARPS + 1 + WS_PROD_WARPS);     // 544
constexpr uint32_t TN_SLAB_ROWS = 32;
constexpr uint32_t TN_OPER_BYTES = TN_SLAB_ROWS * 512;          // one operand slab (hi or lo): 16 KB
constexpr uint32_t IDESC_MN = IDESC | (1u << 15) | (1u << 16);  // A and B MN-major

__device__ __forceinline__ uint64_t make_desc_mn(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
    d |= (uint64_t)(4096u >> 4) << 16;             // LBO: next block of 32 columns
    d |= (uint64_t)(512u >> 4) << 32;              // SBO: next 4-row atom
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)1 << 61;                        // SWIZZLE_128B_BASE32B
    return d;
}
__device__ __forceinline__ void mma_tf32_mn(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(IDESC_MN), "r"(accumulate)
        : "memory");
}
// 16-byte chunk c16 (0..31) of slab row m, hi and lo parts
__device__ __forceinline__ void put_chunk_mn(uint8_t* hi, uint8_t* lo, int m, int c16, float4 v) {
    const int c8 = c16 & 7;                        // 16-byte chunk inside the 128-byte block row
    const uint32_t off = (uint32_t)((c16 >> 3) * 4096 + m * 128 + ((((c8 >> 1) ^ (m & 3)) << 5) | ((c8 & 1) << 4)));
    float4 h = make_float4(tf32_hi(v.x), tf32_hi(v.y), tf32_hi(v.z), tf32_hi(v.w));
    float4 l = make_float4(tf32_lo(v.x, h.x), tf32_lo(v.y, h.y), tf32_lo(v.z, h.z), tf32_lo(v.w, h.w));
    *reinterpret_cast<float4*>(hi + off) = h;
    *reinterpret_cast<float4*>(lo + off) = l;
}

struct TnArgs {
    const float* A; int lda; int a_cols;   // columns of A at or past a_cols (a multiple of 4) are taken as zero
    const float* D; const int32_t* m_dev; int m_host;
    float* part;        // [gridDim.x][128][128]
    int single_pass;
};

__global__ void __launch_bounds__(WS_THREADS, 1) gemm_tn_tc_kernel(TnArgs a) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bar_full[WS_STAGES], bar_empty[WS_STAGES], bar_done;
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int M = dev_size(a.m_dev, a.m_host);
    const int nslabs = (M + (int)TN_SLAB_ROWS - 1) / (int)TN_SLAB_ROWS;
    const int my = ((int)blockIdx.x < nslabs) ? (nslabs - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
    float* part = a.part + (int64_t)blockIdx.x * 128 * 128;
    if (my == 0) {                                    // uniform: this CTA contributes a zero partial
        for (int e = tid; e < 128 * 32; e += WS_THREADS) st4(part + 4 * e, make_float4(0.f, 0.f, 0.f, 0.f));
        return;
    }
    uint8_t* base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // stage: A_hi | A_lo | D_hi | D_lo

    if (warp == WS_EPI_WARPS) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid == 0) {
        for (int i = 0; i < WS_STAGES; ++i) { mbar_init(smem_u32(&bar_full[i]), 128); mbar_init(smem_u32(&bar_empty[i]), 1); }
        mbar_init(smem_u32(&bar_done), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;

    if (warp < WS_EPI_WARPS) {
        // ================= epilogue: TMEM lane = k (row of out), column = n =================
        mbar_wait(smem_u32(&bar_done), 0u);
        tc_fence_after();
        const int k = warp * 32 + lane;
#pragma unroll
        for (int cb = 0; cb < 4; ++cb) {
            uint32_t r[32];
            tmem_ld32(tmem + ((uint32_t)(warp * 32) << 16) + cb * 32, r);
            tmem_ld_wait();
            float* dst = part + (int64_t)k * 128 + cb * 32;
#pragma unroll
            for (int i = 0; i < 8; ++i)
                st4(dst + 4 * i, make_float4(__uint_as_float(r[4 * i]), __uint_as_float(r[4 * i + 1]),
                                             __uint_as_float(r[4 * i + 2]), __uint_as_float(r[4 * i + 3])));
        }
    } else if (warp == WS_EPI_WARPS) {
        // ================= MMA issuer =================
        if (lane == 0) {
            for (int s = 0; s < my; ++s) {
                const int st = s % WS_STAGES;
                mbar_wait(smem_u32(&bar_full[st]), (uint32_t)((s / WS_STAGES) & 1));
                tc_fence_after();
                const uint32_t ah = smem_u32(base) + st * 4 * TN_OPER_BYTES, al = ah + TN_OPER_BYTES;
                const uint32_t dh = al + TN_OPER_BYTES, dl = dh + TN_OPER_BYTES;
#pragma unroll
                for (int b = 0; b < 4; ++b) {              // 8 rows per UMMA_K step
                    const uint32_t ko = b * 1024;
                    const uint32_t accum = (s | b) ? 1u : 0u;
                    if (a.single_pass) {
                        mma_tf32_mn(tmem, make_desc_mn(ah + ko), make_desc_mn(dh + ko), accum);
                    } else {
                        mma_tf32_mn(tmem, make_desc_mn(al + ko), make_desc_mn(dh + ko), accum);
                        mma_tf32_mn(tmem, make_desc_mn(ah + ko), make_desc_mn(dl + ko), 1u);
                        mma_tf32_mn(tmem, make_desc_mn(ah + ko), make_desc_mn(dh + ko), 1u);
                    }
                }
                mma_commit(smem_u32(&bar_empty[st]));
            }
            mma_commit(smem_u32(&bar_done));
        }
        __syncwarp();
    } else {
        // ================= producers =================
        const int g = (warp - WS_EPI_WARPS - 1) >> 2;
        const int t = tid - 32 * (WS_EPI_WARPS + 1) - g * 128;
        uint8_t* ah = base + g * 4 * TN_OPER_BYTES;
        uint8_t* al = ah + TN_OPER_BYTES;
        uint8_t* dh = al + TN_OPER_BYTES;
        uint8_t* dl = dh + TN_OPER_BYTES;
        for (int s = g, u = 0; s < my; s += WS_STAGES, ++u) {
            const int row0 = ((int)blockIdx.x + s * (int)gridDim.x) * (int)TN_SLAB_ROWS;
            float4 va[8], vd[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const int e = t + q * 128;                 // 32 rows x 32 chunks
                const int m = e >> 5, c16 = e & 31;
                const int gr = row0 + m;
                if (gr < M) {
                    va[q] = (c16 * 4 < a.a_cols) ? ldg4(a.A + (int64_t)gr * a.lda + c16 * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
                    vd[q] = ldg4(a.D + (int64_t)gr * 128 + c16 * 4);
                } else {
                    va[q] = make_float4(0.f, 0.f, 0.f, 0.f);
                    vd[q] = make_float4(0.f, 0.f, 0.f, 0.f);
                }
            }
            mbar_wait(smem_u32(&bar_empty[g]), (uint32_t)((u & 1) ^ 1));
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const int e = t + q * 128;
                put_chunk_mn(ah, al, e >> 5, e & 31, va[q]);
                put_chunk_mn(dh, dl, e >> 5, e & 31, vd[q]);
            }
            fence_async_smem();
            mbar_arrive(smem_u32(&bar_full[g]));
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == WS_EPI_WARPS)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(TMEM_COLS) : "memory");
}

// Tensor map of a row-major fp32 matrix [rows, cols] (row stride lda floats): boxes of 32 columns x 128 rows,
// SWIZZLE_128B (the 16-byte chunk index XORed with row & 7 inside 1024-byte groups = the UMMA K-major layout).
// cuTensorMapEncodeTiled is a driver entry point; it is resolved through the runtime so that libnpi links
// against cudart only.
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
int make_tmap_rows(CUtensorMap* tmap, const float* A, int lda, int rows, int cols) {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        NPI_CHECK_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres));
        NPI_REQUIRE(p && qres == cudaDriverEntryPointSuccess, "gemm_nn_tc: cuTensorMapEncodeTiled is not available in this driver");
        fn = (EncodeTiledFn)p;
    }
    const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)lda * sizeof(float)};
    const cuuint32_t box[2] = {32u, 128u};
    const cuuint32_t estr[2] = {1u, 1u};
    const CUresult rc = fn(tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(A), dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    NPI_REQUIRE(rc == CUDA_SUCCESS, "gemm_nn_tc: cuTensorMapEncodeTiled failed (CUresult %d; A=%p lda=%d rows=%d cols=%d)", (int)rc,
                (const void*)A, lda, rows, cols);
    return NPI_OK;
}

}  // namespace tc
}  // namespace npi

using namespace npi;

extern "C" int npi_gemm_nn_tc(const float* A, int32_t lda, const int32_t* m_dev, int32_t m_host, int32_t K,
                              const float* B, int32_t transB, float* C, int32_t single_pass, npi_stream_t stream) {
    NPI_REQUIRE(A && B && C, "gemm_nn_tc: null argument");
    NPI_REQUIRE(K >= 1 && K <= 192, "gemm_nn_tc: K must be in 1..192 (got %d)", K);
    NPI_REQUIRE(!transB || (K % 32 == 0 && K <= 128), "gemm_nn_tc: transB needs K in {32, 64, 96, 128} (got %d)", K);
    NPI_REQUIRE(lda >= K && lda % 4 == 0 && (reinterpret_cast<uintptr_t>(A) & 15) == 0 && (reinterpret_cast<uintptr_t>(B) & 15) == 0,
                "gemm_nn_tc: operands must be 16-byte aligned with lda %% 4 == 0");
    NPI_REQUIRE(m_host > 0, "gemm_nn_tc: m_host must be positive");
    tc::Args a{A, lda, m_dev, m_host, K, B, transB, C, single_pass & 1};
    int tiles = (m_host + 127) / 128;
    int grid = num_sms();
    if (tiles < grid) grid = tiles;
    CUtensorMap tmap;
    if (int rc = tc::make_tmap_rows(&tmap, A, lda, m_host, K)) return rc;
    const size_t smem = (size_t)(2 * tc::TM_OPS + tc::TM_RAW) * tc::TILE_BYTES + 1024;
    static OncePerDevice configured;
    if (configured.need()) {
        NPI_CHECK_CUDA(cudaFuncSetAttribute(tc::gemm_tc_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    NPI_CHECK_CUDA(launch_dep(tc::gemm_tc_tma_kernel, grid, tc::TM_THREADS, smem, (cudaStream_t)stream, a, tmap));
    NPI_CHECK_LAUNCH();
    return NPI_OK;
}

extern "C" int64_t npi_gemm_tn_tc_workspace_bytes(void) { return (int64_t)num_sms() * 128 * 128 * sizeof(float); }

extern "C" int npi_gemm_tn_tc(const float* A, int32_t lda, int32_t K, const float* D, const int32_t* m_dev, int32_t m_host,
                              const float* row0_partials, int32_t R, float* out, int32_t single_pass,
                              void* workspace, int64_t workspace_bytes, npi_stream_t stream) {
    NPI_REQUIRE(A && D && out && workspace, "gemm_tn_tc: null argument");
    NPI_REQUIRE(K >= 1 && lda >= K && lda % 4 == 0 && (reinterpret_cast<uintptr_t>(A) & 15) == 0 && (reinterpret_cast<uintptr_t>(D) & 15) == 0,
                "gemm_tn_tc: operands must be 16-byte aligned, lda %% 4 == 0, lda >= K");
    NPI_REQUIRE(workspace_bytes >= npi_gemm_tn_tc_workspace_bytes(), "gemm_tn_tc: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t smem = (size_t)tc::WS_STAGES * 4 * tc::TN_OPER_BYTES + 1024;
    static OncePerDevice configured;
    if (configured.need()) {
        NPI_CHECK_CUDA(cudaFuncSetAttribute(tc::gemm_tn_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    const int grid = num_sms();
    // out rows in tiles of 128 columns of A: the 178-column feature table of the layer-1 weight gradient takes two
    // passes over G (columns 0..127, then 128..lda-1 with the rest of the tile read as zero)
    for (int k0 = 0; k0 < K; k0 += 128) {
        const int rows = K - k0 < 128 ? K - k0 : 128;
        int cols = lda - k0 < 128 ? lda - k0 : 128;         // lda % 4 == 0; columns K..lda-1 are zero by the table's contract
        tc::TnArgs a{A + k0, lda, cols, D, m_dev, m_host, (float*)workspace, single_pass & 1};
        tc::gemm_tn_tc_kernel<<<grid, tc::WS_THREADS, smem, st>>>(a);
        NPI_CHECK_LAUNCH();
        if (int rc = launch_gemm_tn_reduce((const float*)workspace, grid, 1, rows, k0 == 0 ? row0_partials : nullptr, R,
                                           out + (int64_t)k0 * 128, st)) return rc;
    }
    return NPI_OK;
}
