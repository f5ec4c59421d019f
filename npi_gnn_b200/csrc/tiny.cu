// Small-subgraph path: conv1..3 + pool1..3 + readout of ONE enclosing subgraph per CTA, forward and backward.
//
// Replaces, for batches of small subgraphs, the per-layer launches of reference src/classes.py:62-72 (Net_1.forward:
// SAGEConv -> TopKPooling -> cat[gmp, gap], three times) and of their backward.  RPI2241's two-hop enclosing subgraphs
// have 15 nodes on average (87 at most): a batch of 200 is ~3 k rows, and the layer-by-layer path needs 58 launches of
// 5-25 us each for it -- the step is launch- and dependency-bound (0.236 ms for 3 k rows, 0.014 of the roofline).  Nothing
// in the three layers crosses a subgraph except the parameter gradients, so a CTA takes one subgraph through all of
// them, with block barriers where the layer-by-layer path has kernel boundaries.  What a CTA is bound by is the number of
// DEPENDENT round trips to L2 (~0.7 us each), so the kernels are organised around removing them:
//   * the subgraph's index structures (row pointers, local column indices, global ids / hop labels, and in the backward
//     new_id, scores, 1/(deg+1)) are fetched ONCE per layer into shared memory by the whole CTA (two round trips), and
//     filter_adj produces the next layer's CSR in shared memory as well as in global memory;
//   * the 128 x 128 weight of the next projection is staged into shared memory by one bulk asynchronous copy
//     (cp.async.bulk + mbarrier, 64 KB) issued a layer ahead, so it lands while the CTA aggregates, sorts and gates;
//   * the first 16 rows of every intermediate (gated rows, projected rows, h, dpre, dxa, dX: most subgraphs have no more)
//     are kept in shared-memory tiles next to their global copies;
//   * a HALF-warp owns a row (16 rows in flight per CTA, two float4 per lane), entries are read from shared memory, four
//     feature-row loads in flight per row.
// Activations also land in the SAME global buffers the layer-by-layer path uses (a batch is 1.5 MB: L2 resident), so
// the head, the weight-gradient GEMMs (X^T . DXA on tcgen05, the feature-table route for conv1), the tests and the
// scorer read them unchanged.  Everything a CTA wrote earlier in the same launch is read back with plain (coherent)
// loads -- __ldg only for inputs no kernel of the launch writes.
// The filtered adjacency of the pooled layers is kept per subgraph: subgraph g's rows of layer l >= 1 own the n_g + 1
// row pointers rowptr_f[l-1][lo_g + g ...], its entries start where its entries of the input layer start (a filtered
// edge list is never longer) -- no scan over the batch, hence no dependency between CTAs.
// Sums run in a fixed order (CSR order then the self row; half-warps combined in order): reruns are bit-identical, and
// layer 1's h is bit-identical to aggregate_fwd_kernel's.
#include "common.cuh"

namespace npi {

constexpr int TN_THREADS = 256;
constexpr int TN_WARPS = TN_THREADS / 32;
constexpr int TN_HW = TN_THREADS / 16;    // half-warps: rows in flight per CTA
constexpr int TN_TILE = 16;               // rows per projection tile (two halves of the CTA, 8 rows each) = rows kept in shared memory
constexpr int TN_MAX_NODES = 1024;        // index arrays / sort keys of one subgraph in shared memory
constexpr int TN_RANK_MAX = 256;          // up to this many nodes the top-k is a rank count (one thread per node), beyond: bitonic network
constexpr int TN_PART = 2 * H + 4;        // per-subgraph partial: sum dz*h [128] | sum dz*z | pad[3] | sum dpre [128]  (npi_pool_bwd's layout)
constexpr uint32_t TN_W_BYTES = H * H * sizeof(float);

// -DNPI_TN_TRACE: thread 0 of every CTA records %globaltimer at the phase boundaries (tools/tiny_trace.py); the forward
// borrows dxa[0], the backward y[1] (buffers the kernel itself does not touch) for 32 stamps per CTA
#ifdef NPI_TN_TRACE
#define TN_STAMP(buf, idx)                                                                         \
    do {                                                                                           \
        if (threadIdx.x == 0) {                                                                    \
            unsigned long long t_;                                                                 \
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_));                                 \
            reinterpret_cast<unsigned long long*>(buf)[(size_t)blockIdx.x * 32 + (idx)] = t_;      \
        }                                                                                          \
    } while (0)
#else
#define TN_STAMP(buf, idx) do { } while (0)
#endif

__device__ __forceinline__ float4 tn_ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void tn_fma4(float4& acc, const float4& v, float w) {
    acc.x = fmaf(v.x, w, acc.x); acc.y = fmaf(v.y, w, acc.y); acc.z = fmaf(v.z, w, acc.z); acc.w = fmaf(v.w, w, acc.w);
}
__device__ __forceinline__ float4 tn_zero4() { return make_float4(0.f, 0.f, 0.f, 0.f); }
__device__ __forceinline__ uint32_t tn_orderable(float f) {
    uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float tn_half_sum(float v) {         // over the 16 lanes of a half-warp (all 32 lanes call it)
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---- bulk asynchronous copy of one 128 x 128 weight into shared memory (one thread issues, everybody waits on the barrier)
__device__ __forceinline__ uint32_t tn_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void tn_bar_init(uint64_t* bar) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(tn_smem_u32(bar)) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void tn_stage_weight(float* dst, const float* src, uint64_t* bar) {
    const uint32_t b = tn_smem_u32(bar);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      // the CTA's earlier reads of dst come before the copy's writes
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(b), "r"(TN_W_BYTES) : "memory");
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(tn_smem_u32(dst + q * (H * H / 4))), "l"(src + q * (H * H / 4)), "r"(TN_W_BYTES / 4), "r"(b)
                     : "memory");
    }
}
__device__ __forceinline__ void tn_bar_wait(uint64_t* bar, uint32_t parity) {
    const uint32_t b = tn_smem_u32(bar);
    for (int it = 0;; ++it) {
        uint32_t ok;
        asm volatile(
            "{\n\t"
            ".reg .pred P1;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, P1;\n\t"
            "}\n" : "=r"(ok) : "r"(b), "r"(parity) : "memory");
        if (ok) break;
        if (it > (1 << 22)) __trap();          // a copy that never lands must not hang the device
    }
}

// ---- shared-memory layout (dynamic part), the same for both kernels
struct TnSmem {
    float* W;            // [128*128] staged weight
    uint64_t* bar;
    uint64_t* keys;      // [cap]   sort keys (forward)
    float* sS;           // [cap]   scores
    float* sZ;           // [cap]   pre-tanh scores (backward)
    float* sInv;         // [cap]   1/(deg+1) (backward)
    int* sNew;           // [cap]   local new id after the layer's top-k, or -1
    int* sPerm;          // [cap]   local old row of every selected row
    int* sCnt;           // [cap]   filter_adj: kept entries per new row / their exclusive prefix
    int* sGid;           // [cap]   gid | dist << 29 (input layer)
    int* sRp[2];         // [cap+1] row pointers relative to the subgraph's first entry (ping-pong over the layers)
    int* sCol[2];        // [ecap]  local column indices
    int cap, ecap;
};
__host__ __device__ inline int tn_ecap(int cap) { return cap * 4 < 4096 ? cap * 4 : 4096; }
__host__ __device__ inline size_t tn_smem_bytes(int cap) {
    return (size_t)TN_W_BYTES + 16 + (size_t)cap * 8 + (size_t)cap * 4 * 7 + (size_t)(cap + 4) * 4 * 2 + (size_t)tn_ecap(cap) * 4 * 2;
}
__device__ __forceinline__ TnSmem tn_carve(unsigned char* base, int cap) {
    TnSmem s;
    s.cap = cap; s.ecap = tn_ecap(cap);
    s.W = reinterpret_cast<float*>(base); base += TN_W_BYTES;
    s.bar = reinterpret_cast<uint64_t*>(base); base += 16;
    s.keys = reinterpret_cast<uint64_t*>(base); base += (size_t)cap * 8;
    s.sS = reinterpret_cast<float*>(base); base += (size_t)cap * 4;
    s.sZ = reinterpret_cast<float*>(base); base += (size_t)cap * 4;
    s.sInv = reinterpret_cast<float*>(base); base += (size_t)cap * 4;
    s.sNew = reinterpret_cast<int*>(base); base += (size_t)cap * 4;
    s.sPerm = reinterpret_cast<int*>(base); base += (size_t)cap * 4;
    s.sCnt = reinterpret_cast<int*>(base); base += (size_t)cap * 4;
    s.sGid = reinterpret_cast<int*>(base); base += (size_t)cap * 4;
    s.sRp[0] = reinterpret_cast<int*>(base); base += (size_t)(cap + 4) * 4;
    s.sRp[1] = reinterpret_cast<int*>(base); base += (size_t)(cap + 4) * 4;
    s.sCol[0] = reinterpret_cast<int*>(base); base += (size_t)s.ecap * 4;
    s.sCol[1] = reinterpret_cast<int*>(base);
    return s;
}
// local column index of entry e of the subgraph: shared memory for the first ecap entries, global memory beyond
__device__ __forceinline__ int tn_col(const int* sCol, int ecap, const int32_t* colg, int e, int lo) {
    return e < ecap ? sCol[e] : colg[e] - lo;
}

// Y[lo + r][:] = X[lo + r][:] . W for r < n, W [128,128] row-major in shared memory, in tiles of 8 rows.  Thread = (output
// column, half of K): the two halves of the CTA run the same rows over k < 64 and k >= 64 (k ascending, one fma chain per
// output and half), the upper half's sums go through pbuf and are added by the lower half.  R = rows computed (2, 4 or 8: a
// subgraph's pooled layers have 8 / 4 rows on average, and the FMAs + shared-memory reads of padding rows were most of the
// projection's time).  first_staged: the caller left rows 0..15 (zero padded) in xs already.  ytile (nullable): rows 0..15 of
// the result also go there.
template <int R>
__device__ __forceinline__ void tn_project_tile(const float* xr, const float* Ws, float* Y, int lo, int row0, int n, float* pbuf, float* ytile) {
    const int tid = threadIdx.x, c = tid & (H - 1), kh = tid >> 7;
    float acc[R];
#pragma unroll
    for (int r = 0; r < R; ++r) acc[r] = 0.f;
    const int kb = kh * (H / 2);
#pragma unroll 4
    for (int kk = kb; kk < kb + H / 2; kk += 4) {
        const float w0 = Ws[(kk + 0) * H + c], w1 = Ws[(kk + 1) * H + c], w2 = Ws[(kk + 2) * H + c], w3 = Ws[(kk + 3) * H + c];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const float4 x = tn_ld4(xr + r * H + kk);
            acc[r] = fmaf(x.x, w0, acc[r]); acc[r] = fmaf(x.y, w1, acc[r]);
            acc[r] = fmaf(x.z, w2, acc[r]); acc[r] = fmaf(x.w, w3, acc[r]);
        }
    }
    if (kh == 1) {
#pragma unroll
        for (int r = 0; r < R; ++r) pbuf[r * H + c] = acc[r];
    }
    __syncthreads();
    if (kh == 0) {
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int row = row0 + r;
            if (row < n) {
                const float v = acc[r] + pbuf[r * H + c];
                Y[(int64_t)(lo + row) * H + c] = v;
                if (ytile && row < TN_TILE) ytile[row * H + c] = v;
            }
        }
    }
}

__device__ __forceinline__ void tn_project(const float* X, const float* Ws, float* Y, int lo, int n, float* xs, bool first_staged, float* ytile,
                                           float* pbuf) {
    const int tid = threadIdx.x;
#pragma unroll 1
    for (int r0 = 0; r0 < n; r0 += 8) {
        const bool in_xs = first_staged && r0 < TN_TILE;
        const float* xr = in_xs ? xs + r0 * H : xs;
        if (!in_xs) {
            __syncthreads();
            {
                const int r = tid >> 5, q = tid & 31;                       // 8 rows x 32 float4 = one load per thread
                float4 v = tn_zero4();
                if (r0 + r < n) v = tn_ld4(X + (int64_t)(lo + r0 + r) * H + 4 * q);
                reinterpret_cast<float4*>(xs)[tid] = v;
            }
        }
        __syncthreads();
        const int rows = n - r0;
        if (rows > 4) tn_project_tile<8>(xr, Ws, Y, lo, r0, n, pbuf, ytile);
        else if (rows > 2) tn_project_tile<4>(xr, Ws, Y, lo, r0, n, pbuf, ytile);
        else tn_project_tile<2>(xr, Ws, Y, lo, r0, n, pbuf, ytile);
    }
    __syncthreads();
}

// ------------------------------------------------------------------ forward
// h_i = relu((sum_{j in row(i)} y_j + y_i) / (deg_i + 1) + b), z_i = h_i . p / |p|, s_i = tanh(z_i): a half-warp per row, lane =
// columns 4*l16.. and 64 + 4*l16...  VIRT: y_j = T[gid_j] + dist_j * W1[0,:] (same order of operations as aggregate_fwd_kernel).
template <bool VIRT>
__device__ __forceinline__ void tn_aggregate(const npi_tiny_args_t& a, int l, int lo, int n, const TnSmem& sm, const int* sRp, const int* sCol,
                                             const int32_t* colg, const float* Y, const float* ytile, float* htile) {
    const int tid = threadIdx.x, hw = tid >> 4, l16 = tid & 15;
    const int c0 = 4 * l16, c1 = 64 + 4 * l16;
    const float4 p0 = ldg4(a.pool_w[l] + c0), p1 = ldg4(a.pool_w[l] + c1);
    const float norm = sqrtf(tn_half_sum(dot4(p0, p0) + dot4(p1, p1)));
    const float4 b0 = ldg4(a.bias[l] + c0), b1 = ldg4(a.bias[l] + c1);
    float4 w00 = tn_zero4(), w01 = tn_zero4();
    if (VIRT) { w00 = ldg4(a.w_label + c0); w01 = ldg4(a.w_label + c1); }
    for (int i0 = 0; i0 < n; i0 += TN_HW) {
        if (i0 + (hw & ~1) >= n) continue;        // neither half of this warp has a row in this round: straight to the barrier
        const int i = i0 + hw;
        const bool valid = i < n;
        const int beg = valid ? sRp[i] : 0, end = valid ? sRp[i + 1] : 0;
        float4 acc0 = tn_zero4(), acc1 = tn_zero4();
        int dsum = 0;
        // the self row's load is issued first (it is added last): rows of up to four entries cost one round trip
        float4 self0 = tn_zero4(), self1 = tn_zero4();
        int dself = 0;
        if (valid) {
            const float* src;
            if (VIRT) {
                const int pk = sm.sGid[i];
                dself = (int)((uint32_t)pk >> 29);
                src = Y + (int64_t)(pk & 0x1fffffff) * H;
                self0 = ldg4(src + c0); self1 = ldg4(src + c1);
            } else {
                src = i < TN_TILE ? ytile + i * H : Y + (int64_t)(lo + i) * H;
                self0 = tn_ld4(src + c0); self1 = tn_ld4(src + c1);
            }
        }
        for (int e = beg; e < end; e += 4) {
            float4 v0[4], v1[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (e + u < end) {
                    const int j = tn_col(sCol, sm.ecap, colg, e + u, lo);
                    const float* src;
                    if (VIRT) {
                        const int pk = sm.sGid[j];
                        dsum += (int)((uint32_t)pk >> 29);
                        src = Y + (int64_t)(pk & 0x1fffffff) * H;
                        v0[u] = ldg4(src + c0); v1[u] = ldg4(src + c1);
                    } else {
                        src = j < TN_TILE ? ytile + j * H : Y + (int64_t)(lo + j) * H;
                        v0[u] = tn_ld4(src + c0); v1[u] = tn_ld4(src + c1);
                    }
                }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (e + u < end) { acc0 = add4(acc0, v0[u]); acc1 = add4(acc1, v1[u]); }
            }
        }
        acc0 = add4(acc0, self0); acc1 = add4(acc1, self1);                      // self loop last
        dsum += dself;
        if (VIRT) { tn_fma4(acc0, w00, (float)dsum); tn_fma4(acc1, w01, (float)dsum); }      // label column (exact integer sum)
        const float dv = (float)(end - beg + 1);
        float4 o0 = make_float4(acc0.x / dv + b0.x, acc0.y / dv + b0.y, acc0.z / dv + b0.z, acc0.w / dv + b0.w);
        float4 o1 = make_float4(acc1.x / dv + b1.x, acc1.y / dv + b1.y, acc1.z / dv + b1.z, acc1.w / dv + b1.w);
        o0.x = fmaxf(o0.x, 0.f); o0.y = fmaxf(o0.y, 0.f); o0.z = fmaxf(o0.z, 0.f); o0.w = fmaxf(o0.w, 0.f);
        o1.x = fmaxf(o1.x, 0.f); o1.y = fmaxf(o1.y, 0.f); o1.z = fmaxf(o1.z, 0.f); o1.w = fmaxf(o1.w, 0.f);
        const float d = tn_half_sum(dot4(o0, p0) + dot4(o1, p1));
        if (valid) {
            float* hr = a.h[l] + (int64_t)(lo + i) * H;
            st4(hr + c0, o0); st4(hr + c1, o1);
            if (i < TN_TILE) { st4(htile + i * H + c0, o0); st4(htile + i * H + c1, o1); }
            if (l16 == 0) {
                const float zz = d / norm;
                const float ss = tanhf(zz) + 0.0f;
                a.z[l][lo + i] = zz;
                a.s[l][lo + i] = ss;
                sm.sS[i] = ss;
            }
        }
    }
}

// per-subgraph top-k: keys (~orderable(score) << 32 | index) ascending = descending score, ties by lower index (Appendix A.3;
// the keys of topk_select_kernel).  Up to TN_RANK_MAX nodes: one thread per node counts the keys below its own (keys are
// distinct, so the counts are a permutation) -- no barrier per sorting step; larger subgraphs: bitonic network.
__device__ __forceinline__ void tn_topk(const npi_tiny_args_t& a, int l, int g, int lo, int n, int olo, int k, const TnSmem& sm) {
    const int tid = threadIdx.x;
    uint64_t* keys = sm.keys;
    int np2 = 1;
    while (np2 < n) np2 <<= 1;
    const int nk = n <= TN_RANK_MAX ? n : np2;
    for (int i = tid; i < nk; i += TN_THREADS)
        keys[i] = i < n ? (((uint64_t)(~tn_orderable(sm.sS[i] + 0.0f)) << 32) | (uint32_t)i) : ~0ull;
    __syncthreads();
    if (n <= TN_RANK_MAX) {
        if (tid < n) {
            const uint64_t mine = keys[tid];
            int r = 0;
#pragma unroll 4
            for (int j = 0; j < n; ++j) r += keys[j] < mine ? 1 : 0;
            if (r < k) {
                a.perm[l][olo + r] = lo + tid;
                a.new_id[l][lo + tid] = olo + r;
                a.batch[l][olo + r] = g;
                sm.sPerm[r] = tid;
                sm.sNew[tid] = r;
            } else {
                a.new_id[l][lo + tid] = -1;
                sm.sNew[tid] = -1;
            }
        }
    } else {
        for (int size = 2; size <= np2; size <<= 1) {
            for (int stride = size >> 1; stride > 0; stride >>= 1) {
                for (int t = tid; t < (np2 >> 1); t += TN_THREADS) {
                    const int pos = 2 * t - (t & (stride - 1));
                    const int par = pos + stride;
                    const bool up = ((pos & size) == 0);
                    const uint64_t x = keys[pos], y = keys[par];
                    if ((x > y) == up) { keys[pos] = y; keys[par] = x; }
                }
                __syncthreads();
            }
        }
        for (int r = tid; r < n; r += TN_THREADS) {
            const int idx = (int)(uint32_t)(keys[r] & 0xffffffffull);
            if (r < k) {
                a.perm[l][olo + r] = lo + idx;
                a.new_id[l][lo + idx] = olo + r;
                a.batch[l][olo + r] = g;
                sm.sPerm[r] = idx;
                sm.sNew[idx] = r;
            } else {
                a.new_id[l][lo + idx] = -1;
                sm.sNew[idx] = -1;
            }
        }
    }
    __syncthreads();
}

// filter_adj of one subgraph: new row r = old row perm[r], dropped sources removed, the rest relabelled, order kept.  Reads
// the layer's CSR from shared memory, leaves the next layer's in shared memory (sRpN, sColN) and in global memory.
__device__ __forceinline__ void tn_filter(const TnSmem& sm, const int* sRp, const int* sCol, const int32_t* colg, int lo, int olo, int k, int base,
                                          int* sRpN, int* sColN, int32_t* rp_out, int32_t* col_out) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int r = warp; r < k; r += TN_WARPS) {
        const int o = sm.sPerm[r];
        const int beg = sRp[o], end = sRp[o + 1];
        int cnt = 0;
        for (int e0 = beg; e0 < end; e0 += 32) {
            const int e = e0 + lane;
            bool keep = false;
            if (e < end) keep = sm.sNew[tn_col(sCol, sm.ecap, colg, e, lo)] >= 0;
            cnt += __popc(__ballot_sync(0xffffffffu, keep));
        }
        if (lane == 0) sm.sCnt[r] = cnt;
    }
    __syncthreads();
    if (warp == 0) {
        int run = 0;
        for (int b0 = 0; b0 < k; b0 += 32) {
            const int v = (b0 + lane < k) ? sm.sCnt[b0 + lane] : 0;
            const int inc = warp_incl_scan_i(v, lane);
            if (b0 + lane < k) sRpN[b0 + lane] = run + inc - v;
            run += __shfl_sync(0xffffffffu, inc, 31);
        }
        if (lane == 0) sRpN[k] = run;
    }
    __syncthreads();
    for (int r = tid; r <= k; r += TN_THREADS) rp_out[r] = base + sRpN[r];
    for (int r = warp; r < k; r += TN_WARPS) {
        const int o = sm.sPerm[r];
        const int beg = sRp[o], end = sRp[o + 1];
        int w = sRpN[r];
        for (int e0 = beg; e0 < end; e0 += 32) {
            const int e = e0 + lane;
            int nj = -1;
            if (e < end) nj = sm.sNew[tn_col(sCol, sm.ecap, colg, e, lo)];
            const unsigned bal = __ballot_sync(0xffffffffu, nj >= 0);
            if (nj >= 0) {
                const int pos = w + __popc(bal & ((1u << lane) - 1u));
                col_out[base + pos] = olo + nj;
                if (pos < sm.ecap) sColN[pos] = nj;
            }
            w += __popc(bal);
        }
    }
}

// one layer of the forward pass; L is a RUN-TIME index and the three layers share one copy of the code: a CTA walks
// through every phase once, so what it waits for is largely instruction fetch (the three-times-unrolled kernel was 111 KB of
// SASS and every phase cost >= 1 us however small the subgraph) -- layers 2 and 3 now run out of the instruction cache
__device__ __forceinline__ void tn_fwd_layer(const npi_tiny_args_t& a, const int L, int g, const TnSmem& sm, int base, float* xs, float* ys, float* hs,
                                             float* pbuf, float& ro_max, float& ro_mean) {
    const int tid = threadIdx.x, hw = tid >> 4, l16 = tid & 15;
    const int lo = a.graph_ptr[L][g];
    const int n = min(a.graph_ptr[L][g + 1] - lo, sm.cap);
    const int olo = a.graph_ptr[L + 1][g];
    const int k = min(a.graph_ptr[L + 1][g + 1] - olo, n);
    int* const sRpC = (L & 1) ? sm.sRp[1] : sm.sRp[0];          // this layer's CSR / the next layer's (ping-pong)
    int* const sRpN = (L & 1) ? sm.sRp[0] : sm.sRp[1];
    int* const sColC = (L & 1) ? sm.sCol[1] : sm.sCol[0];
    int* const sColN = (L & 1) ? sm.sCol[0] : sm.sCol[1];
    const int Lm = L > 0 ? L - 1 : 0;
    const int32_t* colg = (L == 0 ? a.col0 : a.col_f[Lm]) + base;      // entry e of the subgraph at colg[e] (global row ids)
    if (L == 0) {
        // the subgraph's input CSR and node keys into shared memory: two dependent round trips for the whole CTA
        const int E = a.rowptr0[lo + n] - base;
        for (int i = tid; i <= n; i += TN_THREADS) sm.sRp[0][i] = a.rowptr0[lo + i] - base;
        for (int i = tid; i < n; i += TN_THREADS) sm.sGid[i] = a.gid[lo + i] | ((int)a.dist[lo + i] << 29);
        for (int e = tid; e < min(E, sm.ecap); e += TN_THREADS) sm.sCol[0][e] = a.col0[base + e] - lo;
        __syncthreads();
        TN_STAMP(a.dxa[0], 1 + 5 * L);
        tn_aggregate<true>(a, L, lo, n, sm, sRpC, sColC, colg, a.T, nullptr, hs);
    } else {
        tn_bar_wait(sm.bar, (uint32_t)(L - 1) & 1u);                           // conv(L+1).weight has landed in shared memory
        tn_project(a.xp[Lm], sm.W, a.y[L], lo, n, xs, true, ys, pbuf);
        if (tid == 0 && L == 1) tn_stage_weight(sm.W, a.weight[2], sm.bar);      // conv3.weight lands while this layer aggregates, sorts and gates
        TN_STAMP(a.dxa[0], 1 + 5 * L);
        tn_aggregate<false>(a, L, lo, n, sm, sRpC, sColC, colg, a.y[L], ys, hs);
    }
    __syncthreads();
    TN_STAMP(a.dxa[0], 2 + 5 * L);
    tn_topk(a, L, g, lo, n, olo, k, sm);
    TN_STAMP(a.dxa[0], 3 + 5 * L);
    // gating: x'_r = h[perm_r] * s[perm_r]; rows 0..15 also into the shared tile the next projection reads (zero padded)
    for (int r0 = 0; r0 < max(k, TN_TILE); r0 += TN_HW) {
        const int r = r0 + hw;
        if (r < k) {
            const int o = sm.sPerm[r];
            const float sv = sm.sS[o];
            const float* hr = o < TN_TILE ? hs + o * H : a.h[L] + (int64_t)(lo + o) * H;
            const float4 v0 = mul4(tn_ld4(hr + 4 * l16), sv), v1 = mul4(tn_ld4(hr + 64 + 4 * l16), sv);
            float* xr = a.xp[L] + (int64_t)(olo + r) * H;
            st4(xr + 4 * l16, v0); st4(xr + 64 + 4 * l16, v1);
            if (r < TN_TILE) { st4(xs + r * H + 4 * l16, v0); st4(xs + r * H + 64 + 4 * l16, v1); }
        } else if (r < TN_TILE) {
            st4(xs + r * H + 4 * l16, tn_zero4()); st4(xs + r * H + 64 + 4 * l16, tn_zero4());
        }
    }
    __syncthreads();
    TN_STAMP(a.dxa[0], 4 + 5 * L);
    // readout: column max (lowest row among equal maxima) and mean over the selected rows, in row order
    if (tid < H) {
        float m = -INFINITY, t = 0.f;
        int am = -1;
        const int ks = min(k, TN_TILE);
        for (int r = 0; r < ks; ++r) {
            const float v = xs[r * H + tid];
            if (v > m) { m = v; am = olo + r; }
            t += v;
        }
        for (int r = ks; r < k; r += 4) {                                        // beyond the shared tile: four loads in flight
            float v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) v[u] = r + u < k ? a.xp[L][(int64_t)(olo + r + u) * H + tid] : 0.f;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (r + u < k) {
                    if (v[u] > m) { m = v[u]; am = olo + r + u; }
                    t += v[u];
                }
            }
        }
        ro_max += m;
        ro_mean += t / (float)k;
        a.argmax[L][(int64_t)g * H + tid] = am;
    }
    if (L < 2) tn_filter(sm, sRpC, sColC, colg, lo, olo, k, base, sRpN, sColN,
                         a.rowptr_f[L] + olo + g, a.col_f[L]);
    __syncthreads();
    TN_STAMP(a.dxa[0], 5 + 5 * L);
}

__global__ void __launch_bounds__(TN_THREADS, 2) tiny_fwd_kernel(const __grid_constant__ npi_tiny_args_t a, int cap) {
    pdl_trigger();
    pdl_wait();
    extern __shared__ __align__(128) unsigned char tn_smem[];
    __shared__ __align__(16) float xs[TN_TILE * H], ys[TN_TILE * H], hs[TN_TILE * H], pbuf[8 * H];
    const TnSmem sm = tn_carve(tn_smem, cap);
    const int g = blockIdx.x;
    if (g >= a.B) return;
    TN_STAMP(a.dxa[0], 0);
    if (threadIdx.x == 0) tn_bar_init(sm.bar);
    __syncthreads();
    if (threadIdx.x == 0) tn_stage_weight(sm.W, a.weight[1], sm.bar);          // conv2.weight lands while layer 1 runs
    const int base = a.rowptr0[a.graph_ptr[0][g]];
    float ro_max = 0.f, ro_mean = 0.f;
#pragma unroll 1
    for (int L = 0; L < 3; ++L) tn_fwd_layer(a, L, g, sm, base, xs, ys, hs, pbuf, ro_max, ro_mean);
    if (threadIdx.x < H) {
        a.readout[(int64_t)g * 2 * H + threadIdx.x] = ro_max;                  // x1 + x2 + x3 (src/classes.py:74)
        a.readout[(int64_t)g * 2 * H + H + threadIdx.x] = ro_mean;
    }
}

// ------------------------------------------------------------------ backward
__device__ __forceinline__ void tn_bwd_layer(const npi_tiny_args_t& a, const int L, int g, const TnSmem& sm, int base, float* xs, float* ds, float* gs,
                                             float* pbuf, float (*sred)[H + 4], float (*sdb)[H]) {
    const int tid = threadIdx.x, hw = tid >> 4, l16 = tid & 15;
    const int c0 = 4 * l16, c1 = 64 + 4 * l16;
    const int lo = a.graph_ptr[L][g];
    const int n = min(a.graph_ptr[L][g + 1] - lo, sm.cap);
    const int olo = a.graph_ptr[L + 1][g];
    const int k = min(a.graph_ptr[L + 1][g + 1] - olo, n);
    const int Lm = L > 0 ? L - 1 : 0, Ld = L < 2 ? L : 0;
    const int32_t* rp = L == 0 ? a.rowptr0 + lo : a.rowptr_f[Lm] + lo + g;
    const int32_t* colg = (L == 0 ? a.col0 : a.col_f[Lm]) + base;
    int* sRp = sm.sRp[0];
    int* sCol = sm.sCol[0];
    // ---- everything index-like of this layer into shared memory (two dependent round trips for the whole CTA)
    {
        const int E = rp[n] - base;
        for (int i = tid; i < n; i += TN_THREADS) {
            const int r0 = rp[i], r1 = rp[i + 1];
            sRp[i] = r0 - base;
            if (i == n - 1) sRp[n] = r1 - base;
            sm.sInv[i] = 1.0f / (float)(r1 - r0 + 1);
            const int ni = a.new_id[L][lo + i];
            sm.sNew[i] = ni >= 0 ? ni - olo : -1;
            sm.sS[i] = a.s[L][lo + i];
            sm.sZ[i] = a.z[L][lo + i];
        }
        for (int r = tid; r < k; r += TN_THREADS) sm.sPerm[r] = a.perm[L][olo + r] - lo;
        for (int e = tid; e < min(E, sm.ecap); e += TN_THREADS) sCol[e] = colg[e] - lo;
    }
    __syncthreads();
    TN_STAMP(a.y[1], 1 + 5 * (2 - L));
    // ---- readout + gate + score + ReLU backward of the selected rows (the formulas of pool_bwd_kernel), a half-warp per row
    {
        const float4 p0 = ldg4(a.pool_w[L] + c0), p1 = ldg4(a.pool_w[L] + c1);
        const float norm = sqrtf(tn_half_sum(dot4(p0, p0) + dot4(p1, p1)));
        const float4 pn0 = make_float4(p0.x / norm, p0.y / norm, p0.z / norm, p0.w / norm);
        const float4 pn1 = make_float4(p1.x / norm, p1.y / norm, p1.z / norm, p1.w / norm);
        const float* dr = a.d_readout + (int64_t)g * 2 * H;
        const float4 gm0 = tn_ld4(dr + H + c0), gm1 = tn_ld4(dr + H + c1);
        const float4 gx0 = tn_ld4(dr + c0), gx1 = tn_ld4(dr + c1);
        const int4 am0 = *reinterpret_cast<const int4*>(a.argmax[L] + (int64_t)g * H + c0);
        const int4 am1 = *reinterpret_cast<const int4*>(a.argmax[L] + (int64_t)g * H + c1);
        const float kd = (float)k;
        float4 accA0 = tn_zero4(), accA1 = tn_zero4(), accB0 = tn_zero4(), accB1 = tn_zero4();
        float accS = 0.f;
        for (int r0 = 0; r0 < k; r0 += TN_HW) {
            if (r0 + (hw & ~1) >= k) continue;    // no selected row for either half of this warp
            const int r = r0 + hw;
            const bool valid = r < k;
            const int row = olo + r;
            const int o = valid ? sm.sPerm[r] : 0;
            const float sv = valid ? sm.sS[o] : 0.f, zv = valid ? sm.sZ[o] : 0.f;
            float4 x0 = tn_zero4(), x1 = tn_zero4(), h0 = tn_zero4(), h1 = tn_zero4();
            if (valid) {
                if (L < 2) {
                    const float* xr = r < TN_TILE ? gs + r * H : a.dxp[Ld] + (int64_t)row * H;
                    x0 = tn_ld4(xr + c0); x1 = tn_ld4(xr + c1);
                }
                const float* hr = a.h[L] + (int64_t)(lo + o) * H;
                h0 = tn_ld4(hr + c0); h1 = tn_ld4(hr + c1);
                x0.x += gm0.x / kd; x0.y += gm0.y / kd; x0.z += gm0.z / kd; x0.w += gm0.w / kd;
                x1.x += gm1.x / kd; x1.y += gm1.y / kd; x1.z += gm1.z / kd; x1.w += gm1.w / kd;
                if (am0.x == row) x0.x += gx0.x;
                if (am0.y == row) x0.y += gx0.y;
                if (am0.z == row) x0.z += gx0.z;
                if (am0.w == row) x0.w += gx0.w;
                if (am1.x == row) x1.x += gx1.x;
                if (am1.y == row) x1.y += gx1.y;
                if (am1.z == row) x1.z += gx1.z;
                if (am1.w == row) x1.w += gx1.w;
            }
            const float dsum = tn_half_sum(dot4(x0, h0) + dot4(x1, h1));
            if (valid) {
                const float dz = dsum * (1.f - sv * sv);
                float4 d0 = make_float4(x0.x * sv + dz * pn0.x, x0.y * sv + dz * pn0.y, x0.z * sv + dz * pn0.z, x0.w * sv + dz * pn0.w);
                float4 d1 = make_float4(x1.x * sv + dz * pn1.x, x1.y * sv + dz * pn1.y, x1.z * sv + dz * pn1.z, x1.w * sv + dz * pn1.w);
                d0.x = h0.x > 0.f ? d0.x : 0.f; d0.y = h0.y > 0.f ? d0.y : 0.f; d0.z = h0.z > 0.f ? d0.z : 0.f; d0.w = h0.w > 0.f ? d0.w : 0.f;
                d1.x = h1.x > 0.f ? d1.x : 0.f; d1.y = h1.y > 0.f ? d1.y : 0.f; d1.z = h1.z > 0.f ? d1.z : 0.f; d1.w = h1.w > 0.f ? d1.w : 0.f;
                float* dp = a.dpre[L] + (int64_t)row * H;
                st4(dp + c0, d0); st4(dp + c1, d1);
                if (r < TN_TILE) { st4(ds + r * H + c0, d0); st4(ds + r * H + c1, d1); }
                accB0 = add4(accB0, d0); accB1 = add4(accB1, d1);
                tn_fma4(accA0, h0, dz); tn_fma4(accA1, h1, dz);
                accS = fmaf(dz, zv, accS);
            }
        }
        // the two half-warps of a warp first (lower + upper), then the warps in order below
#define TN_XADD(v) v += __shfl_xor_sync(0xffffffffu, v, 16)
        TN_XADD(accA0.x); TN_XADD(accA0.y); TN_XADD(accA0.z); TN_XADD(accA0.w);
        TN_XADD(accA1.x); TN_XADD(accA1.y); TN_XADD(accA1.z); TN_XADD(accA1.w);
        TN_XADD(accB0.x); TN_XADD(accB0.y); TN_XADD(accB0.z); TN_XADD(accB0.w);
        TN_XADD(accB1.x); TN_XADD(accB1.y); TN_XADD(accB1.z); TN_XADD(accB1.w);
        TN_XADD(accS);
#undef TN_XADD
        if ((tid & 16) == 0) {
            const int warp = tid >> 5;
            st4(&sred[warp][c0], accA0); st4(&sred[warp][c1], accA1);
            st4(&sdb[warp][c0], accB0); st4(&sdb[warp][c1], accB1);
            if (l16 == 0) sred[warp][H] = accS;
        }
    }
    __syncthreads();
    TN_STAMP(a.y[1], 2 + 5 * (2 - L));
    {
        float* part = a.partials + ((int64_t)L * a.B + g) * TN_PART;
        if (tid <= H) {
            float t = 0.f;
#pragma unroll
            for (int w = 0; w < TN_WARPS; ++w) t += sred[w][tid];
            part[tid] = t;
        }
        if (tid < H) {
            float t = 0.f;
#pragma unroll
            for (int w = 0; w < TN_WARPS; ++w) t += sdb[w][tid];
            part[H + 4 + tid] = t;
        }
    }
    // ---- transposed aggregation: dxa_j = sum_{i in row(j) U {j}, selected} dpre[new_id[i]] / (deg_i + 1), a half-warp per row
    for (int j0 = 0; j0 < max(n, TN_TILE); j0 += TN_HW) {
        const int j = j0 + hw;
        if (j < n) {
            const int beg = sRp[j], end = sRp[j + 1];
            float4 acc0 = tn_zero4(), acc1 = tn_zero4();
            for (int e = beg; e < end; e += 4) {
                float4 v0[4], v1[4];
                float w[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    w[u] = 0.f;
                    v0[u] = tn_zero4(); v1[u] = tn_zero4();
                    if (e + u < end) {
                        const int i = tn_col(sCol, sm.ecap, colg, e + u, lo);
                        const int ni = sm.sNew[i];
                        if (ni >= 0) {
                            w[u] = sm.sInv[i];
                            const float* src = ni < TN_TILE ? ds + ni * H : a.dpre[L] + (int64_t)(olo + ni) * H;
                            v0[u] = tn_ld4(src + c0); v1[u] = tn_ld4(src + c1);
                        }
                    }
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    if (w[u] != 0.f) { tn_fma4(acc0, v0[u], w[u]); tn_fma4(acc1, v1[u], w[u]); }
                }
            }
            const int ns = sm.sNew[j];
            if (ns >= 0) {
                const float* src = ns < TN_TILE ? ds + ns * H : a.dpre[L] + (int64_t)(olo + ns) * H;
                const float w = sm.sInv[j];
                tn_fma4(acc0, tn_ld4(src + c0), w); tn_fma4(acc1, tn_ld4(src + c1), w);
            }
            float* out = a.dxa[L] + (int64_t)(lo + j) * H;
            st4(out + c0, acc0); st4(out + c1, acc1);
            if (L > 0 && j < TN_TILE) { st4(xs + j * H + c0, acc0); st4(xs + j * H + c1, acc1); }
        } else if (L > 0 && j < TN_TILE) {
            st4(xs + j * H + c0, tn_zero4()); st4(xs + j * H + c1, tn_zero4());
        }
    }
    __syncthreads();
    TN_STAMP(a.y[1], 3 + 5 * (2 - L));
    // ---- gradient of the pooled rows of the layer below: dX = DXA . W^T (weight_t = W^T in shared memory)
    if (L > 0) {
        tn_bar_wait(sm.bar, (uint32_t)(2 - L) & 1u);
        tn_project(a.dxa[L], sm.W, a.dxp[Lm], lo, n, xs, true, gs, pbuf);
        if (L == 2 && tid == 0) tn_stage_weight(sm.W, a.weight_t[1], sm.bar);   // conv2.weight^T lands while layer 2's backward runs
    }
    TN_STAMP(a.y[1], 4 + 5 * (2 - L));
}

__global__ void __launch_bounds__(TN_THREADS, 2) tiny_bwd_kernel(const __grid_constant__ npi_tiny_args_t a, int cap) {
    pdl_trigger();
    pdl_wait();
    extern __shared__ __align__(128) unsigned char tn_smem[];
    __shared__ __align__(16) float xs[TN_TILE * H], ds[TN_TILE * H], gs[TN_TILE * H], pbuf[8 * H];
    __shared__ __align__(16) float sred[TN_WARPS][H + 4];
    __shared__ __align__(16) float sdb[TN_WARPS][H];
    const TnSmem sm = tn_carve(tn_smem, cap);
    const int g = blockIdx.x;
    if (g >= a.B) return;
    TN_STAMP(a.y[1], 0);
    if (threadIdx.x == 0) tn_bar_init(sm.bar);
    __syncthreads();
    if (threadIdx.x == 0) tn_stage_weight(sm.W, a.weight_t[2], sm.bar);        // conv3.weight^T lands while layer 3's backward runs
    const int base = a.rowptr0[a.graph_ptr[0][g]];
#pragma unroll 1
    for (int L = 2; L >= 0; --L) tn_bwd_layer(a, L, g, sm, base, xs, ds, gs, pbuf, sred, sdb);
}

// d_pool_w / d_bias of the three layers from the per-subgraph partials, fixed order: grid (128/32 column blocks, 3 layers),
// 32 interleaved slices of the subgraph list summed in parallel, then the slices in order
constexpr int TR_SLICES = 32, TR_COLS = 32;
__global__ void __launch_bounds__(TR_SLICES * TR_COLS) tiny_reduce_kernel(const __grid_constant__ npi_tiny_args_t a) {
    __shared__ float sa[TR_SLICES][TR_COLS + 1], sb[TR_SLICES][TR_COLS + 1], ss[TR_SLICES];
    __shared__ float sS, sN;
    const int l = blockIdx.y;
    const int cl = threadIdx.x % TR_COLS, sl = threadIdx.x / TR_COLS;
    const int c = blockIdx.x * TR_COLS + cl;
    const float* partial = a.partials + (int64_t)l * a.B * TN_PART;
    const float* pw = a.pool_w[l];
    float sumA = 0.f, sumB = 0.f, t = 0.f;
    for (int g = sl; g < a.B; g += TR_SLICES) {
        const float* row = partial + (int64_t)g * TN_PART;
        sumA += row[c]; sumB += row[H + 4 + c];
        if (cl == 0) t += row[H];
    }
    sa[sl][cl] = sumA; sb[sl][cl] = sumB;
    if (cl == 0) ss[sl] = t;
    __syncthreads();
    if (threadIdx.x == 0) {
        float tt = 0.f;
        for (int q = 0; q < TR_SLICES; ++q) tt += ss[q];
        float nn = 0.f;
        for (int q = 0; q < H; ++q) nn = fmaf(pw[q], pw[q], nn);
        sS = tt; sN = nn;
    }
    __syncthreads();
    if (sl == 0) {
        float at = 0.f, bt = 0.f;
#pragma unroll
        for (int q = 0; q < TR_SLICES; ++q) { at += sa[q][cl]; bt += sb[q][cl]; }
        a.d_bias[l][c] = bt;
        // z = (h.w)/|w|  =>  dw = (sum dz h)/|w| - w (sum dz z)/|w|^2
        a.d_pool_w[l][c] = at / sqrtf(sN) - pw[c] * sS / sN;
    }
}

// out[m][c][k] = in_m[k][c] for the two 128 x 128 weights (conv2, conv3)
__global__ void __launch_bounds__(256) tiny_transpose_kernel(const float* w2, const float* w3, float* t2, float* t3) {
    __shared__ float tile[32][33];
    const float* in = blockIdx.z == 0 ? w2 : w3;
    float* out = blockIdx.z == 0 ? t2 : t3;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int k0 = blockIdx.y * 32, c0 = blockIdx.x * 32;
#pragma unroll
    for (int r = ty; r < 32; r += 8) tile[r][tx] = in[(k0 + r) * H + c0 + tx];
    __syncthreads();
#pragma unroll
    for (int r = ty; r < 32; r += 8) out[(c0 + r) * H + k0 + tx] = tile[tx][r];
}

// d conv1.weight [F,128] = sum_j x_j^T . dxa_j over the rows of the batch, x_j = [hop label | table[gid_j][1:F]] (the virtual
// input row of src/classes.py:706-717), in ONE launch.  For a small batch (3 k rows) this replaces the route through the
// feature table (by-node reduction of dxa, then table^T . G with per-CTA partials and a reduce: three dependent launches,
// ~30 us of the chain) -- and, in the same launch (grid.z = job), the dense weight gradients X^T . DXA of conv2 / conv3, whose
// tcgen05 route costs two launches each with a ~9 us floor for 1.6 k rows.  CTA = (8 feature rows of the result, one row range of the batch; the ranges per layer are dealt out on the host so that the launch is about one wave of two CTAs per SM
// and every CTA walks about the same number of rows): a warp walks rows, a lane owns
// four columns -- per row one 16-byte load of dxa and two broadcast loads of the table row feed 32 FMAs (a first version with a
// lane per column issued five loads for eight FMAs and ran at the instruction-issue limit of 36 SMs: 26 us).  The eight warps
// are combined in order through shared memory, the range's partial goes to the workspace, and the LAST CTA of a feature tile
// (ticket counter) adds the partials in range order: fixed summation order, no float atomics, bit-reproducible.
constexpr int WG_F = 8, WG_WARPS = 8, WG_SPLIT = 16, WG_UNROLL = 4, WG_JOBS = 3, WG_HEADER = 1024;      // WG_SPLIT: most row ranges per job
__host__ __device__ inline int wg_tiles(int F) { return (F + WG_F - 1) / WG_F; }
// one weight gradient out[F,128] = sum_j x_j^T . dxa_j: x_j = row j of a dense matrix (gid == nullptr) or the virtual input
// row [dist_j | table[gid_j][1:F]]
struct WgJob {
    const float* x; int ldx; int F;
    const int32_t* gid; const uint8_t* dist;
    const float* dxa; const int32_t* n_dev; int n_host;
    float* out; float* part; unsigned int* ticket;
    int splits;          // row ranges of this job (<= WG_SPLIT): chosen on the host so that every CTA of the launch walks about as many rows
};
struct WgJobs { WgJob job[WG_JOBS]; };

__global__ void __launch_bounds__(WG_WARPS * 32, 2) tiny_weight_grad_kernel(const __grid_constant__ WgJobs jobs) {
    pdl_trigger();
    pdl_wait();
    __shared__ __align__(16) float red[WG_WARPS][WG_F][H];
    __shared__ int s_last;
    const WgJob& jb = jobs.job[blockIdx.z];
    const int ft = blockIdx.x, f0 = ft * WG_F, sp = blockIdx.y;
    if (jb.out == nullptr || ft >= wg_tiles(jb.F) || sp >= jb.splits) return;
    const int n = dev_size(jb.n_dev, jb.n_host);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int chunk = (n + jb.splits - 1) / jb.splits;
    const int r0 = sp * chunk, r1 = min(n, r0 + chunk);
    const float* __restrict__ X = jb.x;
    const float* __restrict__ dxa = jb.dxa;
    const int32_t* __restrict__ gid = jb.gid;
    const int ld = jb.ldx;
    float4 acc[WG_F];
#pragma unroll
    for (int f = 0; f < WG_F; ++f) acc[f] = make_float4(0.f, 0.f, 0.f, 0.f);
    const bool two = f0 + 4 < ld;
    // a warp takes rows r0 + warp, + 8, + 16, ...; the row keys (global id, hop label) of its next 32 rows are fetched
    // lane-parallel and broadcast by shuffles, so the loop body is ONE round of independent loads (four rows in flight)
    for (int base = r0 + warp; base < r1; base += WG_WARPS * 32) {
        const int jl = base + WG_WARPS * lane;
        int rowl = jl, dl = 0;
        if (gid && jl < r1) { rowl = gid[jl]; dl = jb.dist[jl]; }
        for (int q = 0; q < 32 && base + WG_WARPS * q < r1; q += WG_UNROLL) {
            float4 xa[WG_UNROLL], xb[WG_UNROLL], g[WG_UNROLL];
#pragma unroll
            for (int u = 0; u < WG_UNROLL; ++u) {
                const int j = base + WG_WARPS * (q + u);
                const int row = __shfl_sync(0xffffffffu, rowl, (q + u) & 31);
                const int dd = __shfl_sync(0xffffffffu, dl, (q + u) & 31);
                xa[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                xb[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                g[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (j < r1) {
                    const float* tr = X + (int64_t)row * ld + f0;
                    xa[u] = tn_ld4(tr);
                    if (two) xb[u] = tn_ld4(tr + 4);
                    if (gid && f0 == 0) xa[u].x = (float)dd;
                    g[u] = tn_ld4(dxa + (int64_t)j * H + 4 * lane);
                }
            }
#pragma unroll
            for (int u = 0; u < WG_UNROLL; ++u) {
                tn_fma4(acc[0], g[u], xa[u].x); tn_fma4(acc[1], g[u], xa[u].y); tn_fma4(acc[2], g[u], xa[u].z); tn_fma4(acc[3], g[u], xa[u].w);
                tn_fma4(acc[4], g[u], xb[u].x); tn_fma4(acc[5], g[u], xb[u].y); tn_fma4(acc[6], g[u], xb[u].z); tn_fma4(acc[7], g[u], xb[u].w);
            }
        }
    }
#pragma unroll
    for (int f = 0; f < WG_F; ++f) st4(&red[warp][f][4 * lane], acc[f]);
    __syncthreads();
    const int f = tid >> 5;                                  // 256 threads = 8 feature rows x 32 column quads
    {
        float4 t = tn_ld4(&red[0][f][4 * lane]);
#pragma unroll
        for (int w = 1; w < WG_WARPS; ++w) t = add4(t, tn_ld4(&red[w][f][4 * lane]));
        st4(jb.part + (((int64_t)ft * WG_SPLIT + sp) * WG_F + f) * H + 4 * lane, t);
    }
    __threadfence();
    __syncthreads();
    if (tid == 0) s_last = (atomicAdd(&jb.ticket[ft], 1u) == (unsigned)jb.splits - 1u) ? 1 : 0;
    __syncthreads();
    if (s_last) {
        __threadfence();
        float4 t = __ldcg(reinterpret_cast<const float4*>(jb.part + (((int64_t)ft * WG_SPLIT) * WG_F + f) * H + 4 * lane));
#pragma unroll 4
        for (int q = 1; q < jb.splits; ++q)
            t = add4(t, __ldcg(reinterpret_cast<const float4*>(jb.part + (((int64_t)ft * WG_SPLIT + q) * WG_F + f) * H + 4 * lane)));
        if (f0 + f < jb.F) st4(jb.out + (int64_t)(f0 + f) * H + 4 * lane, t);
        if (tid == 0) jb.ticket[ft] = 0;                     // rewound for the next launch
    }
}

static int tn_cap(int max_graph_nodes) {
    int cap = 32;
    while (cap < max_graph_nodes) cap <<= 1;
    return cap;
}

}  // namespace npi

using namespace npi;

extern "C" int32_t npi_tiny_max_nodes(void) { return TN_MAX_NODES; }

extern "C" int64_t npi_tiny_partials_bytes(int32_t B) { return (int64_t)3 * (B > 0 ? B : 1) * TN_PART * sizeof(float); }

extern "C" int npi_tiny_transpose(const float* w2, const float* w3, float* w2_t, float* w3_t, npi_stream_t stream) {
    NPI_REQUIRE(w2 && w3 && w2_t && w3_t, "tiny_transpose: null argument");
    tiny_transpose_kernel<<<dim3(H / 32, H / 32, 2), 256, 0, (cudaStream_t)stream>>>(w2, w3, w2_t, w3_t);
    NPI_CHECK_LAUNCH();
    return NPI_OK;
}

static int tiny_check_common(const npi_tiny_args_t* a, const char* who) {
    NPI_REQUIRE(a, "%s: null argument", who);
    NPI_REQUIRE(a->max_graph_nodes >= 1 && a->max_graph_nodes <= TN_MAX_NODES, "%s: subgraphs of up to %d nodes exceed the per-CTA path (%d)",
                who, a->max_graph_nodes, TN_MAX_NODES);
    for (int l = 0; l < 4; ++l) NPI_REQUIRE(a->graph_ptr[l], "%s: null graph_ptr[%d]", who, l);
    NPI_REQUIRE(a->rowptr0 && a->col0 && a->rowptr_f[0] && a->rowptr_f[1] && a->col_f[0] && a->col_f[1], "%s: null adjacency", who);
    for (int l = 0; l < 3; ++l) {
        NPI_REQUIRE(a->pool_w[l] && a->h[l] && a->z[l] && a->s[l] && a->perm[l] && a->new_id[l] && a->argmax[l], "%s: null layer state (layer %d)", who, l);
    }
    return NPI_OK;
}

extern "C" int npi_tiny_fwd(const npi_tiny_args_t* a, npi_stream_t stream) {
    int rc = tiny_check_common(a, "tiny_fwd");
    if (rc != NPI_OK) return rc;
    NPI_REQUIRE(a->T && a->w_label && a->gid && a->dist && a->weight[1] && a->weight[2] && a->y[1] && a->y[2] && a->readout, "tiny_fwd: null argument");
    NPI_REQUIRE((((uintptr_t)a->weight[1] | (uintptr_t)a->weight[2]) & 15) == 0, "tiny_fwd: weights must be 16-byte aligned (bulk copy)");
    for (int l = 0; l < 3; ++l) NPI_REQUIRE(a->bias[l] && a->batch[l] && a->xp[l], "tiny_fwd: null layer output (layer %d)", l);
    if (a->B <= 0) return NPI_OK;
    const int cap = tn_cap(a->max_graph_nodes);
    static OncePerDevice cfg;
    if (cfg.need()) {
        NPI_CHECK_CUDA(cudaFuncSetAttribute(tiny_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tn_smem_bytes(TN_MAX_NODES)));
        NPI_CHECK_CUDA(cudaFuncSetAttribute(tiny_fwd_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    }
    NPI_CHECK_CUDA(launch_dep(tiny_fwd_kernel, a->B, TN_THREADS, tn_smem_bytes(cap), (cudaStream_t)stream, *a, cap));
    return NPI_OK;
}

extern "C" int npi_tiny_bwd(const npi_tiny_args_t* a, int32_t phases, npi_stream_t stream) {
    int rc = tiny_check_common(a, "tiny_bwd");
    if (rc != NPI_OK) return rc;
    NPI_REQUIRE(phases >= 0 && phases <= 2, "tiny_bwd: phases must be 0 (both), 1 (per-subgraph backward) or 2 (d_pool_w / d_bias)");
    NPI_REQUIRE(a->d_readout && a->weight_t[1] && a->weight_t[2] && a->dxp[0] && a->dxp[1] && a->partials, "tiny_bwd: null argument");
    NPI_REQUIRE((((uintptr_t)a->weight_t[1] | (uintptr_t)a->weight_t[2]) & 15) == 0, "tiny_bwd: transposed weights must be 16-byte aligned (bulk copy)");
    for (int l = 0; l < 3; ++l) NPI_REQUIRE(a->dpre[l] && a->dxa[l] && a->d_pool_w[l] && a->d_bias[l], "tiny_bwd: null gradient buffer (layer %d)", l);
    if (a->B <= 0) return NPI_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if (phases == 0 || phases == 1) {
        const int cap = tn_cap(a->max_graph_nodes);
        static OncePerDevice cfg;
        if (cfg.need()) {
            NPI_CHECK_CUDA(cudaFuncSetAttribute(tiny_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tn_smem_bytes(TN_MAX_NODES)));
        NPI_CHECK_CUDA(cudaFuncSetAttribute(tiny_bwd_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        }
        NPI_CHECK_CUDA(launch_dep(tiny_bwd_kernel, a->B, TN_THREADS, tn_smem_bytes(cap), st, *a, cap));
    }
    if (phases == 0 || phases == 2) {
        tiny_reduce_kernel<<<dim3(H / TR_COLS, 3), TR_SLICES * TR_COLS, 0, st>>>(*a);
        NPI_CHECK_LAUNCH();
    }
    return NPI_OK;
}

static int64_t wg_part_bytes(int F) { return (int64_t)wg_tiles(F > 0 ? F : 1) * WG_SPLIT * WG_F * H * sizeof(float); }

extern "C" int64_t npi_tiny_weight_grads_workspace_bytes(int32_t F) { return WG_HEADER + wg_part_bytes(F) + 2 * wg_part_bytes(H); }

/* workspace: npi_tiny_weight_grads_workspace_bytes(F) bytes whose first 1024 are ZERO before the first call (ticket
 * counters of the in-kernel reductions; every call leaves them zero) */
extern "C" int npi_tiny_weight_grads(const float* table, int32_t ld, int32_t F, const int32_t* gid, const uint8_t* dist,
                                     const float* dxa1, const int32_t* n0_dev, int32_t n0_host, float* d_weight1,
                                     const float* x1, const float* dxa2, const int32_t* n1_dev, int32_t n1_host, float* d_weight2,
                                     const float* x2, const float* dxa3, const int32_t* n2_dev, int32_t n2_host, float* d_weight3,
                                     void* workspace, int64_t workspace_bytes, npi_stream_t stream) {
    NPI_REQUIRE(table && gid && dist && dxa1 && d_weight1 && workspace, "tiny_weight_grads: null argument");
    NPI_REQUIRE((x1 == nullptr) == (d_weight2 == nullptr) && (x2 == nullptr) == (d_weight3 == nullptr) && (!x1 || dxa2) && (!x2 || dxa3),
                "tiny_weight_grads: x / dxa / d_weight of a dense layer come together");
    NPI_REQUIRE(F >= 1 && ld >= ((F + 3) / 4) * 4 && (ld & 3) == 0 && ((uintptr_t)table & 15) == 0,
                "tiny_weight_grads: the table needs 16-byte aligned rows of at least round_up(F, 4) columns");
    NPI_REQUIRE(wg_tiles(F) <= 64 && workspace_bytes >= npi_tiny_weight_grads_workspace_bytes(F) && ((uintptr_t)workspace & 15) == 0,
                "tiny_weight_grads: workspace too small or misaligned (F <= 512)");
    char* ws = (char*)workspace;
    unsigned int* tick = (unsigned int*)ws;
    WgJobs jobs;
    jobs.job[0] = WgJob{table, ld, F, gid, dist, dxa1, n0_dev, n0_host, d_weight1, (float*)(ws + WG_HEADER), tick, 1};
    jobs.job[1] = WgJob{x1, H, H, nullptr, nullptr, dxa2, n1_dev, n1_host, d_weight2, (float*)(ws + WG_HEADER + wg_part_bytes(F)), tick + 64, 1};
    jobs.job[2] = WgJob{x2, H, H, nullptr, nullptr, dxa3, n2_dev, n2_host, d_weight3,
                        (float*)(ws + WG_HEADER + wg_part_bytes(F) + wg_part_bytes(H)), tick + 128, 1};
    int tiles = wg_tiles(F);
    if ((x1 || x2) && tiles < wg_tiles(H)) tiles = wg_tiles(H);
    const int njobs = x2 ? 3 : (x1 ? 2 : 1);
    // row ranges per job: about two CTAs per SM in total, dealt out in proportion to rows x tiles, so that every CTA walks about
    // the same number of rows (with equal range counts the conv1 CTAs of a 3 k-row batch walked 57 rows per warp, conv3's 15)
    {
        double w[WG_JOBS], tot = 0.0;
        for (int k = 0; k < njobs; ++k) { w[k] = (double)(jobs.job[k].n_host > 0 ? jobs.job[k].n_host : 1) * wg_tiles(jobs.job[k].F); tot += w[k]; }
        const double budget = 2.0 * num_sms();
        int maxs = 1;
        for (int k = 0; k < njobs; ++k) {
            int sp = (int)(budget * w[k] / tot / wg_tiles(jobs.job[k].F) + 0.5);
            sp = sp < 1 ? 1 : (sp > WG_SPLIT ? WG_SPLIT : sp);
            jobs.job[k].splits = sp;
            if (sp > maxs) maxs = sp;
        }
        tiny_weight_grad_kernel<<<dim3(tiles, maxs, njobs), WG_WARPS * 32, 0, (cudaStream_t)stream>>>(jobs);
    }
    NPI_CHECK_LAUNCH();
    return NPI_OK;
}
