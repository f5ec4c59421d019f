// CSR segment-reduce kernels of SAGEConv (mean aggregation over neighbours U self) -- the
// HBM/L2-bound half of reference src/classes.py:62,66,70 (PyG SAGEConv propagate, SURVEY K2) and
// of its backward (the edge set is symmetric, so the transposed CSR is the CSR: atomic-free).
//
// Rows are short (mean degree 3-4, 62 % have ONE entry) with a heavy tail (hub proteins, > 1000
// entries; 30 % of all entries sit in rows longer than 16), and every element is a 512-byte feature
// row gathered out of L2.  A warp works on FOUR short rows at a time: lanes 8g..8g+7 own one row,
// fetch up to 8 of its CSR entries lane-parallel and then stream the source rows two at a time, each
// lane holding four float4 (16 of the 128 columns: column 32s + 4*l8 .. +3 for s = 0..3, so the 8
// lanes of a group read 128 contiguous bytes per load instruction).  The row itself rides as the
// last element of its entry stream (PyG appends the self loop last; one dependent round fewer).
//
// Rows with more than AG_HUB (= AG_SHORT = 16) entries are cut into SEGMENTS of AG_SEG = 32 entries,
// listed once per CSR when the CSR is produced (npi_hub_rows_build: next to the extraction /
// filter_adj, off the critical path).  The kernel that reduces the short rows deals the segments to
// its warps first (whole warp, one float4 per lane, 8 row loads in flight) and every warp leaves its
// partial sum in the queue; the warp that completes a row (per-row arrival counter) adds the
// partials IN SEGMENT ORDER, then the self row, and runs the epilogue.  Which warp does that is
// timing dependent, what it computes is not: results stay bit-reproducible, with no float atomics.
// Measured history (DESIGN.md 4): a CTA per hub row in a second launch left the GPU idle
// (profiles/r01p); 128-entry segments reached only the first third of the warps (r02e/r02f: 345 us
// over the six launches of a step vs 274 us with 32-entry segments, 2-3 per warp); a shared-memory
// ring with one accumulator per warp was 2-3x slower (r02b: the per-row epilogue dominates).
// Sums run in CSR order, then the self row (PyG appends the self loop last).
//
//  aggregate_fwd : h_i = act( (sum_{j in row(i) U {i}} y_j) / (deg_i+1) + b ),  y = x.W projected
//                  beforehand (gemm.cu); layer 1 reads y_j = T[gid_j] + label_j * W[0,:] from the
//                  projected feature table; epilogue also emits the TopKPooling score.
//  aggregate_bwd : dxa_j = sum_{i in row(j) U {j}, new_id[i] >= 0} dpre[new_id[i]] / (deg_i+1)
//  gid index / gid_reduce : layer-1 weight gradient through the feature table:
//                  G[v] = sum_{j : gid_j = v} dxa_j  (deterministic: per-v lists sorted by node id).
#include "hub.cuh"

namespace npi {

struct AggFwdArgs {
    const float* Y; const int32_t* gid; const uint8_t* dist; const float* w0;
    const int32_t* rowptr; const int32_t* col; const int32_t* n_dev; int n_host;
    const float* bias; int relu; const float* pool_w;
    float* h; float* z; float* s;
    int32_t* hubq;                               // hub queue of this CSR (npi_hub_rows_build)
    const int32_t* ent;                          // pipelined virtual layer: gid | dist << 29 per CSR entry (npi_entry_pack_virt)
    const int4* rows;                            // pipelined: rows binned by length class {row, beg, end, gid | dist << 29}
};

__device__ __forceinline__ void fma4(float4& acc, const float4& v, float w) {
    acc.x = fmaf(v.x, w, acc.x); acc.y = fmaf(v.y, w, acc.y); acc.z = fmaf(v.z, w, acc.z); acc.w = fmaf(v.w, w, acc.w);
}
__device__ __forceinline__ float4 lds4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ float4 ldcg4(const float* p) { return __ldcg(reinterpret_cast<const float4*>(p)); }

// Arrival of one finished part of a hub row; true for the warp that completes the row (it may then
// read every part: the writers fenced before arriving).
__device__ __forceinline__ bool hub_arrive(const HubQueue& hq, int base, int nseg, int lane) {
    __threadfence();
    __syncwarp();
    int last = 0;
    if (lane == 0) last = (atomicAdd(&hq.arrive[base], 1) == nseg - 1) ? 1 : 0;
    last = __shfl_sync(0xffffffffu, last, 0);
    if (last) __threadfence();
    return last != 0;
}

// sum of entries [k0, k1) of a CSR row by one warp (one float4 per lane, 8 row loads in flight)
template <bool VIRT>
__device__ __forceinline__ void fwd_span(const AggFwdArgs& a, int k0beg, int k1, int lane, float4& accl, int& dsl) {
    for (int k0 = k0beg; k0 < k1; k0 += 32) {
        const int k = k0 + lane;
        int j = 0;
        if (k < k1) {
            j = a.col[k];
            if (VIRT) { dsl += a.dist[j]; j = a.gid[j]; }
        }
        const int cnt = min(32, k1 - k0);
        int q = 0;
        for (; q + 8 <= cnt; q += 8) {
            float4 v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) v[u] = ldg4(a.Y + (int64_t)__shfl_sync(0xffffffffu, j, q + u) * H + 4 * lane);
#pragma unroll
            for (int u = 0; u < 8; ++u) accl = add4(accl, v[u]);
        }
        for (; q < cnt; ++q) accl = add4(accl, ldg4(a.Y + (int64_t)__shfl_sync(0xffffffffu, j, q) * H + 4 * lane));
    }
}

// self row, label column, mean, bias, ReLU, store, pooling score -- for a row summed by a whole warp
template <bool VIRT>
__device__ __forceinline__ void fwd_finish_row(const AggFwdArgs& a, int64_t ir, int js, int dsl, int deg, float4 accl, int lane,
                                               const float* s_b, const float* s_p, const float* s_w0, float norm) {
    accl = add4(accl, ldg4(a.Y + (int64_t)js * H + 4 * lane));                    // self loop last
    if (VIRT) fma4(accl, lds4(s_w0 + 4 * lane), (float)dsl);                       // label column (exact integer sum)
    const float dv = (float)(deg + 1);
    const float4 b = lds4(s_b + 4 * lane);
    float4 o = make_float4(accl.x / dv + b.x, accl.y / dv + b.y, accl.z / dv + b.z, accl.w / dv + b.w);
    if (a.relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
    st4(a.h + ir * H + 4 * lane, o);
    if (a.pool_w) {
        const float d = warp_sum(dot4(o, lds4(s_p + 4 * lane)));
        if (lane == 0) {
            const float zz = d / norm;
            if (a.z) a.z[ir] = zz;
            if (a.s) a.s[ir] = tanhf(zz) + 0.0f;
        }
    }
}

template <bool VIRT>
__global__ void __launch_bounds__(AG_THREADS, 3) aggregate_fwd_kernel(AggFwdArgs a) {
    __shared__ __align__(16) float s_b[H], s_p[H], s_w0[H];
    __shared__ float s_norm;
    const int n = dev_size(a.n_dev, a.n_host);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 3, l8 = lane & 7, gbase = lane & 24;
    if (tid < H) {
        s_b[tid] = a.bias ? a.bias[tid] : 0.f;
        s_p[tid] = a.pool_w ? a.pool_w[tid] : 0.f;
        s_w0[tid] = (VIRT && a.w0) ? a.w0[tid] : 0.f;
    }
    if (warp == 0) {
        float4 p = a.pool_w ? ldg4(a.pool_w + 4 * lane) : make_float4(0.f, 0.f, 0.f, 0.f);
        float nn = sqrtf(warp_sum(dot4(p, p)));
        if (lane == 0) s_norm = a.pool_w ? nn : 1.f;
    }
    __syncthreads();
    const float norm = s_norm;
    const int64_t warp0 = (int64_t)blockIdx.x * AG_WARPS + warp;
    const int64_t nwarps = (int64_t)gridDim.x * AG_WARPS;

    // ---- hub rows: one segment per warp, the warp that completes a row combines its parts
    {
        const HubQueue hq = hub_view(a.hubq, a.hubq[1]);
        const int nsegs = min(hq.hdr[0], a.hubq[1]);
        for (int64_t sidx = warp0; sidx < nsegs; sidx += nwarps) {
            const int i = hq.seg_row[sidx], base = hq.seg_base[sidx];
            const int rb = a.rowptr[i], re = a.rowptr[i + 1];
            const int nseg = (re - rb + AG_SEG - 1) / AG_SEG;
            const int sb = rb + ((int)sidx - base) * AG_SEG;
            float4 accl = make_float4(0.f, 0.f, 0.f, 0.f);
            int dsl = 0;
            fwd_span<VIRT>(a, sb, min(re, sb + AG_SEG), lane, accl, dsl);
            st4(hq.part + sidx * H + 4 * lane, accl);
            if (VIRT) {
                dsl = warp_sum_i(dsl);
                if (lane == 0) hq.dsum[sidx] = dsl;
            }
            if (!hub_arrive(hq, base, nseg, lane)) continue;
            float4 t = ldcg4(hq.part + (int64_t)base * H + 4 * lane);
            int ds = VIRT ? __ldcg(hq.dsum + base) : 0;
            for (int q = 1; q < nseg; ++q) {
                t = add4(t, ldcg4(hq.part + (int64_t)(base + q) * H + 4 * lane));
                if (VIRT) ds += __ldcg(hq.dsum + base + q);
            }
            if (lane == 0) hq.arrive[base] = 0;                    // rewound for the next launch on this queue
            int js = i;
            if (VIRT) { ds += a.dist[i]; js = a.gid[i]; }
            fwd_finish_row<VIRT>(a, i, js, ds, re - rb, t, lane, s_b, s_p, s_w0, norm);
        }
    }

    for (int64_t base = warp0 * 4; base < n; base += nwarps * 4) {
        const int64_t i = base + g;
        const bool valid = i < n;
        int beg = 0, end = 0, jself = 0, dself = 0;
        if (valid) {
            beg = a.rowptr[i]; end = a.rowptr[i + 1];
            if (VIRT) { jself = a.gid[i]; dself = a.dist[i]; } else jself = (int)i;
        }
        const bool is_long = (end - beg) > AG_SHORT;
        const bool is_hub = (end - beg) > AG_HUB;          // done above
        const int kend = is_long ? beg : end;
        // the self row rides as one more element behind the last entry (same summation order, one
        // dependent round of loads fewer per row: 62 % of the rows have a single entry)
        const int kx = (valid && !is_long) ? end + 1 : beg;
        float4 acc[4];
#pragma unroll
        for (int s = 0; s < 4; ++s) acc[s] = make_float4(0.f, 0.f, 0.f, 0.f);
        int dsum = 0;
        // ---- short rows: one 8-lane group per row
        for (int k0 = beg; __any_sync(0xffffffffu, k0 < kx); k0 += 8) {
            int j = 0;
            if (k0 + l8 < kend) {
                j = a.col[k0 + l8];
                if (VIRT) { dsum += a.dist[j]; j = a.gid[j]; }
            } else if (k0 + l8 < kx) j = jself;
            const int cnt = min(8, kx - k0);         // <= 0 for groups that are done
#pragma unroll
            for (int u = 0; u < 8; u += 2) {
                const int j0 = __shfl_sync(0xffffffffu, j, gbase | u);
                const int j1 = __shfl_sync(0xffffffffu, j, gbase | (u + 1));
                float4 v0[4], v1[4];
                if (u < cnt) {
#pragma unroll
                    for (int s = 0; s < 4; ++s) v0[s] = ldg4(a.Y + (int64_t)j0 * H + s * 32 + l8 * 4);
                }
                if (u + 1 < cnt) {
#pragma unroll
                    for (int s = 0; s < 4; ++s) v1[s] = ldg4(a.Y + (int64_t)j1 * H + s * 32 + l8 * 4);
                }
                if (u < cnt) {
#pragma unroll
                    for (int s = 0; s < 4; ++s) acc[s] = add4(acc[s], v0[s]);
                }
                if (u + 1 < cnt) {
#pragma unroll
                    for (int s = 0; s < 4; ++s) acc[s] = add4(acc[s], v1[s]);
                }
            }
        }
        {   // finish the short rows (shuffles are executed by all lanes, stores are predicated)
            const bool fin = valid && !is_long;
            if (VIRT) {
                dsum += __shfl_xor_sync(0xffffffffu, dsum, 1);
                dsum += __shfl_xor_sync(0xffffffffu, dsum, 2);
                dsum += __shfl_xor_sync(0xffffffffu, dsum, 4);
                dsum += dself;
            }
            float dotp = 0.f;
            if (fin) {
                const float ds = (float)dsum;
                const float dv = (float)(end - beg + 1);
#pragma unroll
                for (int s = 0; s < 4; ++s) {
                    const int c = s * 32 + l8 * 4;
                    float4 t = acc[s];                                                  // entries in CSR order, self row last
                    if (VIRT) fma4(t, lds4(s_w0 + c), ds);                              // label column (exact integer sum)
                    const float4 b = lds4(s_b + c);
                    float4 o = make_float4(t.x / dv + b.x, t.y / dv + b.y, t.z / dv + b.z, t.w / dv + b.w);
                    if (a.relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
                    st4(a.h + i * H + c, o);
                    dotp += dot4(o, lds4(s_p + c));
                }
            }
            if (a.pool_w) {
                dotp += __shfl_xor_sync(0xffffffffu, dotp, 1);
                dotp += __shfl_xor_sync(0xffffffffu, dotp, 2);
                dotp += __shfl_xor_sync(0xffffffffu, dotp, 4);
                if (fin && l8 == 0) {
                    const float zz = dotp / norm;
                    if (a.z) a.z[i] = zz;
                    if (a.s) a.s[i] = tanhf(zz) + 0.0f;
                }
            }
        }
        // ---- long rows: the whole warp on one row, one float4 per lane
        unsigned longmask = __ballot_sync(0xffffffffu, valid && is_long && !is_hub && l8 == 0);
        while (longmask) {
            const int src = __ffs(longmask) - 1;
            longmask &= longmask - 1;
            const int64_t ir = base + (src >> 3);
            const int rb = __shfl_sync(0xffffffffu, beg, src), re = __shfl_sync(0xffffffffu, end, src);
            const int js = __shfl_sync(0xffffffffu, jself, src);
            int dsl = 0;
            float4 accl = make_float4(0.f, 0.f, 0.f, 0.f);
            fwd_span<VIRT>(a, rb, re, lane, accl, dsl);
            if (VIRT) dsl = warp_sum_i(dsl) + __shfl_sync(0xffffffffu, dself, src);
            fwd_finish_row<VIRT>(a, ir, js, dsl, re - rb, accl, lane, s_b, s_p, s_w0, norm);
        }
    }
}

struct AggBwdArgs {
    const float* dpre; const int32_t* new_id; const int32_t* rowptr; const int32_t* col;
    const int32_t* n_dev; int n_host; float* dxa;
    int32_t* hubq;
    const int2* sel;                             // pipelined variant: {new_id[col], 1/(deg_col+1) bits} per CSR entry (npi_entry_pack_sel)
    const int4* rows;                            // pipelined: rows binned by length class (npi_hub_rows_build)
    int no_self;                                 // pipelined: rows have no self term (CSR by global id, npi_ctx_gid_reduce)
};

// weighted sum over entries [k0, k1) of a CSR row by one warp: sum_i dpre[new_id[i]] / (deg_i + 1)
__device__ __forceinline__ void bwd_span(const AggBwdArgs& a, int k0beg, int k1, int lane, float4& accl) {
    for (int k0 = k0beg; k0 < k1; k0 += 32) {
        const int k = k0 + lane;
        int id = -1;
        float inv = 0.f;
        if (k < k1) {
            const int i = a.col[k];
            id = a.new_id ? a.new_id[i] : i;
            if (id >= 0) inv = 1.0f / (float)(a.rowptr[i + 1] - a.rowptr[i] + 1);
        }
        const int cnt = min(32, k1 - k0);
        for (int q = 0; q < cnt; q += 8) {
            float4 v[8]; float w[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int idu = __shfl_sync(0xffffffffu, id, (q + u) & 31);
                w[u] = __shfl_sync(0xffffffffu, inv, (q + u) & 31);
                if (q + u < cnt && idu >= 0) v[u] = ldg4(a.dpre + (int64_t)idu * H + 4 * lane);
                else { v[u] = make_float4(0.f, 0.f, 0.f, 0.f); w[u] = 0.f; }
            }
#pragma unroll
            for (int u = 0; u < 8; ++u)
                if (w[u] != 0.f) fma4(accl, v[u], w[u]);
        }
    }
}

__global__ void __launch_bounds__(AG_THREADS, 3) aggregate_bwd_kernel(AggBwdArgs a) {
    const int n = dev_size(a.n_dev, a.n_host);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 3, l8 = lane & 7, gbase = lane & 24;
    const int64_t warp0 = (int64_t)blockIdx.x * AG_WARPS + warp;
    const int64_t nwarps = (int64_t)gridDim.x * AG_WARPS;

    {   // ---- hub rows by segments (see the header)
        const HubQueue hq = hub_view(a.hubq, a.hubq[1]);
        const int nsegs = min(hq.hdr[0], a.hubq[1]);
        for (int64_t sidx = warp0; sidx < nsegs; sidx += nwarps) {
            const int jr = hq.seg_row[sidx], base = hq.seg_base[sidx];
            const int rb = a.rowptr[jr], re = a.rowptr[jr + 1];
            const int nseg = (re - rb + AG_SEG - 1) / AG_SEG;
            const int sb = rb + ((int)sidx - base) * AG_SEG;
            float4 accl = make_float4(0.f, 0.f, 0.f, 0.f);
            bwd_span(a, sb, min(re, sb + AG_SEG), lane, accl);
            st4(hq.part + sidx * H + 4 * lane, accl);
            if (!hub_arrive(hq, base, nseg, lane)) continue;
            float4 t = ldcg4(hq.part + (int64_t)base * H + 4 * lane);
            for (int q = 1; q < nseg; ++q) t = add4(t, ldcg4(hq.part + (int64_t)(base + q) * H + 4 * lane));
            if (lane == 0) hq.arrive[base] = 0;
            const int ids = a.new_id ? a.new_id[jr] : jr;
            if (ids >= 0) fma4(t, ldg4(a.dpre + (int64_t)ids * H + 4 * lane), 1.0f / (float)(re - rb + 1));
            st4(a.dxa + (int64_t)jr * H + 4 * lane, t);
        }
    }

    for (int64_t base = warp0 * 4; base < n; base += nwarps * 4) {
        const int64_t jrow = base + g;
        const bool valid = jrow < n;
        int beg = 0, end = 0, idself = -1;
        if (valid) {
            beg = a.rowptr[jrow]; end = a.rowptr[jrow + 1];
            idself = a.new_id ? a.new_id[jrow] : (int)jrow;
        }
        const bool is_long = (end - beg) > AG_SHORT;
        const bool is_hub = (end - beg) > AG_HUB;          // done above
        const int kend = is_long ? beg : end;
        const int kx = (valid && !is_long) ? end + 1 : beg;      // entries + the row itself as last element
        float4 acc[4];
#pragma unroll
        for (int s = 0; s < 4; ++s) acc[s] = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int k0 = beg; __any_sync(0xffffffffu, k0 < kx); k0 += 8) {
            int id = -1;
            float inv = 0.f;
            if (k0 + l8 < kend) {
                const int i = a.col[k0 + l8];
                id = a.new_id ? a.new_id[i] : i;
                if (id >= 0) inv = 1.0f / (float)(a.rowptr[i + 1] - a.rowptr[i] + 1);
            } else if (k0 + l8 < kx) {
                id = idself;
                if (id >= 0) inv = 1.0f / (float)(end - beg + 1);
            }
#pragma unroll
            for (int u = 0; u < 8; u += 2) {
                const int id0 = __shfl_sync(0xffffffffu, id, gbase | u);
                const int id1 = __shfl_sync(0xffffffffu, id, gbase | (u + 1));
                const float w0 = __shfl_sync(0xffffffffu, inv, gbase | u);
                const float w1 = __shfl_sync(0xffffffffu, inv, gbase | (u + 1));
                float4 v0[4], v1[4];
                if (id0 >= 0) {
#pragma unroll
                    for (int s = 0; s < 4; ++s) v0[s] = ldg4(a.dpre + (int64_t)id0 * H + s * 32 + l8 * 4);
                }
                if (id1 >= 0) {
#pragma unroll
                    for (int s = 0; s < 4; ++s) v1[s] = ldg4(a.dpre + (int64_t)id1 * H + s * 32 + l8 * 4);
                }
                if (id0 >= 0) {
#pragma unroll
                    for (int s = 0; s < 4; ++s) fma4(acc[s], v0[s], w0);
                }
                if (id1 >= 0) {
#pragma unroll
                    for (int s = 0; s < 4; ++s) fma4(acc[s], v1[s], w1);
                }
            }
        }
        if (valid && !is_long) {
#pragma unroll
            for (int s = 0; s < 4; ++s) st4(a.dxa + jrow * H + s * 32 + l8 * 4, acc[s]);
        }
        unsigned longmask = __ballot_sync(0xffffffffu, valid && is_long && !is_hub && l8 == 0);
        while (longmask) {
            const int src = __ffs(longmask) - 1;
            longmask &= longmask - 1;
            const int64_t jr = base + (src >> 3);
            const int rb = __shfl_sync(0xffffffffu, beg, src), re = __shfl_sync(0xffffffffu, end, src);
            const int ids = __shfl_sync(0xffffffffu, idself, src);
            float4 accl = make_float4(0.f, 0.f, 0.f, 0.f);
            bwd_span(a, rb, re, lane, accl);
            if (ids >= 0) fma4(accl, ldg4(a.dpre + (int64_t)ids * H + 4 * lane), 1.0f / (float)(re - rb + 1));
            st4(a.dxa + jr * H + 4 * lane, accl);
        }
    }
}

// =====================================================================================================
// Pipelined variants (the ones the engine launches).
//  * Short rows are taken in LENGTH-CLASS ORDER (rows[] of npi_hub_rows_build, a counting sort by the
//    number of load rounds a row needs): the four groups of a warp run in lock step, so with rows in
//    index order a warp waited for its longest row (3.2 rounds per iteration on average instead of
//    1.75); a row record {row, beg, end, self} is one coalesced 16-byte load.
//  * The per-entry indirections are resolved ONCE per CSR, off the critical path, into a packed entry
//    stream in CSR order (npi_entry_pack_virt: gid | dist << 29 next to the extraction;
//    npi_entry_pack_sel: {new_id[col], 1/(deg_col+1)} next to filter_adj), so an entry costs one
//    coalesced load instead of three gathers.
//  * The row loop is software pipelined: row records are fetched two iterations ahead and the first
//    eight packed entries of every row one iteration ahead, so they arrive while the current rows'
//    feature loads are in flight.  (Deeper pipelines / L1 prefetches only added spills: r02g.)
// Every row is summed in exactly the order of the kernels above (results are bit-identical; the test
// suite compares the two).
constexpr int PK_SHIFT = 29;
constexpr int PK_MASK = (1 << PK_SHIFT) - 1;
#ifndef AG_PIPE_CTAS
#define AG_PIPE_CTAS 3
#endif

template <bool VIRT>
__device__ __forceinline__ void fwd_span_p(const AggFwdArgs& a, const int32_t* __restrict__ ent, int k0beg, int k1, int lane,
                                           float4& accl, int& dsl) {
    int jn = (k0beg + lane < k1) ? ent[k0beg + lane] : 0;
    for (int k0 = k0beg; k0 < k1; k0 += 32) {
        int j = jn;
        jn = 0;
        if (k0 + 32 + lane < k1) jn = ent[k0 + 32 + lane];      // next 32 entries while this chunk streams
        if (VIRT) { dsl += (int)((unsigned)j >> PK_SHIFT); j &= PK_MASK; }      // lanes past k1 hold 0
        const int cnt = min(32, k1 - k0);
        int q = 0;
        for (; q + 8 <= cnt; q += 8) {
            float4 v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) v[u] = ldg4(a.Y + (int64_t)__shfl_sync(0xffffffffu, j, q + u) * H + 4 * lane);
#pragma unroll
            for (int u = 0; u < 8; ++u) accl = add4(accl, v[u]);
        }
        for (; q < cnt; ++q) accl = add4(accl, ldg4(a.Y + (int64_t)__shfl_sync(0xffffffffu, j, q) * H + 4 * lane));
    }
}

template <bool VIRT>
__global__ void __launch_bounds__(AG_THREADS, AG_PIPE_CTAS) aggregate_fwd_pipe_kernel(AggFwdArgs a) {
    __shared__ __align__(16) float s_b[H], s_p[H], s_w0[H];
    __shared__ float s_norm;
    pdl_trigger();                                   // the weights below were written in an earlier step: before the wait
    const int n = dev_size(a.n_dev, a.n_host);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 3, l8 = lane & 7, gbase = lane & 24;
    const int32_t* __restrict__ ent = VIRT ? a.ent : a.col;
    if (tid < H) {
        s_b[tid] = a.bias ? a.bias[tid] : 0.f;
        s_p[tid] = a.pool_w ? a.pool_w[tid] : 0.f;
        s_w0[tid] = (VIRT && a.w0) ? a.w0[tid] : 0.f;
    }
    if (warp == 0) {
        float4 p = a.pool_w ? ldg4(a.pool_w + 4 * lane) : make_float4(0.f, 0.f, 0.f, 0.f);
        float nn = sqrtf(warp_sum(dot4(p, p)));
        if (lane == 0) s_norm = a.pool_w ? nn : 1.f;
    }
    __syncthreads();
    pdl_wait();
    const float norm = s_norm;
    const int64_t warp0 = (int64_t)blockIdx.x * AG_WARPS + warp;
    const int64_t nwarps = (int64_t)gridDim.x * AG_WARPS;

    // ---- hub rows: one segment per warp, the warp that completes a row combines its parts
    {
        const HubQueue hq = hub_view(a.hubq, a.hubq[1]);
        const int nsegs = min(hq.hdr[0], a.hubq[1]);
        for (int64_t sidx = warp0; sidx < nsegs; sidx += nwarps) {
            const int i = hq.seg_row[sidx], base = hq.seg_base[sidx];
            const int rb = a.rowptr[i], re = a.rowptr[i + 1];
            const int nseg = (re - rb + AG_SEG - 1) / AG_SEG;
            const int sb = rb + ((int)sidx - base) * AG_SEG;
            float4 accl = make_float4(0.f, 0.f, 0.f, 0.f);
            int dsl = 0;
            fwd_span_p<VIRT>(a, ent, sb, min(re, sb + AG_SEG), lane, accl, dsl);
            st4(hq.part + sidx * H + 4 * lane, accl);
            if (VIRT) {
                dsl = warp_sum_i(dsl);
                if (lane == 0) hq.dsum[sidx] = dsl;
            }
            if (!hub_arrive(hq, base, nseg, lane)) continue;
            float4 t = ldcg4(hq.part + (int64_t)base * H + 4 * lane);
            int ds = VIRT ? __ldcg(hq.dsum + base) : 0;
            for (int q = 1; q < nseg; ++q) {
                t = add4(t, ldcg4(hq.part + (int64_t)(base + q) * H + 4 * lane));
                if (VIRT) ds += __ldcg(hq.dsum + base + q);
            }
            if (lane == 0) hq.arrive[base] = 0;                    // rewound for the next launch on this queue
            int js = i;
            if (VIRT) { ds += a.dist[i]; js = a.gid[i]; }
            fwd_finish_row<VIRT>(a, i, js, ds, re - rb, t, lane, s_b, s_p, s_w0, norm);
        }
    }

    // ---- regular rows in length-class order (rows[] of npi_hub_rows_build: the four rows of a warp need
    // the same number of load rounds), software pipelined: the row records of iterations t+1 / t+2 and
    // the first eight entries of iteration t+1 are in registers while iteration t streams its rows
    const int32_t* hdr = a.hubq;
    int n_short = 0;
#pragma unroll
    for (int cc = 0; cc < 6; ++cc) n_short += hdr[HQ_CLS + cc];
    const int n_long = hdr[HQ_CLS + 6];
    const int4* __restrict__ rows = a.rows;

    // whole-warp rows (AG_SHORT+1 .. AG_HUB entries; none at the shipped AG_HUB = AG_SHORT = 16) first, one per
    // warp: the warps that get one start their share of the short rows a little later instead of finishing alone
    for (int64_t idx = n_short + warp0; idx < (int64_t)n_short + n_long; idx += nwarps) {
        const int4 R = rows[idx];
        int dsl = 0;
        float4 accl = make_float4(0.f, 0.f, 0.f, 0.f);
        fwd_span_p<VIRT>(a, ent, R.y, R.z, lane, accl, dsl);
        int js = R.x;
        if (VIRT) { dsl = warp_sum_i(dsl) + (int)((unsigned)R.w >> PK_SHIFT); js = R.w & PK_MASK; }
        fwd_finish_row<VIRT>(a, R.x, js, dsl, R.z - R.y, accl, lane, s_b, s_p, s_w0, norm);
    }

    const int64_t stride = nwarps * 4;
    int64_t base = warp0 * 4;
    const int4 RZ = make_int4(0, 0, 0, 0);
    int4 RA = RZ, RB = RZ;
    if (base + g < n_short) RA = rows[base + g];
    if (base + stride + g < n_short) RB = rows[base + stride + g];
    int entA = 0;
    if (l8 < RA.z - RA.y) entA = ent[RA.y + l8];
    for (; base < n_short; base += stride) {
        int4 RC = RZ;
        if (base + 2 * stride + g < n_short) RC = rows[base + 2 * stride + g];
        int entB = 0;
        if (l8 < RB.z - RB.y) entB = ent[RB.y + l8];

        const bool valid = base + g < n_short;
        const int64_t i = RA.x;
        const int beg = RA.y, end = RA.z;
        const int jself = VIRT ? (RA.w & PK_MASK) : RA.x;
        const int dself = VIRT ? (int)((unsigned)RA.w >> PK_SHIFT) : 0;
        const int kend = end;
        const int kx = valid ? end + 1 : beg;                    // entries + the self row as last element
        float4 acc[4];
#pragma unroll
        for (int s = 0; s < 4; ++s) acc[s] = make_float4(0.f, 0.f, 0.f, 0.f);
        int dsum = 0;
        int round = 0;
        for (int k0 = beg; __any_sync(0xffffffffu, k0 < kx); k0 += 8, ++round) {
            int j = 0;
            if (k0 + l8 < kend) {
                int e = (round == 0) ? entA : ent[k0 + l8];
                if (VIRT) { dsum += (int)((unsigned)e >> PK_SHIFT); e &= PK_MASK; }
                j = e;
            } else if (k0 + l8 < kx) j = jself;
            const int cnt = min(8, kx - k0);         // <= 0 for groups that are done
#pragma unroll
            for (int u = 0; u < 8; u += 2) {
                const int j0 = __shfl_sync(0xffffffffu, j, gbase | u);
                const int j1 = __shfl_sync(0xffffffffu, j, gbase | (u + 1));
                float4 v0[4], v1[4];
                if (u < cnt) {
#pragma unroll
                    for (int s = 0; s < 4; ++s) v0[s] = ldg4(a.Y + (int64_t)j0 * H + s * 32 + l8 * 4);
                }
                if (u + 1 < cnt) {
#pragma unroll
                    for (int s = 0; s < 4; ++s) v1[s] = ldg4(a.Y + (int64_t)j1 * H + s * 32 + l8 * 4);
                }
                if (u < cnt) {
#pragma unroll
                    for (int s = 0; s < 4; ++s) acc[s] = add4(acc[s], v0[s]);
                }
                if (u + 1 < cnt) {
#pragma unroll
                    for (int s = 0; s < 4; ++s) acc[s] = add4(acc[s], v1[s]);
                }
            }
        }
        {   // finish (shuffles are executed by all lanes, stores are predicated)
            if (VIRT) {
                dsum += __shfl_xor_sync(0xffffffffu, dsum, 1);
                dsum += __shfl_xor_sync(0xffffffffu, dsum, 2);
                dsum += __shfl_xor_sync(0xffffffffu, dsum, 4);
                dsum += dself;
            }
            float dotp = 0.f;
            if (valid) {
                const float ds = (float)dsum;
                const float dv = (float)(end - beg + 1);
#pragma unroll
                for (int s = 0; s < 4; ++s) {
                    const int c = s * 32 + l8 * 4;
                    float4 t = acc[s];                                                  // entries in CSR order, self row last
                    if (VIRT) fma4(t, lds4(s_w0 + c), ds);                              // label column (exact integer sum)
                    const float4 b = lds4(s_b + c);
                    float4 o = make_float4(t.x / dv + b.x, t.y / dv + b.y, t.z / dv + b.z, t.w / dv + b.w);
                    if (a.relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
                    st4(a.h + i * H + c, o);
                    dotp += dot4(o, lds4(s_p + c));
                }
            }
            if (a.pool_w) {
                dotp += __shfl_xor_sync(0xffffffffu, dotp, 1);
                dotp += __shfl_xor_sync(0xffffffffu, dotp, 2);
                dotp += __shfl_xor_sync(0xffffffffu, dotp, 4);
                if (valid && l8 == 0) {
                    const float zz = dotp / norm;
                    if (a.z) a.z[i] = zz;
                    if (a.s) a.s[i] = tanhf(zz) + 0.0f;
                }
            }
        }
        RA = RB; RB = RC; entA = entB;
    }
}

// weighted sum over packed entries [k0, k1) of a CSR row by one warp
__device__ __forceinline__ void bwd_span_p(const AggBwdArgs& a, const int2* __restrict__ sel, int k0beg, int k1, int lane, float4& accl) {
    int2 pn = make_int2(-1, 0);
    if (k0beg + lane < k1) pn = sel[k0beg + lane];
    for (int k0 = k0beg; k0 < k1; k0 += 32) {
        const int id = pn.x;
        const float inv = __int_as_float(pn.y);
        pn = make_int2(-1, 0);
        if (k0 + 32 + lane < k1) pn = sel[k0 + 32 + lane];
        const int cnt = min(32, k1 - k0);
        for (int q = 0; q < cnt; q += 8) {
            float4 v[8]; float w[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int idu = __shfl_sync(0xffffffffu, id, (q + u) & 31);
                w[u] = __shfl_sync(0xffffffffu, inv, (q + u) & 31);
                if (q + u < cnt && idu >= 0) v[u] = ldg4(a.dpre + (int64_t)idu * H + 4 * lane);
                else { v[u] = make_float4(0.f, 0.f, 0.f, 0.f); w[u] = 0.f; }
            }
#pragma unroll
            for (int u = 0; u < 8; ++u)
                if (w[u] != 0.f) fma4(accl, v[u], w[u]);
        }
    }
}

__global__ void __launch_bounds__(AG_THREADS, AG_PIPE_CTAS) aggregate_bwd_pipe_kernel(AggBwdArgs a) {
    pdl_trigger();
    pdl_wait();
    const int n = dev_size(a.n_dev, a.n_host);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 3, l8 = lane & 7, gbase = lane & 24;
    const int64_t warp0 = (int64_t)blockIdx.x * AG_WARPS + warp;
    const int64_t nwarps = (int64_t)gridDim.x * AG_WARPS;
    const int2* __restrict__ sel = a.sel;

    {   // ---- hub rows by segments (see the header)
        const HubQueue hq = hub_view(a.hubq, a.hubq[1]);
        const int nsegs = min(hq.hdr[0], a.hubq[1]);
        for (int64_t sidx = warp0; sidx < nsegs; sidx += nwarps) {
            const int jr = hq.seg_row[sidx], base = hq.seg_base[sidx];
            const int rb = a.rowptr[jr], re = a.rowptr[jr + 1];
            const int nseg = (re - rb + AG_SEG - 1) / AG_SEG;
            const int sb = rb + ((int)sidx - base) * AG_SEG;
            float4 accl = make_float4(0.f, 0.f, 0.f, 0.f);
            bwd_span_p(a, sel, sb, min(re, sb + AG_SEG), lane, accl);
            st4(hq.part + sidx * H + 4 * lane, accl);
            if (a.no_self && nseg > 2 * HUB_GRP) {
                // Rows of the CSR by node are LONG (a hub protein occurs in thousands of contexts: hundreds of
                // segments), and one warp adding 300 partials in sequence was the length of the whole kernel.  Two
                // levels: the warp that completes a GROUP of HUB_GRP consecutive segments folds them into the group's
                // first slot (in segment order), then arrives at the row; the warp that completes the row adds the
                // group sums in group order.  Fixed order, no atomics on floats; group counters live in the arrival
                // slots behind the row's own (a row of nseg segments owns nseg slots) and are rewound like it.
                const int part_i = (int)sidx - base, grp = part_i / HUB_GRP;
                const int ngrp = (nseg + HUB_GRP - 1) / HUB_GRP, gsize = min(HUB_GRP, nseg - grp * HUB_GRP);
                __threadfence();
                __syncwarp();
                int lastg = 0;
                if (lane == 0) lastg = (atomicAdd(&hq.arrive[base + 1 + grp], 1) == gsize - 1) ? 1 : 0;
                lastg = __shfl_sync(0xffffffffu, lastg, 0);
                if (!lastg) continue;
                __threadfence();
                const int64_t g0 = (int64_t)base + (int64_t)grp * HUB_GRP;
                float4 pv[HUB_GRP];
#pragma unroll
                for (int u = 0; u < HUB_GRP; ++u) pv[u] = (u < gsize) ? ldcg4(hq.part + (g0 + u) * H + 4 * lane) : make_float4(0.f, 0.f, 0.f, 0.f);
                float4 tg = pv[0];
#pragma unroll
                for (int u = 1; u < HUB_GRP; ++u) if (u < gsize) tg = add4(tg, pv[u]);
                st4(hq.part + g0 * H + 4 * lane, tg);
                if (lane == 0) hq.arrive[base + 1 + grp] = 0;
                if (!hub_arrive(hq, base, ngrp, lane)) continue;
                float4 t = ldcg4(hq.part + (int64_t)base * H + 4 * lane);
                int q = 1;
                for (; q + 4 <= ngrp; q += 4) {
                    float4 pw[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u) pw[u] = ldcg4(hq.part + ((int64_t)base + (int64_t)(q + u) * HUB_GRP) * H + 4 * lane);
#pragma unroll
                    for (int u = 0; u < 4; ++u) t = add4(t, pw[u]);
                }
                for (; q < ngrp; ++q) t = add4(t, ldcg4(hq.part + ((int64_t)base + (int64_t)q * HUB_GRP) * H + 4 * lane));
                if (lane == 0) hq.arrive[base] = 0;
                st4(a.dxa + (int64_t)jr * H + 4 * lane, t);
                continue;
            }
            if (!hub_arrive(hq, base, nseg, lane)) continue;
            float4 t = ldcg4(hq.part + (int64_t)base * H + 4 * lane);
            int q = 1;
            for (; q + 4 <= nseg; q += 4) {                        // four partials in flight, added in segment order (a node of the
                float4 pv[4];                                      // graph occurs in thousands of contexts: hundreds of parts per row)
#pragma unroll
                for (int u = 0; u < 4; ++u) pv[u] = ldcg4(hq.part + (int64_t)(base + q + u) * H + 4 * lane);
#pragma unroll
                for (int u = 0; u < 4; ++u) t = add4(t, pv[u]);
            }
            for (; q < nseg; ++q) t = add4(t, ldcg4(hq.part + (int64_t)(base + q) * H + 4 * lane));
            if (lane == 0) hq.arrive[base] = 0;
            const int ids = a.no_self ? -1 : (a.new_id ? a.new_id[jr] : jr);
            if (ids >= 0) fma4(t, ldg4(a.dpre + (int64_t)ids * H + 4 * lane), 1.0f / (float)(re - rb + 1));
            st4(a.dxa + (int64_t)jr * H + 4 * lane, t);
        }
    }

    const int32_t* hdr = a.hubq;
    int n_short = 0;
#pragma unroll
    for (int cc = 0; cc < 6; ++cc) n_short += hdr[HQ_CLS + cc];
    const int n_long = hdr[HQ_CLS + 6];
    const int4* __restrict__ rows = a.rows;

    for (int64_t idx = n_short + warp0; idx < (int64_t)n_short + n_long; idx += nwarps) {      // whole-warp rows (class 6)
        const int4 R = rows[idx];
        const int ids = a.no_self ? -1 : (a.new_id ? a.new_id[R.x] : R.x);
        float4 accl = make_float4(0.f, 0.f, 0.f, 0.f);
        bwd_span_p(a, sel, R.y, R.z, lane, accl);
        if (ids >= 0) fma4(accl, ldg4(a.dpre + (int64_t)ids * H + 4 * lane), 1.0f / (float)(R.z - R.y + 1));
        st4(a.dxa + (int64_t)R.x * H + 4 * lane, accl);
    }

    const int64_t stride = nwarps * 4;
    int64_t base = warp0 * 4;
    const int4 RZ = make_int4(0, 0, 0, 0);
    int4 RA = RZ, RB = RZ;
    if (base + g < n_short) RA = rows[base + g];
    if (base + stride + g < n_short) RB = rows[base + stride + g];
    int idsA = -1;
    if (base + g < n_short && !a.no_self) idsA = a.new_id ? a.new_id[RA.x] : RA.x;
    int2 entA = make_int2(-1, 0);
    if (l8 < RA.z - RA.y) entA = sel[RA.y + l8];
    for (; base < n_short; base += stride) {
        int4 RC = RZ;
        if (base + 2 * stride + g < n_short) RC = rows[base + 2 * stride + g];
        int2 entB = make_int2(-1, 0);
        if (l8 < RB.z - RB.y) entB = sel[RB.y + l8];
        int idsB = -1;
        if (base + stride + g < n_short && !a.no_self) idsB = a.new_id ? a.new_id[RB.x] : RB.x;

        const bool valid = base + g < n_short;
        const int64_t jrow = RA.x;
        const int beg = RA.y, end = RA.z, idself = idsA;
        const int kend = end;
        const int kx = valid ? end + 1 : beg;                    // entries + the row itself as last element
        float4 acc[4];
#pragma unroll
        for (int s = 0; s < 4; ++s) acc[s] = make_float4(0.f, 0.f, 0.f, 0.f);
        int round = 0;
        for (int k0 = beg; __any_sync(0xffffffffu, k0 < kx); k0 += 8, ++round) {
            int id = -1;
            float inv = 0.f;
            if (k0 + l8 < kend) {
                const int2 p = (round == 0) ? entA : sel[k0 + l8];
                id = p.x; inv = __int_as_float(p.y);
            } else if (k0 + l8 < kx) {
                id = idself;
                if (id >= 0) inv = 1.0f / (float)(end - beg + 1);
            }
#pragma unroll
            for (int u = 0; u < 8; u += 2) {
                const int id0 = __shfl_sync(0xffffffffu, id, gbase | u);
                const int id1 = __shfl_sync(0xffffffffu, id, gbase | (u + 1));
                const float w0 = __shfl_sync(0xffffffffu, inv, gbase | u);
                const float w1 = __shfl_sync(0xffffffffu, inv, gbase | (u + 1));
                float4 v0[4], v1[4];
                if (id0 >= 0) {
#pragma unroll
                    for (int s = 0; s < 4; ++s) v0[s] = ldg4(a.dpre + (int64_t)id0 * H + s * 32 + l8 * 4);
                }
                if (id1 >= 0) {
#pragma unroll
                    for (int s = 0; s < 4; ++s) v1[s] = ldg4(a.dpre + (int64_t)id1 * H + s * 32 + l8 * 4);
                }
                if (id0 >= 0) {
#pragma unroll
                    for (int s = 0; s < 4; ++s) fma4(acc[s], v0[s], w0);
                }
                if (id1 >= 0) {
#pragma unroll
                    for (int s = 0; s < 4; ++s) fma4(acc[s], v1[s], w1);
                }
            }
        }
        if (valid) {
#pragma unroll
            for (int s = 0; s < 4; ++s) st4(a.dxa + jrow * H + s * 32 + l8 * 4, acc[s]);
        }
        RA = RB; RB = RC; entA = entB; idsA = idsB;
    }
}

// ---- packed entry streams (one thread per CSR entry; E = rowptr[n] read on the device)
__global__ void entry_pack_virt_kernel(const int32_t* rowptr, const int32_t* col, const int32_t* gid, const uint8_t* dist,
                                       const int32_t* n_dev, int n_host, int64_t e_max, int32_t* out) {
    const int n = dev_size(n_dev, n_host);
    const int64_t E = min((int64_t)rowptr[n], e_max);
    for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < E; k += (int64_t)gridDim.x * blockDim.x) {
        const int j = col[k];
        out[k] = gid[j] | ((int)dist[j] << PK_SHIFT);
    }
}

__global__ void entry_pack_sel_kernel(const int32_t* rowptr, const int32_t* col, const int32_t* new_id, const int32_t* n_dev,
                                      int n_host, int64_t e_max, int2* out) {
    const int n = dev_size(n_dev, n_host);
    const int64_t E = min((int64_t)rowptr[n], e_max);
    for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < E; k += (int64_t)gridDim.x * blockDim.x) {
        const int i = col[k];
        const int id = new_id ? new_id[i] : i;
        const float inv = id >= 0 ? 1.0f / (float)(rowptr[i + 1] - rowptr[i] + 1) : 0.f;
        out[k] = make_int2(id, __float_as_int(inv));
    }
}

// ---- hub queue of a CSR: every row with more than AG_HUB entries reserves ceil(L/AG_SEG) consecutive
// segment slots (slot order is timing dependent and irrelevant: rows are independent)
// keep != nullptr: only rows with keep[i] == i are listed (the representatives of csrc/ctx.cu)
__global__ void __launch_bounds__(256) hub_scan_kernel(const int32_t* rowptr, const int32_t* n_dev, int n_host, int32_t* buf, int cap,
                                                       const int32_t* __restrict__ keep) {
    __shared__ int hist[N_CLS];
    const int n = dev_size(n_dev, n_host);
    const HubQueue hq = hub_view(buf, cap);
    if (threadIdx.x < N_CLS) hist[threadIdx.x] = 0;
    __syncthreads();
    if (blockIdx.x == 0 && threadIdx.x == 0) hq.hdr[1] = cap;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        if (keep && keep[i] != (int)i) continue;
        hub_list_row(hq, cap, hist, (int)i, rowptr[i + 1] - rowptr[i]);
    }
    __syncthreads();
    if (threadIdx.x < N_CLS && hist[threadIdx.x]) atomicAdd(&hq.hdr[HQ_CLS + threadIdx.x], hist[threadIdx.x]);
}

// Rows binned by length class (a counting sort on the class totals of hub_scan_kernel): a CTA owns
// ROF_ROWS consecutive rows, reserves one range per class with a single atomic each and places its
// rows.  The order inside a class depends on timing and is irrelevant: rows are independent, a
// row's sum never depends on which rows share its warp.  rows[pos] = {row, beg, end, self payload}.
constexpr int ROF_ROWS = 1024;
__global__ void __launch_bounds__(256) row_order_fill_kernel(const int32_t* rowptr, const int32_t* n_dev, int n_host, const int32_t* gid,
                                                             const uint8_t* dist, int32_t* buf, int cap, int4* rows,
                                                             const int32_t* __restrict__ keep) {
    __shared__ int hist[N_CLS], start[N_CLS];
    const int n = dev_size(n_dev, n_host);
    const HubQueue hq = hub_view(buf, cap);
    if (threadIdx.x < N_CLS) hist[threadIdx.x] = 0;
    __syncthreads();
    const int64_t r0 = (int64_t)blockIdx.x * ROF_ROWS;
    int cls[ROF_ROWS / 256], rank[ROF_ROWS / 256], beg[ROF_ROWS / 256], end[ROF_ROWS / 256];
#pragma unroll
    for (int q = 0; q < ROF_ROWS / 256; ++q) {
        const int64_t i = r0 + q * 256 + threadIdx.x;
        cls[q] = -1;
        if (i < n && (!keep || keep[i] == (int)i)) {
            beg[q] = rowptr[i]; end[q] = rowptr[i + 1];
            cls[q] = row_class(end[q] - beg[q]);
            rank[q] = atomicAdd(&hist[cls[q]], 1);
        }
    }
    __syncthreads();
    if (threadIdx.x < N_CLS) {
        int base = 0;
        for (int c = 0; c < (int)threadIdx.x; ++c) base += hq.hdr[HQ_CLS + c];
        start[threadIdx.x] = base + (hist[threadIdx.x] ? atomicAdd(&hq.hdr[HQ_CUR + threadIdx.x], hist[threadIdx.x]) : 0);
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < ROF_ROWS / 256; ++q) {
        const int64_t i = r0 + q * 256 + threadIdx.x;
        if (cls[q] >= 0 && cls[q] < N_CLS - 1) {          // hub rows are not listed here (segments)
            const int self = gid ? (gid[i] | ((int)dist[i] << 29)) : (int)i;
            rows[start[cls[q]] + rank[q]] = make_int4((int)i, beg[q], end[q], self);
        }
    }
}

// ------------------------------------------------------------------ occurrence lists by global id
__global__ void gid_count_kernel(const int32_t* gid, const int32_t* n_dev, int n_host, int32_t* cnt) {
    const int n = dev_size(n_dev, n_host);
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        atomicAdd(&cnt[gid[i]], 1);
}

__global__ void __launch_bounds__(1024) gid_scan_kernel(const int32_t* cnt, int V, int32_t* occ_ptr) {
    __shared__ int sh[1024 / 32 + 2];
    int run = 0;
    for (int c = 0; c < V; c += 1024) {
        int i = c + threadIdx.x;
        int v = (i < V) ? cnt[i] : 0;
        int tot;
        int ex = block_excl_scan<1024>(v, sh, &tot);
        if (i < V) occ_ptr[i] = run + ex;
        run += tot;
    }
    if (threadIdx.x == 0) occ_ptr[V] = run;
}

__global__ void gid_fill_kernel(const int32_t* gid, const int32_t* n_dev, int n_host, const int32_t* occ_ptr, int32_t* cursor,
                                int32_t* occ_tmp) {
    const int n = dev_size(n_dev, n_host);
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        int v = gid[i];
        occ_tmp[occ_ptr[v] + atomicAdd(&cursor[v], 1)] = (int)i;
    }
}

// the atomic cursor scrambles the order inside a list; restore ascending node id by rank counting
__global__ void __launch_bounds__(256) gid_sort_kernel(int V, const int32_t* occ_ptr, const int32_t* occ_tmp, int32_t* occ_node) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t v = warp0; v < V; v += nwarps) {
        const int beg = occ_ptr[v], end = occ_ptr[v + 1];
        for (int k = beg + lane; k < end; k += 32) {
            int me = occ_tmp[k], rank = 0;
            for (int q = beg; q < end; ++q) rank += (occ_tmp[q] < me);
            occ_node[beg + rank] = me;
        }
    }
}

// One CTA per occurrence list (persistent over v): the 8 warps take the list's rows interleaved,
// four independent row loads in flight each, and their sums are combined in warp order -- hub
// nodes that occur in every subgraph of the batch no longer serialise on one warp.
constexpr int GR_CTAS_PER_SM = 4;
#ifndef NPI_GR_SHORT
#define NPI_GR_SHORT 16
#endif
constexpr int GR_SHORT = NPI_GR_SHORT;          // lists up to this length are summed by one warp
__global__ void __launch_bounds__(AG_THREADS) gid_reduce_kernel(const float* dxa, const uint8_t* dist, const int32_t* occ_ptr,
                                                                const int32_t* occ_node, int V, float* G, float* label_part) {
    __shared__ __align__(16) float sred[AG_WARPS][H];
    __shared__ int s_list[AG_THREADS];
    __shared__ int s_scan[AG_THREADS / 32 + 2];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float4 lab = make_float4(0.f, 0.f, 0.f, 0.f);
    // The CTA owns v = blockIdx.x + k * gridDim.x.  Nodes that do not occur in the batch (most of a large graph:
    // at 508 k nodes and 512 subgraphs the walk over EMPTY lists, two block barriers each, took 0.8 of 1.07 ms --
    // gpurun_out/r2l) are found AG_THREADS at a time: their rows of G are zeroed warp-cooperatively, the occupied
    // ones are compacted in ascending order (same order as before: the label-row sum stays bit-identical).
    for (int k0 = 0; (int64_t)blockIdx.x + (int64_t)k0 * gridDim.x < V; k0 += AG_THREADS) {
        const int64_t vq = (int64_t)blockIdx.x + (int64_t)(k0 + (int)threadIdx.x) * gridDim.x;
        const bool in = vq < V;
        const bool ne = in && occ_ptr[vq + 1] > occ_ptr[vq];
        unsigned me = __ballot_sync(0xffffffffu, in && !ne);
        while (me) {
            const int b = __ffs(me) - 1;
            me &= me - 1;
            const int64_t vv = (int64_t)blockIdx.x + (int64_t)(k0 + warp * 32 + b) * gridDim.x;
            st4(G + vv * H + 4 * lane, make_float4(0.f, 0.f, 0.f, 0.f));
        }
        int tot;
        const int pos = block_excl_scan<AG_THREADS>(ne ? 1 : 0, s_scan, &tot);
        if (ne) s_list[pos] = (int)vq;
        __syncthreads();
        // short lists (most nodes of a large graph occur in a handful of subgraphs: 3.7 on average at 508 k nodes /
        // 512 subgraphs, where one CTA per list spent 1 ms on block barriers): ONE WARP per list, eight lists of the
        // CTA in flight, four row loads each, no barrier; the assignment (list q -> warp q % 8) is fixed, so sums
        // stay deterministic
        for (int q = warp; q < tot; q += AG_WARPS) {
            const int v = s_list[q];
            const int beg = occ_ptr[v], end = occ_ptr[v + 1];
            if (end - beg > GR_SHORT) continue;
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
            int k = beg;
            for (; k + 3 < end; k += 4) {
                int j[4]; float d[4]; float4 x[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) j[u] = occ_node[k + u];
#pragma unroll
                for (int u = 0; u < 4; ++u) { d[u] = (float)dist[j[u]]; x[u] = ldg4(dxa + (int64_t)j[u] * H + 4 * lane); }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    acc = add4(acc, x[u]);
                    lab.x = fmaf(d[u], x[u].x, lab.x); lab.y = fmaf(d[u], x[u].y, lab.y);
                    lab.z = fmaf(d[u], x[u].z, lab.z); lab.w = fmaf(d[u], x[u].w, lab.w);
                }
            }
            for (; k < end; ++k) {
                const int j = occ_node[k];
                const float d = (float)dist[j];
                const float4 x = ldg4(dxa + (int64_t)j * H + 4 * lane);
                acc = add4(acc, x);
                lab.x = fmaf(d, x.x, lab.x); lab.y = fmaf(d, x.y, lab.y);
                lab.z = fmaf(d, x.z, lab.z); lab.w = fmaf(d, x.w, lab.w);
            }
            st4(G + (int64_t)v * H + 4 * lane, acc);
        }
        for (int q = 0; q < tot; ++q) {
            const int v = s_list[q];
            const int beg = occ_ptr[v], end = occ_ptr[v + 1];
            if (end - beg <= GR_SHORT) continue;              // uniform over the CTA
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
            int k = beg + warp;
            for (; k + 3 * AG_WARPS < end; k += 4 * AG_WARPS) {
                int j[4]; float d[4]; float4 x[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) j[u] = occ_node[k + u * AG_WARPS];
#pragma unroll
                for (int u = 0; u < 4; ++u) { d[u] = (float)dist[j[u]]; x[u] = ldg4(dxa + (int64_t)j[u] * H + 4 * lane); }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    acc = add4(acc, x[u]);
                    lab.x = fmaf(d[u], x[u].x, lab.x); lab.y = fmaf(d[u], x[u].y, lab.y);
                    lab.z = fmaf(d[u], x[u].z, lab.z); lab.w = fmaf(d[u], x[u].w, lab.w);
                }
            }
            for (; k < end; k += AG_WARPS) {
                const int j = occ_node[k];
                const float d = (float)dist[j];
                const float4 x = ldg4(dxa + (int64_t)j * H + 4 * lane);
                acc = add4(acc, x);
                lab.x = fmaf(d, x.x, lab.x); lab.y = fmaf(d, x.y, lab.y);
                lab.z = fmaf(d, x.z, lab.z); lab.w = fmaf(d, x.w, lab.w);
            }
            st4(&sred[warp][4 * lane], acc);
            __syncthreads();
            if (threadIdx.x < H) {
                float t = 0.f;
#pragma unroll
                for (int w = 0; w < AG_WARPS; ++w) t += sred[w][threadIdx.x];
                G[(int64_t)v * H + threadIdx.x] = t;
            }
            __syncthreads();
        }
        __syncthreads();
    }
    st4(&sred[warp][4 * lane], lab);
    __syncthreads();
    if (threadIdx.x < H) {
        float t = 0.f;
#pragma unroll
        for (int w = 0; w < AG_WARPS; ++w) t += sred[w][threadIdx.x];
        label_part[(int64_t)blockIdx.x * H + threadIdx.x] = t;
    }
}

static int gid_reduce_grid() { return num_sms() * GR_CTAS_PER_SM; }

}  // namespace npi

using namespace npi;

extern "C" int64_t npi_hub_rows_bytes(int64_t e_max) {
    const int64_t cap = hub_cap(e_max);
    return (HUB_HDR + 4 * cap) * 4 + cap * H * 4;
}

extern "C" int npi_hub_rows_reset(int32_t* hub_queue, npi_stream_t stream) {
    NPI_REQUIRE(hub_queue, "hub_rows_reset: null argument");
    NPI_CHECK_CUDA(cudaMemsetAsync(hub_queue, 0, sizeof(int32_t) * HUB_HDR, (cudaStream_t)stream));
    return NPI_OK;
}

extern "C" int npi_hub_rows_build(const int32_t* rowptr, const int32_t* n_dev, int32_t n_host, int64_t e_max,
                                  int32_t* hub_queue, int64_t hub_queue_bytes, const int32_t* gid, const uint8_t* dist,
                                  void* row_order, const int32_t* keep, npi_stream_t stream) {
    NPI_REQUIRE(rowptr && hub_queue, "hub_rows_build: null argument");
    NPI_REQUIRE(hub_queue_bytes >= npi_hub_rows_bytes(e_max), "hub_rows_build: queue too small for %lld entries", (long long)e_max);
    NPI_REQUIRE((gid == nullptr) == (dist == nullptr), "hub_rows_build: gid and dist come together");
    NPI_REQUIRE(((uintptr_t)row_order & 15) == 0, "hub_rows_build: row_order must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    NPI_CHECK_CUDA(cudaMemsetAsync(hub_queue, 0, sizeof(int32_t) * HUB_HDR, st));
    int grid = (n_host + 255) / 256;
    if (grid > grid_for(4)) grid = grid_for(4);
    hub_scan_kernel<<<grid > 0 ? grid : 1, 256, 0, st>>>(rowptr, n_dev, n_host, hub_queue, hub_cap(e_max), keep);
    NPI_CHECK_LAUNCH();
    if (row_order) {
        const int g2 = (n_host + ROF_ROWS - 1) / ROF_ROWS;
        row_order_fill_kernel<<<g2 > 0 ? g2 : 1, 256, 0, st>>>(rowptr, n_dev, n_host, gid, dist, hub_queue, hub_cap(e_max), (int4*)row_order, keep);
        NPI_CHECK_LAUNCH();
    }
    return NPI_OK;
}

static int agg_grid(int n_host) {
    int grid = grid_for(3);
    int need = (n_host + 4 * AG_WARPS - 1) / (4 * AG_WARPS);
    if (need < grid) grid = need > 0 ? need : 1;
    return grid;
}

extern "C" int npi_entry_pack_virt(const int32_t* rowptr, const int32_t* col, const int32_t* gid, const uint8_t* dist,
                                   const int32_t* n_dev, int32_t n_host, int32_t V, int64_t e_max, int32_t* packed,
                                   npi_stream_t stream) {
    NPI_REQUIRE(rowptr && col && gid && dist && packed, "entry_pack_virt: null argument");
    NPI_REQUIRE(V > 0 && V <= PK_MASK, "entry_pack_virt: %d graph nodes do not fit the 29-bit id field", V);
    int grid = (int)((e_max + 255) / 256);
    if (grid > grid_for(8)) grid = grid_for(8);
    entry_pack_virt_kernel<<<grid > 0 ? grid : 1, 256, 0, (cudaStream_t)stream>>>(rowptr, col, gid, dist, n_dev, n_host, e_max, packed);
    NPI_CHECK_LAUNCH();
    return NPI_OK;
}

extern "C" int npi_entry_pack_sel(const int32_t* rowptr, const int32_t* col, const int32_t* new_id, const int32_t* n_dev,
                                  int32_t n_host, int64_t e_max, void* packed, npi_stream_t stream) {
    NPI_REQUIRE(rowptr && col && packed, "entry_pack_sel: null argument");
    NPI_REQUIRE(((uintptr_t)packed & 7) == 0, "entry_pack_sel: packed must be 8-byte aligned");
    int grid = (int)((e_max + 255) / 256);
    if (grid > grid_for(8)) grid = grid_for(8);
    entry_pack_sel_kernel<<<grid > 0 ? grid : 1, 256, 0, (cudaStream_t)stream>>>(rowptr, col, new_id, n_dev, n_host, e_max, (int2*)packed);
    NPI_CHECK_LAUNCH();
    return NPI_OK;
}

static int agg_pipe_grid(int n_host) {
    int grid = grid_for(AG_PIPE_CTAS);
    int need = (n_host + 4 * AG_WARPS - 1) / (4 * AG_WARPS);
    if (need < grid) grid = need > 0 ? need : 1;
    return grid;
}

extern "C" int npi_sage_aggregate_fwd(const float* Y, const int32_t* gid, const uint8_t* dist, const float* w0,
                                      const int32_t* rowptr, const int32_t* col, const int32_t* n_dev, int32_t n_host,
                                      const float* bias, int32_t relu, const float* pool_w,
                                      float* h, float* z, float* s, int32_t* hub_queue, const int32_t* packed,
                                      const void* row_order, int32_t pipelined, npi_stream_t stream) {
    NPI_REQUIRE(Y && rowptr && col && h && hub_queue, "sage_aggregate_fwd: null argument");
    NPI_REQUIRE((gid == nullptr) == (dist == nullptr), "sage_aggregate_fwd: gid and dist come together");
    NPI_REQUIRE(!(pipelined && gid) || packed, "sage_aggregate_fwd: the pipelined virtual layer needs the packed entries");
    NPI_REQUIRE(!pipelined || row_order, "sage_aggregate_fwd: the pipelined kernel needs the binned row order of npi_hub_rows_build");
    NPI_REQUIRE(((uintptr_t)row_order & 15) == 0 && ((uintptr_t)packed & 3) == 0,
                "sage_aggregate_fwd: row_order must be 16-byte and packed 4-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    AggFwdArgs a{Y, gid, dist, w0, rowptr, col, n_dev, n_host, bias, relu, pool_w, h, z, s, hub_queue, packed, (const int4*)row_order};
    if (pipelined) {
        const int grid = agg_pipe_grid(n_host);
        if (gid) NPI_CHECK_CUDA(launch_dep(aggregate_fwd_pipe_kernel<true>, grid, AG_THREADS, 0, st, a));
        else NPI_CHECK_CUDA(launch_dep(aggregate_fwd_pipe_kernel<false>, grid, AG_THREADS, 0, st, a));
    } else {
        const int grid = agg_grid(n_host);
        if (gid) aggregate_fwd_kernel<true><<<grid, AG_THREADS, 0, st>>>(a);
        else aggregate_fwd_kernel<false><<<grid, AG_THREADS, 0, st>>>(a);
    }
    NPI_CHECK_LAUNCH();
    return NPI_OK;
}

extern "C" int npi_sage_aggregate_bwd(const float* dpre, const int32_t* new_id, const int32_t* rowptr, const int32_t* col,
                                      const int32_t* n_dev, int32_t n_host, float* dxa,
                                      int32_t* hub_queue, const void* packed, const void* row_order, npi_stream_t stream) {
    NPI_REQUIRE(dpre && rowptr && col && dxa && hub_queue, "sage_aggregate_bwd: null argument");
    NPI_REQUIRE(!packed || row_order, "sage_aggregate_bwd: the pipelined kernel needs the binned row order of npi_hub_rows_build");
    NPI_REQUIRE(((uintptr_t)row_order & 15) == 0 && ((uintptr_t)packed & 7) == 0,
                "sage_aggregate_bwd: row_order must be 16-byte and packed 8-byte aligned");
    AggBwdArgs a{dpre, new_id, rowptr, col, n_dev, n_host, dxa, hub_queue, (const int2*)packed, (const int4*)row_order, 0};
    if (packed) NPI_CHECK_CUDA(launch_dep(aggregate_bwd_pipe_kernel, agg_pipe_grid(n_host), AG_THREADS, 0, (cudaStream_t)stream, a));
    else aggregate_bwd_kernel<<<agg_grid(n_host), AG_THREADS, 0, (cudaStream_t)stream>>>(a);
    NPI_CHECK_LAUNCH();
    return NPI_OK;
}

extern "C" int npi_csr_gather_sum(const float* src, const int32_t* rowptr, const void* packed, int32_t n_rows, float* out,
                                  int32_t* hub_queue, const void* row_order, npi_stream_t stream) {
    NPI_REQUIRE(src && rowptr && packed && out && hub_queue && row_order && n_rows > 0, "csr_gather_sum: bad argument");
    NPI_REQUIRE(((uintptr_t)row_order & 15) == 0 && ((uintptr_t)packed & 7) == 0,
                "csr_gather_sum: row_order must be 16-byte and packed 8-byte aligned");
    AggBwdArgs a{src, nullptr, rowptr, nullptr, nullptr, n_rows, out, hub_queue, (const int2*)packed, (const int4*)row_order, 1};
    // the per-context backward of conv1 uses it on CSRs whose work sits in a few long rows (a node of the graph occurs
    // in ~100 contexts of a batch) as well as on the class CSR: the grid is the full machine whatever n_rows is
    NPI_CHECK_CUDA(launch_dep(aggregate_bwd_pipe_kernel, grid_for(AG_PIPE_CTAS), AG_THREADS, 0, (cudaStream_t)stream, a));
    NPI_CHECK_LAUNCH();
    return NPI_OK;
}

extern "C" int64_t npi_gid_index_workspace_bytes(int32_t V, int32_t n_max) {
    return (2 * (int64_t)(V + 1) + (int64_t)n_max + 4 + 4100) * 4;
}

extern "C" int npi_gid_index_build(const int32_t* gid, const int32_t* n_dev, int32_t n_host, int32_t V,
                                   int32_t* occ_ptr, int32_t* occ_node, void* workspace, int64_t workspace_bytes,
                                   npi_stream_t stream) {
    NPI_REQUIRE(gid && occ_ptr && occ_node && workspace && V > 0, "gid_index_build: bad argument");
    NPI_REQUIRE(workspace_bytes >= npi_gid_index_workspace_bytes(V, n_host), "gid_index_build: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    int32_t* cnt = (int32_t*)workspace;
    int32_t* cursor = cnt + (V + 1);
    int32_t* occ_tmp = cursor + (V + 1);
    NPI_CHECK_CUDA(cudaMemsetAsync(cnt, 0, sizeof(int32_t) * 2 * (size_t)(V + 1), st));
    gid_count_kernel<<<grid_for(4), 256, 0, st>>>(gid, n_dev, n_host, cnt);
    NPI_CHECK_LAUNCH();
    if (V <= 8192) {
        gid_scan_kernel<<<1, 1024, 0, st>>>(cnt, V, occ_ptr);
        NPI_CHECK_LAUNCH();
    } else {      // many buckets (rows of a batch by representative: 215 k; nodes of the 100x graph: 508 k): three-kernel scan
        NPI_REQUIRE((int64_t)V + 1 <= (int64_t)4096 * 4096, "gid_index_build: too many buckets");
        int32_t* tile_sums = occ_tmp + n_host + 4;
        if (int rc = launch_excl_scan_i32(cnt, (int64_t)V + 1, occ_ptr, nullptr, tile_sums, st)) return rc;      // cnt[V] == 0
    }
    gid_fill_kernel<<<grid_for(4), 256, 0, st>>>(gid, n_dev, n_host, occ_ptr, cursor, occ_tmp);
    NPI_CHECK_LAUNCH();
    gid_sort_kernel<<<grid_for(8), 256, 0, st>>>(V, occ_ptr, occ_tmp, occ_node);
    NPI_CHECK_LAUNCH();
    return NPI_OK;
}

extern "C" int32_t npi_gid_reduce_partials(void) { return gid_reduce_grid(); }

extern "C" int npi_gid_reduce(const float* dxa, const uint8_t* dist, const int32_t* occ_ptr, const int32_t* occ_node,
                              int32_t V, float* G, float* label_partials, npi_stream_t stream) {
    NPI_REQUIRE(dxa && dist && occ_ptr && occ_node && G && label_partials && V > 0, "gid_reduce: bad argument");
    gid_reduce_kernel<<<gid_reduce_grid(), AG_THREADS, 0, (cudaStream_t)stream>>>(dxa, dist, occ_ptr, occ_node, V, G, label_partials);
    NPI_CHECK_LAUNCH();
    return NPI_OK;
}
