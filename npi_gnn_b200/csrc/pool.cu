// TopKPooling(128, ratio) + global max/mean readout -- forward and backward.
//
// Replaces self.poolN(x, edge_index, None, batch) and cat[gmp, gap] of reference
// src/classes.py:63-64,67-68,71-72 (PyG 1.4.2 semantics, SURVEY.md Appendix A.3/A.4; K4/K5 in
// SURVEY 2.3): score, per-graph top-k, gating, filter_adj, readout -- with no host sync, no
// dense [B,max_n] padding and no Python loop over graphs.
#include "hub.cuh"

namespace npi {

// ------------------------------------------------------------------ score (module API only)
__global__ void __launch_bounds__(256) topk_score_kernel(const float* h, const int32_t* n_dev, int n_host,
                                                          const float* pw, float* z_out, float* s_out) {
    const int n = dev_size(n_dev, n_host);
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    float4 p = ldg4(pw + 4 * lane);
    float norm = sqrtf(warp_sum(dot4(p, p)));
    for (int64_t i = warp0; i < n; i += nwarps) {
        float d = warp_sum(dot4(ldg4(h + i * H + 4 * lane), p));
        if (lane == 0) {
            float z = d / norm;
            if (z_out) z_out[i] = z;
            if (s_out) s_out[i] = tanhf(z) + 0.0f;
        }
    }
}

// ------------------------------------------------------------------ per-graph top-k selection
// 64-bit key = (~orderable(score) << 32) | local index: an ascending sort yields descending
// score with ties broken by the lower node index (stable rule of Appendix A.3), with no
// stability requirement on the sort itself.  Bitonic sort in shared memory for graphs up to
// SEL_SMEM_KEYS nodes, in the caller's workspace beyond that.
#ifndef NPI_SEL_THREADS
#define NPI_SEL_THREADS 512
#endif
constexpr int SEL_THREADS = NPI_SEL_THREADS;      // 512: two CTAs (graphs) per SM, a batch of 200 graphs is one wave
constexpr int SEL_CTAS_PER_SM = SEL_THREADS <= 512 ? 2 : 1;
constexpr int SEL_SMEM_KEYS = 8192;

__device__ __forceinline__ uint32_t orderable(float f) {
    uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// keys is either the shared-memory array or the global workspace; the helper is inlined at both call
// sites so the shared-memory instance compiles to LDS/STS (not generic loads).
__device__ __forceinline__ void topk_sort_emit(uint64_t* keys, const float* s, int lo, int n, int np2, int olo, int k, int g,
                                               int32_t* perm, int32_t* new_id, int32_t* batch_out,
                                               const int32_t* __restrict__ row_map, int32_t* perm_src) {
    for (int i = threadIdx.x; i < np2; i += SEL_THREADS) {
        uint64_t key = ~0ull;
        // +0.0f folds -0.0 into +0.0 so that they tie (torch's sort compares values, not bits)
        if (i < n) key = ((uint64_t)(~orderable(s[row_map ? row_map[lo + i] : lo + i] + 0.0f)) << 32) | (uint32_t)i;
        keys[i] = key;
    }
    // compare-exchange t of a step with stride <= 32 only touches the 64-key block 64*(t/32)..+63,
    // which the same warp owns in every such step: those steps need a warp barrier only; block
    // barriers are kept around the steps that cross 64-key blocks (21 of 78 steps at 4096 keys)
    bool wide_prev = true;
    for (int size = 2; size <= np2; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            const bool wide = stride > 32;
            if (wide || wide_prev) __syncthreads(); else __syncwarp();
            wide_prev = wide;
            for (int t = threadIdx.x; t < (np2 >> 1); t += SEL_THREADS) {
                int pos = 2 * t - (t & (stride - 1));
                int par = pos + stride;
                bool up = ((pos & size) == 0);
                uint64_t a = keys[pos], b = keys[par];
                if ((a > b) == up) { keys[pos] = b; keys[par] = a; }
            }
        }
    }
    __syncthreads();
    for (int r = threadIdx.x; r < n; r += SEL_THREADS) {
        int idx = (int)(uint32_t)(keys[r] & 0xffffffffull);
        if (r < k) {
            perm[olo + r] = lo + idx;
            if (perm_src) perm_src[olo + r] = row_map[lo + idx];
            new_id[lo + idx] = olo + r;
            if (batch_out) batch_out[olo + r] = g;
        } else {
            new_id[lo + idx] = -1;
        }
    }
}

// LSD radix sort of one graph in shared memory (256 < n <= SEL_SMEM_KEYS): 32-bit keys
// ~orderable(score) (ascending = descending score), 16-bit local indices as payload, four stable
// 8-bit passes.  Stability keeps equal scores in index order, which is the tie rule above.  Each
// warp owns a CONTIGUOUS run of items; ranks inside a (warp, digit) bucket come from match_any,
// bucket bases from one block scan over the [digit][warp] counts -- ~6x fewer instructions than
// the bitonic network at n = 4096.
constexpr int RS_WARPS = SEL_THREADS / 32;
constexpr int RS_MAXSL = SEL_SMEM_KEYS / SEL_THREADS;      // 32-item slots per warp (<= 8)
constexpr int RS_SMALL = 256;                              // graphs up to this size keep the bitonic network

__host__ __device__ inline size_t topk_radix_smem_bytes(int cap) {      // cap: multiple of 32
    return (size_t)cap * (4 + 4 + 2 + 2) + (size_t)(256 * RS_WARPS + 40) * 4;
}

__device__ __forceinline__ void topk_radix_emit(unsigned char* smem, int cap, const float* s, int lo, int n, int olo, int k, int g,
                                                int32_t* perm, int32_t* new_id, int32_t* batch_out,
                                                const int32_t* __restrict__ row_map, int32_t* perm_src) {
    uint32_t* keyA = reinterpret_cast<uint32_t*>(smem);
    uint32_t* keyB = keyA + cap;
    uint16_t* idxA = reinterpret_cast<uint16_t*>(keyB + cap);
    uint16_t* idxB = idxA + cap;
    uint32_t* hist = reinterpret_cast<uint32_t*>(idxB + cap);          // [warp][256]
    int* sscan = reinterpret_cast<int*>(hist + 256 * RS_WARPS);
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const uint32_t lt = (1u << lane) - 1u;
    const int chunk = ((n + SEL_THREADS - 1) / SEL_THREADS) * 32;       // items per warp, multiple of 32
    const int nslots = chunk >> 5;
    for (int i = tid; i < n; i += SEL_THREADS) {
        keyA[i] = ~orderable(s[row_map ? row_map[lo + i] : lo + i] + 0.0f);      // +0.0f folds -0.0 into +0.0 (torch compares values)
        idxA[i] = (uint16_t)i;
    }
    uint32_t* ks = keyA; uint32_t* kd = keyB; uint16_t* is = idxA; uint16_t* id = idxB;
#pragma unroll 1
    for (int pass = 0; pass < 4; ++pass) {
        const int shift = 8 * pass;
        for (int e = tid; e < 256 * RS_WARPS; e += SEL_THREADS) hist[e] = 0;
        __syncthreads();
        uint32_t myrank[RS_MAXSL];
#pragma unroll
        for (int sl = 0; sl < RS_MAXSL; ++sl) {
            if (sl < nslots) {
                const int i = w * chunk + sl * 32 + lane;
                const bool valid = i < n;
                const unsigned act = __ballot_sync(0xffffffffu, valid);
                uint32_t d = 0, peers = 0, base = 0;
                if (valid) {
                    d = (ks[i] >> shift) & 255u;
                    peers = __match_any_sync(act, d);
                    base = hist[w * 256 + d];
                }
                __syncwarp();
                if (valid) {
                    const uint32_t r = __popc(peers & lt);
                    if (r == 0) hist[w * 256 + d] = base + __popc(peers);
                    myrank[sl] = base + r;
                }
                __syncwarp();
            }
        }
        __syncthreads();
        // exclusive scan in (digit, warp) order: thread t owns digit t/G, warps (t%G)*8 .. +7, G = RS_WARPS/8
        {
            constexpr int G = RS_WARPS / 8;
            static_assert(G * 256 == SEL_THREADS && RS_WARPS % 8 == 0, "one thread per (digit, group of 8 warps)");
            const int d = tid / G, w0 = (tid % G) * 8;
            uint32_t v[8];
            int sum = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) { v[j] = hist[(w0 + j) * 256 + d]; sum += (int)v[j]; }
            int total;
            int run = block_excl_scan<SEL_THREADS>(sum, sscan, &total);
#pragma unroll
            for (int j = 0; j < 8; ++j) { hist[(w0 + j) * 256 + d] = (uint32_t)run; run += (int)v[j]; }
        }
        __syncthreads();
#pragma unroll
        for (int sl = 0; sl < RS_MAXSL; ++sl) {
            if (sl < nslots) {
                const int i = w * chunk + sl * 32 + lane;
                if (i < n) {
                    const uint32_t key = ks[i];
                    const uint32_t dst = hist[w * 256 + ((key >> shift) & 255u)] + myrank[sl];
                    kd[dst] = key;
                    id[dst] = is[i];
                }
            }
        }
        __syncthreads();
        uint32_t* tk = ks; ks = kd; kd = tk;
        uint16_t* ti = is; is = id; id = ti;
    }
    for (int r = tid; r < n; r += SEL_THREADS) {
        const int idx = (int)is[r];
        if (r < k) {
            perm[olo + r] = lo + idx;
            if (perm_src) perm_src[olo + r] = row_map[lo + idx];
            new_id[lo + idx] = olo + r;
            if (batch_out) batch_out[olo + r] = g;
        } else {
            new_id[lo + idx] = -1;
        }
    }
}

__global__ void __launch_bounds__(SEL_THREADS, SEL_CTAS_PER_SM) topk_select_kernel(const float* s, const int32_t* gin, const int32_t* gout, int B,
                                                                   int32_t* perm, int32_t* new_id, int32_t* batch_out,
                                                                   const int32_t* row_map, int32_t* perm_src,
                                                                   uint64_t* ws, int64_t ws_keys_per_graph, int radix_cap) {
    pdl_trigger();
    pdl_wait();
    extern __shared__ __align__(16) uint64_t skeys[];
    const int g = blockIdx.x;
    if (g >= B) return;
    const int lo = gin[g], n = gin[g + 1] - lo;
    const int olo = gout[g], k = gout[g + 1] - olo;
    int np2 = 1;
    while (np2 < n) np2 <<= 1;
    if (n > RS_SMALL && n <= radix_cap)
        topk_radix_emit(reinterpret_cast<unsigned char*>(skeys), radix_cap, s, lo, n, olo, k, g, perm, new_id, batch_out, row_map, perm_src);
    else if (np2 <= SEL_SMEM_KEYS && n <= RS_SMALL) topk_sort_emit(skeys, s, lo, n, np2, olo, k, g, perm, new_id, batch_out, row_map, perm_src);
    else topk_sort_emit(ws + (int64_t)g * ws_keys_per_graph, s, lo, n, np2, olo, k, g, perm, new_id, batch_out, row_map, perm_src);
}

// ------------------------------------------------------------------ gating + readout
// Every graph is cut into GR_SPLIT contiguous row ranges, one CTA each (B*GR_SPLIT CTAs keep all
// SMs busy although graph sizes span 1..~1400 rows); a CTA gates its rows (x' = h[perm]*s[perm],
// written once) and leaves per-column max / argmax / sum partials; a second small kernel combines
// the GR_SPLIT partials of a graph in a fixed order (deterministic mean, lowest-row argmax).
constexpr int GR_THREADS = 256;
constexpr int GR_WARPS = GR_THREADS / 32;
#ifndef NPI_GR_SPLIT
#define NPI_GR_SPLIT 8
#endif
constexpr int GR_SPLIT = NPI_GR_SPLIT;
constexpr int GR_PART = 3 * H;          // max[128] | sum[128] | argmax[128] (int bits)

__device__ __forceinline__ void gr_take(float4& mx, int4& ar, const float4& v, int r) {
    if (v.x > mx.x) { mx.x = v.x; ar.x = r; }
    if (v.y > mx.y) { mx.y = v.y; ar.y = r; }
    if (v.z > mx.z) { mx.z = v.z; ar.z = r; }
    if (v.w > mx.w) { mx.w = v.w; ar.w = r; }
}

__global__ void __launch_bounds__(GR_THREADS) gate_readout_kernel(const float* h, const float* s, const int32_t* perm,
                                                                   const int32_t* gout, int B, float* xp, float* part) {
    pdl_trigger();
    pdl_wait();
    __shared__ __align__(16) float smax[GR_WARPS][H];
    __shared__ __align__(16) float ssum[GR_WARPS][H];
    __shared__ __align__(16) int sarg[GR_WARPS][H];
    const int g = blockIdx.x / GR_SPLIT, sp = blockIdx.x % GR_SPLIT;
    if (g >= B) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int lo = gout[g], hi = gout[g + 1];
    const int chunk = (hi - lo + GR_SPLIT - 1) / GR_SPLIT;
    const int r0 = lo + sp * chunk, r1 = min(hi, r0 + chunk);
    float4 mx = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
    float4 sm = make_float4(0.f, 0.f, 0.f, 0.f);
    int4 ar = make_int4(-1, -1, -1, -1);
    int r = r0 + warp;
    for (; r + 3 * GR_WARPS < r1; r += 4 * GR_WARPS) {          // 4 independent row gathers in flight per warp
        int o[4]; float sv[4]; float4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) o[u] = perm[r + u * GR_WARPS];
#pragma unroll
        for (int u = 0; u < 4; ++u) { sv[u] = s[o[u]]; v[u] = ldg4(h + (int64_t)o[u] * H + 4 * lane); }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            v[u] = mul4(v[u], sv[u]);
            st4(xp + (int64_t)(r + u * GR_WARPS) * H + 4 * lane, v[u]);
            gr_take(mx, ar, v[u], r + u * GR_WARPS);
            sm = add4(sm, v[u]);
        }
    }
    for (; r < r1; r += GR_WARPS) {
        const int o = perm[r];
        const float4 v = mul4(ldg4(h + (int64_t)o * H + 4 * lane), s[o]);
        st4(xp + (int64_t)r * H + 4 * lane, v);
        gr_take(mx, ar, v, r);
        sm = add4(sm, v);
    }
    st4(&smax[warp][4 * lane], mx);
    st4(&ssum[warp][4 * lane], sm);
    *reinterpret_cast<int4*>(&sarg[warp][4 * lane]) = ar;
    __syncthreads();
    if (threadIdx.x < H) {
        const int c = threadIdx.x;
        float m = smax[0][c], t = ssum[0][c];
        int a = sarg[0][c];
#pragma unroll
        for (int w = 1; w < GR_WARPS; ++w) {
            const float mv = smax[w][c];
            const int av = sarg[w][c];
            if (av >= 0 && (a < 0 || mv > m || (mv == m && av < a))) { m = mv; a = av; }
            t += ssum[w][c];
        }
        float* pp = part + (int64_t)blockIdx.x * GR_PART;
        pp[c] = m; pp[H + c] = t; pp[2 * H + c] = __int_as_float(a);
    }
}

__global__ void __launch_bounds__(H) readout_combine_kernel(const float* part, const int32_t* gout, int B, float* readout,
                                                            int accumulate, int32_t* argmax) {
    const int g = blockIdx.x, c = threadIdx.x;
    if (g >= B) return;
    const float* pp = part + (int64_t)g * GR_SPLIT * GR_PART;
    float m = pp[c], t = pp[H + c];
    int a = __float_as_int(pp[2 * H + c]);
#pragma unroll
    for (int sp = 1; sp < GR_SPLIT; ++sp) {
        const float mv = pp[sp * GR_PART + c];
        const int av = __float_as_int(pp[sp * GR_PART + 2 * H + c]);
        if (av >= 0 && (a < 0 || mv > m || (mv == m && av < a))) { m = mv; a = av; }
        t += pp[sp * GR_PART + H + c];
    }
    // an empty graph (operator API only: a gap in `batch` or a `size` beyond it) reads 0 for max and mean, as
    // PyG's scatter does; its argmax stays -1, so no row gets a max gradient
    const int cnt = gout[g + 1] - gout[g];
    if (cnt == 0) m = 0.f;
    const float mean = cnt ? t / (float)cnt : 0.f;
    float* ro = readout + (int64_t)g * 2 * H;
    if (accumulate) { ro[c] += m; ro[H + c] += mean; }
    else { ro[c] = m; ro[H + c] = mean; }
    if (argmax) argmax[(int64_t)g * H + c] = a;
}

// ------------------------------------------------------------------ filter_adj on CSR
// New row r = old row perm[r] with dropped sources removed and the rest relabelled, order kept.
// A warp owns 32 consecutive new rows: their old-row extents are fetched lane-parallel, then the
// warp sweeps the FLATTENED entries of the 32 rows (lane <-> entry, row found by a 5-step shuffle
// search in the warp's prefix of row lengths), so hub rows and leaf rows cost the same per entry
// and there is one col -> new_id pointer chase per 32 entries instead of one per row.  Because the
// 32 rows are consecutive, their kept entries in flattened order ARE the output order: the fill
// pass only needs the warp's start offset and a running ballot prefix.
constexpr int FA_THREADS = 256;   // one CTA handles 256 consecutive new rows
constexpr int FA_WARPS = FA_THREADS / 32;
#ifndef NPI_FA_CHUNKS
#define NPI_FA_CHUNKS 8
#endif
constexpr int FA_CHUNKS = NPI_FA_CHUNKS;   // 32-entry chunks in flight per sweep iteration: the kernel's length is the sweep of the warp that
                                           // holds a hub row (thousands of entries, two dependent loads per iteration)

struct FaRows { int b; int off; int total; };     // per lane: old-row begin, exclusive prefix of lengths; warp total

__device__ __forceinline__ FaRows fa_rows(const int32_t* rowptr, const int32_t* perm, int r, int nnew, int lane) {
    int b = 0, len = 0;
    if (r < nnew) { const int o = perm[r]; b = rowptr[o]; len = rowptr[o + 1] - b; }
    const int inc = warp_incl_scan_i(len, lane);
    FaRows f;
    f.b = b; f.off = inc - len; f.total = __shfl_sync(0xffffffffu, inc, 31);
    return f;
}
// entry at flattened position pos of the warp's 32 rows -> (row slot q, CSR index k)
__device__ __forceinline__ void fa_locate(const FaRows& f, int pos, int& q, int& k) {
    int lo = 0, hi = 32;
#pragma unroll
    for (int it = 0; it < 5; ++it) {
        const int mid = (lo + hi) >> 1;
        const int v = __shfl_sync(0xffffffffu, f.off, mid);
        if (v <= pos) lo = mid; else hi = mid;
    }
    q = lo;
    k = __shfl_sync(0xffffffffu, f.b, lo) + (pos - __shfl_sync(0xffffffffu, f.off, lo));
}

__global__ void __launch_bounds__(FA_THREADS) filter_count_kernel(const int32_t* rowptr, const int32_t* col, const int32_t* perm,
                                                                   const int32_t* new_id, const int32_t* nnew_dev, int nnew_host,
                                                                   int32_t* rowptr_out, int32_t* partial, int32_t* hubq, int hubq_cap) {
    __shared__ int sh[FA_THREADS / 32 + 2];
    __shared__ int s_cnt[FA_WARPS][32];
    __shared__ int s_hist[N_CLS];
    const int nnew = dev_size(nnew_dev, nnew_host);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int base = blockIdx.x * FA_THREADS;
    if (hubq && blockIdx.x == 0 && threadIdx.x == 0) hubq[1] = hubq_cap;
    if (base >= nnew) { if (threadIdx.x == 0) partial[blockIdx.x] = 0; return; }
    if (threadIdx.x < N_CLS) s_hist[threadIdx.x] = 0;
    s_cnt[warp][lane] = 0;
    __syncthreads();
    const FaRows f = fa_rows(rowptr, perm, base + warp * 32 + lane, nnew, lane);
    for (int p0 = 0; p0 < f.total; p0 += 32 * FA_CHUNKS) {
        int q[FA_CHUNKS], c[FA_CHUNKS];
#pragma unroll
        for (int u = 0; u < FA_CHUNKS; ++u) {
            const int p = p0 + 32 * u + lane;
            int k;
            c[u] = -1; q[u] = 0;
            if (p0 + 32 * u < f.total) {                       // warp-uniform: chunks behind the end cost nothing
                fa_locate(f, min(p, f.total - 1), q[u], k);
                if (p < f.total) c[u] = col[k];
            }
        }
#pragma unroll
        for (int u = 0; u < FA_CHUNKS; ++u) c[u] = (c[u] >= 0) ? new_id[c[u]] : -1;
#pragma unroll
        for (int u = 0; u < FA_CHUNKS; ++u)
            if (c[u] >= 0) atomicAdd(&s_cnt[warp][q[u]], 1);
    }
    __syncwarp();
    const int mine = s_cnt[warp][lane];
    int tot;
    const int ex = block_excl_scan<FA_THREADS>(mine, sh, &tot);
    const int r = base + threadIdx.x;
    if (r < nnew) rowptr_out[r] = ex;        // chunk-local exclusive prefix for now
    if (threadIdx.x == 0) partial[blockIdx.x] = tot;
    if (hubq) {
        // the new CSR's hub queue is listed on the way (what hub_scan_kernel does from the finished rowptr): the
        // aggregation of the next layer waits for this chain, and a row's segments only need its LENGTH
        const HubQueue hq = hub_view(hubq, hubq_cap);
        if (r < nnew) hub_list_row(hq, hubq_cap, s_hist, r, mine);
        __syncthreads();
        if (threadIdx.x < N_CLS && s_hist[threadIdx.x]) atomicAdd(&hq.hdr[HQ_CLS + threadIdx.x], s_hist[threadIdx.x]);
    }
}

__global__ void __launch_bounds__(1024) scan_partials_kernel(int32_t* partial, int nchunks, const int32_t* nnew_dev, int nnew_host,
                                                              int32_t* rowptr_out) {
    __shared__ int sh[1024 / 32 + 2];
    int run = 0;
    for (int c = 0; c < nchunks; c += 1024) {
        int i = c + threadIdx.x;
        int v = (i < nchunks) ? partial[i] : 0;
        int tot;
        int ex = block_excl_scan<1024>(v, sh, &tot);
        if (i < nchunks) partial[i] = run + ex;
        run += tot;
    }
    if (threadIdx.x == 0) {
        const int nnew = dev_size(nnew_dev, nnew_host);
        rowptr_out[nnew] = run;
    }
}

__global__ void __launch_bounds__(FA_THREADS) filter_fill_kernel(const int32_t* rowptr, const int32_t* col, const int32_t* perm,
                                                                  const int32_t* new_id, const int32_t* nnew_dev, int nnew_host,
                                                                  int32_t* rowptr_out, int32_t* col_out, const int32_t* partial,
                                                                  int32_t* hubq, int hubq_cap, int4* __restrict__ rows, int nchunks) {
    __shared__ int s_pre[FA_THREADS + 1];
    __shared__ int s_hist[N_CLS], s_start[N_CLS];
    const int nnew = dev_size(nnew_dev, nnew_host);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int base = blockIdx.x * FA_THREADS;
    if (base >= nnew) return;
    const int cbase = partial[blockIdx.x];
    const int r_own = base + threadIdx.x;
    int start_own = 0;
    if (r_own < nnew) start_own = cbase + rowptr_out[r_own];
    if (rows) {
        // binned row order of the new CSR (what row_order_fill_kernel builds from the finished rowptr): the class totals
        // are complete (filter_count_kernel), a row's extent is its final start and the next row's
        if (threadIdx.x < N_CLS) s_hist[threadIdx.x] = 0;
        s_pre[threadIdx.x] = start_own;
        if (threadIdx.x == 0) {
            const bool last = base + FA_THREADS >= nnew;
            s_pre[FA_THREADS] = last ? rowptr_out[nnew] : partial[blockIdx.x + 1];      // scan_partials_kernel wrote both
        }
    }
    __syncthreads();                               // all chunk-local prefixes read before being overwritten
    if (r_own < nnew) rowptr_out[r_own] = start_own;
    if (rows) {
        int cls = -1, rank = 0, end_own = 0;
        if (r_own < nnew) {
            end_own = (threadIdx.x + 1 < FA_THREADS && r_own + 1 < nnew) ? s_pre[threadIdx.x + 1] : s_pre[FA_THREADS];
            cls = row_class(end_own - start_own);
            rank = atomicAdd(&s_hist[cls], 1);
        }
        __syncthreads();
        if (threadIdx.x < N_CLS) {
            int b0 = 0;
            for (int c = 0; c < (int)threadIdx.x; ++c) b0 += hubq[HQ_CLS + c];
            s_start[threadIdx.x] = b0 + (s_hist[threadIdx.x] ? atomicAdd(&hubq[HQ_CUR + threadIdx.x], s_hist[threadIdx.x]) : 0);
        }
        __syncthreads();
        if (cls >= 0 && cls < N_CLS - 1) rows[s_start[cls] + rank] = make_int4(r_own, start_own, end_own, r_own);
    }
    const FaRows f = fa_rows(rowptr, perm, r_own, nnew, lane);
    int w = __shfl_sync(0xffffffffu, start_own, 0);        // output slot of the warp's first kept entry
    for (int p0 = 0; p0 < f.total; p0 += 32 * FA_CHUNKS) {
        int id[FA_CHUNKS];
#pragma unroll
        for (int u = 0; u < FA_CHUNKS; ++u) {
            const int p = p0 + 32 * u + lane;
            int q, k;
            id[u] = -1;
            if (p0 + 32 * u < f.total) {                       // warp-uniform
                fa_locate(f, min(p, f.total - 1), q, k);
                if (p < f.total) id[u] = col[k];
            }
        }
#pragma unroll
        for (int u = 0; u < FA_CHUNKS; ++u) id[u] = (id[u] >= 0) ? new_id[id[u]] : -1;
#pragma unroll
        for (int u = 0; u < FA_CHUNKS; ++u) {
            const unsigned b = __ballot_sync(0xffffffffu, id[u] >= 0);
            if (id[u] >= 0) col_out[w + __popc(b & ((1u << lane) - 1u))] = id[u];
            w += __popc(b);
        }
    }
}

// ------------------------------------------------------------------ backward
constexpr int PB_THREADS = 256;
#ifndef NPI_PB_CHUNK
#define NPI_PB_CHUNK 8
#endif
constexpr int PB_CHUNK = NPI_PB_CHUNK;    // selected rows per warp task (<= 32)
constexpr int PB_PART = 2 * H + 4;     // per-CTA partial: sum dz*h [128] | sum dz*z | pad[3] | sum dpre [128]
__global__ void __launch_bounds__(PB_THREADS, 3) pool_bwd_kernel(const float* d_xp, const float* d_readout, const float* h, const float* z,
                                                               const float* s, const int32_t* perm, const int32_t* batch_out,
                                                               const int32_t* argmax, const int32_t* gout,
                                                               const int32_t* nnew_dev, int nnew_host, const float* pw, int relu,
                                                               float* dpre, float* partial /*[G][PB_PART]*/) {
    pdl_trigger();
    pdl_wait();
    __shared__ __align__(16) float sred[PB_THREADS / 32][H + 4];
    __shared__ __align__(16) float sdb[PB_THREADS / 32][H];
    const int nnew = dev_size(nnew_dev, nnew_host);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t warp0 = (int64_t)blockIdx.x * (PB_THREADS / 32) + warp;
    const int64_t nwarps = (int64_t)gridDim.x * (PB_THREADS / 32);
    float4 p = ldg4(pw + 4 * lane);
    const float norm = sqrtf(warp_sum(dot4(p, p)));
    const float4 pn = make_float4(p.x / norm, p.y / norm, p.z / norm, p.w / norm);
    float4 accA = make_float4(0.f, 0.f, 0.f, 0.f);
    float4 accB = make_float4(0.f, 0.f, 0.f, 0.f);
    float accS = 0.f;
    // a warp takes PB_CHUNK consecutive selected rows: the per-row scalars (old row id, graph, score,
    // pre-tanh score, 1/k) are fetched lane-parallel first, so the row loop below only issues
    // independent 512-byte row loads (two rows in flight).  The chunk is short because a warp walks
    // it serially, one dependent load round trip per pair of rows: with 32-row chunks every launch
    // cost at least 16 round trips (~25 us) however few rows the layer had (profiles/r02j_ncu.md).
    for (int64_t r0 = warp0 * PB_CHUNK; r0 < nnew; r0 += nwarps * PB_CHUNK) {
        const int64_t rl = r0 + lane;
        int o_l = 0, g_l = 0;
        float s_l = 0.f, z_l = 0.f, kinv_l = 0.f;
        if (lane < PB_CHUNK && rl < nnew) {
            o_l = perm[rl]; g_l = batch_out[rl];
            s_l = s[o_l]; z_l = z[o_l];
            kinv_l = (float)(gout[g_l + 1] - gout[g_l]);
        }
        const int cnt = (int)min((int64_t)PB_CHUNK, nnew - r0);
        for (int q = 0; q < cnt; q += 2) {
            const bool two = q + 1 < cnt;
            int o[2], g[2]; float sv[2], zv[2], kd[2];
            float4 gx[2], gm[2], gmx[2], hv[2]; int4 am[2];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const int src = min(q + u, cnt - 1);
                o[u] = __shfl_sync(0xffffffffu, o_l, src); g[u] = __shfl_sync(0xffffffffu, g_l, src);
                sv[u] = __shfl_sync(0xffffffffu, s_l, src); zv[u] = __shfl_sync(0xffffffffu, z_l, src);
                kd[u] = __shfl_sync(0xffffffffu, kinv_l, src);
            }
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                if (u == 0 || two) {
                    const int64_t r = r0 + q + u;
                    gx[u] = d_xp ? ldg4(d_xp + r * H + 4 * lane) : make_float4(0.f, 0.f, 0.f, 0.f);
                    gm[u] = ldg4(d_readout + (int64_t)g[u] * 2 * H + H + 4 * lane);
                    am[u] = *reinterpret_cast<const int4*>(argmax + (int64_t)g[u] * H + 4 * lane);
                    gmx[u] = ldg4(d_readout + (int64_t)g[u] * 2 * H + 4 * lane);
                    hv[u] = ldg4(h + (int64_t)o[u] * H + 4 * lane);
                }
            }
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                if (u == 0 || two) {
                    const int64_t r = r0 + q + u;
                    float4 x = gx[u];
                    x.x += gm[u].x / kd[u]; x.y += gm[u].y / kd[u]; x.z += gm[u].z / kd[u]; x.w += gm[u].w / kd[u];
                    if (am[u].x == r) x.x += gmx[u].x;
                    if (am[u].y == r) x.y += gmx[u].y;
                    if (am[u].z == r) x.z += gmx[u].z;
                    if (am[u].w == r) x.w += gmx[u].w;
                    const float ds = warp_sum(dot4(x, hv[u]));
                    const float dz = ds * (1.f - sv[u] * sv[u]);
                    float4 dh = make_float4(x.x * sv[u] + dz * pn.x, x.y * sv[u] + dz * pn.y,
                                            x.z * sv[u] + dz * pn.z, x.w * sv[u] + dz * pn.w);
                    if (relu) {
                        dh.x = hv[u].x > 0.f ? dh.x : 0.f; dh.y = hv[u].y > 0.f ? dh.y : 0.f;
                        dh.z = hv[u].z > 0.f ? dh.z : 0.f; dh.w = hv[u].w > 0.f ? dh.w : 0.f;
                    }
                    st4(dpre + r * H + 4 * lane, dh);
                    accB = add4(accB, dh);
                    accA.x = fmaf(dz, hv[u].x, accA.x); accA.y = fmaf(dz, hv[u].y, accA.y);
                    accA.z = fmaf(dz, hv[u].z, accA.z); accA.w = fmaf(dz, hv[u].w, accA.w);
                    accS = fmaf(dz, zv[u], accS);
                }
            }
        }
    }
    st4(&sred[warp][4 * lane], accA);
    st4(&sdb[warp][4 * lane], accB);
    if (lane == 0) sred[warp][H] = accS;
    __syncthreads();
    if (threadIdx.x <= H) {
        float t = 0.f;
#pragma unroll
        for (int w = 0; w < PB_THREADS / 32; ++w) t += sred[w][threadIdx.x];
        partial[(int64_t)blockIdx.x * PB_PART + threadIdx.x] = t;
    }
    if (threadIdx.x < H) {
        float t = 0.f;
#pragma unroll
        for (int w = 0; w < PB_THREADS / 32; ++w) t += sdb[w][threadIdx.x];
        partial[(int64_t)blockIdx.x * PB_PART + H + 4 + threadIdx.x] = t;
    }
}

// partial sums of the CTAs are combined in a fixed order: a CTA owns PBR_COLS columns; PBR_SLICES
// interleaved slices of the CTA list are summed in parallel (independent loads, 4 in flight per
// thread), then the slices in order.  The scalar sum(dz*z) is recomputed by every CTA.
constexpr int PBR_SLICES = 32, PBR_COLS = 32;
__global__ void __launch_bounds__(PBR_SLICES * PBR_COLS) pool_bwd_reduce_kernel(const float* __restrict__ partial, int G,
                                                                              const float* __restrict__ pw, float* d_pw, float* d_bias) {
    __shared__ float sa[PBR_SLICES][PBR_COLS + 1], sb[PBR_SLICES][PBR_COLS + 1], ss[PBR_SLICES];
    __shared__ float sS, sN;
    const int cl = threadIdx.x % PBR_COLS, sl = threadIdx.x / PBR_COLS;
    const int c = blockIdx.x * PBR_COLS + cl;
    float a = 0.f, bsum = 0.f, t = 0.f;
    int g = sl;
    for (; g + 3 * PBR_SLICES < G; g += 4 * PBR_SLICES) {
        float av[4], bv[4], tv[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const float* row = partial + (int64_t)(g + u * PBR_SLICES) * PB_PART;
            av[u] = row[c]; bv[u] = row[H + 4 + c]; tv[u] = (cl == 0) ? row[H] : 0.f;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) { a += av[u]; bsum += bv[u]; t += tv[u]; }
    }
    for (; g < G; g += PBR_SLICES) {
        const float* row = partial + (int64_t)g * PB_PART;
        a += row[c]; bsum += row[H + 4 + c];
        if (cl == 0) t += row[H];
    }
    sa[sl][cl] = a; sb[sl][cl] = bsum;
    if (cl == 0) ss[sl] = t;
    __syncthreads();
    if (threadIdx.x == 0) {
        float tt = 0.f;
        for (int q = 0; q < PBR_SLICES; ++q) tt += ss[q];
        float nn = 0.f;
        for (int q = 0; q < H; ++q) nn = fmaf(pw[q], pw[q], nn);
        sS = tt; sN = nn;
    }
    __syncthreads();
    if (sl == 0) {
        float at = 0.f, bt = 0.f;
#pragma unroll
        for (int q = 0; q < PBR_SLICES; ++q) { at += sa[q][cl]; bt += sb[q][cl]; }
        if (d_bias) d_bias[c] = bt;
        // z = (h.w)/||w||  =>  dw = (sum dz h)/||w|| - w (sum dz z)/||w||^2
        d_pw[c] = at / sqrtf(sN) - pw[c] * sS / sN;
    }
}

static int pool_bwd_grid() { return num_sms() * 3; }

}  // namespace npi

using namespace npi;

extern "C" int npi_topk_score(const float* h, const int32_t* n_dev, int32_t n_host, const float* pool_w,
                              float* z_out, float* s_out, npi_stream_t stream) {
    NPI_REQUIRE(h && pool_w, "topk_score: null argument");
    topk_score_kernel<<<grid_for(8), 256, 0, (cudaStream_t)stream>>>(h, n_dev, n_host, pool_w, z_out, s_out);
    NPI_CHECK_LAUNCH();
    return NPI_OK;
}

static int next_pow2(int n) { int p = 1; while (p < n) p <<= 1; return p; }

extern "C" int64_t npi_topk_select_workspace_bytes(int32_t B, int32_t max_graph_nodes) {
    int np2 = next_pow2(max_graph_nodes);
    if (np2 <= SEL_SMEM_KEYS) return 16;
    return (int64_t)B * np2 * 8;
}

extern "C" int npi_topk_select(const float* s, const int32_t* graph_ptr_in, const int32_t* graph_ptr_out, int32_t B,
                               int32_t max_graph_nodes, int32_t* perm, int32_t* new_id, int32_t* batch_out,
                               const int32_t* row_map, int32_t* perm_src,
                               void* workspace, int64_t workspace_bytes, npi_stream_t stream) {
    NPI_REQUIRE(s && graph_ptr_in && graph_ptr_out && perm && new_id, "topk_select: null argument");
    NPI_REQUIRE((row_map == nullptr) == (perm_src == nullptr), "topk_select: row_map and perm_src come together");
    if (B <= 0) return NPI_OK;
    int np2 = next_pow2(max_graph_nodes > 1 ? max_graph_nodes : 2);
    NPI_REQUIRE(workspace_bytes >= npi_topk_select_workspace_bytes(B, max_graph_nodes), "topk_select: workspace too small");
    // shared memory: the radix layout for the largest graph of the batch (<= SEL_SMEM_KEYS nodes), which
    // also covers the bitonic network of the small graphs; larger graphs sort in the workspace
    int cap = max_graph_nodes > RS_SMALL ? ((max_graph_nodes < SEL_SMEM_KEYS ? max_graph_nodes : SEL_SMEM_KEYS) + 31) / 32 * 32 : 0;
    size_t smem = cap ? topk_radix_smem_bytes(cap) : 0;
    if (smem < (size_t)RS_SMALL * 8) smem = (size_t)RS_SMALL * 8;
    static OncePerDevice cfg;
    if (cfg.need()) {
        NPI_CHECK_CUDA(cudaFuncSetAttribute(topk_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                            (int)topk_radix_smem_bytes(SEL_SMEM_KEYS)));
    }
    NPI_CHECK_CUDA(launch_dep(topk_select_kernel, B, SEL_THREADS, smem, (cudaStream_t)stream, s, graph_ptr_in, graph_ptr_out, B, perm, new_id,
                              batch_out, row_map, perm_src, (uint64_t*)workspace, np2, cap));
    return NPI_OK;
}

extern "C" int64_t npi_pool_gate_readout_workspace_bytes(int32_t B) {
    return (int64_t)(B > 0 ? B : 1) * GR_SPLIT * GR_PART * sizeof(float);
}

extern "C" int npi_pool_gate_readout(const float* h, const float* s, const int32_t* perm, const int32_t* graph_ptr_out, int32_t B,
                                     float* xp, float* readout, int32_t accumulate, int32_t* argmax,
                                     void* workspace, int64_t workspace_bytes, int32_t phases, npi_stream_t stream) {
    NPI_REQUIRE(h && s && perm && graph_ptr_out && xp && readout && workspace, "pool_gate_readout: null argument");
    NPI_REQUIRE(workspace_bytes >= npi_pool_gate_readout_workspace_bytes(B), "pool_gate_readout: workspace too small");
    NPI_REQUIRE(phases >= 0 && phases <= 2, "pool_gate_readout: phases must be 0 (both), 1 (gating + partials) or 2 (readout)");
    if (B <= 0) return NPI_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if (phases == 0 || phases == 1) {      // x' (what the next projection waits for) + per-range partials into the workspace
        NPI_CHECK_CUDA(launch_dep(gate_readout_kernel, B * GR_SPLIT, GR_THREADS, 0, st, h, s, perm, graph_ptr_out, B, xp, (float*)workspace));
    }
    if (phases == 0 || phases == 2) {      // readout / argmax from the partials: nothing before the head reads them
        readout_combine_kernel<<<B, H, 0, st>>>((const float*)workspace, graph_ptr_out, B, readout, accumulate, argmax);
        NPI_CHECK_LAUNCH();
    }
    return NPI_OK;
}

extern "C" int64_t npi_filter_adj_workspace_bytes(int32_t n_new_max) {
    return ((int64_t)(n_new_max + FA_THREADS - 1) / FA_THREADS + 1) * 4;
}

extern "C" int npi_filter_adj(const int32_t* rowptr, const int32_t* col, const int32_t* perm, const int32_t* new_id,
                              const int32_t* nnew_dev, int32_t nnew_host, int32_t* rowptr_out, int32_t* col_out,
                              int32_t* hub_queue, int64_t hub_e_max, void* row_order,
                              void* workspace, int64_t workspace_bytes, npi_stream_t stream) {
    NPI_REQUIRE(rowptr && col && perm && new_id && rowptr_out && col_out && workspace, "filter_adj: null argument");
    NPI_REQUIRE(!row_order || hub_queue, "filter_adj: row_order comes with hub_queue");
    NPI_REQUIRE(((uintptr_t)row_order & 15) == 0, "filter_adj: row_order must be 16-byte aligned");
    const int hcap = hub_queue ? hub_cap(hub_e_max) : 0;
    NPI_REQUIRE(workspace_bytes >= npi_filter_adj_workspace_bytes(nnew_host), "filter_adj: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    int nchunks = (nnew_host + FA_THREADS - 1) / FA_THREADS;
    int32_t* partial = (int32_t*)workspace;
    if (nchunks > 0) {
        filter_count_kernel<<<nchunks, FA_THREADS, 0, st>>>(rowptr, col, perm, new_id, nnew_dev, nnew_host, rowptr_out, partial, hub_queue, hcap);
        NPI_CHECK_LAUNCH();
    }
    scan_partials_kernel<<<1, 1024, 0, st>>>(partial, nchunks, nnew_dev, nnew_host, rowptr_out);
    NPI_CHECK_LAUNCH();
    if (nchunks > 0) {
        filter_fill_kernel<<<nchunks, FA_THREADS, 0, st>>>(rowptr, col, perm, new_id, nnew_dev, nnew_host, rowptr_out, col_out, partial,
                                                           hub_queue, hcap, (int4*)row_order, nchunks);
        NPI_CHECK_LAUNCH();
    }
    return NPI_OK;
}

extern "C" int64_t npi_pool_bwd_workspace_bytes(void) { return (int64_t)pool_bwd_grid() * PB_PART * sizeof(float); }

extern "C" int npi_pool_bwd(const float* d_xp, const float* d_readout, const float* h, const float* z, const float* s,
                            const int32_t* perm, const int32_t* batch_out, const int32_t* argmax, const int32_t* graph_ptr_out,
                            const int32_t* nnew_dev, int32_t nnew_host, int32_t B, const float* pool_w, int32_t relu,
                            float* dpre, float* d_pool_w, float* d_bias, void* workspace, int64_t workspace_bytes,
                            int32_t phases, npi_stream_t stream) {
    NPI_REQUIRE(d_readout && h && z && s && perm && batch_out && argmax && graph_ptr_out && pool_w && dpre && d_pool_w && workspace,
                "pool_bwd: null argument");
    NPI_REQUIRE(workspace_bytes >= npi_pool_bwd_workspace_bytes(), "pool_bwd: workspace too small");
    NPI_REQUIRE(phases >= 0 && phases <= 2, "pool_bwd: phases must be 0 (both), 1 (dpre + partials) or 2 (parameter gradients)");
    (void)B;
    const int G = pool_bwd_grid();
    cudaStream_t st = (cudaStream_t)stream;
    if (phases == 0 || phases == 1) {      // dpre (what the layer below waits for) + per-CTA partials into the workspace
        NPI_CHECK_CUDA(launch_dep(pool_bwd_kernel, G, PB_THREADS, 0, st, d_xp, d_readout, h, z, s, perm, batch_out, argmax, graph_ptr_out,
                                  nnew_dev, nnew_host, pool_w, relu, dpre, (float*)workspace));
    }
    if (phases == 0 || phases == 2) {      // d_pool_w / d_bias from the partials: only the optimizer waits for them
        pool_bwd_reduce_kernel<<<H / PBR_COLS, PBR_SLICES * PBR_COLS, 0, st>>>((const float*)workspace, G, pool_w, d_pool_w, d_bias);
        NPI_CHECK_LAUNCH();
    }
    return NPI_OK;
}
