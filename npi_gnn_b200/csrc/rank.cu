// Ranking metrics of a scored pair set (ROC AUC, average precision, the ROC and PR curves) -- the evaluation of the
// reference's src/compare_withKmer_noKmer.py:39-74,213-368 (sklearn roc_curve / roc_auc_score / precision_recall_curve /
// average_precision_score / auc), on the device and over ONE global order of all scores.  Semantics: include/npi.h.
//
//   rank_key_kernel     key = ~orderable(score) (ascending key = descending score, -0.0 folded to +0.0), value = label;
//                       per-CTA status bits (NaN score, label not 0/1)
//   npi_sort_pairs_u32  32 key bits, four passes of three kernels (sort.cu)
//   rank_tile_kernel    per tile of the sorted run: positives and run ends (key[i] != key[i+1])
//   rank_scan_kernel    one CTA: exclusive scans of both tile counts over the tiles, n_pos, n_thresholds, status
//   rank_emit_kernel    for every run end i: threshold r = number of run ends before i, tps[r] = positives in [0, i],
//                       fps[r] = i + 1 - tps[r]
//   rank_area_kernel    per-CTA partials of twice_u (int64) and of the two PR areas (fp64) over the thresholds; the last
//                       CTA (ticket) combines them in a fixed order and writes summary / areas
// Only run ends are written, and the count of positives at a run end does not depend on the order inside the run of
// tied keys, so every output is bit-identical under any permutation of the input.  No floating-point atomics.
#include "common.cuh"

namespace npi {

constexpr int RK_THREADS = 1024;
constexpr int RK_ITEMS = 4;
constexpr int RK_TILE = RK_THREADS * RK_ITEMS;      // 4096 items per CTA
constexpr int RA_THREADS = 256;
constexpr int RA_MAX_CTAS = 1024;                   // area partials (one per CTA), summed by the last CTA

__device__ __forceinline__ float rank_score(uint32_t key) {
    const uint32_t o = ~key;
    return __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o);
}

struct RankWs {
    uint32_t* keys_a; int32_t* vals_a; uint32_t* keys_b; int32_t* vals_b;
    void* sort_ws; int64_t sort_bytes;
    int32_t* tile_status; int32_t* tile_pos; int32_t* tile_end;
    int32_t* totals;                  // [0] n_pos, [1] n_thresholds
    unsigned int* ticket;
    long long* part_u; double* part_ap; double* part_tr;
};

// carves the workspace; returns the bytes it needs (ws may be null for the query)
static int64_t rank_layout(int64_t n, char* ws, RankWs* w) {
    const int64_t ntiles = (n + RK_TILE - 1) / RK_TILE;
    WsCarver c{ws};
    w->keys_a = c.take<uint32_t>(4 * n);
    w->vals_a = c.take<int32_t>(4 * n);
    w->keys_b = c.take<uint32_t>(4 * n);
    w->vals_b = c.take<int32_t>(4 * n);
    w->sort_bytes = npi_sort_workspace_bytes(n);
    w->sort_ws = c.take<void>(w->sort_bytes);
    w->tile_status = c.take<int32_t>(4 * ntiles);
    w->tile_pos = c.take<int32_t>(4 * ntiles);
    w->tile_end = c.take<int32_t>(4 * ntiles);
    w->totals = c.take<int32_t>(8);
    w->ticket = c.take<unsigned int>(4);
    w->part_u = c.take<long long>(8 * RA_MAX_CTAS);
    w->part_ap = c.take<double>(8 * RA_MAX_CTAS);
    w->part_tr = c.take<double>(8 * RA_MAX_CTAS);
    return c.off;
}

__global__ void __launch_bounds__(RK_THREADS) rank_key_kernel(const float* __restrict__ scores, const int32_t* __restrict__ labels,
                                                              int64_t n, uint32_t* __restrict__ keys, int32_t* __restrict__ vals,
                                                              int32_t* __restrict__ tile_status, unsigned int* __restrict__ ticket) {
    const int64_t i0 = (int64_t)blockIdx.x * RK_TILE + threadIdx.x;
    int bad = 0;
#pragma unroll
    for (int q = 0; q < RK_ITEMS; ++q) {
        const int64_t i = i0 + (int64_t)q * RK_THREADS;
        if (i < n) {
            const float s = scores[i];
            const int32_t y = labels[i];
            bad |= (s != s ? 1 : 0) | (y != 0 && y != 1 ? 2 : 0);
            keys[i] = rank_key(s);
            vals[i] = y;
        }
    }
    bad = block_or_bits<2>(bad);
    if (threadIdx.x == 0) {
        tile_status[blockIdx.x] = bad;
        if (blockIdx.x == 0) *ticket = 0u;       // the caller's workspace need not be zeroed: the area kernel runs later in stream order
    }
}

// positives (low 16 bits) and run ends (high 16 bits) of items i0 .. i0 + RK_ITEMS - 1, strided by RK_THREADS
__device__ __forceinline__ int rank_flags(const uint32_t* __restrict__ keys, const int32_t* __restrict__ vals, int64_t n, int64_t i,
                                          int* pos, int* end) {
    *pos = 0; *end = 0;
    if (i >= n) return 0;
    *pos = vals[i] == 1;
    *end = (i == n - 1) || (keys[i] != keys[i + 1]);
    return *pos + (*end << 16);
}

__global__ void __launch_bounds__(RK_THREADS) rank_tile_kernel(const uint32_t* __restrict__ keys, const int32_t* __restrict__ vals, int64_t n,
                                                               int32_t* __restrict__ tile_pos, int32_t* __restrict__ tile_end) {
    __shared__ int sh[RK_THREADS / 32 + 2];
    const int64_t i0 = (int64_t)blockIdx.x * RK_TILE + (int64_t)threadIdx.x * RK_ITEMS;
    int v = 0;
#pragma unroll
    for (int q = 0; q < RK_ITEMS; ++q) { int p, e; v += rank_flags(keys, vals, n, i0 + q, &p, &e); }
    int tot;
    block_excl_scan<RK_THREADS>(v, sh, &tot);                // a tile holds at most 4096 of each: no carry across 16 bits
    if (threadIdx.x == 0) { tile_pos[blockIdx.x] = tot & 0xffff; tile_end[blockIdx.x] = tot >> 16; }
}

__global__ void __launch_bounds__(RK_THREADS) rank_scan_kernel(int32_t* __restrict__ tile_pos, int32_t* __restrict__ tile_end,
                                                               const int32_t* __restrict__ tile_status, int ntiles,
                                                               int32_t* __restrict__ totals, int32_t* __restrict__ status) {
    __shared__ int sh[RK_THREADS / 32 + 2];
    int run_p = 0, run_e = 0, st = 0;
    for (int c = 0; c < ntiles; c += RK_THREADS) {
        const int t = c + threadIdx.x;
        const int p = t < ntiles ? tile_pos[t] : 0;
        const int e = t < ntiles ? tile_end[t] : 0;
        if (t < ntiles) st |= tile_status[t];
        int tp, te;
        const int xp = block_excl_scan<RK_THREADS>(p, sh, &tp);
        const int xe = block_excl_scan<RK_THREADS>(e, sh, &te);
        if (t < ntiles) { tile_pos[t] = run_p + xp; tile_end[t] = run_e + xe; }
        run_p += tp; run_e += te;
    }
    st = block_or_bits<2>(st);
    if (threadIdx.x == 0) { totals[0] = run_p; totals[1] = run_e; *status = st; }
}

__global__ void __launch_bounds__(RK_THREADS) rank_emit_kernel(const uint32_t* __restrict__ keys, const int32_t* __restrict__ vals, int64_t n,
                                                               const int32_t* __restrict__ tile_pos, const int32_t* __restrict__ tile_end,
                                                               int32_t* __restrict__ w_tps, int32_t* __restrict__ w_fps,
                                                               float* __restrict__ thresholds, int32_t* __restrict__ tps, int32_t* __restrict__ fps) {
    __shared__ int sh[RK_THREADS / 32 + 2];
    const int64_t i0 = (int64_t)blockIdx.x * RK_TILE + (int64_t)threadIdx.x * RK_ITEMS;
    int p[RK_ITEMS], e[RK_ITEMS], v = 0;
#pragma unroll
    for (int q = 0; q < RK_ITEMS; ++q) v += rank_flags(keys, vals, n, i0 + q, &p[q], &e[q]);
    int tot;
    const int ex = block_excl_scan<RK_THREADS>(v, sh, &tot);
    int cp = tile_pos[blockIdx.x] + (ex & 0xffff);
    int ce = tile_end[blockIdx.x] + (ex >> 16);
#pragma unroll
    for (int q = 0; q < RK_ITEMS; ++q) {
        cp += p[q];
        if (e[q]) {
            const int64_t i = i0 + q;
            const int32_t t = cp, f = (int32_t)(i + 1 - cp);
            w_tps[ce] = t; w_fps[ce] = f;
            if (tps) tps[ce] = t;
            if (fps) fps[ce] = f;
            if (thresholds) thresholds[ce] = rank_score(keys[i]);
            ++ce;
        }
    }
}

__global__ void __launch_bounds__(RA_THREADS) rank_area_kernel(const int32_t* __restrict__ w_tps, const int32_t* __restrict__ w_fps, int64_t n,
                                                               const int32_t* __restrict__ totals, long long* __restrict__ part_u,
                                                               double* __restrict__ part_ap, double* __restrict__ part_tr,
                                                               unsigned int* __restrict__ ticket, int64_t* __restrict__ summary,
                                                               double* __restrict__ areas) {
    __shared__ long long sh_u[RA_THREADS / 32];
    __shared__ double sh_d[RA_THREADS / 32];
    const int T = totals[1];
    long long u = 0;
    double ap = 0.0, tr = 0.0;
    for (int64_t r = (int64_t)blockIdx.x * RA_THREADS + threadIdx.x; r < T; r += (int64_t)gridDim.x * RA_THREADS) {
        const int t = w_tps[r], f = w_fps[r];
        const int tp = r > 0 ? w_tps[r - 1] : 0, fp = r > 0 ? w_fps[r - 1] : 0;
        u += (long long)(f - fp) * (long long)(t + tp);
        if (t != tp) {
            const double prec = (double)t / (double)(t + f);
            const double prev = r > 0 ? (double)tp / (double)(tp + fp) : 1.0;   // precision_recall_curve's end point (0, 1)
            ap += (double)(t - tp) * prec;
            tr += (double)(t - tp) * (prec + prev);
        }
    }
    u = block_sum<RA_THREADS>(u, sh_u);
    ap = block_sum<RA_THREADS>(ap, sh_d);
    tr = block_sum<RA_THREADS>(tr, sh_d);
    if (threadIdx.x == 0) { part_u[blockIdx.x] = u; part_ap[blockIdx.x] = ap; part_tr[blockIdx.x] = tr; }
    if (!last_cta(ticket)) return;
    u = 0; ap = 0.0; tr = 0.0;
    for (int b = threadIdx.x; b < (int)gridDim.x; b += RA_THREADS) {      // CTA b always lands in thread b % 256, in order
        u += __ldcg(&part_u[b]); ap += __ldcg(&part_ap[b]); tr += __ldcg(&part_tr[b]);
    }
    u = block_sum<RA_THREADS>(u, sh_u);
    ap = block_sum<RA_THREADS>(ap, sh_d);
    tr = block_sum<RA_THREADS>(tr, sh_d);
    if (threadIdx.x == 0) {
        const int64_t n_pos = totals[0];
        summary[0] = n_pos; summary[1] = n - n_pos; summary[2] = T; summary[3] = u;
        areas[0] = ap / (double)n_pos;
        areas[1] = 0.5 * tr / (double)n_pos;
    }
}

}  // namespace npi

using namespace npi;

extern "C" int64_t npi_rank_workspace_bytes(int64_t n_max) {
    RankWs w;
    return rank_layout(n_max > 0 ? n_max : 1, nullptr, &w);
}

extern "C" int npi_rank_curve(const float* scores, const int32_t* labels, int64_t n, int64_t* summary, double* areas,
                              float* thresholds, int32_t* tps, int32_t* fps, int32_t* status,
                              void* workspace, int64_t workspace_bytes, npi_stream_t stream) {
    NPI_REQUIRE(scores && labels && summary && areas && status && workspace, "rank_curve: null argument");
    NPI_REQUIRE(n >= 1 && n < (int64_t)1 << 31, "rank_curve: n = %lld out of range [1, 2^31)", (long long)n);
    NPI_REQUIRE(workspace_bytes >= npi_rank_workspace_bytes(n), "rank_curve: workspace of %lld bytes, %lld needed",
                (long long)workspace_bytes, (long long)npi_rank_workspace_bytes(n));
    cudaStream_t st = (cudaStream_t)stream;
    RankWs w;
    rank_layout(n, (char*)workspace, &w);
    const int ntiles = (int)((n + RK_TILE - 1) / RK_TILE);
    rank_key_kernel<<<ntiles, RK_THREADS, 0, st>>>(scores, labels, n, w.keys_a, w.vals_a, w.tile_status, w.ticket);
    NPI_CHECK_LAUNCH();
    SortedPairs sp;
    int rc = sort_pairs(w.keys_a, w.vals_a, w.keys_b, w.vals_b, n, 32, w.sort_ws, w.sort_bytes, st, &sp);
    if (rc != NPI_OK) return rc;
    int32_t* w_tps = (int32_t*)sp.free_keys;                         // the sort's other buffer pair holds the curve
    int32_t* w_fps = sp.free_vals;
    rank_tile_kernel<<<ntiles, RK_THREADS, 0, st>>>(sp.keys, sp.vals, n, w.tile_pos, w.tile_end);
    NPI_CHECK_LAUNCH();
    rank_scan_kernel<<<1, RK_THREADS, 0, st>>>(w.tile_pos, w.tile_end, w.tile_status, ntiles, w.totals, status);
    NPI_CHECK_LAUNCH();
    rank_emit_kernel<<<ntiles, RK_THREADS, 0, st>>>(sp.keys, sp.vals, n, w.tile_pos, w.tile_end, w_tps, w_fps, thresholds, tps, fps);
    NPI_CHECK_LAUNCH();
    const int64_t want = (n + 8 * RA_THREADS - 1) / (8 * RA_THREADS);
    const int actas = (int)(want < RA_MAX_CTAS ? want : RA_MAX_CTAS);
    rank_area_kernel<<<actas, RA_THREADS, 0, st>>>(w_tps, w_fps, n, w.totals, w.part_u, w.part_ap, w.part_tr, w.ticket, summary, areas);
    NPI_CHECK_LAUNCH();
    return NPI_OK;
}
