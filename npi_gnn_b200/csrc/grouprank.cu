// Filtered rank of every held-out interaction among its node's candidates (npi_group_rank) -- MRR, Hits@K and the
// per-node ROC AUC of a scoring sweep: for each RNA, where do its true partners rank among all the proteins it could pair
// with (and for each protein among its RNAs), the question of the reference's case studies (src/case_study.py,
// src/case_study_negativeSample.py).  Semantics: include/npi.h.
//
//   gr_key_kernel        (rank_key(score), position) pairs; per-tile status bits (NaN score, label not 0/1, group id out
//                        of range); resets the ticket
//   npi_sort_pairs_u32   32 key bits: descending score, ties by ascending position (sort.cu)
//   gr_gather_kernel     (group id, position | query << 31) in that order
//   npi_sort_pairs_u32   ceil(log2 num_groups) key bits, stable: the items are now sorted by (group, descending score)
//   topk_bounds_kernel   gptr[g] = first sorted item of group g; the status word (topk.cu)
//   gr_flags_kernel      score key and competitor flag of every sorted item
//   exclusive scan       cumneg[j] = competitors among the sorted items [0, j), three launches (sort.cu)
//   gr_group_kernel      n_pos, n_neg and twice_u = 2 n_pos n_neg per group; per-CTA counts of ranked and unranked
//                        queries and of scored groups
//   gr_emit_kernel       per item: its tie run [lo, hi) inside the group (binary search), above / tied from cumneg,
//                        written at the item's position.  At a run end whose run holds queries: the run's term of sum_rr
//                        and of hits into per-CTA partials, and -npos_run (2 above + tied) into twice_u[g] (an integer
//                        atomic); the last CTA (ticket) combines the partials in a fixed order
// Only run ends contribute to sum_rr, hits and twice_u, and the sorted index of a run end and its counts do not depend on
// the order of the input, so every output is bit-identical on reruns and under any permutation of the input.  No
// floating-point atomics, no host synchronisation.
#include "common.cuh"

namespace npi {

constexpr int GR_THREADS = 1024;
constexpr int GR_ITEMS = 4;
constexpr int GR_TILE = GR_THREADS * GR_ITEMS;     // 4096 items per CTA
constexpr int GG_THREADS = 256;                    // groups per CTA of gr_group_kernel
constexpr int GR_MAXH = 8;                         // Hits@K cut-offs per call

struct GrHits { int32_t k[GR_MAXH]; int32_t n; };

struct GrWs {
    // n + 1 entries each: the pair the second sort leaves free holds the sorted score keys and cumneg[0 .. n]
    uint32_t* keys_a; int32_t* vals_a; uint32_t* keys_b; int32_t* vals_b;
    void* sort_ws; int64_t sort_bytes;
    int32_t* neg;                       // [n] competitor flags in sorted order, the input of the scan
    int32_t* tile_status; int32_t* scan_tiles;
    int32_t* gptr;                      // [num_groups + 1]
    int32_t* gpart;                     // [3][group CTAs]: ranked queries, unranked queries, scored groups
    unsigned int* ticket;
    double* part_rr;                    // [item tiles]
    int32_t* part_hits;                 // [GR_MAXH][item tiles]
};

// carves the workspace; returns the bytes it needs (ws may be null for the query)
static int64_t group_rank_layout(int64_t n, int32_t num_groups, char* ws, GrWs* w) {
    const int64_t ntiles = (n + GR_TILE - 1) / GR_TILE;
    const int64_t gctas = ((int64_t)num_groups + GG_THREADS - 1) / GG_THREADS;
    WsCarver c{ws};
    w->keys_a = c.take<uint32_t>(4 * (n + 1));
    w->vals_a = c.take<int32_t>(4 * (n + 1));
    w->keys_b = c.take<uint32_t>(4 * (n + 1));
    w->vals_b = c.take<int32_t>(4 * (n + 1));
    w->sort_bytes = npi_sort_workspace_bytes(n);
    w->sort_ws = c.take<void>(w->sort_bytes);
    w->neg = c.take<int32_t>(4 * n);
    w->tile_status = c.take<int32_t>(4 * ntiles);
    w->scan_tiles = c.take<int32_t>(4 * ntiles);
    w->gptr = c.take<int32_t>(4 * ((int64_t)num_groups + 1));
    w->gpart = c.take<int32_t>(4 * 3 * gctas);
    w->ticket = c.take<unsigned int>(4);
    w->part_rr = c.take<double>(8 * ntiles);
    w->part_hits = c.take<int32_t>(4 * GR_MAXH * ntiles);
    return c.off;
}

__global__ void __launch_bounds__(GR_THREADS) gr_key_kernel(const float* __restrict__ scores, const int32_t* __restrict__ labels,
                                                            const int32_t* __restrict__ group, int64_t n, int32_t num_groups,
                                                            uint32_t* __restrict__ keys, int32_t* __restrict__ vals,
                                                            int32_t* __restrict__ tile_status, unsigned int* __restrict__ ticket) {
    const int64_t i0 = (int64_t)blockIdx.x * GR_TILE + threadIdx.x;
    int bad = 0;
#pragma unroll
    for (int q = 0; q < GR_ITEMS; ++q) {
        const int64_t i = i0 + (int64_t)q * GR_THREADS;
        if (i < n) {
            const float s = scores[i];
            const int32_t y = labels[i], g = group[i];
            bad |= (s != s ? 1 : 0) | (y != 0 && y != 1 ? 2 : 0) | (g < 0 || g >= num_groups ? 4 : 0);
            keys[i] = rank_key(s);
            vals[i] = (int32_t)i;
        }
    }
    bad = block_or_bits<3>(bad);
    if (threadIdx.x == 0) {
        tile_status[blockIdx.x] = bad;
        if (blockIdx.x == 0) *ticket = 0u;       // the caller's workspace need not be zeroed: the emit kernel runs later in stream order
    }
}

// the score-sorted positions -> (group id, position | query << 31); an id out of range becomes 0 so that every later access
// stays in bounds (the status marks the result void)
__global__ void __launch_bounds__(GR_THREADS) gr_gather_kernel(const int32_t* __restrict__ pos, const int32_t* __restrict__ labels,
                                                               const int32_t* __restrict__ group, int64_t n, int32_t num_groups,
                                                               uint32_t* __restrict__ gkeys, int32_t* __restrict__ gvals) {
    const int64_t j0 = (int64_t)blockIdx.x * GR_TILE + threadIdx.x;
#pragma unroll
    for (int q = 0; q < GR_ITEMS; ++q) {
        const int64_t j = j0 + (int64_t)q * GR_THREADS;
        if (j < n) {
            const int32_t p = pos[j];
            const int32_t g = __ldg(group + p);
            gkeys[j] = (g < 0 || g >= num_groups) ? 0u : (uint32_t)g;
            gvals[j] = (int32_t)((uint32_t)p | (__ldg(labels + p) == 1 ? 0x80000000u : 0u));
        }
    }
}

__global__ void __launch_bounds__(GR_THREADS) gr_flags_kernel(const int32_t* __restrict__ gvals, const float* __restrict__ scores, int64_t n,
                                                              uint32_t* __restrict__ skey, int32_t* __restrict__ neg) {
    const int64_t j0 = (int64_t)blockIdx.x * GR_TILE + threadIdx.x;
#pragma unroll
    for (int q = 0; q < GR_ITEMS; ++q) {
        const int64_t j = j0 + (int64_t)q * GR_THREADS;
        if (j < n) {
            const int32_t v = gvals[j];
            skey[j] = rank_key(__ldg(scores + (v & 0x7fffffff)));
            neg[j] = v >= 0;
        }
    }
}

__global__ void __launch_bounds__(GG_THREADS) gr_group_kernel(const int32_t* __restrict__ gptr, const int32_t* __restrict__ cumneg,
                                                              int32_t num_groups, int32_t* __restrict__ n_pos, int32_t* __restrict__ n_neg,
                                                              int64_t* __restrict__ twice_u, int32_t* __restrict__ gpart) {
    __shared__ int sh[GG_THREADS / 32];
    const int64_t g = (int64_t)blockIdx.x * GG_THREADS + threadIdx.x;
    int ranked = 0, unranked = 0, scored = 0;
    if (g < num_groups) {
        const int gs = gptr[g], ge = gptr[g + 1];
        const int nn = cumneg[ge] - cumneg[gs], np = ge - gs - nn;
        n_pos[g] = np;
        n_neg[g] = nn;
        twice_u[g] = 2 * (int64_t)np * nn;                         // gr_emit_kernel subtracts what the queries lose
        if (nn > 0) ranked = np; else unranked = np;
        scored = np > 0 && nn > 0;
    }
    ranked = block_sum<GG_THREADS>(ranked, sh);
    unranked = block_sum<GG_THREADS>(unranked, sh);
    scored = block_sum<GG_THREADS>(scored, sh);
    if (threadIdx.x == 0) {
        gpart[blockIdx.x] = ranked;
        gpart[gridDim.x + blockIdx.x] = unranked;
        gpart[2 * gridDim.x + blockIdx.x] = scored;
    }
}

__global__ void __launch_bounds__(GR_THREADS) gr_emit_kernel(const uint32_t* __restrict__ gkeys, const int32_t* __restrict__ gvals,
                                                             const uint32_t* __restrict__ skey, const int32_t* __restrict__ cumneg,
                                                             const int32_t* __restrict__ gptr, int64_t n, GrHits hk,
                                                             int32_t* __restrict__ above_out, int32_t* __restrict__ tied_out,
                                                             int64_t* __restrict__ twice_u, double* __restrict__ part_rr,
                                                             int32_t* __restrict__ part_hits, const int32_t* __restrict__ gpart, int gctas,
                                                             unsigned int* __restrict__ ticket, int64_t* __restrict__ summary,
                                                             double* __restrict__ sum_rr) {
    __shared__ double sh_d[GR_THREADS / 32];
    __shared__ long long sh_l[GR_THREADS / 32];
    __shared__ int sh_i[GR_THREADS / 32];
    const int ntiles = (int)gridDim.x;
    const int64_t j0 = (int64_t)blockIdx.x * GR_TILE + threadIdx.x;
    double rr = 0.0;
    int hits[GR_MAXH];
#pragma unroll
    for (int h = 0; h < GR_MAXH; ++h) hits[h] = 0;
#pragma unroll 1
    for (int q = 0; q < GR_ITEMS; ++q) {
        const int64_t j = j0 + (int64_t)q * GR_THREADS;
        if (j >= n) break;
        const int32_t v = gvals[j];
        const bool query = v < 0;
        const uint32_t g = gkeys[j];
        const int gs = gptr[g], ge = gptr[g + 1];
        const uint32_t k = skey[j];
        const bool end = j + 1 == ge || skey[j + 1] != k;
        int32_t a = -1, t = -1;
        if (query || end) {
            int lo = (int)j, hi = (int)j + 1;
            if (lo > gs && skey[lo - 1] == k) {                    // first member of the run: lower bound of k in [gs, j)
                int L = gs, R = (int)j;
                while (L < R) { const int m = (L + R) >> 1; if (skey[m] < k) L = m + 1; else R = m; }
                lo = L;
            }
            if (!end) {                                            // one past the run: upper bound of k in [j + 1, ge)
                int L = (int)j + 1, R = ge;
                while (L < R) { const int m = (L + R) >> 1; if (skey[m] <= k) L = m + 1; else R = m; }
                hi = L;
            }
            const int c0 = cumneg[gs], cl = cumneg[lo], ch = cumneg[hi];
            a = cl - c0;
            t = ch - cl;
            const int npos_run = hi - lo - t;
            if (end && npos_run > 0) {
                const long long lost = (long long)npos_run * (2 * (long long)a + t);
                if (lost) atomicAdd(reinterpret_cast<unsigned long long*>(twice_u + g), (unsigned long long)(-lost));
                if (cumneg[ge] > c0) {                             // the group has a competitor: its queries are ranked
                    const long long twice_rank = 2 * (long long)a + t + 2;
                    rr += (double)npos_run * (2.0 / (double)twice_rank);
#pragma unroll
                    for (int h = 0; h < GR_MAXH; ++h)
                        if (h < hk.n && twice_rank <= 2 * (long long)hk.k[h]) hits[h] += npos_run;
                }
            }
        }
        const int32_t p = v & 0x7fffffff;
        if (above_out) above_out[p] = query ? a : -1;
        if (tied_out) tied_out[p] = query ? t : -1;
    }

    rr = block_sum<GR_THREADS>(rr, sh_d);
    if (threadIdx.x == 0) part_rr[blockIdx.x] = rr;
#pragma unroll
    for (int h = 0; h < GR_MAXH; ++h) {
        if (h < hk.n) {
            const int s = block_sum<GR_THREADS>(hits[h], sh_i);      // <= 4096: the tile's items
            if (threadIdx.x == 0) part_hits[(int64_t)h * ntiles + blockIdx.x] = s;
        }
    }
    if (!last_cta(ticket)) return;
    rr = 0.0;
    for (int b = threadIdx.x; b < ntiles; b += GR_THREADS) rr += __ldcg(&part_rr[b]);     // CTA b always lands in thread b % 1024, in order
    rr = block_sum<GR_THREADS>(rr, sh_d);
    if (threadIdx.x == 0) *sum_rr = rr;
#pragma unroll
    for (int h = 0; h < GR_MAXH; ++h) {
        if (h < hk.n) {
            long long s = 0;
            for (int b = threadIdx.x; b < ntiles; b += GR_THREADS) s += __ldcg(&part_hits[(int64_t)h * ntiles + b]);
            s = block_sum<GR_THREADS>(s, sh_l);
            if (threadIdx.x == 0) summary[3 + h] = s;
        }
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) {                                  // ranked queries, unranked queries, scored groups
        long long s = 0;
        for (int b = threadIdx.x; b < gctas; b += GR_THREADS) s += gpart[(int64_t)c * gctas + b];
        s = block_sum<GR_THREADS>(s, sh_l);
        if (threadIdx.x == 0) summary[c] = s;
    }
}

}  // namespace npi

using namespace npi;

extern "C" int64_t npi_group_rank_workspace_bytes(int64_t n_max, int32_t num_groups) {
    GrWs w;
    return group_rank_layout(n_max > 0 ? n_max : 1, num_groups > 0 ? num_groups : 1, nullptr, &w);
}

extern "C" int npi_group_rank(const float* scores, const int32_t* labels, const int32_t* group, int64_t n, int32_t num_groups,
                              const int32_t* hits_k, int32_t n_hits, int32_t* n_pos, int32_t* n_neg, int64_t* twice_u,
                              int64_t* summary, double* sum_rr, int32_t* above, int32_t* tied, int32_t* status,
                              void* workspace, int64_t workspace_bytes, npi_stream_t stream) {
    NPI_REQUIRE(scores && labels && group && hits_k && n_pos && n_neg && twice_u && summary && sum_rr && status && workspace,
                "group_rank: null argument");
    NPI_REQUIRE(n >= 1 && n < (int64_t)1 << 31, "group_rank: n = %lld out of range [1, 2^31)", (long long)n);
    NPI_REQUIRE(num_groups >= 1 && num_groups < (1 << 24), "group_rank: num_groups = %d out of range [1, 2^24)", num_groups);
    NPI_REQUIRE(n_hits >= 1 && n_hits <= GR_MAXH, "group_rank: n_hits = %d out of range [1, %d]", n_hits, GR_MAXH);
    GrHits hk = {};
    hk.n = n_hits;
    for (int h = 0; h < n_hits; ++h) {
        NPI_REQUIRE(hits_k[h] >= 1, "group_rank: hits K = %d must be >= 1", hits_k[h]);
        hk.k[h] = hits_k[h];
    }
    NPI_REQUIRE(workspace_bytes >= npi_group_rank_workspace_bytes(n, num_groups), "group_rank: workspace of %lld bytes, %lld needed",
                (long long)workspace_bytes, (long long)npi_group_rank_workspace_bytes(n, num_groups));
    cudaStream_t st = (cudaStream_t)stream;
    GrWs w;
    group_rank_layout(n, num_groups, (char*)workspace, &w);
    const int ntiles = (int)((n + GR_TILE - 1) / GR_TILE);
    const int gctas = (int)(((int64_t)num_groups + GG_THREADS - 1) / GG_THREADS);
    gr_key_kernel<<<ntiles, GR_THREADS, 0, st>>>(scores, labels, group, n, num_groups, w.keys_a, w.vals_a, w.tile_status, w.ticket);
    NPI_CHECK_LAUNCH();
    SortedPairs by_score, by_group;
    int rc = sort_pairs(w.keys_a, w.vals_a, w.keys_b, w.vals_b, n, 32, w.sort_ws, w.sort_bytes, st, &by_score);
    if (rc != NPI_OK) return rc;
    gr_gather_kernel<<<ntiles, GR_THREADS, 0, st>>>(by_score.vals, labels, group, n, num_groups, by_score.free_keys,
                                                    by_score.free_vals);
    NPI_CHECK_LAUNCH();
    rc = sort_pairs(by_score.free_keys, by_score.free_vals, by_score.keys, by_score.vals, n, group_bits(num_groups), w.sort_ws,
                    w.sort_bytes, st, &by_group);
    if (rc != NPI_OK) return rc;
    const uint32_t* gkeys = by_group.keys;
    const int32_t* gvals = by_group.vals;
    uint32_t* skey = by_group.free_keys;                          // the free pair: sorted score keys and cumneg
    int32_t* cumneg = by_group.free_vals;
    rc = launch_group_bounds(gkeys, n, num_groups, w.tile_status, ntiles, w.gptr, status, st);
    if (rc != NPI_OK) return rc;
    gr_flags_kernel<<<ntiles, GR_THREADS, 0, st>>>(gvals, scores, n, skey, w.neg);
    NPI_CHECK_LAUNCH();
    rc = launch_excl_scan_i32(w.neg, n, cumneg, cumneg + n, w.scan_tiles, st);
    if (rc != NPI_OK) return rc;
    gr_group_kernel<<<gctas, GG_THREADS, 0, st>>>(w.gptr, cumneg, num_groups, n_pos, n_neg, twice_u, w.gpart);
    NPI_CHECK_LAUNCH();
    gr_emit_kernel<<<ntiles, GR_THREADS, 0, st>>>(gkeys, gvals, skey, cumneg, w.gptr, n, hk, above, tied, twice_u, w.part_rr,
                                                 w.part_hits, w.gpart, gctas, w.ticket, summary, sum_rr);
    NPI_CHECK_LAUNCH();
    return NPI_OK;
}
