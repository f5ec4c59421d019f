// Top-K of scored items per group (npi_group_topk) -- the ranking a case study reads off a scoring sweep (the
// reference's src/case_study_negativeSample.py / src/case_study.py): for every RNA its most likely protein partners,
// for every protein its most likely RNAs.  Semantics: include/npi.h.
//
//   topk_key_kernel     (group id, position) pairs; per-tile status bits (NaN score, group id out of range)
//   npi_sort_pairs_u32  ceil(log2 num_groups) key bits (sort.cu); stable, so the members of a group stay in ascending
//                       position
//   topk_bounds_kernel  gptr[g] = first sorted item of group g (binary search: empty groups need no special case);
//                       the status word
//   group_topk_kernel   one CTA per group: MSB-first radix select of the k-th smallest score key (rank_key: ascending
//                       key = descending score), then every member strictly below it plus the first members equal to
//                       it in position order (block scan), then a bitonic sort of the <= k winners by (key, position)
// The members taken and their order depend on the scores and positions only, never on scheduling: outputs are
// bit-identical on reruns.  No floating-point atomics, no host synchronisation.
#include "common.cuh"

namespace npi {

constexpr int TK_THREADS = 256;         // one bin of the 8-bit digit histogram per thread
constexpr int TK_MAXK = 1024;
// The score keys of a group of up to TK_STAGE members are staged once in shared memory; a larger group rereads its
// slice from global memory on every radix pass.  Sized for four CTAs per SM in the 228 KB of an SM (up to 227 KB for
// one block, 1 KB reserved per CTA): 4 * (47,104 B of stage + 9.3 KB static + 1 KB) <= 233,472 B.
constexpr int TK_STAGE = 11776;
constexpr int KK_THREADS = 1024;
constexpr int KK_ITEMS = 4;
constexpr int KK_TILE = KK_THREADS * KK_ITEMS;
constexpr int TB_THREADS = 256;

struct TopkWs {
    uint32_t* keys_a; int32_t* vals_a; uint32_t* keys_b; int32_t* vals_b;
    void* sort_ws; int64_t sort_bytes;
    int32_t* tile_status;
    int32_t* gptr;                      // [num_groups + 1]
};

// carves the workspace; returns the bytes it needs (ws may be null for the query)
static int64_t topk_layout(int64_t n, int32_t num_groups, char* ws, TopkWs* w) {
    const int64_t ntiles = (n + KK_TILE - 1) / KK_TILE;
    WsCarver c{ws};
    w->keys_a = c.take<uint32_t>(4 * n);
    w->vals_a = c.take<int32_t>(4 * n);
    w->keys_b = c.take<uint32_t>(4 * n);
    w->vals_b = c.take<int32_t>(4 * n);
    w->sort_bytes = npi_sort_workspace_bytes(n);
    w->sort_ws = c.take<void>(w->sort_bytes);
    w->tile_status = c.take<int32_t>(4 * ntiles);
    w->gptr = c.take<int32_t>(4 * ((int64_t)num_groups + 1));
    return c.off;
}

__global__ void __launch_bounds__(KK_THREADS) topk_key_kernel(const float* __restrict__ scores, const int32_t* __restrict__ group,
                                                              int64_t n, int32_t num_groups, uint32_t* __restrict__ keys,
                                                              int32_t* __restrict__ vals, int32_t* __restrict__ tile_status) {
    const int64_t i0 = (int64_t)blockIdx.x * KK_TILE + threadIdx.x;
    int bad = 0;
#pragma unroll
    for (int q = 0; q < KK_ITEMS; ++q) {
        const int64_t i = i0 + (int64_t)q * KK_THREADS;
        if (i < n) {
            const float s = scores[i];
            const int32_t g = group[i];
            const bool out = g < 0 || g >= num_groups;
            bad |= (s != s ? 1 : 0) | (out ? 2 : 0);
            keys[i] = out ? 0u : (uint32_t)g;      // keeps every later access in bounds; the status marks the result void
            vals[i] = (int32_t)i;
        }
    }
    bad = block_or_bits<2>(bad);
    if (threadIdx.x == 0) tile_status[blockIdx.x] = bad;
}

__global__ void __launch_bounds__(TB_THREADS) topk_bounds_kernel(const uint32_t* __restrict__ keys, int64_t n, int32_t num_groups,
                                                                 const int32_t* __restrict__ tile_status, int ntiles,
                                                                 int32_t* __restrict__ gptr, int32_t* __restrict__ status) {
    const int64_t g = (int64_t)blockIdx.x * TB_THREADS + threadIdx.x;
    if (g <= num_groups) {
        int64_t lo = 0, hi = n;                       // first sorted item with key >= g
        while (lo < hi) {
            const int64_t mid = (lo + hi) >> 1;
            if (keys[mid] < (uint32_t)g) lo = mid + 1; else hi = mid;
        }
        gptr[g] = (int32_t)lo;
    }
    if (blockIdx.x == 0) {
        int st = 0;
        for (int t = threadIdx.x; t < ntiles; t += TB_THREADS) st |= tile_status[t];
        st = block_or_bits<3>(st);
        if (threadIdx.x == 0) *status = st;
    }
}

int launch_group_bounds(const uint32_t* keys, int64_t n, int32_t num_groups, const int32_t* tile_status, int ntiles,
                        int32_t* gptr, int32_t* status, cudaStream_t st) {
    topk_bounds_kernel<<<(int)(((int64_t)num_groups + TB_THREADS) / TB_THREADS), TB_THREADS, 0, st>>>(keys, n, num_groups, tile_status,
                                                                                                     ntiles, gptr, status);
    NPI_CHECK_LAUNCH();
    return NPI_OK;
}

__global__ void __launch_bounds__(TK_THREADS) group_topk_kernel(const float* __restrict__ scores, const int32_t* __restrict__ pos_sorted,
                                                                const int32_t* __restrict__ gptr, int32_t k,
                                                                int32_t* __restrict__ out_pos, float* __restrict__ out_score,
                                                                int32_t* __restrict__ out_count) {
    extern __shared__ uint32_t stage[];                  // TK_STAGE score keys
    __shared__ unsigned long long win[TK_MAXK];          // (key << 32) | position of the winners
    __shared__ int hist[256];
    __shared__ int sh[TK_THREADS / 32 + 2];
    __shared__ uint32_t s_prefix;
    __shared__ int s_rem, s_done;
    const int tid = threadIdx.x, lane = tid & 31;
    const int g = blockIdx.x;
    const int base = gptr[g], c = gptr[g + 1] - base;
    const int kk = c < k ? c : k;
    const int32_t* __restrict__ pos = pos_sorted + base;
    const bool staged = c <= TK_STAGE;
    auto key_at = [&](int j) -> uint32_t { return staged ? stage[j] : rank_key(__ldg(scores + __ldg(pos + j))); };

    if (staged)
        for (int j = tid; j < c; j += TK_THREADS) stage[j] = rank_key(__ldg(scores + __ldg(pos + j)));
    __syncthreads();

    // Radix select, 8 bits at a time from the top: the kk-th smallest key agrees with `prefix` in the bits above `lo`,
    // and `rem` of the members that agree there are taken.  It stops early once every member of the chosen digit is
    // taken.  With c <= k nothing is selected: lo = 32 and every member is an "equal" one.
    uint32_t prefix = 0u;
    int lo = 32, rem = kk;
    if (c > k) {
        for (int lo_next = 24; ; lo_next -= 8) {
            hist[tid] = 0;
            __syncthreads();
            for (int j0 = 0; j0 < c; j0 += TK_THREADS) {
                const int j = j0 + tid;
                uint32_t key = 0u;
                bool in = false;
                if (j < c) { key = key_at(j); in = ((uint64_t)key >> lo) == ((uint64_t)prefix >> lo); }
                const unsigned act = __ballot_sync(0xffffffffu, in);
                if (in) {                                // one shared-memory atomic per distinct digit of the warp
                    const uint32_t d = (key >> lo_next) & 255u;
                    const unsigned peers = __match_any_sync(act, d);
                    if ((peers & ((1u << lane) - 1u)) == 0) atomicAdd(&hist[d], __popc(peers));
                }
            }
            __syncthreads();
            const int h = hist[tid];
            int tot;
            const int ex = block_excl_scan<TK_THREADS>(h, sh, &tot);
            if (ex < rem && ex + h >= rem) {             // exactly one digit holds the rem-th member
                s_prefix = prefix | ((uint32_t)tid << lo_next);
                s_rem = rem - ex;
                s_done = (h == rem - ex) || lo_next == 0;
            }
            __syncthreads();
            prefix = s_prefix; rem = s_rem; lo = lo_next;
            if (s_done) break;
        }
    }

    // Take: members below the prefix all win (n_strict of them); of the members equal to it, the first rem in position
    // order.  The block scan numbers both kinds in position order, so the slots do not depend on scheduling.
    const int n_strict = kk - rem;
    const uint64_t pre = (uint64_t)prefix >> lo;
    int carry_s = 0, carry_e = 0;
    for (int j0 = 0; j0 < c && (carry_s < n_strict || carry_e < rem); j0 += TK_THREADS) {
        const int j = j0 + tid;
        int s = 0, e = 0;
        uint32_t key = 0u;
        if (j < c) {
            key = key_at(j);
            const uint64_t a = (uint64_t)key >> lo;
            s = a < pre; e = a == pre;
        }
        int tot;
        const int ex = block_excl_scan<TK_THREADS>(s | (e << 16), sh, &tot);     // <= 256 of each: no carry across 16 bits
        int slot = -1;
        if (s) slot = carry_s + (ex & 0xffff);
        else if (e && carry_e + (ex >> 16) < rem) slot = n_strict + carry_e + (ex >> 16);
        if (slot >= 0) win[slot] = ((unsigned long long)key << 32) | (uint32_t)__ldg(pos + j);
        carry_s += tot & 0xffff;
        carry_e += tot >> 16;
    }

    // bitonic sort of the winners by (key, position), padded to a power of two
    int m = 1;
    while (m < kk) m <<= 1;
    for (int t = kk + tid; t < m; t += TK_THREADS) win[t] = ~0ull;
    __syncthreads();
    for (int size = 2; size <= m; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int t = tid; t < (m >> 1); t += TK_THREADS) {
                const int i = 2 * t - (t & (stride - 1));
                const unsigned long long a = win[i], b = win[i + stride];
                if ((a > b) == ((i & size) == 0)) { win[i] = b; win[i + stride] = a; }
            }
            __syncthreads();
        }
    }

    const int64_t row = (int64_t)g * k;
    for (int r = tid; r < k; r += TK_THREADS) {
        int32_t p = -1;
        float v = __uint_as_float(0x7fc00000u);
        if (r < kk) { p = (int32_t)(uint32_t)win[r]; v = __ldg(scores + p); }
        out_pos[row + r] = p;
        out_score[row + r] = v;
    }
    if (tid == 0) out_count[g] = kk;
}

}  // namespace npi

using namespace npi;

extern "C" int64_t npi_group_topk_workspace_bytes(int64_t n_max, int32_t num_groups) {
    TopkWs w;
    return topk_layout(n_max > 0 ? n_max : 1, num_groups > 0 ? num_groups : 1, nullptr, &w);
}

extern "C" int npi_group_topk(const float* scores, const int32_t* group, int64_t n, int32_t num_groups, int32_t k,
                              int32_t* out_pos, float* out_score, int32_t* out_count, int32_t* status,
                              void* workspace, int64_t workspace_bytes, npi_stream_t stream) {
    NPI_REQUIRE(scores && group && out_pos && out_score && out_count && status && workspace, "group_topk: null argument");
    NPI_REQUIRE(n >= 1 && n < (int64_t)1 << 31, "group_topk: n = %lld out of range [1, 2^31)", (long long)n);
    NPI_REQUIRE(num_groups >= 1 && num_groups < (1 << 24), "group_topk: num_groups = %d out of range [1, 2^24)", num_groups);
    NPI_REQUIRE(k >= 1 && k <= TK_MAXK, "group_topk: k = %d out of range [1, %d]", k, TK_MAXK);
    NPI_REQUIRE(workspace_bytes >= npi_group_topk_workspace_bytes(n, num_groups), "group_topk: workspace of %lld bytes, %lld needed",
                (long long)workspace_bytes, (long long)npi_group_topk_workspace_bytes(n, num_groups));
    cudaStream_t st = (cudaStream_t)stream;
    TopkWs w;
    topk_layout(n, num_groups, (char*)workspace, &w);
    const int ntiles = (int)((n + KK_TILE - 1) / KK_TILE);
    topk_key_kernel<<<ntiles, KK_THREADS, 0, st>>>(scores, group, n, num_groups, w.keys_a, w.vals_a, w.tile_status);
    NPI_CHECK_LAUNCH();
    const int bits = group_bits(num_groups);
    SortedPairs sp;
    int rc = sort_pairs(w.keys_a, w.vals_a, w.keys_b, w.vals_b, n, bits, w.sort_ws, w.sort_bytes, st, &sp);
    if (rc != NPI_OK) return rc;
    rc = launch_group_bounds(sp.keys, n, num_groups, w.tile_status, ntiles, w.gptr, status, st);
    if (rc != NPI_OK) return rc;
    static OncePerDevice once;
    if (once.need())
        NPI_CHECK_CUDA(cudaFuncSetAttribute(group_topk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TK_STAGE * 4));
    group_topk_kernel<<<num_groups, TK_THREADS, TK_STAGE * 4, st>>>(scores, sp.vals, w.gptr, k, out_pos, out_score, out_count);
    NPI_CHECK_LAUNCH();
    return NPI_OK;
}
