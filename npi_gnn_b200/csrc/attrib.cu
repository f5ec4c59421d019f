// Input attribution of scored pairs (npi_input_attribution): the gradient of a pair's target with respect to the layer-1
// input rows of its enclosing subgraph, and gradient x input summed per row and per (pair, feature).  Semantics:
// include/npi.h.
//
// The unit of work is a chunk: AT_ROWS consecutive rows of ONE pair, counted from the pair's first row (a pair of n
// rows has ceil(n / AT_ROWS) chunks).  Chunks start at the pair, not at a multiple of AT_ROWS in the batch, so every sum
// groups a pair's rows the same way wherever the pair sits in its batch: a pair gives the same bits in any batch.
//   attrib_chunks_kernel  one CTA: chunk_ptr[p] = chunks of the pairs before p (block scan in steps of 1024 pairs)
//   attrib_rows_kernel    persistent CTAs (one per SM), conv1.weight staged once per CTA in shared memory, transposed.
//                         Per chunk: g_i = dxa_i . W1^T, register-blocked (a thread computes 4 rows x 8 columns from one
//                         float4 of dxa^T and two of W1^T per k: 32 FMAs per 3 shared-memory loads), x_i * g_i into
//                         shared memory, node_attr_i = its row sum (fixed lane order, then a butterfly), grad_x_i = g_i;
//                         then a thread per feature adds the chunk's rows in order: the pair's feature_attr row when the
//                         pair has one chunk, else the chunk's partial.
//   attrib_pairs_kernel   a CTA per pair of two or more chunks: feature_attr = its chunk partials added in chunk order.
//                         A hub subgraph of thousands of rows is spread over many CTAs of attrib_rows_kernel; this
//                         kernel adds one partial per 32 rows.
// Every sum has a fixed order: no float atomics, bit-identical on reruns, no host synchronisation.
#include "common.cuh"

namespace npi {

constexpr int AT_THREADS = 256;
constexpr int AT_WARPS = AT_THREADS / WARP;
constexpr int AT_RPW = 4;                          // rows per warp: a thread's tile of g is AT_RPW rows x AT_CPT columns
constexpr int AT_ROWS = AT_WARPS * AT_RPW;         // 32 rows per chunk
constexpr int AT_MAXF = 256;
constexpr int AT_CPT = AT_MAXF / WARP;             // 8 feature columns per thread
constexpr int AT_DLD = AT_ROWS + 4;                // row stride of the transposed dxa stage: conflict-free stores, 16-byte rows
constexpr int AT_SCAN = 1024;                      // threads of attrib_chunks_kernel

static size_t at_smem_bytes(int F) {               // W1^T [128][F rounded to 8] | dxa^T [128][AT_DLD] | x * g [AT_ROWS][F]
    return sizeof(float) * ((size_t)H * ((F + 7) & ~7) + (size_t)H * AT_DLD + (size_t)AT_ROWS * F);
}

// chunks of a batch of B pairs and at most n_rows rows: sum ceil(n_p / AT_ROWS) <= n_rows / AT_ROWS + B
static int64_t at_max_chunks(int32_t n_rows, int32_t B) {
    return (int64_t)(n_rows > 0 ? n_rows : 0) / AT_ROWS + (B > 0 ? B : 0);
}

// carves the workspace: chunk_ptr [B + 1] | part [max chunks][F]; returns the bytes it needs (ws may be null for the query).
// The last region is not padded.
static int64_t attrib_layout(int32_t n_rows, int32_t B, int32_t F, char* ws, int32_t** chunk_ptr, float** part) {
    WsCarver c{ws};
    *chunk_ptr = c.take<int32_t>(4 * ((int64_t)B + 1));
    *part = c.take<float>(0);
    return c.off + at_max_chunks(n_rows, B) * (int64_t)F * (int64_t)sizeof(float);
}

__device__ __forceinline__ int at_rows_of(const int32_t* gptr, int p, int N) {
    return min(gptr[p + 1], N) - min(gptr[p], N);
}

__global__ void __launch_bounds__(AT_SCAN) attrib_chunks_kernel(const int32_t* __restrict__ gptr, int B, int n_rows,
                                                               int32_t* __restrict__ chunk_ptr) {
    __shared__ int sh[AT_SCAN / 32 + 1];
    const int N = min(n_rows, gptr[B]);
    int carry = 0;
    for (int base = 0; base < B; base += AT_SCAN) {
        const int p = base + (int)threadIdx.x;
        const int n = p < B ? max(at_rows_of(gptr, p, N), 0) : 0;
        int total;
        const int ex = block_excl_scan<AT_SCAN>((n + AT_ROWS - 1) / AT_ROWS, sh, &total);
        if (p < B) chunk_ptr[p] = carry + ex;
        carry += total;
    }
    if (threadIdx.x == 0) chunk_ptr[B] = carry;
}

__global__ void __launch_bounds__(AT_THREADS) attrib_rows_kernel(
    const float* __restrict__ dxa, const int32_t* __restrict__ gid, const uint8_t* __restrict__ dist,
    const int32_t* __restrict__ gptr, const int32_t* __restrict__ chunk_ptr, int B, int n_rows,
    const float* __restrict__ table, int ld, int F, const float* __restrict__ w1, float* __restrict__ node_attr,
    float* __restrict__ feature_attr, float* __restrict__ grad_x, float* __restrict__ part) {
    extern __shared__ __align__(16) float at_sm[];
    const int Fp = (F + 7) & ~7;
    float* sW = at_sm;                             // sW[k * Fp + c] = W1[c][k], zero for F <= c < Fp
    float* sD = sW + H * Fp;                       // sD[k * AT_DLD + r] = dxa of the chunk's row r
    float* sP = sD + H * AT_DLD;
    __shared__ int s_p;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int e = tid; e < Fp * H; e += AT_THREADS) {
        const int c = e >> 7, k = e & (H - 1);
        sW[k * Fp + c] = c < F ? __ldg(w1 + e) : 0.f;
    }
    const int N = min(n_rows, gptr[B]);
    const int nchunks = chunk_ptr[B];
    for (int w = blockIdx.x; w < nchunks; w += gridDim.x) {
        __syncthreads();                           // the W1 stage, or the previous chunk's readers of sD / sP / s_p
        if (tid == 0) {                            // the pair of chunk w: the last p < B with chunk_ptr[p] <= w
            int lo = 0, hi = B - 1;
            while (lo < hi) { const int m = (lo + hi + 1) >> 1; if (chunk_ptr[m] <= w) lo = m; else hi = m - 1; }
            s_p = lo;
        }
        __syncthreads();
        const int p = s_p;
        const int c0 = chunk_ptr[p], nch = chunk_ptr[p + 1] - c0;
        const int t0 = min(gptr[p], N) + (w - c0) * AT_ROWS, t1 = min(t0 + AT_ROWS, min(gptr[p + 1], N));
        for (int e = tid; e < AT_ROWS * (H / 4); e += AT_THREADS) {      // transposed; a warp stores 32 rows of one k
            const int r = e % AT_ROWS, q = e / AT_ROWS;
            const float4 v = t0 + r < t1 ? ldg4(dxa + (int64_t)(t0 + r) * H + 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
            sD[(4 * q) * AT_DLD + r] = v.x;
            sD[(4 * q + 1) * AT_DLD + r] = v.y;
            sD[(4 * q + 2) * AT_DLD + r] = v.z;
            sD[(4 * q + 3) * AT_DLD + r] = v.w;
        }
        __syncthreads();

        // g = dxa . W1^T for the chunk: warp = 4 rows (AT_RPW), lane = 8 columns (AT_CPT); both operands as float4
        const int r0 = warp * AT_RPW, cb = lane * AT_CPT;
        float acc[AT_RPW][AT_CPT];
#pragma unroll
        for (int r = 0; r < AT_RPW; ++r)
#pragma unroll
            for (int j = 0; j < AT_CPT; ++j) acc[r][j] = 0.f;
        if (cb < F) {
#pragma unroll 4
            for (int k = 0; k < H; ++k) {
                const float4 a = *reinterpret_cast<const float4*>(sD + k * AT_DLD + r0);
                const float4 b0 = *reinterpret_cast<const float4*>(sW + k * Fp + cb);
                const float4 b1 = *reinterpret_cast<const float4*>(sW + k * Fp + cb + 4);
                const float av[AT_RPW] = {a.x, a.y, a.z, a.w};
                const float bv[AT_CPT] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
                for (int r = 0; r < AT_RPW; ++r)
#pragma unroll
                    for (int j = 0; j < AT_CPT; ++j) acc[r][j] = fmaf(av[r], bv[j], acc[r][j]);
            }
        }
#pragma unroll
        for (int r = 0; r < AT_RPW; ++r) {
            const int rt = r0 + r, i = t0 + rt;
            if (i >= t1) continue;                 // warp-uniform
            const float* xr = table + (int64_t)__ldg(gid + i) * ld;
            const float lab = (float)__ldg(dist + i);
            float s = 0.f;
#pragma unroll
            for (int j = 0; j < AT_CPT; ++j) {
                const int c = cb + j;
                if (c < F) {
                    const float xg = (c == 0 ? lab : __ldg(xr + c)) * acc[r][j];
                    s += xg;
                    sP[rt * F + c] = xg;
                    if (grad_x) grad_x[(int64_t)i * F + c] = acc[r][j];
                }
            }
            s = warp_sum(s);
            if (lane == 0) node_attr[i] = s;
        }
        __syncthreads();
        if (tid < F) {                             // the chunk's rows in order
            float sum = 0.f;
            for (int r = 0; r < t1 - t0; ++r) sum += sP[r * F + tid];
            if (nch == 1) feature_attr[(int64_t)p * F + tid] = sum;
            else part[(int64_t)w * F + tid] = sum;
        }
    }
}

__global__ void __launch_bounds__(AT_THREADS) attrib_pairs_kernel(const int32_t* __restrict__ chunk_ptr, int F,
                                                                  const float* __restrict__ part,
                                                                  float* __restrict__ feature_attr) {
    const int p = blockIdx.x, c = threadIdx.x;
    if (c >= F) return;
    const int c0 = chunk_ptr[p], c1 = chunk_ptr[p + 1];
    if (c1 - c0 == 1) return;                      // written by attrib_rows_kernel
    float sum = 0.f;                               // no rows (below n_rows): 0
    for (int w = c0; w < c1; ++w) sum += part[(int64_t)w * F + c];
    feature_attr[(int64_t)p * F + c] = sum;
}

}  // namespace npi

using namespace npi;

extern "C" int64_t npi_input_attribution_workspace_bytes(int32_t n_rows, int32_t B, int32_t F) {
    int32_t* chunk_ptr;
    float* part;
    return attrib_layout(n_rows, B > 0 ? B : 0, F > 0 ? F : 1, nullptr, &chunk_ptr, &part);
}

extern "C" int npi_input_attribution(const float* dxa, const int32_t* gid, const uint8_t* dist, const int32_t* graph_ptr,
                                     int32_t B, int32_t n_rows, const float* table, int32_t ld, int32_t F, const float* w1,
                                     float* node_attr, float* feature_attr, float* grad_x,
                                     void* workspace, int64_t workspace_bytes, npi_stream_t stream) {
    NPI_REQUIRE(F >= 1 && F <= AT_MAXF, "input_attribution: F = %d out of range [1, %d]", F, AT_MAXF);
    NPI_REQUIRE(B >= 1, "input_attribution: B = %d, expected >= 1", B);
    NPI_REQUIRE(n_rows >= 0, "input_attribution: n_rows = %d, expected >= 0", n_rows);
    NPI_REQUIRE(graph_ptr && w1 && feature_attr && workspace, "input_attribution: null argument");
    NPI_REQUIRE(n_rows == 0 || (dxa && gid && dist && table && node_attr), "input_attribution: null argument");
    NPI_REQUIRE(ld >= F, "input_attribution: table row stride %d below F = %d", ld, F);
    NPI_REQUIRE(((uintptr_t)dxa & 15) == 0, "input_attribution: dxa must be 16-byte aligned");
    const int64_t need = npi_input_attribution_workspace_bytes(n_rows, B, F);
    NPI_REQUIRE(workspace_bytes >= need, "input_attribution: workspace of %lld bytes, %lld needed", (long long)workspace_bytes,
                (long long)need);
    cudaStream_t st = (cudaStream_t)stream;
    int32_t* chunk_ptr;
    float* part;
    attrib_layout(n_rows, B, F, (char*)workspace, &chunk_ptr, &part);
    attrib_chunks_kernel<<<1, AT_SCAN, 0, st>>>(graph_ptr, B, n_rows, chunk_ptr);
    NPI_CHECK_LAUNCH();
    const int64_t max_chunks = at_max_chunks(n_rows, B);
    if (n_rows > 0) {
        const size_t smem = at_smem_bytes(F);
        static MaxPerDevice configured;
        if (configured.need(smem))
            NPI_CHECK_CUDA(cudaFuncSetAttribute(attrib_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        const int grid = (int)(max_chunks < num_sms() ? max_chunks : num_sms());
        attrib_rows_kernel<<<grid, AT_THREADS, smem, st>>>(dxa, gid, dist, graph_ptr, chunk_ptr, B, n_rows, table, ld, F, w1,
                                                           node_attr, feature_attr, grad_x, part);
        NPI_CHECK_LAUNCH();
    }
    attrib_pairs_kernel<<<B, AT_THREADS, 0, st>>>(chunk_ptr, F, part, feature_attr);
    NPI_CHECK_LAUNCH();
    return NPI_OK;
}
