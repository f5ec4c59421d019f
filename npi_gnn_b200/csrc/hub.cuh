// Hub queue of a CSR (segments of the rows longer than AG_HUB entries, arrival counters, partial sums) and the binned
// row order -- shared by the aggregation kernels (agg.cu), which consume them, and by the kernels that produce a CSR and
// can list its rows on the way (agg.cu: npi_hub_rows_build; pool.cu: filter_adj).
#pragma once
#include "common.cuh"

namespace npi {

constexpr int AG_THREADS = 256;
constexpr int AG_WARPS = AG_THREADS / 32;
constexpr int AG_SHORT = 16;      // rows up to this many entries are reduced by an 8-lane group
#ifndef NPI_AG_HUB
#define NPI_AG_HUB 16
#endif
#ifndef NPI_AG_SEG
#define NPI_AG_SEG 32
#endif
constexpr int AG_HUB = NPI_AG_HUB;   // rows with more entries are cut into segments
constexpr int AG_SEG = NPI_AG_SEG;   // entries per segment of a hub row (one warp each)

// Hub queue = caller's buffer, sized by npi_hub_rows_bytes(e_max):
//   int32 hdr[32]     [0] segments listed, [1] capacity `cap` (segments),
//                     [4+c] rows of length class c (c = 0..7, row_class below), [16+c] fill cursors
//   int32 seg_row[cap], seg_base[cap]   row of segment s / first segment of that row (a row's
//                                       segments are consecutive: segment s is part s - seg_base[s])
//   int32 arrive[cap]                   arrive[base]: parts of the row finished, arrive[base+1+g]: segments of group g
//                                       finished (two-level combine); zeroed by hub_list_row, rewound by the last
//   int32 dsum[cap]                     integer label sum of a part (virtual input layer)
//   float part[cap][128]                partial sums
// sum_rows ceil(L/AG_SEG) <= E/AG_SEG + #hub rows <= E/AG_SEG + E/(AG_HUB+1)  (= hub_cap).
struct HubQueue { int32_t* hdr; int32_t* seg_row; int32_t* seg_base; int32_t* arrive; int32_t* dsum; float* part; };
constexpr int HUB_HDR = 32;
constexpr int HUB_GRP = 8;              // segments per group of the two-level combine (rows without a self term)
constexpr int HQ_CLS = 4, HQ_CUR = 16;      // class totals / fill cursors inside hdr
constexpr int N_CLS = 8;

__host__ __device__ inline int hub_cap(int64_t e_max) {
    const int64_t e = e_max > 0 ? e_max : 0;
    return (int)((e / AG_SEG + e / (AG_HUB + 1) + 8 + 3) & ~(int64_t)3);
}
__host__ __device__ inline HubQueue hub_view(int32_t* buf, int cap) {
    HubQueue q;
    q.hdr = buf; q.seg_row = buf + HUB_HDR; q.seg_base = q.seg_row + cap; q.arrive = q.seg_base + cap; q.dsum = q.arrive + cap;
    q.part = reinterpret_cast<float*>(q.dsum + cap);
    return q;
}

// Length class of a row: the 8-lane groups of a warp work in lock step, two elements (entries, then
// the row itself) per round, so a warp should hold four rows that need the same number of rounds.
// Classes 0..5: 1, 2, 3, 4, 5-6, 7-9 rounds (short rows); 6: whole-warp rows (AG_SHORT+1 .. AG_HUB entries: empty
// at the shipped AG_HUB = AG_SHORT = 16, reachable in a -DNPI_AG_HUB build); 7: hub rows (segments).
__host__ __device__ inline int row_class(int len) {
    return len <= 1 ? 0 : len <= 3 ? 1 : len <= 5 ? 2 : len <= 7 ? 3 : len <= 11 ? 4 : len <= AG_SHORT ? 5 : len <= AG_HUB ? 6 : 7;
}

// one row of `len` entries joins the queue: class histogram (the caller's shared-memory hist[N_CLS]) and, for a hub row,
// its consecutive segment slots (slot order is timing dependent and irrelevant: rows are independent).  Every arrival
// counter a launch may use is zeroed here, so the queue works whatever memory it was allocated in: arrive[base] counts
// the row, and a row of more than 2*HUB_GRP segments also counts its groups in arrive[base + 1 + g] (the two-level
// combine of agg.cu).
__device__ __forceinline__ void hub_list_row(const HubQueue& hq, int cap, int* hist, int row, int len) {
    atomicAdd(&hist[row_class(len)], 1);
    if (len > AG_HUB) {
        const int nseg = (len + AG_SEG - 1) / AG_SEG;
        const int base = atomicAdd(&hq.hdr[0], nseg);
        if (base + nseg <= cap) {
            for (int k = 0; k < nseg; ++k) { hq.seg_row[base + k] = row; hq.seg_base[base + k] = base; }
            const int ncnt = nseg > 2 * HUB_GRP ? 1 + (nseg + HUB_GRP - 1) / HUB_GRP : 1;
            for (int k = 0; k < ncnt; ++k) hq.arrive[base + k] = 0;
        }
    }
}

}  // namespace npi
