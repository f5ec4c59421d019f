// MLP head of Net_1 (src/classes.py:74-80) as device functions shared by head_fwd_kernel and head_fwd_delta_kernel (head.cu, one
// CTA per sample).
#pragma once
#include "common.cuh"

namespace npi {

constexpr int HD_THREADS = 128;
constexpr int D0 = 256, D1 = 128, D2 = 64, D3 = 2;
// forward: 16 warps per sample -- every warp owns 8 lin1 outputs (two rounds of 4, 8 weight loads in
// flight each) and 4 lin2 outputs (one round), so a sample is three short dependent phases instead of
// eight rounds of L2 latency; the per-output arithmetic (hence the result) does not depend on it
constexpr int HF_THREADS = 512;
constexpr int HF_WARPS = HF_THREADS / 32;

struct HeadSmem {
    __align__(16) float sx[D0];
    __align__(16) float s1[D1];
    __align__(16) float s2[D2];
    float s3[D3];
    float lp[D3];            // log-probabilities
    uint8_t keep[D1];        // dropout decisions (1 when not training)
};

// forward of sample b by the whole CTA of NT threads (the per-output arithmetic, a full-warp dot product, does not depend on NT);
// leaves a1 (after dropout), a2, the log-probabilities and the dropout decisions in S as well as in global memory; ends with a
// block barrier
template <int NT>
__device__ __forceinline__ void head_fwd_body(HeadSmem& S, const int b,
    const float* readout, const float* w1, const float* b1, const float* w2, const float* b2,
    const float* w3, const float* b3, int training, const uint8_t* mask_in, uint64_t seed, const int32_t* step_dev,
    const int32_t* sample_ids, int sample_id_base,
    float* a1_out, uint8_t* mask_out, float* a2_out, float* logp) {
    float* const sx = S.sx; float* const s1 = S.s1; float* const s2 = S.s2; float* const s3 = S.s3;
    constexpr int NW = NT / 32;
    static_assert((D1 / NW) % 4 == 0 && (D2 / NW) % 4 == 0, "four outputs per warp and round");
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int i = tid; i < D0; i += NT) sx[i] = readout[(int64_t)b * D0 + i];
    __syncthreads();
    // lin1 + ReLU + dropout
    const int sid = sample_ids ? sample_ids[b] : sample_id_base + b;
    const uint32_t stepv = step_dev ? (uint32_t)(*step_dev) : 0u;
    float4 x0 = *reinterpret_cast<const float4*>(sx + 4 * lane);
    float4 x1 = *reinterpret_cast<const float4*>(sx + 128 + 4 * lane);
    // four outputs per iteration: eight independent 16-byte weight loads in flight, four interleaved
    // butterfly reductions; lane u (< 4) finishes output o + u
#pragma unroll
    for (int o0 = warp * (D1 / NW); o0 < (warp + 1) * (D1 / NW); o0 += 4) {
        float4 wa[4], wb[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const float* wr = w1 + (int64_t)(o0 + u) * D0;
            wa[u] = ldg4(wr + 4 * lane); wb[u] = ldg4(wr + 128 + 4 * lane);
        }
        float d[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) d[u] = dot4(wa[u], x0) + dot4(wb[u], x1);
#pragma unroll
        for (int sh = 16; sh > 0; sh >>= 1) {
#pragma unroll
            for (int u = 0; u < 4; ++u) d[u] += __shfl_xor_sync(0xffffffffu, d[u], sh);
        }
        if (lane < 4) {
            const int o = o0 + lane;
            const float dd = lane == 0 ? d[0] : lane == 1 ? d[1] : lane == 2 ? d[2] : d[3];
            float v = fmaxf(dd + b1[o], 0.f);
            uint8_t keep = 1;
            if (training) {
                if (mask_in) keep = mask_in[(int64_t)b * D1 + o];
                else {
                    uint4 r = philox4x32_10(make_uint4((uint32_t)sid, (uint32_t)(o >> 2), stepv, 0u),
                                            make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
                    uint32_t rv = (o & 3) == 0 ? r.x : (o & 3) == 1 ? r.y : (o & 3) == 2 ? r.z : r.w;
                    keep = (rv & 0x80000000u) ? 1 : 0;
                }
                v = keep ? v * 2.0f : 0.f;                 // F.dropout(p=0.5): scale 1/(1-p)
            }
            s1[o] = v;
            S.keep[o] = keep;
            a1_out[(int64_t)b * D1 + o] = v;
            if (mask_out) mask_out[(int64_t)b * D1 + o] = keep;
        }
    }
    __syncthreads();
    // lin2 + ReLU
    float4 y0 = *reinterpret_cast<const float4*>(s1 + 4 * lane);
    for (int o0 = warp * (D2 / NW); o0 < (warp + 1) * (D2 / NW); o0 += 4) {
        float d[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) d[u] = dot4(ldg4(w2 + (int64_t)(o0 + u) * D1 + 4 * lane), y0);
#pragma unroll
        for (int sh = 16; sh > 0; sh >>= 1) {
#pragma unroll
            for (int u = 0; u < 4; ++u) d[u] += __shfl_xor_sync(0xffffffffu, d[u], sh);
        }
        if (lane < 4) {
            const int o = o0 + lane;
            const float dd = lane == 0 ? d[0] : lane == 1 ? d[1] : lane == 2 ? d[2] : d[3];
            float v = fmaxf(dd + b2[o], 0.f);
            s2[o] = v;
            a2_out[(int64_t)b * D2 + o] = v;
        }
    }
    __syncthreads();
    // lin3
    if (warp < D3) {
        float d = warp_sum(w3[warp * D2 + lane] * s2[lane] + w3[warp * D2 + 32 + lane] * s2[32 + lane]);
        if (lane == 0) s3[warp] = d + b3[warp];
    }
    __syncthreads();
    if (tid == 0) {
        float l0 = s3[0], l1 = s3[1];
        float m = fmaxf(l0, l1);
        float lse = m + logf(expf(l0 - m) + expf(l1 - m));
        logp[(int64_t)b * 2] = l0 - lse;
        logp[(int64_t)b * 2 + 1] = l1 - lse;
        S.lp[0] = l0 - lse;
        S.lp[1] = l1 - lse;
    }
    __syncthreads();
}

constexpr int DW = D1 + D2 + D3;          // per-sample deltas: ws[b] = { d1[128] | d2[64] | d3[2] }
struct HeadDeltaSmem { float d3[D3], d2[D2], d1[D1]; };

// per-sample deltas of the mean NLL and d_readout from what head_fwd_body left in S -- the operations of
// head_bwd_delta_kernel in the same order (bit-identical results)
template <int NT>
__device__ __forceinline__ void head_delta_body(const HeadSmem& S, HeadDeltaSmem& Dl, const int b, const float* w1, const float* w2, const float* w3,
                                                int training, const int32_t* y, float scale, float* ws, float* d_readout) {
    const int tid = threadIdx.x;
    if (tid < D3) {                                      // mean NLL: d logits = (softmax - onehot) * scale
        const float d = (expf(S.lp[tid]) - (y[b] == tid ? 1.f : 0.f)) * scale;
        Dl.d3[tid] = d;
        ws[(int64_t)b * DW + D1 + D2 + tid] = d;
    }
    __syncthreads();
    if (tid < D2) {
        float d = Dl.d3[0] * w3[tid] + Dl.d3[1] * w3[D2 + tid];
        d = S.s2[tid] > 0.f ? d : 0.f;
        Dl.d2[tid] = d;
        ws[(int64_t)b * DW + D1 + tid] = d;
    }
    __syncthreads();
    if (tid < D1) {
        float d = 0.f;
#pragma unroll 16
        for (int j = 0; j < D2; ++j) d = fmaf(Dl.d2[j], w2[j * D1 + tid], d);
        if (training) d = S.keep[tid] ? d * 2.0f : 0.f;
        d = S.s1[tid] > 0.f ? d : 0.f;
        Dl.d1[tid] = d;
        ws[(int64_t)b * DW + tid] = d;
    }
    __syncthreads();
    for (int i = tid; i < D0; i += NT) {
        float d = 0.f;
#pragma unroll 32
        for (int o = 0; o < D1; ++o) d = fmaf(Dl.d1[o], w1[o * D0 + i], d);
        d_readout[(int64_t)b * D0 + i] = d;
    }
}

}  // namespace npi
