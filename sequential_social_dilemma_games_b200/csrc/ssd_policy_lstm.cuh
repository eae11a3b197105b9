// What the fused policy head (ssd_policy_head.cu) and the model of other agents (ssd_policy_moa.cu) share of their LSTM(128)
// gate stage: per group of 128 agents (= UMMA M, one TMEM lane per agent) and 256 threads, each builds
//
//   A[128 x 160] = fp16([features | h])        from HBM into shared memory
//   G[128 x 512] = A * [W; U]                  20 MMAs 128 x 256 x 16, all of tensor memory (Keras gate order i, f, c~, o)
//
// The B operand [W; U] (160 KB as fp16) stays resident at the start of shared memory; the kernels add their constants and
// scratch behind it.  gate_operand below builds A for the head and for the MOA pool (the Shared / PerAgent MOA keeps its own
// builder, ssd_policy_moa.cu).  The recurrent state lives in HBM in a TILED layout: [group of 128 agents][block of 16 units (8)][agent
// in group (128)][16 floats] -- element (agent m, unit u) at ((m / 128 * 8 + u / 16) * 128 + m % 128) * 16 + u % 16.  A thread
// owns an agent and works through 16 units at a time, so a warp's loads and stores of c / h are 2 KB contiguous (with
// row-major [M][128] state they were 64-byte pieces 512 bytes apart and the cell update ran at 2.9 TB/s of HBM).
#pragma once
#include <cuda_fp16.h>

#include "ssd_policy.h"
#include "ssd_umma.cuh"

namespace ssd {
namespace lstm {
using namespace ssd::umma;

constexpr int GA = 128, U = 128, KX = 32, K = KX + U, NG = 4 * U;
constexpr int kThreads = 256;
constexpr int kBBytes = (K / 8) * NG * 16;   // 163 840: [W; U] K-major, element (n, k) at ((k / 8) * 512 + n) * 16 + (k % 8) * 2
constexpr int kABytes = (K / 8) * GA * 16;   // 40 960: A [128 x 160] fp16

__device__ __forceinline__ uint32_t pack_h2(float lo, float hi) {
    const __half2 v = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<const uint32_t*>(&v);
}
// one MUFU op each (tanh.approx.f32, ~2^-11 relative error: below the fp16 rounding of the GEMM operands); the cell update
// is transcendental-bound: 5 per unit, 640 per agent
__device__ __forceinline__ float tanh_fast(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float sigmoid_fast(float x) { return fmaf(tanh_fast(0.5f * x), 0.5f, 0.5f); }

__device__ __forceinline__ void copy_blob(uint8_t* smem, const uint8_t* blob, int bytes) {
    for (int i = threadIdx.x; i < (bytes >> 4); i += kThreads) reinterpret_cast<uint4*>(smem)[i] = reinterpret_cast<const uint4*>(blob)[i];
}

// G = A * [W; U] into tensor memory columns 0-511, two column halves of 256 with the k-steps interleaved, completion on `bar`.
// Issued by one elected thread.
__device__ __forceinline__ void gate_gemm(uint32_t tmem, uint32_t sA, uint32_t sB, uint64_t* bar) {
    constexpr uint32_t kIG = umma_idesc(GA, 256);
    tc_fence_after();
#pragma unroll
    for (int ks = 0; ks < K / 16; ++ks)
#pragma unroll
        for (int half = 0; half < 2; ++half)
            umma_f16(tmem + half * 256, umma_desc(sA + ks * 2 * GA * 16, GA * 16, 128), umma_desc(sB + half * 256 * 16 + ks * 2 * NG * 16, NG * 16, 128),
                     kIG, ks > 0);
    umma_commit(bar);
}

// A = fp16([features | h]) of the group's `rem` live rows into `a`, rows past them zero.  agent(r): the feature row of row r;
// state(r): the offset, in 16-float pieces, of row r's first unit block in the tiled state (block b at + b * 128).  HBM is read
// in long contiguous runs (features: a 128-byte row per eight lanes; h: the tiled state, 64 bytes per lane, 2 KB per warp -- a
// thread walking a row-major row in 32-byte steps reached 2.3 TB/s).  All loads before the stores: the compiler keeps a
// global load below a store through a generic pointer.
template <class Agent, class State>
__device__ __forceinline__ void gate_operand(uint8_t* a, const float* __restrict__ feat, const float* h_in, int rem, Agent agent, State state) {
    const int tid = threadIdx.x;
    const int seg = tid & 7, r8 = tid >> 3;                  // features: 32 rows per pass, 4 passes, a 128-byte row per eight lanes
    const int hrow = tid & (GA - 1), hb0 = (tid >> 7) * 4;   // h: thread = (agent, four of the eight 16-unit blocks), 64 bytes per block
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    float4 vx[4], vh[4][4];
#pragma unroll
    for (int ps = 0; ps < 4; ++ps) {
        const int row = ps * 32 + r8;
        vx[ps] = row < rem ? __ldcs(reinterpret_cast<const float4*>(feat + agent(row) * KX) + seg) : z;
    }
    const long long hbase = state(hrow);
#pragma unroll
    for (int b = 0; b < 4; ++b) {
        const float4* src = reinterpret_cast<const float4*>(h_in + (hbase + (hb0 + b) * GA) * 16);
#pragma unroll
        for (int j = 0; j < 4; ++j) vh[b][j] = hrow < rem ? __ldcs(src + j) : z;
    }
#pragma unroll
    for (int ps = 0; ps < 4; ++ps)   // elements 4 seg .. 4 seg + 3 of the 32 features: half of operand chunk seg / 2
        *reinterpret_cast<uint2*>(a + (seg >> 1) * (GA * 16) + (ps * 32 + r8) * 16 + (seg & 1) * 8) =
            make_uint2(pack_h2(vx[ps].x, vx[ps].y), pack_h2(vx[ps].z, vx[ps].w));
#pragma unroll
    for (int b = 0; b < 4; ++b)      // units 16 (hb0 + b) .. + 15: operand chunks 4 + 2 (hb0 + b) and the next
#pragma unroll
        for (int hf = 0; hf < 2; ++hf)
            *reinterpret_cast<uint4*>(a + (KX / 8 + 2 * (hb0 + b) + hf) * (GA * 16) + hrow * 16) =
                make_uint4(pack_h2(vh[b][2 * hf].x, vh[b][2 * hf].y), pack_h2(vh[b][2 * hf].z, vh[b][2 * hf].w),
                           pack_h2(vh[b][2 * hf + 1].x, vh[b][2 * hf + 1].y), pack_h2(vh[b][2 * hf + 1].z, vh[b][2 * hf + 1].w));
}

// Host: packs [W; U] (Keras LSTM kernel [32][512] and recurrent kernel [128][512], gates i, f, c~, o) K-major as fp16 into b,
// and the gate bias into bias[512].
inline void pack_gates(__half* b, float* bias, const float* w, const float* u, const float* gate_bias) {
    for (int n = 0; n < NG; ++n) {
        for (int k = 0; k < KX; ++k) b[ssd::policy::kmajor(NG, n, k)] = __float2half_rn(w[k * NG + n]);
        for (int k = 0; k < U; ++k) b[ssd::policy::kmajor(NG, n, KX + k)] = __float2half_rn(u[k * NG + n]);
        bias[n] = gate_bias[n];
    }
}

}  // namespace lstm
}  // namespace ssd
