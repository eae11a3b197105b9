// What the fused policy head (ssd_policy_head.cu) and the model of other agents (ssd_policy_moa.cu) share of their LSTM(128)
// gate stage: per group of 128 agents (= UMMA M, one TMEM lane per agent) and 256 threads, each builds
//
//   A[128 x 160] = fp16([features | h])        from HBM into shared memory
//   G[128 x 512] = A * [W; U]                  20 MMAs 128 x 256 x 16, all of tensor memory (Keras gate order i, f, c~, o)
//
// The B operand [W; U] (160 KB as fp16) stays resident at the start of shared memory; the kernels add their constants and
// scratch behind it.  The recurrent state lives in HBM in a TILED layout: [group of 128 agents][block of 16 units (8)][agent
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
