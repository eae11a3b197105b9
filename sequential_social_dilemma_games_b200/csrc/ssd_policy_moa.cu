// Model of other agents (MOA) of the reference's causal-influence models (models/moa_model.py, MOA_LSTM) and the social-influence
// reward (common_funcs.py, compute_influence_reward) as ONE kernel behind ssd_moa_step: per group of 128 agents (= UMMA M, one
// TMEM lane per agent), for agent m = b * N + i (env b, agent i) with joint action a_{b, .}:
//
//   input(a')    = [x | onehot(a') | onehot(a_{b,j}) for j != i, increasing j]          width 32 + N A
//   gates(a')    = x Wx + h U + b + W_own[a'] + sum_j W_j[a_{b,j}]                     the one-hot input enters linearly:
//   G[128 x 512] = fp16([x | h]) * fp16([Wx; U])                                       ONE tcgen05 GEMM, all of tensor memory
//   G           += b + sum_j W_j[a_{b,j}]                                              pass 0: fp32 rows gathered from L2, in place
//   for every own action a' (A of them): c', h' = cell(G + W_own[a'], c)               pass 1: A cell updates per agent
//                                        y(a') = h' * moa_logits_w + moa_logits_b      CUDA-core product, fp32 rows from L2
//                                        q_k  += softmax(logits_pi)[a'] softmax(y(a')_k)
//   influence_k  = KL(softmax(y(a_{b,i})_k) || q_k / sum q_k)  (or the Jensen-Shannon divergence)
//
// Budget: [Wx; U] as fp16 (160 KB) stays resident in shared memory as in the fused policy head (ssd_policy_head.cu), and the
// base gates fill all 512 columns of tensor memory and stay live across the A counterfactual drains, so neither the one-hot
// rows (N A x 512 fp32, up to 158 KB) nor the head product's accumulators fit on chip next to them: the rows and
// moa_logits_w (fp32) are read from global memory (L2-resident, warp-uniform addresses for the own-action rows and the head
// weights), and the head product runs on the CUDA cores into a 64 KB scratch that reuses the A operand's buffer.
//
// Threads: pass 0 as the head's drain (thread = agent, warps 0-3 / 4-7 take units 0-63 / 64-127); pass 1 thread = agent and
// half of the own actions (warps 0-3 take a' = 0, 2, ..., warps 4-7 a' = 1, 3, ...), each thread owning all 128 units of its
// agent for its a'.  The counterfactual at the actual action writes pred and (h', c').  An own action outside 0..A-1 runs one
// more drain with no own row for pred / h' / c'.  Gate operand, gate GEMM and recurrent state: ssd_policy_lstm.cuh.
#include <cmath>
#include <new>
#include <vector>

#include "ssd_policy_lstm.cuh"

namespace ssd {
namespace moa {
using namespace ssd::lstm;

constexpr int NJ = 64, AMAX = 15;
constexpr int kConstFloats = NG + NJ;                  // gate bias, moa_logits_b
constexpr int kBlobBytes = kBBytes + kConstFloats * 4;  // 166 144
constexpr int kOffB = 0, kOffConst = kBBytes;
constexpr int kOffS = (kBlobBytes + 127) & ~127;       // A operand [128 x 160] fp16, then the scratch [NJ / 4][256][4] fp32
constexpr int kSBytes = NJ * kThreads * 4;             // 65 536
constexpr int kOffBar = kOffS + kSBytes;
constexpr int kSmemBytes = kOffBar + 16;
static_assert(kABytes <= kSBytes && kBlobBytes % 16 == 0 && kSmemBytes <= 227 * 1024, "one CTA per SM");

// fp32 rows per weight set in global memory: the one-hot rows of moa_lstm_w (own block, then the others' blocks) [N A][512],
// then moa_logits_w [128][NJ] zero padded
inline long long rows_floats(int n, int a) { return static_cast<long long>(n) * a * NG + U * NJ; }

// kMap Shared: agent m = a0 + row, own index i = m % N.  PerAgent (P = N): the groups of GroupMap (ssd_policy.h), as the
// policy head.
template <WeightMap kMap>
__global__ void __launch_bounds__(kThreads, 1)
moa_kernel(const float* __restrict__ feat, const int8_t* __restrict__ joint, const float* __restrict__ pol_logits, const float* h_in,
           const float* c_in, float* h_out, float* c_out, float* pred, float* __restrict__ cf, float* __restrict__ ipa, float* __restrict__ infl,
           long long M, int N, int A, const uint8_t* __restrict__ blob, const float* __restrict__ rows, long long rows_stride, int divergence,
           float clip, int ctas_per_policy) {
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ uint32_t s_tmem;
    const int tid = threadIdx.x, warp = tid >> 5;
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + kOffBar);
    const float* s_bias = reinterpret_cast<const float*>(smem + kOffConst);
    float* ys = reinterpret_cast<float*>(smem + kOffS);   // scratch: column j of thread t at ((j / 4) * kThreads + t) * 4 + j % 4
    const GroupMap<kMap> gm(M, N, ctas_per_policy);
    blob += static_cast<long long>(gm.pol) * kBlobBytes;
    rows += gm.pol * rows_stride;
    const float* wl = rows + static_cast<long long>(N) * A * NG;   // moa_logits_w [128][NJ]
    const int nc = (N - 1) * A;
    if (tid == 0) mbar_init(bar, 1);
    if (warp == 0) tmem_alloc(&s_tmem, 512);
    for (int i = tid; i < (kBlobBytes >> 4); i += kThreads) reinterpret_cast<uint4*>(smem)[i] = reinterpret_cast<const uint4*>(blob)[i];
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = s_tmem;
    const uint32_t sA = smem_u32(smem + kOffS), sB = smem_u32(smem + kOffB);
    uint32_t parity = 0;

    for (long long g = gm.cta; g < gm.n_groups; g += gm.stride) {
        const long long a0 = g * GA, sg = gm.state_group(g);
        const int rem = static_cast<int>(gm.rows - a0 < GA ? gm.rows - a0 : GA);
        {   // A = fp16([features | h]), as the policy head.  Built here rather than by the head's builder: with that builder this
            // kernel's register allocation and instruction order changed and it measured 0.5 % slower.
            const int seg = tid & 7, r8 = tid >> 3;
            const int hrow = tid & (GA - 1), hb0 = (tid >> 7) * 4;
            const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
            float4 vx[4], vh[4][4];
#pragma unroll
            for (int ps = 0; ps < 4; ++ps) {
                const int row = ps * 32 + r8;
                vx[ps] = row < rem ? __ldcs(reinterpret_cast<const float4*>(feat + gm.agent(a0, row) * KX) + seg) : z;
            }
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                const float4* src = reinterpret_cast<const float4*>(h_in + ((sg * (U / 16) + hb0 + b) * GA + hrow) * 16);
#pragma unroll
                for (int j = 0; j < 4; ++j) vh[b][j] = hrow < rem ? __ldcs(src + j) : z;
            }
#pragma unroll
            for (int ps = 0; ps < 4; ++ps)
                *reinterpret_cast<uint2*>(smem + kOffS + (seg >> 1) * (GA * 16) + (ps * 32 + r8) * 16 + (seg & 1) * 8) =
                    make_uint2(pack_h2(vx[ps].x, vx[ps].y), pack_h2(vx[ps].z, vx[ps].w));
#pragma unroll
            for (int b = 0; b < 4; ++b)
#pragma unroll
                for (int hf = 0; hf < 2; ++hf)
                    *reinterpret_cast<uint4*>(smem + kOffS + (KX / 8 + 2 * (hb0 + b) + hf) * (GA * 16) + hrow * 16) =
                        make_uint4(pack_h2(vh[b][2 * hf].x, vh[b][2 * hf].y), pack_h2(vh[b][2 * hf].z, vh[b][2 * hf].w),
                                   pack_h2(vh[b][2 * hf + 1].x, vh[b][2 * hf + 1].y), pack_h2(vh[b][2 * hf + 1].z, vh[b][2 * hf + 1].w));
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (warp == 0 && elect_one()) gate_gemm(tmem, sA, sB, bar);
        mbar_wait(bar, parity);
        parity ^= 1;
        tc_fence_after();

        // this thread's agent (TMEM lane r); both halves of the CTA see the same 128 agents
        const int r = tid & (GA - 1), half = warp >> 2;
        const uint32_t trow = tmem + (static_cast<uint32_t>((warp & 3) * 32) << 16);
        const bool live = r < rem;
        const long long m = gm.agent(a0, r), b = m / N;
        const int i = static_cast<int>(m - b * N);
        const int8_t* ja = joint + b * N;
        const int own = live ? ja[i] : 0;
        const bool own_ok = own >= 0 && own < A;
        bool env_ok = true;
        if (live)
            for (int j = 0; j < N; ++j) env_ok = env_ok && ja[j] >= 0 && ja[j] < A;
        {   // pass 0: gates += bias + the others' actual one-hot rows (an invalid action adds nothing)
#pragma unroll 1
            for (int ub = 0; ub < 4; ++ub) {
                const int u0 = half * 64 + ub * 16;
#pragma unroll 1
                for (int gq = 0; gq < 4; ++gq) {
                    uint32_t v[16];
                    tmem_ld16(trow + gq * U + u0, v);
                    tmem_ld_wait();
                    float s[16];
#pragma unroll
                    for (int e = 0; e < 16; ++e) s[e] = __uint_as_float(v[e]) + s_bias[gq * U + u0 + e];
                    if (live) {
                        for (int k = 0; k < N - 1; ++k) {
                            const int a = ja[k < i ? k : k + 1];
                            if (a < 0 || a >= A) continue;
                            const float4* src = reinterpret_cast<const float4*>(rows + static_cast<long long>(A + k * A + a) * NG + gq * U + u0);
#pragma unroll
                            for (int e = 0; e < 4; ++e) {
                                const float4 w = __ldg(src + e);
                                s[4 * e] += w.x, s[4 * e + 1] += w.y, s[4 * e + 2] += w.z, s[4 * e + 3] += w.w;
                            }
                        }
                    }
#pragma unroll
                    for (int e = 0; e < 16; ++e) v[e] = __float_as_uint(s[e]);
                    tmem_st8(trow + gq * U + u0, v);
                    tmem_st8(trow + gq * U + u0 + 8, v + 8);
                }
            }
            tmem_st_wait();
        }
        tc_fence_before();
        __syncthreads();
        tc_fence_after();

        float lse = 0.f;   // log-sum-exp of the policy logits: pi(a') = exp(l[a'] - lse)
        if (live) {
            const float* pl = pol_logits + m * A;
            float mx = pl[0];
            for (int a = 1; a < A; ++a) mx = fmaxf(mx, pl[a]);
            float se = 0.f;
            for (int a = 0; a < A; ++a) se += expf(pl[a] - mx);
            lse = mx + logf(se);
        }
        float qa[NJ];   // this thread's part of the marginal: sum over its a' of pi(a') p(. | a')
#pragma unroll
        for (int j = 0; j < NJ; ++j) qa[j] = 0.f;
        auto ys_at = [&](int j) -> float& { return ys[((j >> 2) * kThreads + tid) * 4 + (j & 3)]; };
        const int a_end = __any_sync(0xffffffffu, live && !own_ok) ? A + 1 : A;   // a' = A: no own row (pred of an invalid own action)
#pragma unroll 1
        for (int ap = half; ap < a_end; ap += 2) {
            const bool actual = live && (own_ok ? ap == own : ap == A);
            const float* wo = rows + static_cast<long long>(ap < A ? ap : 0) * NG;   // own row a' (warp-uniform)
#pragma unroll 1
            for (int ub = 0; ub < U / 16; ++ub) {
                const int u0 = ub * 16;
                uint32_t gi[16], gf[16], gg[16], go[16];
                tmem_ld16(trow + u0, gi);
                tmem_ld16(trow + U + u0, gf);
                tmem_ld16(trow + 2 * U + u0, gg);
                tmem_ld16(trow + 3 * U + u0, go);
                const long long tile = ((sg * (U / 16) + ub) * GA + r) * 16;
                float c[16];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float4 v = live ? *(reinterpret_cast<const float4*>(c_in + tile) + e) : make_float4(0.f, 0.f, 0.f, 0.f);
                    c[4 * e] = v.x, c[4 * e + 1] = v.y, c[4 * e + 2] = v.z, c[4 * e + 3] = v.w;
                }
                float wi[16], wf[16], wg[16], wo4[16];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
                    const float4 x0 = ap < A ? __ldg(reinterpret_cast<const float4*>(wo + u0) + e) : z;
                    const float4 x1 = ap < A ? __ldg(reinterpret_cast<const float4*>(wo + U + u0) + e) : z;
                    const float4 x2 = ap < A ? __ldg(reinterpret_cast<const float4*>(wo + 2 * U + u0) + e) : z;
                    const float4 x3 = ap < A ? __ldg(reinterpret_cast<const float4*>(wo + 3 * U + u0) + e) : z;
                    wi[4 * e] = x0.x, wi[4 * e + 1] = x0.y, wi[4 * e + 2] = x0.z, wi[4 * e + 3] = x0.w;
                    wf[4 * e] = x1.x, wf[4 * e + 1] = x1.y, wf[4 * e + 2] = x1.z, wf[4 * e + 3] = x1.w;
                    wg[4 * e] = x2.x, wg[4 * e + 1] = x2.y, wg[4 * e + 2] = x2.z, wg[4 * e + 3] = x2.w;
                    wo4[4 * e] = x3.x, wo4[4 * e + 1] = x3.y, wo4[4 * e + 2] = x3.z, wo4[4 * e + 3] = x3.w;
                }
                tmem_ld_wait();
                float c2[16], hn[16];
#pragma unroll
                for (int e = 0; e < 16; ++e) {
                    const float si = sigmoid_fast(__uint_as_float(gi[e]) + wi[e]), sf = sigmoid_fast(__uint_as_float(gf[e]) + wf[e]);
                    const float so = sigmoid_fast(__uint_as_float(go[e]) + wo4[e]);
                    c2[e] = sf * c[e] + si * tanh_fast(__uint_as_float(gg[e]) + wg[e]);
                    hn[e] = so * tanh_fast(c2[e]);
                }
                if (actual) {
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        __stcs(reinterpret_cast<float4*>(c_out + tile) + e, make_float4(c2[4 * e], c2[4 * e + 1], c2[4 * e + 2], c2[4 * e + 3]));
                        __stcs(reinterpret_cast<float4*>(h_out + tile) + e, make_float4(hn[4 * e], hn[4 * e + 1], hn[4 * e + 2], hn[4 * e + 3]));
                    }
                }
                // y(a') += h'[u0 .. u0 + 15] * moa_logits_w[u0 .. u0 + 15][:]  (warp-uniform weight rows)
#pragma unroll
                for (int j4 = 0; j4 < NJ / 4; ++j4) {
                    if (4 * j4 < nc) {
                        float4* acc_p = reinterpret_cast<float4*>(ys) + j4 * kThreads + tid;
                        float4 acc = ub ? *acc_p : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                        for (int e = 0; e < 16; ++e) {
                            const float4 w = __ldg(reinterpret_cast<const float4*>(wl + (u0 + e) * NJ) + j4);
                            acc.x = fmaf(hn[e], w.x, acc.x), acc.y = fmaf(hn[e], w.y, acc.y);
                            acc.z = fmaf(hn[e], w.z, acc.z), acc.w = fmaf(hn[e], w.w, acc.w);
                        }
                        *acc_p = acc;
                    }
                }
            }
            // logits of a': outputs, then softmax per other agent in place, then the marginal
            const float* lb = s_bias + NG;
            if (live) {
                float* cfm = cf != nullptr && ap < A ? cf + (m * A + ap) * nc : nullptr;
                float* pm = actual ? pred + m * nc : nullptr;
                for (int j = 0; j < nc; ++j) {
                    const float l = ys_at(j) + lb[j];
                    ys_at(j) = l;
                    if (cfm) cfm[j] = l;
                    if (pm) pm[j] = l;
                }
            }
            if (ap < A) {
                const float pi = live ? expf(pol_logits[m * A + ap] - lse) : 0.f;
                for (int k = 0; k < N - 1; ++k) {
                    float mx = ys_at(k * A);
                    for (int a = 1; a < A; ++a) mx = fmaxf(mx, ys_at(k * A + a));
                    float se = 0.f;
                    for (int a = 0; a < A; ++a) se += expf(ys_at(k * A + a) - mx);
                    const float w = pi / se;
                    for (int a = 0; a < A; ++a) ys_at(k * A + a) = w * expf(ys_at(k * A + a) - mx);
                }
#pragma unroll
                for (int j = 0; j < NJ; ++j)
                    if (j < nc) qa[j] += ys_at(j);
            }
        }
        __syncthreads();   // the scratch is free; pred is complete
        if (half == 1) {
#pragma unroll
            for (int j = 0; j < NJ; ++j)
                if (j < nc) ys_at(j) = qa[j];
        }
        __syncthreads();
        if (half == 0 && live) {
#pragma unroll
            for (int j = 0; j < NJ; ++j)
                if (j < nc) ys_at(j) = qa[j] + ys[((j >> 2) * kThreads + tid + GA) * 4 + (j & 3)];
            const float* pm = pred + m * nc;
            float total = 0.f;
            for (int k = 0; k < N - 1; ++k) {
                float qs = 0.f, mx = pm[k * A];
                for (int a = 0; a < A; ++a) qs += ys_at(k * A + a), mx = fmaxf(mx, pm[k * A + a]);
                float se = 0.f;
                for (int a = 0; a < A; ++a) se += expf(pm[k * A + a] - mx);
                float d = 0.f;
                for (int a = 0; a < A; ++a) {
                    const float p = expf(pm[k * A + a] - mx) / se, q = ys_at(k * A + a) / qs;
                    if (divergence == SSD_DIV_KL) {
                        if (p > 0.f) d += p * (logf(p) - logf(q));
                    } else {
                        const float mu = 0.5f * (p + q);
                        if (p > 0.f) d += 0.5f * p * (logf(p) - logf(mu));
                        if (q > 0.f) d += 0.5f * q * (logf(q) - logf(mu));
                    }
                }
                if (!env_ok) d = __int_as_float(0x7fc00000);
                ipa[m * (N - 1) + k] = d;
                total += d;
            }
            infl[m] = total > clip ? clip : total < -clip ? -clip : total;   // NaN stays NaN
        }
        tc_fence_before();
        __syncthreads();   // tensor memory and the scratch are free for the next group
        tc_fence_after();
    }
    __syncthreads();
    if (warp == 0) tmem_free(tmem, 512);
}

inline auto moa_kernel_for(WeightMap m) { return m == WeightMap::Shared ? moa_kernel<WeightMap::Shared> : moa_kernel<WeightMap::PerAgent>; }

}  // namespace moa
}  // namespace ssd

#pragma GCC visibility push(default)
extern "C" {

int ssd_moa_create(int device, int num_policies, int num_agents, int num_actions, const float* lstm_w, const float* lstm_u, const float* lstm_b,
                   const float* logits_w, const float* logits_b, ssd_moa_t* out) {
    using namespace ssd::moa;
    if (!out) return ssd::set_error(SSD_ERR_INVALID, "null argument");
    *out = nullptr;
    if (!lstm_w || !lstm_u || !lstm_b || !logits_w || !logits_b) return ssd::set_error(SSD_ERR_INVALID, "null weight pointer");
    const int n = num_agents, na = num_actions;
    if (n < 2 || n > SSD_MAX_AGENTS) return ssd::set_error(SSD_ERR_INVALID, "the MOA needs 2..SSD_MAX_AGENTS agents");
    if (na < 1 || na > AMAX) return ssd::set_error(SSD_ERR_INVALID, "num_actions must be 1..15");
    if ((n - 1) * na > NJ) return ssd::set_error(SSD_ERR_INVALID, "(num_agents - 1) * num_actions must be at most 64");
    if (num_policies != 1 && num_policies != n) return ssd::set_error(SSD_ERR_INVALID, "num_policies must be 1 or num_agents");
    const int kin = KX + n * na, nc = (n - 1) * na;
    const long long rf = rows_floats(n, na);
    std::vector<uint8_t> blobs(static_cast<size_t>(num_policies) * kBlobBytes, 0);
    std::vector<float> rows(static_cast<size_t>(num_policies * rf), 0.f);
    for (int q = 0; q < num_policies; ++q) {   // weight set q: arrays q of the num_policies consecutive ones behind each pointer
        const float* lw = lstm_w + static_cast<size_t>(q) * kin * NG;
        const float* ow = logits_w + static_cast<size_t>(q) * U * nc;
        const float* ob = logits_b + q * nc;
        float* cst = reinterpret_cast<float*>(blobs.data() + static_cast<size_t>(q) * kBlobBytes + kOffConst);
        pack_gates(reinterpret_cast<__half*>(blobs.data() + static_cast<size_t>(q) * kBlobBytes + kOffB), cst, lw, lstm_u + static_cast<size_t>(q) * U * NG,
                   lstm_b + q * NG);   // the features' rows of moa_lstm_w (its first 32) and moa_lstm_u
        for (int j = 0; j < nc; ++j) cst[NG + j] = ob[j];
        float* rq = rows.data() + q * rf;
        for (size_t e = 0; e < static_cast<size_t>(n) * na * NG; ++e) rq[e] = lw[KX * NG + e];   // rows 32 .. 32 + N A of moa_lstm_w
        for (int k = 0; k < U; ++k)
            for (int j = 0; j < nc; ++j) rq[static_cast<long long>(n) * na * NG + k * NJ + j] = ow[k * nc + j];
    }
    SsdPolicy* p = new (std::nothrow) SsdPolicy();
    if (!p) return ssd::set_error(SSD_ERR_INVALID, "out of host memory");
    p->device = device;
    p->num_policies = num_policies;
    p->kind = HandleKind::Moa;
    p->moa_agents = n;
    p->num_outputs = na;
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&p->sms, cudaDevAttrMultiProcessorCount, device);
    if (e == cudaSuccess) e = cudaMalloc(&p->d_head_blob, blobs.size());
    if (e == cudaSuccess) e = cudaMemcpyAsync(p->d_head_blob, blobs.data(), blobs.size(), cudaMemcpyHostToDevice, 0);
    if (e == cudaSuccess) e = cudaMalloc(&p->d_moa_rows, rows.size() * sizeof(float));
    if (e == cudaSuccess) e = cudaMemcpyAsync(p->d_moa_rows, rows.data(), rows.size() * sizeof(float), cudaMemcpyHostToDevice, 0);
    if (e == cudaSuccess) e = cudaStreamSynchronize(0);   // the host staging buffers go out of scope
    if (e == cudaSuccess) e = cudaFuncSetAttribute(moa_kernel_for(ssd::policy::weight_map(p)), cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
    if (e != cudaSuccess) {
        ssd_policy_destroy(p);
        return ssd::set_error(SSD_ERR_CUDA, cudaGetErrorString(e));
    }
    *out = p;
    return SSD_OK;
}

void ssd_moa_destroy(ssd_moa_t p) { ssd_policy_destroy(p); }

int ssd_moa_step(ssd_moa_t p, const float* features, const int8_t* joint_actions, const float* policy_logits, const float* h_in, const float* c_in,
                 float* h_out, float* c_out, float* pred, float* counterfactual, float* influence_per_agent, float* influence, int64_t num_agents,
                 int divergence, float clip, void* stream) {
    using namespace ssd::moa;
    using namespace ssd::policy;
    if (!p || !features || !joint_actions || !policy_logits || !h_in || !c_in || !h_out || !c_out || !pred || !influence_per_agent || !influence ||
        num_agents < 0)
        return ssd::set_error(SSD_ERR_INVALID, "bad argument");
    int rc = check_kind(p, HandleKind::Moa, "not an MOA handle (ssd_moa_create)");
    if (rc != SSD_OK) return rc;
    if (divergence != SSD_DIV_KL && divergence != SSD_DIV_JSD) return ssd::set_error(SSD_ERR_INVALID, "divergence must be SSD_DIV_KL or SSD_DIV_JSD");
    if (!(clip >= 0.f)) return ssd::set_error(SSD_ERR_INVALID, "clip must be >= 0 (+inf: no clamp), not NaN");
    rc = check_aligned({features, h_in, c_in, h_out, c_out}, "features and state pointers must be 16-byte aligned");
    if (rc != SSD_OK) return rc;
    if (h_out == h_in || c_out == c_in) return ssd::set_error(SSD_ERR_INVALID, "h_out / c_out must not alias h_in / c_in");
    const int n = p->moa_agents;
    if (num_agents % n != 0) return ssd::set_error(SSD_ERR_INVALID, "num_agents must be a multiple of the MOA's num_agents");
    if (num_agents == 0) return SSD_OK;
    rc = setup(p, nullptr, num_agents, stream);
    if (rc != SSD_OK) return rc;
    const Grid g = grid(p, num_agents);
    moa_kernel_for(weight_map(p))<<<g.ctas, kThreads, kSmemBytes, static_cast<cudaStream_t>(stream)>>>(
        features, joint_actions, policy_logits, h_in, c_in, h_out, c_out, pred, counterfactual, influence_per_agent, influence, num_agents, n,
        p->num_outputs, p->d_head_blob, p->d_moa_rows, rows_floats(n, p->num_outputs), divergence, clip, g.ctas_per_policy);
    return launched();
}

}  // extern "C"
#pragma GCC visibility pop
