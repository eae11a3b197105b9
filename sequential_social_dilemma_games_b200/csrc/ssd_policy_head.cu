// LSTM(128) + logits / value heads + action sampling of the reference's policy network (models/conv_to_fcnet_v2.py:68-92)
// as ONE kernel behind ssd_policy_lstm_heads: per group of 128 agents (= UMMA M, one TMEM lane per agent)
//
//   A[128 x 160]  = fp16([features | h])                                  built from HBM into shared memory
//   G[128 x 512]  = A * [W; U]                                            the gate GEMM of ssd_policy_lstm.cuh
//   c' = sigmoid(f) c + sigmoid(i) tanh(c~),  h' = sigmoid(o) tanh(c')     drain: thread = agent, 8 warps split the units
//   Y[128 x 16]   = fp16(h') * [logits_w | value_w]                        8 MMAs 128 x 16 x 16 into the freed columns
//   action        = argmax(logits + Gumbel noise)                          Philox4x32-10 keyed (seed; agent, counter)
//
// The recurrent state lives in HBM in the tiled layout of ssd_policy_lstm.cuh.  HBM traffic per agent: 128 B features + 1 KB
// (h, c) in, 1 KB (h', c') + logits / value / action out -- one pass, against ~7.5 KB for the unfused gate GEMMs + cell
// update.  The B operand [W; U] (160 KB as fp16) stays resident in shared memory; the grid is persistent (one CTA per SM).
#include <cstdio>
#include <vector>

#include "ssd_policy_lstm.cuh"

#ifdef SSD_POLICY_TIMING  // profiles/micro/policy_head_timing.cu: cycles per phase of thread 0 of CTA 0
__device__ unsigned long long g_head_cycles[8];
#define SSD_HT_DECL unsigned long long ht_[8] = {0, 0, 0, 0, 0, 0, 0, 0}; long long ht_t = clock64()
#define SSD_HT(slot) do { const long long n_ = clock64(); ht_[slot] += n_ - ht_t; ht_t = n_; } while (0)
#define SSD_HT_FLUSH do { if (blockIdx.x == 0 && threadIdx.x == 0) for (int q_ = 0; q_ < 8; ++q_) g_head_cycles[q_] = ht_[q_]; } while (0)
#else
#define SSD_HT_DECL
#define SSD_HT(slot)
#define SSD_HT_FLUSH
#endif

namespace ssd {
namespace policy_head {
using namespace ssd::lstm;

constexpr int NH = 16;
constexpr int kBHBytes = (U / 8) * NH * 16;        // 4 096: [logits_w | value_w | 0]
constexpr int kConstFloats = NG + NH;              // gate bias, head bias
constexpr int kBlobBytes = kBBytes + kBHBytes + kConstFloats * 4;   // 170 048
constexpr int kOffB = 0, kOffBH = kBBytes, kOffConst = kOffBH + kBHBytes;
constexpr int kOffA = (kOffConst + kConstFloats * 4 + 127) & ~127;   // [128 x 160] fp16, later fp16(h') [128 x 128]
constexpr int kOffBar = kOffA + kABytes;
constexpr int kSmemBytes = kOffBar + 16;
static_assert(kBlobBytes % 16 == 0 && kSmemBytes <= 227 * 1024, "one CTA per SM");

// Start of a kernel: the mbarrier, all 512 columns of tensor memory and the resident weights (`bytes` of blob) at smem[0].
// Returns the tensor-memory base.
__device__ __forceinline__ uint32_t prologue(uint8_t* smem, const uint8_t* blob, int bytes, uint64_t* bar, uint32_t* s_tmem) {
    if (threadIdx.x == 0) mbar_init(bar, 1);
    if (threadIdx.x < 32) tmem_alloc(s_tmem, 512);
    copy_blob(smem, blob, bytes);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    return *s_tmem;
}

// Shared / PerAgent: the groups of GroupMap (ssd_policy.h); features are read as 128-byte rows P * 128 bytes apart and
// outputs are written to agent-major rows.  The sampler keys Philox by the agent-major index m in all variants.
//
// WeightMap::Pool: a group is one tile of the assignment (ssd_policy_pool.cu), agents perm[first, first + count) of one policy;
// CTA c takes tiles [c T / G, (c + 1) T / G) and reloads the resident weights when the policy changes (the tiles are in
// policy order).  Feature rows are gathered by perm, h and c are read and written per agent in the agent-major tiled layout
// (64-byte pieces, one per 16 units), outputs go to row m.
//
// kDist (ssd_policy_lstm_heads_dist): the action is chosen by `mode` (SSD_ACT_SAMPLE: the sampler above; SSD_ACT_GREEDY: the
// first argmax of the logits; SSD_ACT_GIVEN: read from `actions`, which is then not written), and the epilogue adds
// logp = l[a] - logsumexp(l) of that action and the entropy of softmax(l), from the fp32 logits it writes (accurate expf /
// logf, at most 15 of each per agent).  Without kDist these parameters are unused and the code is that of the plain head.
template <WeightMap kMap, bool kDist>
__global__ void __launch_bounds__(kThreads, 1)
lstm_heads_kernel(const float* __restrict__ feat, const float* h_in, const float* c_in, float* h_out, float* c_out, float* __restrict__ logits,
                  float* __restrict__ value, int8_t* __restrict__ actions, long long M, int num_outputs, const uint8_t* __restrict__ blob,
                  uint32_t seed_lo, uint32_t seed_hi, uint32_t counter, int num_policies, int ctas_per_policy, const uint32_t* __restrict__ perm,
                  const PoolTile* __restrict__ tiles, const uint32_t* __restrict__ num_tiles, int mode, float* __restrict__ logp,
                  float* __restrict__ entropy) {
    constexpr bool kPerAgent = kMap != WeightMap::Shared, kPool = kMap == WeightMap::Pool;
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ uint32_t s_tmem;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + kOffBar);
    const float* s_bias = reinterpret_cast<const float*>(smem + kOffConst);
    const GroupMap<kMap> gm(M, num_policies, ctas_per_policy);
    const long long nt = kPool ? *num_tiles : 0;
    const long long first = kPool ? nt * blockIdx.x / gridDim.x : gm.cta;                  // pool: its first tile
    const long long end = kPool ? nt * (blockIdx.x + 1) / gridDim.x : gm.n_groups;          // pool: the end of its tiles
    const long long stride = kPool ? 1 : gm.stride;
    const uint8_t* const blob0 = blob;
    int cur = 0;   // pool: the weight set in shared memory
    if (kPool) {
        cur = first < end ? tiles[first].policy : 0;
        blob += static_cast<long long>(cur) * kBlobBytes;
    } else if (kPerAgent) {
        blob += static_cast<long long>(gm.pol) * kBlobBytes;
    }
    const uint32_t tmem = prologue(smem, blob, kBlobBytes, bar, &s_tmem);
    const uint32_t sA = smem_u32(smem + kOffA), sB = smem_u32(smem + kOffB), sBH = smem_u32(smem + kOffBH);
    constexpr uint32_t kIH = umma_idesc(GA, NH);
    uint32_t parity = 0;

    SSD_HT_DECL;
    for (long long g = first; g < end; g += stride) {
        const long long a0 = g * GA, sg = gm.state_group(g);   // first agent row of the group in its policy; its state group
        const PoolTile tile = kPool ? tiles[g] : PoolTile{};
        if (kPool && tile.policy != cur) {   // the previous group is complete (the barrier at the end of the loop)
            cur = tile.policy;
            copy_blob(smem, blob0 + static_cast<long long>(cur) * kBlobBytes, kBlobBytes);
            fence_async_smem();
            __syncthreads();
        }
        const int rem = kPool ? tile.count : static_cast<int>(gm.rows - a0 < GA ? gm.rows - a0 : GA);
        // agent of row r; its offset in the tiled state (pool: agent-major, element (m, u) at (that + u / 16 * 128) * 16 + u % 16)
        auto agent = [&](int r) { return kPool ? static_cast<long long>(perm[tile.first + r]) : gm.agent(a0, r); };
        auto state = [&](int r) -> long long {
            if (!kPool) return sg * (U / 16) * GA + r;
            if (r >= rem) return 0;   // a pool tile's rows past its count have no perm entry
            const long long m = agent(r);
            return (m >> 7) * (U / 16) * GA + (m & (GA - 1));
        };
        gate_operand(smem + kOffA, feat, h_in, rem, agent, state);
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        SSD_HT(0);
        if (warp == 0 && elect_one()) gate_gemm(tmem, sA, sB, bar);
        mbar_wait(bar, parity);
        parity ^= 1;
        tc_fence_after();
        SSD_HT(1);
        {   // cell update: thread = agent (TMEM lane), warps 0-3 take units 0-63, warps 4-7 units 64-127
            const int q = warp & 3, row = q * 32 + lane, uh = warp >> 2;
            const uint32_t trow = tmem + (static_cast<uint32_t>(q * 32) << 16);
            const bool live = row < rem;
            const long long tile0 = (state(row) + uh * 4 * GA) * 16;   // this agent's 16 floats of unit block 4 uh; + GA * 16 per block
            float4 cn[4];   // the next 16 units of c, fetched one iteration ahead
#pragma unroll
            for (int e = 0; e < 4; ++e) cn[e] = live ? __ldcs(reinterpret_cast<const float4*>(c_in + tile0) + e) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 1
            for (int ub = 0; ub < 4; ++ub) {
                const int u0 = uh * 64 + ub * 16;
                uint32_t gi[16], gf[16], gg[16], go[16];
                tmem_ld16(trow + u0, gi);
                tmem_ld16(trow + U + u0, gf);
                tmem_ld16(trow + 2 * U + u0, gg);
                tmem_ld16(trow + 3 * U + u0, go);
                const float c[16] = {cn[0].x, cn[0].y, cn[0].z, cn[0].w, cn[1].x, cn[1].y, cn[1].z, cn[1].w,
                                     cn[2].x, cn[2].y, cn[2].z, cn[2].w, cn[3].x, cn[3].y, cn[3].z, cn[3].w};
                if (ub < 3) {
#pragma unroll
                    for (int e = 0; e < 4; ++e)
                        cn[e] = live ? __ldcs(reinterpret_cast<const float4*>(c_in + tile0 + (ub + 1) * (GA * 16)) + e) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
                tmem_ld_wait();
                float c2[16], hn[16];
#pragma unroll
                for (int e = 0; e < 16; ++e) {
                    const float si = sigmoid_fast(__uint_as_float(gi[e]) + s_bias[u0 + e]), sf = sigmoid_fast(__uint_as_float(gf[e]) + s_bias[U + u0 + e]);
                    const float so = sigmoid_fast(__uint_as_float(go[e]) + s_bias[3 * U + u0 + e]);
                    c2[e] = sf * c[e] + si * tanh_fast(__uint_as_float(gg[e]) + s_bias[2 * U + u0 + e]);
                    hn[e] = so * tanh_fast(c2[e]);
                }
                if (live) {
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        __stcs(reinterpret_cast<float4*>(c_out + tile0 + ub * (GA * 16)) + e, make_float4(c2[4 * e], c2[4 * e + 1], c2[4 * e + 2], c2[4 * e + 3]));
                        __stcs(reinterpret_cast<float4*>(h_out + tile0 + ub * (GA * 16)) + e, make_float4(hn[4 * e], hn[4 * e + 1], hn[4 * e + 2], hn[4 * e + 3]));
                    }
                }
                // fp16(h') is the A operand of the heads: the gate MMAs are complete, their operand buffer is free
                uint4* dst = reinterpret_cast<uint4*>(smem + kOffA + (u0 / 8) * (GA * 16) + row * 16);
                dst[0] = make_uint4(pack_h2(hn[0], hn[1]), pack_h2(hn[2], hn[3]), pack_h2(hn[4], hn[5]), pack_h2(hn[6], hn[7]));
                dst[GA] = make_uint4(pack_h2(hn[8], hn[9]), pack_h2(hn[10], hn[11]), pack_h2(hn[12], hn[13]), pack_h2(hn[14], hn[15]));
            }
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();  // every gate column has been read: tensor memory can take the heads
        SSD_HT(2);
        if (warp == 0 && elect_one()) {
            tc_fence_after();
#pragma unroll
            for (int ks = 0; ks < U / 16; ++ks)
                umma_f16(tmem, umma_desc(sA + ks * 2 * GA * 16, GA * 16, 128), umma_desc(sBH + ks * 2 * NH * 16, NH * 16, 128), kIH, ks > 0);
            umma_commit(bar);
        }
        mbar_wait(bar, parity);
        parity ^= 1;
        tc_fence_after();
        SSD_HT(3);
        if (warp < 4) {  // heads: logits, value, sampled action
            const int row = warp * 32 + lane;
            uint32_t y[16];
            tmem_ld16(tmem + (static_cast<uint32_t>(warp * 32) << 16), y);
            tmem_ld_wait();
            if (row < rem) {
                const long long m = agent(row);
                const float* hb = s_bias + NG;
                float best = -3.0e38f;
                int arg = 0;
                uint4 rnd = make_uint4(0, 0, 0, 0);
                float lv[NH - 1];   // kDist: the logits as written
#pragma unroll
                for (int a = 0; a < NH - 1; ++a) {
                    if (a < num_outputs) {
                        const float l = __uint_as_float(y[a]) + hb[a];
                        logits[m * num_outputs + a] = l;
                        if (kDist) lv[a] = l;
                        if (kDist ? mode == SSD_ACT_SAMPLE : actions != nullptr) {  // Gumbel-max: argmax(l - log(-log u)), u uniform in (0, 1)
                            if ((a & 3) == 0) rnd = philox4x32_10(static_cast<uint32_t>(m), static_cast<uint32_t>(m >> 32), counter, a >> 2, seed_lo, seed_hi);
                            const float u = (static_cast<float>(pick_word(rnd, a & 3) >> 8) + 0.5f) * (1.0f / 16777216.0f);
                            const float s = l - __logf(-__logf(u));
                            if (s > best) { best = s; arg = a; }
                        }
                    }
                }
                // y[] is indexed statically: read the value column with a select chain
                float v = 0.f;
#pragma unroll
                for (int a = 0; a < NH; ++a) {
                    if (!kPerAgent) {
                        if (a == num_outputs) v = __uint_as_float(y[a]) + hb[a];
                    } else {  // an explicit selp: ptxas turned the chain into y[num_outputs] through a stack copy of y[] here
                        asm("{\n\t.reg .pred q;\n\tsetp.eq.s32 q, %2, %3;\n\tselp.f32 %0, %1, %0, q;\n\t}\n"
                            : "+f"(v) : "f"(__uint_as_float(y[a]) + hb[a]), "r"(a), "r"(num_outputs));
                    }
                }
                value[m] = v;
                if (kDist) {
                    float mx = lv[0];   // first argmax: the greedy action, and the shift of the logsumexp
                    int am = 0;
#pragma unroll
                    for (int a = 1; a < NH - 1; ++a)
                        if (a < num_outputs && lv[a] > mx) { mx = lv[a]; am = a; }
                    const int act = mode == SSD_ACT_SAMPLE ? arg : mode == SSD_ACT_GREEDY ? am : static_cast<int>(actions[m]);
                    float se = 0.f, sed = 0.f, la = __int_as_float(0x7fc00000);   // la: NaN unless act is in 0..A-1
#pragma unroll
                    for (int a = 0; a < NH - 1; ++a) {
                        if (a < num_outputs) {
                            const float d = lv[a] - mx, e = expf(d);
                            se += e;
                            sed = fmaf(e, d, sed);
                            if (a == act) la = d;
                        }
                    }
                    const float lse = logf(se);   // logsumexp(l) - mx; se >= 1
                    if (logp != nullptr) logp[m] = la - lse;
                    if (entropy != nullptr) entropy[m] = lse - sed / se;   // -sum p (d - lse)
                    if (mode != SSD_ACT_GIVEN) actions[m] = static_cast<int8_t>(act);
                } else if (actions != nullptr) {
                    actions[m] = static_cast<int8_t>(arg);
                }
            }
        }
        tc_fence_before();
        __syncthreads();  // tensor memory and the operand buffer are free for the next group
        tc_fence_after();
        SSD_HT(4);
    }
    SSD_HT_FLUSH;
    __syncthreads();
    if (warp == 0) tmem_free(tmem, 512);
}

template <bool kDist>
auto heads_kernel(WeightMap m) {
    return m == WeightMap::Shared ? lstm_heads_kernel<WeightMap::Shared, kDist>
                                  : m == WeightMap::PerAgent ? lstm_heads_kernel<WeightMap::PerAgent, kDist> : lstm_heads_kernel<WeightMap::Pool, kDist>;
}

// both instantiations of a weight map (plain head and ssd_policy_lstm_heads_dist) take the whole of shared memory
cudaError_t allow_smem(WeightMap m) {
    const cudaError_t e = cudaFuncSetAttribute(heads_kernel<false>(m), cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
    return e != cudaSuccess ? e : cudaFuncSetAttribute(heads_kernel<true>(m), cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
}

// the arguments only ssd_policy_lstm_heads_dist / ssd_policy_pool_lstm_heads_dist take
bool bad_dist_args(int mode, const int8_t* actions) {
    if (mode != SSD_ACT_SAMPLE && mode != SSD_ACT_GREEDY && mode != SSD_ACT_GIVEN) {
        ssd::set_error(SSD_ERR_INVALID, "mode must be SSD_ACT_SAMPLE, SSD_ACT_GREEDY or SSD_ACT_GIVEN");
        return true;
    }
    if (!actions) {
        ssd::set_error(SSD_ERR_INVALID, "the _dist entry points need actions (output, or input for SSD_ACT_GIVEN)");
        return true;
    }
    return false;
}

// ssd_policy_[pool_]lstm_heads[_dist]: policy_ids is null for a network handle (kDist false: mode, logp and entropy unused)
template <bool kDist>
int heads(ssd_policy_t p, const float* features, const uint8_t* policy_ids, const float* h_in, const float* c_in, float* h_out, float* c_out,
          float* logits, float* value, int mode, int8_t* actions, float* logp, float* entropy, int64_t num_agents, uint64_t seed,
          uint32_t counter, void* stream) {
    using namespace ssd::policy;
    const bool pool = policy_ids != nullptr;
    if (!p || !features || !h_in || !c_in || !h_out || !c_out || !logits || !value || num_agents < 0) return ssd::set_error(SSD_ERR_INVALID, "bad argument");
    if (kDist && bad_dist_args(mode, actions)) return SSD_ERR_INVALID;
    int rc = pool ? check_kind(p, HandleKind::Pool, "not a policy pool handle (ssd_policy_create_pool)")
                  : check_kind(p, HandleKind::Net, kDist ? "a policy pool handle takes ssd_policy_pool_lstm_heads_dist"
                                                         : "a policy pool handle takes ssd_policy_pool_lstm_heads");
    if (rc != SSD_OK) return rc;
    if (!p->d_head_blob) return ssd::set_error(SSD_ERR_INVALID, "ssd_policy_set_head has not been called");
    rc = check_aligned({features, h_in, c_in, h_out, c_out}, "features and state pointers must be 16-byte aligned");
    if (rc != SSD_OK) return rc;
    if (!pool && num_agents % p->num_policies != 0) return ssd::set_error(SSD_ERR_INVALID, "num_agents must be a multiple of num_policies");
    if (num_agents == 0) return SSD_OK;
    rc = setup(p, policy_ids, num_agents, stream);
    if (rc != SSD_OK) return rc;
    const Grid g = grid(p, num_agents);
    heads_kernel<kDist>(weight_map(p))<<<g.ctas, kThreads, kSmemBytes, static_cast<cudaStream_t>(stream)>>>(
        features, h_in, c_in, h_out, c_out, logits, value, actions, num_agents, p->num_outputs, p->d_head_blob, static_cast<uint32_t>(seed),
        static_cast<uint32_t>(seed >> 32), counter, p->num_policies, g.ctas_per_policy, p->d_perm, p->d_tiles, ssd::policy_pool::num_tiles(p), mode,
        logp, entropy);
    return launched();
}

}  // namespace policy_head
}  // namespace ssd

#pragma GCC visibility push(default)
extern "C" {

int ssd_policy_set_head_n(ssd_policy_t p, int num_policies, int units, int num_outputs, const float* lstm_w, const float* lstm_u,
                          const float* lstm_b, const float* logits_w, const float* logits_b, const float* value_w, const float* value_b) {
    if (!p) return ssd::set_error(SSD_ERR_INVALID, "null argument");
    if (num_policies < 1 || num_policies > SSD_MAX_AGENTS) return ssd::set_error(SSD_ERR_INVALID, "num_policies must be 1..SSD_MAX_AGENTS");
    if (num_policies != p->num_policies) return ssd::set_error(SSD_ERR_INVALID, "the head must have as many weight sets as the trunk");
    const int rc = ssd::policy::check_kind(p, HandleKind::Net, "a policy pool's head is loaded by ssd_policy_create_pool",
                                           "an MOA handle is loaded by ssd_moa_create");
    if (rc != SSD_OK) return rc;
    return ssd::policy_head::set_head(p, units, num_outputs, lstm_w, lstm_u, lstm_b, logits_w, logits_b, value_w, value_b);
}
#pragma GCC visibility pop
}  // extern "C"

int ssd::policy_head::set_head(SsdPolicy* p, int units, int num_outputs, const float* lstm_w, const float* lstm_u, const float* lstm_b,
                               const float* logits_w, const float* logits_b, const float* value_w, const float* value_b) {
    using namespace ssd::policy_head;
    if (!lstm_w || !lstm_u || !lstm_b || !logits_w || !logits_b || !value_w || !value_b) return ssd::set_error(SSD_ERR_INVALID, "null argument");
    const int num_policies = p->num_policies;
    if (units != U) return ssd::set_error(SSD_ERR_UNSUPPORTED, "the fused LSTM kernel is built for cell_size 128 (conv_to_fcnet_v2.py's custom_options)");
    if (num_outputs < 1 || num_outputs > NH - 1) return ssd::set_error(SSD_ERR_UNSUPPORTED, "1..15 policy outputs");
    const size_t blob_bytes = static_cast<size_t>(num_policies) * kBlobBytes;
    std::vector<uint8_t> blobs(blob_bytes, 0);
    using ssd::policy::kmajor;
    for (int q = 0; q < num_policies; ++q) {  // weight set q: arrays q of the num_policies consecutive ones behind each pointer
        uint8_t* blob = blobs.data() + static_cast<size_t>(q) * kBlobBytes;
        const float* ow = logits_w + q * U * num_outputs;
        const float* ob = logits_b + q * num_outputs;
        const float* vw = value_w + q * U;
        const float* vb = value_b + q;
        __half* bh = reinterpret_cast<__half*>(blob + kOffBH);
        float* cst = reinterpret_cast<float*>(blob + kOffConst);
        pack_gates(reinterpret_cast<__half*>(blob + kOffB), cst, lstm_w + static_cast<size_t>(q) * KX * NG, lstm_u + static_cast<size_t>(q) * U * NG,
                   lstm_b + q * NG);
        for (int k = 0; k < U; ++k) {
            for (int n = 0; n < num_outputs; ++n) bh[kmajor(NH, n, k)] = __float2half_rn(ow[k * num_outputs + n]);
            bh[kmajor(NH, num_outputs, k)] = __float2half_rn(vw[k]);
        }
        for (int n = 0; n < num_outputs; ++n) cst[NG + n] = ob[n];
        cst[NG + num_outputs] = vb[0];
    }
    cudaError_t e = cudaSetDevice(p->device);
    if (e == cudaSuccess && !p->d_head_blob) e = cudaMalloc(&p->d_head_blob, blob_bytes);
    if (e == cudaSuccess) e = cudaMemcpy(p->d_head_blob, blobs.data(), blob_bytes, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = allow_smem(ssd::policy::weight_map(p));
    if (e != cudaSuccess) return ssd::set_error(SSD_ERR_CUDA, cudaGetErrorString(e));
    p->units = units;
    p->num_outputs = num_outputs;
    return SSD_OK;
}

#pragma GCC visibility push(default)
extern "C" {

int ssd_policy_set_head(ssd_policy_t p, int units, int num_outputs, const float* lstm_w, const float* lstm_u, const float* lstm_b,
                        const float* logits_w, const float* logits_b, const float* value_w, const float* value_b) {
    return ssd_policy_set_head_n(p, 1, units, num_outputs, lstm_w, lstm_u, lstm_b, logits_w, logits_b, value_w, value_b);
}

int ssd_policy_lstm_heads(ssd_policy_t p, const float* features, const float* h_in, const float* c_in, float* h_out, float* c_out, float* logits,
                          float* value, int8_t* actions, int64_t num_agents, uint64_t seed, uint32_t counter, void* stream) {
    return ssd::policy_head::heads<false>(p, features, nullptr, h_in, c_in, h_out, c_out, logits, value, 0, actions, nullptr, nullptr, num_agents,
                                          seed, counter, stream);
}

int ssd_policy_lstm_heads_dist(ssd_policy_t p, const float* features, const float* h_in, const float* c_in, float* h_out, float* c_out,
                               float* logits, float* value, int mode, int8_t* actions, float* logp, float* entropy, int64_t num_agents,
                               uint64_t seed, uint32_t counter, void* stream) {
    return ssd::policy_head::heads<true>(p, features, nullptr, h_in, c_in, h_out, c_out, logits, value, mode, actions, logp, entropy, num_agents,
                                         seed, counter, stream);
}

int ssd_policy_pool_lstm_heads(ssd_policy_t p, const float* features, const uint8_t* policy_ids, const float* h_in, const float* c_in, float* h_out,
                               float* c_out, float* logits, float* value, int8_t* actions, int64_t num_agents, uint64_t seed, uint32_t counter,
                               void* stream) {
    if (!policy_ids) return ssd::set_error(SSD_ERR_INVALID, "bad argument");
    return ssd::policy_head::heads<false>(p, features, policy_ids, h_in, c_in, h_out, c_out, logits, value, 0, actions, nullptr, nullptr,
                                          num_agents, seed, counter, stream);
}

int ssd_policy_pool_lstm_heads_dist(ssd_policy_t p, const float* features, const uint8_t* policy_ids, const float* h_in, const float* c_in,
                                    float* h_out, float* c_out, float* logits, float* value, int mode, int8_t* actions, float* logp,
                                    float* entropy, int64_t num_agents, uint64_t seed, uint32_t counter, void* stream) {
    if (!policy_ids) return ssd::set_error(SSD_ERR_INVALID, "bad argument");
    return ssd::policy_head::heads<true>(p, features, policy_ids, h_in, c_in, h_out, c_out, logits, value, mode, actions, logp, entropy, num_agents,
                                         seed, counter, stream);
}

}  // extern "C"
#pragma GCC visibility pop
