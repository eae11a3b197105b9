// Advantages and value targets of a [T][M] trajectory on the device: RLlib's compute_advantages (GAE and discounted returns) and
// V-trace's from_importance_weights, with episode ends and the weighted influence reward (DESIGN.md section 5.8).
//
// All three modes are one affine recurrence per agent, run backwards in time:
//     acc_t = x_t + k_t * acc_{t+1}                       no done at t
//     acc_t = x_t, every (t+1) term of x_t dropped        done at t (a select: nothing of t+1 is multiplied by zero)
// with r_t = float(rewards_t) + w * intrinsic_t, V_T = bootstrap and
//     GAE      x_t = (r_t + g V_{t+1}) - V_t              k_t = g lambda   adv = acc, value_targets = acc + V_t        acc_T = 0
//     returns  x_t = r_t                                  k_t = g          adv = acc                                   acc_T = bootstrap
//     V-trace  x_t = rho_bar_t ((r_t + g V_{t+1}) - V_t)  k_t = g c_t      vs = acc + V_t,                             acc_T = 0
//              pg_t = rho_pg_t ((r_t + g vs_{t+1}) - V_t), vs_T = bootstrap;  rho = exp(target_logp - behaviour_logp),
//              rho_bar = min(rho_bar_max, rho), c = min(1, rho), rho_pg = min(rho_pg_max, rho) (the min passes a NaN rho on)
//
// Two paths, chosen from (T, M, SM count) by num_chunks():
//   - C = 1: one thread per agent walks t = T-1 .. 0.  Loads of a step are coalesced across the agents of a warp, and the loads of
//     kGroup steps are issued before any of them is used (they do not depend on acc).  Every input is read once, every output
//     written once.
//   - C > 1 (few agents, long T): time is split into C chunks of L steps.  summary_kernel composes each chunk's affine map
//     acc_s = D ? X : X + K acc_e ("D": the chunk contains a done) into the caller's workspace; finish_kernel then gives every
//     (chunk, agent) its carry acc_e by applying the later chunks' maps to acc_T, and walks its chunk from that carry.
#include <cstdint>

#include "ssd_internal.h"

namespace ssd {
namespace adv {

enum Mode { kGae = 0, kReturns = 1, kVtrace = 2 };

constexpr int kThreads = 128;
constexpr int kUnroll = 8;          // steps whose loads are in flight together (chunk maps in finish_kernel, too)
// V-trace loads six words a step: with eight steps ptxas sinks most of the 48 loads next to their uses (about two steps in
// flight), with four it issues all 24 first, as it does for the 32 loads of eight GAE steps.
template <int kMode>
constexpr int kGroup = kMode == kVtrace ? 4 : kUnroll;
constexpr int kMinChunk = 16;       // steps per chunk at least
constexpr int kMaxChunks = 64;      // the carry walk of finish_kernel is O(C) per thread
constexpr int kThreadsPerSm = 2048;
constexpr int kMaxSms = 256;        // ssd_advantages_workspace_bytes sizes the workspace for any device up to this many SMs

struct Args {
    int64_t T, M, B, L;             // B = M / N envs; L = steps per chunk (T for C = 1)
    int N;
    const uint32_t* rew;            // int32 or float32 words, as rew_int says
    bool rew_int;
    const float* intr;              // may be null
    float w;
    const float* v;
    const uint8_t* d;               // [T][B]
    const float* boot;
    const float* tl;                // V-trace only
    const float* bl;
    float gamma, k, rho_max, pg_max; // k = g lambda (GAE), g (returns, V-trace)
    float* out0;                    // advantages (GAE, returns) or vs (V-trace)
    float* out1;                    // value_targets (GAE) or pg_advantages (V-trace)
    float2* sum_kx;                 // [C][M] (K, X) of each chunk
    uint8_t* sum_d;                 // [C][M] D of each chunk
};

// The words of one step as loaded: nothing here is converted or compared, so that no instruction between the loads of a group
// waits for one of them.
struct StepIn {
    uint32_t r, d;
    float i, v, tl, bl;
};

__device__ __forceinline__ float min_nan(float thr, float x) { return x > thr ? thr : x; }   // min(thr, x); a NaN x stays NaN

// Read-only loads as volatile asm: the compiler keeps them in program order, ahead of the arithmetic that consumes them, instead
// of sinking each next to its first use (which it does for the V-trace group, whose expf raises the register pressure).
__device__ __forceinline__ uint32_t ld_u32(const void* p) {
    uint32_t x;
    asm volatile("ld.global.nc.u32 %0, [%1];" : "=r"(x) : "l"(p));
    return x;
}
__device__ __forceinline__ uint32_t ld_u8(const uint8_t* p) {
    uint32_t x;
    asm volatile("ld.global.nc.u8 %0, [%1];" : "=r"(x) : "l"(p));
    return x;
}
__device__ __forceinline__ float ld_f32(const float* p) { return __uint_as_float(ld_u32(p)); }

// o = t M + m (the agent's element of step t), od = t B + b (its env's done byte).
template <int kMode>
__device__ __forceinline__ StepIn load_step(const Args& a, int64_t o, int64_t od) {
    StepIn s;
    s.r = ld_u32(a.rew + o);
    s.i = a.intr ? ld_f32(a.intr + o) : 0.0f;
    s.v = kMode != kReturns ? ld_f32(a.v + o) : 0.0f;
    s.d = ld_u8(a.d + od);
    if (kMode == kVtrace) {
        s.tl = ld_f32(a.tl + o);
        s.bl = ld_f32(a.bl + o);
    }
    return s;
}

// r_t = float(rewards_t) + w * intrinsic_t
__device__ __forceinline__ float step_reward(const Args& a, const StepIn& s) {
    float r = a.rew_int ? static_cast<float>(static_cast<int32_t>(s.r)) : __uint_as_float(s.r);
    if (a.intr) r += a.w * s.i;
    return r;
}

// Runs steps t0-1 .. t0-kCount of agent m from acc = acc_{t0}, vn = V_{t0}: all kCount steps' loads are issued first (they do
// not depend on acc), then the serial part.  kSummary: writes nothing and composes the map instead: started at acc = 0, K = 1,
// D = false, the walk of a chunk returns acc_s = D ? acc : acc + K acc_e.
template <int kMode, bool kSummary, int kCount>
__device__ __forceinline__ void steps(const Args& a, int64_t m, int64_t b, int64_t t0, float& acc, float& vn, float& K, bool& D) {
    const int64_t o0 = (t0 - 1) * a.M + m, od0 = (t0 - 1) * a.B + b;
    StepIn in[kCount];
#pragma unroll
    for (int j = 0; j < kCount; ++j) in[j] = load_step<kMode>(a, o0 - j * a.M, od0 - j * a.B);
#pragma unroll
    for (int j = 0; j < kCount; ++j) {
        const bool done = in[j].d != 0;
        const float r = step_reward(a, in[j]), v = in[j].v;
        float x, k, rho = 0.0f;
        if (kMode == kReturns) {
            x = r;
            k = a.k;
        } else {
            const float delta = done ? r - v : (r + a.gamma * vn) - v;
            if (kMode == kGae) {
                x = delta;
                k = a.k;
            } else {
                rho = expf(in[j].tl - in[j].bl);
                x = min_nan(a.rho_max, rho) * delta;
                k = a.gamma * min_nan(1.0f, rho);
            }
        }
        const float vs_next = acc + vn;   // V-trace: vs_{t+1} (acc_T + V_T = 0 + bootstrap at t = T-1)
        acc = done ? x : x + k * acc;
        if (kSummary) {
            K *= k;                       // not used once D is set
            D = D || done;
        } else {
            const int64_t o = o0 - j * a.M;
            if (kMode == kGae) {
                a.out0[o] = acc;
                a.out1[o] = acc + v;
            } else if (kMode == kReturns) {
                a.out0[o] = acc;
            } else {
                a.out0[o] = acc + v;
                const float pg = done ? r - v : (r + a.gamma * vs_next) - v;
                a.out1[o] = min_nan(a.pg_max, rho) * pg;
            }
        }
        vn = v;
    }
}

// Walks steps e-1 .. s of agent m backwards: full groups of kGroup steps without a bound check, then the rest one by one.
template <int kMode, bool kSummary>
__device__ __forceinline__ void walk(const Args& a, int64_t m, int64_t s, int64_t e, float& acc, float vn, float& K, bool& D) {
    const int64_t b = m / a.N;
    int64_t t0 = e;
    for (; t0 - kGroup<kMode> >= s; t0 -= kGroup<kMode>) steps<kMode, kSummary, kGroup<kMode>>(a, m, b, t0, acc, vn, K, D);
    for (; t0 > s; --t0) steps<kMode, kSummary, 1>(a, m, b, t0, acc, vn, K, D);
}

template <int kMode>
__device__ __forceinline__ float acc_end(const Args& a, int64_t m) { return kMode == kReturns ? __ldg(a.boot + m) : 0.0f; }

// V_e: values[e], or the bootstrap at e = T (the returns mode reads neither).
template <int kMode>
__device__ __forceinline__ float v_at(const Args& a, int64_t e, int64_t m) {
    if (kMode == kReturns) return 0.0f;
    return e < a.T ? __ldg(a.v + e * a.M + m) : __ldg(a.boot + m);
}

__device__ __forceinline__ int64_t chunk_end(const Args& a, int64_t s) { return s + a.L < a.T ? s + a.L : a.T; }

// C = 1: one thread per agent over the whole trajectory.
template <int kMode>
__global__ void __launch_bounds__(kThreads) single_kernel(Args a) {
    const int64_t m = static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x;
    if (m >= a.M) return;
    float acc = acc_end<kMode>(a, m), K = 1.0f;
    bool D = false;
    walk<kMode, false>(a, m, 0, a.T, acc, v_at<kMode>(a, a.T, m), K, D);
}

// C > 1, pass 1: the map (K, X, D) of chunk blockIdx.y + 1 (chunk 0's map is never needed).
template <int kMode>
__global__ void __launch_bounds__(kThreads) summary_kernel(Args a) {
    const int64_t m = static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x;
    if (m >= a.M) return;
    const int64_t c = blockIdx.y + 1, s = c * a.L, e = chunk_end(a, s);
    float X = 0.0f, K = 1.0f;
    bool D = false;
    walk<kMode, true>(a, m, s, e, X, v_at<kMode>(a, e, m), K, D);
    a.sum_kx[c * a.M + m] = make_float2(K, X);
    a.sum_d[c * a.M + m] = D;
}

// Applies the map of chunk q to acc.
__device__ __forceinline__ float apply_map(float2 kx, uint8_t d, float acc) { return d ? kx.y : kx.y + kx.x * acc; }

// C > 1, pass 2: chunk blockIdx.y from its carry acc_e, the maps of chunks C-1 .. c+1 applied to acc_T.  The maps are loaded
// kUnroll at a time before they are applied, so the carry costs about (C - 1 - c) / kUnroll round trips to L2, not C - 1 - c.
template <int kMode>
__global__ void __launch_bounds__(kThreads) finish_kernel(Args a, int C) {
    const int64_t m = static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x;
    if (m >= a.M) return;
    const int c = blockIdx.y;
    float acc = acc_end<kMode>(a, m), K = 1.0f;
    int q = C - 1;
    for (; q - kUnroll >= c; q -= kUnroll) {
        float2 kx[kUnroll];
        uint8_t d[kUnroll];
#pragma unroll
        for (int j = 0; j < kUnroll; ++j) {
            kx[j] = a.sum_kx[static_cast<int64_t>(q - j) * a.M + m];
            d[j] = a.sum_d[static_cast<int64_t>(q - j) * a.M + m];
        }
#pragma unroll
        for (int j = 0; j < kUnroll; ++j) acc = apply_map(kx[j], d[j], acc);
    }
    for (; q > c; --q) acc = apply_map(a.sum_kx[static_cast<int64_t>(q) * a.M + m], a.sum_d[static_cast<int64_t>(q) * a.M + m], acc);
    const int64_t s = c * a.L, e = chunk_end(a, s);
    bool D = false;
    walk<kMode, false>(a, m, s, e, acc, v_at<kMode>(a, e, m), K, D);
}

// C for a call: one chunk when the agents alone give every SM a quarter of its threads (the chunked path reads the inputs twice),
// else enough chunks of at least kMinChunk steps to fill the SMs, at most kMaxChunks.  Non-decreasing in sms.
inline int num_chunks(int64_t T, int64_t M, int sms) {
    const int64_t target = static_cast<int64_t>(sms < kMaxSms ? sms : kMaxSms) * kThreadsPerSm;
    if (4 * M >= target) return 1;
    int64_t c = (target + M - 1) / M;
    if (c > T / kMinChunk) c = T / kMinChunk;
    if (c > kMaxChunks) c = kMaxChunks;
    if (c <= 1) return 1;
    const int64_t L = (T + c - 1) / c;   // no empty chunk
    return static_cast<int>((T + L - 1) / L);
}

// (K, X) as float2 then D as bytes, each array 16-byte aligned.
inline int64_t kx_bytes(int64_t C, int64_t M) { return (C * M * 8 + 15) / 16 * 16; }
inline int64_t workspace_bytes(int64_t C, int64_t M) { return C <= 1 ? 0 : kx_bytes(C, M) + (C * M + 15) / 16 * 16; }

inline bool aligned4(const void* p) { return reinterpret_cast<uintptr_t>(p) % 4 == 0; }

template <int kMode>
int launch(Args a, void* workspace, cudaStream_t stream) {
    int dev = 0, sms = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess) return set_error(SSD_ERR_CUDA, cudaGetErrorString(e));
    const int C = num_chunks(a.T, a.M, sms);
    const unsigned blocks = static_cast<unsigned>((a.M + kThreads - 1) / kThreads);
    if (C == 1) {
        a.L = a.T;
        single_kernel<kMode><<<blocks, kThreads, 0, stream>>>(a);
    } else {
        a.L = (a.T + C - 1) / C;
        a.sum_kx = static_cast<float2*>(workspace);
        a.sum_d = static_cast<uint8_t*>(workspace) + kx_bytes(C, a.M);
        summary_kernel<kMode><<<dim3(blocks, C - 1), kThreads, 0, stream>>>(a);
        finish_kernel<kMode><<<dim3(blocks, C), kThreads, 0, stream>>>(a, C);
    }
    e = cudaGetLastError();
    return e == cudaSuccess ? SSD_OK : set_error(SSD_ERR_CUDA, cudaGetErrorString(e));
}

// The checks every mode shares; SSD_OK or SSD_ERR_INVALID.  Nothing here touches a device.
int check_common(int64_t T, int64_t M, int N, const void* rewards, int reward_dtype, const float* intrinsic, const float* values,
                 const uint8_t* dones, const float* bootstrap, float gamma, const void* workspace, int64_t workspace_bytes_given) {
    if (!rewards || !values || !dones || !bootstrap) return set_error(SSD_ERR_INVALID, "null input pointer");
    if (T <= 0 || M <= 0) return set_error(SSD_ERR_INVALID, "T and M must be positive");
    if (N <= 0 || M % N != 0) return set_error(SSD_ERR_INVALID, "M must be a positive multiple of num_agents");
    if (reward_dtype != SSD_DTYPE_I32 && reward_dtype != SSD_DTYPE_F32) return set_error(SSD_ERR_INVALID, "unknown reward dtype");
    if (!(gamma >= 0.0f && gamma <= 1.0f)) return set_error(SSD_ERR_INVALID, "gamma must be in [0, 1]");
    if (!aligned4(rewards) || !aligned4(intrinsic) || !aligned4(values) || !aligned4(bootstrap))
        return set_error(SSD_ERR_INVALID, "float and int32 arrays must be 4-byte aligned");
    const int64_t need = workspace_bytes(num_chunks(T, M, kMaxSms), M);
    if (need > 0 && (!workspace || workspace_bytes_given < need)) return set_error(SSD_ERR_INVALID, "workspace too small (ssd_advantages_workspace_bytes)");
    if (need > 0 && reinterpret_cast<uintptr_t>(workspace) % 16 != 0) return set_error(SSD_ERR_INVALID, "workspace must be 16-byte aligned");
    return SSD_OK;
}

Args make_args(int64_t T, int64_t M, int N, const void* rewards, int reward_dtype, const float* intrinsic, float intrinsic_weight,
               const float* values, const uint8_t* dones, const float* bootstrap, float gamma) {
    Args a{};
    a.T = T;
    a.M = M;
    a.N = N;
    a.B = M / N;
    a.rew = static_cast<const uint32_t*>(rewards);
    a.rew_int = reward_dtype == SSD_DTYPE_I32;
    a.intr = intrinsic;
    a.w = intrinsic_weight;
    a.v = values;
    a.d = dones;
    a.boot = bootstrap;
    a.gamma = gamma;
    return a;
}

}  // namespace adv
}  // namespace ssd

#pragma GCC visibility push(default)
extern "C" {

int64_t ssd_advantages_workspace_bytes(int64_t T, int64_t M) {
    if (T <= 0 || M <= 0) return 0;
    using namespace ssd::adv;
    return workspace_bytes(num_chunks(T, M, kMaxSms), M);
}

int ssd_advantages(int mode, int64_t T, int64_t M, int num_agents, const void* rewards, int reward_dtype, const float* intrinsic,
                   float intrinsic_weight, const float* values, const uint8_t* dones, const float* bootstrap, float gamma, float lambda,
                   float* advantages, float* value_targets, void* workspace, int64_t workspace_bytes, void* stream) {
    using namespace ssd::adv;
    if (mode != SSD_ADV_GAE && mode != SSD_ADV_RETURNS) return ssd::set_error(SSD_ERR_INVALID, "mode must be SSD_ADV_GAE or SSD_ADV_RETURNS");
    const int rc = check_common(T, M, num_agents, rewards, reward_dtype, intrinsic, values, dones, bootstrap, gamma, workspace, workspace_bytes);
    if (rc != SSD_OK) return rc;
    if (!advantages) return ssd::set_error(SSD_ERR_INVALID, "null output pointer");
    if (mode == SSD_ADV_GAE && !value_targets) return ssd::set_error(SSD_ERR_INVALID, "null output pointer");
    if (mode == SSD_ADV_RETURNS && value_targets) return ssd::set_error(SSD_ERR_INVALID, "SSD_ADV_RETURNS writes no value targets: pass NULL");
    if (mode == SSD_ADV_GAE && !(lambda >= 0.0f && lambda <= 1.0f)) return ssd::set_error(SSD_ERR_INVALID, "lambda must be in [0, 1]");
    if (!aligned4(advantages) || !aligned4(value_targets)) return ssd::set_error(SSD_ERR_INVALID, "float and int32 arrays must be 4-byte aligned");
    Args a = make_args(T, M, num_agents, rewards, reward_dtype, intrinsic, intrinsic_weight, values, dones, bootstrap, gamma);
    a.out0 = advantages;
    a.out1 = value_targets;
    const cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (mode == SSD_ADV_GAE) {
        a.k = gamma * lambda;
        return launch<kGae>(a, workspace, s);
    }
    a.k = gamma;
    return launch<kReturns>(a, workspace, s);
}

int ssd_vtrace(int64_t T, int64_t M, int num_agents, const void* rewards, int reward_dtype, const float* intrinsic, float intrinsic_weight,
               const float* values, const uint8_t* dones, const float* bootstrap, const float* target_logp, const float* behaviour_logp,
               float gamma, float clip_rho_threshold, float clip_pg_rho_threshold, float* vs, float* pg_advantages, void* workspace,
               int64_t workspace_bytes, void* stream) {
    using namespace ssd::adv;
    if (!target_logp || !behaviour_logp) return ssd::set_error(SSD_ERR_INVALID, "null input pointer");
    const int rc = check_common(T, M, num_agents, rewards, reward_dtype, intrinsic, values, dones, bootstrap, gamma, workspace, workspace_bytes);
    if (rc != SSD_OK) return rc;
    if (!vs || !pg_advantages) return ssd::set_error(SSD_ERR_INVALID, "null output pointer");
    if (!(clip_rho_threshold >= 0.0f) || !(clip_pg_rho_threshold >= 0.0f)) return ssd::set_error(SSD_ERR_INVALID, "clip thresholds must be >= 0 (+inf: no clip)");
    if (!aligned4(target_logp) || !aligned4(behaviour_logp) || !aligned4(vs) || !aligned4(pg_advantages))
        return ssd::set_error(SSD_ERR_INVALID, "float and int32 arrays must be 4-byte aligned");
    Args a = make_args(T, M, num_agents, rewards, reward_dtype, intrinsic, intrinsic_weight, values, dones, bootstrap, gamma);
    a.tl = target_logp;
    a.bl = behaviour_logp;
    a.k = gamma;
    a.rho_max = clip_rho_threshold;
    a.pg_max = clip_pg_rho_threshold;
    a.out0 = vs;
    a.out1 = pg_advantages;
    return launch<kVtrace>(a, workspace, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
#pragma GCC visibility pop
