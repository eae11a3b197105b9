// Policy pool (ssd_policy_create_pool): K <= 255 weight sets loaded once, agent m evaluated with set policy_ids[m] of the
// call.  The trunk and head kernels take the grouping of agents by policy from the assignment built here, on the device:
//
//   count    per-policy counts: a CTA histograms a chunk of ids in shared memory (one atomic per run of equal ids in a warp),
//            then adds its nonzero bins to the global counts;
//   plan     one CTA: exclusive prefix sums of the counts and of the tile counts ceil(count / 128); the tile table
//            (policy, first, count <= 128) in policy order; the cursors of the scatter; the counts are zeroed for the next
//            call (the handle allocates them zeroed);
//   scatter  a CTA histograms its chunk again, reserves a range per policy with one global atomic per bin, and writes each
//            agent to perm[cursor + rank].  The order of agents within a policy depends on the timing of those atomics; it
//            does not change any result (an agent is one accumulator row / one drain thread in both kernels).
//
// Ids >= K are skipped: they get no perm entry and no tile, so the kernels write nothing for those agents.
#include <new>

#include "ssd_internal.h"
#include "ssd_policy.h"

namespace ssd {
namespace policy_pool {

constexpr int kThreads = 256, kPerThread = 16, kChunk = kThreads * kPerThread;   // agents per CTA of count / scatter
constexpr int kGA = 128;                                                          // agents per tile (UMMA M)

// Histogram of the chunk's ids < K into h[kBins] (zeroed by the caller).  Every lane of every warp runs the same iterations.
__device__ __forceinline__ void chunk_histogram(const uint8_t* __restrict__ ids, long long M, int K, uint32_t* h) {
    const long long c0 = static_cast<long long>(blockIdx.x) * kChunk;
    const int lane = threadIdx.x & 31;
#pragma unroll 4
    for (int j = 0; j < kPerThread; ++j) {
        const long long m = c0 + j * kThreads + threadIdx.x;
        const int id = m < M ? ids[m] : kBins;
        const unsigned peers = __match_any_sync(0xffffffffu, id);
        if (id < K && lane == __ffs(peers) - 1) atomicAdd(h + id, __popc(peers));
    }
}

__global__ void __launch_bounds__(kThreads) pool_count_kernel(const uint8_t* __restrict__ ids, long long M, int K, uint32_t* __restrict__ counts) {
    __shared__ uint32_t h[kBins];
    h[threadIdx.x] = 0;
    __syncthreads();
    chunk_histogram(ids, M, K, h);
    __syncthreads();
    if (h[threadIdx.x]) atomicAdd(counts + threadIdx.x, h[threadIdx.x]);
}

__global__ void __launch_bounds__(kBins) pool_plan_kernel(int K, uint32_t* __restrict__ counts, PoolTile* __restrict__ tiles) {
    __shared__ uint32_t s_off[kBins + 1], s_tile[kBins + 1];
    const int k = threadIdx.x;
    const uint32_t c = k < K ? counts[k] : 0;
    counts[k] = 0;
    // inclusive scans (Hillis-Steele over 256 entries) of the agent and tile counts; entry k + 1 = everything before policy k + 1
    s_off[k + 1] = c;
    s_tile[k + 1] = (c + kGA - 1) / kGA;
    if (k == 0) s_off[0] = s_tile[0] = 0;
    __syncthreads();
    for (int d = 1; d < kBins; d <<= 1) {
        const uint32_t a = k >= d ? s_off[k + 1 - d] : 0, t = k >= d ? s_tile[k + 1 - d] : 0;
        __syncthreads();
        s_off[k + 1] += a;
        s_tile[k + 1] += t;
        __syncthreads();
    }
    counts[kOffCursor + k] = s_off[k];
    const uint32_t n_tiles = s_tile[kBins];
    if (k == 0) counts[kOffNumTiles] = n_tiles;
    for (uint32_t j = k; j < n_tiles; j += kBins) {   // tile j belongs to the policy q with s_tile[q] <= j < s_tile[q + 1]
        int lo = 0, hi = kBins - 1;
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (s_tile[mid] <= j) lo = mid; else hi = mid - 1;
        }
        const uint32_t i = j - s_tile[lo], n = s_off[lo + 1] - s_off[lo];
        tiles[j] = PoolTile{s_off[lo] + i * kGA, static_cast<uint16_t>(lo), static_cast<uint16_t>(n - i * kGA < kGA ? n - i * kGA : kGA)};
    }
}

__global__ void __launch_bounds__(kThreads) pool_scatter_kernel(const uint8_t* __restrict__ ids, long long M, int K, uint32_t* __restrict__ cursor,
                                                                 uint32_t* __restrict__ perm) {
    __shared__ uint32_t h[kBins], base[kBins];
    h[threadIdx.x] = 0;
    __syncthreads();
    chunk_histogram(ids, M, K, h);
    __syncthreads();
    if (h[threadIdx.x]) base[threadIdx.x] = atomicAdd(cursor + threadIdx.x, h[threadIdx.x]);
    h[threadIdx.x] = 0;
    __syncthreads();
    const long long c0 = static_cast<long long>(blockIdx.x) * kChunk;
    const int lane = threadIdx.x & 31;
#pragma unroll 4
    for (int j = 0; j < kPerThread; ++j) {
        const long long m = c0 + j * kThreads + threadIdx.x;
        const int id = m < M ? ids[m] : kBins;
        const unsigned peers = __match_any_sync(0xffffffffu, id);
        const int leader = __ffs(peers) - 1;
        uint32_t at = 0;
        if (id < K && lane == leader) at = atomicAdd(h + id, __popc(peers));
        at = __shfl_sync(0xffffffffu, at, leader);
        if (id < K) perm[base[id] + at + __popc(peers & ((1u << lane) - 1))] = static_cast<uint32_t>(m);
    }
}

int assign(SsdPolicy* p, const uint8_t* policy_ids, long long M, void* stream) {
    if (M > 0x7fffffffLL) return ssd::set_error(SSD_ERR_INVALID, "a policy pool takes at most 2^31 - 1 agents per call");
    if (cudaSetDevice(p->device) != cudaSuccess) return ssd::set_error(SSD_ERR_CUDA, "cudaSetDevice failed");
    const int K = p->num_policies;
    const long long need_tiles = max_tiles(M, K);
    cudaError_t e = cudaSuccess;
    if (M > p->perm_cap || need_tiles > p->tile_cap) {   // grow the scratch (cudaFree waits for work that may still read it)
        cudaFree(p->d_perm);
        cudaFree(p->d_tiles);
        p->d_perm = nullptr;
        p->d_tiles = nullptr;
        p->perm_cap = p->tile_cap = 0;
        e = cudaMalloc(&p->d_perm, M * sizeof(uint32_t));
        if (e == cudaSuccess) e = cudaMalloc(&p->d_tiles, need_tiles * sizeof(PoolTile));
        if (e != cudaSuccess) return ssd::set_error(SSD_ERR_CUDA, cudaGetErrorString(e));
        p->perm_cap = M;
        p->tile_cap = need_tiles;
    }
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    const unsigned chunks = static_cast<unsigned>((M + kChunk - 1) / kChunk);
    pool_count_kernel<<<chunks, kThreads, 0, st>>>(policy_ids, M, K, p->d_counts);
    pool_plan_kernel<<<1, kBins, 0, st>>>(K, p->d_counts, p->d_tiles);
    pool_scatter_kernel<<<chunks, kThreads, 0, st>>>(policy_ids, M, K, p->d_counts + kOffCursor, p->d_perm);
    return ssd::policy::launched();
}

}  // namespace policy_pool
}  // namespace ssd

#pragma GCC visibility push(default)
extern "C" {

int ssd_policy_create_pool(int view_radius, int device, int num_policies, int units, int num_outputs, const float* conv_w, const float* conv_b,
                           const float* fc1_w, const float* fc1_b, const float* fc2_w, const float* fc2_b, const float* lstm_w, const float* lstm_u,
                           const float* lstm_b, const float* logits_w, const float* logits_b, const float* value_w, const float* value_b,
                           ssd_policy_t* out) {
    using namespace ssd::policy_pool;
    if (!out) return ssd::set_error(SSD_ERR_INVALID, "null argument");
    *out = nullptr;
    if (num_policies < 1 || num_policies > kBins - 1) return ssd::set_error(SSD_ERR_INVALID, "a policy pool holds 1..255 weight sets");
    if (!lstm_w || !lstm_u || !lstm_b || !logits_w || !logits_b || !value_w || !value_b) return ssd::set_error(SSD_ERR_INVALID, "null weight pointer");
    if (units != 128) return ssd::set_error(SSD_ERR_UNSUPPORTED, "a policy pool needs the fused LSTM kernel: cell_size 128");
    if (num_outputs < 1 || num_outputs > 15) return ssd::set_error(SSD_ERR_UNSUPPORTED, "a policy pool needs the fused heads: 1..15 policy outputs");
    ssd_policy_t p = nullptr;
    int rc = ssd::policy::create_trunk(view_radius, device, num_policies, WeightMap::Pool, conv_w, conv_b, fc1_w, fc1_b, fc2_w, fc2_b, &p);
    if (rc != SSD_OK) return rc;
    rc = ssd::policy_head::set_head(p, units, num_outputs, lstm_w, lstm_u, lstm_b, logits_w, logits_b, value_w, value_b);
    if (rc == SSD_OK) {
        cudaError_t e = cudaMalloc(&p->d_counts, kCountWords * sizeof(uint32_t));
        if (e == cudaSuccess) e = cudaMemset(p->d_counts, 0, kCountWords * sizeof(uint32_t));
        if (e != cudaSuccess) rc = ssd::set_error(SSD_ERR_CUDA, cudaGetErrorString(e));
    }
    if (rc != SSD_OK) {
        ssd_policy_destroy(p);
        return rc;
    }
    *out = p;
    return SSD_OK;
}

}  // extern "C"
#pragma GCC visibility pop
