// Host-side handle of the policy kernels (ssd_policy.cu: trunk; ssd_policy_head.cu: LSTM + heads; ssd_policy_moa.cu: model of
// other agents; ssd_policy_pool.cu: the assignment of agents to the weight sets of a policy pool), and what their kernels and
// entry points share: the map of agents to groups, the grid, the launch and argument checks.
#pragma once
#include <cstdint>
#include <initializer_list>

#include "ssd_internal.h"

// How the policy kernels map agents to weight sets: one set for all agents, set m % P for agent m (one network per agent id),
// or set policy_ids[m] for agent m (a policy pool; agents grouped by ssd::policy_pool::assign).
enum class WeightMap { Shared, PerAgent, Pool };

// What made a handle: ssd_policy_create[_n] (Net), ssd_policy_create_pool (Pool) or ssd_moa_create (Moa).
enum class HandleKind { Net, Pool, Moa };

// One tile of a pool's assignment: agents perm[first, first + count), count <= 128, all evaluated with weight set `policy`.
struct PoolTile {
    uint32_t first;
    uint16_t policy, count;
};

struct SsdPolicy {
    int device = 0;
    int sms = 0;
    HandleKind kind = HandleKind::Net;
    uint8_t* d_blob = nullptr;       // packed trunk weights
    uint8_t* d_head_blob = nullptr;  // packed LSTM / head weights (ssd_policy_set_head)
    int units = 0, num_outputs = 0;
    int num_policies = 1;            // weight sets: agent m = b * P + p uses set p (ssd_policy_create_n), or set ids[m] (pool)
    // Moa: d_head_blob holds the MOA's resident weights, d_moa_rows its one-hot rows and moa_logits_w, num_outputs its A,
    // moa_agents its N
    int moa_agents = 0;
    float* d_moa_rows = nullptr;
    // pool scratch, grown on demand: per-policy counts [256] and cursors [256], the tile count, perm [M], tiles [M / 128 + K]
    uint32_t* d_counts = nullptr;
    uint32_t* d_perm = nullptr;
    PoolTile* d_tiles = nullptr;
    long long perm_cap = 0, tile_cap = 0;
};

// Shared and PerAgent weight maps, per CTA: agent m = b * P + p uses weight set p, and CTA c serves set pol = c % P only, its
// groups g = cta, cta + stride, ... < n_groups of 128 agents (b, pol), b in [128 g, 128 g + 128).  A UMMA tile cannot change
// its B operand per row, so each CTA loads one set's weights once.  The recurrent state of group g is state group
// pol * n_groups + g.  Shared is P = 1.
template <WeightMap kMap>
struct GroupMap {
    static constexpr bool kPerAgent = kMap != WeightMap::Shared;
    int np, pol;                              // P; this CTA's weight set
    long long cta, stride, rows, n_groups;    // its first group, the step to its next one; agents and groups per weight set
    __device__ __forceinline__ GroupMap(long long M, int num_policies, int ctas_per_policy)
        : np(kPerAgent ? num_policies : 1),
          pol(kPerAgent ? static_cast<int>(blockIdx.x) % np : 0),
          cta(kPerAgent ? blockIdx.x / np : blockIdx.x),
          stride(kPerAgent ? ctas_per_policy : gridDim.x),
          rows(kPerAgent ? M / np : M),
          n_groups((rows + 127) / 128) {}
    __device__ __forceinline__ long long agent(long long a0, int row) const { return (a0 + row) * np + pol; }   // a0 = 128 g
    __device__ __forceinline__ long long state_group(long long g) const { return pol * n_groups + g; }
};

namespace ssd {
namespace policy {
// Packs num_policies trunk weight sets into a new handle (ssd_policy_create_n without its limit on num_policies).
int create_trunk(int view_radius, int device, int num_policies, WeightMap map, const float* conv_w, const float* conv_b, const float* fc1_w,
                 const float* fc1_b, const float* fc2_w, const float* fc2_b, SsdPolicy** out);

// Element (n, k) of a [rows x K] B operand in the canonical K-major layout without swizzle (8 x 16-byte core matrices).
inline int kmajor(int rows, int n, int k) { return ((k >> 3) * rows + n) * 8 + (k & 7); }

inline WeightMap weight_map(const SsdPolicy* p) {
    return p->kind == HandleKind::Pool ? WeightMap::Pool : p->num_policies == 1 ? WeightMap::Shared : WeightMap::PerAgent;
}

// SSD_OK when p is of kind `want`; else SSD_ERR_INVALID with `msg`, or for a network entry point given an MOA handle `moa_msg`.
inline int check_kind(const SsdPolicy* p, HandleKind want, const char* msg, const char* moa_msg = "an MOA handle takes ssd_moa_step") {
    if (p->kind == want) return SSD_OK;
    return ssd::set_error(SSD_ERR_INVALID, want == HandleKind::Net && p->kind == HandleKind::Moa ? moa_msg : msg);
}

inline int check_aligned(std::initializer_list<const void*> ptrs, const char* msg) {
    for (const void* q : ptrs)
        if (reinterpret_cast<uintptr_t>(q) % 16 != 0) return ssd::set_error(SSD_ERR_INVALID, msg);
    return SSD_OK;
}

// After a launch: SSD_OK, or SSD_ERR_CUDA with the launch error.
inline int launched() {
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? SSD_OK : ssd::set_error(SSD_ERR_CUDA, cudaGetErrorString(e));
}
}  // namespace policy

namespace policy_head {
// Packs the head weight sets of a handle (ssd_policy_set_head_n without its limit on num_policies).
int set_head(SsdPolicy* p, int units, int num_outputs, const float* lstm_w, const float* lstm_u, const float* lstm_b, const float* logits_w,
             const float* logits_b, const float* value_w, const float* value_b);
}  // namespace policy_head

namespace policy_pool {
constexpr int kBins = 256;                                                        // u8 ids
constexpr int kOffCursor = kBins, kOffNumTiles = 2 * kBins, kCountWords = 2 * kBins + 1;   // words of d_counts
// Bucket agents [0, M) by policy_ids (ids >= K skipped) into p->d_perm / p->d_tiles / num_tiles(p), all on `stream` with no
// host synchronisation.  Returns SSD_OK or an SSD_ERR_* code (message set).
int assign(SsdPolicy* p, const uint8_t* policy_ids, long long M, void* stream);
// tiles at most for M agents of K policies: every policy's last tile may be partial
inline long long max_tiles(long long M, int K) { return (M + 127) / 128 + K; }
// the tile count of the last assign, on the device (null for a handle that is not a pool)
inline const uint32_t* num_tiles(const SsdPolicy* p) { return p->d_counts ? p->d_counts + kOffNumTiles : nullptr; }
}  // namespace policy_pool

namespace policy {
// The persistent grid of a call on M agents: ctas CTAs, ctas_per_policy of them per weight set.  Shared: min(groups, #SMs);
// PerAgent: P * min(groups per set, #SMs / P); Pool: min(tiles, #SMs) over the tile table, whose length only the device knows.
struct Grid {
    int ctas, ctas_per_policy;
};
inline Grid grid(const SsdPolicy* p, long long M) {
    const int np = p->num_policies;
    if (p->kind == HandleKind::Pool) {
        const long long tiles = ssd::policy_pool::max_tiles(M, np);
        const int g = static_cast<int>(tiles < p->sms ? tiles : p->sms);
        return {g, g};
    }
    const long long groups = (M / np + 127) / 128;
    const int per = static_cast<int>(groups < p->sms / np ? groups : p->sms / np);
    return {np * per, per};
}

// Before a launch: makes the handle's device current (its weights and the caller's stream live there) and, for a pool call
// (policy_ids not null), groups the agents by policy on `stream`.
inline int setup(SsdPolicy* p, const uint8_t* policy_ids, long long M, void* stream) {
    if (policy_ids) return ssd::policy_pool::assign(p, policy_ids, M, stream);   // sets the device
    return cudaSetDevice(p->device) == cudaSuccess ? SSD_OK : ssd::set_error(SSD_ERR_CUDA, "cudaSetDevice failed");
}
}  // namespace policy
}  // namespace ssd
