// Host-side handle of the policy kernels (ssd_policy.cu: trunk; ssd_policy_head.cu: LSTM + heads; ssd_policy_pool.cu: the
// assignment of agents to the weight sets of a policy pool).
#pragma once
#include <cstdint>

// How the policy kernels map agents to weight sets: one set for all agents, set m % P for agent m (one network per agent id),
// or set policy_ids[m] for agent m (a policy pool; agents grouped by ssd::policy_pool::assign).
enum class WeightMap { Shared, PerAgent, Pool };

// One tile of a pool's assignment: agents perm[first, first + count), count <= 128, all evaluated with weight set `policy`.
struct PoolTile {
    uint32_t first;
    uint16_t policy, count;
};

struct SsdPolicy {
    int device = 0;
    int sms = 0;
    uint8_t* d_blob = nullptr;       // packed trunk weights
    uint8_t* d_head_blob = nullptr;  // packed LSTM / head weights (ssd_policy_set_head)
    int units = 0, num_outputs = 0;
    int num_policies = 1;            // weight sets: agent m = b * P + p uses set p (ssd_policy_create_n), or set ids[m] (pool)
    bool pool = false;               // made by ssd_policy_create_pool
    // made by ssd_moa_create: d_head_blob holds the MOA's resident weights, d_moa_rows its one-hot rows and moa_logits_w,
    // num_outputs its A, moa_agents its N
    bool moa = false;
    int moa_agents = 0;
    float* d_moa_rows = nullptr;
    // pool scratch, grown on demand: per-policy counts [256] and cursors [256], the tile count, perm [M], tiles [M / 128 + K]
    uint32_t* d_counts = nullptr;
    uint32_t* d_perm = nullptr;
    PoolTile* d_tiles = nullptr;
    long long perm_cap = 0, tile_cap = 0;
};

namespace ssd {
namespace policy {
// Packs num_policies trunk weight sets into a new handle (ssd_policy_create_n without its limit on num_policies).
int create_trunk(int view_radius, int device, int num_policies, WeightMap map, const float* conv_w, const float* conv_b, const float* fc1_w,
                 const float* fc1_b, const float* fc2_w, const float* fc2_b, SsdPolicy** out);
}  // namespace policy
namespace policy_head {
// Packs the head weight sets of a handle (ssd_policy_set_head_n without its limit on num_policies).
int set_head(SsdPolicy* p, int units, int num_outputs, const float* lstm_w, const float* lstm_u, const float* lstm_b, const float* logits_w,
             const float* logits_b, const float* value_w, const float* value_b);
}  // namespace policy_head
namespace policy_pool {
// Bucket agents [0, M) by policy_ids (ids >= K skipped) into p->d_perm / p->d_tiles / the tile count at p->d_counts + 512,
// all on `stream` with no host synchronisation.  Returns SSD_OK or an SSD_ERR_* code (message set).
int assign(SsdPolicy* p, const uint8_t* policy_ids, long long M, void* stream);
// tiles at most for M agents of K policies: every policy's last tile may be partial
inline long long max_tiles(long long M, int K) { return (M + 127) / 128 + K; }
}  // namespace policy_pool
}  // namespace ssd
