// Host-side handle of the policy kernels (ssd_policy.cu: trunk; ssd_policy_head.cu: LSTM + heads).
#pragma once
#include <cstdint>

struct SsdPolicy {
    int device = 0;
    int sms = 0;
    uint8_t* d_blob = nullptr;       // packed trunk weights
    uint8_t* d_head_blob = nullptr;  // packed LSTM / head weights (ssd_policy_set_head)
    int units = 0, num_outputs = 0;
    int num_policies = 1;            // weight sets: agent m = b * P + p uses set p (ssd_policy_create_n)
};
