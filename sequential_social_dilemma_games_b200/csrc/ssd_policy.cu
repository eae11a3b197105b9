// Policy-side consumer of the observation tensor (SURVEY.md 8f-4): the feature trunk of the reference's policy network,
// models/conv_to_fcnet_v2.py:36-66 -- Conv2D(6, 3x3, stride 1, 'valid') -> ReLU -> flatten -> Dense(32) -> ReLU -> Dense(32) -> ReLU --
// reading the uint8 observations the step kernel left in HBM (the (x - 128) / 255 of map_env.py:199 is folded into the first
// layer).  One fused kernel on the 5th-generation tensor cores: nothing but the [M, 32] features goes back to HBM.
//
//   per group of 128 agents (= UMMA M: one tensor-memory lane per agent; one persistent CTA per SM):
//     for each of the 15 image rows r:   A_r[agent][k] = fp16(1024 + obs[agent][45 r + k]), k < 48  (0x6400 | byte IS that fp16; taps
//                                         45..47 belong to the next row and meet zero weights) -- converted once, kept in a ring
//     for each of the 13 output rows i of the convolution (image rows i..i+2 are the three operand blocks i, i+1, i+2):
//       D1[128 x 80]  = sum_di A_(i+di)[128 x 48] * B1_di[48 x 80]   banded weights: column (j, f) holds filter f at taps 3 (j + dj) + c
//       C [agent][n]  = fp16(relu(D1 / 255 + cb[n]))                cb folds the bias, the -128 / 255 and the 1024 offset
//       D2[128 x 32] += C[128 x 80] * W1_i[80 x 32]                 Dense(32) accumulated over the 13 row blocks of its 1014 inputs
//     D3[128 x 32] = fp16(relu(D2 + b1)) * W2;  features = relu(D3 + b2)
//
// The A operands (image-row ring, C, the fc2 operand) and the accumulators live in tensor memory -- the lane that owns an agent
// writes them with tcgen05.st -- the B operands (weights) in shared memory in the canonical K-major no-swizzle layout (8 x 16-byte
// core matrices: element (n, k) at (k / 8) * rows * 16 + n * 16 + (k % 8) * 2); all MMAs are issued by one elected thread.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <cstdio>
#include <cstring>
#include <new>
#include <vector>

#include "ssd_internal.h"
#include "ssd_policy.h"
#include "ssd_umma.cuh"

#ifdef SSD_POLICY_TIMING  // profiles/micro/policy_timing.cu: cycles per phase of one thread per role of CTA 0
__device__ unsigned long long g_policy_cycles[3][8];
#define SSD_PT_DECL unsigned long long pt_[8] = {0, 0, 0, 0, 0, 0, 0, 0}; long long pt_t = clock64()
#define SSD_PT(slot) do { const long long n_ = clock64(); pt_[slot] += n_ - pt_t; pt_t = n_; } while (0)
#define SSD_PT_FLUSH(role) do { if (blockIdx.x == 0) for (int q_ = 0; q_ < 8; ++q_) g_policy_cycles[role][q_] = pt_[q_]; } while (0)
__device__ long long g_policy_tl[3][32][4];   // [role][step - 40][event] clock64 stamps of CTA 0
#define SSD_TL(role, idx, ev) do { if (blockIdx.x == 0 && (idx) >= 40 && (idx) < 72) g_policy_tl[role][(idx) - 40][ev] = clock64(); } while (0)
#else
#define SSD_TL(role, idx, ev)
#define SSD_PT_DECL
#define SSD_PT(slot)
#define SSD_PT_FLUSH(role)
#endif

namespace ssd {
namespace policy {
using namespace ssd::umma;

constexpr int V = 15, IMG = V * V * 3, ROWB = V * 3, CO = V - 2, NF = 6, FEAT = 32;
constexpr int GA = 128;                       // agents per group = UMMA M
constexpr int ROWK = 48;                      // one image row: 45 taps padded to 3 k-steps
constexpr int N1 = 80;                        // 13 * 6 = 78 conv outputs of one output row, padded
constexpr int K2 = 80, N2 = FEAT;             // one row block of Dense(32)
constexpr int K3 = FEAT, N3 = FEAT;
constexpr int RING = 6;                       // image-row operand blocks in flight (tensor memory)
constexpr int kProducerWarps = 4, kMmaWarp = 4, kDrainWarp0 = 5, kDrainWarps = 8, kLoadWarp = kDrainWarp0 + kDrainWarps, kThreads = 32 * (kLoadWarp + 1);
// tensor memory (512 columns x 128 lanes x 32 bit): accumulators, and the A operands -- a lane is an agent, a column two fp16
constexpr int kTmemCols = 512;
constexpr int kColD1a = 0, kColD1b = 144;     // conv accumulators of even / odd output rows (80 columns)
constexpr int kColD2a = 80, kColD2b = 112;    // Dense(32) accumulators of even / odd groups
constexpr int kColD3 = 224;                   // fc2 accumulator
constexpr int kColX3 = 256;                   // fc2 operand, 16 columns
constexpr int kColC = 272;                    // + 40 * buffer: relu(conv) of one output row, 40 columns
constexpr int kColRing = 352;                 // + 24 * slot: one image row, 24 columns
constexpr int kDrainSplit = 48;               // conv columns [0, 48) drain on warps 5-8, [48, 80) on warps 9-12

// shared-memory carve-up (bytes): two groups of observation bytes and the B operands
constexpr int kB1Bytes = (3 * ROWK / 8) * N1 * 16;        // 23 040
constexpr int kB2Bytes = (K2 / 8) * N2 * 16;              // 5 120 per row block of Dense(32)
constexpr int kB3Bytes = (K3 / 8) * N3 * 16;              // 2 048
constexpr int kConstFloats = N1 + N2 + N3;                // cb[80], b1[32], b2[32]
constexpr int kHeadBytes = kB1Bytes + kB3Bytes + kConstFloats * 4;   // resident part of the blob: 25 664
constexpr int kBlobBytes = kHeadBytes + CO * kB2Bytes;    // + the 13 row blocks of Dense(32), streamed: 92 224
constexpr int kObsSlot = 704;                             // per-agent variant: one agent's 16-byte-aligned span (<= 690 bytes) + reads past it
enum { BAR_OBS = 0, BAR_OBS_FREE = 2, BAR_ROW_FULL = 4, BAR_D1_FREE = 10, BAR_C_FULL = 12, BAR_W1_FULL = 14, BAR_X3 = 20, BAR_D3 = 21, BAR_STEP = 22,
       BAR_COUNT = 30 };
constexpr int STEPS = 8;                      // ring of "first block of MMA step s has completed" barriers
// Shared-memory layout of the two variants of the kernel.  Shared weights: a group is 128 consecutive agents, one contiguous
// run of 86 400 bytes.  Per-agent weights: a group is 128 agents of one policy, rows P * 675 bytes apart, each gathered into
// a 704-byte slot; the two observation buffers grow by 7 168 bytes, which the weight ring pays for with one block (6 -> 5:
// 5 KB; the blocks come from L2 and the ring still runs five output rows ahead of their use).
template <bool kPerAgent>
struct TrunkSmem {
    static constexpr int WRING = kPerAgent ? 5 : 6;         // Dense weight blocks in flight (shared memory)
    static constexpr int kSlot = kPerAgent ? kObsSlot : IMG; // bytes from one agent's observation to the next
    static constexpr int kObsStride = kPerAgent ? GA * kObsSlot : 86528;  // 128 * 675 = 86 400 + slack for the padded taps of the last agent
    static constexpr int kOffObs = 0;
    static constexpr int kOffB1 = 2 * kObsStride, kOffB3 = kOffB1 + kB1Bytes, kOffConst = kOffB3 + kB3Bytes;
    static constexpr int kOffW1 = kOffB1 + kHeadBytes;
    static constexpr int kOffBar = kOffW1 + WRING * kB2Bytes;
    static constexpr int kSmemBytes = kOffBar + BAR_COUNT * 8;
    static_assert(kHeadBytes % 16 == 0 && kOffB1 % 128 == 0 && kOffW1 % 16 == 0 && kOffBar % 8 == 0, "alignment");
    static_assert(kSmemBytes <= 227 * 1024, "one CTA per SM");
    static_assert(BAR_W1_FULL + WRING <= BAR_X3, "weight-ring barriers");
};

// The CTA works through its groups g = blockIdx.x, blockIdx.x + gridDim.x, ... as ONE sequence of output rows
// T = 13 * (group ordinal) + i and image rows R = 15 * (group ordinal) + r; three roles run that sequence concurrently:
//   producers (warps 0-3, thread = agent = TMEM lane): image row R -> fp16(1024 + byte) in ring block R % 6 of tensor
//       memory;
//   loader thread (warp 13): TMA bulk copies -- two groups of observation bytes in flight, the Dense(32) weight blocks
//       through a 6-deep ring in shared memory;
//   MMA thread (warp 4): step s issues the last six MMAs of conv(s) interleaved with the five of the Dense partial of
//       row s - 2, then -- once the drain warps have read the accumulator of row s - 1 -- the first three of conv(s + 1)
//       into it, so the tensor pipe always has queued work while an accumulator is drained; fc2 of a group four steps
//       after its last row;
//   drain warps (5-12, thread = accumulator lane = agent, two warps per lane quarter splitting the columns):
//       D1[T % 2] -> relu -> fp16 -> C[T % 2] (tensor memory again: the A operand of the Dense partial); two rows into
//       the next group D2 -> fc2 operand, four rows in D3 -> features in HBM.
// Hand-offs: mbarriers.  "Full" barriers (image row published, C written, weight block landed, ...) are waited on parity
// n & 1 at their n-th use.  Everything the MMAs release -- accumulator full, image-row block / C buffer / weight block free,
// D2 complete -- hangs on ONE tcgen05.commit per step into a ring of eight step barriers (a commit costs the issuing
// thread ~40 cycles, five per step were 15 % of the kernel): whoever needs "the first block of step x is complete" waits
// barrier x % 8 on parity (x / 8) & 1; no waiter is ever more than six steps from the MMA thread, so phases cannot alias.
//
// kPerAgent: agent m = b * P + p of the [B, P] batch is evaluated with weight set p (blob + p * kBlobBytes); the CTAs take the
// groups of GroupMap (ssd_policy.h) and load their policy's resident weights once, as the shared kernel does.
//
// WeightMap::Pool: a group is one tile of the assignment (ssd_policy_pool.cu): agents perm[first, first + count) of one
// policy, gathered and written back as the per-agent variant does, at rows perm[i].  CTA c takes tiles
// [c T / G, (c + 1) T / G) and runs them as segments of consecutive tiles of one policy.  Each segment is the pipeline above
// from a clean start: at a switch of policy every role has finished the previous segment (its last fc2 committed, its
// features written), the CTA synchronises, re-initialises the barriers and loads the new policy's resident block.  The
// Dense(32) blocks stream from the segment's blob.  Tiles are in policy order, so a CTA switches at most once per policy
// boundary inside its range.
template <WeightMap kMap>
__global__ void __launch_bounds__(kThreads, 1) policy_features_kernel(const uint8_t* __restrict__ obs, long long M, const uint8_t* __restrict__ blob,
                                                                     float* __restrict__ out, int num_policies, int ctas_per_policy,
                                                                     const uint32_t* __restrict__ perm, const PoolTile* __restrict__ tiles,
                                                                     const uint32_t* __restrict__ num_tiles) {
    constexpr bool kPerAgent = kMap != WeightMap::Shared, kPool = kMap == WeightMap::Pool;
    using L = TrunkSmem<kPerAgent>;
    constexpr int WRING = L::WRING, kObsStride = L::kObsStride, kOffObs = L::kOffObs, kOffB1 = L::kOffB1, kOffB3 = L::kOffB3;
    constexpr int kOffConst = L::kOffConst, kOffW1 = L::kOffW1, kOffBar = L::kOffBar;
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ uint32_t s_tmem;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kOffBar);
    const float* s_const = reinterpret_cast<const float*>(smem + kOffConst);
    const GroupMap<kMap> gm(M, num_policies, ctas_per_policy);
    const long long cta = gm.cta, stride = gm.stride, rows = gm.rows, n_groups = gm.n_groups;
    const uint8_t* const blob0 = blob;
    if (kPerAgent && !kPool) blob += static_cast<long long>(gm.pol) * kBlobBytes;
    long long seg_end = 0, tile_end = 0;   // pool: the CTA's tiles not yet run are [seg_end, tile_end)
    if (kPool) {
        const long long nt = *num_tiles;
        seg_end = nt * blockIdx.x / gridDim.x;
        tile_end = nt * (blockIdx.x + 1) / gridDim.x;
    }
    int seg = 0;
    uint32_t tmem_base = 0;
    do {   // pool: one pass per segment; otherwise one pass
    long long tb = seg_end;   // pool: the segment's first tile = group 0
    if (kPool && seg_end < tile_end) {
        tb = seg_end;
        const int k = tiles[tb].policy;
        while (++seg_end < tile_end && tiles[seg_end].policy == k) {
        }
        blob = blob0 + static_cast<long long>(k) * kBlobBytes;
    }
    const uint32_t n_my = kPool ? static_cast<uint32_t>(seg_end - tb)
                                : cta < n_groups ? static_cast<uint32_t>((n_groups - cta + stride - 1) / stride) : 0;  // groups of this CTA
    const uint32_t NT = n_my * CO;

    if (kPool && seg > 0) {   // every role is done with the previous segment: its barriers can start over
        tc_fence_after();
        if (tid == 0)
            for (int b = 0; b < BAR_COUNT; ++b) asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(smem_u32(bars + b)) : "memory");
    }
    if (tid == 0) {
        for (int b = 0; b < BAR_COUNT; ++b) {
            const int count = (b >= BAR_OBS_FREE && b < BAR_D1_FREE) ? kProducerWarps      // one arrival per producer warp
                              : ((b >= BAR_D1_FREE && b < BAR_W1_FULL) || b == BAR_X3) ? kDrainWarps : 1;  // per drain warp; else TMA / commit
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bars + b)), "r"(count) : "memory");
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (seg == 0 && warp == kMmaWarp) {  // all of the SM's tensor memory (one CTA per SM)
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s_tmem)), "r"(kTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    for (int i = tid; i < kHeadBytes / 16; i += kThreads)  // conv and fc2 weights, constants: once per CTA (the grid is persistent)
        reinterpret_cast<uint4*>(smem + kOffB1)[i] = reinterpret_cast<const uint4*>(blob)[i];
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = s_tmem;
    tmem_base = tmem;

    if (warp < kProducerWarps) {
        // ------------------------------------------------------------------ producers
        const int t = tid;
        const uint32_t tlane = tmem + (static_cast<uint32_t>(warp * 32) << 16);
        uint32_t R = 0;
        SSD_PT_DECL;
        // The stores of a row into tensor memory complete while the next row is assembled in registers: a row is published
        // (wait::st, fence, arrive) one iteration after its stores were issued.
        auto publish = [&](uint32_t Rp) {
            tmem_st_wait();
            SSD_PT(6);
            tc_fence_before();
            __syncwarp();
            SSD_PT(7);
            if (lane == 0) mbar_arrive(bars + BAR_ROW_FULL + Rp % RING);
        };
        for (uint32_t gi = 0; gi < n_my; ++gi) {
            warp_wait(bars + BAR_OBS + (gi & 1), (gi >> 1) & 1);
            SSD_PT(0);
            const uint8_t* img = smem + kOffObs + (gi & 1) * kObsStride + t * L::kSlot;
            if (kPool) {
                const PoolTile tile = tiles[tb + gi];
                img += t < tile.count ? (perm[tile.first + t] * static_cast<uint32_t>(IMG)) & 15u : 0u;
            } else if (kPerAgent)  // the slot starts at the 16-byte boundary below the agent's row (obs is 16-byte aligned)
                img += (static_cast<uint32_t>(gm.agent((cta + gi * stride) * GA, t)) * IMG) & 15u;
#pragma unroll 1
            for (int r = 0; r < V; ++r, ++R) {
                const uint32_t slot = R % RING;
                uint32_t h[ROWK / 2];
                {   // fp16(1024 + byte) of this agent's 48-byte window: 0x6400 | byte
                    const uint32_t base = smem_u32(img + r * ROWB);
                    const uint32_t sh = (base & 3u) * 8;
                    uint32_t x[ROWK / 4 + 1];
#pragma unroll
                    for (int q = 0; q <= ROWK / 4; ++q) asm volatile("ld.shared.u32 %0, [%1];" : "=r"(x[q]) : "r"((base & ~3u) + 4 * q));
#pragma unroll
                    for (int q = 0; q < ROWK / 4; ++q) {
                        const uint32_t b4 = __funnelshift_r(x[q], x[q + 1], sh);
                        h[2 * q] = __byte_perm(b4, 0x64646464u, 0x4140);
                        h[2 * q + 1] = __byte_perm(b4, 0x64646464u, 0x4342);
                    }
                }
                SSD_PT(2);
                if (t == 0) SSD_TL(0, R, 0);
                if (R > 0) publish(R - 1);
                SSD_PT(3);
                if (t == 0) SSD_TL(0, R, 3);
                if (R >= RING) {  // the block's previous image row: last read by conv of its own output row (rows 13, 14: of row 12)
                    const uint32_t Rq = R - RING, iq = Rq % V, xs = (Rq / V) * CO + (iq < CO ? iq : CO - 1);
                    warp_wait(bars + BAR_STEP + xs % STEPS, (xs / STEPS) & 1);
                }
                SSD_PT(1);
                if (t == 0) SSD_TL(0, R, 1);
                tc_fence_after();
#pragma unroll
                for (int c = 0; c < ROWK / 2; c += 8) tmem_st8(tlane + kColRing + slot * (ROWK / 2) + c, h + c);
                SSD_PT(5);
                if (t == 0) SSD_TL(0, R, 2);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(bars + BAR_OBS_FREE + (gi & 1));  // this warp is done with the buffer of observation bytes
            SSD_PT(4);
        }
        if (R > 0) publish(R - 1);
        if (t == 0) SSD_PT_FLUSH(0);
    } else if (warp == kMmaWarp) {
        // ------------------------------------------------------------------ MMA issue (one elected thread)
        // Everything an MMA needs is a 32-bit add away: descriptors are (lo, hi) pairs whose lo word advances by a constant
        // per k-step, tensor-memory operands are base + 24 * ring slot + 8 * k-step.  elect.sync (not `lane == 0`) tells ptxas
        // the block runs on one lane, so the UTCHMMAs are issued without a per-instruction convergence loop.
        if (NT > 0 && elect_one()) {
            constexpr uint32_t kI1 = umma_idesc(GA, N1), kI2 = umma_idesc(GA, N2), kI3 = umma_idesc(GA, N3);
            constexpr uint32_t kDescHi = (128u >> 4) | 1u << 14;   // SBO = 128 bytes, descriptor version 1
            auto desc_lo = [](uint32_t saddr, uint32_t lbo) { return ((saddr & 0x3FFFFu) >> 4) | (lbo >> 4) << 16; };
            auto mk = [](uint32_t lo) { return static_cast<uint64_t>(kDescHi) << 32 | lo; };
            const uint32_t b1_lo = desc_lo(smem_u32(smem + kOffB1), N1 * 16);   // + (2 * N1 * 16 >> 4) per k-step
            const uint32_t w1_lo = desc_lo(smem_u32(smem + kOffW1), N2 * 16);   // + (kB2Bytes >> 4) per buffer, + (2 * N2 * 16 >> 4) per k-step
            const uint32_t b3_lo = desc_lo(smem_u32(smem + kOffB3), N3 * 16);
            constexpr uint32_t kB1Step = 2 * N1 * 16 >> 4, kW1Step = 2 * N2 * 16 >> 4, kW1Buf = kB2Bytes >> 4, kB3Step = 2 * N3 * 16 >> 4;
            const uint32_t ring = tmem + kColRing;
            uint32_t rows_seen = 0;
            SSD_PT_DECL;
            auto wait_rows = [&](uint32_t need) {  // image rows [0, need) of the CTA's sequence
                while (rows_seen < need) {
                    wait_sleep(bars + BAR_ROW_FULL + rows_seen % RING, (rows_seen / RING) & 1);
                    ++rows_seen;
                }
            };
            auto fc2 = [&](uint32_t gi) {
                wait_sleep(bars + BAR_X3, gi & 1);
                tc_fence_after();
#pragma unroll
                for (int ks = 0; ks < K3 / 16; ++ks) umma_f16_ts(tmem + kColD3, tmem + kColX3 + ks * 8, mk(b3_lo + ks * kB3Step), kI3, ks > 0);
                umma_commit(bars + BAR_D3);
            };
            // state of output row s (e), s + 1 (o) and s - 2 (d): index in its group, ring slot of its first image row, group parity
            uint32_t i_e = 0, slot_e = 0, row_e = 0, g_e = 0;   // row_e = first image row of conv(s) in the CTA's sequence
            uint32_t i_d1 = 0, g_d1 = 0, i_d = 0, g_d = 0;      // rows s - 1 and s - 2
            wait_rows(1);
            tc_fence_after();
#pragma unroll
            for (int k = 0; k < 3; ++k) umma_f16_ts(tmem + kColD1a, ring + k * 8, mk(b1_lo + k * kB1Step), kI1, k != 0);
#pragma unroll 1
            for (uint32_t s = 0; s < NT + 2; ++s) {
                const bool has_e = s < NT, has_o = s + 1 < NT, has_d = s >= 2;
                const bool last_e = i_e == CO - 1;
                const uint32_t slot_o = (slot_e + (last_e ? 3 : 1)) % RING, row_o = row_e + (last_e ? 3 : 1);
                // ---- first block: the six remaining MMAs of conv(s) (image rows i + 1, i + 2) interleaved with the Dense partial of
                // row s - 2.  Nothing here needs the accumulator the drain warps are reading.
                if (has_e) wait_rows(row_e + 3);
                SSD_PT(0);
                if (has_d) {
                    wait_sleep(bars + BAR_C_FULL + (s & 1), ((s - 2) >> 1) & 1);
                    wait_sleep(bars + BAR_W1_FULL + (s - 2) % WRING, ((s - 2) / WRING) & 1);
                }
                SSD_PT(3);
                SSD_TL(1, s, 0);
                tc_fence_after();
                {
                    const uint32_t d_e = tmem + ((s & 1) ? kColD1b : kColD1a);
                    const uint32_t a_e1 = ring + ((slot_e + 1) % RING) * (ROWK / 2), a_e2 = ring + ((slot_e + 2) % RING) * (ROWK / 2);
                    const uint32_t d_d = tmem + (g_d ? kColD2b : kColD2a), a_d = tmem + kColC + (s & 1) * (K2 / 2);
                    const uint32_t w_d = w1_lo + ((s - 2) % WRING) * kW1Buf;
                    const uint32_t acc_d = i_d != 0;
                    if (has_e) umma_f16_ts(d_e, a_e1, mk(b1_lo + 3 * kB1Step), kI1, 1);
                    if (has_d) umma_f16_ts(d_d, a_d, mk(w_d), kI2, acc_d);
                    if (has_e) umma_f16_ts(d_e, a_e1 + 8, mk(b1_lo + 4 * kB1Step), kI1, 1);
                    if (has_d) umma_f16_ts(d_d, a_d + 8, mk(w_d + kW1Step), kI2, 1);
                    if (has_e) umma_f16_ts(d_e, a_e1 + 16, mk(b1_lo + 5 * kB1Step), kI1, 1);
                    if (has_d) umma_f16_ts(d_d, a_d + 16, mk(w_d + 2 * kW1Step), kI2, 1);
                    if (has_e) umma_f16_ts(d_e, a_e2, mk(b1_lo + 6 * kB1Step), kI1, 1);
                    if (has_d) umma_f16_ts(d_d, a_d + 24, mk(w_d + 3 * kW1Step), kI2, 1);
                    if (has_e) umma_f16_ts(d_e, a_e2 + 8, mk(b1_lo + 7 * kB1Step), kI1, 1);
                    if (has_d) umma_f16_ts(d_d, a_d + 32, mk(w_d + 4 * kW1Step), kI2, 1);
                    if (has_e) umma_f16_ts(d_e, a_e2 + 16, mk(b1_lo + 8 * kB1Step), kI1, 1);
                }
                // ONE commit per step: conv(s) is complete (accumulator full, image row i -- and at the end of a group rows
                // 13, 14 -- free) and so is the Dense partial of row s - 2 (C buffer and weight block free, D2 full after row 12)
                umma_commit(bars + BAR_STEP + s % STEPS);
                SSD_TL(1, s, 1);
                SSD_PT(2);
                if (s >= 4 && (s - 4) % CO == CO - 1) fc2((s - 4) / CO);  // the drain warps delivered its operand a step ago
                // ---- second block: the first image row of conv(s + 1), into the accumulator of row s - 1 once it is drained
                if (has_o) {
                    wait_rows(row_o + 1);
                    wait_sleep(bars + BAR_D1_FREE + ((s + 1) & 1), (((s + 1) >> 1) & 1) ^ 1);
                    SSD_PT(1);
                    SSD_TL(1, s, 2);
                    tc_fence_after();
                    const uint32_t d_o = tmem + ((s & 1) ? kColD1a : kColD1b), a_o0 = ring + slot_o * (ROWK / 2);
                    umma_f16_ts(d_o, a_o0, mk(b1_lo), kI1, 0);
                    umma_f16_ts(d_o, a_o0 + 8, mk(b1_lo + kB1Step), kI1, 1);
                    umma_f16_ts(d_o, a_o0 + 16, mk(b1_lo + 2 * kB1Step), kI1, 1);
                    SSD_TL(1, s, 3);
                }
                // shift the window of rows
                i_d = i_d1; g_d = g_d1; i_d1 = i_e; g_d1 = g_e;
                if (last_e) { i_e = 0; g_e ^= 1; } else { ++i_e; }
                slot_e = slot_o; row_e = row_o;
                SSD_PT(4);
            }
            fc2(n_my - 1);  // the last group's fc2 step lies beyond the sequence
            SSD_PT(6);
            SSD_PT_FLUSH(1);
        }
    } else if (warp == kLoadWarp) {
        // ------------------------------------------------------------------ loader: TMA bulk copies only.  Shared weights: one
        // elected thread.  Per-agent weights: the whole warp -- a group is 128 copies, which one thread issued too slowly to keep
        // the weight ring fed -- with lane 0 polling the barriers for the warp and issuing the weight blocks.
        if (n_my > 0 && (kPerAgent || elect_one())) {
            const bool lead = !kPerAgent || lane == 0;
            auto ready = [&](uint64_t* b, uint32_t parity) {  // per-agent: lane 0's view, the same for the whole warp
                if (!kPerAgent) return mbar_try_wait(b, parity);
                return __shfl_sync(0xffffffffu, lane == 0 ? static_cast<int>(mbar_try_wait(b, parity)) : 0, 0) != 0;
            };
            auto load_obs = [&](uint32_t gi) {
                const long long a0 = (cta + static_cast<long long>(gi) * stride) * GA;
                const PoolTile tile = kPool ? tiles[tb + gi] : PoolTile{};
                const int rem = kPool ? tile.count : static_cast<int>(rows - a0 < GA ? rows - a0 : GA);
                uint8_t* dst = smem + kOffObs + (gi & 1) * kObsStride;
                uint64_t* bar = bars + BAR_OBS + (gi & 1);
                if (!kPerAgent) {  // the group's rem * 675 contiguous bytes (a group starts 16-byte aligned)
                    const uint8_t* src = obs + a0 * IMG;
                    const uint32_t bytes = static_cast<uint32_t>(rem) * IMG, b16 = bytes & ~15u;
                    for (uint32_t i = b16; i < bytes; ++i) dst[i] = src[i];
                    mbar_expect_tx(bar, b16);
                    bulk_g2s(dst, src, b16, bar);
                } else {  // gather: per agent the 16-byte-aligned span around its row, into its slot; nothing past the tensor's end
                    const long long end = M * IMG, end16 = end & ~15ll;
                    auto span = [&](int t, long long& s0) {
                        const long long s = (kPool ? static_cast<long long>(perm[tile.first + t]) : gm.agent(a0, t)) * IMG, s1 = (s + IMG + 15) & ~15ll;
                        s0 = s & ~15ll;
                        return static_cast<uint32_t>((s1 < end16 ? s1 : end16) - s0);
                    };
                    uint32_t bytes = 0;
                    for (int t = lane; t < rem; t += 32) {
                        long long s0;
                        bytes += span(t, s0);
                        if (s0 + span(t, s0) == end16)  // the last agent of the tensor: its bytes past the last 16-byte boundary by hand
                            for (long long i = end16; i < end; ++i) dst[t * L::kSlot + (i - s0)] = obs[i];
                    }
                    bytes = __reduce_add_sync(0xffffffffu, bytes);
                    __syncwarp();
                    if (lane == 0) mbar_expect_tx(bar, bytes);  // before any copy can complete; releases the tail bytes
                    __syncwarp();
                    for (int t = lane; t < rem; t += 32) {
                        long long s0;
                        const uint32_t n = span(t, s0);
                        bulk_g2s(dst + t * L::kSlot, obs + s0, n, bar);
                    }
                }
            };
            load_obs(0);
            if (n_my > 1) load_obs(1);
            uint32_t next_obs = 2;  // next group whose bytes want a buffer: group next_obs - 2 must have been consumed
#pragma unroll 1
            for (uint32_t T = 0; T < NT; ++T) {  // Dense(32) weight block of output row T, WRING rows ahead of its use
                const uint32_t ws = T % WRING, tf = T - WRING + 2;  // step tf issued the Dense partial of row T - WRING
                while (T >= WRING && !ready(bars + BAR_STEP + tf % STEPS, (tf / STEPS) & 1)) {
                    if (next_obs < n_my && ready(bars + BAR_OBS_FREE + (next_obs & 1), ((next_obs - 2) >> 1) & 1)) load_obs(next_obs++);
                    __nanosleep(200);
                }
                if (lead) {
                    mbar_expect_tx(bars + BAR_W1_FULL + ws, kB2Bytes);
                    bulk_g2s(smem + kOffW1 + ws * kB2Bytes, blob + kHeadBytes + (T % CO) * kB2Bytes, kB2Bytes, bars + BAR_W1_FULL + ws);
                }
                if (next_obs < n_my && ready(bars + BAR_OBS_FREE + (next_obs & 1), ((next_obs - 2) >> 1) & 1)) load_obs(next_obs++);
            }
            while (next_obs < n_my) {
                if (kPerAgent) {
                    while (!ready(bars + BAR_OBS_FREE + (next_obs & 1), ((next_obs - 2) >> 1) & 1)) {
                    }
                } else {
                    wait_sleep(bars + BAR_OBS_FREE + (next_obs & 1), ((next_obs - 2) >> 1) & 1);
                }
                load_obs(next_obs++);
            }
        }
    } else {
        // ------------------------------------------------------------------ drain warps: thread = accumulator lane = agent
        const int q = warp & 3, row = q * 32 + lane, half = (warp - kDrainWarp0) >> 2;
        const uint32_t trow = tmem + (static_cast<uint32_t>(q * 32) << 16);
        const int col0 = half ? kDrainSplit : 0;   // this warp's conv columns [col0, col0 + ncol)
        float cb[kDrainSplit];  // bias, -128 / 255 and the 1024 offset of the operand, per conv column
#pragma unroll
        for (int c = 0; c < kDrainSplit; ++c) cb[c] = (col0 + c < N1) ? s_const[col0 + c] : 0.f;
        SSD_PT_DECL;
        auto tail1 = [&](uint32_t gi) {  // this warp's 16 columns of the fc2 operand = fp16(relu(D2 + b1))
            const uint32_t xs = gi * CO + CO + 1;  // the step that issued the Dense partial of the group's last row
            warp_wait(bars + BAR_STEP + xs % STEPS, (xs / STEPS) & 1);
            tc_fence_after();
            uint32_t acc[16], h[8];
            tmem_ld16(trow + ((gi & 1) ? kColD2b : kColD2a) + 16 * half, acc);
            tmem_ld_wait();
#pragma unroll
            for (int c = 0; c < 16; c += 2)
                h[c / 2] = pack_relu_h2(__uint_as_float(acc[c]) + s_const[N1 + 16 * half + c], __uint_as_float(acc[c + 1]) + s_const[N1 + 16 * half + c + 1]);
            tmem_st8(trow + kColX3 + 8 * half, h);
            tmem_st_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bars + BAR_X3);
        };
        auto tail2 = [&](uint32_t gi) {  // this warp's 16 features = relu(D3 + b2): 64 of the agent's 128 bytes
            warp_wait(bars + BAR_D3, gi & 1);
            tc_fence_after();
            uint32_t acc[16];
            tmem_ld16(trow + kColD3 + 16 * half, acc);
            tmem_ld_wait();
            tc_fence_before();
            const long long a0 = (cta + static_cast<long long>(gi) * stride) * GA;
            const PoolTile tile = kPool ? tiles[tb + gi] : PoolTile{};
            if (kPool ? row < tile.count : a0 + row < rows) {
                float4* dst = reinterpret_cast<float4*>(out + (kPool ? static_cast<long long>(perm[tile.first + row]) : gm.agent(a0, row)) * FEAT + 16 * half);
                const float* b2 = s_const + N1 + N2 + 16 * half;
#pragma unroll
                for (int c = 0; c < 16; c += 4)
                    dst[c / 4] = make_float4(fmaxf(__uint_as_float(acc[c]) + b2[c], 0.f), fmaxf(__uint_as_float(acc[c + 1]) + b2[c + 1], 0.f),
                                             fmaxf(__uint_as_float(acc[c + 2]) + b2[c + 2], 0.f), fmaxf(__uint_as_float(acc[c + 3]) + b2[c + 3], 0.f));
            }
        };
#pragma unroll 1
        for (uint32_t T = 0; T < NT; ++T) {
            const uint32_t b = T & 1;
            warp_wait(bars + BAR_STEP + T % STEPS, (T / STEPS) & 1);   // conv(T) complete; so is the Dense partial that read C[b]
            SSD_PT(0);
            if (tid == 32 * kDrainWarp0) SSD_TL(2, T, 0);
            tc_fence_after();
            uint32_t acc[kDrainSplit];
            const uint32_t src = trow + (b ? kColD1b : kColD1a) + col0;
            tmem_ld16(src, acc);
            tmem_ld16(src + 16, acc + 16);
            if (half == 0) tmem_ld16(src + 32, acc + 32);
            tmem_ld_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bars + BAR_D1_FREE + b);
            SSD_PT(1);
            if (tid == 32 * kDrainWarp0) SSD_TL(2, T, 1);
            uint32_t h[kDrainSplit / 2];   // C = fp16(relu(D1 / 255 + cb))
#pragma unroll
            for (int c = 0; c < kDrainSplit; c += 2)
                if (half == 0 || c < N1 - kDrainSplit)
                    h[c / 2] = pack_relu_h2(fmaf(__uint_as_float(acc[c]), 1.0f / 255.0f, cb[c]), fmaf(__uint_as_float(acc[c + 1]), 1.0f / 255.0f, cb[c + 1]));
            SSD_PT(2);
            const uint32_t dstc = trow + kColC + b * (K2 / 2) + col0 / 2;
            tmem_st8(dstc, h);
            tmem_st8(dstc + 8, h + 8);
            if (half == 0) tmem_st8(dstc + 16, h + 16);
            tmem_st_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bars + BAR_C_FULL + b);
            SSD_PT(4);
            if (tid == 32 * kDrainWarp0) SSD_TL(2, T, 2);
            if (T >= 2 && (T - 2) % CO == CO - 1) tail1((T - 2) / CO);
            if (T >= 4 && (T - 4) % CO == CO - 1) tail2((T - 4) / CO);
            SSD_PT(5);
            if (tid == 32 * kDrainWarp0) SSD_TL(2, T, 3);
        }
        if (n_my > 0) {
            tail1(n_my - 1);
            tail2(n_my - 1);
        }
        if (tid == 32 * kDrainWarp0) SSD_PT_FLUSH(2);
    }
    if (kPool) {
        tc_fence_before();
        __syncthreads();
    }
    ++seg;
    } while (kPool && seg_end < tile_end);
    tc_fence_before();
    __syncthreads();
    if (warp == kMmaWarp) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
}

// LSTM cell update after the gate GEMM (conv_to_fcnet_v2.py:68-80, Keras gate order i, f, c~, o):
//   c' = sigmoid(f) * c + sigmoid(i) * tanh(c~),  h' = sigmoid(o) * tanh(c').
// One pass over HBM: bf16 gate pre-activations [M][4u] (+ fp32 bias) and c in, c', h' (fp32) and h' (bf16, the next GEMM
// operand) out.  A thread owns eight consecutive units of one agent.
__global__ void __launch_bounds__(256) lstm_cell_kernel(const uint4* __restrict__ gates, const float* __restrict__ bias, const float4* __restrict__ c_prev,
                                                        float4* __restrict__ c_out, float4* __restrict__ h_out, uint4* __restrict__ h16_out, long long M, int units) {
    const int per_row = units >> 3;
    const long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (idx >= M * per_row) return;
    const long long m = idx / per_row;
    const int j8 = static_cast<int>(idx - m * per_row);
    float g[4][8];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const uint4 v = gates[(m * 4 + q) * per_row + j8];
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
        const float* b = bias + q * units + j8 * 8;
#pragma unroll
        for (int e = 0; e < 4; ++e) {  // bf16 -> fp32 is a shift
            g[q][2 * e] = __uint_as_float(w[e] << 16) + b[2 * e];
            g[q][2 * e + 1] = __uint_as_float(w[e] & 0xffff0000u) + b[2 * e + 1];
        }
    }
    const float4 c0 = c_prev[idx * 2], c1 = c_prev[idx * 2 + 1];
    const float c[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
    float cn[8], hn[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        const float si = 1.f / (1.f + __expf(-g[0][e])), sf = 1.f / (1.f + __expf(-g[1][e])), so = 1.f / (1.f + __expf(-g[3][e]));
        cn[e] = sf * c[e] + si * tanhf(g[2][e]);
        hn[e] = so * tanhf(cn[e]);
    }
    c_out[idx * 2] = make_float4(cn[0], cn[1], cn[2], cn[3]);
    c_out[idx * 2 + 1] = make_float4(cn[4], cn[5], cn[6], cn[7]);
    h_out[idx * 2] = make_float4(hn[0], hn[1], hn[2], hn[3]);
    h_out[idx * 2 + 1] = make_float4(hn[4], hn[5], hn[6], hn[7]);
    uint32_t p[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        const __nv_bfloat162 v = __floats2bfloat162_rn(hn[2 * e], hn[2 * e + 1]);
        p[e] = *reinterpret_cast<const uint32_t*>(&v);
    }
    h16_out[idx] = make_uint4(p[0], p[1], p[2], p[3]);
}

inline auto features_kernel(WeightMap m) {
    return m == WeightMap::Shared ? policy_features_kernel<WeightMap::Shared>
                                  : m == WeightMap::PerAgent ? policy_features_kernel<WeightMap::PerAgent> : policy_features_kernel<WeightMap::Pool>;
}
inline int smem_bytes(WeightMap m) { return m == WeightMap::Shared ? TrunkSmem<false>::kSmemBytes : TrunkSmem<true>::kSmemBytes; }

// ssd_policy_[pool_]features: policy_ids is null for a network handle
int features(ssd_policy_t p, const uint8_t* obs, const uint8_t* policy_ids, int64_t num_agents, float* features, void* stream) {
    const bool pool = policy_ids != nullptr;
    if (!p || !obs || !features || num_agents < 0) return ssd::set_error(SSD_ERR_INVALID, "bad argument");
    // ssd_policy_features reports misaligned pointers before a wrong kind of handle, ssd_policy_pool_features after it
    const char* misaligned = "obs and features must be 16-byte aligned";
    if (!pool && check_aligned({obs, features}, misaligned) != SSD_OK) return SSD_ERR_INVALID;
    int rc = pool ? check_kind(p, HandleKind::Pool, "not a policy pool handle (ssd_policy_create_pool)")
                  : check_kind(p, HandleKind::Net, "a policy pool handle takes ssd_policy_pool_features");
    if (rc == SSD_OK) rc = check_aligned({obs, features}, misaligned);
    if (rc != SSD_OK) return rc;
    if (!pool && num_agents % p->num_policies != 0) return ssd::set_error(SSD_ERR_INVALID, "num_agents must be a multiple of num_policies");
    if (num_agents == 0) return SSD_OK;
    rc = setup(p, policy_ids, num_agents, stream);
    if (rc != SSD_OK) return rc;
    const Grid g = grid(p, num_agents);
    const WeightMap map = weight_map(p);
    features_kernel(map)<<<g.ctas, kThreads, smem_bytes(map), static_cast<cudaStream_t>(stream)>>>(
        obs, num_agents, p->d_blob, features, p->num_policies, g.ctas_per_policy, p->d_perm, p->d_tiles, ssd::policy_pool::num_tiles(p));
    return launched();
}

// Packs num_policies trunk weight sets (Keras layouts, consecutive behind each pointer) into a new handle; the caller has
// checked num_policies against its map's limit.
int create_trunk(int view_radius, int device, int num_policies, WeightMap map, const float* conv_w, const float* conv_b, const float* fc1_w,
                 const float* fc1_b, const float* fc2_w, const float* fc2_b, SsdPolicy** out) {
    if (!out) return ssd::set_error(SSD_ERR_INVALID, "null argument");
    *out = nullptr;
    if (!conv_w || !conv_b || !fc1_w || !fc1_b || !fc2_w || !fc2_b) return ssd::set_error(SSD_ERR_INVALID, "null weight pointer");
    if (2 * view_radius + 1 != V) return ssd::set_error(SSD_ERR_UNSUPPORTED, "the feature kernel is built for 15x15 observations (view radius 7)");
    const size_t blob_bytes = static_cast<size_t>(num_policies) * kBlobBytes;
    std::vector<uint8_t> blobs(blob_bytes, 0);
    for (int q = 0; q < num_policies; ++q) {  // weight set q: arrays q of the num_policies consecutive ones behind each pointer
        uint8_t* blob = blobs.data() + static_cast<size_t>(q) * kBlobBytes;
        const float* cw = conv_w + q * (9 * 3 * NF);
        const float* cbias = conv_b + q * NF;
        const float* w1 = fc1_w + static_cast<size_t>(q) * (CO * CO * NF * N2);
        const float* b1v = fc1_b + q * N2;
        const float* w2 = fc2_w + q * (K3 * N3);
        const float* b2v = fc2_b + q * N3;
        __half* b1 = reinterpret_cast<__half*>(blob);                          // resident: conv, fc2, constants
        __half* b3 = reinterpret_cast<__half*>(blob + kB1Bytes);
        float* cst = reinterpret_cast<float*>(blob + kB1Bytes + kB3Bytes);
        __half* b2 = reinterpret_cast<__half*>(blob + kHeadBytes);             // streamed: the 13 row blocks of Dense(32)
        // banded conv weights: conv_w[di][dj][c][f] (Keras kernel layout) at tap k = 48 di + 3 (j + dj) + c of column n = 6 j + f
        for (int j = 0; j < CO; ++j)
            for (int f = 0; f < NF; ++f) {
                double sum16 = 0.0;
                for (int di = 0; di < 3; ++di)
                    for (int dj = 0; dj < 3; ++dj)
                        for (int c = 0; c < 3; ++c) {
                            const __half h = __float2half_rn(cw[((di * 3 + dj) * 3 + c) * NF + f]);
                            b1[kmajor(N1, j * NF + f, di * ROWK + (j + dj) * 3 + c)] = h;
                            sum16 += static_cast<double>(__half2float(h));
                        }
                // relu(conv((x - 128) / 255) + b) with the operand holding 1024 + x
                cst[j * NF + f] = static_cast<float>(static_cast<double>(cbias[f]) - (1024.0 + 128.0) * sum16 / 255.0);
            }
        for (int i = 0; i < CO; ++i)  // Dense(32) kernel [1014][32], inputs flattened (i, j, f)
            for (int k = 0; k < CO * NF; ++k)
                for (int n = 0; n < N2; ++n) b2[i * (K2 * N2) + kmajor(N2, n, k)] = __float2half_rn(w1[(i * CO * NF + k) * N2 + n]);
        for (int k = 0; k < K3; ++k)
            for (int n = 0; n < N3; ++n) b3[kmajor(N3, n, k)] = __float2half_rn(w2[k * N3 + n]);
        for (int n = 0; n < N2; ++n) cst[N1 + n] = b1v[n];
        for (int n = 0; n < N3; ++n) cst[N1 + N2 + n] = b2v[n];
    }

    SsdPolicy* p = new (std::nothrow) SsdPolicy();
    if (!p) return ssd::set_error(SSD_ERR_INVALID, "out of host memory");
    p->device = device;
    p->num_policies = num_policies;
    p->kind = map == WeightMap::Pool ? HandleKind::Pool : HandleKind::Net;
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&p->sms, cudaDevAttrMultiProcessorCount, device);
    if (e == cudaSuccess) e = cudaMalloc(&p->d_blob, blob_bytes);
    if (e == cudaSuccess) e = cudaMemcpy(p->d_blob, blobs.data(), blob_bytes, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(features_kernel(weight_map(p)), cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes(weight_map(p)));
    if (e != cudaSuccess) {
        if (p->d_blob) cudaFree(p->d_blob);
        delete p;
        return ssd::set_error(SSD_ERR_CUDA, cudaGetErrorString(e));
    }
    *out = p;
    return SSD_OK;
}


}  // namespace policy
}  // namespace ssd


#pragma GCC visibility push(default)
extern "C" {

int ssd_policy_create_n(int view_radius, int device, int num_policies, const float* conv_w, const float* conv_b, const float* fc1_w,
                        const float* fc1_b, const float* fc2_w, const float* fc2_b, ssd_policy_t* out) {
    if (out) *out = nullptr;
    if (num_policies < 1 || num_policies > SSD_MAX_AGENTS) return ssd::set_error(SSD_ERR_INVALID, "num_policies must be 1..SSD_MAX_AGENTS");
    return ssd::policy::create_trunk(view_radius, device, num_policies, WeightMap::PerAgent, conv_w, conv_b, fc1_w, fc1_b, fc2_w, fc2_b, out);
}
int ssd_policy_create(int view_radius, int device, const float* conv_w, const float* conv_b, const float* fc1_w, const float* fc1_b,
                      const float* fc2_w, const float* fc2_b, ssd_policy_t* out) {
    return ssd_policy_create_n(view_radius, device, 1, conv_w, conv_b, fc1_w, fc1_b, fc2_w, fc2_b, out);
}

int ssd_policy_features(ssd_policy_t p, const uint8_t* obs, int64_t num_agents, float* features, void* stream) {
    return ssd::policy::features(p, obs, nullptr, num_agents, features, stream);
}

int ssd_policy_pool_features(ssd_policy_t p, const uint8_t* obs, const uint8_t* policy_ids, int64_t num_agents, float* features, void* stream) {
    if (!policy_ids) return ssd::set_error(SSD_ERR_INVALID, "bad argument");
    return ssd::policy::features(p, obs, policy_ids, num_agents, features, stream);
}

int ssd_policy_lstm_cell(const void* gates_bf16, const float* bias, const float* c_prev, float* c_out, float* h_out, void* h_bf16_out,
                         int64_t num_agents, int units, void* stream) {
    using namespace ssd::policy;
    if (!gates_bf16 || !bias || !c_prev || !c_out || !h_out || !h_bf16_out || num_agents < 0) return ssd::set_error(SSD_ERR_INVALID, "bad argument");
    if (units <= 0 || units % 8 != 0) return ssd::set_error(SSD_ERR_INVALID, "units must be a positive multiple of 8");
    const int rc = check_aligned({gates_bf16, bias, c_prev, c_out, h_out, h_bf16_out}, "pointers must be 16-byte aligned");
    if (rc != SSD_OK) return rc;
    if (num_agents == 0) return SSD_OK;
    const long long n = num_agents * (units / 8);
    lstm_cell_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const uint4*>(gates_bf16), bias, reinterpret_cast<const float4*>(c_prev), reinterpret_cast<float4*>(c_out),
        reinterpret_cast<float4*>(h_out), static_cast<uint4*>(h_bf16_out), num_agents, units);
    return launched();
}

void ssd_policy_destroy(ssd_policy_t p) {
    if (!p) return;
    cudaSetDevice(p->device);
    cudaFree(p->d_blob);
    if (p->d_head_blob) cudaFree(p->d_head_blob);
    if (p->d_counts) cudaFree(p->d_counts);
    if (p->d_perm) cudaFree(p->d_perm);
    if (p->d_tiles) cudaFree(p->d_tiles);
    if (p->d_moa_rows) cudaFree(p->d_moa_rows);
    delete p;
}

}  // extern "C"
#pragma GCC visibility pop
