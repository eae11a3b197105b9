/* libssd_b200 -- C ABI of the B200-native batched SSD gridworld step path.
 *
 * Drop-in boundary for the `MapEnv.step` / `MapEnv.reset` path of
 * vermashresth/sequential_social_dilemma_games (Harvest, Cleanup).  The reference has no FFI of its
 * own (it is pure Python behind RLlib's MultiAgentEnv, map_env.py:9,60); each entry point below
 * names the reference method(s) it replaces, and INTEGRATION.md shows the ctypes binding a
 * maintainer would add to social_dilemmas/envs/map_env.py.
 *
 * Conventions
 *   - plain C, no exceptions: every call returns 0 on success or a negative SSD_ERR_* code;
 *     ssd_last_error() returns a thread-local message for the last failure.
 *   - a handle owns the state of `num_envs` independent environments resident in the HBM of ONE
 *     GPU.  It is not thread-safe; use one handle per GPU (one process per GPU).
 *   - "dev" pointers are device pointers (e.g. PyTorch tensors); "host" pointers are host memory.
 *     `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  Calls are
 *     asynchronous with respect to the host unless stated otherwise.
 *   - encodings: grid cells are ASCII codes as in the reference's `world_map` (' ', '@', 'A', 'H',
 *     'R', 'S'); positions are (row, col) int16; orientations 0 UP, 1 RIGHT, 2 DOWN, 3 LEFT;
 *     actions follow agent.py:7-13,148-149,186-188 (0 MOVE_LEFT, 1 MOVE_RIGHT, 2 MOVE_UP, 3 MOVE_DOWN,
 *     4 STAY, 5 TURN_CLOCKWISE, 6 TURN_COUNTERCLOCKWISE, 7 FIRE, 8 CLEAN), -1 = the agent is absent
 *     from the action dict (map_env.py:171 iterates only the given keys).
 *   - observations are uint8 RGB [B][N][V][V][3], V = 2*view_radius+1, i.e. the array the
 *     reference holds just before `(rgb - 128.0) / 255.0` (map_env.py:197-199).
 */
#ifndef SSD_B200_H
#define SSD_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SSD_ABI_VERSION 2
#define SSD_MAX_AGENTS 16

#define SSD_KIND_HARVEST 0 /* social_dilemmas/envs/harvest.py:18  HarvestEnv */
#define SSD_KIND_CLEANUP 1 /* social_dilemmas/envs/cleanup.py:30  CleanupEnv */
#define SSD_KIND_PLAIN 2   /* MapEnv without custom_action / custom_map_update (tests' DummyMapEnv) */

#define SSD_OK 0
#define SSD_ERR_INVALID -1     /* bad argument / unsupported configuration */
#define SSD_ERR_CUDA -2        /* a CUDA runtime call failed */
#define SSD_ERR_UNSUPPORTED -3 /* configuration does not fit the device (shared memory) */

/* Phases of MapEnv.step (map_env.py:152-212), for callers that override a hook
 * (custom_action / custom_map_update, map_env.py:108-125) and need the rest on the GPU. */
#define SSD_PHASE_MOVES 1    /* update_moves                       map_env.py:176, 357-543 */
#define SSD_PHASE_CONSUME 2  /* agent.consume loop                 map_env.py:178-181 */
#define SSD_PHASE_BEAMS 4    /* update_custom_moves/custom_action  map_env.py:184, 545-649 */
#define SSD_PHASE_SPAWN 8    /* custom_map_update                  map_env.py:187 */
#define SSD_PHASE_RENDER 16  /* get_map_with_agents..rotate_view   map_env.py:189-199 */
#define SSD_PHASE_ALL 31

#define SSD_NUM_STATS 8
/* ssd_stats order: env_steps, reward_sum, apples_eaten, fires, hits, cleaned, apples_spawned, waste_spawned */

typedef struct SsdEnv* ssd_handle;

/* Static description of a game: what MapEnv.__init__ (map_env.py:62-102), HarvestEnv.__init__
 * (harvest.py:20-28) and CleanupEnv.__init__ (cleanup.py:32-66) derive from their arguments and the
 * module constants.  All pointers are HOST pointers, read during ssd_create only. */
typedef struct SsdConfig {
    int32_t abi_version;   /* SSD_ABI_VERSION */
    int32_t kind;          /* SSD_KIND_* */
    int32_t height, width; /* ascii_map shape; <= 255 each; the map must be wall-enclosed (agent.py:111) */
    int32_t num_agents;    /* 1..SSD_MAX_AGENTS; ids are 'agent-0'..'agent-(N-1)' (harvest.py:50) */
    int32_t view_radius;   /* HARVEST_VIEW_SIZE / CLEANUP_VIEW_SIZE (harvest.py:15, cleanup.py:22) */
    int32_t beam_len;      /* ACTIONS['FIRE'] (harvest.py:11, cleanup.py:11-12) */
    int32_t num_envs;      /* B: environments owned by this handle */
    int32_t device;        /* CUDA device ordinal */
    int32_t envs_per_cta;  /* 0 = choose automatically */
    uint64_t env_id_offset;/* global id of local env 0 (shard offset): Philox streams are keyed by
                              global ids, so trajectories do not depend on the sharding */
    const uint8_t* base_map;            /* [height*width] ASCII (map_env.py:80 ascii_to_numpy) */
    const uint8_t* color_lut;           /* [128*3] RGB by ASCII code (map_env.py:24-41, cleanup.py:15-18) */
    const double* harvest_spawn_prob;   /* [4] SPAWN_PROB (harvest.py:13) */
    const double* cleanup_apple_prob;   /* [potential_waste_area+1] by #'H' cells (cleanup.py:156-171) */
    const double* cleanup_waste_prob;   /* [potential_waste_area+1] */
    int32_t potential_waste_area;       /* cleanup.py:36-38 */
    int32_t num_spawn_points;
    const int16_t* spawn_points;        /* [num_spawn_points][2] sorted (row, col); Cleanup lists every
                                           'P' twice (map_env.py:96-99 + cleanup.py:51-52) */
} SsdConfig;

/* RNG replay ("tape-out", SURVEY.md 8c): the results of the reference's random calls for ONE step.
 * All pointers are dev pointers.  NULL tape => the production Philox4x32-10 streams. */
typedef struct SsdTape {
    const uint8_t* move_order;   /* [B][N] agent indices after np.random.shuffle (map_env.py:422), 0xFF padded */
    const double* uniforms;      /* [B][u_stride] np.random.rand(1)[0] in call order (harvest.py:101, cleanup.py:139,150) */
    int32_t u_stride;
    const uint16_t* waste_order; /* [B][num_waste_points] cell ids (row*W+col) after random.shuffle (cleanup.py:145); may be NULL for non-Cleanup */
    int32_t* n_draws_out;        /* [B] or NULL: number of uniforms the spawn pass consumed, so a caller that feeds
                                    np.random.rand values can advance its generator by exactly that many draws */
} SsdTape;

const char* ssd_last_error(void);
int ssd_abi_version(void);

/* MapEnv.__init__ .. without the RNG-consuming setup_agents() (map_env.py:102): state is
 * the post-reset_map() grid with all agents parked on the first 'P' spawn point of the map (cell (1,1) when the
 * map has none) until ssd_reset or ssd_set_state places them. */
int ssd_create(const SsdConfig* cfg, ssd_handle* out);
int ssd_destroy(ssd_handle h);

/* Sizes (elements) of the arrays the other calls take. */
int ssd_num_apple_points(ssd_handle h);
int ssd_num_waste_points(ssd_handle h);
int64_t ssd_obs_bytes_per_env(ssd_handle h);
int ssd_envs_per_cta(ssd_handle h);
int64_t ssd_algorithmic_bytes_per_env_step(ssd_handle h); /* SURVEY.md 8d definition, for rooflines */

/* np.random.seed / random.seed analogue for the production streams: Philox key = seed, and
 * the per-env step counter t (incremented by every ssd_step; ssd_reset uses but keeps it). */
int ssd_seed(ssd_handle h, uint64_t seed, uint32_t t);
int ssd_get_counter(ssd_handle h, uint32_t* t);

/* State upload / download (parity, checkpoint/resume).  Pointers may be host or dev (UVA).
 * grid u8[B][H*W], pos i16[B][N][2], ori u8[B][N].  Reference fields: MapEnv.world_map
 * (map_env.py:85), Agent.pos / Agent.orientation (agent.py:37-38).
 * ssd_set_state validates every position (0 <= row < H, 0 <= col < W) before it touches the state and returns
 * SSD_ERR_INVALID otherwise (it synchronises `stream` to do so).  An agent placed on a '@' cell -- which the
 * reference never does -- is accepted as PARKED: it keeps its place, never acts, is never painted or hit, so
 * that no beam ever starts outside the wall enclosure. */
int ssd_set_state(ssd_handle h, const uint8_t* grid, const int16_t* pos, const uint8_t* ori, void* stream);
int ssd_get_state(ssd_handle h, uint8_t* grid, int16_t* pos, uint8_t* ori, void* stream);

/* MapEnv.reset (map_env.py:214-249): setup_agents (spawn_point :651, spawn_rotation :664),
 * reset_map (:560), one custom_map_update (:230), un-rotated observations (:239-240).
 * mask dev u8[B] (NULL = all envs): only envs with mask != 0 are reset and rendered.
 * obs_out dev u8[B][N][V][V][3] or NULL. */
int ssd_reset(ssd_handle h, const uint8_t* mask, uint8_t* obs_out, void* stream);

/* MapEnv.reset of the listed environments only (RLlib resets sub-environments one at a time at the episode
 * horizon, map_env.py:214-249 is per env): ONE launch over n_rows warps instead of a masked pass over all B.
 * rows: host or dev i32[n_rows], each in 0..B-1 (a host list is range-checked; out-of-range device entries are
 * skipped).  obs_out is the full dev u8[B][N][V][V][3] tensor (or NULL); only the listed rows are written. */
int ssd_reset_rows(ssd_handle h, const int32_t* rows, int n_rows, uint8_t* obs_out, void* stream);

/* MapEnv.step (map_env.py:152-212) for all B envs in one fused launch.
 * actions dev i8[B][N]; action_order dev u8[B][N] = iteration order of the action dict as agent
 * indices (NULL = 0..N-1); tape NULL or replayed RNG; obs_out dev u8[B][N][V][V][3] (NULL skips
 * rendering); reward_out dev i32[B][N] (Agent.compute_reward, agent.py:80-83).  dones are always
 * False in the reference (agent.py:174,209; map_env.py:211) and are not materialised. */
int ssd_step(ssd_handle h, const int8_t* actions, const uint8_t* action_order, const SsdTape* tape,
             uint8_t* obs_out, int32_t* reward_out, void* stream);

/* A scripted rollout: `num_steps` consecutive ssd_step calls whose actions all exist up front -- actions dev
 * i8[num_steps][B][N] in agent order, rewards dev i32[num_steps][B][N], observations of step s into slot s % ring_slots of
 * obs_ring dev u8[ring_slots][B][N][V][V][3].  Because no input of a later step is produced between the launches, the
 * library chains the step kernels (see SSD_OPT_CHAIN_STEPS) regardless of the option; results equal num_steps calls of
 * ssd_step.  This is the reference's own benchmark shape (random-action rollouts). */
int ssd_rollout(ssd_handle h, int num_steps, const int8_t* actions, uint8_t* obs_ring, int ring_slots, int32_t* reward_out, void* stream);

/* A subset of the phases of one step (SSD_PHASE_* mask), for overridden hooks: e.g. run
 * MOVES|CONSUME, apply a Python custom_action through ssd_get_state/ssd_set_state, then
 * SPAWN|RENDER.  Beam cells persist on the device between the phase calls of one step; rewards
 * accumulate in reward_out (the caller zeroes it at the start of the step).  The step counter
 * advances when `phases` contains SSD_PHASE_SPAWN. */
int ssd_step_phases(ssd_handle h, int phases, const int8_t* actions, const uint8_t* action_order,
                    const SsdTape* tape, uint8_t* obs_out, int32_t* reward_out, void* stream);

/* Beam cells of the last SSD_PHASE_BEAMS call that did not render (phase-split stepping), for
 * MapEnv.beam_pos / test_map (map_env.py:169,275-276,648).  out dev-or-host u8[B][64]:
 * bytes 0..47 = painted cells of ray s of the k-th action-dict entry at [k*3+s], bytes 48..63 = beam
 * character of entry k (0 none, 'F', 'C').  Synchronises `stream` when `out` is host memory. */
int ssd_get_beams(ssd_handle h, uint8_t* out, void* stream);

/* Observations of the current state without beams: rotate != 0 as step renders them
 * (map_env.py:197-198), 0 as reset does (map_env.py:239).  Backs Agent.get_state /
 * MapEnv.map_to_colors for the adapters. */
int ssd_render(ssd_handle h, int rotate, uint8_t* obs_out, void* stream);

/* Full-map frames for video / visualisation: MapEnv.map_to_colors(get_map_with_agents()) (map_env.py:280-339,
 * rollout.py:48-82) of every env.  rgb_out dev u8[B][H][W][3].  Beams live for one step only
 * (map_env.py:169) and are not drawn. */
int ssd_render_map(ssd_handle h, uint8_t* rgb_out, void* stream);

/* End-to-end step with HOST buffers: H2D actions, fused step, D2H observations and rewards,
 * pipelined in chunks over two internal streams; returns after everything landed.
 * actions_host i8[B][N], obs_host u8[B][N][V][V][3] (NULL to skip), reward_host i32[B][N].
 * Pinned host memory gives full PCIe bandwidth; pageable memory works but is slower.
 * The internal streams first wait for everything already queued on `stream` (NULL = legacy default stream), so
 * the call is ordered after an asynchronous ssd_reset / ssd_set_state / ssd_step issued there. */
int ssd_step_host(ssd_handle h, const int8_t* actions_host, uint8_t* obs_host, int32_t* reward_host, void* stream);

/* ---- Policy-side consumer of the observation tensor (SURVEY 8f-4) -------------------------------------------------
 * The feature trunk of the reference's policy network, models/conv_to_fcnet_v2.py:36-66: Conv2D(6, 3x3, stride 1,
 * 'valid') -> ReLU -> flatten -> Dense(32) -> ReLU -> Dense(32) -> ReLU, applied to (obs - 128) / 255 (map_env.py:199)
 * of uint8 observations resident in HBM -- what ssd_step / ssd_rollout wrote -- in one fused tensor-core kernel
 * (fp16 operands, fp32 accumulation; nothing but the features returns to HBM).  The LSTM and the two heads that
 * follow (conv_to_fcnet_v2.py:68-92) are ssd_policy_lstm_heads below (one fused kernel); ssd_policy_lstm_cell is the
 * elementwise cell update for callers that run the gate GEMMs of another cell size through their own BLAS.
 *
 * Weights are HOST fp32 arrays in the Keras layouts: conv_w [3][3][3][6] (kh, kw, in, out), conv_b [6],
 * fc1_w [1014][32] (inputs flattened (row, col, filter) as keras Flatten does), fc1_b [32], fc2_w [32][32], fc2_b [32].
 * Only view_radius 7 (15x15 observations, the reference's HARVEST_VIEW_SIZE / CLEANUP_VIEW_SIZE) is built. */
typedef struct SsdPolicy* ssd_policy_t;
int ssd_policy_create(int view_radius, int device, const float* conv_w, const float* conv_b, const float* fc1_w, const float* fc1_b,
                      const float* fc2_w, const float* fc2_b, ssd_policy_t* out);
/* obs dev u8[num_agents][15][15][3] (16-byte aligned; the [B][N][...] tensor of ssd_step with num_agents = B*N),
 * features dev f32[num_agents][32] (16-byte aligned). */
int ssd_policy_features(ssd_policy_t p, const uint8_t* obs, int64_t num_agents, float* features, void* stream);
void ssd_policy_destroy(ssd_policy_t p);
/* LSTM(128) + logits / value heads + action sampling in ONE kernel (conv_to_fcnet_v2.py:68-92; Keras gate order i, f, c~, o,
 * sigmoid recurrent activation).  ssd_policy_set_head packs HOST fp32 weights in the Keras layouts: lstm_w [32][4u],
 * lstm_u [u][4u], lstm_b [4u], logits_w [u][num_outputs], logits_b, value_w [u][1], value_b [1]; units must be 128,
 * num_outputs 1..15.  ssd_policy_lstm_heads: features dev f32[M][32] (ssd_policy_features); h_in / c_in / h_out / c_out dev
 * f32 recurrent state in the library's TILED layout [ceil(M/128)][8][128][16]: element (agent m, unit u) at
 * ((m / 128 * 8 + u / 16) * 128 + m % 128) * 16 + u % 16 -- buffers of ceil(M/128) * 16384 floats, zero for an initial
 * state, out may alias in (a warp then moves 2 KB contiguous per access instead of 64-byte row pieces);
 * logits dev f32[M][num_outputs], value dev f32[M], actions dev i8[M] or NULL: a sample
 * of softmax(logits) by the Gumbel-max rule on Philox4x32-10 (key = seed, counter words = agent index, `counter`) -- pass a
 * fresh `counter` every step.  fp16 GEMM operands, fp32 accumulation and state. */
int ssd_policy_set_head(ssd_policy_t p, int units, int num_outputs, const float* lstm_w, const float* lstm_u, const float* lstm_b,
                        const float* logits_w, const float* logits_b, const float* value_w, const float* value_b);
int ssd_policy_lstm_heads(ssd_policy_t p, const float* features, const float* h_in, const float* c_in, float* h_out, float* c_out, float* logits,
                          float* value, int8_t* actions, int64_t num_agents, uint64_t seed, uint32_t counter, void* stream);
/* One network per agent id, as the reference's training scripts build them (a policy per 'agent-i', policy_mapping_fn
 * mapping agent i to it): num_policies = P weight sets, 1..SSD_MAX_AGENTS.  Every weight pointer points to P consecutive
 * arrays, each in the layout above.  Agent m = b*P + p of the [B][P][15][15][3] observation tensor (num_agents = B*P) is
 * evaluated with weight set p; features, logits, value and actions stay agent-major ([M][...], M = B*P), and the Philox
 * counter words of the sampler are the agent-major index m, so P copies of one weight set give exactly the outputs of the
 * shared network.  ssd_policy_set_head_n must be given the P of ssd_policy_create_n; on a handle with P > 1,
 * ssd_policy_features and ssd_policy_lstm_heads return SSD_ERR_INVALID unless num_agents % P == 0.
 * The TILED recurrent state of such a handle is grouped per policy: P*G groups, G = ceil(B/128), shape [P*G][8][128][16];
 * state group p*G + g holds policy p and envs b in [128 g, 128 g + 128): element (agent m = b*P + p, unit u) at
 * (((p*G + b/128) * 8 + u/16) * 128 + b % 128) * 16 + u % 16.  P = 1 is the shared network (ssd_policy_create /
 * ssd_policy_set_head are that case). */
int ssd_policy_create_n(int view_radius, int device, int num_policies, const float* conv_w, const float* conv_b, const float* fc1_w,
                        const float* fc1_b, const float* fc2_w, const float* fc2_b, ssd_policy_t* out);
int ssd_policy_set_head_n(ssd_policy_t p, int num_policies, int units, int num_outputs, const float* lstm_w, const float* lstm_u,
                          const float* lstm_b, const float* logits_w, const float* logits_b, const float* value_w, const float* value_b);
/* A policy pool: num_policies = K weight sets, 1..255, loaded once; every call takes a device u8 policy id per agent, and the
 * ids may change from call to call (several runs or seeds on one GPU, cross-play teams, population play, scripted agents).
 * ssd_policy_create_pool loads trunk and head together: every weight pointer points to K consecutive arrays in the layouts of
 * ssd_policy_create / ssd_policy_set_head; the fused head is required.  K outside 1..255 or a null pointer returns
 * SSD_ERR_INVALID; view_radius != 7, units != 128 or num_outputs outside 1..15 SSD_ERR_UNSUPPORTED; nothing is allocated then.
 * ssd_policy_pool_features / ssd_policy_pool_lstm_heads take the arguments of ssd_policy_features / ssd_policy_lstm_heads plus
 * policy_ids dev u8[num_agents], agent-major like obs: agent m is evaluated with weight set policy_ids[m].
 *   - An id >= K means "no pool policy": nothing is written for that agent -- none of its rows of features, logits, value,
 *     actions, h_out or c_out -- so a caller can drive it with its own code (as ssd_reset_rows ignores out-of-range rows).
 *   - The recurrent state is in the TILED layout of the shared network, [ceil(M/128)][8][128][16] (element (agent m, unit u) at
 *     ((m / 128 * 8 + u / 16) * 128 + m % 128) * 16 + u % 16): it does not depend on the ids, so they may change between two
 *     steps of a live state.  An agent's rows of h_out / c_out are written only when it has a pool policy.
 *   - Sampling keys Philox by (seed; m, counter) as ssd_policy_lstm_heads does: weight set k gives agent m exactly the action
 *     a shared network with set k draws for m.
 * Each call first groups the agents by id on the device (no host synchronisation) into scratch that belongs to the handle
 * and grows on demand, so calls on one pool handle must be ordered (one stream).  Pool handles are rejected by
 * ssd_policy_features / ssd_policy_lstm_heads / ssd_policy_set_head(_n), other handles by the pool entry points
 * (SSD_ERR_INVALID).  At most 2^31 - 1 agents per call. */
int ssd_policy_create_pool(int view_radius, int device, int num_policies, int units, int num_outputs, const float* conv_w, const float* conv_b,
                           const float* fc1_w, const float* fc1_b, const float* fc2_w, const float* fc2_b, const float* lstm_w, const float* lstm_u,
                           const float* lstm_b, const float* logits_w, const float* logits_b, const float* value_w, const float* value_b,
                           ssd_policy_t* out);
int ssd_policy_pool_features(ssd_policy_t p, const uint8_t* obs, const uint8_t* policy_ids, int64_t num_agents, float* features, void* stream);
int ssd_policy_pool_lstm_heads(ssd_policy_t p, const float* features, const uint8_t* policy_ids, const float* h_in, const float* c_in, float* h_out,
                               float* c_out, float* logits, float* value, int8_t* actions, int64_t num_agents, uint64_t seed, uint32_t counter,
                               void* stream);
/* The policy's distribution at the chosen action, in the same kernel: ssd_policy_lstm_heads / ssd_policy_pool_lstm_heads (same
 * handles, state layouts and rules; the _dist form of each rejects the other kind of handle) that also return, per agent,
 *   logp    dev f32[M] or NULL: log softmax(logits)[a] = l[a] - logsumexp(l) of the agent's action a, computed from the fp32
 *           logits the call writes (max subtracted first, accurate expf / logf);
 *   entropy dev f32[M] or NULL: -sum_i softmax(l)_i log softmax(l)_i.
 * `mode` chooses the action a:
 *   SSD_ACT_SAMPLE  the Gumbel-max sampler of ssd_policy_lstm_heads: with the same seed and counter the actions are bitwise those
 *                   of the plain entry point; written to actions dev i8[M];
 *   SSD_ACT_GREEDY  the first index of the maximum of the fp32 logits as written (np.argmax of them where they are
 *                   finite; a NaN logit is passed over unless it is the first); written to actions;
 *   SSD_ACT_GIVEN   actions dev i8[M] is an INPUT and is not written (a scripted agent, another policy's action, a recorded
 *                   trajectory: the pi(a) of an importance ratio); a value outside 0..num_outputs-1 (-1 included) gives logp NaN
 *                   for that agent and changes nothing else.
 * logits, value, h_out and c_out are exactly what the plain entry point writes; a pool's agents with an id >= K get nothing
 * written, logp and entropy included.  logp is the model's probability of the action; in SSD_ACT_SAMPLE it is not the
 * sampler's realised frequency, which deviates where the sampler's fast -log(u) is inexact for u close to 1.  A mode outside
 * the three, NULL actions, or a handle of the other kind returns SSD_ERR_INVALID before anything is launched. */
#define SSD_ACT_SAMPLE 0
#define SSD_ACT_GREEDY 1
#define SSD_ACT_GIVEN 2
int ssd_policy_lstm_heads_dist(ssd_policy_t p, const float* features, const float* h_in, const float* c_in, float* h_out, float* c_out,
                               float* logits, float* value, int mode, int8_t* actions, float* logp, float* entropy, int64_t num_agents,
                               uint64_t seed, uint32_t counter, void* stream);
int ssd_policy_pool_lstm_heads_dist(ssd_policy_t p, const float* features, const uint8_t* policy_ids, const float* h_in, const float* c_in,
                                    float* h_out, float* c_out, float* logits, float* value, int mode, int8_t* actions, float* logp,
                                    float* entropy, int64_t num_agents, uint64_t seed, uint32_t counter, void* stream);
/* Model of other agents (MOA) and social-influence reward of the causal-influence models (models/moa_model.py MOA_LSTM,
 * common_funcs.py compute_influence_reward), forward only, in ONE kernel.  For agent m = b*N + i (env b, agent i):
 *   input(a') = [features(32) | onehot(a') | onehot(a_{b,j}) for j != i, increasing j], width 32 + N*A; an action outside 0..A-1
 *   is a zero one-hot row.  LSTM(128) (Keras gate order i, f, c~, o, as ssd_policy_set_head), then Dense((N-1)*A), columns
 *   (other k in the same order, action).
 * ssd_moa_create packs HOST fp32 weights in the Keras layouts: lstm_w [32 + N*A][512], lstm_u [128][512], lstm_b [512],
 * logits_w [128][(N-1)*A], logits_b [(N-1)*A]; num_policies 1 (shared) or N (agent i uses weight set i, the pointers then point
 * to N consecutive arrays, as ssd_policy_create_n).  N = num_agents 2..SSD_MAX_AGENTS, A = num_actions 1..15, (N-1)*A <= 64.
 * ssd_moa_step, M = num_agents a multiple of N:
 *   features dev f32[M][32] (ssd_policy_features), joint_actions dev i8[M] ([B][N], the actions the step took),
 *   policy_logits dev f32[M][A] (the policy's logits of that step); h_in / c_in / h_out / c_out the MOA's recurrent state in the
 *   TILED layout of ssd_policy_lstm_heads (grouped per weight set for num_policies = N, as ssd_policy_create_n), out must not
 *   alias in; all five 16-byte aligned.
 *   pred dev f32[M][N-1][A]: the MOA logits at the actual joint action; h_out / c_out: the next state at the actual action.
 *   counterfactual dev f32[M][A][N-1][A] or NULL: the logits with the own action replaced by a' (equal to pred at a' = a_{b,i}).
 *   influence_per_agent dev f32[M][N-1]: D(p_k(.|a_{b,i}) || q_k), p_k(.|a') = softmax(counterfactual[m][a'][k]),
 *     q_k = sum_{a'} softmax(policy_logits[m])[a'] p_k(.|a') renormalised to sum 1; D = KL (SSD_DIV_KL, terms with p = 0
 *     skipped) or the Jensen-Shannon divergence (SSD_DIV_JSD).
 *   influence dev f32[M]: clamp(sum_k influence_per_agent[m][k], -clip, clip); clip >= 0, +inf disables the clamp.
 *   An action outside 0..A-1 anywhere in env b sets influence and influence_per_agent of every agent of b to NaN; pred,
 *   h_out and c_out are still written.
 * Bad arguments return SSD_ERR_INVALID before anything is launched, as do policy handles here and MOA handles at the policy
 * entry points.  fp16 gate GEMM operands; one-hot rows, Dense((N-1)*A) and the influence in fp32. */
typedef struct SsdPolicy* ssd_moa_t;
#define SSD_DIV_KL 0
#define SSD_DIV_JSD 1
int ssd_moa_create(int device, int num_policies, int num_agents, int num_actions, const float* lstm_w, const float* lstm_u, const float* lstm_b,
                   const float* logits_w, const float* logits_b, ssd_moa_t* out);
void ssd_moa_destroy(ssd_moa_t p);
int ssd_moa_step(ssd_moa_t p, const float* features, const int8_t* joint_actions, const float* policy_logits, const float* h_in, const float* c_in,
                 float* h_out, float* c_out, float* pred, float* counterfactual, float* influence_per_agent, float* influence, int64_t num_agents,
                 int divergence, float clip, void* stream);
/* The unfused alternative for other cell sizes: LSTM cell update after the gate GEMM (conv_to_fcnet_v2.py:68-80; Keras gate order i, f, c~, o; sigmoid recurrent
 * activation): gates dev bf16[num_agents][4*units] = x W + h U without the bias, bias dev f32[4*units],
 * c_prev / c_out / h_out dev f32[num_agents][units] (c_out may alias c_prev), h_bf16_out dev bf16[num_agents][units]
 * (the operand of the next step's GEMM).  One pass over HBM; all pointers 16-byte aligned, units a multiple of 8. */
int ssd_policy_lstm_cell(const void* gates_bf16, const float* bias, const float* c_prev, float* c_out, float* h_out, void* h_bf16_out,
                         int64_t num_agents, int units, void* stream);

/* Tuning options.
 * SSD_OPT_CHAIN_STEPS (default 0): when 1, consecutive ssd_step calls on the same stream are launched
 * with programmatic dependent launch: the kernel of step t+1 starts filling SMs while the last CTAs of
 * step t are still running, and every warp waits only for the environments IT steps (a per-warp
 * completion word written by step t).  Results are unchanged.  Precondition: the `actions` of a
 * chained step must already be complete when the previous ssd_step was enqueued (a rollout with
 * pre-generated or scripted actions); work enqueued between two chained steps is NOT waited for.
 * Any other call on the handle (reset, set_state, phases, render, ...) breaks the chain safely.  The library
 * only chains launches of 1.5 to 12 waves of CTAs (about 28K to 230K Harvest envs on a B200): smaller grids
 * have no tail to hide, larger ones amortise it. */
#define SSD_OPT_CHAIN_STEPS 1
#define SSD_OPT_GENERAL_KERNEL 2 /* 1: step everything with the general kernel (tests compare the two kernels) */
int ssd_set_option(ssd_handle h, int option, int64_t value);

/* Running counters since creation (host i64[SSD_NUM_STATS]); synchronises `stream`. */
int ssd_stats(ssd_handle h, int64_t* out_host, void* stream);

/* Number of kernel launches issued by this handle so far (bench.py's gpu_launches). */
int64_t ssd_launch_count(ssd_handle h);

/* Test hook: Philox4x32-10 of one (counter, key) evaluated ON THE DEVICE; out_host u32[4]. */
int ssd_philox_selftest(int device, const uint32_t ctr[4], const uint32_t key[2], uint32_t* out_host);

#ifdef __cplusplus
}
#endif
#endif /* SSD_B200_H */
