/*
 * mpe_b200.h -- C ABI of libmpe_b200.so: batched multi-agent particle worlds on B200 (sm_100a).
 *
 * The reference (openai/multiagent-particle-envs) exposes a *Python* API and no FFI; each entry
 * point below names the reference interface (file:line under /root/reference) whose work it
 * replaces for a batch of n_env independent worlds.  See INTEGRATION.md for the ctypes binding a
 * maintainer of the reference would add.
 *
 * Conventions
 *   - plain pointers and sizes only; no C++/torch types cross this boundary;
 *   - every pointer marked "dev" is a device pointer on the handle's device, borrowed for the
 *     duration of the stream-ordered call; the library allocates nothing per step;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *   - every function returns 0 on success or a negative MPE_ERR_* code; mpe_strerror() names it;
 *   - calls are asynchronous w.r.t. the host; a handle is bound to one device and is not
 *     thread-safe (the reference is single-threaded too: environment.py:80-104).
 *
 * Device state layout (fp32, struct-of-arrays over the world index w in [0, n_env)):
 *   agent_pv  float4 [A][n_env]        (p_pos.x, p_pos.y, p_vel.x, p_vel.y)   core.py:4-9
 *   lm_p      float2 [L][n_env]        landmark p_pos (landmarks never move in any scenario)
 *   comm      float  [S*dim_c][n_env]  state.c of the S non-silent agents     core.py:11-16
 *   goal      int32  [G][n_env]        per-world goal indices (push/adversary/... scenarios)
 * API-facing per-agent tensors are row-major exactly as a trainer holds them:
 *   act_n[i]  float  [n_env][act_dim_i]  (5 physical one-hot/probabilities, then dim_c comm)
 *   obs_n[i]  float  [n_env][obs_dim_i]    (base pointer 16-byte aligned; act_n[i] may be 4-byte aligned,
 *                                           16-byte alignment enables the TMA path)
 *   rew       float  [A][n_env],  done uint8 [A][n_env],  info float [A][info_dim][n_env]
 */
#ifndef MPE_B200_H
#define MPE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define MPE_API __attribute__((visibility("default")))
#else
#define MPE_API
#endif

#define MPE_ABI_VERSION 1
#define MPE_MAX_AGENTS 8
#define MPE_MAX_LANDMARKS 8

/* scenario programs (multiagent/scenarios/<name>.py) */
enum mpe_scenario {
    MPE_SCN_SIMPLE = 0,           /* simple.py */
    MPE_SCN_SPREAD = 1,           /* simple_spread.py (A = L = N) */
    MPE_SCN_TAG = 2,              /* simple_tag.py */
    MPE_SCN_WORLD_COMM = 3,       /* simple_world_comm.py */
    MPE_SCN_ADVERSARY = 4,        /* simple_adversary.py */
    MPE_SCN_PUSH = 5,             /* simple_push.py */
    MPE_SCN_SPEAKER_LISTENER = 6, /* simple_speaker_listener.py */
    MPE_SCN_REFERENCE = 7,        /* simple_reference.py */
    MPE_SCN_CRYPTO = 8,           /* simple_crypto.py */
    MPE_SCN_CUSTOM = 9,           /* user scenario: native _set_action + World.step for ANY entity table (<= 8 agents,
                                     <= 8 landmarks); observation / reward stay in the caller's (GPU) code, so only
                                     mpe_set_action, mpe_world_step and mpe_reset are available */
    MPE_SCN_COUNT_
};

/* error codes */
enum mpe_error {
    MPE_OK = 0,
    MPE_ERR_BAD_ARG = -1,         /* null/misaligned pointer, n_env <= 0, bad agent index */
    MPE_ERR_BAD_DESC = -2,        /* descriptor inconsistent with its scenario program */
    MPE_ERR_UNSUPPORTED = -3,     /* no compiled kernel for this scenario/shape */
    MPE_ERR_CUDA = -4,            /* CUDA runtime error; see mpe_last_cuda_error() */
    MPE_ERR_NO_DEVICE = -5        /* no sm_100 device / device index out of range */
};

/* step flags (MultiAgentEnv attributes, environment.py:29-35) */
enum mpe_step_flags {
    MPE_FLAG_SHARED_REWARD = 1,         /* env.shared_reward: every agent gets sum_i r_i   :100-102 */
    MPE_FLAG_FORCE_DISCRETE_ACTION = 2, /* env.force_discrete_action: argmax one-hot       :169-172 */
    MPE_FLAG_DISCRETE_ACTION_INPUT = 4, /* env.discrete_action_input (:161-167,185-187): act_n[i] is int32
                                           [n_env][n_sub_i], one index per sub-action -- movement (0 none, 1 -x,
                                           2 +x, 3 -y, 4 +y) if the agent is movable, then the utterance
                                           (one-hot of the index) if it is not silent; decoded inside the kernel */
    MPE_FLAG_HOST_SLAB = 8,             /* mpe_step_host only: obs_n_host[0..A), rew_host, done_host (, info_host)
                                           are consecutive parts of ONE host allocation and their device
                                           counterparts of ONE device allocation, with equal gaps < 512 B:
                                           the D2H copies are coalesced into a single DMA */
    MPE_FLAG_SAMPLE_ACTIONS = 16        /* mpe_collect only: act with MADDPG's Gumbel-softmax exploration sample */
};

/*
 * Immutable world descriptor: what Scenario.make_world() writes onto World / Entity objects
 * (core.py:25-99 defaults; e.g. simple_spread.py:7-29), flattened.  Doubles keep the Python
 * values exact; the library rounds derived constants to fp32 once at create time.
 */
typedef struct mpe_desc {
    int32_t abi_version;                       /* MPE_ABI_VERSION */
    int32_t scenario;                          /* enum mpe_scenario */
    int32_t n_agents;                          /* len(world.agents) == len(world.policy_agents) */
    int32_t n_landmarks;                       /* len(world.landmarks) */
    int32_t dim_c;                             /* world.dim_c                       core.py:88 */
    int32_t n_adversaries;                     /* agents [0, n_adv) have .adversary (tag/world_comm/adversary/push) */
    int32_t n_obstacles;                       /* world_comm: landmarks = obstacles ++ food ++ forests */
    int32_t n_food;
    int32_t n_forests;
    int32_t reserved_i[7];
    double dt;                                 /* core.py:94  */
    double damping;                            /* core.py:96  */
    double contact_force;                      /* core.py:98  */
    double contact_margin;                     /* core.py:99  */
    double agent_size[MPE_MAX_AGENTS];         /* core.py:32  */
    double agent_mass[MPE_MAX_AGENTS];         /* core.py:47-51 */
    double agent_sens[MPE_MAX_AGENTS];         /* accel or 5.0: environment.py:178-181 */
    double agent_max_speed[MPE_MAX_AGENTS];    /* < 0 means None: core.py:41,164 */
    double landmark_size[MPE_MAX_LANDMARKS];
    uint8_t agent_movable[MPE_MAX_AGENTS];     /* core.py:58  */
    uint8_t agent_collide[MPE_MAX_AGENTS];     /* core.py:36  */
    uint8_t agent_silent[MPE_MAX_AGENTS];      /* core.py:60  */
    uint8_t agent_adversary[MPE_MAX_AGENTS];
    uint8_t agent_leader[MPE_MAX_AGENTS];      /* simple_world_comm.py:23 */
    uint8_t landmark_collide[MPE_MAX_LANDMARKS];
    uint8_t reserved_b[16];
} mpe_desc;

typedef struct mpe_env *mpe_handle;

/* ---- lifetime -------------------------------------------------------------------------- */

/* Validates the descriptor against its scenario program and binds a batch of n_env worlds to a
 * device.  Replaces: World() + Scenario.make_world() + MultiAgentEnv.__init__ shape discovery
 * (make_env.py:36-43, environment.py:14-78). */
MPE_API int mpe_create(const mpe_desc *desc, int64_t n_env, int device, mpe_handle *out);
MPE_API int mpe_destroy(mpe_handle h);

/* ---- shape queries (environment.py:39-70: action_space / observation_space construction) -- */
MPE_API int mpe_num_agents(mpe_handle h);
MPE_API int64_t mpe_num_envs(mpe_handle h);
MPE_API int mpe_obs_dim(mpe_handle h, int agent);     /* len(scenario.observation(agent, world)) :68 */
MPE_API int mpe_act_dim(mpe_handle h, int agent);     /* 5 if movable (+ dim_c if not silent)    :45-63 */
MPE_API int mpe_num_speakers(mpe_handle h);           /* S: agents with silent == False */
MPE_API int mpe_num_goals(mpe_handle h);              /* G: rows of the goal tensor */
MPE_API int mpe_info_dim(mpe_handle h);               /* floats of benchmark_data per agent */
MPE_API int64_t mpe_bytes_per_env_step(mpe_handle h); /* compulsory HBM bytes of one fused step (SURVEY 8d) */

/* ---- reset (scenario.reset_world: e.g. simple_spread.py:31-45; environment.py:106-116) ---- */
/* Worlds with mask[w] != 0 (all if mask == NULL) get i.i.d. uniform positions from a Philox4x32
 * stream keyed by (seed, world_offset + w, epoch): results do not depend on how the batch is
 * sharded.  Velocities, comm state are zeroed; goal indices redrawn. */
MPE_API int mpe_reset(mpe_handle h, void *agent_pv_dev, void *lm_p_dev, float *comm_dev, int32_t *goal_dev,
              const uint8_t *mask_dev, uint64_t seed, uint64_t world_offset, uint64_t epoch,
              void *stream);

/* Same reset, but the epoch is read from device memory (*epoch_dev) and incremented afterwards on the stream:
 * a reset captured in a CUDA graph then draws fresh initial conditions on every replay. */
MPE_API int mpe_reset_dev_epoch(mpe_handle h, void *agent_pv_dev, void *lm_p_dev, float *comm_dev, int32_t *goal_dev,
                                const uint8_t *mask_dev, uint64_t seed, uint64_t world_offset,
                                unsigned long long *epoch_dev, void *stream);

/* ---- the hot path ------------------------------------------------------------------------ */

/* MultiAgentEnv._set_action for all agents (environment.py:144-192): act_n -> action.u, action.c.
 * u: float2 [A][n_env]; c: float [S*dim_c][n_env]. */
MPE_API int mpe_set_action(mpe_handle h, const float *const *act_n_dev, float *u_dev, float *c_dev,
                   uint32_t flags, void *stream);

/* World.step (core.py:117-131): apply_action_force, apply_environment_force /
 * get_collision_force, integrate_state, update_agent_state -- from already decoded actions. */
MPE_API int mpe_world_step(mpe_handle h, void *agent_pv_dev, const void *lm_p_dev, float *comm_dev,
                   const float *u_dev, const float *c_dev, void *stream);

/* scenario.observation / reward / benchmark_data for every agent plus the done/shared-reward
 * glue of MultiAgentEnv.step (environment.py:92-102,119-141) on the current state.
 * info_dev may be NULL. */
MPE_API int mpe_observe(mpe_handle h, const void *agent_pv_dev, const void *lm_p_dev, const float *comm_dev,
                const int32_t *goal_dev, float *const *obs_n_dev, float *rew_dev, uint8_t *done_dev,
                float *info_dev, uint32_t flags, void *stream);

/* MultiAgentEnv.step (environment.py:80-104) fused into one launch:
 * _set_action -> World.step -> observation/reward/done/info -> shared-reward sum. */
MPE_API int mpe_step(mpe_handle h, void *agent_pv_dev, const void *lm_p_dev, float *comm_dev,
             const int32_t *goal_dev, const float *const *act_n_dev, float *const *obs_n_dev,
             float *rew_dev, uint8_t *done_dev, float *info_dev, uint32_t flags, void *stream);

/* n_steps consecutive MultiAgentEnv.step calls (environment.py:80-104; the loop of bin/interactive.py:27-39 with the
 * policy's outputs known in advance) on pre-generated actions, in ONE launch: act_seq_dev[i] is float
 * [n_steps][n_env][act_dim_i].  A world's state stays in registers between the steps; per step only the actions are read.
 * Outputs: the state after the last step, obs_n_dev / done_dev for that final state, rew_sum_dev [A][n_env] = the
 * per-agent rewards summed over the steps in step order, and -- if rew_steps_dev is not NULL -- every step's rewards
 * [n_steps][A][n_env].  Bit-identical to n_steps calls of mpe_step.  (CEM / MPPI style planners, evaluation of
 * recorded action sequences.)  MPE_FLAG_DISCRETE_ACTION_INPUT is not supported here. */
MPE_API int mpe_rollout(mpe_handle h, void *agent_pv_dev, const void *lm_p_dev, float *comm_dev,
                        const int32_t *goal_dev, const float *const *act_seq_dev, int32_t n_steps,
                        float *const *obs_n_dev, float *rew_sum_dev, float *rew_steps_dev, uint8_t *done_dev,
                        uint32_t flags, void *stream);

/* n_steps consecutive MultiAgentEnv.step calls in ONE launch with the policy INSIDE the kernel (the trainer's loop
 * obs -> actor network -> env.step, bin/interactive.py:27-39 with `policy.action(obs_n[i])` being a small actor): agent i
 * acts with  a_i = softmax(W2_i . relu(W1_i^T . obs_i + b1_i) + b2_i),  obs_dim_i -> hidden -> 5 movement probabilities.
 * w1_n[i]: float [obs_dim_i][hidden] (input-major, 16-byte aligned), b1_n[i]: [hidden], w2_n[i]: [5][hidden], b2_n[i]: [5];
 * hidden = 32 or 64.  World state stays in registers, observations are never written between steps.  Outputs as
 * mpe_rollout; act_record_n (NULL or per agent float [n_steps][n_env][5]) receives the actions taken -- feeding them to
 * mpe_rollout / mpe_step reproduces state, observations and reward sums bit for bit.  Only for scenarios whose agents
 * all move and are silent and for which the program was built (simple, simple_spread N = 3, simple_tag 3 + 1,
 * simple_adversary 1 + 2, simple_push); otherwise, speaking or immovable agents included, MPE_ERR_UNSUPPORTED. */
MPE_API int mpe_rollout_policy(mpe_handle h, void *agent_pv_dev, const void *lm_p_dev, float *comm_dev,
                               const int32_t *goal_dev, const float *const *w1_n, const float *const *b1_n,
                               const float *const *w2_n, const float *const *b2_n, int32_t hidden, int32_t n_steps,
                               float *const *obs_n_dev, float *rew_sum_dev, float *rew_steps_dev,
                               float *const *act_record_n, uint8_t *done_dev, uint32_t flags, void *stream);

/* Training experience in ONE launch: the closed loop of mpe_rollout_policy, with a one- or two-hidden-layer actor,
 * optional exploration noise and a record of every step's observations -- everything a replay buffer needs:
 * (obs_record[t], act_record[t], rew_steps[t], obs_record[t + 1]), with obs_n_dev holding the observation after the
 * last step.  Agent i's actor has act_dim_i = mpe_act_dim(h, i) outputs:
 *   depth 1:  logits_i = W2_i . relu(W1_i^T . obs_i + b1_i) + b2_i                          (obs_dim_i -> H -> act_dim_i)
 *   depth 2:  logits_i = W3_i . relu(W2_i . relu(W1_i^T . obs_i + b1_i) + b2_i) + b3_i      (obs_dim_i -> H -> H ->
 *             act_dim_i, the MADDPG actor: fc 64 relu, fc 64 relu, fc act_dim_i)
 * The logits are the heads of the reference's action space (environment.py:58-64): 5 movement logits if the agent
 * moves, then dim_c communication logits if it speaks.  Each head gets its own max-subtracted softmax; the action is
 * [softmax(movement) | softmax(comm)], the comm head's probabilities becoming the agent's utterance (action.c) once
 * every agent has acted on the current state, as in mpe_step.
 * hidden = H = 32 or 64.  Weights, all 16-byte aligned except b2 / b3 (4-byte):
 *   w1_n[i] float [obs_dim_i][H] (input-major, W1^T of a torch Linear(obs_dim_i, H)), b1_n[i] [H];
 *   depth 1: w2_n[i] [act_dim_i][H], b2_n[i] [act_dim_i], w3_n = b3_n = NULL;
 *   depth 2: w2_n[i] [H][H] (torch Linear(H, H).weight), b2_n[i] [H], w3_n[i] [act_dim_i][H], b3_n[i] [act_dim_i].
 * Every unit sums bias + inputs in ascending input order with FMAs.  comm_dev (the speakers' utterances) is read
 * before the first step and written after the last; it is required when the scenario has speakers.
 * flags: MPE_FLAG_SHARED_REWARD as for mpe_step; MPE_FLAG_SAMPLE_ACTIONS replaces each head's softmax(logits) by the
 * exploration sample softmax(logits - log(-log u)), u = (2 (bits >> 9) + 1) 2^-24 from Philox4x32-10 with key
 * (sample_seed lo, hi) and counter (w lo, w hi, sample_step + t, tag), w = world_offset + world index:
 *   movement logit c < 5: tag 0x40000000 | agent << 1 | block, blocks 0 and 1 giving words 0-3 and 4;
 *   comm logit q < dim_c: word q & 3 of block q >> 2 with tag 0x40000100 | agent << 2 | block.
 * These counters are disjoint from each other and from mpe_reset's (small block numbers, 0x80000000 in word 3).  Draws
 * depend on the global world index and the global step only, so a sharded batch or a rollout split into several calls
 * draws exactly what one call over the whole batch draws.
 * Records (NULL, or per agent): act_record_n[i] float [n_steps][n_env][act_dim_i], the actions taken (sampled ones when
 * sampling); obs_record_n[i] float [n_steps][n_env][obs_dim_i] (16-byte aligned, all agents or none), row t = the
 * observation agent i acted on at step t (row 0 = the state before the call).  Feeding act_record_n to mpe_step
 * reproduces state, utterances, observations and rewards bit for bit.  Outputs otherwise as mpe_rollout_policy.
 * For scenarios whose agents all move and are silent nothing differs from a 5-wide actor.
 * Errors: MPE_ERR_BAD_ARG for NULL / misaligned pointers, depth not 1 or 2, hidden not 32 or 64, n_steps < 0 or
 * sample_step + n_steps > 2^32; MPE_ERR_NO_DEVICE for a device-less handle; MPE_ERR_UNSUPPORTED for a scenario
 * without the kernel (mpe_collect_supported) or MPE_FLAG_FORCE_DISCRETE_ACTION / MPE_FLAG_DISCRETE_ACTION_INPUT. */
MPE_API int mpe_collect(mpe_handle h, void *agent_pv_dev, const void *lm_p_dev, float *comm_dev, const int32_t *goal_dev,
                        int32_t depth, int32_t hidden,
                        const float *const *w1_n, const float *const *b1_n,
                        const float *const *w2_n, const float *const *b2_n,
                        const float *const *w3_n, const float *const *b3_n,
                        int32_t n_steps, uint64_t sample_seed, uint32_t sample_step, uint64_t world_offset,
                        float *const *obs_n_dev, float *rew_sum_dev, float *rew_steps_dev,
                        float *const *act_record_n, float *const *obs_record_n, uint8_t *done_dev,
                        uint32_t flags, void *stream);

/* Is mpe_collect built for this handle's scenario at this depth and hidden width?  MPE_OK; MPE_ERR_UNSUPPORTED (built
 * for simple, simple_spread N = 3, simple_tag 3 + 1, simple_adversary 1 + 2, simple_push, simple_speaker_listener,
 * simple_reference and simple_crypto; not for user scenarios or other entity counts); MPE_ERR_BAD_ARG for a NULL handle,
 * depth not 1 or 2 or hidden not 32 or 64.  Needs no device: answers for shape-only handles as well. */
MPE_API int mpe_collect_supported(mpe_handle h, int32_t depth, int32_t hidden);

/* Same step for a caller that holds HOST buffers (what the reference's callers hold):
 * act_n_host[i] -> (async H2D into act_n_dev[i]) -> mpe_step -> (async D2H) obs_n_host[i],
 * rew_host, done_host, all ordered on `stream`.  Host buffers should be pinned for the copies
 * to be asynchronous.  The caller synchronises the stream before reading the outputs.
 * Large batches are cut into MPE_B200_HOST_CHUNKS (default 4) world ranges that alternate
 * between two library-owned streams forked from / joined to `stream`, so that the upload + step of one range
 * overlaps the download of the previous one (full-duplex PCIe).  Pipelining starts at MPE_B200_HOST_CHUNK_MIN worlds (default 262144: below that the
 * extra copy calls cost more than the overlap gains on PCIe Gen5). */
MPE_API int mpe_step_host(mpe_handle h, void *agent_pv_dev, const void *lm_p_dev, float *comm_dev,
                  const int32_t *goal_dev, const float *const *act_n_host, float *const *act_n_dev,
                  float *const *obs_n_dev, float *rew_dev, uint8_t *done_dev, float *info_dev,
                  float *const *obs_n_host, float *rew_host, uint8_t *done_host, float *info_host,
                  uint32_t flags, void *stream);

/* ---- diagnostics --------------------------------------------------------------------------- */
MPE_API const char *mpe_strerror(int err);
MPE_API const char *mpe_last_cuda_error(void);  /* text of the last CUDA failure on this thread */
MPE_API int mpe_abi_version(void);
MPE_API int64_t mpe_kernel_launches(void);      /* kernels launched by this library so far (process-wide) */
/* Measurement aid (bench.py "size-matched streaming ceiling"): one launch of a pure streaming kernel that reads
 * read_bytes from src_dev and then writes write_bytes to dst_dev (both 16-byte aligned) with `threads` threads,
 * through the same launch path as mpe_step.  Not counted by mpe_kernel_launches; computes nothing. */
MPE_API int mpe_probe_stream(int device, const void *src_dev, int64_t read_bytes, void *dst_dev, int64_t write_bytes,
                             int64_t threads, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* MPE_B200_H */
