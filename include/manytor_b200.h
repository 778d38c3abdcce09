/*
 * manytor_b200 -- C ABI of the B200-native batched ManyTor step loop.
 *
 * This header is the drop-in boundary for the hot path of victorkich/ManyTor
 * (Environment.step / reset and the Multienv loop).  The reference has no FFI
 * of its own: its boundary is the Python surface of manytor.py, so every entry
 * point below names the reference method (file:line under /root/reference) it
 * replaces, vectorised over N lock-step environments.
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / C++ types.
 *   - "_dev" pointers are device pointers on the handle's device, 16-byte
 *     aligned; "_host" pointers are host memory (pinned where the call is
 *     asynchronous).  `stream` is a cudaStream_t passed as void* (NULL = the
 *     legacy default stream).  Calls are asynchronous on that stream unless
 *     documented as synchronous.
 *   - every call returns MT_OK (0) or a negative mt_status; mt_last_error()
 *     returns a per-thread message for the last failure.
 *   - one handle = one shard of environments on one device; handles are not
 *     thread-safe.
 *   - angles are DEGREES, actions are absolute joint targets (manytor.py:182-184).
 *
 * Array layouts (row-major, fp32 unless noted)
 *   actions [N][J]        obs [N][3*X]  (per objective: distance, r, theta;
 *   reward  [N]                          zeros for a dead objective, manytor.py:141-153),
 *                         elements of the handle's format: fp32, or binary16 when
 *                         mt_config.obs_dtype = MT_OBS_F16 (6*X bytes per row)
 *   done    [N] uint8     bit0 = terminated (no objective alive, manytor.py:170-171,
 *                                  or ground contact when terminate_on_ground)
 *                         bit1 = truncated (episode reached cfg.horizon steps)
 *   points  [N][X][3]     goals [N][J]     alive [N] uint32 bitmask (bit p = objective p)
 *   joints  [N][J][3]     the reference's joints_coordinates: rows = base, frame 2 .. frame J
 */
#ifndef MANYTOR_B200_H
#define MANYTOR_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MT_ABI_VERSION 3
#define MT_MAX_JOINTS 8
#define MT_MAX_OBJ 32

/* mt_config.obs_dtype: the element type of every observation a handle writes */
#define MT_OBS_F32 0   /* float                                                         */
#define MT_OBS_F16 1   /* IEEE binary16, rounded to nearest even from the fp32 result   */

typedef enum mt_status {
    MT_OK = 0,
    MT_ERR_INVALID = -1,   /* bad argument / configuration                     */
    MT_ERR_CUDA = -2,      /* a CUDA runtime call failed (message has details) */
    MT_ERR_NO_DEVICE = -3, /* no usable sm_100 device: there is NO CPU fallback */
    MT_ERR_STATE = -4      /* call not valid in the handle's current state     */
} mt_status;

typedef struct mt_env mt_env; /* opaque handle */

/* Everything the reference hard-codes (SURVEY.md section 5, "Config / flags"). */
typedef struct mt_config {
    uint32_t struct_size;          /* = sizeof(mt_config), checked by mt_create          */
    int32_t device;                /* CUDA device ordinal                                 */
    int64_t n_envs;                /* N: environments in this shard                       */
    int64_t env_id_base;           /* global id of env 0 (keys the RNG: shard-invariant)  */
    int32_t n_joints;              /* J, 2..MT_MAX_JOINTS (reference: 4)                  */
    int32_t n_obj;                 /* X, 1..MT_MAX_OBJ (Environment(obj_number), :130)    */
    float dh[MT_MAX_JOINTS][4];    /* rows (a, alpha, d, theta_offset), radians (:42-48)  */
    int32_t obs_frame;             /* frame anchoring observations (reference: 3, :143)   */
    int32_t ground_frame_a;        /* frames whose z<0 is ground contact (3 and 4, :191)  */
    int32_t ground_frame_b;
    int32_t catch_frame;           /* frame that catches objectives (4, :162)             */
    float radius;                  /* objective half-ball radius (51.3, :231,236)         */
    float catch_tol;               /* per-axis inclusive tolerance (8.0, :162)            */
    int32_t substeps;              /* interpolated poses per step (25, :178)              */
    int32_t horizon;               /* max steps per episode, 0 = none (max_steps in the
                                      reference's driver scripts, test_single.py:6), at most
                                      65535.  The per-env episode-length counter saturates: at
                                      65535 when n_obj <= 16 or horizon = 0, else at
                                      2^(32 - n_obj) - 1 when the horizon fits below that (the
                                      counter then shares a word with the alive mask), else 65535 */
    int32_t terminate_on_ground;   /* 0 = reference code (reward -1 only), 1 = README     */
    int32_t auto_reset;            /* 1: envs that end are reset inside the step kernel   */
    int32_t obs_after_reset;       /* with auto_reset: 0 = emit obs2 of the ending step,
                                      1 = emit the first observation of the new episode   */
    int32_t fk_mode;               /* 0 auto (closed form / preset / NVRTC-specialised / run-time
                                      table, in that order), 1 run-time DH table, 2 closed form
                                      required, 3 NVRTC specialisation required              */
    int32_t action_low;            /* action_sample range [low, high) (-180, 180, :216)   */
    int32_t action_high;
    uint64_t seed;                 /* Philox key for on-device actions / objectives       */
    int32_t obs_dtype;             /* MT_OBS_F32 (default) or MT_OBS_F16: the format of the
                                      obs buffers of mt_step, mt_observe, mt_rollout_random,
                                      mt_rollout and mt_step_host (the values are the fp32
                                      ones rounded) */
} mt_config;

/* Episode statistics; summed over the shard, reducible across shards by plain
 * addition (the one collective of a multi-GPU rollout). */
typedef struct mt_stats {
    int64_t env_steps;       /* env-steps executed since create / stats reset            */
    int64_t episodes;        /* episodes finished (terminated or truncated)              */
    int64_t terminated;      /* ... of which all objectives were collected               */
    int64_t reward_sum;      /* sum of total_reward over finished episodes               */
    int64_t length_sum;      /* sum of episode lengths over finished episodes            */
    int64_t catches;         /* objectives collected in finished episodes                */
    int64_t ground_steps;    /* env-steps with ground contact (every executed step)      */
    int64_t live_reward_sum; /* sum of total_reward over episodes still in progress      */
} mt_stats;
#define MT_STATS_WORDS 8

int mt_abi_version(void);
const char *mt_last_error(void);

/* Fill cfg with the reference arm and constants (manytor.py:42-48,162,178,216,231). */
int mt_config_init(mt_config *cfg);

/* Environment(obj_number) / Multienv(env_shape, obj_number) -- manytor.py:77-82,130-139.
 * Allocates the structure-of-arrays state in HBM.  Envs start un-reset, as in the
 * reference; call mt_reset before mt_step. */
int mt_create(const mt_config *cfg, mt_env **out);
int mt_destroy(mt_env *env);
int mt_get_config(const mt_env *env, mt_config *out);
/* Re-seed the on-device Philox streams (actions, objective refresh): new key AND the counters that
 * index the streams (per-env reset count of mt_get_reset_counts, step index) back to zero, so
 * reset(seed=s) reproduces the same objectives and actions every time it is called with the same s
 * (Gymnasium's reset(seed=...) contract).  Synchronous (waits for the device). */
int mt_set_seed(mt_env *env, uint64_t seed);

/* The step index that keys the action stream of mt_sample_actions / mt_rollout_random.  It lives in
 * DEVICE memory and is advanced by the step kernel itself (the last block of every mt_step,
 * mt_step_host and of each step of mt_rollout_random), as are mt_stats.env_steps and the other
 * statistics.  Consequence for CUDA graphs: a captured mt_step / mt_rollout_random can be replayed
 * any number of times -- every replay counts its env-steps and draws fresh actions, exactly like the
 * same calls issued eagerly.  Get/set are synchronous 8-byte copies on the legacy default stream
 * (checkpoint / resume, with the state listed at mt_set_points), ordered after everything submitted
 * earlier to it / blocking streams (work on cudaStreamNonBlocking streams must be synchronised by the
 * caller); the set has landed on return.
 * The index lies in [0, MT_STEP_INDEX_MAX]; mt_set_step_index returns MT_ERR_INVALID above it and leaves
 * the index as it was.  The bound exists because the kernels' launch bookkeeping needs bit 63 of the index
 * to be clear: each warp orders its launch ticket after its read of the index through that bit.  At most
 * 4096 steps pass per launch, so climbing from 2^62 to 2^63 would take more than 10^15 launches. */
#define MT_STEP_INDEX_MAX 0x4000000000000000ull /* 2^62 */
int mt_get_step_index(mt_env *env, uint64_t *out);
int mt_set_step_index(mt_env *env, uint64_t value);

/* Environment.reset / Multienv.reset -- manytor.py:219-253, 106-109.
 * mask_dev: NULL = all envs, else [N] uint8 selecting the envs to reset.  The FIRST reset of a handle
 * must cover every env (NULL or an all-ones mask; a partial first mask returns MT_ERR_STATE after one
 * small synchronous check): the reference raises IndexError when a never-reset env is stepped.
 * Fresh objectives come from the objective stream if one is set, else from the
 * on-device half-ball sampler (uniform in {|p|<=radius, z>=0}). */
int mt_reset(mt_env *env, const uint8_t *mask_dev, void *stream);

/* Environment.get_observations -- manytor.py:141-153: current obs of every env. */
int mt_observe(mt_env *env, void *obs_dev, void *stream);

/* Environment.step / Multienv.step -- manytor.py:255-260, 115-122: ONE fused kernel
 * (FK over the 25 sub-poses, ground flag, obs2, catch, reward, done, auto-reset).
 * joints_dev may be NULL. */
int mt_step(mt_env *env, const float *actions_dev, void *obs_dev, float *reward_dev,
            uint8_t *done_dev, float *joints_dev, void *stream);

/* mt_step plus what an episode that ends in this step leaves behind, which the in-kernel auto-reset
 * otherwise wipes (Gymnasium's info["final_obs"] and the per-episode return / length of
 * RecordEpisodeStatistics; V(final_obs) bootstraps a truncated episode):
 *   final_obs_dev    [N][3X]  obs2 of the ending step (manytor.py:204), in the handle's obs format, bit for bit
 *                             what mt_step returns for that env with obs_after_reset = 0
 *   final_return_dev [N] fp32 total reward of the episode
 *   final_length_dev [N] i32  its length: the episode-length counter, which saturates as
 *                             mt_config.horizon documents
 * Row n of each final array is written exactly when done[n] != 0; the other rows keep their contents.
 * Everything else (obs, reward, done, joints, state, statistics, step index) is what mt_step computes.
 * obs_dev and the three final pointers are required and 16-byte aligned; argument errors are reported
 * before the handle is looked at.  A handle created without auto_reset returns MT_ERR_INVALID (without
 * auto-reset nothing is lost: obs2 is the returned obs and mt_get_state holds the return and length);
 * a call before the first mt_reset returns MT_ERR_STATE. */
int mt_step_final(mt_env *env, const float *actions_dev, void *obs_dev, float *reward_dev, uint8_t *done_dev,
                  float *joints_dev, void *final_obs_dev, float *final_return_dev, int32_t *final_length_dev,
                  void *stream);

/* Environment.action_sample / Multienv.action_sample -- manytor.py:215-217, 111-113:
 * integer degrees uniform on [action_low, action_high), Philox keyed by
 * (seed, global env id, step index). */
int mt_sample_actions(mt_env *env, float *actions_dev, void *stream);

/* n_steps x step(action_sample()) with the actions drawn inside the kernel (same stream
 * of actions as mt_sample_actions).  obs_dev/reward_dev/done_dev are overwritten every
 * step; obs_dev may be NULL to skip the observation write; reward_dev / done_dev may be
 * NULL, the results then go to buffers the handle owns (a host without CUDA headers can
 * drive a rollout and read only the statistics).
 * For n_steps >= 2 this is ONE launch per 4096 steps of the multi-step rollout kernel:
 * every tile of 32 envs keeps its pose / alive word / total reward in registers and its
 * objectives in shared memory for all the steps, and only what a step produces
 * (observations, reward, done) leaves the SM each step.  Results are bit-identical to
 * n_steps launches of the step kernel, which run-time DH tables without NVRTC still
 * take (MT_ROLLOUT_PERSISTENT=0 forces them for everyone). */
int mt_rollout_random(mt_env *env, int32_t n_steps, void *obs_dev, float *reward_dev,
                      uint8_t *done_dev, void *stream);

/* n_steps x step() in one call, keeping EVERY step (a trajectory).  Slice s of each array holds exactly
 * what the s-th of n_steps consecutive mt_step calls would have written, bit for bit.
 *   actions_dev [n_steps][N][J]  the caller's actions; step s reads actions_dev + s*N*J.
 *                                NULL = drawn in-kernel: the stream of mt_rollout_random / mt_sample_actions
 *                                (Philox keyed by seed, env id, step index + s)
 *   drawn_dev   [n_steps][N][J]  receives the drawn actions when actions_dev is NULL; may be NULL;
 *                                must be NULL when actions_dev is given
 *   obs_dev     [n_steps][N][3X] in the handle's obs format, or NULL (no observations written)
 *   reward_dev  [n_steps][N] fp32, done_dev [n_steps][N] u8: required
 * Slices are packed (a stride of exactly N rows); every base pointer is 16-byte aligned.  n_steps < 0 is
 * MT_ERR_INVALID, n_steps = 0 does nothing, a call before the first mt_reset is MT_ERR_STATE.
 * The step index, env-step count and statistics advance exactly as for n_steps mt_step calls.
 * Like mt_rollout_random this is one launch of the multi-step rollout kernel per 4096 steps (state in
 * registers, objectives in shared memory), and n_steps launches of the step kernel for run-time DH
 * tables without NVRTC or under MT_ROLLOUT_PERSISTENT=0.  The caller's actions are read once each, so
 * an open-loop planner or a replay of logged actions moves 4J bytes of actions per env-step instead of
 * the full state round trip of one mt_step per step. */
int mt_rollout(mt_env *env, int32_t n_steps, const float *actions_dev, float *drawn_dev, void *obs_dev,
               float *reward_dev, uint8_t *done_dev, void *stream);

/* mt_rollout plus, for every step, what mt_step_final adds to mt_step: the final observation, return and
 * length of each episode that ends inside the trajectory, which the in-kernel auto-reset otherwise wipes.
 *   actions_dev, drawn_dev, reward_dev, done_dev  exactly as in mt_rollout
 *   obs_dev            [n_steps][N][3X] required (the final observation is the step's obs2)
 *   final_obs_dev      [n_steps][N][3X] in the handle's obs format
 *   final_return_dev   [n_steps][N] fp32
 *   final_length_dev   [n_steps][N] i32
 * Slice s of every output, the final arrays included, is bit for bit what the s-th of n_steps consecutive
 * mt_step_final calls writes (with the caller's actions, or the draws mt_rollout makes).  Row n of final
 * slice s is written exactly when done[s][n] != 0; every other row keeps its contents.  Every pointer
 * but drawn_dev is required, and all are 16-byte aligned.  Argument errors are reported before the
 * handle is looked at, in mt_rollout's order and then mt_step_final's.  A handle without auto_reset
 * returns MT_ERR_INVALID, a call before the first mt_reset MT_ERR_STATE; n_steps < 0 is MT_ERR_INVALID,
 * n_steps = 0 does nothing.  One launch of the multi-step rollout kernel per 4096 steps, as mt_rollout;
 * where mt_rollout takes one step-kernel launch per step, in-kernel draws here take two (the draw, as
 * mt_sample_actions makes it, then the step with those actions).  The final rows cost 12X + 8 bytes per
 * ending episode and nothing for the envs that go on. */
int mt_rollout_final(mt_env *env, int32_t n_steps, const float *actions_dev, float *drawn_dev, void *obs_dev,
                     float *reward_dev, uint8_t *done_dev, void *final_obs_dev, float *final_return_dev,
                     int32_t *final_length_dev, void *stream);

/* Score action sequences from copies of chosen envs in one launch, leaving the handle untouched -- what an
 * open-loop planner (random shooting, CEM, MPPI, MPC with a terminal value) asks many times per decision.
 *   src_dev     [M] int64: branch m starts from the current state of env src[m]: its goals, alive word, episode
 *                          length and raw objectives (dead ones included).  Sources may repeat, in any order; M may
 *                          be smaller or larger than N.
 *   actions_dev [n_steps][M][J] fp32 degrees: step s of branch m reads actions_dev + (s*M + m)*J (mt_rollout's layout)
 * Every step is computed as mt_step computes it for an env in that state with those actions (reward, catches,
 * ground test, terminate_on_ground, truncation at the handle's horizon counted from the source's episode length).
 * A branch ends at the first step whose done byte is non-zero, that step included; nothing resets inside a branch.
 * Outputs, one row per branch:
 *   return_dev  [M] fp32: the discounted return up to and including the ending step, in this fp32 order:
 *               d_0 = 1, d_{s+1} = fl(d_s * gamma), G_{s+1} = fl(G_s + d_s * r_s) (d_s * r_s is exact: r_s is -1, 0, +1)
 *   length_dev  [M] i32: the steps the branch executed, T in [1, n_steps] when it ended at step T-1, else n_steps
 *   done_dev    [M] u8: the done byte of the ending step (bit0 terminated, bit1 truncated), 0 if it ran all steps
 *   obs_dev     [M][3X] in the handle's obs format, or NULL (not written): the observation mt_step returns at the
 *               branch's last executed step with obs_after_reset = 0 (obs2; where the branch ended, what
 *               mt_step_final writes as the final observation)
 * A branch whose source is outside [0, N) reads nothing of any env: it gets return NaN, length -1, done 0, and its
 * obs row is not written.  The handle is not changed: goals, alive words, episode lengths, total rewards, objectives,
 * reset counts, step index and statistics stay as they were; auto_reset and the objective stream play no part.
 * Only mt_launch_count moves.  Every pointer but obs_dev is required, and all are 16-byte aligned.  Argument errors
 * are reported before the handle is looked at: n_steps outside [0, 4096], n_branches outside [0, 2e9] and gamma
 * not in [0, 1] (NaN included) are MT_ERR_INVALID.  A call before the first mt_reset is MT_ERR_STATE; n_steps = 0
 * or n_branches = 0 then does nothing.  ONE launch: a branch's state stays in registers and its objectives in shared
 * memory for all the steps, so a branch-step moves its 4J bytes of actions plus (state + 12X + outputs) / n_steps.
 * Every arm runs it: the built-in ones at X = 10, 20 and any X, and any other DH table through the run-time-table
 * kernel.  For a handle whose steps NVRTC specialises to its table, branches are therefore bit for bit the step of the
 * same table with fk_mode = 1; the specialised kernel folds the table's zeros and orders two multiply-adds differently,
 * so positions, and with them observations, can differ in the last bits from that handle's own mt_step. */
int mt_rollout_branches(mt_env *env, int32_t n_steps, int64_t n_branches, const int64_t *src_dev,
                        const float *actions_dev, float gamma, float *return_dev, int32_t *length_dev,
                        uint8_t *done_dev, void *obs_dev, void *stream);

/* mt_rollout_branches with the actions of steps n_prefix .. n_steps-1 drawn in the kernel from the environment's own
 * random policy (mt_sample_actions: integer degrees uniform on [action_low, action_high)) -- random shooting,
 * Monte-Carlo state values, rollout-based Q estimates -- in O(M) memory instead of O(n_steps M).
 *   prefix_dev   [n_prefix][M][J] fp32 degrees, mt_rollout_branches' layout: the actions of steps s < n_prefix.  Required
 *                when n_prefix > 0, and NULL when n_prefix = 0; 0 <= n_prefix <= n_steps <= 4096.
 *   draw_key_dev one uint64 on the device, read by the kernel (so a CUDA graph that captures this call and an increment
 *                of the key draws fresh actions at every replay); required, 8-byte aligned.
 * Draw contract: step s >= n_prefix of branch m (s counted from the start of the branch) takes exactly what
 * mt_sample_actions draws for GLOBAL ENV ID m at STEP INDEX key + s (mod 2^64), with the handle's current seed (after
 * any mt_set_seed), action range and J.  So a branch's draws depend on (seed, m, key) only: not on src, on M, on
 * env_id_base or on the handle's step index.  Two calls whose [key, key + n_steps) ranges overlap reuse draws for the
 * same m: advance the key by n_steps per call.  Two handles with the same seed and key draw the same actions for the
 * same m: sharded callers give each rank its own key range.
 * Everything else is mt_rollout_branches': sources, steps, endings, the fp32 return order, the outputs, sources outside
 * [0, N) (NaN / -1 / 0, obs row untouched), the handle left untouched, the argument errors and their order (n_prefix
 * outside [0, n_steps] and a prefix_dev that disagrees with n_prefix are MT_ERR_INVALID too) and MT_ERR_STATE before
 * mt_reset.  The result is bit for bit mt_rollout_branches fed concat(prefix, mt_branch_actions(key, n_prefix,
 * n_steps - n_prefix, rows 0 .. M-1)).  A branch-step reads no action bytes past the prefix. */
int mt_rollout_branches_random(mt_env *env, int32_t n_steps, int32_t n_prefix, int64_t n_branches,
                               const int64_t *src_dev, const float *prefix_dev, const uint64_t *draw_key_dev,
                               float gamma, float *return_dev, int32_t *length_dev, uint8_t *done_dev,
                               void *obs_dev, void *stream);

/* The draws of chosen branches of mt_rollout_branches_random: out_dev [n_steps][n_rows][J] fp32, slice s, row r =
 * the actions of branch id branch_dev[r] at branch step first_step + s under the key *draw_key_dev, i.e. what
 * mt_sample_actions draws for global env id branch_dev[r] at step index key + first_step + s (mod 2^64).  Any int64
 * id is valid (its 64-bit pattern is the global id).  A planner that picked branch b of a call gets the action it
 * executes with first_step = 0, n_steps = 1.  Reads only the seed, the action range and J of the handle: it needs no
 * mt_reset, and writes nothing of the handle.  Asynchronous on `stream`.  Argument errors come before the handle is
 * looked at: draw_key_dev NULL or not 8-byte aligned, first_step < 0, n_steps < 0, n_rows outside [0, 2e9], and
 * branch_dev / out_dev NULL or not 16-byte aligned are MT_ERR_INVALID; n_steps = 0 or n_rows = 0 does nothing. */
int mt_branch_actions(mt_env *env, const uint64_t *draw_key_dev, int32_t first_step, int32_t n_steps,
                      int64_t n_rows, const int64_t *branch_dev, float *out_dev, void *stream);

/* Host-buffer step: actions_host/obs_host/reward_host/done_host must be pinned
 * (mt_host_alloc).  Copies actions H2D, steps, copies results D2H, chunked over
 * internal streams so copies overlap the kernels; synchronous on return.  Ordered after
 * everything submitted earlier to the legacy default stream / blocking streams (work on
 * cudaStreamNonBlocking streams must be synchronised by the caller). */
int mt_step_host(mt_env *env, const float *actions_host, void *obs_host, float *reward_host,
                 uint8_t *done_host);
/* mt_step_host has two implementations with identical results -- chunks staged through device buffers,
 * or one launch reading and writing the pinned host buffers across PCIe itself -- and by default times
 * both on a handle's first six calls and keeps the faster (MT_HOST_ZEROCOPY=0/1 pins it).  Returns 0
 * staged, 1 zero-copy, 2 still deciding. */
int mt_host_step_mode(const mt_env *env);
int mt_host_alloc(void **out, uint64_t bytes);
int mt_host_free(void *p);

/* State exchange (parity upload of reference objectives, checkpoint, render copy-back).
 * Any pointer may be NULL to skip that array; mask_dev as in mt_reset.
 * A checkpoint from which a new handle continues bit for bit holds: the config (mt_get_config: the seed may
 * have been changed by mt_set_seed), goals / alive / total_reward / ep_len (mt_get_state), the reset counts
 * (mt_get_reset_counts), the raw objectives (mt_get_points with zero_dead = 0) and the step index
 * (mt_get_step_index).  To restore, create a handle with that config, mt_reset it, then set all of them
 * (and the same objective stream, if one was set).  Statistics restart at zero in the new handle: a caller
 * who wants running totals adds the checkpoint's statistics. */
int mt_set_points(mt_env *env, const float *points_dev, const uint8_t *mask_dev, void *stream);
int mt_get_points(mt_env *env, float *points_dev, int32_t zero_dead, void *stream);
int mt_set_state(mt_env *env, const float *goals_dev, const uint32_t *alive_dev,
                 const float *total_reward_dev, const int32_t *ep_len_dev,
                 const uint8_t *mask_dev, void *stream);
int mt_get_state(mt_env *env, float *goals_dev, uint32_t *alive_dev, float *total_reward_dev,
                 int32_t *ep_len_dev, void *stream);
/* counts_dev [N] uint32: the resets each env has had so far (mt_reset and the in-kernel auto-reset each add
 * one).  The count keys the on-device objective sampler -- the e-th reset of an env draws with Philox counter
 * e*32 + objective, mod 2^32, so the sampler repeats after 2^27 episodes of one env -- and selects the set
 * e mod n_sets of an objective stream.  Counts wrap mod 2^32.  mt_set_seed zeroes them.  mask_dev as in
 * mt_reset; counts_dev is required.  A restore sets them AFTER the new handle's first mt_reset, because
 * mt_reset advances the counts of the envs it resets. */
int mt_get_reset_counts(mt_env *env, uint32_t *counts_dev, void *stream);
int mt_set_reset_counts(mt_env *env, const uint32_t *counts_dev, const uint8_t *mask_dev, void *stream);

/* Objective refresh stream for parity runs: points_dev [n_sets][N][X][3], borrowed.
 * The e-th reset of env n takes set (e mod n_sets).  NULL/0 restores the sampler. */
int mt_set_objective_stream(mt_env *env, const float *points_dev, int32_t n_sets);

/* One-env copy-back for the render shim and per-env attribute reads (manytor.py:131-139,
 * 196-201).  Synchronous, on the legacy default stream: one small kernel + one copy through
 * scratch buffers the handle owns (no allocation, no device-wide synchronisation).  Ordered after
 * everything submitted earlier to the legacy default stream / blocking streams (work on
 * cudaStreamNonBlocking streams must be synchronised by the caller). */
int mt_fetch_env(mt_env *env, int64_t index, float *goals_host, float *joints_host,
                 float *points_host, uint32_t *alive_host, float *total_reward_host);

/* Episode statistics.  mt_stats_device writes MT_STATS_WORDS int64 to a device
 * buffer (for an NCCL all-reduce); mt_stats_host is the synchronous host read, on the legacy default
 * stream: ordered after everything submitted earlier to it / blocking streams (work on
 * cudaStreamNonBlocking streams must be synchronised by the caller). */
int mt_stats_device(mt_env *env, int64_t *stats_dev, void *stream);
int mt_stats_host(mt_env *env, mt_stats *out);
int mt_stats_clear(mt_env *env, void *stream);

/* The ONE collective of a multi-GPU rollout (SURVEY.md section 8e): every shard's statistics summed
 * with ncclAllReduce (NVLink / NVSwitch).  NCCL is dlopen'ed at first use (libnccl.so.2).
 *   mt_stats_allreduce       one process driving n handles on n distinct devices; communicators
 *                            from ncclCommInitAll, cached per device list.  Synchronous; the sum
 *                            over all handles is written to *out_host.
 *   mt_stats_allreduce_comm  one process per GPU: `nccl_comm` is the caller's ncclComm_t
 *                            (ncclCommInitRank); stats_dev [MT_STATS_WORDS] int64 on the handle's
 *                            device receives the global sum, asynchronously on `stream`. */
int mt_stats_allreduce(mt_env *const *envs, int32_t n, mt_stats *out_host);
int mt_stats_allreduce_comm(mt_env *env, void *nccl_comm, int64_t *stats_dev, void *stream);
/* The same sum by the library's own kernel over NVLink peer memory (one process per GPU): every rank
 * owns a zero-initialised buffer of mt_stats_peer_buffer_bytes(world) bytes that all peers can write
 * (torch symmetric memory, cuMem IPC, ...); peers_dev is a DEVICE array of the `world` buffer
 * addresses as seen from this rank.  One small kernel per rank stores this rank's 64 bytes into every
 * peer's buffer, raises a flag there and waits for the peers' flags in its own: ~4 us instead of
 * ~30 us for the NCCL call.  Asynchronous on `stream`; the epoch that keys the flags lives in device
 * memory (graph-replay safe).  Every rank of the group must make the call; if a peer never does, the
 * kernel gives up after ~10 s and writes -1 into every word instead of hanging the GPU. */
int64_t mt_stats_peer_buffer_bytes(int32_t world);
int mt_stats_allreduce_peers(mt_env *env, int64_t *const *peers_dev, int32_t rank, int32_t world,
                             int64_t *stats_dev, void *stream);

/* Module-level helpers of the reference, batched over M rows:
 * fk(mode, goals) manytor.py:35-53 -> out [M][16]; dh(a, alfa, d, theta) :25-32 ->
 * out [M][16] from params [M][4]; r_theta(v1, v2) :17-22 -> out [M][2]. */
int mt_fk(const mt_config *cfg, int32_t mode, const float *goals_dev, float *out_dev, int64_t m,
          void *stream);
int mt_dh(const float *params_dev, float *out_dev, int64_t m, void *stream);
/* joints_coordinates (manytor.py:188-189) of M poses: goals [M][J] -> out [M][J][3]
 * (rows base, frame 2 .. frame J) with the handle's arm; used by the render shim. */
int mt_joints(mt_env *env, const float *goals_dev, float *out_dev, int64_t m, void *stream);
int mt_r_theta(const float *v1_dev, const float *v2_dev, float *out_dev, int64_t m, void *stream);

/* Introspection for bench.py: kernels launched by this handle since create, and
 * the algorithmic bytes per env-step of mt_step (SURVEY.md section 8d): 12J + 24X + 21
 * for an fp32 handle, 12J + 18X + 21 for a binary16 one (observations 6X instead of 12X). */
int64_t mt_launch_count(const mt_env *env);
int64_t mt_bytes_per_env_step(const mt_env *env, int32_t actions_from_hbm, int32_t obs_written);
/* Device time (ms) of the step kernels launched by the last mt_rollout_random /
 * mt_step call when timing was enabled with mt_set_timing(env, 1). */
int mt_set_timing(mt_env *env, int32_t enabled);
int mt_last_kernel_ms(mt_env *env, float *ms_out);

#ifdef __cplusplus
}
#endif
#endif /* MANYTOR_B200_H */
