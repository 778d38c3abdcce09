// C ABI of manytor_b200 (see include/manytor_b200.h): handle, state in HBM,
// kernel dispatch and the non-hot helper kernels.  There is deliberately no CPU
// path here: without a CUDA device every entry point fails with MT_ERR_NO_DEVICE.
#include <cuda_runtime.h>

#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <new>
#include <unordered_map>
#include <utility>
#include <vector>

#include "mt_jit.cuh"
#include "mt_step.cuh"

using namespace mt;

// ----------------------------------------------------------------------------
// errors
// ----------------------------------------------------------------------------
static thread_local char g_err[512] = "";

static int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CU(call)                                                                                     \
    do {                                                                                             \
        cudaError_t e_ = (call);                                                                     \
        if (e_ != cudaSuccess)                                                                       \
            return fail(e_ == cudaErrorNoDevice || e_ == cudaErrorInsufficientDriver ? MT_ERR_NO_DEVICE \
                                                                                     : MT_ERR_CUDA, \
                        "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) {
        cudaGetDevice(&prev);
        if (prev != dev) cudaSetDevice(dev);
        else prev = -1;
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

// ----------------------------------------------------------------------------
// handle
// ----------------------------------------------------------------------------
// mt_fetch_env scratch: goals[J] | joints[J][3] | points[X][3] | alive | total_reward
constexpr int kFetchFloats = MT_MAX_JOINTS * 4 + MT_MAX_OBJ * 3 + 2;

struct mt_env {
    mt_config cfg;
    long long n, n_pad, n_tiles;
    int arm;  // 0 = closed form reference arm, 2..8 = J (run-time DH table), >= 100 = preset arm
    bool f16 = false;  // observations written as binary16 (mt_config.obs_dtype)
    // NVRTC-specialised step kernels for this handle's own DH table (mt_jit.cuh); the helper kernels
    // keep using the run-time table (`arm`)
    bool jit = false;
    int jit_id = 0, jit_x = 0;
    std::string jit_preset;
    cudaKernel_t jit_kernel[2][2][2] = {};   // [in-kernel actions][observations written] (in the handle's format)[final outputs]
    cudaKernel_t jit_rollout[3][2][2] = {};  // multi-step rollout kernel, [RolloutMode][observations written][final outputs]
    bool jit_rollout_failed = false;
    float *goals = nullptr, *total_reward = nullptr, *points = nullptr;
    uint32_t *alive = nullptr, *counters = nullptr, *episode = nullptr;
    unsigned long long *stats = nullptr;   // MT_STATS_WORDS: env_steps, finished-episode sums, ground steps (device side)
    unsigned long long *ctrl = nullptr;    // kCtrlWords: step index + launch tickets (mt_step.cuh)
    float keep_fraction = 1.f; // share of the state lines marked evict_last (StepParams::pol_state)
    int32_t ep_shift = 0;      // > 0: ep_len packed into the alive word above bit ep_shift
    uint32_t ep_max = 65535u;
    int num_sms = 0;
    std::unordered_map<const void *, int> block_shape;   // per step-kernel variant: most warps one block can have on an SM
    std::unordered_map<unsigned long long, int> occupancy;   // (variant, warps per block) -> blocks per SM
    const float *obj_stream = nullptr;
    int32_t obj_sets = 0;
    long long launches = 0;
    bool was_reset = false;
    // mt_fetch_env scratch (device + pinned host), mt_stats_host / mt_stats_allreduce buffers
    float *scratch_reward = nullptr;       // mt_rollout_random with reward_dev / done_dev = NULL
    uint8_t *scratch_done = nullptr;
    void *scratch_obs = nullptr;           // mt_rollout's per-step path: one step's observations for a misaligned slice
    float *scratch_actions = nullptr;      // mt_rollout_final's per-step path: one step's draws when drawn_dev is NULL
    float *fetch_dev = nullptr, *fetch_host = nullptr;
    int64_t *stats_dev = nullptr, *stats_pin = nullptr;
    StepParams base;
    // mt_step_host resources
    static constexpr int kStreams = 4;
    cudaStream_t hs[kStreams] = {};
    cudaEvent_t hev[kStreams + 1] = {};       // per stream "kernels done"; [kStreams] = entry fence
    // mt_step_host variant: 0 staged, 1 zero-copy, 2 auto (decided from the first calls' own timings)
    int host_mode = 2, host_calls = 0;
    double host_best[2] = {1e30, 1e30};
    float *h_actions = nullptr, *h_reward = nullptr;
    void *h_obs = nullptr;
    uint8_t *h_done = nullptr;
    // timing
    bool timing = false;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    bool ev_valid = false;
};

static const float kRefDh[4][4] = {{0.0f, -1.57079632679f, 4.3f, 0.0f},
                                   {0.0f, 1.57079632679f, 0.0f, 0.0f},
                                   {0.0f, -1.57079632679f, 24.3f, 0.0f},
                                   {27.0f, 1.57079632679f, 0.0f, -1.57079632679f}};

static bool is_reference_arm(const mt_config &c) {
    if (c.n_joints != 4) return false;
    for (int i = 0; i < 4; ++i)
        for (int k = 0; k < 4; ++k)
            if (std::fabs(c.dh[i][k] - kRefDh[i][k]) > 1e-6f) return false;
    return c.obs_frame == 3 && c.ground_frame_a == 3 && c.ground_frame_b == 4 && c.catch_frame == 4;
}

// does the configuration describe the preset arm `id` (table within 1e-6, usual frame selectors)?
template <int ID>
static bool is_preset_arm(const mt_config &c) {
    constexpr int J = ArmJoints<ID>::value;
    if (c.n_joints != J) return false;
    for (int i = 0; i < J; ++i) {
        const JointConst q = Preset<ID>::row(i);
        const double ca = std::cos((double)c.dh[i][1]), sa = std::sin((double)c.dh[i][1]);
        const double co = std::cos((double)c.dh[i][3]), so = std::sin((double)c.dh[i][3]);
        if (std::fabs(c.dh[i][0] - q.a) > 1e-6 || std::fabs(c.dh[i][2] - q.d) > 1e-6 || std::fabs(ca - q.ca) > 1e-6 ||
            std::fabs(sa - q.sa) > 1e-6 || std::fabs(co - q.co) > 1e-6 || std::fabs(so - q.so) > 1e-6)
            return false;
    }
    return c.obs_frame == J - 1 && c.ground_frame_a == J - 1 && c.ground_frame_b == J && c.catch_frame == J;
}

// cos/sin of the table's alpha and theta offsets: the table arrives as fp32 (pi/2 -> 1.57079637, whose
// cosine is -4.4e-8, where the reference's fp64 np.pi/2 gives 6e-17), so values within fp32 rounding of
// 0 or +-1 are snapped; this is also what lets the specialised kernels fold them away.
static double snap(double v) { return std::fabs(v) < 5e-7 ? 0.0 : (std::fabs(std::fabs(v) - 1.0) < 5e-7 ? (v > 0 ? 1.0 : -1.0) : v); }

extern "C" int mt_abi_version(void) { return MT_ABI_VERSION; }
extern "C" const char *mt_last_error(void) { return g_err; }

extern "C" int mt_config_init(mt_config *cfg) {
    if (!cfg) return fail(MT_ERR_INVALID, "cfg is NULL");
    std::memset(cfg, 0, sizeof(*cfg));
    cfg->struct_size = sizeof(mt_config);
    cfg->n_envs = 1;
    cfg->n_joints = 4;
    cfg->n_obj = 10;
    for (int i = 0; i < 4; ++i)
        for (int k = 0; k < 4; ++k) cfg->dh[i][k] = kRefDh[i][k];
    cfg->obs_frame = 3;
    cfg->ground_frame_a = 3;
    cfg->ground_frame_b = 4;
    cfg->catch_frame = 4;
    cfg->radius = 51.3f;
    cfg->catch_tol = 8.0f;
    cfg->substeps = 25;
    cfg->horizon = 0;
    cfg->terminate_on_ground = 0;
    cfg->auto_reset = 0;
    cfg->obs_after_reset = 0;
    cfg->fk_mode = 0;
    cfg->action_low = -180;
    cfg->action_high = 180;
    cfg->seed = 0;
    cfg->obs_dtype = MT_OBS_F32;
    return MT_OK;
}

// the L2 eviction policies of a handle (StepParams::pol_state / pol_stream / pol_store); kind: 0 evict_first (the
// default for everything streamed), 1 evict_normal, 2 evict_last (MT_POL_LOAD / MT_POL_STORE = first|normal|last, tuning)
__device__ unsigned long long policy_of(int kind) {
    return kind == 1 ? policy_evict_normal() : (kind == 2 ? policy_evict_last() : policy_evict_first());
}
__global__ void policy_kernel(unsigned long long *out, float keep_fraction, int load_kind, int store_kind) {
#ifdef MT_NO_L2_HINTS
    out[0] = out[1] = out[2] = policy_evict_last();      // A/B builds: evict_normal everywhere
#else
    out[0] = keep_fraction > 0.f ? policy_evict_last_fraction(fminf(keep_fraction, 1.0f)) : policy_evict_normal();
    out[1] = policy_of(load_kind);
    out[2] = policy_of(store_kind);
#endif
}

static int policy_kind(const char *name, int fallback) {
    const char *v = std::getenv(name);
    if (!v) return fallback;
    return v[0] == 'n' ? 1 : (v[0] == 'l' ? 2 : 0);
}

static int validate(const mt_config &c) {
    if (c.struct_size != sizeof(mt_config)) return fail(MT_ERR_INVALID, "mt_config.struct_size %u != %zu (ABI mismatch)", c.struct_size, sizeof(mt_config));
    if (c.n_envs < 1 || c.n_envs > 2000000000LL) return fail(MT_ERR_INVALID, "n_envs must be in [1, 2e9] (32-bit env index per shard)");
    if (c.n_joints < 2 || c.n_joints > MT_MAX_JOINTS) return fail(MT_ERR_INVALID, "n_joints must be in [2, %d]", MT_MAX_JOINTS);
    if (c.n_obj < 1 || c.n_obj > MT_MAX_OBJ) return fail(MT_ERR_INVALID, "n_obj must be in [1, %d]", MT_MAX_OBJ);
    const int J = c.n_joints;
    const int fr[4] = {c.obs_frame, c.ground_frame_a, c.ground_frame_b, c.catch_frame};
    for (int f : fr)
        if (f < 0 || f > J) return fail(MT_ERR_INVALID, "frame selector %d outside [0, %d]", f, J);
    if (c.substeps < 2 || c.substeps > 4096) return fail(MT_ERR_INVALID, "substeps must be in [2, 4096]");
    if (c.horizon < 0 || c.horizon > 65535) return fail(MT_ERR_INVALID, "horizon must be in [0, 65535]");
    if (c.action_high <= c.action_low) return fail(MT_ERR_INVALID, "action_high must exceed action_low");
    if (!(c.radius > 0.f) || !(c.catch_tol >= 0.f)) return fail(MT_ERR_INVALID, "radius must be > 0 and catch_tol >= 0");
    if (c.fk_mode < 0 || c.fk_mode > 3) return fail(MT_ERR_INVALID, "fk_mode must be 0, 1, 2 or 3");
    if (c.fk_mode == 2 && !is_reference_arm(c)) return fail(MT_ERR_INVALID, "fk_mode=2 (closed form) needs the reference DH table and frames");
    if (c.obs_dtype != MT_OBS_F32 && c.obs_dtype != MT_OBS_F16)
        return fail(MT_ERR_INVALID, "obs_dtype must be MT_OBS_F32 (0) or MT_OBS_F16 (1), not %d", c.obs_dtype);
    return MT_OK;
}

static void fill_arm(const mt_config &c, StepParams &P) {
    const int J = c.n_joints;
    for (int i = 0; i < MT_MAX_JOINTS; ++i) P.arm[i] = JointConst{0, 0, 1, 0, 1, 0};
    for (int i = 0; i < J; ++i) {
        P.arm[i].a = c.dh[i][0];
        P.arm[i].d = c.dh[i][2];
        P.arm[i].ca = (float)snap(std::cos((double)c.dh[i][1]));
        P.arm[i].sa = (float)snap(std::sin((double)c.dh[i][1]));
        P.arm[i].co = (float)snap(std::cos((double)c.dh[i][3]));
        P.arm[i].so = (float)snap(std::sin((double)c.dh[i][3]));
    }
    // obs anchor at the zero pose (manytor.py:224-225), fp64 chain on the snapped table
    double R[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}}, t[3] = {0, 0, 0};
    double anchor[3] = {0, 0, 0};
    for (int i = 0; i < J; ++i) {
        const double ct = P.arm[i].co, st = P.arm[i].so, ca = P.arm[i].ca, sa = P.arm[i].sa;
        for (int r = 0; r < 3; ++r) {
            double u = R[r][0] * ct + R[r][1] * st, v = R[r][1] * ct - R[r][0] * st, r2 = R[r][2];
            t[r] += P.arm[i].a * u + P.arm[i].d * r2;
            R[r][0] = u;
            R[r][1] = v * ca + r2 * sa;
            R[r][2] = r2 * ca - v * sa;
        }
        if (i + 1 == c.obs_frame) { anchor[0] = t[0]; anchor[1] = t[1]; anchor[2] = t[2]; }
    }
    for (int k = 0; k < 3; ++k) P.zero_anchor[k] = (float)anchor[k];
}

static void fill_params(const mt_config &c, StepParams &P) {
    std::memset(&P, 0, sizeof(P));
    P.n_obj = c.n_obj;
    P.n_joints = c.n_joints;
    P.substeps = c.substeps;
    P.horizon = c.horizon;
    P.flags = (c.terminate_on_ground ? kTerminateOnGround : 0) | (c.auto_reset ? kAutoReset : 0) |
              (c.obs_after_reset ? kObsAfterReset : 0);
    P.action_low = c.action_low;
    P.action_span = (uint32_t)(c.action_high - c.action_low);
    P.radius = c.radius;
    P.catch_tol = c.catch_tol;
    P.inv_div = 1.0f / (float)(c.substeps - 1);
    P.obs_frame = c.obs_frame;
    P.ground_a = c.ground_frame_a;
    P.ground_b = c.ground_frame_b;
    P.catch_frame = c.catch_frame;
    P.seed_lo = (uint32_t)c.seed;
    P.seed_hi = (uint32_t)(c.seed >> 32);
    P.env_id_base = c.env_id_base;
    P.tile_bytes = (uint32_t)(kTile * 3 * c.n_obj * 4);
    fill_arm(c, P);
}

extern "C" int mt_create(const mt_config *cfg, mt_env **out) {
    if (!cfg || !out) return fail(MT_ERR_INVALID, "cfg/out is NULL");
    *out = nullptr;
    if (int rc = validate(*cfg)) return rc;
    int count = 0;
    cudaError_t ce = cudaGetDeviceCount(&count);
    if (ce != cudaSuccess || count == 0)
        return fail(MT_ERR_NO_DEVICE, "no CUDA device (%s); manytor_b200 has no CPU fallback",
                    ce == cudaSuccess ? "device count is 0" : cudaGetErrorString(ce));
    if (cfg->device < 0 || cfg->device >= count) return fail(MT_ERR_INVALID, "device %d outside [0, %d)", cfg->device, count);
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, cfg->device));
    if (prop.major != 10)
        return fail(MT_ERR_NO_DEVICE, "device %d is sm_%d%d; this library is built for sm_100a (B200) only", cfg->device,
                    prop.major, prop.minor);
    DeviceGuard guard(cfg->device);
    mt_env *e = new (std::nothrow) mt_env();
    if (!e) return fail(MT_ERR_INVALID, "out of host memory");
    e->cfg = *cfg;
    e->n = cfg->n_envs;
    e->n_tiles = (e->n + kTile - 1) / kTile;
    e->n_pad = e->n_tiles * kTile;
    e->f16 = cfg->obs_dtype == MT_OBS_F16;
    e->arm = cfg->n_joints;                                   // run-time DH table
    if (cfg->fk_mode != 1) {
        if (is_reference_arm(*cfg)) e->arm = 0;               // closed form
#define MT_MATCH(ID) else if (is_preset_arm<ID>(*cfg)) e->arm = ID;   /* compile-time table */
        MT_FOR_EACH_PRESET_ARM(MT_MATCH)
#undef MT_MATCH
    }
    const size_t np = (size_t)e->n_pad, J = cfg->n_joints, X = cfg->n_obj;
#define ALLOC(ptr, bytes)                                        \
    do {                                                         \
        cudaError_t e_ = cudaMalloc((void **)&(ptr), (bytes));   \
        if (e_ == cudaSuccess) e_ = cudaMemset((ptr), 0, (bytes)); \
        if (e_ != cudaSuccess) {                                 \
            int rc_ = fail(MT_ERR_CUDA, "cudaMalloc(%zu) failed: %s", (size_t)(bytes), cudaGetErrorString(e_)); \
            mt_destroy(e);                                       \
            return rc_;                                          \
        }                                                        \
    } while (0)
    ALLOC(e->goals, np * J * 4);
    ALLOC(e->alive, np * 4);
    ALLOC(e->total_reward, np * 4);
    // episode length: in the spare bits of the alive word when they can hold it (mt_step.cuh, StepParams::ep_shift)
    {
        const int shift = cfg->n_obj <= 16 ? 16 : cfg->n_obj;
        const bool packed = cfg->n_obj <= 16 || (cfg->n_obj < 32 && cfg->horizon > 0 && cfg->horizon < (1 << (32 - shift)));
        e->ep_shift = packed ? shift : 0;
        e->ep_max = packed ? (uint32_t)((1ull << (32 - shift)) - 1ull) : 65535u;
        if (e->ep_max > 65535u) e->ep_max = 65535u;
    }
    if (!e->ep_shift) ALLOC(e->counters, np * 4);
    ALLOC(e->episode, np * 4);
    ALLOC(e->points, np * X * 3 * 4);
    ALLOC(e->stats, MT_STATS_WORDS * 8);
    ALLOC(e->ctrl, kCtrlWords * 8);
    ALLOC(e->fetch_dev, kFetchFloats * 4);
    ALLOC(e->stats_dev, MT_STATS_WORDS * 8);
#undef ALLOC
    if (cudaHostAlloc((void **)&e->fetch_host, kFetchFloats * 4, cudaHostAllocDefault) != cudaSuccess ||
        cudaHostAlloc((void **)&e->stats_pin, MT_STATS_WORDS * 8, cudaHostAllocDefault) != cudaSuccess) {
        int rc = fail(MT_ERR_CUDA, "cudaHostAlloc of the handle's scratch failed: %s", cudaGetErrorString(cudaGetLastError()));
        mt_destroy(e);
        return rc;
    }
    e->num_sms = prop.multiProcessorCount;
    fill_params(*cfg, e->base);
    e->base.goals = e->goals;
    e->base.alive = e->alive;
    e->base.total_reward = e->total_reward;
    e->base.counters = e->counters;
    e->base.episode = e->episode;
    e->base.points = e->points;
    e->base.stats = e->stats;
    e->base.ctrl = e->ctrl;
    e->base.n = e->n;
    e->base.tile_begin = 0;
    e->base.tile_end = e->n_tiles;
    e->base.pair_layout = (cfg->n_obj % 2 == 0) ? 1 : 0;      // even X: pair-interleaved objectives (mt_step.cuh)
    e->base.ep_shift = e->ep_shift;
    e->base.ep_max = e->ep_max;
    {
        // evict_last budget for the per-env state: 36 MB of the 126 MB L2 (MT_L2_KEEP_MB overrides, 0 = none)
        double keep_mb = 36.0;
        if (const char *kb = std::getenv("MT_L2_KEEP_MB")) keep_mb = std::atof(kb);
        const double state_bytes = (4.0 * J + 8.0 + (e->ep_shift ? 0.0 : 4.0)) * (double)np;
        e->keep_fraction = (float)(keep_mb * 1048576.0 >= state_bytes ? 1.0 : keep_mb * 1048576.0 / state_bytes);
        // Streamed arrays (objectives, actions in; observations, reward, done out): evict_normal while the whole state fits
        // its evict_last budget -- measured 44.0 vs 47.1 us per step at 2^20 envs, 98.1 vs 100.3 for the UR5 config
        // (profiles/r2_ab_l2_policies.txt) -- and evict_first once it does not (2^22 envs: 231.5 vs 237.6 us), where the
        // streams would otherwise push the protected part of the state out.
        const int stream_kind = e->keep_fraction >= 1.0f ? 1 : 0;
        policy_kernel<<<1, 1>>>(e->stats, e->keep_fraction, policy_kind("MT_POL_LOAD", stream_kind),
                                policy_kind("MT_POL_STORE", stream_kind));   // the stats words are zeroed again right below
        unsigned long long pol[3] = {0, 0, 0};
        cudaError_t pe = cudaMemcpy(pol, e->stats, sizeof(pol), cudaMemcpyDeviceToHost);
        if (pe == cudaSuccess) pe = cudaMemset(e->stats, 0, sizeof(pol));
        if (pe != cudaSuccess) {
            int rc = fail(MT_ERR_CUDA, "L2 policy setup failed: %s", cudaGetErrorString(pe));
            mt_destroy(e);
            return rc;
        }
        e->base.pol_state = pol[0];
        e->base.pol_stream = pol[1];
        e->base.pol_store = pol[2];
    }
    // Run-time specialisation (mt_jit.cuh): a run-time table with the usual frame selectors gets its own
    // Preset<>; a built-in arm with an objective count other than the pre-compiled 10 / 20 gets the same arm
    // code with X as a compile-time constant (unrolled objective walk).
    const int nj = cfg->n_joints;
    const bool usual = cfg->obs_frame == nj - 1 && cfg->ground_frame_a == nj - 1 && cfg->ground_frame_b == nj && cfg->catch_frame == nj;
    const char *off = std::getenv("MT_DISABLE_JIT");
    const bool allowed = cfg->fk_mode == 3 || (cfg->fk_mode == 0 && !(off && off[0] == '1'));
    const bool runtime_table = e->arm >= 2 && e->arm <= MT_MAX_JOINTS;
    const bool other_x = !runtime_table && cfg->n_obj != 10 && cfg->n_obj != 20;
    if (allowed && (runtime_table || other_x)) {
        std::string err;
        if (runtime_table && !usual) {
            err = "run-time specialisation needs the usual frame selectors (obs J-1, ground J-1 and J, catch J)";
        } else {
            e->jit_id = runtime_table ? 1000 + nj : e->arm;
            e->jit_x = cfg->n_obj;                                    // compile-time X: unrolled objective walk
            e->jit_preset = runtime_table ? preset_source(e->jit_id, nj, e->base.arm) : std::string();
            JitKernel k = jit_step_kernel(e->jit_preset, e->jit_id, e->jit_x, false, true, e->f16, false, err);
            if (k.kernel) {
                e->jit = true;
                e->jit_kernel[0][1][0] = k.kernel;
            }
        }
        if (!e->jit && cfg->fk_mode == 3 && runtime_table) {
            int rc = fail(MT_ERR_INVALID, "fk_mode=3 (run-time specialisation) unavailable: %s", err.c_str());
            mt_destroy(e);
            return rc;
        }
    }
    *out = e;
    return MT_OK;
}

extern "C" int mt_destroy(mt_env *e) {
    if (!e) return MT_OK;
    DeviceGuard guard(e->cfg.device);
    cudaDeviceSynchronize();
    cudaFree(e->goals); cudaFree(e->alive); cudaFree(e->total_reward); cudaFree(e->counters);
    cudaFree(e->episode); cudaFree(e->points); cudaFree(e->stats); cudaFree(e->ctrl);
    cudaFree(e->fetch_dev); cudaFree(e->stats_dev); cudaFree(e->scratch_reward); cudaFree(e->scratch_done);
    cudaFree(e->scratch_obs); cudaFree(e->scratch_actions);
    if (e->fetch_host) cudaFreeHost(e->fetch_host);
    if (e->stats_pin) cudaFreeHost(e->stats_pin);
    cudaFree(e->h_actions); cudaFree(e->h_obs); cudaFree(e->h_reward); cudaFree(e->h_done);
    for (auto &s : e->hs) if (s) cudaStreamDestroy(s);
    for (auto &v : e->hev) if (v) cudaEventDestroy(v);
    if (e->ev0) cudaEventDestroy(e->ev0);
    if (e->ev1) cudaEventDestroy(e->ev1);
    delete e;
    return MT_OK;
}

// Re-seeding restarts the on-device streams: the Philox key changes AND the counters that index the
// streams (per-env episode count, step index) go back to zero, so reset(seed=s) reproduces the same
// objectives and actions whenever it is called with the same s (Gymnasium's contract).  Synchronous.
extern "C" int mt_set_seed(mt_env *e, uint64_t seed) {
    if (!e) return fail(MT_ERR_INVALID, "env is NULL");
    DeviceGuard guard(e->cfg.device);
    CU(cudaDeviceSynchronize());
    CU(cudaMemset(e->episode, 0, (size_t)e->n_pad * 4));
    CU(cudaMemset(e->ctrl + kCtrlStep, 0, 8));
    CU(cudaDeviceSynchronize());
    e->cfg.seed = seed;
    e->base.seed_lo = (uint32_t)seed;
    e->base.seed_hi = (uint32_t)(seed >> 32);
    return MT_OK;
}

// The step index that keys the action stream (mt_sample_actions / mt_rollout_random): part of a
// checkpoint next to mt_get_state.  Synchronous (one 8-byte copy on the legacy default stream; the set waits for
// its copy to land, which a copy from pageable memory does not promise on return, so that a launch on any stream
// issued after it reads the new index).
extern "C" int mt_get_step_index(mt_env *e, uint64_t *out) {
    if (!e || !out) return fail(MT_ERR_INVALID, "NULL argument");
    DeviceGuard guard(e->cfg.device);
    unsigned long long v = 0;
    CU(cudaMemcpy(&v, e->ctrl + kCtrlStep, 8, cudaMemcpyDeviceToHost));
    *out = v;
    return MT_OK;
}
extern "C" int mt_set_step_index(mt_env *e, uint64_t value) {
    if (!e) return fail(MT_ERR_INVALID, "env is NULL");
    // the kernels' launch ticket depends on bit 63 of the index being clear (launch_ticket, mt_step.cuh)
    if (value > MT_STEP_INDEX_MAX)
        return fail(MT_ERR_INVALID, "step index %llu is above MT_STEP_INDEX_MAX (2^62)", (unsigned long long)value);
    DeviceGuard guard(e->cfg.device);
    const unsigned long long v = value;
    CU(cudaMemcpy(e->ctrl + kCtrlStep, &v, 8, cudaMemcpyHostToDevice));
    CU(cudaStreamSynchronize(nullptr));
    return MT_OK;
}

extern "C" int mt_get_config(const mt_env *e, mt_config *out) {
    if (!e || !out) return fail(MT_ERR_INVALID, "NULL argument");
    *out = e->cfg;
    return MT_OK;
}

// ----------------------------------------------------------------------------
// helper kernels (not on the hot path; one thread per env, plain accesses)
// ----------------------------------------------------------------------------
__device__ __forceinline__ void pose_of(const StepParams &P, int arm, const float *g, Frames &f, float *jout) {
    // final pose only: the same code as the step kernel with no interior sub-poses
    switch (arm) {
        case 0: ref_arm<false>(g, g, 1, 0.f, f, jout); break;
#define MT_CASE(JJ) case JJ: { StepParams Q = P; Q.substeps = 1; generic_arm<JJ, false>(Q, g, g, f, jout); } break;
        MT_CASE(2) MT_CASE(3) MT_CASE(4) MT_CASE(5) MT_CASE(6) MT_CASE(7) MT_CASE(8)
        MT_FOR_EACH_PRESET_ARM(MT_CASE)
#undef MT_CASE
    }
}

__global__ void reset_kernel(const __grid_constant__ StepParams P, const uint8_t *mask) {
    const long long env = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= P.n) return;
    if (mask && !mask[env]) return;
    const int x = P.n_obj, J = P.n_joints;
    const uint32_t ep = P.episode[env];
    P.episode[env] = ep + 1u;
    float *row = P.points + env * 3 * x;
    for (int pt = 0; pt < x; ++pt) {
        float px, py, pz;
        if (P.obj_stream) {
            const float *src = P.obj_stream + (((long long)(ep % (uint32_t)P.obj_sets) * P.n + env) * x + pt) * 3;
            px = src[0]; py = src[1]; pz = src[2];
        } else {
            sample_point(P, P.env_id_base + env, ep, pt, px, py, pz);
        }
        row[point_index(P.pair_layout, pt, 0)] = px;
        row[point_index(P.pair_layout, pt, 1)] = py;
        row[point_index(P.pair_layout, pt, 2)] = pz;
    }
    for (int i = 0; i < J; ++i) P.goals[env * J + i] = 0.f;           // manytor.py:220
    P.total_reward[env] = 0.f;                                        // manytor.py:221
    P.alive[env] = (x >= 32) ? 0xffffffffu : ((1u << x) - 1u);        // manytor.py:222 (and ep_len = 0 when packed)
    if (!P.ep_shift) P.counters[env] = 0u;
}

template <bool F16>
__global__ void observe_kernel(const __grid_constant__ StepParams P, int arm, void *obs) {
    const long long env = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= P.n) return;
    const int x = P.n_obj, J = P.n_joints;
    float g[MT_MAX_JOINTS];
    for (int i = 0; i < J; ++i) g[i] = P.goals[env * J + i];
    Frames f;
    pose_of(P, arm, g, f, nullptr);
    const uint32_t alive = alive_mask_of(P, P.alive[env]);
    const float *row = P.points + env * 3 * x;
    void *dst = obs_at<F16>(obs, (size_t)env * 3 * x);
    for (int pt = 0; pt < x; ++pt) {
        float px = row[point_index(P.pair_layout, pt, 0)], py = row[point_index(P.pair_layout, pt, 1)],
              pz = row[point_index(P.pair_layout, pt, 2)];
        one_objective<true>(px, py, pz, f, P.catch_tol, (alive >> pt) & 1u);
        store_obs<F16>(dst, pt * 3, px); store_obs<F16>(dst, pt * 3 + 1, py); store_obs<F16>(dst, pt * 3 + 2, pz);
    }
}

__global__ void joints_kernel(const __grid_constant__ StepParams P, int arm, const float *goals, long long m, float *out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const int J = P.n_joints;
    float g[MT_MAX_JOINTS], jb[MT_MAX_JOINTS * 3];
    for (int k = 0; k < J; ++k) g[k] = goals[i * J + k];
    Frames f;
    pose_of(P, arm, g, f, jb);
    for (int k = 0; k < J * 3; ++k) out[i * J * 3 + k] = jb[k];
}

__global__ void set_points_kernel(const __grid_constant__ StepParams P, const float *src, const uint8_t *mask) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long row = 3LL * P.n_obj;
    if (i >= P.n * row) return;
    const long long env = i / row;
    if (mask && !mask[env]) return;
    const int k = (int)(i - env * row);                               // public row-major [X][3]
    P.points[env * row + point_index(P.pair_layout, k / 3, k % 3)] = src[i];
}

__global__ void get_points_kernel(const __grid_constant__ StepParams P, float *dst, int zero_dead) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long row = 3LL * P.n_obj;
    if (i >= P.n * row) return;
    const long long env = i / row;
    const int k = (int)(i - env * row), pt = k / 3;
    const bool dead = zero_dead && !((alive_mask_of(P, P.alive[env]) >> pt) & 1u);   // manytor.py:148
    dst[i] = dead ? 0.f : P.points[env * row + point_index(P.pair_layout, pt, k % 3)];
}

__global__ void set_state_kernel(const __grid_constant__ StepParams P, const float *goals, const uint32_t *alive,
                                 const float *total, const int32_t *eplen, const uint8_t *mask) {
    const long long env = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= P.n) return;
    if (mask && !mask[env]) return;
    const int J = P.n_joints;
    if (goals) for (int i = 0; i < J; ++i) P.goals[env * J + i] = goals[env * J + i];
    const uint32_t len = eplen ? (uint32_t)min(max(eplen[env], 0), (int)P.ep_max) : 0u;
    if (P.ep_shift) {
        const uint32_t amask = (1u << P.ep_shift) - 1u;
        uint32_t w = P.alive[env];
        if (alive) w = (w & ~amask) | (alive[env] & amask);
        if (eplen) w = (w & amask) | (len << P.ep_shift);
        P.alive[env] = w;
    } else {
        if (alive) P.alive[env] = alive[env];
        if (eplen) P.counters[env] = len;
    }
    if (total) P.total_reward[env] = total[env];
}

__global__ void get_state_kernel(const __grid_constant__ StepParams P, float *goals, uint32_t *alive, float *total,
                                 int32_t *eplen) {
    const long long env = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= P.n) return;
    const int J = P.n_joints;
    if (goals) for (int i = 0; i < J; ++i) goals[env * J + i] = P.goals[env * J + i];
    const uint32_t w = P.alive[env];
    if (alive) alive[env] = alive_mask_of(P, w);
    if (total) total[env] = P.total_reward[env];
    if (eplen) eplen[env] = (int32_t)(P.ep_shift ? (w >> P.ep_shift) : P.counters[env]);
}

__global__ void set_reset_counts_kernel(const __grid_constant__ StepParams P, const uint32_t *counts,
                                        const uint8_t *mask) {
    const long long env = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= P.n) return;
    if (mask && !mask[env]) return;
    P.episode[env] = counts[env];
}

__global__ void get_reset_counts_kernel(const __grid_constant__ StepParams P, uint32_t *counts) {
    const long long env = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= P.n) return;
    counts[env] = P.episode[env];
}

__global__ void sample_actions_kernel(const __grid_constant__ StepParams P, float *actions) {
    const long long env = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= P.n) return;
    float a[MT_MAX_JOINTS];
    draw_actions(P, ld_volatile_u64(P.ctrl + kCtrlStep), P.env_id_base + env, P.n_joints, a);
    for (int i = 0; i < P.n_joints; ++i) actions[env * P.n_joints + i] = a[i];
}

// mt_branch_actions: out[s][r] = the draws of branch id ids[r] at branch step first + s, i.e. what mt_sample_actions
// draws for global env id ids[r] at step index *key + first + s (mod 2^64) -- what branch_kernel<.., DRAW = true>
// draws.  One thread per (s, r), grid-stride.
__global__ void branch_actions_kernel(const __grid_constant__ StepParams P, const unsigned long long *key, int first,
                                      int n_steps, long long rows, const int64_t *ids, float *out) {
    const long long total = (long long)n_steps * rows;
    const unsigned long long k0 = *key + (unsigned long long)first;
    const int J = P.n_joints;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long s = i / rows, r = i - s * rows;
        float a[MT_MAX_JOINTS];
        draw_actions(P, k0 + (unsigned long long)s, (long long)ids[r], J, a);
#pragma unroll
        for (int j = 0; j < MT_MAX_JOINTS; ++j)       // constant indices: `a` stays in registers
            if (j < J) out[i * J + j] = a[j];
    }
}

// stats: the device-side counters (env-steps, finished-episode sums, ground-contact steps) + a
// block/warp-shuffle reduction of the in-progress total_reward, written as MT_STATS_WORDS int64.
__global__ void stats_kernel(const __grid_constant__ StepParams P, long long *out) {
    long long local = 0;
    for (long long env = (long long)blockIdx.x * blockDim.x + threadIdx.x; env < P.n;
         env += (long long)gridDim.x * blockDim.x)
        local += (long long)P.total_reward[env];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) local += __shfl_xor_sync(0xffffffffu, local, o);
    __shared__ long long part[32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) part[warp] = local;
    __syncthreads();
    if (warp == 0) {
        local = (lane < (int)(blockDim.x >> 5)) ? part[lane] : 0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) local += __shfl_xor_sync(0xffffffffu, local, o);
        if (lane == 0 && local) atomicAdd((unsigned long long *)(out + 7), (unsigned long long)local);
    }
    if (blockIdx.x == 0 && threadIdx.x < 7) out[threadIdx.x] = (long long)P.stats[threadIdx.x];
}

__global__ void fk_kernel(const __grid_constant__ StepParams P, int mode, const float *goals, long long m, float *out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const int J = P.n_joints;
    float R[3][3] = {{1.f, 0.f, 0.f}, {0.f, 1.f, 0.f}, {0.f, 0.f, 1.f}}, t[3] = {0.f, 0.f, 0.f};
    for (int k = 0; k < mode && k < J; ++k) {
        float sk, ck;
        sincos_deg(goals[i * J + k], sk, ck);
        const JointConst q = P.arm[k];
        float c = fmaf(ck, q.co, -(sk * q.so)), s = fmaf(sk, q.co, ck * q.so);
        for (int r = 0; r < 3; ++r) {
            float u = fmaf(R[r][0], c, R[r][1] * s), v = fmaf(R[r][1], c, -(R[r][0] * s)), r2 = R[r][2];
            t[r] = fmaf(q.a, u, fmaf(q.d, r2, t[r]));
            R[r][0] = u;
            R[r][1] = fmaf(v, q.ca, r2 * q.sa);
            R[r][2] = fmaf(r2, q.ca, -(v * q.sa));
        }
    }
    float *o = out + i * 16;
    for (int r = 0; r < 3; ++r) {
        o[r * 4 + 0] = R[r][0]; o[r * 4 + 1] = R[r][1]; o[r * 4 + 2] = R[r][2]; o[r * 4 + 3] = t[r];
    }
    o[12] = 0.f; o[13] = 0.f; o[14] = 0.f; o[15] = 1.f;
}

__global__ void dh_kernel(const float *params, long long m, float *out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const float a = params[i * 4], alfa = params[i * 4 + 1], d = params[i * 4 + 2], th = params[i * 4 + 3];
    float st, ct, sa, ca;
    sincosf(th, &st, &ct);
    sincosf(alfa, &sa, &ca);
    float *o = out + i * 16;
    o[0] = ct; o[1] = -st * ca; o[2] = st * sa; o[3] = a * ct;
    o[4] = st; o[5] = ct * ca; o[6] = -ct * sa; o[7] = a * st;
    o[8] = 0.f; o[9] = sa; o[10] = ca; o[11] = d;
    o[12] = 0.f; o[13] = 0.f; o[14] = 0.f; o[15] = 1.f;
}

__global__ void r_theta_kernel(const float *v1, const float *v2, long long m, float *out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    float dx = fabsf(v1[i * 3] - v2[i * 3]), dy = fabsf(v1[i * 3 + 1] - v2[i * 3 + 1]),
          dz = fabsf(v1[i * 3 + 2] - v2[i * 3 + 2]);
    const float h2 = fmaf(dx, dx, dy * dy), h = fast_sqrt(h2);
    out[i * 2] = atan2_deg_pos(dx, dy, h);
    out[i * 2 + 1] = atan2_deg_pos(h, dz, fast_sqrt(fmaf(dz, dz, h2)));
}

// ----------------------------------------------------------------------------
// step dispatch
// ----------------------------------------------------------------------------
typedef void (*StepFn)(const StepParams);
typedef void (*BranchFn)(const StepParams, const BranchParams);

// final: the FINAL = true kernels of mt_step_final, built only for the caller's actions with observations written
template <int ARM, int X, bool RAND>
static StepFn pick_obs(bool wobs, bool f16, bool final) {
    if (final) {
        if constexpr (RAND) return nullptr;
        else if (!wobs) return nullptr;
        else return f16 ? step_kernel<ARM, X, false, true, true, true> : step_kernel<ARM, X, false, true, false, true>;
    }
    if (!wobs) return step_kernel<ARM, X, RAND, false, false, false>;
    return f16 ? step_kernel<ARM, X, RAND, true, true, false> : step_kernel<ARM, X, RAND, true, false, false>;
}

template <int ARM, int X>
static StepFn pick_flags(bool rnd, bool wobs, bool f16, bool final) {
    return rnd ? pick_obs<ARM, X, true>(wobs, f16, final) : pick_obs<ARM, X, false>(wobs, f16, final);
}

template <int ARM>
static StepFn pick_x(int x, bool rnd, bool wobs, bool f16, bool final) {
    switch (x) {
        case 10: return pick_flags<ARM, 10>(rnd, wobs, f16, final);
        case 20: return pick_flags<ARM, 20>(rnd, wobs, f16, final);
        default: return pick_flags<ARM, 0>(rnd, wobs, f16, final);
    }
}

static StepFn pick_kernel(int arm, int x, bool rnd, bool wobs, bool f16, bool final) {
    switch (arm) {
        case 0: return pick_x<0>(x, rnd, wobs, f16, final);
        case 2: return pick_flags<2, 0>(rnd, wobs, f16, final);
        case 3: return pick_flags<3, 0>(rnd, wobs, f16, final);
        case 4: return pick_flags<4, 0>(rnd, wobs, f16, final);
        case 5: return pick_flags<5, 0>(rnd, wobs, f16, final);
        case 6: return pick_x<6>(x, rnd, wobs, f16, final);
        case 7: return pick_flags<7, 0>(rnd, wobs, f16, final);
        case 8: return pick_flags<8, 0>(rnd, wobs, f16, final);
#define MT_PICK(ID) case ID: return pick_x<ID>(x, rnd, wobs, f16, final);
        MT_FOR_EACH_PRESET_ARM(MT_PICK)
#undef MT_PICK
    }
    return nullptr;
}

static int check_ptr(const void *p, const char *name, bool required) {
    if (!p) return required ? fail(MT_ERR_INVALID, "%s is NULL", name) : MT_OK;
    if (((uintptr_t)p & 15u) != 0) return fail(MT_ERR_INVALID, "%s must be 16-byte aligned", name);
    return MT_OK;
}

// Entries of the per-block sin/cos table for in-kernel (integer-degree) actions (ActionTrig, mt_step.cuh): the whole
// action range when it is small enough to sit beside the tile buffers, else none (the kernels then evaluate).
static int trig_table_entries(const mt_env *e) {
    if (const char *v = std::getenv("MT_ACTION_TABLE"))
        if (v[0] == '0') return 0;
    const long long span = (long long)e->cfg.action_high - (long long)e->cfg.action_low;
    return span >= 1 && span <= 720 ? (int)span : 0;
}

// Block shape and grid of a persistent launch of `fn` over `tiles` tiles: as many warps as ONE block can have on
// an SM (they share the block's tile queue), bounded by the kernel's __launch_bounds__ and by shared memory
// (`per_warp` bytes each); MT_WARPS_PER_BLOCK overrides the target (tuning / A-B runs).  A launch with fewer
// tiles than that x SMs (small shards, the chunks of mt_step_host) uses smaller blocks, several per SM, so that
// it still spreads over every SM.
struct LaunchShape {
    int wpb = 0;
    unsigned grid = 0;
    size_t smem = 0;
};

static int plan_launch(mt_env *e, const void *fn, size_t per_warp, size_t extra, long long tiles, LaunchShape &out) {
    int max_wpb = 0;
    auto hit = e->block_shape.find(fn);
    if (hit != e->block_shape.end()) {
        max_wpb = hit->second;
    } else {
        max_wpb = e->arm == 0 ? kMaxWarpsRefArm : kMaxWarpsGeneric;
        if (const char *w = std::getenv("MT_WARPS_PER_BLOCK")) {
            const int v = std::atoi(w);
            if (v >= 1 && v <= max_wpb) max_wpb = v;
        }
        const size_t smem_cap = 227 * 1024 - 2048 - extra;        // per-SM limit minus the per-block reserve (and the action table)
        if ((size_t)max_wpb * per_warp > smem_cap) max_wpb = (int)(smem_cap / per_warp);
        if (max_wpb < 1) return fail(MT_ERR_CUDA, "step kernel does not fit on an SM (%zu B of shared memory per warp)", per_warp);
        const size_t smem_max = (size_t)max_wpb * per_warp + extra;
        if (smem_max > 48 * 1024) CU(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
        int per_sm = 0;
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, max_wpb * kTile, smem_max));
        if (per_sm < 1) return fail(MT_ERR_CUDA, "step kernel does not fit on an SM (%d warps, %zu B of shared memory)", max_wpb, smem_max);
        e->block_shape[fn] = max_wpb;
    }
    long long fair = (tiles + e->num_sms - 1) / e->num_sms;
    const int wpb = (int)(fair < 1 ? 1 : (fair > max_wpb ? max_wpb : fair));
    int per_sm = 1;                                               // blocks of this shape one SM can hold
    if (wpb < max_wpb || wpb < (e->arm == 0 ? kMaxWarpsRefArm : kMaxWarpsGeneric)) {
        const unsigned long long key = (unsigned long long)(uintptr_t)fn ^ ((unsigned long long)wpb << 52);
        auto occ = e->occupancy.find(key);
        if (occ != e->occupancy.end()) {
            per_sm = occ->second;
        } else {
            CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, wpb * kTile, (size_t)wpb * per_warp + extra));
            if (per_sm < 1) per_sm = 1;
            e->occupancy[key] = per_sm;
        }
    }
    const long long want = (tiles + wpb - 1) / wpb;
    const long long cap = (long long)per_sm * e->num_sms;
    out.wpb = wpb;
    out.grid = (unsigned)(want < cap ? want : cap);
    out.smem = (size_t)wpb * per_warp + extra;
    return MT_OK;
}

// programmatic dependent launch: see griddep_wait() in mt_ptx.cuh.  B: branch_kernel's second parameter
static int launch_pdl(const void *fn, const LaunchShape &shape, const StepParams &P, cudaStream_t st,
                      const BranchParams *B = nullptr) {
    cudaLaunchConfig_t lc = {};
    lc.gridDim = dim3(shape.grid);
    lc.blockDim = dim3(shape.wpb * kTile);
    lc.dynamicSmemBytes = shape.smem;
    lc.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    lc.attrs = attr;
    lc.numAttrs = 1;
    void *args[] = {(void *)&P, (void *)B};
    CU(cudaLaunchKernelExC(&lc, fn, args));
    return MT_OK;
}

// launch the fused step kernel over tiles [t0, t1): a persistent grid sized to the SMs.  final_obs != nullptr selects
// the FINAL = true kernel (mt_step_final), which also writes final_return / final_length.
static int launch_step(mt_env *e, const float *actions, void *obs, float *reward, uint8_t *done, float *joints,
                       bool rnd, long long t0, long long t1, cudaStream_t st, int ticket_slot = 0, bool advance = true,
                       void *final_obs = nullptr, float *final_return = nullptr, int32_t *final_length = nullptr) {
    StepParams P = e->base;
    P.actions = actions;
    P.obs = obs;
    P.reward = reward;
    P.done = done;
    P.joints = joints;
    P.obj_stream = e->obj_stream;
    P.obj_sets = e->obj_sets;
    P.tile_begin = t0;
    P.tile_end = t1;
    // device-side bookkeeping done by the launch's last block (mt_step.cuh, block_epilogue)
    P.ticket_slot = ticket_slot;
    P.advance = advance ? 1 : 0;
    P.n_steps = 1;
    P.launch_envs = ((t1 * kTile < e->n) ? t1 * kTile : e->n) - t0 * kTile;
    P.final_obs = final_obs;
    P.final_return = final_return;
    P.final_length = final_length;
    const bool wobs = obs != nullptr, final = final_obs != nullptr;
    const void *fn = nullptr;
    if (e->jit) {
        cudaKernel_t &k = e->jit_kernel[rnd ? 1 : 0][wobs ? 1 : 0][final ? 1 : 0];
        if (!k) {                                             // other variants compile on first use
            std::string err;
            k = jit_step_kernel(e->jit_preset, e->jit_id, e->jit_x, rnd, wobs, e->f16, final, err).kernel;
            if (!k) return fail(MT_ERR_CUDA, "run-time specialisation failed: %s", err.c_str());
        }
        fn = (const void *)k;
    } else {
        fn = (const void *)pick_kernel(e->arm, e->cfg.n_obj, rnd, wobs, e->f16, final);
    }
    if (!fn) return fail(MT_ERR_INVALID, "no kernel for arm=%d", e->arm);
    const size_t nb = e->arm == 0 ? StepBuffers<0>::value : StepBuffers<1>::value;   // tile buffers per warp
    P.trig_span = rnd ? trig_table_entries(e) : 0;
    LaunchShape shape;
    if (int rc = plan_launch(e, fn, nb * P.tile_bytes + nb * sizeof(uint64_t), (size_t)P.trig_span * 8, t1 - t0, shape)) return rc;
    if (int rc = launch_pdl(fn, shape, P, st)) return rc;
    e->launches++;
    return MT_OK;
}

// Multi-step rollout in ONE launch (rollout_kernel, mt_step.cuh): built-in arms and handles whose kernels come
// from NVRTC; run-time DH tables take the per-step launches instead (`launched` stays false).
// final: the FINAL = true kernels of mt_rollout_final, built only for the trajectory modes with observations written
template <int ARM, int X, RolloutMode MODE>
static StepFn pick_rollout_obs(bool wobs, bool f16, bool final) {
    if (final) {
        if constexpr (MODE == RolloutMode::kDrawLast) return nullptr;
        else if (!wobs) return nullptr;
        else return f16 ? rollout_kernel<ARM, X, true, true, MODE, true> : rollout_kernel<ARM, X, true, false, MODE, true>;
    }
    if (!wobs) return rollout_kernel<ARM, X, false, false, MODE, false>;
    return f16 ? rollout_kernel<ARM, X, true, true, MODE, false> : rollout_kernel<ARM, X, true, false, MODE, false>;
}

template <int ARM, int X>
static StepFn pick_rollout_mode(RolloutMode mode, bool wobs, bool f16, bool final) {
    switch (mode) {
        case RolloutMode::kDrawLast: return pick_rollout_obs<ARM, X, RolloutMode::kDrawLast>(wobs, f16, final);
        case RolloutMode::kDrawTrajectory: return pick_rollout_obs<ARM, X, RolloutMode::kDrawTrajectory>(wobs, f16, final);
        case RolloutMode::kActionsTrajectory: return pick_rollout_obs<ARM, X, RolloutMode::kActionsTrajectory>(wobs, f16, final);
    }
    return nullptr;
}

template <int ARM>
static StepFn pick_rollout_x(int x, RolloutMode mode, bool wobs, bool f16, bool final) {
    switch (x) {
        case 10: return pick_rollout_mode<ARM, 10>(mode, wobs, f16, final);
        case 20: return pick_rollout_mode<ARM, 20>(mode, wobs, f16, final);
        default: return pick_rollout_mode<ARM, 0>(mode, wobs, f16, final);
    }
}

static StepFn pick_rollout(int arm, int x, RolloutMode mode, bool wobs, bool f16, bool final) {
    switch (arm) {
        case 0: return pick_rollout_x<0>(x, mode, wobs, f16, final);
#define MT_PICK(ID) case ID: return pick_rollout_x<ID>(x, mode, wobs, f16, final);
        MT_FOR_EACH_PRESET_ARM(MT_PICK)
#undef MT_PICK
    }
    return nullptr;
}

// n_steps (<= 4096) steps of `mode` in one launch.  The trajectory modes take the bases of slice 0 (mt_rollout);
// final_obs != nullptr selects the FINAL = true kernel (mt_rollout_final), which also writes the final slices.
static int launch_rollout(mt_env *e, RolloutMode mode, int n_steps, const float *actions, float *drawn, void *obs,
                          float *reward, uint8_t *done, cudaStream_t st, bool &launched, void *final_obs = nullptr,
                          float *final_return = nullptr, int32_t *final_length = nullptr) {
    launched = false;
    if (n_steps < 2) return MT_OK;
    if (const char *v = std::getenv("MT_ROLLOUT_PERSISTENT"))
        if (v[0] == '0') return MT_OK;
    const bool final = final_obs != nullptr;
    const void *fn = nullptr;
    if (e->jit) {                                             // this handle's own table: compiled on first use
        if (e->jit_rollout_failed) return MT_OK;
        cudaKernel_t &k = e->jit_rollout[(int)mode][obs ? 1 : 0][final ? 1 : 0];
        if (!k) {
            std::string err;
            k = jit_step_kernel(e->jit_preset, e->jit_id, e->jit_x, true, obs != nullptr, e->f16, final, err, (int)mode).kernel;
            if (!k) {
                e->jit_rollout_failed = true;                 // keep working through the per-step launches
                return MT_OK;
            }
        }
        fn = (const void *)k;
    } else {
        fn = (const void *)pick_rollout(e->arm, e->cfg.n_obj, mode, obs != nullptr, e->f16, final);
    }
    if (!fn) return MT_OK;
    StepParams P = e->base;
    P.actions = actions;
    P.drawn = drawn;
    P.obs = obs;
    P.reward = reward;
    P.done = done;
    P.joints = nullptr;
    P.obj_stream = e->obj_stream;
    P.obj_sets = e->obj_sets;
    P.tile_begin = 0;
    P.tile_end = e->n_tiles;
    P.ticket_slot = 0;
    P.advance = n_steps;
    P.n_steps = n_steps;
    P.launch_envs = e->n * (long long)n_steps;
    P.final_obs = final_obs;
    P.final_return = final_return;
    P.final_length = final_length;
    const size_t nb = obs ? 2 : 1;                            // objectives (+ observations) per warp, one barrier
    P.trig_span = mode == RolloutMode::kActionsTrajectory ? 0 : trig_table_entries(e);   // the caller's actions: any float
    LaunchShape shape;
    if (int rc = plan_launch(e, fn, nb * P.tile_bytes + sizeof(uint64_t), (size_t)P.trig_span * 8, e->n_tiles, shape)) return rc;
    if (int rc = launch_pdl(fn, shape, P, st)) return rc;
    e->launches++;
    launched = true;
    return MT_OK;
}

static inline unsigned blocks_for(long long n, int bs = 256) { return (unsigned)((n + bs - 1) / bs); }

__global__ void mask_gap_kernel(const uint8_t *mask, long long n, int64_t *flag) {
    const long long env = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (env < n && !mask[env]) *flag = 1;
}

extern "C" int mt_reset(mt_env *e, const uint8_t *mask_dev, void *stream) {
    if (!e) return fail(MT_ERR_INVALID, "env is NULL");
    DeviceGuard guard(e->cfg.device);
    cudaStream_t st = (cudaStream_t)stream;
    if (mask_dev && !e->was_reset) {
        // The reference raises IndexError when an env that was never reset is stepped (manytor.py:143);
        // here the first reset has to cover every env, so that no env can be stepped with empty state.
        CU(cudaMemsetAsync(e->stats_dev, 0, 8, st));
        mask_gap_kernel<<<blocks_for(e->n), 256, 0, st>>>(mask_dev, e->n, e->stats_dev);
        CU(cudaMemcpyAsync(e->stats_pin, e->stats_dev, 8, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        if (e->stats_pin[0]) return fail(MT_ERR_STATE, "the first mt_reset must cover every env (mask leaves some env un-reset; the reference raises IndexError when such an env is stepped, manytor.py:143)");
    }
    StepParams P = e->base;
    P.obj_stream = e->obj_stream;
    P.obj_sets = e->obj_sets;
    reset_kernel<<<blocks_for(e->n), 256, 0, st>>>(P, mask_dev);
    CU(cudaGetLastError());
    e->launches++;
    e->was_reset = true;
    return MT_OK;
}

extern "C" int mt_observe(mt_env *e, void *obs_dev, void *stream) {
    if (!e) return fail(MT_ERR_INVALID, "env is NULL");
    if (int rc = check_ptr(obs_dev, "obs_dev", true)) return rc;
    if (!e->was_reset) return fail(MT_ERR_STATE, "mt_observe before mt_reset (the reference raises IndexError here, manytor.py:143)");
    DeviceGuard guard(e->cfg.device);
    (e->f16 ? observe_kernel<true> : observe_kernel<false>)<<<blocks_for(e->n, 128), 128, 0, (cudaStream_t)stream>>>(
        e->base, e->arm, obs_dev);
    CU(cudaGetLastError());
    e->launches++;
    return MT_OK;
}

static int timing_begin(mt_env *e, cudaStream_t st) {
    if (!e->timing) return MT_OK;
    if (!e->ev0) { CU(cudaEventCreate(&e->ev0)); CU(cudaEventCreate(&e->ev1)); }
    CU(cudaEventRecord(e->ev0, st));
    return MT_OK;
}
static int timing_end(mt_env *e, cudaStream_t st) {
    if (!e->timing) return MT_OK;
    CU(cudaEventRecord(e->ev1, st));
    e->ev_valid = true;
    return MT_OK;
}

extern "C" int mt_step(mt_env *e, const float *actions_dev, void *obs_dev, float *reward_dev, uint8_t *done_dev,
                       float *joints_dev, void *stream) {
    if (!e) return fail(MT_ERR_INVALID, "env is NULL");
    if (!e->was_reset) return fail(MT_ERR_STATE, "mt_step before mt_reset (the reference raises IndexError here, manytor.py:143)");
    int rc;
    if ((rc = check_ptr(actions_dev, "actions_dev", true))) return rc;
    if ((rc = check_ptr(obs_dev, "obs_dev", false))) return rc;
    if (!reward_dev || !done_dev) return fail(MT_ERR_INVALID, "reward_dev/done_dev is NULL");
    DeviceGuard guard(e->cfg.device);
    cudaStream_t st = (cudaStream_t)stream;
    if ((rc = timing_begin(e, st))) return rc;
    if ((rc = launch_step(e, actions_dev, obs_dev, reward_dev, done_dev, joints_dev, false, 0, e->n_tiles, st))) return rc;
    return timing_end(e, st);
}

extern "C" int mt_step_final(mt_env *e, const float *actions_dev, void *obs_dev, float *reward_dev, uint8_t *done_dev,
                             float *joints_dev, void *final_obs_dev, float *final_return_dev, int32_t *final_length_dev,
                             void *stream) {
    // the arguments first: none of these checks needs the handle or a device
    int rc;
    if ((rc = check_ptr(actions_dev, "actions_dev", true))) return rc;
    if ((rc = check_ptr(obs_dev, "obs_dev", true))) return rc;
    if (!reward_dev || !done_dev) return fail(MT_ERR_INVALID, "reward_dev/done_dev is NULL");
    if ((rc = check_ptr(final_obs_dev, "final_obs_dev", true))) return rc;
    if ((rc = check_ptr(final_return_dev, "final_return_dev", true))) return rc;
    if ((rc = check_ptr(final_length_dev, "final_length_dev", true))) return rc;
    if (!e) return fail(MT_ERR_INVALID, "env is NULL");
    if (!e->cfg.auto_reset)
        return fail(MT_ERR_INVALID, "mt_step_final needs a handle created with auto_reset (without it obs2 is the returned "
                                    "observation and mt_get_state holds the return and length)");
    if (!e->was_reset) return fail(MT_ERR_STATE, "mt_step_final before mt_reset (the reference raises IndexError here, manytor.py:143)");
    DeviceGuard guard(e->cfg.device);
    cudaStream_t st = (cudaStream_t)stream;
    if ((rc = timing_begin(e, st))) return rc;
    if ((rc = launch_step(e, actions_dev, obs_dev, reward_dev, done_dev, joints_dev, false, 0, e->n_tiles, st, 0, true,
                          final_obs_dev, final_return_dev, final_length_dev)))
        return rc;
    return timing_end(e, st);
}

extern "C" int mt_sample_actions(mt_env *e, float *actions_dev, void *stream) {
    if (!e) return fail(MT_ERR_INVALID, "env is NULL");
    if (int rc = check_ptr(actions_dev, "actions_dev", true)) return rc;
    DeviceGuard guard(e->cfg.device);
    sample_actions_kernel<<<blocks_for(e->n), 256, 0, (cudaStream_t)stream>>>(e->base, actions_dev);
    CU(cudaGetLastError());
    e->launches++;
    return MT_OK;
}

extern "C" int mt_rollout_random(mt_env *e, int32_t n_steps, void *obs_dev, float *reward_dev, uint8_t *done_dev,
                                 void *stream) {
    if (!e) return fail(MT_ERR_INVALID, "env is NULL");
    if (!e->was_reset) return fail(MT_ERR_STATE, "mt_rollout_random before mt_reset");
    if (n_steps < 0) return fail(MT_ERR_INVALID, "n_steps < 0");
    int rc;
    if ((rc = check_ptr(obs_dev, "obs_dev", false))) return rc;
    DeviceGuard guard(e->cfg.device);
    if (!reward_dev || !done_dev) {                   // outputs nobody reads: buffers the handle owns
        if (!e->scratch_reward) {
            CU(cudaMalloc((void **)&e->scratch_reward, (size_t)e->n_pad * 4));
            CU(cudaMalloc((void **)&e->scratch_done, (size_t)e->n_pad));
        }
        if (!reward_dev) reward_dev = e->scratch_reward;
        if (!done_dev) done_dev = e->scratch_done;
    }
    cudaStream_t st = (cudaStream_t)stream;
    if ((rc = timing_begin(e, st))) return rc;
    // chunks of at most 4096 steps per launch keep a launch's work bounded (a tile's warp holds it for the chunk)
    for (int s = 0; s < n_steps;) {
        const int chunk = n_steps - s < 4096 ? n_steps - s : 4096;
        bool launched = false;
        if ((rc = launch_rollout(e, RolloutMode::kDrawLast, chunk, nullptr, nullptr, obs_dev, reward_dev, done_dev, st, launched)))
            return rc;
        if (launched) {
            s += chunk;
        } else {
            if ((rc = launch_step(e, nullptr, obs_dev, reward_dev, done_dev, nullptr, true, 0, e->n_tiles, st))) return rc;
            ++s;
        }
    }
    return timing_end(e, st);
}

// One step of mt_rollout through the step kernel, into the slice pointers of that step.  step_kernel bulk-stores
// every full observation tile, so a slice whose base may not take a bulk copy (obs_bulk_ok false) gets the step's
// observations through the handle's own buffer and one device-to-device copy.  The final observations
// (mt_rollout_final) are stored lane by lane and go to their slice directly.  step_kernel<.., FINAL = true> exists
// for the caller's actions only, so in-kernel draws are drawn first, as mt_sample_actions draws them at this step
// index, and stepped as the caller's actions: bit for bit the same step, as the ActionTrig table is bit for bit the
// kernel's own sin / cos evaluation (fill_action_trig).
static int rollout_one_step(mt_env *e, const float *actions, float *drawn, void *obs, bool obs_bulk_ok, float *reward,
                            uint8_t *done, cudaStream_t st, void *final_obs, float *final_return, int32_t *final_length) {
    if (!actions && final_obs && !drawn) {
        if (!e->scratch_actions) CU(cudaMalloc((void **)&e->scratch_actions, (size_t)e->n * e->cfg.n_joints * 4));
        drawn = e->scratch_actions;
    }
    if (!actions && drawn) {                          // what mt_sample_actions returns at this step index
        sample_actions_kernel<<<blocks_for(e->n), 256, 0, st>>>(e->base, drawn);
        CU(cudaGetLastError());
        e->launches++;
        if (final_obs) actions = drawn;
    }
    const size_t obs_bytes = (size_t)e->n * 3 * e->cfg.n_obj * (e->f16 ? 2 : 4);
    void *dst = obs;
    if (obs && !obs_bulk_ok) {
        if (!e->scratch_obs) CU(cudaMalloc(&e->scratch_obs, obs_bytes));
        dst = e->scratch_obs;
    }
    if (int rc = launch_step(e, actions, dst, reward, done, nullptr, actions == nullptr, 0, e->n_tiles, st, 0, true,
                             final_obs, final_return, final_length))
        return rc;
    if (dst != obs) CU(cudaMemcpyAsync(obs, dst, obs_bytes, cudaMemcpyDeviceToDevice, st));
    return MT_OK;
}

// The chunk loop of mt_rollout and mt_rollout_final (that of mt_rollout_random, with slices): every pointer below is
// the base of slice s (64-bit offsets).  final_obs = nullptr: mt_rollout.
static int rollout_trajectory(mt_env *e, int32_t n_steps, const float *actions_dev, float *drawn_dev, void *obs_dev,
                              float *reward_dev, uint8_t *done_dev, void *final_obs_dev, float *final_return_dev,
                              int32_t *final_length_dev, cudaStream_t st) {
    const RolloutMode mode = actions_dev ? RolloutMode::kActionsTrajectory : RolloutMode::kDrawTrajectory;
    const size_t n = (size_t)e->n, J = (size_t)e->cfg.n_joints, obs_row = (size_t)3 * e->cfg.n_obj * (e->f16 ? 2 : 4);
    int rc;
    if ((rc = timing_begin(e, st))) return rc;
    for (int s = 0; s < n_steps;) {
        const int chunk = n_steps - s < 4096 ? n_steps - s : 4096;
        const size_t rows = (size_t)s * n;
        const float *a = actions_dev ? actions_dev + rows * J : nullptr;
        float *d = drawn_dev ? drawn_dev + rows * J : nullptr;
        void *o = obs_dev ? (void *)((char *)obs_dev + rows * obs_row) : nullptr;
        void *fo = final_obs_dev ? (void *)((char *)final_obs_dev + rows * obs_row) : nullptr;
        float *fr = final_obs_dev ? final_return_dev + rows : nullptr;
        int32_t *fl = final_obs_dev ? final_length_dev + rows : nullptr;
        bool launched = false;
        if ((rc = launch_rollout(e, mode, chunk, a, d, o, reward_dev + rows, done_dev + rows, st, launched, fo, fr, fl)))
            return rc;
        if (launched) {
            s += chunk;
        } else {
            const bool bulk_ok = slice_bulk_ok((uintptr_t)obs_dev, (unsigned long long)s, n, 0, obs_row);
            if ((rc = rollout_one_step(e, a, d, o, bulk_ok, reward_dev + rows, done_dev + rows, st, fo, fr, fl))) return rc;
            ++s;
        }
    }
    return timing_end(e, st);
}

extern "C" int mt_rollout(mt_env *e, int32_t n_steps, const float *actions_dev, float *drawn_dev, void *obs_dev,
                          float *reward_dev, uint8_t *done_dev, void *stream) {
    // the arguments first: none of these checks needs the handle or a device
    if (n_steps < 0) return fail(MT_ERR_INVALID, "n_steps < 0");
    int rc;
    if ((rc = check_ptr(actions_dev, "actions_dev", false))) return rc;
    if ((rc = check_ptr(drawn_dev, "drawn_dev", false))) return rc;
    if (actions_dev && drawn_dev) return fail(MT_ERR_INVALID, "drawn_dev must be NULL when actions_dev is given");
    if ((rc = check_ptr(obs_dev, "obs_dev", false))) return rc;
    if ((rc = check_ptr(reward_dev, "reward_dev", true))) return rc;
    if ((rc = check_ptr(done_dev, "done_dev", true))) return rc;
    if (!e) return fail(MT_ERR_INVALID, "env is NULL");
    if (!e->was_reset) return fail(MT_ERR_STATE, "mt_rollout before mt_reset");
    if (n_steps == 0) return MT_OK;
    DeviceGuard guard(e->cfg.device);
    return rollout_trajectory(e, n_steps, actions_dev, drawn_dev, obs_dev, reward_dev, done_dev, nullptr, nullptr, nullptr,
                              (cudaStream_t)stream);
}

extern "C" int mt_rollout_final(mt_env *e, int32_t n_steps, const float *actions_dev, float *drawn_dev, void *obs_dev,
                                float *reward_dev, uint8_t *done_dev, void *final_obs_dev, float *final_return_dev,
                                int32_t *final_length_dev, void *stream) {
    // the arguments first, in mt_rollout's order and then mt_step_final's: none of these checks needs the handle
    if (n_steps < 0) return fail(MT_ERR_INVALID, "n_steps < 0");
    int rc;
    if ((rc = check_ptr(actions_dev, "actions_dev", false))) return rc;
    if ((rc = check_ptr(drawn_dev, "drawn_dev", false))) return rc;
    if (actions_dev && drawn_dev) return fail(MT_ERR_INVALID, "drawn_dev must be NULL when actions_dev is given");
    if ((rc = check_ptr(obs_dev, "obs_dev", true))) return rc;
    if ((rc = check_ptr(reward_dev, "reward_dev", true))) return rc;
    if ((rc = check_ptr(done_dev, "done_dev", true))) return rc;
    if ((rc = check_ptr(final_obs_dev, "final_obs_dev", true))) return rc;
    if ((rc = check_ptr(final_return_dev, "final_return_dev", true))) return rc;
    if ((rc = check_ptr(final_length_dev, "final_length_dev", true))) return rc;
    if (!e) return fail(MT_ERR_INVALID, "env is NULL");
    if (!e->cfg.auto_reset)
        return fail(MT_ERR_INVALID, "mt_rollout_final needs a handle created with auto_reset (without it obs2 is the "
                                    "returned observation and mt_get_state holds the return and length)");
    if (!e->was_reset) return fail(MT_ERR_STATE, "mt_rollout_final before mt_reset");
    if (n_steps == 0) return MT_OK;
    DeviceGuard guard(e->cfg.device);
    return rollout_trajectory(e, n_steps, actions_dev, drawn_dev, obs_dev, reward_dev, done_dev, final_obs_dev,
                              final_return_dev, final_length_dev, (cudaStream_t)stream);
}

// Branch kernels (branch_kernel, mt_step.cuh): the built-in arms at X = 10, 20 and run time, as pick_rollout; every other
// DH table -- run-time tables and the tables of NVRTC handles alike (`arm` is J for both, StepParams::arm holds the
// table) -- through the run-time-table instantiation ARM = J, X = 0.
// DRAW: the kernels of mt_rollout_branches_random (in-kernel draws after the caller's prefix).
template <int ARM, int X, bool DRAW>
static BranchFn pick_branch_obs(bool wobs, bool f16) {
    if (!wobs) return branch_kernel<ARM, X, false, false, DRAW>;
    return f16 ? branch_kernel<ARM, X, true, true, DRAW> : branch_kernel<ARM, X, true, false, DRAW>;
}

template <int ARM, bool DRAW>
static BranchFn pick_branch_x(int x, bool wobs, bool f16) {
    switch (x) {
        case 10: return pick_branch_obs<ARM, 10, DRAW>(wobs, f16);
        case 20: return pick_branch_obs<ARM, 20, DRAW>(wobs, f16);
        default: return pick_branch_obs<ARM, 0, DRAW>(wobs, f16);
    }
}

template <bool DRAW>
static BranchFn pick_branch(int arm, int x, bool wobs, bool f16) {
    switch (arm) {
        case 0: return pick_branch_x<0, DRAW>(x, wobs, f16);
        case 2: return pick_branch_obs<2, 0, DRAW>(wobs, f16);
        case 3: return pick_branch_obs<3, 0, DRAW>(wobs, f16);
        case 4: return pick_branch_obs<4, 0, DRAW>(wobs, f16);
        case 5: return pick_branch_obs<5, 0, DRAW>(wobs, f16);
        case 6: return pick_branch_obs<6, 0, DRAW>(wobs, f16);
        case 7: return pick_branch_obs<7, 0, DRAW>(wobs, f16);
        case 8: return pick_branch_obs<8, 0, DRAW>(wobs, f16);
#define MT_PICK(ID) case ID: return pick_branch_x<ID, DRAW>(x, wobs, f16);
        MT_FOR_EACH_PRESET_ARM(MT_PICK)
#undef MT_PICK
    }
    return nullptr;
}

constexpr long long kMaxBranches = 2000000000ll;   // the 32-bit env index of mt_create

extern "C" int mt_rollout_branches(mt_env *e, int32_t n_steps, int64_t n_branches, const int64_t *src_dev,
                                   const float *actions_dev, float gamma, float *return_dev, int32_t *length_dev,
                                   uint8_t *done_dev, void *obs_dev, void *stream) {
    // the arguments first: none of these checks needs the handle or a device
    if (n_steps < 0 || n_steps > 4096) return fail(MT_ERR_INVALID, "n_steps must be in [0, 4096]");
    if (n_branches < 0 || n_branches > kMaxBranches) return fail(MT_ERR_INVALID, "n_branches must be in [0, 2000000000]");
    if (!(gamma >= 0.0f && gamma <= 1.0f)) return fail(MT_ERR_INVALID, "gamma must be finite and in [0, 1]");
    int rc;
    if ((rc = check_ptr(src_dev, "src_dev", true))) return rc;
    if ((rc = check_ptr(actions_dev, "actions_dev", true))) return rc;
    if ((rc = check_ptr(return_dev, "return_dev", true))) return rc;
    if ((rc = check_ptr(length_dev, "length_dev", true))) return rc;
    if ((rc = check_ptr(done_dev, "done_dev", true))) return rc;
    if ((rc = check_ptr(obs_dev, "obs_dev", false))) return rc;
    if (!e) return fail(MT_ERR_INVALID, "env is NULL");
    if (!e->was_reset) return fail(MT_ERR_STATE, "mt_rollout_branches before mt_reset");
    if (n_steps == 0 || n_branches == 0) return MT_OK;
    DeviceGuard guard(e->cfg.device);
    const bool wobs = obs_dev != nullptr;
    const void *fn = (const void *)pick_branch<false>(e->arm, e->cfg.n_obj, wobs, e->f16);
    if (!fn) return fail(MT_ERR_INVALID, "no branch kernel for arm=%d", e->arm);
    StepParams P = e->base;
    P.flags &= ~kAutoReset;                       // settle_step then resets nothing and writes nothing
    P.actions = actions_dev;
    P.obs = obs_dev;
    P.done = done_dev;
    P.n_steps = n_steps;
    P.tile_begin = 0;
    P.tile_end = (n_branches + kTile - 1) / kTile;
    const BranchParams B{src_dev, return_dev, length_dev, (long long)n_branches, gamma};
    const size_t nb = wobs ? 2 : 1;               // objectives (+ observations) per warp
    LaunchShape shape;
    if ((rc = plan_launch(e, fn, nb * P.tile_bytes, 0, P.tile_end, shape))) return rc;
    if ((rc = launch_pdl(fn, shape, P, (cudaStream_t)stream, &B))) return rc;
    e->launches++;
    return MT_OK;
}

// The draw key is one uint64 word on the device, read by the kernels: 8-byte alignment is all it needs.
static int check_key(const uint64_t *key) {
    if (!key) return fail(MT_ERR_INVALID, "draw_key_dev is NULL");
    if (((uintptr_t)key & 7u) != 0) return fail(MT_ERR_INVALID, "draw_key_dev must be 8-byte aligned");
    return MT_OK;
}

extern "C" int mt_rollout_branches_random(mt_env *e, int32_t n_steps, int32_t n_prefix, int64_t n_branches,
                                          const int64_t *src_dev, const float *prefix_dev, const uint64_t *draw_key_dev,
                                          float gamma, float *return_dev, int32_t *length_dev, uint8_t *done_dev,
                                          void *obs_dev, void *stream) {
    // the arguments first, in mt_rollout_branches' order: none of these checks needs the handle or a device
    if (n_steps < 0 || n_steps > 4096) return fail(MT_ERR_INVALID, "n_steps must be in [0, 4096]");
    if (n_prefix < 0 || n_prefix > n_steps) return fail(MT_ERR_INVALID, "n_prefix must be in [0, n_steps]");
    if (n_branches < 0 || n_branches > kMaxBranches) return fail(MT_ERR_INVALID, "n_branches must be in [0, 2000000000]");
    if (!(gamma >= 0.0f && gamma <= 1.0f)) return fail(MT_ERR_INVALID, "gamma must be finite and in [0, 1]");
    int rc;
    if ((rc = check_ptr(src_dev, "src_dev", true))) return rc;
    if ((rc = check_ptr(prefix_dev, "prefix_dev", n_prefix > 0))) return rc;
    if (n_prefix == 0 && prefix_dev) return fail(MT_ERR_INVALID, "prefix_dev must be NULL when n_prefix is 0");
    if ((rc = check_key(draw_key_dev))) return rc;
    if ((rc = check_ptr(return_dev, "return_dev", true))) return rc;
    if ((rc = check_ptr(length_dev, "length_dev", true))) return rc;
    if ((rc = check_ptr(done_dev, "done_dev", true))) return rc;
    if ((rc = check_ptr(obs_dev, "obs_dev", false))) return rc;
    if (!e) return fail(MT_ERR_INVALID, "env is NULL");
    if (!e->was_reset) return fail(MT_ERR_STATE, "mt_rollout_branches_random before mt_reset");
    if (n_steps == 0 || n_branches == 0) return MT_OK;
    DeviceGuard guard(e->cfg.device);
    const bool wobs = obs_dev != nullptr;
    const void *fn = (const void *)pick_branch<true>(e->arm, e->cfg.n_obj, wobs, e->f16);
    if (!fn) return fail(MT_ERR_INVALID, "no branch kernel for arm=%d", e->arm);
    StepParams P = e->base;
    P.flags &= ~kAutoReset;                       // settle_step then resets nothing and writes nothing
    P.actions = prefix_dev;
    P.obs = obs_dev;
    P.done = done_dev;
    P.n_steps = n_steps;
    P.tile_begin = 0;
    P.tile_end = (n_branches + kTile - 1) / kTile;
    P.trig_span = trig_table_entries(e);          // the drawn steps' sin / cos table, after the per-warp buffers
    const BranchParams B{src_dev, return_dev, length_dev, (long long)n_branches, gamma, n_prefix,
                         reinterpret_cast<const unsigned long long *>(draw_key_dev)};
    const size_t nb = wobs ? 2 : 1;               // objectives (+ observations) per warp
    LaunchShape shape;
    if ((rc = plan_launch(e, fn, nb * P.tile_bytes, (size_t)P.trig_span * 8, P.tile_end, shape))) return rc;
    if ((rc = launch_pdl(fn, shape, P, (cudaStream_t)stream, &B))) return rc;
    e->launches++;
    return MT_OK;
}

extern "C" int mt_branch_actions(mt_env *e, const uint64_t *draw_key_dev, int32_t first_step, int32_t n_steps,
                                 int64_t n_rows, const int64_t *branch_dev, float *out_dev, void *stream) {
    // the arguments first: none of these checks needs the handle or a device
    int rc;
    if ((rc = check_key(draw_key_dev))) return rc;
    if (first_step < 0) return fail(MT_ERR_INVALID, "first_step must be >= 0");
    if (n_steps < 0) return fail(MT_ERR_INVALID, "n_steps must be >= 0");
    if (n_rows < 0 || n_rows > kMaxBranches) return fail(MT_ERR_INVALID, "n_rows must be in [0, 2000000000]");
    if ((rc = check_ptr(branch_dev, "branch_dev", true))) return rc;
    if ((rc = check_ptr(out_dev, "out_dev", true))) return rc;
    if (!e) return fail(MT_ERR_INVALID, "env is NULL");
    if (n_steps == 0 || n_rows == 0) return MT_OK;
    DeviceGuard guard(e->cfg.device);
    const long long total = (long long)n_steps * n_rows;
    const long long blocks = (total + 255) / 256, cap = (long long)e->num_sms * 64;
    branch_actions_kernel<<<(unsigned)(blocks < cap ? blocks : cap), 256, 0, (cudaStream_t)stream>>>(
        e->base, reinterpret_cast<const unsigned long long *>(draw_key_dev), first_step, n_steps, n_rows, branch_dev, out_dev);
    CU(cudaGetLastError());
    e->launches++;
    return MT_OK;
}

extern "C" int mt_host_alloc(void **out, uint64_t bytes) {
    if (!out) return fail(MT_ERR_INVALID, "out is NULL");
    CU(cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocPortable | cudaHostAllocMapped));
    return MT_OK;
}
extern "C" int mt_host_free(void *p) {
    if (p) CU(cudaFreeHost(p));
    return MT_OK;
}

// Host-buffer step, two variants.
//   staged     chunks of whole tiles round-robin over internal streams, each chunk H2D(actions) -> step kernel ->
//              D2H(observations), then reward/done in two copies at the end; the copies of one chunk overlap the
//              kernels and copies of the others.
//   zero-copy  ONE step launch on the pinned host buffers themselves: the kernel reads the actions and bulk-stores
//              the observations across PCIe, no staging copy, no chunking.
// Either way the call is bound by the PCIe read-back of the observations (120 of the 125 B per env).  Which one is
// faster depends on the box: alone on a link staging wins (93 % vs 87 % of the link), with 8 GPUs sharing the host's
// 93 GB/s zero-copy does (99 % vs 94 %).  So by default the handle TIMES both on its first six calls (the call is
// synchronous, results are identical) and keeps the faster; MT_HOST_ZEROCOPY=0/1 pins the choice.  The internal
// streams are ordered after everything submitted earlier to blocking streams (an event on the legacy default stream),
// not by a device-wide synchronisation.
static bool device_visible_host(const void *p) {
    if (!p) return true;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        (void)cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeHost && a.devicePointer == p && ((uintptr_t)p & 15u) == 0;
}

extern "C" int mt_step_host(mt_env *e, const float *actions_host, void *obs_host, float *reward_host,
                            uint8_t *done_host) {
    if (!e) return fail(MT_ERR_INVALID, "env is NULL");
    if (!e->was_reset) return fail(MT_ERR_STATE, "mt_step_host before mt_reset");
    if (!actions_host || !reward_host || !done_host) return fail(MT_ERR_INVALID, "NULL host buffer");
    DeviceGuard guard(e->cfg.device);
    const size_t J = e->cfg.n_joints, R = 3 * (size_t)e->cfg.n_obj * (e->f16 ? 2 : 4);   // R: bytes per observation row
    if (!e->hs[0]) {
        for (auto &s : e->hs) CU(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
        for (auto &v : e->hev) CU(cudaEventCreateWithFlags(&v, cudaEventDisableTiming));
        if (const char *zc = std::getenv("MT_HOST_ZEROCOPY"))
            if (zc[0] == '0' || zc[0] == '1') e->host_mode = zc[0] - '0';
    }
    // calls 0-2 staged, 3-5 zero-copy (the first of each triple untimed: allocations, first-touch; the better of the
    // other two counts), then the faster variant
    const int call = e->host_calls;
    bool zero_copy = e->host_mode == 1 || (e->host_mode == 2 && call >= 3);
    if (zero_copy && !(device_visible_host(actions_host) && device_visible_host(obs_host) && device_visible_host(reward_host) &&
                       device_visible_host(done_host))) {
        if (e->host_mode == 1) return fail(MT_ERR_INVALID, "MT_HOST_ZEROCOPY=1 needs buffers from mt_host_alloc (pinned, mapped, 16-byte aligned)");
        e->host_mode = 0;                                     // pageable or unaligned buffers: staging only
        zero_copy = false;
    }
    const auto t_begin = std::chrono::steady_clock::now();
    auto finish = [&]() {
        if (e->host_mode != 2) return;
        const double dt = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_begin).count();
        if (call % 3 != 0 && dt < e->host_best[zero_copy ? 1 : 0]) e->host_best[zero_copy ? 1 : 0] = dt;
        if (++e->host_calls == 6) e->host_mode = e->host_best[1] < 0.98 * e->host_best[0] ? 1 : 0;
    };
    if (zero_copy) {
        // one launch on the legacy stream: ordered after everything submitted so far on blocking streams, like the
        // event fence of the staged variant below, without the two extra calls (a batch of one env is pure latency)
        if (int rc = launch_step(e, actions_host, obs_host, reward_host, done_host, nullptr, false, 0, e->n_tiles, nullptr))
            return rc;
        CU(cudaStreamSynchronize(nullptr));
        finish();
        return MT_OK;
    }
    CU(cudaEventRecord(e->hev[mt_env::kStreams], nullptr));       // everything submitted so far (blocking streams)
    if (!e->h_actions) {
        CU(cudaMalloc((void **)&e->h_actions, (size_t)e->n_pad * J * 4));
        CU(cudaMalloc(&e->h_obs, (size_t)e->n_pad * R));
        CU(cudaMalloc((void **)&e->h_reward, (size_t)e->n_pad * 4));
        CU(cudaMalloc((void **)&e->h_done, (size_t)e->n_pad));
    }
    for (auto &s : e->hs) CU(cudaStreamWaitEvent(s, e->hev[mt_env::kStreams], 0));
    const long long chunks = e->n_tiles < 16 ? 1 : 16;
    const long long per = (e->n_tiles + chunks - 1) / chunks;
    int k = 0;
    for (long long t0 = 0; t0 < e->n_tiles; t0 += per, ++k) {
        const long long t1 = (t0 + per < e->n_tiles) ? t0 + per : e->n_tiles;
        const long long e0 = t0 * kTile, e1 = (t1 * kTile < e->n) ? t1 * kTile : e->n, cnt = e1 - e0;
        cudaStream_t st = e->hs[k % mt_env::kStreams];
        CU(cudaMemcpyAsync(e->h_actions + e0 * J, actions_host + e0 * J, cnt * J * 4, cudaMemcpyHostToDevice, st));
        // every chunk has its own launch ticket (the chunks overlap in time); the last one completes the step
        if (int rc = launch_step(e, e->h_actions, obs_host ? e->h_obs : nullptr, e->h_reward, e->h_done, nullptr, false,
                                 t0, t1, st, 1 + k, t1 == e->n_tiles))
            return rc;
        if (obs_host)
            CU(cudaMemcpyAsync((char *)obs_host + e0 * R, (char *)e->h_obs + e0 * R, cnt * R, cudaMemcpyDeviceToHost, st));
    }
    // reward / done of the whole shard: two copies once every chunk's kernel has run
    for (int i = 1; i < mt_env::kStreams; ++i) {
        CU(cudaEventRecord(e->hev[i], e->hs[i]));
        CU(cudaStreamWaitEvent(e->hs[0], e->hev[i], 0));
    }
    CU(cudaMemcpyAsync(reward_host, e->h_reward, (size_t)e->n * 4, cudaMemcpyDeviceToHost, e->hs[0]));
    CU(cudaMemcpyAsync(done_host, e->h_done, (size_t)e->n, cudaMemcpyDeviceToHost, e->hs[0]));
    CU(cudaStreamSynchronize(e->hs[0]));
    finish();
    return MT_OK;
}

// which variant mt_step_host uses: 0 staged, 1 zero-copy, 2 still deciding (see above)
extern "C" int mt_host_step_mode(const mt_env *e) { return e ? e->host_mode : -1; }

extern "C" int mt_set_points(mt_env *e, const float *points_dev, const uint8_t *mask_dev, void *stream) {
    if (!e || !points_dev) return fail(MT_ERR_INVALID, "NULL argument");
    DeviceGuard guard(e->cfg.device);
    set_points_kernel<<<blocks_for(e->n * 3 * e->cfg.n_obj), 256, 0, (cudaStream_t)stream>>>(e->base, points_dev, mask_dev);
    CU(cudaGetLastError());
    e->launches++;
    return MT_OK;
}

extern "C" int mt_get_points(mt_env *e, float *points_dev, int32_t zero_dead, void *stream) {
    if (!e || !points_dev) return fail(MT_ERR_INVALID, "NULL argument");
    DeviceGuard guard(e->cfg.device);
    get_points_kernel<<<blocks_for(e->n * 3 * e->cfg.n_obj), 256, 0, (cudaStream_t)stream>>>(e->base, points_dev, zero_dead);
    CU(cudaGetLastError());
    e->launches++;
    return MT_OK;
}

extern "C" int mt_set_state(mt_env *e, const float *goals_dev, const uint32_t *alive_dev, const float *total_reward_dev,
                            const int32_t *ep_len_dev, const uint8_t *mask_dev, void *stream) {
    if (!e) return fail(MT_ERR_INVALID, "env is NULL");
    DeviceGuard guard(e->cfg.device);
    set_state_kernel<<<blocks_for(e->n), 256, 0, (cudaStream_t)stream>>>(e->base, goals_dev, alive_dev, total_reward_dev,
                                                                          ep_len_dev, mask_dev);
    CU(cudaGetLastError());
    e->launches++;
    return MT_OK;
}

extern "C" int mt_get_state(mt_env *e, float *goals_dev, uint32_t *alive_dev, float *total_reward_dev,
                            int32_t *ep_len_dev, void *stream) {
    if (!e) return fail(MT_ERR_INVALID, "env is NULL");
    DeviceGuard guard(e->cfg.device);
    get_state_kernel<<<blocks_for(e->n), 256, 0, (cudaStream_t)stream>>>(e->base, goals_dev, alive_dev, total_reward_dev,
                                                                          ep_len_dev);
    CU(cudaGetLastError());
    e->launches++;
    return MT_OK;
}

// The per-env reset counts (StepParams::episode): they key sample_point and pick the objective-stream set, so a
// checkpoint needs them next to mt_get_state.
extern "C" int mt_get_reset_counts(mt_env *e, uint32_t *counts_dev, void *stream) {
    if (!counts_dev) return fail(MT_ERR_INVALID, "counts_dev is NULL");
    if (!e) return fail(MT_ERR_INVALID, "env is NULL");
    DeviceGuard guard(e->cfg.device);
    get_reset_counts_kernel<<<blocks_for(e->n), 256, 0, (cudaStream_t)stream>>>(e->base, counts_dev);
    CU(cudaGetLastError());
    e->launches++;
    return MT_OK;
}

extern "C" int mt_set_reset_counts(mt_env *e, const uint32_t *counts_dev, const uint8_t *mask_dev, void *stream) {
    if (!counts_dev) return fail(MT_ERR_INVALID, "counts_dev is NULL");
    if (!e) return fail(MT_ERR_INVALID, "env is NULL");
    DeviceGuard guard(e->cfg.device);
    set_reset_counts_kernel<<<blocks_for(e->n), 256, 0, (cudaStream_t)stream>>>(e->base, counts_dev, mask_dev);
    CU(cudaGetLastError());
    e->launches++;
    return MT_OK;
}

extern "C" int mt_set_objective_stream(mt_env *e, const float *points_dev, int32_t n_sets) {
    if (!e) return fail(MT_ERR_INVALID, "env is NULL");
    if (points_dev && n_sets < 1) return fail(MT_ERR_INVALID, "n_sets must be >= 1");
    e->obj_stream = points_dev;
    e->obj_sets = points_dev ? n_sets : 0;
    return MT_OK;
}

// one env's state packed into the handle's scratch: goals[J] | joints[J][3] | points[X][3] (dead -> 0) | alive | total
__global__ void fetch_kernel(const __grid_constant__ StepParams P, int arm, long long index, float *out) {
    const int J = P.n_joints, X = P.n_obj, lane = threadIdx.x;
    const uint32_t alive = alive_mask_of(P, P.alive[index]);
    float *goals = out, *joints = out + J, *points = out + J * 4, *tail = out + J * 4 + X * 3;
    if (lane == 0) {
        float g[MT_MAX_JOINTS], jb[MT_MAX_JOINTS * 3];
        for (int k = 0; k < J; ++k) goals[k] = g[k] = P.goals[index * J + k];
        Frames f;
        pose_of(P, arm, g, f, jb);
        for (int k = 0; k < J * 3; ++k) joints[k] = jb[k];
        tail[0] = __uint_as_float(alive);
        tail[1] = P.total_reward[index];
    }
    for (int i = lane; i < X * 3; i += 32) {                                // dead objectives read as zeros, manytor.py:148
        const int pt = i / 3;
        points[i] = ((alive >> pt) & 1u) ? P.points[index * 3 * X + point_index(P.pair_layout != 0, pt, i % 3)] : 0.f;
    }
}

// Synchronous, on the legacy default stream (ordered after everything submitted to blocking streams):
// one small kernel into the handle's scratch and one copy to its pinned mirror -- no allocation and no
// device-wide synchronisation per call.
extern "C" int mt_fetch_env(mt_env *e, int64_t index, float *goals_host, float *joints_host, float *points_host,
                            uint32_t *alive_host, float *total_reward_host) {
    if (!e) return fail(MT_ERR_INVALID, "env is NULL");
    if (index < 0 || index >= e->n) return fail(MT_ERR_INVALID, "env index %lld outside [0, %lld)", (long long)index, e->n);
    DeviceGuard guard(e->cfg.device);
    const size_t J = e->cfg.n_joints, X = e->cfg.n_obj, words = J * 4 + X * 3 + 2;
    fetch_kernel<<<1, 32, 0, nullptr>>>(e->base, e->arm, index, e->fetch_dev);
    CU(cudaGetLastError());
    e->launches++;
    CU(cudaMemcpyAsync(e->fetch_host, e->fetch_dev, words * 4, cudaMemcpyDeviceToHost, nullptr));
    CU(cudaStreamSynchronize(nullptr));
    const float *h = e->fetch_host;
    if (goals_host) std::memcpy(goals_host, h, J * 4);
    if (joints_host) std::memcpy(joints_host, h + J, J * 12);
    if (points_host) std::memcpy(points_host, h + J * 4, X * 12);
    if (alive_host) std::memcpy(alive_host, h + J * 4 + X * 3, 4);
    if (total_reward_host) *total_reward_host = h[J * 4 + X * 3 + 1];
    return MT_OK;
}

extern "C" int mt_stats_device(mt_env *e, int64_t *stats_dev, void *stream) {
    if (!e || !stats_dev) return fail(MT_ERR_INVALID, "NULL argument");
    DeviceGuard guard(e->cfg.device);
    cudaStream_t st = (cudaStream_t)stream;
    CU(cudaMemsetAsync(stats_dev, 0, MT_STATS_WORDS * 8, st));
    // enough threads in flight to read the (L2-resident) total_reward array at full rate: this kernel sits inside
    // the timed region of a rollout, right before the one collective
    stats_kernel<<<e->num_sms * 4, 512, 0, st>>>(e->base, (long long *)stats_dev);
    CU(cudaGetLastError());
    e->launches++;
    return MT_OK;
}

// ----------------------------------------------------------------------------
// The same collective without NCCL's launch latency: every rank owns a small SYMMETRIC buffer that all peers can
// write over NVLink (the caller maps it: torch symmetric memory, cuMem IPC, ...), layout per buffer (int64 words):
//     [2 parities][world ranks][MT_STATS_WORDS]   slots, written by the owning peer's rank
//     [2 parities][world ranks]                   flags, = epoch once the slot is complete
//     [1]                                          this rank's epoch counter
// One kernel per rank (after its stats_kernel): thread r copies this rank's statistics into peer r's slot for this
// rank, fences, raises the flag there, then waits for peer r's flag in its OWN buffer and adds peer r's slot.  Slots
// alternate by epoch parity: a peer can only be one call ahead (it needs everybody's flags of call n to leave call n).
// The epoch lives in device memory, so the call may sit in a replayed CUDA graph.  64 bytes per peer over NVLink:
// ~4 us against ~30 us for ncclAllReduce on the same 64 bytes.
// ----------------------------------------------------------------------------
__global__ void stats_exchange_kernel(const long long *local, long long *const *peers, int rank, int world, long long *out) {
    __shared__ long long acc[MT_STATS_WORDS];
    __shared__ long long epoch_s;
    __shared__ int timed_out;
    const int r = threadIdx.x;
    long long *mine = peers[rank];
    const size_t slot_words = (size_t)2 * world * MT_STATS_WORDS, flag_words = (size_t)2 * world;
    if (r < MT_STATS_WORDS) acc[r] = 0;
    if (r == 0) {
        epoch_s = ++mine[slot_words + flag_words];
        timed_out = 0;
    }
    __syncthreads();
    const long long epoch = epoch_s;
    const size_t par = (size_t)(epoch & 1);
    if (r < world) {
        long long *peer = peers[r];
        long long *slot = peer + (par * world + rank) * MT_STATS_WORDS;
#pragma unroll
        for (int k = 0; k < MT_STATS_WORDS; ++k) slot[k] = local[k];
        __threadfence_system();
        *reinterpret_cast<volatile long long *>(peer + slot_words + par * world + rank) = epoch;
        volatile long long *flag = mine + slot_words + par * world + r;
        const long long t0 = clock64();
        while (*flag != epoch) {
            if (clock64() - t0 > 20000000000LL) {      // ~10 s: a peer never made the call -- give up instead of hanging the GPU
                timed_out = 1;
                break;
            }
        }
        __threadfence_system();
        const long long *got = mine + (par * world + r) * MT_STATS_WORDS;
#pragma unroll
        for (int k = 0; k < MT_STATS_WORDS; ++k)
            atomicAdd(reinterpret_cast<unsigned long long *>(&acc[k]), (unsigned long long)reinterpret_cast<const volatile long long *>(got)[k]);
    }
    __syncthreads();
    if (r < MT_STATS_WORDS) out[r] = timed_out ? -1 : acc[r];      // all words -1: the exchange timed out
}

extern "C" int64_t mt_stats_peer_buffer_bytes(int32_t world) {
    return world < 1 ? 0 : (int64_t)8 * ((int64_t)2 * world * MT_STATS_WORDS + (int64_t)2 * world + 1);
}

// peers_dev: [world] device pointers (in device memory) to every rank's symmetric buffer of mt_stats_peer_buffer_bytes(world)
// bytes, zero-initialised once before the first call; peers_dev[rank] is this rank's own.  stats_dev receives the global sum.
extern "C" int mt_stats_allreduce_peers(mt_env *e, int64_t *const *peers_dev, int32_t rank, int32_t world, int64_t *stats_dev,
                                        void *stream) {
    if (!e || !peers_dev || !stats_dev) return fail(MT_ERR_INVALID, "NULL argument");
    if (world < 1 || world > 1024 || rank < 0 || rank >= world) return fail(MT_ERR_INVALID, "bad rank/world %d/%d", rank, world);
    DeviceGuard guard(e->cfg.device);
    cudaStream_t st = (cudaStream_t)stream;
    if (int rc = mt_stats_device(e, e->stats_dev, stream)) return rc;
    stats_exchange_kernel<<<1, ((world + 31) / 32) * 32 < 32 ? 32 : ((world + 31) / 32) * 32, 0, st>>>(
        (const long long *)e->stats_dev, (long long *const *)peers_dev, rank, world, (long long *)stats_dev);
    CU(cudaGetLastError());
    e->launches++;
    return MT_OK;
}

extern "C" int mt_stats_host(mt_env *e, mt_stats *out) {
    if (!e || !out) return fail(MT_ERR_INVALID, "NULL argument");
    DeviceGuard guard(e->cfg.device);
    if (int rc = mt_stats_device(e, e->stats_dev, nullptr)) return rc;   // legacy default stream: after all blocking streams
    CU(cudaMemcpyAsync(e->stats_pin, e->stats_dev, MT_STATS_WORDS * 8, cudaMemcpyDeviceToHost, nullptr));
    CU(cudaStreamSynchronize(nullptr));
    std::memcpy(out, e->stats_pin, MT_STATS_WORDS * 8);
    return MT_OK;
}

// ----------------------------------------------------------------------------
// The one collective of a multi-GPU rollout (SURVEY.md section 8e): the MT_STATS_WORDS statistics of every
// shard summed with ncclAllReduce over NVLink.  NCCL is dlopen'ed (like NVRTC): a host that already loaded
// one (torch) shares it, and the library has no link-time dependency on it.
// ----------------------------------------------------------------------------
namespace {
struct Nccl {
    typedef struct ncclComm *Comm;
    int (*CommInitAll)(Comm *, int, const int *) = nullptr;
    int (*CommDestroy)(Comm) = nullptr;
    int (*AllReduce)(const void *, void *, size_t, int, int, Comm, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
    bool ok = false;
    static constexpr int kInt64 = 4, kSum = 0;      // ncclInt64, ncclSum (nccl.h)
    static Nccl &get() {
        static Nccl n;
        static std::once_flag once;
        std::call_once(once, [] {
            void *h = nullptr;
            for (const char *name : {"libnccl.so.2", "libnccl.so"}) {
                h = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
                if (h) break;
            }
            if (!h) return;
#define MT_SYM(field, sym) n.field = reinterpret_cast<decltype(n.field)>(dlsym(h, sym)); if (!n.field) return;
            MT_SYM(CommInitAll, "ncclCommInitAll")
            MT_SYM(CommDestroy, "ncclCommDestroy")
            MT_SYM(AllReduce, "ncclAllReduce")
            MT_SYM(GroupStart, "ncclGroupStart")
            MT_SYM(GroupEnd, "ncclGroupEnd")
            MT_SYM(GetErrorString, "ncclGetErrorString")
#undef MT_SYM
            n.ok = true;
        });
        return n;
    }
};
std::mutex g_comm_mu;
std::map<std::vector<int>, std::vector<Nccl::Comm>> g_comms;     // device list -> communicators (one per device), per process
}  // namespace

#define NC(call)                                                                                         \
    do {                                                                                                 \
        int r_ = (call);                                                                                 \
        if (r_ != 0) return fail(MT_ERR_CUDA, "%s failed: %s", #call, Nccl::get().GetErrorString(r_));   \
    } while (0)

// Caller-provided communicator (one process per GPU: the host created `nccl_comm` with ncclCommInitRank):
// writes this shard's statistics to stats_dev and all-reduces them in place on `stream`.  Asynchronous.
extern "C" int mt_stats_allreduce_comm(mt_env *e, void *nccl_comm, int64_t *stats_dev, void *stream) {
    if (!e || !nccl_comm || !stats_dev) return fail(MT_ERR_INVALID, "NULL argument");
    Nccl &nc = Nccl::get();
    if (!nc.ok) return fail(MT_ERR_CUDA, "libnccl.so.2 not found (dlopen)");
    DeviceGuard guard(e->cfg.device);
    if (int rc = mt_stats_device(e, stats_dev, stream)) return rc;
    NC(nc.AllReduce(stats_dev, stats_dev, MT_STATS_WORDS, Nccl::kInt64, Nccl::kSum, (Nccl::Comm)nccl_comm, (cudaStream_t)stream));
    return MT_OK;
}

// Single process driving n handles on n DISTINCT devices: communicators come from ncclCommInitAll (made on
// first use, cached per device list).  Synchronous; every handle's sum lands in *out_host.
extern "C" int mt_stats_allreduce(mt_env *const *envs, int32_t n, mt_stats *out_host) {
    if (!envs || n < 1 || !out_host) return fail(MT_ERR_INVALID, "envs/out is NULL or n < 1");
    for (int i = 0; i < n; ++i)
        if (!envs[i]) return fail(MT_ERR_INVALID, "envs[%d] is NULL", i);
    if (n == 1) return mt_stats_host(envs[0], out_host);
    std::vector<int> devs(n);
    for (int i = 0; i < n; ++i) {
        devs[i] = envs[i]->cfg.device;
        for (int k = 0; k < i; ++k)
            if (devs[k] == devs[i]) return fail(MT_ERR_INVALID, "envs[%d] and envs[%d] share device %d: one handle per device", k, i, devs[i]);
    }
    Nccl &nc = Nccl::get();
    if (!nc.ok) return fail(MT_ERR_CUDA, "libnccl.so.2 not found (dlopen)");
    std::vector<Nccl::Comm> *comms = nullptr;
    {
        std::lock_guard<std::mutex> lock(g_comm_mu);
        auto hit = g_comms.find(devs);
        if (hit == g_comms.end()) {
            std::vector<Nccl::Comm> made(n, nullptr);
            NC(nc.CommInitAll(made.data(), n, devs.data()));
            hit = g_comms.emplace(devs, std::move(made)).first;
        }
        comms = &hit->second;
    }
    for (int i = 0; i < n; ++i) {
        DeviceGuard guard(devs[i]);
        if (int rc = mt_stats_device(envs[i], envs[i]->stats_dev, nullptr)) return rc;
    }
    NC(nc.GroupStart());
    for (int i = 0; i < n; ++i) {
        int r = nc.AllReduce(envs[i]->stats_dev, envs[i]->stats_dev, MT_STATS_WORDS, Nccl::kInt64, Nccl::kSum, (*comms)[i], nullptr);
        if (r != 0) {
            nc.GroupEnd();
            return fail(MT_ERR_CUDA, "ncclAllReduce failed: %s", nc.GetErrorString(r));
        }
    }
    NC(nc.GroupEnd());
    for (int i = 0; i < n; ++i) {
        DeviceGuard guard(devs[i]);
        CU(cudaStreamSynchronize(nullptr));
    }
    DeviceGuard guard(devs[0]);
    CU(cudaMemcpy(out_host, envs[0]->stats_dev, MT_STATS_WORDS * 8, cudaMemcpyDeviceToHost));
    return MT_OK;
}

extern "C" int mt_stats_clear(mt_env *e, void *stream) {
    if (!e) return fail(MT_ERR_INVALID, "env is NULL");
    DeviceGuard guard(e->cfg.device);
    CU(cudaMemsetAsync(e->stats, 0, MT_STATS_WORDS * 8, (cudaStream_t)stream));
    return MT_OK;
}

extern "C" int mt_fk(const mt_config *cfg, int32_t mode, const float *goals_dev, float *out_dev, int64_t m, void *stream) {
    if (!cfg || !goals_dev || !out_dev) return fail(MT_ERR_INVALID, "NULL argument");
    mt_config c = *cfg;
    if (c.n_envs < 1) c.n_envs = 1;
    if (int rc = validate(c)) return rc;
    if (mode < 1 || mode > c.n_joints) return fail(MT_ERR_INVALID, "mode must be in [1, %d]", c.n_joints);
    if (m <= 0) return MT_OK;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) return fail(MT_ERR_NO_DEVICE, "no CUDA device; manytor_b200 has no CPU fallback");
    DeviceGuard guard(c.device);
    StepParams P;
    fill_params(c, P);
    fk_kernel<<<blocks_for(m), 256, 0, (cudaStream_t)stream>>>(P, mode, goals_dev, m, out_dev);
    CU(cudaGetLastError());
    return MT_OK;
}

extern "C" int mt_dh(const float *params_dev, float *out_dev, int64_t m, void *stream) {
    if (!params_dev || !out_dev) return fail(MT_ERR_INVALID, "NULL argument");
    if (m <= 0) return MT_OK;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) return fail(MT_ERR_NO_DEVICE, "no CUDA device; manytor_b200 has no CPU fallback");
    dh_kernel<<<blocks_for(m), 256, 0, (cudaStream_t)stream>>>(params_dev, m, out_dev);
    CU(cudaGetLastError());
    return MT_OK;
}

extern "C" int mt_joints(mt_env *e, const float *goals_dev, float *out_dev, int64_t m, void *stream) {
    if (!e || !goals_dev || !out_dev) return fail(MT_ERR_INVALID, "NULL argument");
    if (m <= 0) return MT_OK;
    DeviceGuard guard(e->cfg.device);
    joints_kernel<<<blocks_for(m, 128), 128, 0, (cudaStream_t)stream>>>(e->base, e->arm, goals_dev, m, out_dev);
    CU(cudaGetLastError());
    e->launches++;
    return MT_OK;
}

extern "C" int mt_r_theta(const float *v1_dev, const float *v2_dev, float *out_dev, int64_t m, void *stream) {
    if (!v1_dev || !v2_dev || !out_dev) return fail(MT_ERR_INVALID, "NULL argument");
    if (m <= 0) return MT_OK;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) return fail(MT_ERR_NO_DEVICE, "no CUDA device; manytor_b200 has no CPU fallback");
    r_theta_kernel<<<blocks_for(m), 256, 0, (cudaStream_t)stream>>>(v1_dev, v2_dev, m, out_dev);
    CU(cudaGetLastError());
    return MT_OK;
}

extern "C" int64_t mt_launch_count(const mt_env *e) { return e ? e->launches : 0; }

// SURVEY.md section 8(d): B = 12J + 24X + 21 with actions read from HBM and fp32 obs
// written (12J + 18X + 21 with binary16 obs); minus 4J when actions are drawn in-kernel,
// minus the observations (12X or 6X) without them.
extern "C" int64_t mt_bytes_per_env_step(const mt_env *e, int32_t actions_from_hbm, int32_t obs_written) {
    if (!e) return 0;
    const int64_t J = e->cfg.n_joints, X = e->cfg.n_obj;
    int64_t b = 8 * J + 12 * X + 21;  // goals r+w, points r, alive r+w, reward w, done w, total_reward r+w
    if (actions_from_hbm) b += 4 * J;
    if (obs_written) b += (e->f16 ? 6 : 12) * X;
    return b;
}

extern "C" int mt_set_timing(mt_env *e, int32_t enabled) {
    if (!e) return fail(MT_ERR_INVALID, "env is NULL");
    e->timing = enabled != 0;
    e->ev_valid = false;
    return MT_OK;
}

extern "C" int mt_last_kernel_ms(mt_env *e, float *ms_out) {
    if (!e || !ms_out) return fail(MT_ERR_INVALID, "NULL argument");
    if (!e->ev_valid) return fail(MT_ERR_STATE, "no timed launch recorded (mt_set_timing)");
    DeviceGuard guard(e->cfg.device);
    CU(cudaEventSynchronize(e->ev1));
    CU(cudaEventElapsedTime(ms_out, e->ev0, e->ev1));
    return MT_OK;
}

#ifdef MT_TRACE
// debug builds only (nvcc -DMT_TRACE): per-warp trace of the most recent step launches, [kTraceWarps][4] u64
extern "C" int mt_debug_trace(unsigned long long *out_host) {
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpyFromSymbol(out_host, g_trace, sizeof(unsigned long long) * kTraceWarps * 4));
    return MT_OK;
}
#endif
