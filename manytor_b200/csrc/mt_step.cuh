// The fused step kernels: one launch of step_kernel = Environment.step for every env of a shard;
// one launch of rollout_kernel = n_steps x step(action_sample()) for every env of a shard.
//
// Both restate, per environment (lane), the reference's
//   step          manytor.py:255-260
//   action        manytor.py:175-213   (25 interpolated poses, ground flag, reward)
//   fk / dh       manytor.py:35-53, 25-32 (closed form for the reference arm,
//                                          z-row / affine chain for a generic DH table)
//   get_observations / r_theta  manytor.py:141-153, 17-22
//   is_done       manytor.py:155-173
//   reset         manytor.py:219-241   (auto-reset with on-device objective refresh)
//
// Mapping: one persistent block per SM; a warp owns a tile of 32 consecutive envs at a time, one lane
// per env, and takes its next tile from the block's queue in shared memory.  The tile's objectives
// (3X fp32 per env, 120 B at X=10) are fetched from HBM by ONE TMA bulk copy into shared memory while
// the lanes do the kinematics (which need no objectives); observations leave by ONE TMA bulk store
// (step_kernel writes them in place over the objectives, rollout_kernel into a second buffer because it
// keeps the objectives for the next step), so the row-major [N][3X] layouts are moved with full-line
// transactions and no per-lane strided access.  All other state is fp32/u32 structure-of-arrays, read
// and written once per step (once per n_steps in rollout_kernel, which keeps it in registers) with
// coalesced vector accesses, prefetched one tile ahead.  Independent fp32 work is packed two lanes per
// instruction (FFMA2 / FADD2 / FMUL2).  DESIGN.md section 4 has the measurements behind each choice.
#pragma once
#include "../../include/manytor_b200.h"
#include "mt_math.cuh"
#include "mt_ptx.cuh"

#include <type_traits>

namespace mt {

#ifndef MT_SUBPOSE_UNROLL
#define MT_SUBPOSE_UNROLL 4      // iterations (pairs of sub-poses) of the ground-test loop unrolled together
#endif
constexpr int kSubposeUnroll = MT_SUBPOSE_UNROLL;
constexpr int kTile = 32;
// Warps per block is a launch-time choice (blockDim.x / 32): as many as one SM can hold in ONE block (28
// for the reference arm at x = 10: 72 registers, 7.7 KB of tile buffers per warp), because the warps of a
// block share the block's tile queue (see step_kernel).  Upper bounds for __launch_bounds__:
constexpr int kMaxWarpsRefArm = 28, kMaxWarpsGeneric = 16;
// Statistics and counters live on the DEVICE, so that a replayed CUDA graph counts its steps and draws
// fresh actions (the host never sees a replay).  Every warp adds its share to accumulators in shared
// memory; the last warp of a block flushes them with one fire-and-forget global atomic per word (148 per
// launch and address: every WARP finishing with a global atomic on one address was measured at +3.6 us
// per launch), and a ticket taken at the START of the launch decides which block advances the step index
// and the env-step count (launch_ticket below).
// Control words (StepParams::ctrl, 64-bit each): [0] step index, [1 + slot] launch tickets.
constexpr int kCtrlStep = 0, kCtrlTicket = 1, kTicketSlots = 31, kCtrlWords = kCtrlTicket + kTicketSlots;
constexpr int kBlockStats = 6;   // episodes, terminated, reward_sum, length_sum, catches, ground_steps = mt_stats words 1..6

enum StepFlags : int32_t {
    kTerminateOnGround = 1,
    kAutoReset = 2,
    kObsAfterReset = 4,
};

struct JointConst {
    float a, d, ca, sa;  // DH row: link length, offset, cos/sin(alpha)
    float co, so;        // cos/sin(theta offset)
};

struct StepParams {
    // state (HBM, padded to a whole number of tiles)
    float *goals;            // [Npad][J]
    uint32_t *alive;         // [Npad]  packed layout: alive mask (bits < ep_shift) | ep_len << ep_shift; wide: mask only
    float *total_reward;     // [Npad]
    uint32_t *counters;      // [Npad]  wide layout only: ep_len (saturating at ep_max); nullptr when packed
    uint32_t *episode;       // [Npad]  resets so far (touched only on reset)
    float *points;           // [Npad][X][3]
    // per-step I/O
    const float *actions;    // [N][J] or nullptr when drawn in-kernel
    void *obs;               // [N][3X] fp32, or binary16 in the kernels built for F16 (mt_config.obs_dtype)
    float *reward;           // [N]
    uint8_t *done;           // [N]
    float *joints;           // [N][J][3] or nullptr
    const float *obj_stream; // [sets][N][X][3] or nullptr
    unsigned long long *stats; // [MT_STATS_WORDS]
    unsigned long long *ctrl;  // [kCtrlWords]: step index, launch tickets (see above)
    long long n;
    long long tile_begin, tile_end;
    long long env_id_base;
    uint32_t seed_lo, seed_hi;
    int32_t ticket_slot;       // which ticket this launch uses (launches that may overlap in time use different ones)
    int32_t advance;           // steps this launch completes: its last block adds them to the step index
    int32_t n_steps;           // rollout_kernel: steps per launch
    long long launch_envs;     // envs this launch advances (added to the env-step count by its last block)
    int32_t n_obj, n_joints, substeps, horizon, flags, obj_sets;
    int32_t action_low;
    uint32_t action_span;
    int32_t trig_span;         // > 0: in-kernel actions take sin/cos from a per-block table of this many entries (ActionTrig)
    float radius, catch_tol, inv_div;
    int32_t obs_frame, ground_a, ground_b, catch_frame;
    float zero_anchor[3];
    JointConst arm[MT_MAX_JOINTS];
    uint32_t tile_bytes;
    int32_t pair_layout;     // objectives stored pair-interleaved (see point_index)
    // Episode length: packed into the alive word above the mask when it fits (every X <= 16; X < 32 when
    // the horizon fits in the 32 - X spare bits), which saves one 4-byte state array read and written per
    // step; otherwise (ep_shift == 0) it lives in `counters`.  Saturates at ep_max either way.
    int32_t ep_shift;
    uint32_t ep_max;
    // L2 eviction policies (createpolicy results), made once per handle and passed as constants, so the
    // step kernel holds no registers for them across its tile loop.  pol_state marks the per-env state
    // evict_last so that it stays in the 126 MB L2 from one step to the next -- for the FRACTION of its
    // lines (chosen by the hardware's address hash, hence the same lines every step) that fits the
    // handle's L2 budget: protecting more lines than the L2 can hold costs more than no hint at all
    // (tools/microbench/bigstreams.cu, N = 2^22).  pol_stream / pol_store are for everything that passes
    // through once per step (actions, objectives in; observations, reward, done out): evict_normal while the
    // whole state fits its budget, evict_first beyond (mt_create; measured both ways in round 2).
    unsigned long long pol_state, pol_stream, pol_store;   // pol_store: the streamed OUTPUTS (observations, reward, done)
    float *drawn;              // rollout_kernel<.., RolloutMode::kDrawTrajectory>: [n_steps][N][J] drawn actions, or nullptr
    // step_kernel<.., FINAL = true> (mt_step_final) and rollout_kernel<.., FINAL = true> (mt_rollout_final): what an
    // ending env's episode leaves behind, written for the rows of the envs that end in this step only (settle_step);
    // the rollout kernel writes step s into slice s of [n_steps][N] arrays, as it does its other outputs
    void *final_obs;           // [N][3X] obs2 of the ending step, in the handle's obs format
    float *final_return;       // [N] total reward of the episode
    int32_t *final_length;     // [N] episode length (the saturating counter)
};

// branch_kernel's own parameters (mt_rollout_branches), beside a StepParams whose actions ([n_steps][M][J]), done ([M]) and
// obs ([M][3X] or nullptr) are per branch.  A second parameter rather than more StepParams fields: every other kernel
// keeps its parameter layout, and with it its code.
struct BranchParams {
    const int64_t *src;        // [M] source env of each branch
    float *ret;                // [M] discounted return
    int32_t *length;           // [M] steps executed
    long long n;               // M
    float gamma;
    // branch_kernel<.., DRAW = true> only (mt_rollout_branches_random); after the fields above, whose offsets stay put
    int32_t n_prefix;          // steps 0 .. n_prefix-1 read P.actions ([n_prefix][M][J]); the others are drawn
    const unsigned long long *draw_key;   // step s >= n_prefix of branch m draws as mt_sample_actions at env m, index key + s
};

// Trajectory buffers (mt_rollout) are arrays of slices: slice s holds step s's rows 0 .. N-1, packed, so row `row` of
// slice s starts at base + (s N + row) row_bytes.  Computed in 64 bits: s N row_bytes passes 2^32 at sizes users run
// (2^20 envs x 36 steps x 120 B of observations).
__host__ __device__ __forceinline__ unsigned long long slice_row_addr(unsigned long long base, unsigned long long s,
                                                                      unsigned long long n, unsigned long long row,
                                                                      unsigned long long row_bytes) {
    return base + (s * n + row) * row_bytes;
}
// May a bulk copy (cp.async.bulk: store of an observation tile, L2 prefetch of an action tile) start at row `row` of
// slice s?  It needs a 16-byte aligned global address; a misaligned one kills the context.  With a 16-byte aligned
// base and `row` a multiple of the 32-env tile that is s N row_bytes % 16 == 0, which fails on some slices unless
// N 3X % 4 == 0 (fp32 observations), N 3X % 8 == 0 (binary16) or N J % 4 == 0 (actions).  Decided per tile from the
// address itself; a tile that may not goes the per-lane way.
__host__ __device__ __forceinline__ bool bulk_aligned(unsigned long long addr) { return (addr & 15ull) == 0ull; }
__host__ __device__ __forceinline__ bool slice_bulk_ok(unsigned long long base, unsigned long long s, unsigned long long n,
                                                       unsigned long long row, unsigned long long row_bytes) {
    return bulk_aligned(slice_row_addr(base, s, n, row, row_bytes));
}

__host__ __device__ __forceinline__ uint32_t alive_mask_of(const StepParams &P, uint32_t word) {
    return P.ep_shift ? (word & ((1u << P.ep_shift) - 1u)) : word;
}

// ---------------------------------------------------------------------------
// kinematics
// ---------------------------------------------------------------------------
struct Frames {
    float anchor[3];   // obs frame origin   (reference: elbow, manytor.py:143)
    float catcher[3];  // catch frame origin (reference: terminal, manytor.py:162)
    float zmin;        // min z of the two ground frames over all sub-poses (manytor.py:191)
};

// Reference arm, closed form (DESIGN.md): with alpha = -+pi/2 the chain of
// manytor.py:42-52 collapses to
//   frame2 = (0, 0, 4.3)
//   elbow  = (24.3 c0 s1, 24.3 s0 s1, 4.3 + 24.3 c1)
//   ee     = elbow + 27 (s3 (c0 c1 c2 - s0 s2) + c3 c0 s1,
//                        s3 (s0 c1 c2 + c0 s2) + c3 s0 s1,
//                        c3 c1 - s3 s1 c2)
// (theta3 before its -pi/2 offset).  Only the two z values are needed at the 24
// interior sub-poses (manytor.py:191), and with A = th1 + th3, B = th1 - th3
//   elbow_z - 4.3 = 24.3 cos th1                                  =: u1
//   ee_z    - 4.3 = u1 + uA + uB + cos th2 (uA - uB),   uA = 13.5 cos A, uB = 13.5 cos B
// The route is linear in angle (np.linspace, manytor.py:182), so u1, cos th2, uA,
// uB are four sampled cosines.  Each is advanced by Reinsch's recurrence
//   x <- x + d;  d <- d - 4 sin^2(delta/2) x
// (2 FMA-class ops per value per sub-pose, error growth linear in the step
// count), run backwards from the exact final pose: 9 instructions per sub-pose
// instead of 3 plane rotations + products (26).  tools/emulate_subpose.py compares
// it with fp64: max |dz| 3.5e-5 over 4e5 random steps, no ground-flag flips.

// Two cosine sequences advanced together (one FADD2 + one FFMA2 per sub-pose).
struct CosSeq2 {
    float2 x, d, na;  // values, backward differences, -4 sin^2(delta/2)
    // amp * cos(theta - k * delta), k = 0, 1, ...; (sh, ch) = sin/cos(delta / 2), per half
    __device__ __forceinline__ void init(float2 amp, float2 cth, float2 sth, float2 sh, float2 ch) {
        float2 t = add2(sh, sh);
        na = neg2(mul2(t, t));            // -4 sh^2
        x = mul2(amp, cth);
        // amp (cos(theta - delta) - cos theta) = amp sin(theta) sin(delta) - 2 sh^2 x
        d = fma2(mul2(amp, sth), mul2(t, ch), mul2(mul2(bc2(0.5f), na), x));
    }
    __device__ __forceinline__ void back() {
        x = add2(x, d);
        d = fma2(na, x, d);
    }
};

// ONE cosine sequence x(k) = amp cos(theta - k delta) at two sub-poses at once: lane .x holds an odd k,
// lane .y the next even k, and back() moves both by 2 delta (Reinsch's recurrence with step 2 delta,
// -4 sin^2(delta) shared by the lanes).  init: (ax, ay) = amp (cos, sin) theta, (sd, cd) = sin/cos delta;
// the lanes start at k = -1 and k = 0, so that the first back() yields k = 1 and k = 2.
struct CosPair {
    float2 x, d;
    float na;
    __device__ __forceinline__ void init(float ax, float ay, float sd, float cd) {
        const float q = (ay + ay) * sd;                       // 2 amp sin(theta) sin(delta) = x(1) - x(-1)
        na = -4.0f * (sd * sd);
        x = make_float2(fmaf(ax, cd, -(ay * sd)), ax);        // amp cos(theta + delta), amp cos(theta)
        d = make_float2(q, fmaf(q, cd, 0.5f * na * ax));      // x(2) - x(0) = amp (sin th sin 2 delta - 2 sin^2 delta cos th)
    }
    __device__ __forceinline__ void back() {
        x = add2(x, d);
        d = fma2(bc2(na), x, d);
    }
};

// Where the sines / cosines of the joint TARGETS come from.  Actions drawn in-kernel are integer degrees in
// [action_low, action_low + span): each block fills a table of (sin, cos) per possible value once per launch -- with
// the very evaluation the kernels would otherwise run per env and step, so a lookup is bit-identical to it -- and the
// per-step cost of 4..8 sin/cos evaluations becomes as many 64-bit shared-memory loads.  table = 0: evaluate.
struct ActionTrig {
    uint32_t table;   // shared-space address of the float2 (sin, cos) entries
    int32_t low;      // action value of entry 0
    __device__ __forceinline__ float2 at(float a) const { return lds_f2(table + (uint32_t)(__float2int_rn(a) - low) * 8u); }
};

template <bool TAB>
__device__ __forceinline__ void ref_arm(const float *g, const float *a, int substeps, float inv_div, Frames &f,
                                        float *jout /* 12 floats or nullptr */, ActionTrig trig = ActionTrig{0u, 0}) {
    float2 s01, c01, s23, c23;
    if (TAB && trig.table) {
        const float2 t0 = trig.at(a[0]), t1 = trig.at(a[1]), t2 = trig.at(a[2]), t3 = trig.at(a[3]);
        s01 = make_float2(t0.x, t1.x); c01 = make_float2(t0.y, t1.y);
        s23 = make_float2(t2.x, t3.x); c23 = make_float2(t2.y, t3.y);
    } else {
        sincos_deg2(make_float2(a[0], a[1]), s01, c01);
        sincos_deg2(make_float2(a[2], a[3]), s23, c23);
    }
    const float s0 = s01.x, c0 = c01.x, s1 = s01.y, c1 = c01.y, s2 = s23.x, c2 = c23.x, s3 = s23.y, c3 = c23.y;
    const float L1 = 24.3f, L2 = 27.0f, H = 4.3f;
    float ez = fmaf(L1, c1, H);
    float k = L1 * s1;
    float ex = k * c0, ey = k * s0;
    float c1c2 = c1 * c2;
    float ux = fmaf(c0, c1c2, -(s0 * s2));
    float uy = fmaf(s0, c1c2, c0 * s2);
    float s1c3 = s1 * c3;
    float tx = fmaf(L2, fmaf(s3, ux, c0 * s1c3), ex);
    float ty = fmaf(L2, fmaf(s3, uy, s0 * s1c3), ey);
    float tz = fmaf(L2, fmaf(c3, c1, -((s3 * s1) * c2)), ez);
    f.anchor[0] = ex; f.anchor[1] = ey; f.anchor[2] = ez;
    f.catcher[0] = tx; f.catcher[1] = ty; f.catcher[2] = tz;
    if (jout) {
        jout[0] = 0.f; jout[1] = 0.f; jout[2] = 0.f;
        jout[3] = 0.f; jout[4] = 0.f; jout[5] = H;
        jout[6] = ex; jout[7] = ey; jout[8] = ez;
        jout[9] = tx; jout[10] = ty; jout[11] = tz;
    }
    float zmin = fminf(ez, tz);
    if (substeps > 1) {
        const float d1 = (a[1] - g[1]) * inv_div, d2 = (a[2] - g[2]) * inv_div, d3 = (a[3] - g[3]) * inv_div;   // degrees per sub-pose
        const float dmax = fmaxf(fmaxf(fabsf(d1), fabsf(d2)), fabsf(d3));
        float m = 3.0e38f;
        if (((substeps - 1) & 1) == 0 && __all_sync(__activemask(), dmax <= 22.5f)) {
            // Usual case (an even number of interior sub-poses, every joint within 540 degrees of its target at
            // 25 sub-poses): TWO sub-poses per packed iteration.  Lane .x of every value walks the odd
            // sub-poses k = 1, 3, ..., lane .y the even ones k = 2, 4, ..., both in steps of 2 delta, so the
            // combination u1 + (uA + uB) + cos(th2)(uA - uB) is packed as well: 14 instructions per two
            // sub-poses against 2 x 9.4.  Same error as the single-step recurrence (tools/emulate_subpose.py:
            // max |dz| 3.8e-5, no ground-flag flips in 4e5 steps).
            float2 sd12, cd12;
            float sd3, cd3;
            sincos_deg_small2(make_float2(d1, d2), sd12, cd12);
            sincos_deg_small(d3, sd3, cd3);
            const float sd1 = sd12.x, cd1 = cd12.x;
            // A = th1 + th3, B = th1 - th3: cos/sin of the angles and of their steps by angle addition
            const float cA = fmaf(c1, c3, -(s1 * s3)), cB = fmaf(c1, c3, s1 * s3);
            const float sA = fmaf(s1, c3, c1 * s3), sB = fmaf(s1, c3, -(c1 * s3));
            const float cdA = fmaf(cd1, cd3, -(sd1 * sd3)), cdB = fmaf(cd1, cd3, sd1 * sd3);
            const float sdA = fmaf(sd1, cd3, cd1 * sd3), sdB = fmaf(sd1, cd3, -(cd1 * sd3));
            CosPair u1, q2, uA, uB;
            u1.init(L1 * c1, L1 * s1, sd1, cd1);
            q2.init(c2, s2, sd12.y, cd12.y);
            uA.init(0.5f * L2 * cA, 0.5f * L2 * sA, sdA, cdA);
            uB.init(0.5f * L2 * cB, 0.5f * L2 * sB, sdB, cdB);
            const int iters = (substeps - 1) >> 1;
#pragma unroll kSubposeUnroll
            for (int it = 0; it < iters; ++it) {
                u1.back(); q2.back(); uA.back(); uB.back();
                const float2 t = fma2(q2.x, add2(uA.x, neg2(uB.x)), add2(u1.x, add2(uA.x, uB.x)));
                m = fminf(m, fminf(t.x, t.y));
                m = fminf(m, fminf(u1.x.x, u1.x.y));
            }
        } else {
            // half steps in degrees; the small-angle sin/cos holds for |half step| <= 45, i.e. any
            // target within +-2160 degrees of the current pose at 25 sub-poses (else: general path)
            const float2 h12 = make_float2(0.5f * d1, 0.5f * d2);
            const float2 h33 = bc2(0.5f * d3);
            float2 sh12, ch12, sh33, ch33;
            if (__all_sync(__activemask(), dmax <= 90.0f)) {
                sincos_deg_small2(h12, sh12, ch12);
                sincos_deg_small2(h33, sh33, ch33);
            } else {
                sincos_deg2(h12, sh12, ch12);
                sincos_deg2(h33, sh33, ch33);
            }
            // A = th1 + th3, B = th1 - th3 and their half steps by angle addition, A in .x, B in .y:
            // cos(th1 +- th3) = c1 c3 -+ s1 s3, sin(th1 +- th3) = s1 c3 +- c1 s3
            const float2 pm = make_float2(1.0f, -1.0f);
            const float2 cAB = fma2(bc2(-(s1 * s3)), pm, bc2(c1 * c3));
            const float2 sAB = fma2(bc2(c1 * s3), pm, bc2(s1 * c3));
            const float sh1 = sh12.x, ch1 = ch12.x, sh3 = sh33.x, ch3 = ch33.x;
            const float2 chAB = fma2(bc2(-(sh1 * sh3)), pm, bc2(ch1 * ch3));
            const float2 shAB = fma2(bc2(ch1 * sh3), pm, bc2(sh1 * ch3));
            CosSeq2 q12, qAB;
            q12.init(make_float2(L1, 1.0f), make_float2(c1, c2), make_float2(s1, s2), sh12, ch12);
            qAB.init(bc2(0.5f * L2), cAB, sAB, shAB, chAB);
#pragma unroll 4
            for (int p = 1; p < substeps; ++p) {
                q12.back();
                qAB.back();
                const float t = fmaf(q12.x.y, qAB.x.x - qAB.x.y, q12.x.x + (qAB.x.x + qAB.x.y));
                m = fminf(m, fminf(q12.x.x, t));
            }
        }
        zmin = fminf(zmin, m + H);
    }
    f.zmin = zmin;
}

// ---------------------------------------------------------------------------
// Generic J-joint DH chain -- the reference's "pluggable fk" (README.md:20, manytor.py:126-127).
//
// ARM template values: 0 = reference arm closed form (above); 2..8 = J joints with the DH table
// read at run time from the kernel parameters; >= 100 = a PRESET arm whose table is a constexpr
// in this header (ARM % 100 joints), so every row's a = 0 / d = 0 / alpha in {0, +-pi/2} folds at
// compile time and most of the chain disappears.  Plugging in a new arm at full speed = adding a
// Preset<> specialisation here and a case in pick_kernel (mt_api.cu); any other table still runs
// through the run-time path.  Presets assume the usual frame selectors (obs J-1, ground J-1 and J,
// catch J); mt_create only picks a preset when the configuration says so.
// ---------------------------------------------------------------------------
constexpr int kArmUr5 = 106;
// every preset arm, once: mt_api.cu expands this list for detection (is_preset_arm), kernel
// dispatch (pick_kernel) and the helper kernels, so adding an arm = one Preset<> + one line here
#define MT_FOR_EACH_PRESET_ARM(X) X(kArmUr5)

template <int ARM> struct ArmJoints { static constexpr int value = ARM == 0 ? 4 : (ARM >= 100 ? ARM % 100 : ARM); };

template <int ARM> struct Preset {
    static constexpr bool value = false;
    __host__ __device__ static constexpr JointConst row(int) { return JointConst{0.f, 0.f, 1.f, 0.f, 1.f, 0.f}; }
};
// UR5 (BASELINE.json config 5), metres: (a, d, cos alpha, sin alpha, cos offset, sin offset)
template <> struct Preset<kArmUr5> {
    static constexpr bool value = true;
    __host__ __device__ static constexpr JointConst row(int i) {
        switch (i) {
            case 0: return JointConst{0.f, 0.089159f, 0.f, 1.f, 1.f, 0.f};
            case 1: return JointConst{-0.425f, 0.f, 1.f, 0.f, 1.f, 0.f};
            case 2: return JointConst{-0.39225f, 0.f, 1.f, 0.f, 1.f, 0.f};
            case 3: return JointConst{0.f, 0.10915f, 0.f, 1.f, 1.f, 0.f};
            case 4: return JointConst{0.f, 0.09465f, 0.f, -1.f, 1.f, 0.f};
            default: return JointConst{0.f, 0.0823f, 1.f, 0.f, 1.f, 0.f};
        }
    }
};

template <int I, int N, class F>
__device__ __forceinline__ void static_for(F &&f) {
    if constexpr (I < N) {
        f(std::integral_constant<int, I>{});
        static_for<I + 1, N>(f);
    }
}

// scalar / packed arithmetic under one name, so a row update is written once
__device__ __forceinline__ float vfma(float a, float b, float c) { return fmaf(a, b, c); }
__device__ __forceinline__ float2 vfma(float2 a, float2 b, float2 c) { return fma2(a, b, c); }
__device__ __forceinline__ float vmul(float a, float b) { return a * b; }
__device__ __forceinline__ float2 vmul(float2 a, float2 b) { return mul2(a, b); }
__device__ __forceinline__ float vneg(float a) { return -a; }
__device__ __forceinline__ float2 vneg(float2 a) { return neg2(a); }
template <class T> __device__ __forceinline__ T vbc(float x);
template <> __device__ __forceinline__ float vbc<float>(float x) { return x; }
template <> __device__ __forceinline__ float2 vbc<float2>(float x) { return bc2(x); }

template <int ARM, int I>
__device__ __forceinline__ JointConst joint_of(const StepParams &P) {
    if constexpr (Preset<ARM>::value) return Preset<ARM>::row(I);
    else return P.arm[I];
}

// Push the row vector (r0, r1, r2 | t) of the accumulated transform through DH row I, whose joint
// angle has cosine c and sine s:  row <- row * [Rz(theta) Tz(d) Tx(a) Rx(alpha)]  (manytor.py:25-32).
template <int ARM, int I, class T>
__device__ __forceinline__ void push_row(const StepParams &P, T &r0, T &r1, T &r2, T &t, T c, T s) {
    const T u = vfma(r0, c, vmul(r1, s));
    const T v = vfma(r1, c, vneg(vmul(r0, s)));
    const T o = r2;
    if constexpr (Preset<ARM>::value) {
        constexpr JointConst q = Preset<ARM>::row(I);
        if constexpr (q.a != 0.f) t = vfma(vbc<T>(q.a), u, t);
        if constexpr (q.d != 0.f) t = vfma(vbc<T>(q.d), o, t);
        if constexpr (q.sa == 0.f && q.ca == 1.f) { r1 = v; }
        else if constexpr (q.sa == 0.f && q.ca == -1.f) { r1 = vneg(v); r2 = vneg(o); }
        else if constexpr (q.ca == 0.f && q.sa == 1.f) { r1 = o; r2 = vneg(v); }
        else if constexpr (q.ca == 0.f && q.sa == -1.f) { r1 = vneg(o); r2 = v; }
        else {
            r1 = vfma(v, vbc<T>(q.ca), vmul(o, vbc<T>(q.sa)));
            r2 = vfma(o, vbc<T>(q.ca), vneg(vmul(v, vbc<T>(q.sa))));
        }
    } else {
        const JointConst q = P.arm[I];
        t = vfma(vbc<T>(q.a), u, vfma(vbc<T>(q.d), o, t));
        r1 = vfma(v, vbc<T>(q.ca), vmul(o, vbc<T>(q.sa)));
        r2 = vfma(o, vbc<T>(q.ca), vneg(vmul(v, vbc<T>(q.sa))));
    }
    r0 = u;
}

// z of the two ground frames at two sub-poses per iteration (lanes .x/.y), minimum over `iters`
// iterations.  The z row e_z^T A_1 .. A_k does not depend on joint 0's angle: after joint 0 it is the
// constant (0, sin a0, cos a0 | d0), and pushing THAT through joint 1 needs no r0 terms.
template <int ARM, bool STD>
__device__ __forceinline__ float subpose_zmin(const StepParams &P, float2 *c2, float2 *s2, const float *cdd,
                                              const float *sdd, int iters, float zmin) {
    constexpr int J = ArmJoints<ARM>::value;
    const JointConst q0 = joint_of<ARM, 0>(P);
    for (int it = 0; it < iters; ++it) {
        float2 r0, r1, r2, tz;
        float2 za = bc2(q0.d), zb = bc2(q0.d);     // frame 1 (only reachable through run-time selectors or J = 2)
        if (!STD) {
            za = bc2((P.ground_a == 1) ? q0.d : 0.f);
            zb = bc2((P.ground_b == 1) ? q0.d : 0.f);
        }
        static_for<1, J>([&](auto ic) {
            constexpr int i = decltype(ic)::value;
            if constexpr (i == 1) {                 // row entering joint 1 is constant with r0 = 0
                const JointConst q = joint_of<ARM, 1>(P);
                const float2 u = mul2(bc2(q0.sa), s2[1]);
                const float2 v = mul2(bc2(q0.sa), c2[1]);
                tz = fma2(bc2(q.a), u, bc2(fmaf(q.d, q0.ca, q0.d)));
                r1 = fma2(v, bc2(q.ca), bc2(q0.ca * q.sa));
                r2 = fma2(v, bc2(-q.sa), bc2(q0.ca * q.ca));
                r0 = u;
            } else {
                push_row<ARM, i, float2>(P, r0, r1, r2, tz, c2[i], s2[i]);
            }
            if (STD ? (i + 1 == J - 1) : (i + 1 == P.ground_a)) za = tz;
            if (STD ? (i + 1 == J) : (i + 1 == P.ground_b)) zb = tz;
            // advance this joint by 2 delta for the next pair of sub-poses
            const float2 nc = fma2(c2[i], bc2(cdd[i]), mul2(s2[i], bc2(sdd[i])));
            s2[i] = fma2(s2[i], bc2(cdd[i]), neg2(mul2(c2[i], bc2(sdd[i]))));
            c2[i] = nc;
        });
        zmin = fminf(zmin, fminf(fminf(za.x, za.y), fminf(zb.x, zb.y)));
    }
    return zmin;
}

// Final pose: 3x4 affine prefix products give the origin of every frame (manytor.py:188-189).
// Sub-poses: only the z row is propagated, two sub-poses per packed iteration.
template <int ARM, bool TAB>
__device__ __forceinline__ void generic_arm(const StepParams &P, const float *g, const float *a, Frames &f,
                                            float *jout /* J*3 floats or nullptr */, ActionTrig trig = ActionTrig{0u, 0}) {
    constexpr int J = ArmJoints<ARM>::value;
    constexpr bool kPreset = Preset<ARM>::value;
    const int obs_frame = kPreset ? J - 1 : P.obs_frame, catch_frame = kPreset ? J : P.catch_frame;
    const int ground_a = kPreset ? J - 1 : P.ground_a, ground_b = kPreset ? J : P.ground_b;
    float c[J], s[J];
    static_for<0, J>([&](auto ic) {
        constexpr int i = decltype(ic)::value;
        float si, ci;
        if (TAB && trig.table) {
            const float2 t = trig.at(a[i]);
            si = t.x; ci = t.y;
        } else {
            sincos_deg(a[i], si, ci);
        }
        const JointConst q = joint_of<ARM, i>(P);
        if (kPreset && q.so == 0.f && q.co == 1.f) {       // no theta offset on this row
            c[i] = ci; s[i] = si;
        } else {
            c[i] = fmaf(ci, q.co, -(si * q.so));
            s[i] = fmaf(si, q.co, ci * q.so);
        }
    });
    // rows of the accumulated transform after joint 0 = the DH matrix of row 0 itself
    const JointConst q0 = joint_of<ARM, 0>(P);
    float R[3][3] = {{c[0], -s[0] * q0.ca, s[0] * q0.sa}, {s[0], c[0] * q0.ca, -c[0] * q0.sa}, {0.f, q0.sa, q0.ca}};
    float t[3] = {q0.a * c[0], q0.a * s[0], q0.d};
    float zA = 0.f, zB = 0.f;
    if (jout) { jout[0] = 0.f; jout[1] = 0.f; jout[2] = 0.f; }
    if (obs_frame == 0) { f.anchor[0] = f.anchor[1] = f.anchor[2] = 0.f; }
    if (catch_frame == 0) { f.catcher[0] = f.catcher[1] = f.catcher[2] = 0.f; }
    static_for<0, J>([&](auto ic) {
        constexpr int i = decltype(ic)::value;
        if constexpr (i > 0) {
#pragma unroll
            for (int r = 0; r < 3; ++r) push_row<ARM, i, float>(P, R[r][0], R[r][1], R[r][2], t[r], c[i], s[i]);
        }
        const int frame = i + 1;
        if (frame == obs_frame) { f.anchor[0] = t[0]; f.anchor[1] = t[1]; f.anchor[2] = t[2]; }
        if (frame == catch_frame) { f.catcher[0] = t[0]; f.catcher[1] = t[1]; f.catcher[2] = t[2]; }
        if (frame == ground_a) zA = t[2];
        if (frame == ground_b) zB = t[2];
        if (jout && frame >= 2) { jout[(frame - 1) * 3 + 0] = t[0]; jout[(frame - 1) * 3 + 1] = t[1]; jout[(frame - 1) * 3 + 2] = t[2]; }
    });
    float zmin = fminf(zA, zB);
    // Interior sub-poses k = 1 .. M (k steps back from the final pose), TWO per iteration: the .x
    // lane of every packed value is sub-pose k, the .y lane sub-pose k+1, and both advance by
    // 2*delta per iteration (FFMA2/FADD2: half the instructions, half the rotations' rounding).
    // M even: pairs (1,2), (3,4), ..; M odd: (0,1), (2,3), .. (re-testing the final pose is harmless).
    const int M = P.substeps - 1;
    if (M > 0) {
        const bool even = (M & 1) == 0;
        float2 c2[J], s2[J];
        float cdd[J], sdd[J];
#pragma unroll
        for (int i = 1; i < J; ++i) {
            float sd, cd;
            sincos_deg((a[i] - g[i]) * P.inv_div, sd, cd);
            const float c1 = fmaf(c[i], cd, s[i] * sd), s1 = fmaf(s[i], cd, -(c[i] * sd));      // one step back
            cdd[i] = fmaf(cd, cd, -(sd * sd));                                                   // cos / sin of 2 delta
            sdd[i] = 2.0f * sd * cd;
            const float cb = fmaf(c[i], cdd[i], s[i] * sdd[i]), sb = fmaf(s[i], cdd[i], -(c[i] * sdd[i]));  // two back
            c2[i] = even ? make_float2(c1, cb) : make_float2(c[i], c1);
            s2[i] = even ? make_float2(s1, sb) : make_float2(s[i], s1);
        }
        const int iters = (M + 1) >> 1;
        // the usual selectors (ground frames J-1 and J) get a copy of the loop with the two z picks
        // resolved at compile time; any other choice takes the run-time-select copy
        if (kPreset || (ground_a == J - 1 && ground_b == J)) zmin = subpose_zmin<ARM, true>(P, c2, s2, cdd, sdd, iters, zmin);
        else if constexpr (!kPreset) zmin = subpose_zmin<ARM, false>(P, c2, s2, cdd, sdd, iters, zmin);
    }
    f.zmin = zmin;
}

// ---------------------------------------------------------------------------
// observations + catch for one objective (manytor.py:141-153, 17-22, 158-168)
// ---------------------------------------------------------------------------
template <bool WOBS>
__device__ __forceinline__ bool one_objective(float &px, float &py, float &pz, const Frames &f, float tol,
                                              bool alive) {
    // catch: inclusive axis-aligned cube around the catch frame (math.isclose abs_tol)
    bool caught = fmaxf(fmaxf(fabsf(f.catcher[0] - px), fabsf(f.catcher[1] - py)), fabsf(f.catcher[2] - pz)) <= tol;
    if (WOBS) {
        float dx = fabsf(f.anchor[0] - px), dy = fabsf(f.anchor[1] - py), dz = fabsf(f.anchor[2] - pz);
        float h2 = fmaf(dx, dx, dy * dy);
        float dist = fast_sqrt(fmaf(dz, dz, h2));
        float h = fast_sqrt(h2);
        float r = atan2_deg_pos(dx, dy, h);
        float th = atan2_deg_pos(h, dz, dist);
        px = alive ? dist : 0.0f;
        py = alive ? r : 0.0f;
        pz = alive ? th : 0.0f;
    }
    return caught;
}

// Layout of one env's objectives inside its row of 3X floats.
//   pair layout (every EVEN X): objectives are stored two by two,
//   component-interleaved -- [x0 x1 | y0 y1 | z0 z1] per pair -- so one 64-bit shared-memory load
//   yields the packed operand (x0, x1) for the FADD2/FFMA2 pipeline; observations are written back
//   in place in the public row-major order [d0 r0 t0 d1 r1 t1], which spans the same 6 floats.
//   plain layout (every ODD X): row-major [x y z] per objective.
// Either way a lane only ever touches its own row, and the row stride (3X words) keeps 64/128-bit
// accesses of consecutive lanes on distinct banks for X = 10 / 20.

__host__ __device__ __forceinline__ int point_index(bool pair_layout, int pt, int comp) {
    return pair_layout ? (pt >> 1) * 6 + comp * 2 + (pt & 1) : pt * 3 + comp;
}

// Two objectives at once, packed (manytor.py:141-153, 17-22, 158-168).  In: (x0,x1), (y0,y1),
// (z0,z1).  Out: o[6] = d0 r0 t0 d1 r1 t1; returns the two catch bits.
template <bool WOBS>
__device__ __forceinline__ uint32_t pair_objective(float2 PX, float2 PY, float2 PZ, const Frames &f, float tol,
                                                   bool alive0, bool alive1, float *o) {
    const float2 cx = add2(PX, bc2(-f.catcher[0])), cy = add2(PY, bc2(-f.catcher[1])), cz = add2(PZ, bc2(-f.catcher[2]));
    // inside the inclusive cube <=> the largest |component| is within the tolerance: one 3-input max
    // (FMNMX3 with |x| operands) and one compare per objective instead of three chained compares
    const bool c0 = fmaxf(fmaxf(fabsf(cx.x), fabsf(cy.x)), fabsf(cz.x)) <= tol;
    const bool c1 = fmaxf(fmaxf(fabsf(cx.y), fabsf(cy.y)), fabsf(cz.y)) <= tol;
    if (WOBS) {
        const float2 dx = add2(PX, bc2(-f.anchor[0])), dy = add2(PY, bc2(-f.anchor[1])), dz = add2(PZ, bc2(-f.anchor[2]));
        // 1e-36 under the square roots keeps both denominators below positive (0/0 -> 0 like math.atan2(0, 0));
        // it is absorbed unless the objective is within 1e-15 of the anchor, where it moves the distance by 1e-18
        const float2 h2 = fma2(dx, dx, fma2(dy, dy, bc2(1e-36f)));
        const float2 d2 = fma2(dz, dz, h2);
        const float2 h = make_float2(fast_sqrt(h2.x), fast_sqrt(h2.y));
        const float2 dist = make_float2(fast_sqrt(d2.x), fast_sqrt(d2.y));
        // atan2(|dx|, |dy|) = 2 atan(|dx| / (|dy| + h)); atan2(h, |dz|) = 2 atan(h / (|dz| + dist))
        const float2 dr = add2(abs2(dy), h);
        const float2 dt = add2(abs2(dz), dist);
        const float2 tr = mul2(abs2(dx), make_float2(fast_rcp(dr.x), fast_rcp(dr.y)));
        const float2 tt = mul2(h, make_float2(fast_rcp(dt.x), fast_rcp(dt.y)));
        const float2 R = atan_half_deg2(tr), T = atan_half_deg2(tt);
        o[0] = alive0 ? dist.x : 0.0f; o[1] = alive0 ? R.x : 0.0f; o[2] = alive0 ? T.x : 0.0f;
        o[3] = alive1 ? dist.y : 0.0f; o[4] = alive1 ? R.y : 0.0f; o[5] = alive1 ? T.y : 0.0f;
    }
    return (c0 ? 1u : 0u) | (c1 ? 2u : 0u);
}

// Walk one env's row of objectives in shared memory (`row` = its shared-space byte address); the
// observations go to `orow` -- the same row for the step kernel (in place), another buffer for the
// multi-step rollout, which keeps the objectives.  Returns the bitmask of objectives inside the catch cube.
template <int X, bool WOBS>
__device__ __forceinline__ uint32_t walk_row(uint32_t row, uint32_t orow, int x, const Frames &f, float tol, uint32_t alive) {
    uint32_t caught = 0;
    const int xx = X ? X : x;
    if ((xx & 1) == 0) {
        // even X: pair-interleaved layout, one 64-bit access per packed operand
#pragma unroll
        for (int pr = 0; pr < (X ? X / 2 : xx >> 1); ++pr) {
            const uint32_t q = row + pr * 24;
            const float2 PX = lds_f2(q), PY = lds_f2(q + 8), PZ = lds_f2(q + 16);
            float o[6];
            const uint32_t c = pair_objective<WOBS>(PX, PY, PZ, f, tol, (alive >> (2 * pr)) & 1u,
                                                    (alive >> (2 * pr + 1)) & 1u, o);
            caught |= c << (2 * pr);
            if (WOBS) {
                const uint32_t w = orow + pr * 24;
                sts_f2(w, make_float2(o[0], o[1]));
                sts_f2(w + 8, make_float2(o[2], o[3]));
                sts_f2(w + 16, make_float2(o[4], o[5]));
            }
        }
    } else {
        // odd X: plain row-major layout (the row stride 3X is odd, so 32-bit accesses of consecutive lanes
        // fall on distinct banks); still two objectives per packed evaluation, plus one left over
        int pt = 0;
#pragma unroll
        for (; pt + 1 < xx; pt += 2) {
            const uint32_t q = row + pt * 12;
            float v[6];
#pragma unroll
            for (int k = 0; k < 6; ++k) v[k] = lds_f(q + 4 * k);
            float o[6];
            const uint32_t c = pair_objective<WOBS>(make_float2(v[0], v[3]), make_float2(v[1], v[4]), make_float2(v[2], v[5]), f,
                                                    tol, (alive >> pt) & 1u, (alive >> (pt + 1)) & 1u, o);
            caught |= c << pt;
            if (WOBS) {
#pragma unroll
                for (int k = 0; k < 6; ++k) sts_f(orow + pt * 12 + 4 * k, o[k]);
            }
        }
        const uint32_t q = row + pt * 12;
        float px = lds_f(q), py = lds_f(q + 4), pz = lds_f(q + 8);
        const bool c = one_objective<WOBS>(px, py, pz, f, tol, (alive >> pt) & 1u);
        caught |= c ? (1u << pt) : 0u;
        if (WOBS) { const uint32_t w = orow + pt * 12; sts_f(w, px); sts_f(w + 4, py); sts_f(w + 8, pz); }
    }
    return caught;
}

// ---------------------------------------------------------------------------
// binary16 observations (mt_config.obs_dtype = MT_OBS_F16).  Every kernel computes a tile's observations in fp32
// in shared memory, exactly as for an fp32 handle; only the way out differs.
// ---------------------------------------------------------------------------
// Pack a full tile of observations, [32][rowlen] fp32 at `buf`, to binary16 in place: element i moves from byte 4i
// to byte 2i, so the packed tile ([32][rowlen] halves, 64 rowlen = 192 X bytes) is contiguous at the start of the
// buffer and leaves by one bulk store.  Lane l converts the 4-element quads l, l + 32, ...: round r reads bytes
// [512r, 512r + 512) and writes [256r, 256r + 256), which round r / 2 <= r has read.  The writes of a round land on
// words other lanes of the SAME round read (r = 0), so each round reads into registers, syncs the warp, then writes;
// later rounds read only above what earlier rounds wrote.  The caller has synced the warp after writing the tile.
template <int X>
__device__ __forceinline__ void pack_tile_f16(uint32_t buf, int rowlen, int lane) {
    const int quads = (X ? 3 * X : rowlen) * (kTile / 4);
#pragma unroll
    for (int q0 = 0; q0 < quads; q0 += kTile) {
        const int q = q0 + lane;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (q < quads) v = lds_f4(buf + 16u * (uint32_t)q);
        __syncwarp();
        if (q < quads) sts_u2(buf + 8u * (uint32_t)q, f32x2_to_f16x2(v.x, v.y), f32x2_to_f16x2(v.z, v.w));
    }
}

// element i of the caller's observation buffer, in the kernel's format
template <bool F16>
__device__ __forceinline__ void *obs_at(void *obs, size_t i) {
    return F16 ? (void *)((uint16_t *)obs + i) : (void *)((float *)obs + i);
}
template <bool F16>
__device__ __forceinline__ void store_obs(void *obs, size_t i, float v) {
    if (F16) ((uint16_t *)obs)[i] = f32_to_f16(v);
    else ((float *)obs)[i] = v;
}

// ---------------------------------------------------------------------------
// objective refresh (manytor.py:228-241): uniform in the upper half ball.
// The reference rejects from the cube; the direct map below has the same
// distribution: r = R u^(1/3), z/r uniform on [0,1], azimuth uniform.
// ---------------------------------------------------------------------------
__device__ __forceinline__ void sample_point(const StepParams &P, long long gid, uint32_t episode, int pt, float &x,
                                             float &y, float &z) {
    Philox u = philox4x32_10((uint32_t)gid, (uint32_t)((unsigned long long)gid >> 32), episode * 32u + (uint32_t)pt,
                             STREAM_POINTS, P.seed_lo, P.seed_hi);
    float r = fminf(P.radius * cbrtf(1.0f - uniform01(u.x)), P.radius);
    float ct = uniform01(u.y);
    float st = sqrtf(fmaxf(1.0f - ct * ct, 0.0f));
    float sphi, cphi;
    sincospif(2.0f * uniform01(u.z), &sphi, &cphi);
    x = r * st * cphi;
    y = r * st * sphi;
    z = r * ct;
}

__device__ __forceinline__ void draw_actions(const StepParams &P, unsigned long long step, long long gid, int J, float *a) {
    const uint32_t lo = (uint32_t)gid, hi = (uint32_t)((unsigned long long)gid >> 32);
    const uint32_t step_lo = (uint32_t)step, step_hi = (uint32_t)(step >> 32);
    Philox u = philox4x32_10(lo, hi, step_lo, STREAM_ACTIONS ^ step_hi, P.seed_lo, P.seed_hi);
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int i = 0; i < 4; ++i)
        if (i < J) a[i] = (float)uniform_int(w[i], P.action_low, P.action_span);
    if (J > 4) {
        Philox u2 = philox4x32_10(lo, hi, step_lo, (STREAM_ACTIONS + 1u) ^ step_hi, P.seed_lo, P.seed_hi);
        const uint32_t w2[4] = {u2.x, u2.y, u2.z, u2.w};
#pragma unroll
        for (int i = 4; i < MT_MAX_JOINTS; ++i)
            if (i < J) a[i] = (float)uniform_int(w2[i - 4], P.action_low, P.action_span);
    }
}

// Per-env scalars of one tile, prefetched into registers one tile ahead.  (Loading the two state words
// that are only needed after the kinematics at the top of their own tile instead -- two registers fewer --
// was measured: +1.2 us per step under back-to-back launches, the kinematics do not cover a loaded HBM.)
template <int J>
struct TileScalars {
    float g[J], a[J];
    uint32_t word;    // the state word: alive mask (| ep_len << ep_shift in the packed layout)
    float total;
    uint32_t cnt;     // ep_len in the wide layout
};

// Where the episode length lives (StepParams::ep_shift): a compile-time objective count of at most 16 always
// has it in the upper half of the alive word (mt_create), which removes the `counters` path, its register
// and its selects from those kernels; otherwise the handle's choice is read at run time.
template <int X>
__device__ __forceinline__ int ep_shift_of(const StepParams &P) {
    return (X > 0 && X <= 16) ? 16 : P.ep_shift;
}

template <int J, int X, bool RAND>
__device__ __forceinline__ void load_scalars(const StepParams &P, int env32, TileScalars<J> &s, uint64_t keep,
                                             uint64_t stream) {
    const size_t env = (size_t)env32;     // indices stay 32-bit in the kernel (n_envs < 2^31); one widening per address
    // goals[0] is never loaded: no sub-pose z depends on joint 0 (it turns about the world z axis), so
    // the register of a prefetched goals[0] would be dead on arrival, ptxas would hand it out as scratch
    // at once, and that write-after-write hazard parks the warp on the prefetch's full memory latency
    // (it was 21 % of all stall samples in ncu with a 128-bit load of the whole row).
    s.g[0] = 0.f;
    if (J == 4) {
        s.g[1] = ld_hint(P.goals + env * 4 + 1, keep);
        float2 t = ld_hint(reinterpret_cast<const float2 *>(P.goals + env * 4 + 2), keep);
        s.g[2] = t.x; s.g[3] = t.y;
    } else if (J % 2 == 0) {
        // rows of J floats are 8-byte aligned: g[1] alone (g[0] stays unread, see above), then pairs
        s.g[1] = ld_hint(P.goals + env * J + 1, keep);
#pragma unroll
        for (int i = 2; i < J; i += 2) {
            const float2 t = ld_hint(reinterpret_cast<const float2 *>(P.goals + env * J + i), keep);
            s.g[i] = t.x; s.g[i + 1] = t.y;
        }
    } else {
#pragma unroll
        for (int i = 1; i < J; ++i) s.g[i] = ld_hint(P.goals + env * J + i, keep);
    }
    if (!RAND) {
        if (env32 >= (int)P.n) {
#pragma unroll
            for (int i = 0; i < J; ++i) s.a[i] = 0.f;
        } else if (J == 4) {
            float4 t = ld_hint(reinterpret_cast<const float4 *>(P.actions + env * 4), stream);
            s.a[0] = t.x; s.a[1] = t.y; s.a[2] = t.z; s.a[3] = t.w;
        } else if (J % 2 == 0) {
#pragma unroll
            for (int i = 0; i < J; i += 2) {
                const float2 t = ld_hint(reinterpret_cast<const float2 *>(P.actions + env * J + i), stream);
                s.a[i] = t.x; s.a[i + 1] = t.y;
            }
        } else {
#pragma unroll
            for (int i = 0; i < J; ++i) s.a[i] = ld_hint(P.actions + env * J + i, stream);
        }
    }
    s.word = ld_hint(P.alive + env, keep);
    s.total = ld_hint(P.total_reward + env, keep);
    s.cnt = ep_shift_of<X>(P) ? 0u : ld_hint(P.counters + env, keep);
}

// One env's row of J actions in a trajectory slice (rollout_kernel's trajectory modes), with the vector widths of
// load_scalars: float4 at J = 4, float2 pairs for even J (rows of J floats are 16- / 8-byte aligned in every slice).
// row = nullptr (an env past the shard's end): zeros, as load_scalars gives it.
template <int J>
__device__ __forceinline__ void load_action_row(const float *row, float *a, uint64_t pol) {
    if (!row) {
#pragma unroll
        for (int i = 0; i < J; ++i) a[i] = 0.f;
    } else if (J == 4) {
        const float4 t = ld_hint(reinterpret_cast<const float4 *>(row), pol);
        a[0] = t.x; a[1] = t.y; a[2] = t.z; a[3] = t.w;
    } else if (J % 2 == 0) {
#pragma unroll
        for (int i = 0; i < J; i += 2) {
            const float2 t = ld_hint(reinterpret_cast<const float2 *>(row + i), pol);
            a[i] = t.x; a[i + 1] = t.y;
        }
    } else {
#pragma unroll
        for (int i = 0; i < J; ++i) a[i] = ld_hint(row + i, pol);
    }
}
template <int J>
__device__ __forceinline__ void store_action_row(float *row, const float *a, uint64_t pol) {
    if (J == 4) {
        st_hint(reinterpret_cast<float4 *>(row), make_float4(a[0], a[1], a[2], a[3]), pol);
    } else if (J % 2 == 0) {
#pragma unroll
        for (int i = 0; i < J; i += 2) st_hint(reinterpret_cast<float2 *>(row + i), make_float2(a[i], a[i + 1]), pol);
    } else {
#pragma unroll
        for (int i = 0; i < J; ++i) st_hint(row + i, a[i], pol);
    }
}

// ---------------------------------------------------------------------------
// What a step does to one env once its kinematics and objective walk are done (per lane, warp-converged):
// reward / done (manytor.py:205-212, 258-259, 170-171), the block's statistics, and the auto-reset with
// objective refresh (manytor.py:219-241; test_single.py:20-21,32).
//   in : neg (ground flag), alive0 / caught (masks), a (the action = new goals), total / eplen (before this step)
//   out: gn (goals after the step), total, alive1, eplen (after the step and a possible reset), rew, done
//   obs_buf   shared-space address of the tile's observations (first observation of a new episode goes there
//             when obs_after_reset is set)
//   pts_buf   shared-space address of a resident copy of the tile's objectives to refresh as well, or 0
// Resets are rare (one env-step in ~550 for random actions), so the warp handles its ending envs one at a
// time and COOPERATIVELY: lane p draws objective p (x <= 32 lanes busy) instead of the one ending lane
// drawing all x while 31 lanes idle.
// FINAL (mt_step_final, mt_rollout_final; needs WOBS): before the reset wipes them, an ending env's return and
// length go to P.final_return / P.final_length, and its obs2 row -- still fp32 at obs_buf, in the public order -- to
// P.final_obs (binary16 when F16, rounded as pack_tile_f16 rounds), lane p copying objective p's three words
// ahead of the first observation of the new episode that replaces them.  Rows of envs that go on are not
// touched.  srow: the first row of the final arrays' slice (0 for step_kernel, s N for step s of a trajectory),
// so env `env` of the slice is row srow + env; the offsets are 64-bit (a slice passes 4 GiB at sizes users run).
// ---------------------------------------------------------------------------
template <int J, bool WOBS, bool FINAL = false, bool F16 = false>
__device__ __forceinline__ void settle_step(const StepParams &P, int lane, int env0, bool valid, int x, int rowlen, bool neg,
                                            uint32_t alive0, uint32_t caught, const float *a, float *gn, float &total,
                                            uint32_t &alive1, uint32_t &eplen, float &rew, uint8_t &done,
                                            uint32_t &ground_steps, unsigned long long *blk_stat, uint32_t obs_buf,
                                            uint32_t pts_buf, size_t srow) {
    static_assert(WOBS || !FINAL, "the final observation is the tile's obs2");
    alive1 = alive0 & ~caught;                                             // manytor.py:168
    rew = (alive1 != alive0) ? 1.0f : 0.0f;
    rew = neg ? -1.0f : rew;
    total += rew;
    eplen = min(eplen + 1u, P.ep_max);
    ground_steps += __popc(__ballot_sync(0xffffffffu, neg & valid));
    const bool term = (alive1 == 0u) | (((P.flags & kTerminateOnGround) != 0) & neg);
    const bool trunc = (P.horizon > 0) & (eplen >= (uint32_t)P.horizon) & !term;
    done = (uint8_t)((term ? 1 : 0) | (trunc ? 2 : 0));
#pragma unroll
    for (int i = 0; i < J; ++i) gn[i] = a[i];                              // goals <- action (manytor.py:184)
    const bool ending = ((P.flags & kAutoReset) != 0) & (done != 0) & valid;
    uint32_t pending = __ballot_sync(0xffffffffu, ending);
    if (pending) {                                                         // warp-uniform, rare
        // fold the ending episodes into the block's statistics: one warp reduction per word and one
        // shared-memory atomic from lane 0 (five same-address GLOBAL atomics per ending env in round 1)
        const uint32_t n_term = __popc(__ballot_sync(0xffffffffu, ending & term));
        const int r_sum = __reduce_add_sync(0xffffffffu, ending ? (int)total : 0);
        const uint32_t l_sum = __reduce_add_sync(0xffffffffu, ending ? eplen : 0u);
        const uint32_t c_sum = __reduce_add_sync(0xffffffffu, ending ? (uint32_t)(x - __popc(alive1)) : 0u);
        if (lane == 0) {
            atomicAdd(&blk_stat[0], (unsigned long long)__popc(pending));
            atomicAdd(&blk_stat[1], (unsigned long long)n_term);
            atomicAdd(&blk_stat[2], (unsigned long long)(long long)r_sum);
            atomicAdd(&blk_stat[3], (unsigned long long)l_sum);
            atomicAdd(&blk_stat[4], (unsigned long long)c_sum);
        }
        if (FINAL && ending) {
            const size_t env = srow + (size_t)(env0 + lane);
            P.final_return[env] = total;
            P.final_length[env] = (int32_t)eplen;
        }
    }
    if (ending) {
#pragma unroll
        for (int i = 0; i < J; ++i) gn[i] = 0.f;
        alive1 = (x >= 32) ? 0xffffffffu : ((1u << x) - 1u);
        total = 0.f;
        eplen = 0u;
    }
    while (pending) {
        const int src = __ffs(pending) - 1;
        pending &= pending - 1u;
        const size_t renv = (size_t)(env0 + src);
        const uint32_t ep = P.episode[renv];                               // resets so far (broadcast load)
        __syncwarp();
        if (lane == src) P.episode[renv] = ep + 1u;
        if (lane < x) {
            if (FINAL) {
                const uint32_t orow = obs_buf + (uint32_t)(src * rowlen + lane * 3) * 4u;
                const size_t i = (srow + renv) * (size_t)rowlen + (size_t)(lane * 3);
                store_obs<F16>(P.final_obs, i, lds_f(orow));
                store_obs<F16>(P.final_obs, i + 1, lds_f(orow + 4));
                store_obs<F16>(P.final_obs, i + 2, lds_f(orow + 8));
            }
            float px, py, pz;
            if (P.obj_stream) {
                const float *srcp = P.obj_stream + (((size_t)(ep % (uint32_t)P.obj_sets) * (size_t)P.n + renv) * x + lane) * 3;
                px = srcp[0]; py = srcp[1]; pz = srcp[2];
            } else {
                sample_point(P, P.env_id_base + (long long)renv, ep, lane, px, py, pz);
            }
            const bool pair = (x & 1) == 0;
            float *grow = P.points + renv * rowlen;
            grow[point_index(pair, lane, 0)] = px;
            grow[point_index(pair, lane, 1)] = py;
            grow[point_index(pair, lane, 2)] = pz;
            if (pts_buf) {
                const uint32_t prow = pts_buf + (uint32_t)(src * rowlen) * 4u;
                sts_f(prow + 4u * point_index(pair, lane, 0), px);
                sts_f(prow + 4u * point_index(pair, lane, 1), py);
                sts_f(prow + 4u * point_index(pair, lane, 2), pz);
            }
            if (WOBS && (P.flags & kObsAfterReset)) {
                Frames f0;
                f0.anchor[0] = P.zero_anchor[0]; f0.anchor[1] = P.zero_anchor[1]; f0.anchor[2] = P.zero_anchor[2];
                f0.catcher[0] = f0.catcher[1] = f0.catcher[2] = 3.0e38f;
                one_objective<true>(px, py, pz, f0, P.catch_tol, true);
                const uint32_t orow = obs_buf + (uint32_t)(src * rowlen + lane * 3) * 4u;
                sts_f(orow, px); sts_f(orow + 4, py); sts_f(orow + 8, pz);
            }
        }
    }
    __syncwarp();
}

// Fill the block's ActionTrig table (before the block's first __syncthreads): entry i = the sin / cos the kernel's own
// evaluation gives for the action value low + i -- the packed evaluation for the reference arm, the scalar one for the
// generic chain, so that a lookup equals what the same kernel without a table computes, bit for bit.
template <int ARM>
__device__ __forceinline__ void fill_action_trig(const StepParams &P, uint32_t table) {
    for (int i = threadIdx.x; i < P.trig_span; i += blockDim.x) {
        const float v = (float)(P.action_low + i);
        float2 sc;
        if (ARM == 0) {
            float2 S, C;
            sincos_deg2(bc2(v), S, C);
            sc = make_float2(S.x, C.x);
        } else {
            sincos_deg(v, sc.x, sc.y);
        }
        sts_f2(table + (uint32_t)i * 8u, sc);
    }
}

// Device-side bookkeeping of a launch, kept OFF the tail of the launch (a returning atomic or a fence at the
// end of every block lengthens the launch by its round trip, and the next step cannot start before the whole
// grid has completed: measured +2 us per step when the ticket sat in the epilogue).
//
// launch_ticket, at the START of a block: every warp calls it once it has read the step index (`seen` carries a
// data dependence on that load); the block's last warp takes the launch's ticket, and the launch's last block --
// at which point every block has read the old step index -- advances it by P.advance and adds the launch's
// env-steps.  The round trip overlaps the warp's first tile fetch.
__device__ __forceinline__ void launch_ticket(const StepParams &P, int lane, int wpb, unsigned long long seen,
                                              unsigned int *warps_seen) {
    if (lane != 0) return;
    if (atomicAdd(warps_seen, 1u + (unsigned)(seen >> 63)) != (unsigned)wpb - 1u) return;
    __threadfence();
    unsigned int *ticket = reinterpret_cast<unsigned int *>(P.ctrl + kCtrlTicket + P.ticket_slot);
    if (atomicAdd(ticket, 1u) == gridDim.x - 1u) {
        atomicExch(ticket, 0u);
        atomicAdd(P.stats, (unsigned long long)P.launch_envs);
        if (P.advance) atomicAdd(P.ctrl + kCtrlStep, (unsigned long long)P.advance);
    }
}

// block_epilogue, at the END: every warp adds its ground-contact count to the block's shared-memory accumulators;
// the block's last warp flushes them with one fire-and-forget atomic per non-zero word.
__device__ __forceinline__ void block_epilogue(const StepParams &P, int lane, int wpb, uint32_t ground_steps,
                                               unsigned long long *blk_stat, unsigned int *warps_done) {
    if (lane != 0) return;
    if (ground_steps) atomicAdd(&blk_stat[5], (unsigned long long)ground_steps);
    __threadfence_block();
    if (atomicAdd(warps_done, 1u) != (unsigned)wpb - 1u) return;
    __threadfence_block();
#pragma unroll
    for (int k = 0; k < kBlockStats; ++k) {
        const unsigned long long v = reinterpret_cast<volatile unsigned long long *>(blk_stat)[k];
        if (v) atomicAdd(P.stats + 1 + k, v);
    }
}

// ---------------------------------------------------------------------------
// the kernel
//   ARM  0 = reference arm closed form (J = 4); else J of the generic chain
//   X    objectives per env, 0 = run-time P.n_obj
//   RAND draw actions in-kernel (mt_rollout_random)   WOBS write observations
//   F16  observations leave as binary16 (pack_tile_f16); only instantiated with WOBS
//   FINAL an ending env's obs2, return and length to P.final_* (mt_step_final, settle_step); only with WOBS
//
// Persistent blocks: one per SM (as many warps as the SM holds; several smaller
// blocks for launches with few tiles), each owning every G-th tile and handing
// them to its warps from a queue in shared memory.  Each warp software-pipelines
// its tiles: while it computes tile i it has tile i+1's scalars in flight to
// registers (coalesced vector loads) and tile i+1's objectives in flight to its
// second shared-memory buffer (TMA bulk copy + mbarrier), and tile i-1's
// observations draining from the other buffer to HBM (TMA bulk store).
// ---------------------------------------------------------------------------
template <int ARM> struct StepBuffers { static constexpr int value = (ARM == 0) ? 2 : 1; };

#ifdef MT_TRACE   // tools/trace_warps.py: per-warp (start ns, end ns, SM id, tiles done) of the last launch
constexpr int kTraceWarps = 8192;
__device__ unsigned long long g_trace[kTraceWarps * 4];
__device__ __forceinline__ unsigned long long trace_now() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#endif

template <int ARM, int X, bool RAND, bool WOBS, bool F16, bool FINAL>
__global__ void __launch_bounds__(((ARM == 0) ? kMaxWarpsRefArm : kMaxWarpsGeneric) * kTile, 1)
step_kernel(const __grid_constant__ StepParams P) {
    static_assert(WOBS || !F16, "F16 is an observation format");
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ int queue_next;
    __shared__ unsigned int warps_done, warps_seen;
    __shared__ unsigned long long blk_stat[kBlockStats];
    constexpr int J = ArmJoints<ARM>::value;
    // Everything that is the same for the whole warp is made PROVABLY warp-uniform (a warp reduction's result
    // lives in a uniform register), so that tile indices, buffer addresses and TMA operands are computed once
    // in the uniform datapath; with `threadIdx.x >> 5` and shuffles ptxas has to assume they diverge and wraps
    // every bulk copy in an elect-and-broadcast loop.
    const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
    const int warp = __reduce_max_sync(0xffffffffu, (int)(threadIdx.x >> 5));
    const int x = X ? X : P.n_obj;
    const int rowlen = 3 * x;
    const uint32_t tile_bytes = (uint32_t)(kTile * rowlen * 4);
    // Tile buffers per warp: two for the reference arm (its kinematics are too short to cover a tile's
    // HBM latency, so tile i+1 is fetched while tile i is still being turned into observations); one
    // for the generic chain, whose long kinematics cover the fetch and where the halved footprint
    // doubles the warps an SM can hold at X = 20.  Buffers and barriers are shared-space byte addresses.
    constexpr int NB = StepBuffers<ARM>::value;
    const uint32_t sbase = smem_addr(smem);
    const uint32_t buf0 = sbase + (uint32_t)(NB * warp) * P.tile_bytes;
    const uint32_t bar0 = sbase + (uint32_t)(NB * wpb) * P.tile_bytes + (uint32_t)(NB * warp) * 8u;
    const uint32_t queue = smem_addr(&queue_next);
    const ActionTrig trig{RAND && P.trig_span > 0 ? bar0 - (uint32_t)(NB * warp) * 8u + (uint32_t)(NB * wpb) * 8u : 0u, P.action_low};
    // The warp's k-th tile uses buffer / barrier k mod NB, and a barrier's phase parity flips every time it
    // completes, so one counter gives buffer, barrier and parity.
    uint32_t k = 0;
    auto buf_of = [&](uint32_t kk) { return buf0 + (NB == 2 ? (kk & 1u) * P.tile_bytes : 0u); };
    auto bar_of = [&](uint32_t kk) { return bar0 + (NB == 2 ? (kk & 1u) * 8u : 0u); };
    auto parity_of = [&](uint32_t kk) { return (NB == 2 ? kk >> 1 : kk) & 1u; };

    // Tile schedule.  Block b owns the tiles b, b + G, b + 2G, ... (G blocks in the grid, one or two per SM),
    // and its warps take them from a queue in shared memory as they become free.  A static share per WARP
    // (the first design) looked balanced -- 7 or 8 tiles each -- but the warp schedulers are not fair: traced
    // per warp (tools/trace_warps.py), the first warp of an SM finished its 8 tiles in 25 us and the last in
    // 50 us, so for the second half of every launch the SM ran with ever fewer warps and ever less latency
    // hiding.  With the queue every warp stays busy until the block's tiles run out.  (One ticket counter
    // for the whole grid was measured earlier: ~37k same-address global atomics per launch serialise in L2;
    // a shared-memory atomic per tile costs nothing.)  What is left is BETWEEN the SMs: a few of them, not the
    // same ones every launch, need up to 12 % longer for their 221 tiles (profiles/r2_warp_trace.txt).  A pool of
    // the launch's last tiles drawn from a global counter -- the draw issued before the kinematics of the tile
    // in hand and read after them, or two tiles ahead -- and a static relief of the highest-numbered blocks
    // were built and measured slower or within the noise (profiles/r2_ab_tile_pool.txt, r2_ab_pool_two_ahead.txt,
    // r2_ab_tail_relief.txt): a second scalar-load site and one more live register cost this kernel 3.6 us.
    const uint64_t pol_stream = P.pol_stream, pol_keep = P.pol_state, pol_store = P.pol_store;
    const int tile_begin = (int)P.tile_begin, tile_end = (int)P.tile_end, n_envs = (int)P.n;
    auto tile_of = [&](int li) -> int {     // (one contiguous range of tiles per block instead: measured, +2.5 us per step)
        const int t = tile_begin + li * (int)gridDim.x + (int)blockIdx.x;
        return t < tile_end ? t : -1;
    };
    auto grab_tile = [&]() -> int {
        int li = 0;
        if (lane == 0) li = atom_add_s(queue, 1);
        return tile_of(__reduce_max_sync(0xffffffffu, li));
    };
    auto fetch_points = [&](int tile, uint32_t buf, uint32_t bar) {   // lane 0 only
        mbar_expect_tx_s(bar, tile_bytes);
        bulk_load_hint_s(buf, P.points + (size_t)tile * (size_t)(kTile * rowlen), tile_bytes, bar, pol_stream);
    };

    if (threadIdx.x == 0) {
        queue_next = wpb;                   // the first wpb tiles of the block go to its warps directly
        warps_done = 0u;
        warps_seen = 0u;
#pragma unroll
        for (int k = 0; k < kBlockStats; ++k) blk_stat[k] = 0ull;
    }
    if (RAND && trig.table) fill_action_trig<ARM>(P, trig.table);
    __syncthreads();
    int cur = tile_of(warp);
#ifdef MT_TRACE
    const unsigned long long trace_t0 = trace_now();
    unsigned trace_tiles = 0;
#endif
    griddep_launch_dependents();            // the next step's grid may start taking free SM slots
    if (cur >= 0 && lane == 0) {
        mbar_init_s(bar0, 1);
        if (NB == 2) mbar_init_s(bar0 + 8u, 1);
        mbar_init_fence();
    }
#ifndef MT_NO_START_PREFETCH
    // While this block waits for the previous step's grid to drain, pull its warps' FIRST tiles towards the L2
    // (objectives by one bulk prefetch, actions by line): the first tile of a warp is the only one whose fetch has
    // nothing to hide behind.  Hints only -- nothing is consumed before the wait below.
    if (cur >= 0) {
        if (lane == 0) bulk_prefetch_l2(P.points + (size_t)cur * (size_t)(kTile * rowlen), tile_bytes);
        if (!RAND && cur * kTile + lane < n_envs) prefetch_l2(P.actions + (size_t)(cur * kTile + lane) * J);
    }
#endif
    griddep_wait();                         // ... but nothing touches the state before the previous step is complete
    uint32_t ground_steps = 0;              // warp-uniform: ground-contact env-steps of this warp's tiles
    // the step index keys the in-kernel action stream; it lives in device memory and was advanced by the
    // previous launch (visible here: griddepcontrol.wait orders after that grid's completion)
    unsigned long long step_index = 0ull;
    if (RAND && cur >= 0) step_index = ld_volatile_u64(P.ctrl + kCtrlStep);
    if (cur < 0) launch_ticket(P, lane, wpb, step_index, &warps_seen);
    if (cur >= 0) {                         // (a warp without a tile still takes part in the block's bookkeeping)
        if (lane == 0) fetch_points(cur, buf0, bar0);
        __syncwarp();
        TileScalars<J> sc;
        load_scalars<J, X, RAND>(P, cur * kTile + lane, sc, pol_keep, pol_stream);
        launch_ticket(P, lane, wpb, step_index, &warps_seen);   // its round trip overlaps the tile's fetch
        int nxt = grab_tile();
        const int ep_shift = ep_shift_of<X>(P);
        const uint32_t amask = ep_shift ? ((1u << ep_shift) - 1u) : 0xffffffffu;

        while (true) {
            const int env0 = cur * kTile, env32 = env0 + lane;
            const size_t env = (size_t)env32;
            const bool full = env0 + kTile <= n_envs;  // warp-uniform
            const bool valid = env32 < n_envs;

            // 1. next tile's scalars on their way to registers
            const uint32_t word = sc.word;
            float total = sc.total;
            uint32_t eplen = sc.cnt;
            TileScalars<J> sn;
            if (nxt >= 0) load_scalars<J, X, RAND>(P, nxt * kTile + lane, sn, pol_keep, pol_stream);

            // 2. kinematics of the current tile (needs no objectives)
            if (RAND) draw_actions(P, step_index, P.env_id_base + env32, J, sc.a);
            Frames f;
            float jbuf[J * 3];
            float *jout = P.joints ? jbuf : nullptr;
            if (ARM == 0) ref_arm<RAND>(sc.g, sc.a, P.substeps, P.inv_div, f, jout, trig);
            else generic_arm<ARM, RAND>(P, sc.g, sc.a, f, jout, trig);
            const bool neg = f.zmin < 0.0f;                                    // manytor.py:191-192

            // 3. next tile's objectives: HBM -> the other buffer by one TMA bulk copy (its previous
            //    contents, tile i-1's observations, have long been read out by their bulk store)
            if (NB == 2 && nxt >= 0 && lane == 0) {
                if (WOBS) bulk_wait_read0();
                fetch_points(nxt, buf_of(k + 1u), bar_of(k + 1u));
            }

            // 4. objectives of the current tile: obs2 in place + catch mask
            const uint32_t buf_cur = buf_of(k);
            mbar_wait_s(bar_of(k), parity_of(k));
            const uint32_t row = buf_cur + (uint32_t)(lane * rowlen) * 4u;
            const uint32_t alive0 = word & amask;
            const uint32_t caught = walk_row<X, WOBS>(row, row, x, f, P.catch_tol, alive0);

            // 5-6. reward / done, statistics, auto-reset with objective refresh
            float gn[J], rew;
            uint32_t alive1;
            uint8_t done;
            if (ep_shift) eplen = word >> ep_shift;
            settle_step<J, WOBS, FINAL, F16>(P, lane, env0, valid, x, rowlen, neg, alive0, caught, sc.a, gn, total, alive1, eplen,
                                             rew, done, ground_steps, blk_stat, buf_cur, 0u, 0);

            // 7. write back: state (coalesced), then the observation tile by one bulk store
            if (J == 4) {
                st_hint(reinterpret_cast<float4 *>(P.goals + env * 4), make_float4(gn[0], gn[1], gn[2], gn[3]), pol_keep);
            } else if (J % 2 == 0) {
#pragma unroll
                for (int i = 0; i < J; i += 2)
                    st_hint(reinterpret_cast<float2 *>(P.goals + env * J + i), make_float2(gn[i], gn[i + 1]), pol_keep);
            } else {
#pragma unroll
                for (int i = 0; i < J; ++i) st_hint(P.goals + env * J + i, gn[i], pol_keep);
            }
            st_hint(P.alive + env, ep_shift ? (alive1 | (eplen << ep_shift)) : alive1, pol_keep);
            st_hint(P.total_reward + env, total, pol_keep);
            if (!ep_shift) st_hint(P.counters + env, eplen, pol_keep);
            if (valid) {
                st_hint(P.reward + env, rew, pol_store);
                st_hint(P.done + env, done, pol_store);
                if (P.joints) {
#pragma unroll
                    for (int i = 0; i < J * 3; ++i) P.joints[env * (J * 3) + i] = jbuf[i];
                }
            }
            if (WOBS) {
                if (full) {
                    if (F16) pack_tile_f16<X>(buf_cur, rowlen, lane);
                    fence_async_smem();
                    __syncwarp();
                    if (lane == 0) {
                        bulk_store_hint_s(obs_at<F16>(P.obs, (size_t)env0 * rowlen), buf_cur, F16 ? tile_bytes / 2 : tile_bytes, pol_store);
                        bulk_commit();
                    }
                } else if (valid) {
                    void *dst = obs_at<F16>(P.obs, env * rowlen);
                    for (int i = 0; i < rowlen; ++i) store_obs<F16>(dst, i, lds_f(row + 4u * i));
                }
            }

#ifdef MT_TRACE
            ++trace_tiles;
#endif
            if (nxt < 0) break;
            if (NB == 1) {   // single buffer: refill it as soon as the observations have been read out
                __syncwarp();
                if (lane == 0) {
                    if (WOBS) bulk_wait_read0();
                    fetch_points(nxt, buf0, bar0);
                }
            }
            cur = nxt;
            nxt = grab_tile();
            sc = sn;
            ++k;
            __syncwarp();
        }
        if (WOBS && lane == 0) bulk_wait_read0();   // shared memory must outlive the last bulk store's read
    }
#ifdef MT_TRACE
    if (lane == 0) {
        const unsigned w = blockIdx.x * wpb + warp;
        unsigned smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        if (w < kTraceWarps) {
            g_trace[w * 4] = trace_t0; g_trace[w * 4 + 1] = trace_now(); g_trace[w * 4 + 2] = smid; g_trace[w * 4 + 3] = trace_tiles;
        }
    }
#endif
    block_epilogue(P, lane, wpb, ground_steps, blk_stat, &warps_done);
}


// ---------------------------------------------------------------------------
// Multi-step random rollout: n_steps x step(action_sample()) in ONE launch (mt_rollout_random).
//
// A tile's step t + 1 depends only on its own step t, so the warp that takes a tile keeps it for all
// P.n_steps steps: pose, alive word and total reward stay in registers, the objectives stay in shared memory
// (fetched once per tile by one TMA bulk copy; a reset refreshes the row in place), and only what a step
// PRODUCES leaves the SM every step -- observations (one bulk store per tile and step, from a second buffer),
// reward, done.  Against n_steps launches of step_kernel<.., RAND = true, ..> this removes, per env-step, the
// read and write of the state (48 B), the read of the objectives (12 X B) and every launch boundary with its
// staggered start and drain; results are bit-identical (same arithmetic, same action stream: step index of
// the launch + s).  Algorithmic bytes per env-step: 12 X + 5 written, plus (48 + 12 X) / n_steps.
//
// MODE (RolloutMode) says where a step's actions come from and where its outputs go.  kDrawLast is
// mt_rollout_random: every step overwrites the same outputs.  The trajectory modes (mt_rollout) write step s's
// observations, reward and done into slice s of [n_steps][N] arrays (slice_row_addr); kDrawTrajectory also stores
// the drawn actions when P.drawn is set, and kActionsTrajectory reads step s's actions from slice s of the caller's
// [n_steps][N][J] array instead of drawing them, evaluating their sin / cos exactly as step_kernel<.., RAND = false, ..>
// does (arbitrary floats: no ActionTrig table), with an L2 prefetch of the next step's action tile that costs no
// register and no shared memory.
// FINAL (mt_rollout_final, trajectory modes with WOBS only): settle_step also writes each ending env's obs2, return
// and length into slice s of P.final_* -- what mt_step_final writes at the s-th step.
// ---------------------------------------------------------------------------
enum class RolloutMode : int {
    kDrawLast = 0,             // in-kernel actions, outputs of the last step (mt_rollout_random)
    kDrawTrajectory = 1,       // in-kernel actions, outputs of every step (mt_rollout, actions_dev = NULL)
    kActionsTrajectory = 2,    // the caller's actions, outputs of every step (mt_rollout)
};

template <int ARM, int X, bool WOBS, bool F16, RolloutMode MODE, bool FINAL = false>
__global__ void __launch_bounds__(((ARM == 0) ? kMaxWarpsRefArm : kMaxWarpsGeneric) * kTile, 1)
rollout_kernel(const __grid_constant__ StepParams P) {
    static_assert(WOBS || !F16, "F16 is an observation format");
    constexpr bool TRAJ = MODE != RolloutMode::kDrawLast;
    static_assert(!FINAL || TRAJ, "final outputs come in slices: trajectory modes only");
    constexpr bool DRAW = MODE != RolloutMode::kActionsTrajectory;
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ int queue_next;
    __shared__ unsigned int warps_done, warps_seen;
    __shared__ unsigned long long blk_stat[kBlockStats];
    constexpr int J = ArmJoints<ARM>::value;
    constexpr int NB = WOBS ? 2 : 1;                      // objectives (+ observations) of the warp's tile
    const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
    const int warp = __reduce_max_sync(0xffffffffu, (int)(threadIdx.x >> 5));
    const int x = X ? X : P.n_obj;
    const int rowlen = 3 * x;
    const uint32_t tile_bytes = (uint32_t)(kTile * rowlen * 4);
    const uint32_t sbase = smem_addr(smem);
    const uint32_t pts = sbase + (uint32_t)(NB * warp) * P.tile_bytes, obuf = pts + P.tile_bytes;
    const uint32_t bar = sbase + (uint32_t)(NB * wpb) * P.tile_bytes + (uint32_t)warp * 8u;
    const ActionTrig trig{P.trig_span > 0 ? sbase + (uint32_t)(NB * wpb) * P.tile_bytes + (uint32_t)wpb * 8u : 0u, P.action_low};
    const uint32_t queue = smem_addr(&queue_next);
    const uint64_t pol_stream = P.pol_stream, pol_keep = P.pol_state, pol_store = P.pol_store;
    const int tile_begin = (int)P.tile_begin, tile_end = (int)P.tile_end, n_envs = (int)P.n;
    auto tile_of = [&](int li) -> int {
        const int t = tile_begin + li * (int)gridDim.x + (int)blockIdx.x;
        return t < tile_end ? t : -1;
    };
    if (threadIdx.x == 0) {
        queue_next = wpb;
        warps_done = 0u;
        warps_seen = 0u;
#pragma unroll
        for (int k = 0; k < kBlockStats; ++k) blk_stat[k] = 0ull;
    }
    if (trig.table) fill_action_trig<ARM>(P, trig.table);
    __syncthreads();
    int cur = tile_of(warp);
    griddep_launch_dependents();
    if (cur >= 0 && lane == 0) {
        mbar_init_s(bar, 1);
        mbar_init_fence();
    }
    griddep_wait();
    uint32_t ground_steps = 0;
    const unsigned long long step0 = cur >= 0 ? ld_volatile_u64(P.ctrl + kCtrlStep) : 0ull;
    launch_ticket(P, lane, wpb, step0, &warps_seen);
    if (cur >= 0) {
        const int ep_shift = ep_shift_of<X>(P);
        const uint32_t amask = ep_shift ? ((1u << ep_shift) - 1u) : 0xffffffffu;
        const uint32_t row = pts + (uint32_t)(lane * rowlen) * 4u, orow = obuf + (uint32_t)(lane * rowlen) * 4u;
        for (uint32_t k = 0; cur >= 0; ++k) {
            const int env0 = cur * kTile, env32 = env0 + lane;
            const size_t env = (size_t)env32;
            const bool full = env0 + kTile <= n_envs, valid = env32 < n_envs;
            if (lane == 0) {                               // objectives: HBM -> shared, once for all the steps
                mbar_expect_tx_s(bar, tile_bytes);
                bulk_load_hint_s(pts, P.points + (size_t)cur * (size_t)(kTile * rowlen), tile_bytes, bar, pol_stream);
            }
            TileScalars<J> sc;
            load_scalars<J, X, true>(P, env32, sc, pol_keep, pol_stream);
            uint32_t alive = sc.word & amask, eplen = ep_shift ? sc.word >> ep_shift : sc.cnt;
            float total = sc.total;
            float rew = 0.f;
            uint8_t done = 0;
            for (int s = 0; s < P.n_steps; ++s) {
                const size_t srow = TRAJ ? (size_t)s * (size_t)n_envs : 0;      // first row of this step's slice
                if constexpr (DRAW) {
                    draw_actions(P, step0 + (unsigned long long)s, P.env_id_base + env32, J, sc.a);
                    if (MODE == RolloutMode::kDrawTrajectory && P.drawn && valid)
                        store_action_row<J>(P.drawn + (srow + env) * J, sc.a, pol_store);
                } else {
                    load_action_row<J>(valid ? P.actions + (srow + env) * J : nullptr, sc.a, pol_stream);
                    // the next step's action tile towards the L2 while this step computes (a hint: aligned full tiles only)
                    // (the address by pointer arithmetic, = slice_row_addr(actions, s + 1, N, env0, 4J): the 64-bit products
                    // of slice_row_addr here cost rollout_kernel<0, 20, .., kActionsTrajectory> a spill)
                    const float *next = P.actions + (srow + (size_t)n_envs + (size_t)env0) * J;
                    if (full && lane == 0 && s + 1 < P.n_steps && bulk_aligned((uintptr_t)next))
                        bulk_prefetch_l2(next, (uint32_t)(kTile * 4 * J));
                }
                Frames f;
                if (ARM == 0) ref_arm<DRAW>(sc.g, sc.a, P.substeps, P.inv_div, f, nullptr, trig);
                else generic_arm<ARM, DRAW>(P, sc.g, sc.a, f, nullptr, trig);
                const bool neg = f.zmin < 0.0f;
                if (s == 0) mbar_wait_s(bar, k & 1u);
                if (WOBS) {                                // the previous step's bulk store must have read the buffer
                    if (lane == 0) bulk_wait_read0();
                    __syncwarp();
                }
                const uint32_t caught = walk_row<X, WOBS>(row, orow, x, f, P.catch_tol, alive);
                float gn[J];
                uint32_t alive1;
                // FINAL: obuf holds this step's obs2 here -- the wait above ordered the previous step's bulk store (which
                // may have packed the buffer to binary16) before walk_row refilled it -- so the final observation is copied
                // out before a reset writes the new episode's first observation over it, as in step_kernel
                settle_step<J, WOBS, FINAL, F16>(P, lane, env0, valid, x, rowlen, neg, alive, caught, sc.a, gn, total, alive1, eplen,
                                                 rew, done, ground_steps, blk_stat, obuf, pts, srow);
                alive = alive1;
#pragma unroll
                for (int i = 0; i < J; ++i) sc.g[i] = gn[i];
                if (valid) {
                    st_hint(P.reward + srow + env, rew, pol_store);
                    st_hint(P.done + srow + env, done, pol_store);
                }
                if (WOBS) {
                    // a full tile whose slice address is misaligned takes the per-lane way (warp-uniform)
                    const bool bulk = TRAJ ? full && slice_bulk_ok((uintptr_t)P.obs, (unsigned long long)s, (unsigned long long)n_envs,
                                                                   (unsigned long long)env0, (unsigned long long)rowlen * (F16 ? 2 : 4))
                                           : full;
                    if (bulk) {
                        if (F16) pack_tile_f16<X>(obuf, rowlen, lane);
                        fence_async_smem();
                        __syncwarp();
                        if (lane == 0) {
                            bulk_store_hint_s(obs_at<F16>(P.obs, (srow + (size_t)env0) * rowlen), obuf, F16 ? tile_bytes / 2 : tile_bytes, pol_store);
                            bulk_commit();
                        }
                    } else if (valid) {
                        void *dst = obs_at<F16>(P.obs, (srow + env) * rowlen);
                        for (int i = 0; i < rowlen; ++i) store_obs<F16>(dst, i, lds_f(orow + 4u * i));
                    }
                }
            }
            // the tile's state goes back to HBM once
            if (J == 4) {
                st_hint(reinterpret_cast<float4 *>(P.goals + env * 4), make_float4(sc.g[0], sc.g[1], sc.g[2], sc.g[3]), pol_keep);
            } else {
#pragma unroll
                for (int i = 0; i < J; ++i) st_hint(P.goals + env * J + i, sc.g[i], pol_keep);
            }
            st_hint(P.alive + env, ep_shift ? (alive | (eplen << ep_shift)) : alive, pol_keep);
            st_hint(P.total_reward + env, total, pol_keep);
            if (!ep_shift) st_hint(P.counters + env, eplen, pol_keep);
            int li = 0;
            if (lane == 0) li = atom_add_s(queue, 1);
            cur = tile_of(__reduce_max_sync(0xffffffffu, li));
            fence_async_smem();                            // a reset's refresh of the row (generic proxy) vs the next bulk copy into it
            __syncwarp();                                  // every lane is done with the objectives before the next fetch
        }
        if (WOBS && lane == 0) bulk_wait_read0();
    }
    block_epilogue(P, lane, wpb, ground_steps, blk_stat, &warps_done);
}

// ---------------------------------------------------------------------------
// Branches: K steps of the caller's actions from copies of chosen envs, leaving the handle untouched (mt_rollout_branches).
//
// Branch m starts from the current state of env B.src[m] -- goals, alive word, episode length and raw objectives --
// and takes the actions of slice s of P.actions ([K][M][J], the layout of mt_rollout) at step s.  A step is the step of
// every other kernel (the arm code, walk_row, settle_step) with kAutoReset cleared in P.flags by the host, so settle_step
// writes nothing and no branch is reset.  A branch ends at the first step whose done byte is non-zero; from then on its
// outputs are frozen: the discounted return (d_0 = 1, d_{s+1} = fl(d_s gamma), G_{s+1} = fl(G_s + d_s r_s), exact
// products as r_s is -1, 0 or +1), the steps executed, the done byte of the ending step (0 after all K) and, when WOBS,
// obs2 of the last executed step.  Nothing of the handle is written: no state, no statistics, no launch ticket.
//
// One lane per branch, a persistent grid over ceil(M / 32) tiles taken from the block's queue, as in rollout_kernel.
// Each lane gathers its source's scalars and copies its source's objective row into its row of the warp's buffer, once
// per call; a gathered row is 12X bytes at an arbitrary row, generally not 16-byte aligned, so this is a per-lane copy and
// not a bulk copy.  The source index is bounds-checked before any load that uses it: a branch whose source is outside
// [0, N) computes as if from row 0 and writes NaN / -1 / 0 and no observation.  A lane past M has the zero goals and
// actions of a padding row.  An ended branch keeps stepping, with its own actions, exactly as an env of a handle without
// auto-reset does: ref_arm picks its sub-pose recurrence for the whole warp (__all_sync), so a lane that froze its pose or
// skipped its actions could change the path, and with it the last bits, of the branches that go on.  The warp leaves
// the step loop once all its branches have ended.
// With WOBS, a step on which some lane of the warp ends (about one env-step in 550 under random actions), and the last
// step, walks the objectives a second time into the warp's second buffer, with the same frames and entry alive mask; each
// lane that ends there, or is still running at the last step, stores its row.  Other steps cost what a rollout without
// observations costs.
// DRAW (mt_rollout_branches_random): steps s < B.n_prefix read slice s of P.actions ([n_prefix][M][J]) as above; every
// later step draws its actions in the kernel, as mt_sample_actions draws them for global env id m at step index
// *B.draw_key + s (mod 2^64): draw_actions with gid = m, whatever the source, M or the handle's step index.  The key is
// read once per lane, after griddep_wait.  A lane past M takes zeros on drawn steps too, so the warp computes what
// branch_kernel<.., DRAW = false> computes when fed the drawn actions, bit for bit.  Drawn steps take sin / cos from the
// block's ActionTrig table (after the per-warp buffers, as in rollout_kernel) when P.trig_span > 0; prefix steps, and
// the zeros of a lane past M (0 is outside a range such as [10, 100), so its entry is not in the table), pass no table
// and evaluate, as DRAW = false does.  No L2 prefetch past the prefix.
// ---------------------------------------------------------------------------
template <int ARM, int X, bool WOBS, bool F16, bool DRAW = false>
__global__ void __launch_bounds__(((ARM == 0) ? kMaxWarpsRefArm : kMaxWarpsGeneric) * kTile, 1)
branch_kernel(const __grid_constant__ StepParams P, const __grid_constant__ BranchParams B) {
    static_assert(WOBS || !F16, "F16 is an observation format");
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ int queue_next;
    constexpr int J = ArmJoints<ARM>::value;
    constexpr int NB = WOBS ? 2 : 1;                      // objectives (+ observations) of the warp's branches
    const int lane = threadIdx.x & 31;
    const int warp = __reduce_max_sync(0xffffffffu, (int)(threadIdx.x >> 5));
    const int x = X ? X : P.n_obj;
    const int rowlen = 3 * x;
    const uint32_t pts = smem_addr(smem) + (uint32_t)(NB * warp) * P.tile_bytes, obuf = pts + P.tile_bytes;
    const uint32_t row = pts + (uint32_t)(lane * rowlen) * 4u, orow = obuf + (uint32_t)(lane * rowlen) * 4u;
    const ActionTrig trig{DRAW && P.trig_span > 0 ? smem_addr(smem) + (uint32_t)(NB * (int)(blockDim.x >> 5)) * P.tile_bytes : 0u,
                          P.action_low};
    const uint32_t queue = smem_addr(&queue_next);
    const uint64_t pol_stream = P.pol_stream, pol_keep = P.pol_state;
    const int tile_end = (int)P.tile_end, n_branches = (int)B.n, n_src = (int)P.n;
    auto tile_of = [&](int li) -> int {
        const int t = li * (int)gridDim.x + (int)blockIdx.x;
        return t < tile_end ? t : -1;
    };
    if (threadIdx.x == 0) queue_next = blockDim.x >> 5;
    if (DRAW && trig.table) fill_action_trig<ARM>(P, trig.table);
    __syncthreads();
    int cur = tile_of(warp);
    griddep_launch_dependents();
    griddep_wait();                                       // nothing is read before the previous grid is complete
    const unsigned long long key = DRAW ? *B.draw_key : 0ull;
    const int ep_shift = ep_shift_of<X>(P);
    const uint32_t amask = ep_shift ? ((1u << ep_shift) - 1u) : 0xffffffffu;
    while (cur >= 0) {
        const int m0 = cur * kTile, m = m0 + lane;
        const bool in = m < n_branches, full = m0 + kTile <= n_branches;
        const long long src64 = in ? (long long)B.src[m] : 0ll;
        const bool ok = in && src64 >= 0 && src64 < (long long)n_src;
        const int src = ok ? (int)src64 : 0;              // every gathered load below reads row `src`, inside [0, N)
        TileScalars<J> sc;
        load_scalars<J, X, true>(P, src, sc, pol_keep, pol_stream);
        if (!in) {
#pragma unroll
            for (int i = 0; i < J; ++i) sc.g[i] = 0.f;
        }
        uint32_t alive = sc.word & amask, eplen = ep_shift ? sc.word >> ep_shift : sc.cnt;
        float total = sc.total;
        const float *prow = P.points + (size_t)src * (size_t)rowlen;
        if ((rowlen & 1) == 0) {                          // even X: rows are 8-byte aligned
            for (int i = 0; i < rowlen; i += 2) sts_f2(row + 4u * i, ld_hint(reinterpret_cast<const float2 *>(prow + i), pol_keep));
        } else {
            for (int i = 0; i < rowlen; ++i) sts_f(row + 4u * i, ld_hint(prow + i, pol_keep));
        }
        bool live = ok;
        float ret = 0.f, disc = 1.f;
        int len = 0;
        uint8_t end_done = 0;
        uint32_t ground_steps = 0;                        // settle_step counts them; nothing reads them here
        for (int s = 0; s < P.n_steps && __any_sync(0xffffffffu, live); ++s) {
            const size_t srow = (size_t)s * (size_t)n_branches;
            const bool drawn = DRAW && s >= B.n_prefix;
            if (drawn) {
                draw_actions(P, key + (unsigned long long)s, (long long)m, J, sc.a);
#pragma unroll
                for (int i = 0; i < J; ++i) sc.a[i] = in ? sc.a[i] : 0.f;
            } else {
                load_action_row<J>(in ? P.actions + (srow + (size_t)m) * J : nullptr, sc.a, pol_stream);
                // the next step's action tile towards the L2 while this step computes (a hint: aligned full tiles only)
                const float *next = P.actions + (srow + (size_t)n_branches + (size_t)m0) * J;
                if (full && lane == 0 && s + 1 < (DRAW ? B.n_prefix : P.n_steps) && bulk_aligned((uintptr_t)next))
                    bulk_prefetch_l2(next, (uint32_t)(kTile * 4 * J));
            }
            Frames f;
            // a lane past M holds zeros, which need not lie in [action_low, action_low + span): it evaluates, never looks up
            const ActionTrig tab = drawn && in ? trig : ActionTrig{0u, 0};
            if (ARM == 0) ref_arm<DRAW>(sc.g, sc.a, P.substeps, P.inv_div, f, nullptr, tab);
            else generic_arm<ARM, DRAW>(P, sc.g, sc.a, f, nullptr, tab);
            const bool neg = f.zmin < 0.0f;
            const uint32_t caught = walk_row<X, false>(row, row, x, f, P.catch_tol, alive);
            float gn[J], rew;
            uint32_t alive1;
            uint8_t done;
            settle_step<J, false>(P, lane, m0, in, x, rowlen, neg, alive, caught, sc.a, gn, total, alive1, eplen, rew, done,
                                  ground_steps, nullptr, 0u, 0u, 0);
            if (WOBS) {
                const bool last = live && (done != 0 || s + 1 == P.n_steps);
                if (__any_sync(0xffffffffu, last)) {      // warp-uniform, rare
                    walk_row<X, true>(row, orow, x, f, P.catch_tol, alive);
                    if (last) {
                        void *dst = obs_at<F16>(P.obs, (size_t)m * rowlen);
                        for (int i = 0; i < rowlen; ++i) store_obs<F16>(dst, i, lds_f(orow + 4u * i));
                    }
                }
            }
            if (live) {
                ret = ret + disc * rew;
                disc = disc * B.gamma;
                len = s + 1;
                end_done = done;
                live = done == 0;
            }
            alive = alive1;
#pragma unroll
            for (int i = 0; i < J; ++i) sc.g[i] = gn[i];
        }
        if (in) {
            B.ret[m] = ok ? ret : __int_as_float(0x7fc00000);
            B.length[m] = ok ? len : -1;
            P.done[m] = ok ? end_done : (uint8_t)0;
        }
        int li = 0;
        if (lane == 0) li = atom_add_s(queue, 1);
        cur = tile_of(__reduce_max_sync(0xffffffffu, li));
        __syncwarp();                                     // every lane is done with its rows before the next tile's copy
    }
}

}  // namespace mt
