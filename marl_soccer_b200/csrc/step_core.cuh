/*
 * step_core.cuh -- per-env arithmetic of the fused soccer step (fp32), shared by every kernel in
 * msoc.cu.  One logical env = one thread; all functions are __host__ __device__ so that the very same
 * arithmetic can also be compiled into the TEST-ONLY host harness tests/hostsim (used to debug
 * parity against the oracle on machines without a GPU; the product never loads it).
 *
 * What is restated here (reference paths relative to soccer_simulation/):
 *   soccer_env.py:118-125      action clip + scale in float32
 *   game/game.py:378-437       Game.step (reward state, forces, space.step, goal, reward, soft reset,
 *                              truncation at max_steps)
 *   game/game.py:399           pymunk Space.step(1/60): Chipmunk2D cpSpaceStep restricted to this scene
 *                              (5 dynamic bodies, 8 static segments), see SURVEY.md Appendix A
 *   game/entities.py:19-28,69-77  custom velocity functions (friction, max_velocity clamp)
 *   game/game.py:129-249       the three spawn modes (Philox4x32-10 instead of PCG64)
 *   game/game.py:258-322       22-float observation frame
 *   marl_vecenv.py:45-53       auto-reset in full-random mode
 *
 * fp32 design notes (the reference computes in fp64):
 *   - narrow phase runs in a frame centred on one of the two bodies so that no O(800) world
 *     coordinate enters a cancellation; contact arms r1/r2 come out of it directly;
 *   - reward shaping (difference of two nearly equal distances, game/game.py:338,345) is computed
 *     from the step displacement:  d_prev - d_cur = -(2 D.dl + dl.dl) / (d_prev + d_cur);
 *   - agent angles are kept wrapped to [-pi, pi] (Cody-Waite 2*pi), the reference keeps them
 *     unwrapped and wraps only in the observation (game/game.py:271-273).
 */
#pragma once
#include <stdint.h>
#include <math.h>
#include <float.h>
#include <string.h>

#if defined(__CUDACC__)
#define MSOC_HD __host__ __device__ __forceinline__
#define MSOC_HD_NOINLINE static __host__ __device__ __noinline__
#else
#define MSOC_HD inline
#define MSOC_HD_NOINLINE static
#endif

/* Debug build only (-DMSOC_CHECKS, marl_soccer_b200/libmsoc_checked.so): bounds and invariant checks of the kernels'
   indices; a failed check sets a bit in a device word that msoc_debug_errors() returns.  (compute-sanitizer is not
   available on the GPU pool this was developed on.) */
#if defined(MSOC_CHECKS) && defined(__CUDA_ARCH__)
extern __device__ unsigned int g_msoc_check_bits;
#define MSOC_CHECK(cond, bit) do { if (!(cond)) atomicOr(&g_msoc_check_bits, 1u << (bit)); } while (0)
#else
#define MSOC_CHECK(cond, bit) do { } while (0)
#endif
enum { CHK_LIST_ENV = 0, CHK_POOL_SLOT = 1, CHK_OVF_SLOT = 2, CHK_CACHE_COUNT = 3, CHK_OBS_ENV = 4, CHK_STEP_COUNTER = 5,
       CHK_CONTACT_COUNT = 6, CHK_FINITE_STATE = 7, CHK_LIST_COUNT = 8 };

namespace msoc {

/* ------------------------------------------------------------------ constants (game/constants.py) */
constexpr float SCREEN_W = 800.0f, SCREEN_H = 600.0f, FIELD_MARGIN = 10.0f;
constexpr float GOAL_Y_BOT = 225.0f, GOAL_Y_TOP = 375.0f; /* 300 -+ 150/2 */
constexpr float AGENT_HALF = 15.0f, BALL_R = 10.0f;
constexpr float FIELD_L = 10.0f, FIELD_R = 790.0f, FIELD_B = 10.0f, FIELD_T = 590.0f;
constexpr float DT = (float)(1.0 / 60.0);
constexpr float PI_F = 3.14159274101257324f;      /* float(pi) */
constexpr float TWO_PI_HI = 6.28318548202514648f; /* float(2 pi) */
constexpr float TWO_PI_LO = -1.74845553e-7f;      /* 2 pi - TWO_PI_HI */
constexpr float SLOP = 0.1f;                      /* cpSpace collisionSlop */
constexpr float BIAS_COEF_OVER_DT = 0.1f * 60.0f; /* (1 - collisionBias^dt) / dt, collisionBias = 0.9^60 */
constexpr int SOLVER_ITERS = 10;                  /* cpSpace iterations default */
/* squared centre distances beyond which two agents / the ball and an agent cannot touch (circumscribed circles + 0.01 px) */
constexpr float AA_REACH2 = (float)((2.0 * 15.0 * 1.4142135623730951 + 0.01) * (2.0 * 15.0 * 1.4142135623730951 + 0.01));
constexpr float BA_REACH2 = (float)((15.0 * 1.4142135623730951 + 10.0 + 0.01) * (15.0 * 1.4142135623730951 + 10.0 + 0.01));

constexpr int N_AGENTS = 4, BALL = 4, STATIC_BODY = 5;
constexpr int FRAME = 22, OBS = 66;
#ifndef MSOC_MAXC
#define MSOC_MAXC 24
#endif
constexpr int MAXC = MSOC_MAXC;      /* contacts solved per env and step */
constexpr int MAX_CACHE = 32; /* == MSOC_MAX_CACHE */

/* pair ids (shared with the oracle and include/msoc.h) */
constexpr int PAIR_AGENT_SEG = 0, PAIR_AGENT_AGENT = 32, PAIR_BALL_AGENT = 38, PAIR_BALL_WALL = 42;

/* restitution / friction products (cpArbiterUpdate: e = ea*eb, u = ua*ub) */
constexpr float E_AGENT_SEG = (float)(0.95 * 0.2), U_AGENT_WALL = (float)(0.2 * 0.8), U_AGENT_GOALLINE = 0.0f;
constexpr float E_AGENT_AGENT = (float)(0.2 * 0.2), U_AGENT_AGENT = (float)(0.8 * 0.8);
constexpr float E_BALL_AGENT = (float)(0.95 * 0.2), U_BALL_AGENT = (float)(0.2 * 0.8);
constexpr float E_BALL_WALL = (float)(0.95 * 0.95), U_BALL_WALL = (float)(0.2 * 0.2);

/* flags word of the per-env counters */
constexpr uint32_t FLAG_CACHE_MASK = 63u, FLAG_MODE_SHIFT = 6, FLAG_MODE_MASK = 3u << 6, FLAG_HAS_BIAS = 1u << 8;
/* set in the CURRENT record of an env whose state was injected after its newest frame had been emitted
   (msoc_set_state): the record keeps the pose behind that frame, the state the next step starts from is in
   Arrays::inject */
constexpr uint32_t FLAG_INJECT = 1u << 9;

/* device-side config: config.json keys as floats plus derived reciprocals */
struct SimCfg {
    float max_velocity, agent_minv, ball_minv, agent_iinv, ball_iinv;
    float agent_friction, ball_friction, force_max, torque_max, max_ang_vel;
    float prox_mult, move_mult, goal_reward, conceded_penalty, alive_penalty, score_diff_mult;
    int32_t max_steps;
    int32_t pad;
    float inv_vmax, inv_wmax; /* 1 / max(max_velocity, 1e-6), 1 / max(max_angular_velocity, 1e-6) (game/game.py:262-264) */
};
MSOC_HD void cfg_derive(SimCfg &s)
{
    s.inv_vmax = 1.0f / fmaxf(s.max_velocity, 1e-6f);
    s.inv_wmax = 1.0f / fmaxf(s.max_ang_vel, 1e-6f);
}

/* State of N envs (device memory in the product, host memory in tests/hostsim).

   An env's state is one 128-byte record; the records live in THREE buffers that rotate: step t reads the state from
   buffer t % 3 and writes the new one to buffer (t + 1) % 3, so after the store the three buffers hold the states of
   steps t-2, t-1 and t -- exactly the poses behind the three frames of the stacked observation
   (soccer_env.py:130-140).  The observation is therefore REBUILT from the three records (3 x 128 B read, L2 hits for
   two of them) instead of being shifted through memory (704 B of 8-byte-aligned history reads per env-step), and a
   frame is the same arithmetic on the same fp32 inputs whenever it is rebuilt: bit-identical to the frame emitted one
   and two steps earlier.  A fresh episode writes its first state to all three buffers (soccer_env.py:92-96). */
constexpr int POSE_F4 = 8; /* float4s per env record: 128 B = one L2 line = four DRAM sectors */
struct Arrays {
    int64_t n;
    float4 *pose[3];   /* per env 8 float4: (px, py, vx, vy) of agent_0..3, ball; agent angles (wrapped); agent angular
                          velocities; (ball angular velocity, steps, flags, running episode return) as bits.
                          flags: arbiter-cache count, spawn mode, has-bias, inject */
    int2 *score;       /* (blue, red), in place: read every step, written on goals and resets only */
    float4 *bias;      /* 4 per env, in place: v_bias agents 0-1, 2-3; (v_bias ball, w_bias agents 0-1); (w_bias agents 2-3, -, -);
                          touched only while the has-bias flag is set */
    float4 *inject;    /* 8 per env or null: the record the next step starts from, for envs flagged FLAG_INJECT */
    uint64_t *seed;    /* per-env Philox key */
    uint32_t *spawn_count;
    uint32_t *cache[2]; /* arbiter cache, ping-pong by step parity: entry j of env e = 3 words at cache_slot(e, j) */
};
/* the step counter lives in device memory and cycles through 0..5 (period of the buffer rotation and of the parity) */
MSOC_HD int buf_prev(int step) { return (step + 2) % 3; } /* state of two steps ago -> oldest frame */
MSOC_HD int buf_cur(int step) { return step % 3; }        /* state the step starts from -> middle frame */
MSOC_HD int buf_next(int step) { return (step + 1) % 3; } /* receives the new state -> newest frame */
MSOC_HD int cache_half(int step) { return step & 1; }

struct Env {
    float px[5], py[5], vx[5], vy[5];
    float ang[4], w[5];
    float vbx[5], vby[5], wb[4];
    float ep_return;
    int32_t steps, score_b, score_r;
    uint32_t flags;
};

/* arbiter cache entry j of env e: (info, accumulated normal impulse, accumulated tangent impulse), the entries of an
   env contiguous (a lane's few live entries share one or two sectors) */
MSOC_HD int64_t cache_slot(int64_t e, int j) { return (e * MAX_CACHE + j) * 3; }

/* ------------------------------------------------------------------------------------ small math */
struct V2 { float x, y; };
MSOC_HD V2 mk(float x, float y) { V2 r; r.x = x; r.y = y; return r; }
MSOC_HD V2 operator+(V2 a, V2 b) { return mk(a.x + b.x, a.y + b.y); }
MSOC_HD V2 operator-(V2 a, V2 b) { return mk(a.x - b.x, a.y - b.y); }
MSOC_HD V2 operator*(V2 a, float s) { return mk(a.x * s, a.y * s); }
MSOC_HD V2 vneg(V2 a) { return mk(-a.x, -a.y); }
MSOC_HD float vdot(V2 a, V2 b) { return a.x * b.x + a.y * b.y; }
MSOC_HD float vcross(V2 a, V2 b) { return a.x * b.y - a.y * b.x; }
MSOC_HD V2 vperp(V2 a) { return mk(-a.y, a.x); }
MSOC_HD V2 vrot(V2 a, V2 r) { return mk(a.x * r.x - a.y * r.y, a.x * r.y + a.y * r.x); }
MSOC_HD V2 vlerp(V2 a, V2 b, float t) { return a * (1.0f - t) + b * t; }
MSOC_HD float clamp01(float t) { return fminf(fmaxf(t, 0.0f), 1.0f); }

/* sin and cos of an angle in [-pi - 1, pi + 1] (agent angles are kept wrapped): quadrant reduction with a
   two-term pi/2 and the Cephes single-precision minimax polynomials on [-pi/4, pi/4]; ~1 ulp, ~30
   instructions, no slow path (the library sincosf carries a Payne-Hanek branch per call site). */
MSOC_HD void sincos_f(float a, float *s, float *c)
{
    const float kf = rintf(a * 0.636619772367581343f);
    const int k = (int)kf;
    float r = fmaf(-kf, 1.57079625129699707031f, a);
    r = fmaf(-kf, 7.54978941586159635335e-08f, r);
    const float z = r * r;
    const float sp = r + r * z * fmaf(z, fmaf(z, -1.9515295891e-4f, 8.3321608736e-3f), -1.6666654611e-1f);
    const float cp = 1.0f + z * fmaf(z, fmaf(z, fmaf(z, 2.443315711809948e-5f, -1.388731625493765e-3f), 4.166664568298827e-2f), -0.5f);
    const bool swap = k & 1;
    const float ss = swap ? cp : sp, cc = swap ? sp : cp;
    *s = (k & 2) ? -ss : ss;
    *c = ((k + 1) & 2) ? -cc : cc;
}
MSOC_HD float rsqrt_f(float x)
{
#if defined(__CUDA_ARCH__)
    return rsqrtf(x);
#else
    return 1.0f / sqrtf(x);
#endif
}
MSOC_HD float wrap_angle(float a)
{
    /* one turn: the common case (|w dt| < pi), bit-for-bit the two-term Cody-Waite subtraction */
    if (a > PI_F) a = (a - TWO_PI_HI) - TWO_PI_LO;
    else if (a < -PI_F) a = (a + TWO_PI_HI) + TWO_PI_LO;
    /* several turns in one step (configs with a huge action_torque_max: the reference default of 100000 spins an
       agent by ~27 rad per step): full range reduction a - 2 pi rint(a / 2 pi), hi/lo split */
    if (fabsf(a) > PI_F) {
        const float k = rintf(a * 0.15915494309189535f);
        a = fmaf(-k, TWO_PI_HI, a);
        a = fmaf(-k, TWO_PI_LO, a);
    }
    return a;
}

/* --------------------------------------------------------------------------------------- Philox */
MSOC_HD void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t out[4])
{
#pragma unroll 1
    for (int r = 0; r < 10; r++) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
MSOC_HD float u01(uint32_t x) { return (float)(x >> 8) * (1.0f / 16777216.0f); }
MSOC_HD float uni(uint32_t x, float lo, float hi) { return fmaf(u01(x), hi - lo, lo); }

/* Spawn positions for one of the three modes (game/game.py:129-249).  Draw order and
   distributions follow the reference; the stream is Philox keyed by (seed, global env index,
   spawn counter).  Returns the incremented spawn counter. */
MSOC_HD_NOINLINE uint32_t spawn_positions(int mode, uint64_t seed, uint64_t gidx, uint32_t spawn_count, float *px, float *py)
{
    if (mode == 1) { /* fixed, game/game.py:129-152 */
        px[0] = 200.0f; py[0] = 198.0f; px[1] = 200.0f; py[1] = 396.0f;
        px[2] = 600.0f; py[2] = 198.0f; px[3] = 600.0f; py[3] = 396.0f;
        px[4] = 400.0f; py[4] = 300.0f;
        return spawn_count;
    }
    uint32_t A[4], B[4], C[4], D[4];
    const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    const uint32_t g0 = (uint32_t)gidx, g1 = (uint32_t)(gidx >> 32);
    philox4x32_10(g0, g1, spawn_count, 0, k0, k1, A);
    philox4x32_10(g0, g1, spawn_count, 1, k0, k1, B);
    philox4x32_10(g0, g1, spawn_count, 2, k0, k1, C);
    philox4x32_10(g0, g1, spawn_count, 3, k0, k1, D);
    const float xmin = 30.0f, xmax = 770.0f, ymin = 30.0f, ymax = 570.0f;
    if (mode == 2) { /* full random, game/game.py:192-249 */
        const bool corners = u01(A[0]) < 0.75f;
        for (int k = 0; k < 2; k++) {
            if (corners) {
                const uint32_t c = A[1 + k] >> 30;
                const bool left = (c == 0 || c == 1), top = (c == 0 || c == 2);
                const float cx = left ? 18.0f : 782.0f, cy = top ? 582.0f : 18.0f;
                px[k] = cx + uni(B[2 * k], -5.0f, 5.0f);
                py[k] = cy + uni(B[2 * k + 1], -5.0f, 5.0f);
            } else {
                px[k] = uni(B[2 * k], xmin, xmax);
                py[k] = uni(B[2 * k + 1], ymin, ymax);
            }
        }
        for (int k = 0; k < 2; k++) { px[2 + k] = uni(C[2 * k], xmin, xmax); py[2 + k] = uni(C[2 * k + 1], ymin, ymax); }
        px[4] = uni(D[0], xmin, xmax); py[4] = uni(D[1], ymin, ymax);
    } else { /* default half-field random, game/game.py:154-190 */
        for (int k = 0; k < 2; k++) { px[k] = uni(B[2 * k], 30.0f, 380.0f); py[k] = uni(B[2 * k + 1], ymin, ymax); }
        for (int k = 0; k < 2; k++) { px[2 + k] = uni(C[2 * k], 420.0f, 770.0f); py[2 + k] = uni(C[2 * k + 1], ymin, ymax); }
        px[4] = 400.0f + uni(D[0], -40.0f, 40.0f); py[4] = 300.0f + uni(D[1], -40.0f, 40.0f);
    }
    return spawn_count + 1;
}

MSOC_HD uint32_t f2u(float f)
{
#if defined(__CUDA_ARCH__)
    return __float_as_uint(f);
#else
    uint32_t u; memcpy(&u, &f, 4); return u;
#endif
}
MSOC_HD float u2f(uint32_t u)
{
#if defined(__CUDA_ARCH__)
    return __uint_as_float(u);
#else
    float f; memcpy(&f, &u, 4); return f;
#endif
}

/* -------------------------------------------------------------------------------- state load/store */
/* what an observation frame is made of (game/game.py:266-321): positions of the five bodies, velocity, angle and
   angular velocity of the four agents */
struct Pose { float px[5], py[5], vx[4], vy[4], ang[4], w[4]; };

MSOC_HD void pose_of(const Env &E, Pose &P)
{
#pragma unroll
    for (int i = 0; i < 5; i++) { P.px[i] = E.px[i]; P.py[i] = E.py[i]; }
#pragma unroll
    for (int i = 0; i < 4; i++) { P.vx[i] = E.vx[i]; P.vy[i] = E.vy[i]; P.ang[i] = E.ang[i]; P.w[i] = E.w[i]; }
}
/* the first seven float4 of an env record */
MSOC_HD void pose_unpack(const float4 *r, Pose &P)
{
#pragma unroll
    for (int i = 0; i < 5; i++) { P.px[i] = r[i].x; P.py[i] = r[i].y; if (i < 4) { P.vx[i] = r[i].z; P.vy[i] = r[i].w; } }
    P.ang[0] = r[5].x; P.ang[1] = r[5].y; P.ang[2] = r[5].z; P.ang[3] = r[5].w;
    P.w[0] = r[6].x; P.w[1] = r[6].y; P.w[2] = r[6].z; P.w[3] = r[6].w;
}
MSOC_HD void pose_pack(const Pose &P, float ball_vx, float ball_vy, float4 *r)
{
#pragma unroll
    for (int i = 0; i < 4; i++) r[i] = make_float4(P.px[i], P.py[i], P.vx[i], P.vy[i]);
    r[4] = make_float4(P.px[4], P.py[4], ball_vx, ball_vy);
    r[5] = make_float4(P.ang[0], P.ang[1], P.ang[2], P.ang[3]);
    r[6] = make_float4(P.w[0], P.w[1], P.w[2], P.w[3]);
}

MSOC_HD void load_env(const Arrays &A, const float4 *rec, int64_t e, Env &E)
{
#pragma unroll
    for (int i = 0; i < 5; i++) {
        const float4 b = rec[i];
        E.px[i] = b.x; E.py[i] = b.y; E.vx[i] = b.z; E.vy[i] = b.w;
    }
    const float4 a = rec[5], w = rec[6], c = rec[7];
    const int2 sc = A.score[e];
    E.ang[0] = a.x; E.ang[1] = a.y; E.ang[2] = a.z; E.ang[3] = a.w;
    E.w[0] = w.x; E.w[1] = w.y; E.w[2] = w.z; E.w[3] = w.w;
    E.w[4] = c.x; E.steps = (int32_t)f2u(c.y); E.flags = f2u(c.z); E.ep_return = c.w;
    E.score_b = sc.x; E.score_r = sc.y;
    if (E.flags & FLAG_HAS_BIAS) {
        const float4 *bp = A.bias + 4 * e;
        const float4 b01 = bp[0], b23 = bp[1], b4w = bp[2], w23 = bp[3];
        E.vbx[0] = b01.x; E.vby[0] = b01.y; E.vbx[1] = b01.z; E.vby[1] = b01.w;
        E.vbx[2] = b23.x; E.vby[2] = b23.y; E.vbx[3] = b23.z; E.vby[3] = b23.w;
        E.vbx[4] = b4w.x; E.vby[4] = b4w.y; E.wb[0] = b4w.z; E.wb[1] = b4w.w;
        E.wb[2] = w23.x; E.wb[3] = w23.y;
    } else {
#pragma unroll
        for (int i = 0; i < 5; i++) { E.vbx[i] = 0.0f; E.vby[i] = 0.0f; }
#pragma unroll
        for (int i = 0; i < 4; i++) E.wb[i] = 0.0f;
    }
}

/* in-place part of the store: the bias velocities (only when there are any) and the has-bias flag */
MSOC_HD void store_env_bias(const Arrays &A, int64_t e, Env &E)
{
    bool any_bias = false;
#pragma unroll
    for (int i = 0; i < 5; i++) any_bias = any_bias || (E.vbx[i] != 0.0f) || (E.vby[i] != 0.0f);
#pragma unroll
    for (int i = 0; i < 4; i++) any_bias = any_bias || (E.wb[i] != 0.0f);
    if (any_bias) {
        float4 *bp = A.bias + 4 * e;
        bp[0] = make_float4(E.vbx[0], E.vby[0], E.vbx[1], E.vby[1]);
        bp[1] = make_float4(E.vbx[2], E.vby[2], E.vbx[3], E.vby[3]);
        bp[2] = make_float4(E.vbx[4], E.vby[4], E.wb[0], E.wb[1]);
        bp[3] = make_float4(E.wb[2], E.wb[3], 0.0f, 0.0f);
        E.flags |= FLAG_HAS_BIAS;
    } else {
        E.flags &= ~FLAG_HAS_BIAS;
    }
}
/* the env record (after store_env_bias) */
MSOC_HD void store_env_record(float4 *rec, const Env &E)
{
#pragma unroll
    for (int i = 0; i < 5; i++) rec[i] = make_float4(E.px[i], E.py[i], E.vx[i], E.vy[i]);
    rec[5] = make_float4(E.ang[0], E.ang[1], E.ang[2], E.ang[3]);
    rec[6] = make_float4(E.w[0], E.w[1], E.w[2], E.w[3]);
    rec[7] = make_float4(E.w[4], u2f((uint32_t)E.steps), u2f(E.flags), E.ep_return);
}
/* bias, record into buffer `buf`, and the score when the caller says it changed (goal, reset, injection) */
MSOC_HD void store_env(const Arrays &A, int buf, int64_t e, Env &E, bool score_dirty)
{
    store_env_bias(A, e, E);
    store_env_record(A.pose[buf] + e * POSE_F4, E);
    if (score_dirty) A.score[e] = make_int2(E.score_b, E.score_r);
}

/* ----------------------------------------------------------------------------- observation frame */
/* game/game.py:258-322; frames for all four agents, 22 floats each.  Pairwise agent vectors are
   computed once and mirrored.  STRIDE is the distance between two agents' frames in `out`.
   The sum of squares is an explicit fma: a frame is rebuilt from its pose by whichever kernel finishes the env one and
   two steps later (Arrays), and must come out bit-identical there whatever the compiler contracts. */
MSOC_HD void unit_mag(float dx, float dy, float &ux, float &uy, float &mag)
{
    const float d2 = fmaf(dx, dx, dy * dy);
    /* mag > 1e-8 (game/game.py:281), else all three are zero; d2 is never subnormal past the test, so the bare
       hardware reciprocal square root (MUFU.RSQ) is what rsqrtf() returns */
#if defined(__CUDA_ARCH__)
    float inv;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(inv) : "f"(d2));
    inv = d2 > 1e-16f ? inv : 0.0f;
#else
    const float inv = d2 > 1e-16f ? 1.0f / sqrtf(d2) : 0.0f;
#endif
    ux = dx * inv; uy = dy * inv; mag = d2 * inv * 0.001f; /* / hypot(800, 600) */
}

/* Frame of agent a (22 floats) from an env record (its first seven float4).  Scaled by reciprocals (within 1.5 ulp
   of the reference's divisions).  u(p_j - p_i) = -u(p_i - p_j) exactly, so the four agents' frames are consistent
   with each other. */
MSOC_HD void frame_of_record(const float4 *rec, int a, const SimCfg &c, float *o)
{
    const int opp = (a & 2) ^ 2;
    const float4 own = rec[a];
    const float2 *xy = reinterpret_cast<const float2 *>(rec); /* positions: float2 0, 2, 4, 6, 8 */
    const float2 mate = xy[2 * (a ^ 1)], o0 = xy[2 * opp], o1 = xy[2 * opp + 2], ball = xy[8];
    const float *fl = reinterpret_cast<const float *>(rec);
    const float ang = fl[20 + a], w = fl[24 + a];
    o[0] = own.z * c.inv_vmax;
    o[1] = own.w * c.inv_vmax;
    o[2] = ang * 0.318309886183790672f;
    o[3] = w * c.inv_wmax;
    unit_mag(mate.x - own.x, mate.y - own.y, o[4], o[5], o[6]);
    unit_mag(o0.x - own.x, o0.y - own.y, o[7], o[8], o[9]);
    unit_mag(o1.x - own.x, o1.y - own.y, o[10], o[11], o[12]);
    unit_mag(ball.x - own.x, ball.y - own.y, o[13], o[14], o[15]);
    const float own_x = (a < 2) ? FIELD_L : FIELD_R, opp_x = (a < 2) ? FIELD_R : FIELD_L;
    unit_mag(own_x - own.x, 300.0f - own.y, o[16], o[17], o[18]);
    unit_mag(opp_x - own.x, 300.0f - own.y, o[19], o[20], o[21]);
}

/* ------------------------------------------------------------------------------------ narrow phase */
struct Manifold { int count; V2 n; V2 p1[2], p2[2]; int key[2]; };
struct Edge { V2 pa, pb; int ia, ib; float r; };
/* box in some frame: v[k] vertices in cpBoxShapeInit2 order, nrm[k] = outward normal of edge k-1 -> k */
struct Box { V2 v[4]; V2 nrm[4]; };

MSOC_HD void make_box(float cs, float sn, V2 off, Box &b)
{
    const float h = AGENT_HALF;
    const V2 a = mk(h * cs + h * sn, h * sn - h * cs); /* R (h,-h) */
    const V2 d = mk(h * cs - h * sn, h * sn + h * cs); /* R (h, h) */
    b.v[0] = off + a; b.v[1] = off + d; b.v[2] = off - a; b.v[3] = off - d;
    b.nrm[0] = mk(sn, -cs); b.nrm[1] = mk(cs, sn); b.nrm[2] = mk(-sn, cs); b.nrm[3] = mk(-cs, -sn);
}

/* Closest features of two convex polygons (a segment is a 2-gon): the (n, d) Chipmunk's GJK
   (separated) / EPA (overlapping) converge to -- exact whenever d <= reach; for shapes further apart than `reach`
   only a lower bound d > reach is returned.  nA[k] / nB[k] are unit outward normals of the edge
   k -> k+1, il2 = 1/|edge|^2 (all edges of one shape have the same length here). */
template <int NA, int NB>
MSOC_HD void closest_convex(const V2 *A, const V2 *nA, float il2A, const V2 *B, const V2 *nB, float il2B, float reach, V2 &n_out, float &d_out)
{
    float best = -INFINITY; V2 bn = mk(0.0f, 0.0f);
#pragma unroll
    for (int k = 0; k < NA; k++) {
        float s = INFINITY;
#pragma unroll
        for (int j = 0; j < NB; j++) s = fminf(s, vdot(B[j] - A[k], nA[k]));
        if (s > best) { best = s; bn = nA[k]; }
    }
#pragma unroll
    for (int k = 0; k < NB; k++) {
        float s = INFINITY;
#pragma unroll
        for (int i = 0; i < NA; i++) s = fminf(s, vdot(A[i] - B[k], nB[k]));
        if (s > best) { best = s; bn = vneg(nB[k]); }
    }
    if (best <= 0.0f) { n_out = bn; d_out = best; return; }
    /* separated along a face normal by more than the caller cares about: the distance is at least that (the caller
       only asks "closer than reach?"), so the closest-feature search below is not needed */
    if (best > reach) { n_out = bn; d_out = best; return; }
    float bd2 = INFINITY; V2 bdel = bn;
#pragma unroll
    for (int k = 0; k < NA; k++) {
        const V2 e = A[(k + 1) % NA] - A[k];
#pragma unroll
        for (int j = 0; j < NB; j++) {
            const V2 rel = B[j] - A[k];
            const float tr = vdot(rel, e) * il2A, t = clamp01(tr);
            /* interior foot point: the offset is exactly along the edge normal (no cancellation of the
               O(800) along-edge component, which would tilt n when the vertex nearly touches the edge) */
            const V2 delta = (tr == t) ? nA[k] * vdot(rel, nA[k]) : rel - e * t;
            const float d2 = vdot(delta, delta);
            if (d2 < bd2) { bd2 = d2; bdel = delta; }
        }
    }
#pragma unroll
    for (int k = 0; k < NB; k++) {
        const V2 e = B[(k + 1) % NB] - B[k];
#pragma unroll
        for (int i = 0; i < NA; i++) {
            const V2 rel = A[i] - B[k];
            const float tr = vdot(rel, e) * il2B, t = clamp01(tr);
            const V2 delta = (tr == t) ? nB[k] * (-vdot(rel, nB[k])) : e * t - rel;
            const float d2 = vdot(delta, delta);
            if (d2 < bd2) { bd2 = d2; bdel = delta; }
        }
    }
    const float inv = rsqrt_f(bd2);
    n_out = bdel * inv; d_out = bd2 * inv;
}

MSOC_HD Edge support_edge_poly(const Box &b, V2 n)
{
    /* cpCollision.c SupportEdgeForPoly */
    float mx = -INFINITY; int i1 = 0;
#pragma unroll
    for (int i = 0; i < 4; i++) { const float d = vdot(b.v[i], n); if (d > mx) { mx = d; i1 = i; } }
    const int i0 = (i1 + 3) & 3, i2 = (i1 + 1) & 3;
    /* dynamic selects instead of dynamic indexing */
    V2 v0, v1, v2, n1, n2;
    v1 = (i1 == 0) ? b.v[0] : (i1 == 1) ? b.v[1] : (i1 == 2) ? b.v[2] : b.v[3];
    v0 = (i0 == 0) ? b.v[0] : (i0 == 1) ? b.v[1] : (i0 == 2) ? b.v[2] : b.v[3];
    v2 = (i2 == 0) ? b.v[0] : (i2 == 1) ? b.v[1] : (i2 == 2) ? b.v[2] : b.v[3];
    n1 = (i1 == 0) ? b.nrm[0] : (i1 == 1) ? b.nrm[1] : (i1 == 2) ? b.nrm[2] : b.nrm[3];
    n2 = (i2 == 0) ? b.nrm[0] : (i2 == 1) ? b.nrm[1] : (i2 == 2) ? b.nrm[2] : b.nrm[3];
    Edge e; e.r = 0.0f;
    if (vdot(n, n1) > vdot(n, n2)) { e.pa = v0; e.ia = i0; e.pb = v1; e.ib = i1; }
    else                           { e.pa = v1; e.ia = i1; e.pb = v2; e.ib = i2; }
    return e;
}

MSOC_HD void contact_points(const Edge &e1, const Edge &e2, V2 n, float d, Manifold &m)
{
    /* cpCollision.c ContactPoints; key = (vertex on shape a) * 4 + (vertex on shape b) */
    m.count = 0;
    const float mindist = e1.r + e2.r;
    if (!(d <= mindist)) return;
    m.n = n;
    const float d_e1_a = vcross(e1.pa, n), d_e1_b = vcross(e1.pb, n);
    const float d_e2_a = vcross(e2.pa, n), d_e2_b = vcross(e2.pb, n);
    const float e1_denom = 1.0f / (d_e1_b - d_e1_a + FLT_MIN);
    const float e2_denom = 1.0f / (d_e2_b - d_e2_a + FLT_MIN);
    {
        const V2 p1 = n * e1.r + vlerp(e1.pa, e1.pb, clamp01((d_e2_b - d_e1_a) * e1_denom));
        const V2 p2 = n * (-e2.r) + vlerp(e2.pa, e2.pb, clamp01((d_e1_a - d_e2_a) * e2_denom));
        if (vdot(p2 - p1, n) <= 0.0f) { m.p1[0] = p1; m.p2[0] = p2; m.key[0] = e1.ia * 4 + e2.ib; m.count = 1; }
    }
    {
        const V2 p1 = n * e1.r + vlerp(e1.pa, e1.pb, clamp01((d_e2_a - d_e1_a) * e1_denom));
        const V2 p2 = n * (-e2.r) + vlerp(e2.pa, e2.pb, clamp01((d_e1_b - d_e2_a) * e2_denom));
        if (vdot(p2 - p1, n) <= 0.0f) {
            const int k = e1.ib * 4 + e2.ia;
            if (m.count == 0) { m.p1[0] = p1; m.p2[0] = p2; m.key[0] = k; }
            else              { m.p1[1] = p1; m.p2[1] = p2; m.key[1] = k; }
            m.count++;
        }
    }
}

/* static segments in setup_field order (game/game.py:50-68) */
struct Seg { V2 a, b, n; float r, il2, u; };
MSOC_HD Seg get_segment(int s)
{
    Seg g;
    if (s < 2) {
        const float y = (s == 0) ? FIELD_B : FIELD_T;
        g.a = mk(FIELD_L, y); g.b = mk(FIELD_R, y); g.n = mk(0.0f, -1.0f);
        g.il2 = 1.0f / (780.0f * 780.0f);
    } else {
        const float x = (s == 2 || s == 3 || s == 6) ? FIELD_L : FIELD_R;
        const float y0 = (s == 2 || s == 4) ? FIELD_B : (s == 3 || s == 5) ? GOAL_Y_TOP : GOAL_Y_BOT;
        const float y1 = (s == 2 || s == 4) ? GOAL_Y_BOT : (s == 3 || s == 5) ? FIELD_T : GOAL_Y_TOP;
        g.a = mk(x, y0); g.b = mk(x, y1); g.n = mk(1.0f, 0.0f);
        const float len = y1 - y0;
        g.il2 = 1.0f / (len * len);
    }
    g.r = (s < 6) ? 2.0f : 1.0f;
    g.u = (s < 6) ? U_AGENT_WALL : U_AGENT_GOALLINE;
    return g;
}

/* cpCollision.c SegmentToPoly (a = segment, b = box), in the frame centred on the box.
   p1 is on the segment side, p2 on the box side; both relative to the box centre. */
MSOC_HD void collide_segment_box(const Seg &g, V2 c, float cs, float sn, Manifold &m)
{
    Box box; make_box(cs, sn, mk(0.0f, 0.0f), box);
    const V2 sv[2] = {g.a - c, g.b - c};
    const V2 sn2[2] = {g.n, vneg(g.n)};
    V2 n; float d;
    if (fminf(vdot(sv[0], sv[0]), vdot(sv[1], sv[1])) > 45.0f * 45.0f) {
        /* Both segment ends are more than 45 px from the box centre while the bounding boxes overlap, so
           the whole box projects onto the segment's interior with >= 38 px to spare at either end.  Then
           neither an end point nor a box face can be the closest feature / the minimum-penetration axis
           (a face tilted by eps against the wall loses by >= 8 |eps| px): the answer is one of the
           segment's two faces, exactly as the general routine finds it, without its 16 point-edge tests. */
        float s0 = INFINITY, s1 = INFINITY;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            s0 = fminf(s0, vdot(box.v[j] - sv[0], g.n));
            s1 = fminf(s1, -vdot(box.v[j] - sv[1], g.n));
        }
        if (s1 > s0) { n = vneg(g.n); d = s1; } else { n = g.n; d = s0; }
    } else {
        const V2 bn[4] = {box.nrm[1], box.nrm[2], box.nrm[3], box.nrm[0]};
        closest_convex<2, 4>(sv, sn2, g.il2, box.v, bn, 1.0f / 900.0f, g.r + 1e-3f, n, d);
    }
    m.count = 0;
    if (d - g.r <= 0.0f) {
        Edge e1; e1.r = g.r;
        if (vdot(g.n, n) > 0.0f) { e1.pa = sv[0]; e1.ia = 0; e1.pb = sv[1]; e1.ib = 1; }
        else                     { e1.pa = sv[1]; e1.ia = 1; e1.pb = sv[0]; e1.ib = 0; }
        contact_points(e1, support_edge_poly(box, vneg(n)), n, d, m);
    }
}

/* cpCollision.c PolyToPoly, in the frame centred on box a; off = centre_b - centre_a */
MSOC_HD void collide_box_box(float csa, float sna, float csb, float snb, V2 off, Manifold &m)
{
    Box A, B; make_box(csa, sna, mk(0.0f, 0.0f), A); make_box(csb, snb, off, B);
    const V2 an[4] = {A.nrm[1], A.nrm[2], A.nrm[3], A.nrm[0]};
    const V2 bn[4] = {B.nrm[1], B.nrm[2], B.nrm[3], B.nrm[0]};
    V2 n; float d;
    closest_convex<4, 4>(A.v, an, 1.0f / 900.0f, B.v, bn, 1.0f / 900.0f, 1e-3f, n, d);
    m.count = 0;
    if (d <= 0.0f) contact_points(support_edge_poly(A, n), support_edge_poly(B, vneg(n)), n, d, m);
}

/* cpCollision.c CircleToPoly (a = ball, b = box), frame centred on the box; c = ball centre.
   p1 = point on the ball, p2 = point on the box. */
MSOC_HD void collide_ball_box(V2 c, float cs, float sn, Manifold &m)
{
    Box box; make_box(cs, sn, mk(0.0f, 0.0f), box);
    m.count = 0;
    float best = -INFINITY; int bk = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) { const float s = vdot(c - box.v[k], box.nrm[k]); if (s > best) { best = s; bk = k; } }
    V2 n, pb; float d;
    if (best <= 0.0f) { /* centre inside the box */
        const V2 nk = (bk == 0) ? box.nrm[0] : (bk == 1) ? box.nrm[1] : (bk == 2) ? box.nrm[2] : box.nrm[3];
        n = vneg(nk); d = best; pb = c - nk * best;
    } else {
        float bd2 = INFINITY; pb = c;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const V2 a0 = box.v[(k + 3) & 3], e = box.v[k] - a0;
            const V2 rel = c - a0;
            const float tr = vdot(rel, e) * (1.0f / 900.0f), t = clamp01(tr);
            const V2 q = (tr == t) ? c - box.nrm[k] * vdot(rel, box.nrm[k]) : a0 + e * t;
            const V2 dl = q - c;
            const float d2 = vdot(dl, dl);
            if (d2 < bd2) { bd2 = d2; pb = q; }
        }
        const float inv = rsqrt_f(bd2);
        d = bd2 * inv; n = (pb - c) * inv;
    }
    if (d <= BALL_R) { m.count = 1; m.n = n; m.key[0] = 0; m.p1[0] = c + n * BALL_R; m.p2[0] = pb; }
}

/* cpCollision.c CircleToSegment (a = ball, b = wall), frame centred on the ball. */
MSOC_HD void collide_ball_segment(const Seg &g, V2 c, Manifold &m)
{
    const V2 a = g.a - c, sd = g.b - g.a;
    const float tr = -vdot(sd, a) * g.il2, t = clamp01(tr);
    /* closest point relative to the ball centre; interior foot point exactly along the wall normal */
    const V2 closest = (tr == t) ? g.n * vdot(a, g.n) : a + sd * t;
    const float mind = BALL_R + g.r;
    const float d2 = vdot(closest, closest);
    m.count = 0;
    if (d2 < mind * mind) {
        V2 n = g.n;
        if (d2 > 0.0f) n = closest * rsqrt_f(d2);
        m.count = 1; m.n = n; m.key[0] = 0;
        m.p1[0] = n * BALL_R;
        m.p2[0] = closest - n * g.r;
    }
}

/* ---------------------------------------------------------------------------------- solver storage */
/* Scratch of the contact path with dynamic indexing.  In the kernel `body` and `con` point into shared
   memory (conflict-free: element (field, index) of thread t lives at (field*K + index)*stride + t), the
   first CON_FAST contacts of an env are kept there and the rare further ones in the per-thread overflow
   array (local memory).  In tests/hostsim both are plain arrays with stride 1. */
#ifndef MSOC_CON_FAST
#define MSOC_CON_FAST 4
#endif
constexpr int CON_FAST = MSOC_CON_FAST; /* contacts per env held in shared memory */
constexpr int CON_FIELDS = 15; /* 14 solver fields + the link to the env's next contact */
constexpr int BODY_FIELDS = 6; /* vx vy w bias_x bias_y bias_w, for the 5 dynamic bodies */
/* contact record: normal, lever arms as scalars (rn = r x n, rt = r x perp(n)), effective masses,
   bounce (restitution e until the pre-step), bias (separation until the pre-step), accumulated
   impulses, meta = a | b<<3 | pair<<6 | key<<12 | first<<16 */
enum { CF_NX, CF_NY, CF_RN1, CF_RT1, CF_RN2, CF_RT2, CF_NMASS, CF_TMASS, CF_BOUNCE, CF_BIAS, CF_JN, CF_JT, CF_JB, CF_META, CF_NEXT };
enum { BF_VX, BF_VY, BF_W, BF_BX, BF_BY, BF_BW };
#if defined(__CUDA_ARCH__)
constexpr int SCR = 32; /* stride between consecutive scratch elements of one lane (shared memory, lane-interleaved) */
#else
constexpr int SCR = 1;
#endif
constexpr int CON_FS = CON_FAST * SCR; /* distance between two fields of a shared-memory contact */
constexpr int BODY_FS = 5 * SCR;       /* distance between two fields of a body */


constexpr int GEOM_WORDS = 22; /* px[5] py[5] cos[4] sin[4] angle[4]: parked while the contact path runs */
enum { GF_PX = 0, GF_PY = 5, GF_CS = 10, GF_SN = 14, GF_ANG = 18 };
#ifndef MSOC_OLD_FAST
#define MSOC_OLD_FAST 4
#endif
constexpr int OLD_FAST = MSOC_OLD_FAST; /* cached arbiter entries (info, jn, jt) preloaded into the scratch; the rest stay in global */
constexpr int SCRATCH_WORDS = BODY_FIELDS * 5 + CON_FIELDS * CON_FAST + GEOM_WORDS + 3 * OLD_FAST; /* per lane */

struct Work {
    float *body; /* field f of body i: body[f*BODY_FS + i*SCR] */
    float *pool; /* contact records of the whole warp: field f of slot s: pool[f*CON_FS + s], CON_FS slots handed out on demand
                    (an env takes as many as it has contacts; on the average that is far fewer than CON_FAST per lane) */
    int *pool_count; /* slots handed out so far (shared by the warp) */
    float *geom; /* word g: geom[g*SCR] */
    float *isl;  /* island modes: contact slot k, field f: isl[(k*ISL_FIELDS + f)*SCR] (in the kernel: the idle contact pool) */
    float *old;  /* preloaded cache entry j < OLD_FAST: info old[j*SCR] (bits), jn old[(OLD_FAST+j)*SCR], jt old[(2*OLD_FAST+j)*SCR] */
    float (*ovf)[CON_FIELDS]; /* only when the pool is exhausted (rare): caller-provided array of MAXC - CON_FAST records, field
                                 stride 1 (a pointer, so that the scalar members of this struct stay in registers) */
    int nc, overflow;
    int head, tail, n_ovf; /* the env's contacts form a linked list in arbiter order: refs >= 0 are pool slots, < 0 overflow records */
    uint64_t touched;
};
/* base pointer and field stride of the contact with reference p */
constexpr int NIL = 0x7fffffff;
MSOC_HD float *contact_ptr(const Work &W, int p, int &fs)
{
    if (p >= 0) { fs = CON_FS; return W.pool + p; }
    fs = 1; return &W.ovf[-1 - p][0];
}
/* a new record at the end of the env's list; NIL if the env already has MAXC contacts */
MSOC_HD int contact_alloc(Work &W)
{
    if (W.nc >= MAXC) { W.overflow++; return NIL; }
    int p;
#if defined(__CUDA_ARCH__)
    const int s_ = atomicAdd(W.pool_count, 1);
#else
    const int s_ = (*W.pool_count)++;
#endif
    if (s_ < CON_FS) p = s_;
    else {
        if (W.n_ovf >= MAXC - CON_FAST) { W.overflow++; return NIL; }
        p = -1 - W.n_ovf++;
    }
    MSOC_CHECK(p < CON_FS && s_ >= 0, CHK_POOL_SLOT);
    MSOC_CHECK(p >= -(MAXC - CON_FAST), CHK_OVF_SLOT);
    MSOC_CHECK(W.nc < MAXC, CHK_CONTACT_COUNT);
    int fs; float *cp = contact_ptr(W, p, fs);
    cp[CF_NEXT * fs] = u2f((uint32_t)NIL);
    if (W.nc == 0) W.head = p;
    else { int fs2; float *tp = contact_ptr(W, W.tail, fs2); tp[CF_NEXT * fs2] = u2f((uint32_t)p); }
    W.tail = p; W.nc++;
    return p;
}

struct CacheIO {
    const uint32_t *oldc; /* previous step's entries of this env: 3 words each */
    uint32_t *newc;       /* next step's */
    int64_t n, e;
    int old_count;
};

/* old (previous step) arbiter cache entry j: the first OLD_FAST come from the scratch (preloaded with one
   batch of independent loads), the rare further ones from global memory */
MSOC_HD uint32_t old_info_at(const Work &W, const CacheIO &cio, int j)
{
    return j < OLD_FAST ? f2u(W.old[j * SCR]) : cio.oldc[3 * j];
}
MSOC_HD float old_jn_at(const Work &W, const CacheIO &cio, int j)
{
    return j < OLD_FAST ? W.old[(OLD_FAST + j) * SCR] : u2f(cio.oldc[3 * j + 1]);
}
MSOC_HD float old_jt_at(const Work &W, const CacheIO &cio, int j)
{
    return j < OLD_FAST ? W.old[(2 * OLD_FAST + j) * SCR] : u2f(cio.oldc[3 * j + 2]);
}

/* friction product of a pair id (cpArbiterUpdate u = ua*ub) */
MSOC_HD float pair_friction(int pair)
{
    if (pair < PAIR_AGENT_AGENT) return ((pair & 7) < 6) ? U_AGENT_WALL : U_AGENT_GOALLINE;
    if (pair < PAIR_BALL_AGENT) return U_AGENT_AGENT;
    if (pair < PAIR_BALL_WALL) return U_BALL_AGENT;
    return U_BALL_WALL;
}

/* cpSpaceCollideShapes + cpArbiterUpdate for one touching pair: append the manifold's contacts,
   carry jnAcc/jtAcc of equal-key contacts from the cache, decide first-contact state. */
MSOC_HD void add_contacts(Work &W, const CacheIO &cio, int pair, int a, int b, float e, const Manifold &m,
                          V2 r1_off, V2 r2_off)
{
    W.touched |= (1ull << pair);
    bool first = true;
    float cjn[2] = {0.0f, 0.0f}, cjt[2] = {0.0f, 0.0f};
    for (int j = 0; j < cio.old_count; j++) {
        const uint32_t info = old_info_at(W, cio, j);
        if ((int)(info & 63u) != pair) continue;
        if (((info >> 10) & 3u) == 0u) first = false;
        const int key = (int)((info >> 6) & 15u);
        const float ojn = old_jn_at(W, cio, j), ojt = old_jt_at(W, cio, j);
        if (m.count > 0 && key == m.key[0]) { cjn[0] = ojn; cjt[0] = ojt; }
        if (m.count > 1 && key == m.key[1]) { cjn[1] = ojn; cjt[1] = ojt; }
    }
    for (int i = 0; i < m.count; i++) {
        const int k = contact_alloc(W);
        if (k == NIL) continue;
        const V2 p1 = (i == 0) ? m.p1[0] : m.p1[1], p2 = (i == 0) ? m.p2[0] : m.p2[1];
        const int key = (i == 0) ? m.key[0] : m.key[1];
        /* stored so that body b is dynamic: a contact (a dynamic, b static) is kept as (static, a) with the
           normal negated and the arms exchanged -- the scalars vrn, vrt, jn, jt, dist are invariant */
        const bool flip = (b == STATIC_BODY);
        const V2 n_ = flip ? vneg(m.n) : m.n, t = vperp(n_);
        const V2 r1 = flip ? p2 - r2_off : p1 - r1_off, r2 = flip ? p1 - r1_off : p2 - r2_off;
        const int a_ = flip ? b : a, b_ = flip ? a : b;
        int fs; float *cp = contact_ptr(W, k, fs);
        cp[CF_NX * fs] = n_.x; cp[CF_NY * fs] = n_.y;
        cp[CF_RN1 * fs] = vcross(r1, n_); cp[CF_RT1 * fs] = vcross(r1, t);
        cp[CF_RN2 * fs] = vcross(r2, n_); cp[CF_RT2 * fs] = vcross(r2, t);
        cp[CF_JN * fs] = (i == 0) ? cjn[0] : cjn[1];
        cp[CF_JT * fs] = (i == 0) ? cjt[0] : cjt[1];
        cp[CF_JB * fs] = 0.0f;
        cp[CF_BOUNCE * fs] = e; /* restitution until the pre-step turns it into the bounce velocity */
        /* signed separation along n from the contact points themselves (translation invariant):
           cpArbiterPreStep dist = ((r2 - r1) + (pb - pa)) . n */
        cp[CF_BIAS * fs] = vdot(p2 - p1, m.n);
        cp[CF_META * fs] = u2f((uint32_t)a_ | ((uint32_t)b_ << 3) | ((uint32_t)pair << 6) | ((uint32_t)key << 12) | ((first ? 1u : 0u) << 16));
    }
}

/* body i's inverse mass / inverse moment; i = 5 is the static body */
MSOC_HD float inv_mass(const SimCfg &c, int i) { return i < 4 ? c.agent_minv : (i == 4 ? c.ball_minv : 0.0f); }
MSOC_HD float inv_moment(const SimCfg &c, int i) { return i < 4 ? c.agent_iinv : (i == 4 ? c.ball_iinv : 0.0f); }

/* cpArbiterPreStep for one contact (FS = field stride of the record): effective masses, bias velocity,
   bounce = e * (relative normal velocity BEFORE the velocity update).  With rn = r x n:
   (v + w perp(r)) . n = v.n + w rn. */
template <int FS>
MSOC_HD void prestep_contact(float *cp, const float *body, const SimCfg &c)
{
    const uint32_t meta = f2u(cp[CF_META * FS]);
    const int a = meta & 7u, b = (meta >> 3) & 7u;
    const float nx = cp[CF_NX * FS], ny = cp[CF_NY * FS];
    const float rn1 = cp[CF_RN1 * FS], rt1 = cp[CF_RT1 * FS], rn2 = cp[CF_RN2 * FS], rt2 = cp[CF_RT2 * FS];
    const float ma = inv_mass(c, a), ia = inv_moment(c, a), mb = inv_mass(c, b), ib = inv_moment(c, b);
    cp[CF_NMASS * FS] = 1.0f / (ma + ia * rn1 * rn1 + mb + ib * rn2 * rn2);
    cp[CF_TMASS * FS] = 1.0f / (ma + ia * rt1 * rt1 + mb + ib * rt2 * rt2);
    cp[CF_BIAS * FS] = -BIAS_COEF_OVER_DT * fminf(0.0f, cp[CF_BIAS * FS] + SLOP);
    float vn = 0.0f;
    if (a < 5) { const float *pa = body + a * SCR; vn -= pa[BF_VX * BODY_FS] * nx + pa[BF_VY * BODY_FS] * ny + pa[BF_W * BODY_FS] * rn1; }
    if (b < 5) { const float *pb = body + b * SCR; vn += pb[BF_VX * BODY_FS] * nx + pb[BF_VY * BODY_FS] * ny + pb[BF_W * BODY_FS] * rn2; }
    cp[CF_BOUNCE * FS] = vn * cp[CF_BOUNCE * FS];
}

/* cpArbiterApplyCachedImpulse for one contact (skipped for arbiters in their first step) */
template <int FS>
MSOC_HD void warmstart_contact(const float *cp, float *body, const SimCfg &c)
{
    const uint32_t meta = f2u(cp[CF_META * FS]);
    if ((meta >> 16) & 1u) return;
    const int a = meta & 7u, b = (meta >> 3) & 7u;
    const float nx = cp[CF_NX * FS], ny = cp[CF_NY * FS], jn = cp[CF_JN * FS], jt = cp[CF_JT * FS];
    const float jx = nx * jn - ny * jt, jy = ny * jn + nx * jt; /* n jn + perp(n) jt */
    if (a < 5) {
        float *pa = body + a * SCR;
        const float ma = inv_mass(c, a), ia = inv_moment(c, a);
        pa[BF_VX * BODY_FS] -= jx * ma; pa[BF_VY * BODY_FS] -= jy * ma;
        pa[BF_W * BODY_FS] -= ia * (cp[CF_RN1 * FS] * jn + cp[CF_RT1 * FS] * jt);
    }
    if (b < 5) {
        float *pb = body + b * SCR;
        const float mb = inv_mass(c, b), ib = inv_moment(c, b);
        pb[BF_VX * BODY_FS] += jx * mb; pb[BF_VY * BODY_FS] += jy * mb;
        pb[BF_W * BODY_FS] += ib * (cp[CF_RN2 * FS] * jn + cp[CF_RT2 * FS] * jt);
    }
}

/* The solver keeps the second body of the contact it is working on in registers: consecutive contacts of
   an arbiter list usually share it (an agent's wall contacts), so the Gauss-Seidel chain does not go
   through shared memory between them.  Contacts are stored so that body b is always dynamic. */
struct BodyCache { int cur; float vx, vy, w, bx, by, bw; };
MSOC_HD void bc_flush(BodyCache &bc, float *body)
{
    if (bc.cur >= 0) {
        float *p = body + bc.cur * SCR;
        p[BF_VX * BODY_FS] = bc.vx; p[BF_VY * BODY_FS] = bc.vy; p[BF_W * BODY_FS] = bc.w;
        p[BF_BX * BODY_FS] = bc.bx; p[BF_BY * BODY_FS] = bc.by; p[BF_BW * BODY_FS] = bc.bw;
    }
}
MSOC_HD void bc_acquire(BodyCache &bc, float *body, int b)
{
    if (bc.cur == b) return;
    bc_flush(bc, body);
    const float *p = body + b * SCR;
    bc.vx = p[BF_VX * BODY_FS]; bc.vy = p[BF_VY * BODY_FS]; bc.w = p[BF_W * BODY_FS];
    bc.bx = p[BF_BX * BODY_FS]; bc.by = p[BF_BY * BODY_FS]; bc.bw = p[BF_BW * BODY_FS];
    bc.cur = b;
}

/* cpArbiterApplyImpulse for one contact: bias impulse on the bias velocities, then normal impulse with
   restitution and Coulomb friction clamped by the accumulated normal impulse. */
template <int FS>
MSOC_HD void solve_contact(float *cp, float *body, const SimCfg &c, BodyCache &bc)
{
    const uint32_t meta = f2u(cp[CF_META * FS]);
    const int a = meta & 7u, b = (meta >> 3) & 7u;
    if (a == bc.cur) { bc_flush(bc, body); bc.cur = -1; }
    bc_acquire(bc, body, b);
    const float nx = cp[CF_NX * FS], ny = cp[CF_NY * FS];
    const float rn1 = cp[CF_RN1 * FS], rt1 = cp[CF_RT1 * FS], rn2 = cp[CF_RN2 * FS], rt2 = cp[CF_RT2 * FS];
    float *pa = body + a * SCR;
    float vrn = bc.vx * nx + bc.vy * ny + bc.w * rn2;
    float vrt = bc.vy * nx - bc.vx * ny + bc.w * rt2;
    float vbn = bc.bx * nx + bc.by * ny + bc.bw * rn2;
    if (a < 5) {
        const float vx = pa[BF_VX * BODY_FS], vy = pa[BF_VY * BODY_FS], w = pa[BF_W * BODY_FS];
        vrn -= vx * nx + vy * ny + w * rn1;
        vrt -= vy * nx - vx * ny + w * rt1;
        vbn -= pa[BF_BX * BODY_FS] * nx + pa[BF_BY * BODY_FS] * ny + pa[BF_BW * BODY_FS] * rn1;
    }
    const float nMass = cp[CF_NMASS * FS];
    const float jbOld = cp[CF_JB * FS], jnOld = cp[CF_JN * FS], jtOld = cp[CF_JT * FS];
    const float jbNew = fmaxf(jbOld + (cp[CF_BIAS * FS] - vbn) * nMass, 0.0f);
    const float jnNew = fmaxf(jnOld - (cp[CF_BOUNCE * FS] + vrn) * nMass, 0.0f);
    const float jtMax = pair_friction((int)((meta >> 6) & 63u)) * jnNew;
    const float jtNew = fminf(fmaxf(jtOld - vrt * cp[CF_TMASS * FS], -jtMax), jtMax);
    cp[CF_JB * FS] = jbNew; cp[CF_JN * FS] = jnNew; cp[CF_JT * FS] = jtNew;
    const float djb = jbNew - jbOld, djn = jnNew - jnOld, djt = jtNew - jtOld;
    const float jx = nx * djn - ny * djt, jy = ny * djn + nx * djt;
    {
        const float mb = inv_mass(c, b), ib = inv_moment(c, b);
        bc.bx += nx * djb * mb; bc.by += ny * djb * mb; bc.bw += ib * rn2 * djb;
        bc.vx += jx * mb; bc.vy += jy * mb; bc.w += ib * (rn2 * djn + rt2 * djt);
    }
    if (a < 5) {
        const float ma = inv_mass(c, a), ia = inv_moment(c, a);
        pa[BF_BX * BODY_FS] -= nx * djb * ma; pa[BF_BY * BODY_FS] -= ny * djb * ma; pa[BF_BW * BODY_FS] -= ia * rn1 * djb;
        pa[BF_VX * BODY_FS] -= jx * ma; pa[BF_VY * BODY_FS] -= jy * ma; pa[BF_W * BODY_FS] -= ia * (rn1 * djn + rt1 * djt);
    }
}

MSOC_HD bool bb_overlap(float cx, float cy, float R, float l, float b, float r, float t)
{
    return (cx - R <= r) && (l <= cx + R) && (cy - R <= t) && (b <= cy + R);
}

MSOC_HD int ctz32(uint32_t x)
{
#if defined(__CUDA_ARCH__)
    return __ffs((int)x) - 1;
#else
    return __builtin_ctz(x);
#endif
}
MSOC_HD int popc32(uint32_t x)
{
#if defined(__CUDA_ARCH__)
    return __popc(x);
#else
    return __builtin_popcount(x);
#endif
}

/* ------------------------------------------------------------------------------------------ step */
struct StepOut {
    float reward;
    float reward_r;       /* red's reward: set by the TEAMS instances of env_step only */
    uint8_t done;
    int8_t goal;
    bool fresh_episode;   /* auto-reset happened: obs = 3 copies of the new frame */
    bool score_dirty;     /* the score changed (goal, auto-reset): store_env must write it */
    float finished_return; /* blue return of the episode that ended on this step */
    int n_contacts, overflow;
    int32_t score_b, score_r; /* info["score"] of this step (before any auto-reset) */
};

/* Full reset of one env (Game.reset, game/game.py:76-118): bodies re-created (all velocities,
   biases and cached arbiters dropped), spawn, counters cleared. */
MSOC_HD void env_full_reset(Env &E, int mode, uint64_t seed, uint64_t gidx, uint32_t &spawn_count)
{
    float px[5], py[5];
    spawn_count = spawn_positions(mode, seed, gidx, spawn_count, px, py);
#pragma unroll
    for (int i = 0; i < 5; i++) {
        E.px[i] = px[i]; E.py[i] = py[i]; E.vx[i] = 0.0f; E.vy[i] = 0.0f; E.w[i] = 0.0f;
        E.vbx[i] = 0.0f; E.vby[i] = 0.0f;
    }
#pragma unroll
    for (int i = 0; i < 4; i++) { E.wb[i] = 0.0f; E.ang[i] = (i < 2) ? 0.0f : PI_F; }
    E.steps = 0; E.score_b = 0; E.score_r = 0; E.ep_return = 0.0f;
    E.flags = ((uint32_t)mode << FLAG_MODE_SHIFT); /* cache count 0, no bias */
}

/* One env-step (everything except the observation frames, which the caller builds from the stored records afterwards).
   MODE_FAST is the contact-free mode of the streaming kernel: it returns false -- leaving E meaningless and every array
   untouched -- as soon as the broad phase finds a candidate pair, and reports the env's work class in `load`; such envs
   are then stepped by the contact kernel in the mode of their class (always returns true), batched by class:
     MODE_LIGHT  exactly one candidate pair, agent x segment: narrow phase + solver for one body and <= 2 contacts in registers
     MODE_PAIR   exactly one agent x agent / ball x agent candidate pair (+ at most one agent x segment pair): one island of
                 two bodies and <= 4 contacts, or that island and a single-body one
     MODE_MULTI  only static candidates, at most two per body: up to five single-body islands, solved one after the other
     MODE_FULL   anything else: the general Chipmunk path (contact pool, linked arbiter-ordered list, all five bodies)
   The modes are run-time values under a compile-time mask (ALLOWED): one copy of the prologue and epilogue per kernel.
   W is only touched by MODE_PAIR / MODE_MULTI (bodies, poses, island slots) and MODE_FULL (everything). */
enum { MODE_FULL = 0, MODE_FAST = 1, MODE_LIGHT = 2, MODE_PAIR = 3, MODE_MULTI = 4 };
/* work classes of the envs the contact-free mode declines (`load`): each has its own list and its own code path */
enum { LOAD_LIGHT = 0, /* exactly one candidate pair, agent x segment: MODE_LIGHT */
       LOAD_HEAVY = 1, /* anything else: the general Chipmunk path, MODE_FULL */
       LOAD_PAIR = 2,  /* exactly one agent x agent or ball x agent candidate pair, at most one agent x segment pair beside it: MODE_PAIR */
       LOAD_MULTI = 3, /* only static candidates (agent x segment, ball x wall), at most two per body: MODE_MULTI */
       N_LOADS = 4 };
MSOC_HD int mode_of_load(int load) { return load == LOAD_LIGHT ? MODE_LIGHT : load == LOAD_PAIR ? MODE_PAIR : load == LOAD_MULTI ? MODE_MULTI : MODE_FULL; }
MSOC_HD float sel4(const float *a, int i) { return i == 0 ? a[0] : i == 1 ? a[1] : i == 2 ? a[2] : a[3]; }

/* Contact slots of an island (MODE_PAIR, MODE_MULTI; Work::isl): the solver fields of a pool record.  The islands of
   these modes share no dynamic body with anything else, so solving them on their own, contacts in arbiter order, is the
   same arithmetic as the general path's sweep over all contacts of the env (bit-identical on the host build:
   tests/test_hostsim_parity.py). */
enum { IF_NX, IF_NY, IF_RN1, IF_RT1, IF_RN2, IF_RT2, IF_NM, IF_TM, IF_BIAS, IF_BNC, IF_JN, IF_JT, IF_JB, IF_INFO, ISL_FIELDS };
enum { IF_U = IF_RN1 }; /* a static x body contact has no first arm: its slot carries the friction coefficient there */
constexpr int ISL_SLOTS = 4;

/* Shaping term of one distance (game/game.py:338,345): |d| - |d + l|, the decrease of the distance d over the step
   displacement l, as the difference of squares over the sum of the two distances (no cancellation); 0 if both are 0. */
MSOC_HD float distance_drop(float dx, float dy, float lx, float ly)
{
    const float dp = sqrtf(dx * dx + dy * dy);
    const float nx_ = dx + lx, ny_ = dy + ly;
    const float dc = sqrtf(nx_ * nx_ + ny_ * ny_);
    const float den = dp + dc;
    return den > 0.0f ? -(2.0f * (dx * lx + dy * ly) + (lx * lx + ly * ly)) / den : 0.0f;
}

/* TEAMS: red's reward too (out.reward_r), blue's reward on the field mirrored about x = 400 (include/msoc.h,
   msoc_step_teams).  The TEAMS = false instances are the blue-only step, instruction for instruction. */
template <bool TEAMS = false>
MSOC_HD bool env_step(const int MODE, const int ALLOWED, Env &E, const float *act, const SimCfg &c, const Arrays &A, int cur, int64_t e,
                      uint64_t gidx, uint32_t step_flags, Work &W, StepOut &out, int &load)
{
    /* ALLOWED: bit m set = the caller may pass MODE == m (a compile-time constant at every call site, so that a kernel
       only carries the code of its own modes even where MODE itself is a run-time value) */
    const bool FAST = (ALLOWED & (1 << MODE_FAST)) && MODE == MODE_FAST, LIGHT = (ALLOWED & (1 << MODE_LIGHT)) && MODE == MODE_LIGHT;
    const bool PAIR = (ALLOWED & (1 << MODE_PAIR)) && MODE == MODE_PAIR, MULTI = (ALLOWED & (1 << MODE_MULTI)) && MODE == MODE_MULTI;
    const bool FULL = (ALLOWED & (1 << MODE_FULL)) && MODE == MODE_FULL;
    /* register-only modes: the first four cached arbiter entries (one or two sectors) are fetched right away, so that
       their latency is covered by the prologue */
    uint32_t pc[12];
#pragma unroll
    for (int k = 0; k < 12; k++) pc[k] = 0u;
    if ((LIGHT || PAIR || MULTI) && (E.flags & FLAG_CACHE_MASK) != 0u) {
#if defined(__CUDA_ARCH__)
        const uint4 *q = reinterpret_cast<const uint4 *>(A.cache[cur] + cache_slot(e, 0));
        const uint4 q0 = q[0], q1 = q[1], q2 = q[2];
        pc[0] = q0.x; pc[1] = q0.y; pc[2] = q0.z; pc[3] = q0.w; pc[4] = q1.x; pc[5] = q1.y; pc[6] = q1.z; pc[7] = q1.w;
        pc[8] = q2.x; pc[9] = q2.y; pc[10] = q2.z; pc[11] = q2.w;
#else
        for (int k = 0; k < 12; k++) pc[k] = A.cache[cur][cache_slot(e, 0) + k];
#endif
    }
    /* ---- soccer_env.py:118-125: clip to [-1, 1], scale in float32 */
    float Fx[4], Fy[4], Tq[4];
    float cs[4], sn[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const float a0 = fminf(fmaxf(act[3 * i + 0], -1.0f), 1.0f) * c.force_max;
        const float a1 = fminf(fmaxf(act[3 * i + 1], -1.0f), 1.0f) * c.force_max;
        Tq[i] = fminf(fmaxf(act[3 * i + 2], -1.0f), 1.0f) * c.torque_max;
        /* apply_force_at_local_point(force, (0,0)): world force = R(angle) force, game/game.py:396 */
        float s_, c_;
        sincos_f(E.ang[i], &s_, &c_);
        Fx[i] = a0 * c_ - a1 * s_;
        Fy[i] = a0 * s_ + a1 * c_;
    }
    /* ---- game/game.py:379 _update_reward_state: distances at the start of the step */
    const float d0x = E.px[0] - E.px[4], d0y = E.py[0] - E.py[4];
    const float d1x = E.px[1] - E.px[4], d1y = E.py[1] - E.py[4];
    const float dgx = E.px[4] - FIELD_R, dgy = E.py[4] - 300.0f;
    /* red's: agents 2, 3 to the ball, the ball to red's target (FIELD_L, 300) (its y offset is dgy) */
    const float d2x = TEAMS ? E.px[2] - E.px[4] : 0.0f, d2y = TEAMS ? E.py[2] - E.py[4] : 0.0f;
    const float d3x = TEAMS ? E.px[3] - E.px[4] : 0.0f, d3y = TEAMS ? E.py[3] - E.py[4] : 0.0f;
    const float dhx = TEAMS ? E.px[4] - FIELD_L : 0.0f;
    E.steps += 1;

    /* ---- cpBodyUpdatePosition: p += (v + v_bias) dt, a += (w + w_bias) dt, bias cleared */
    float incx[5], incy[5];
#pragma unroll
    for (int i = 0; i < 5; i++) {
        incx[i] = (E.vx[i] + E.vbx[i]) * DT; incy[i] = (E.vy[i] + E.vby[i]) * DT;
        E.px[i] += incx[i]; E.py[i] += incy[i];
        E.vbx[i] = 0.0f; E.vby[i] = 0.0f;
    }
#pragma unroll
    for (int i = 0; i < 4; i++) {
        E.ang[i] = wrap_angle(E.ang[i] + (E.w[i] + E.wb[i]) * DT);
        E.wb[i] = 0.0f;
        sincos_f(E.ang[i], &sn[i], &cs[i]);
    }

    /* ---- broad phase (conservative bounding-box reject, cpSpaceCollideShapes QueryReject) */
    uint32_t m_as = 0, m_aa = 0, m_ba = 0, m_bw = 0;
    float R[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        R[i] = AGENT_HALF * (fabsf(cs[i]) + fabsf(sn[i]));
        const float x = E.px[i], y = E.py[i], r = R[i];
        if (x - r <= 12.0f || x + r >= 788.0f || y - r <= 12.0f || y + r >= 588.0f) {
            uint32_t mm = 0;
            mm |= bb_overlap(x, y, r, 8.0f, 8.0f, 792.0f, 12.0f) ? 1u : 0u;
            mm |= bb_overlap(x, y, r, 8.0f, 588.0f, 792.0f, 592.0f) ? 2u : 0u;
            mm |= bb_overlap(x, y, r, 8.0f, 8.0f, 12.0f, 227.0f) ? 4u : 0u;
            mm |= bb_overlap(x, y, r, 8.0f, 373.0f, 12.0f, 592.0f) ? 8u : 0u;
            mm |= bb_overlap(x, y, r, 788.0f, 8.0f, 792.0f, 227.0f) ? 16u : 0u;
            mm |= bb_overlap(x, y, r, 788.0f, 373.0f, 792.0f, 592.0f) ? 32u : 0u;
            mm |= bb_overlap(x, y, r, 9.0f, 224.0f, 11.0f, 376.0f) ? 64u : 0u;
            mm |= bb_overlap(x, y, r, 789.0f, 224.0f, 791.0f, 376.0f) ? 128u : 0u;
            m_as |= mm << (8 * i);
        }
    }
    {
        int p = 0;
#pragma unroll
        for (int i = 0; i < 4; i++) {
#pragma unroll
            for (int j = i + 1; j < 4; j++) {
                const float rr = R[i] + R[j];
                const float dx = E.px[i] - E.px[j], dy = E.py[i] - E.py[j];
                /* bounding boxes overlap AND the circumscribed circles (radius 15 sqrt 2) do: both are necessary for
                   the boxes to touch; the second test spares the general path most near misses */
                if (fabsf(dx) <= rr && fabsf(dy) <= rr && dx * dx + dy * dy <= AA_REACH2) m_aa |= 1u << p;
                p++;
            }
        }
    }
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const float rr = R[i] + BALL_R;
        const float dx = E.px[i] - E.px[4], dy = E.py[i] - E.py[4];
        if (fabsf(dx) <= rr && fabsf(dy) <= rr && dx * dx + dy * dy <= BA_REACH2) m_ba |= 1u << i;
    }
    {
        const float x = E.px[4], y = E.py[4], r = BALL_R;
        if (x - r <= 12.0f || x + r >= 788.0f || y - r <= 12.0f || y + r >= 588.0f) {
            m_bw |= bb_overlap(x, y, r, 8.0f, 8.0f, 792.0f, 12.0f) ? 1u : 0u;
            m_bw |= bb_overlap(x, y, r, 8.0f, 588.0f, 792.0f, 592.0f) ? 2u : 0u;
            m_bw |= bb_overlap(x, y, r, 8.0f, 8.0f, 12.0f, 227.0f) ? 4u : 0u;
            m_bw |= bb_overlap(x, y, r, 8.0f, 373.0f, 12.0f, 592.0f) ? 8u : 0u;
            m_bw |= bb_overlap(x, y, r, 788.0f, 8.0f, 792.0f, 227.0f) ? 16u : 0u;
            m_bw |= bb_overlap(x, y, r, 788.0f, 373.0f, 792.0f, 592.0f) ? 32u : 0u;
        }
    }

    const int old_count = (int)(E.flags & FLAG_CACHE_MASK);
    int n_contacts = 0, overflow = 0;
    int new_count = 0;
    const bool any_candidate = (m_as | m_aa | m_ba | m_bw) != 0u;
#ifndef MSOC_FAST_AGING
#define MSOC_FAST_AGING 1
#endif
#if MSOC_FAST_AGING
    const bool contact_path = any_candidate; /* narrow phase + solver needed */
#else
    const bool contact_path = any_candidate || old_count != 0;
#endif
    load = LOAD_LIGHT;
    const bool run_contacts = FULL && contact_path;
    const bool run_light = LIGHT && contact_path;
    const bool run_pair = PAIR && contact_path, run_multi = MULTI && contact_path;
    if (FAST) {
        if (contact_path) {
            /* work class for the contact lists */
            const uint32_t dyn = m_aa | (m_ba << 6);
            const int n_as = popc32(m_as), n_dyn = popc32(dyn), n_bw = popc32(m_bw);
            if ((E.flags & FLAG_INJECT) || (step_flags & 2u)) load = LOAD_HEAVY; /* 2u: MSOC_STEP_GENERAL_PATH */
            else if (n_dyn == 0) {
                if (n_as == 1 && n_bw == 0) load = LOAD_LIGHT;
                else {
                    bool ok = n_bw <= 2;
#pragma unroll
                    for (int i = 0; i < 4; i++) ok = ok && popc32((m_as >> (8 * i)) & 255u) <= 2;
                    load = ok ? LOAD_MULTI : LOAD_HEAVY;
                }
            } else load = (n_dyn == 1 && n_as <= 1 && n_bw == 0) ? LOAD_PAIR : LOAD_HEAVY;
            return false;
        }
        /* an injected state (Arrays::inject): the general kernel steps it (rare: only the step after msoc_set_state) */
        if (E.flags & FLAG_INJECT) { load = LOAD_HEAVY; return false; }
    }
    const bool age_only = !contact_path && old_count != 0;
#if defined(__CUDA_ARCH__)
    /* the env still carries arbiters of contacts that ended less than collision_persistence (3) steps ago; they are aged
       at the end of the step -- start pulling their cache line now, the shaping and velocity code in between covers the
       latency */
    if (age_only) asm volatile("prefetch.global.L1 [%0];" ::"l"(A.cache[cur] + cache_slot(e, 0)));
#endif

    /* ---- shaping rewards (game/game.py:324-349) from the step displacement; only positions enter, so
       they are final here and their inputs need not stay live across the contact path */
    float r = 0.0f, r_red = 0.0f;
    {
        const float ibx = incx[4], iby = incy[4];
        if (c.prox_mult != 0.0f) {
            float imp = 0.0f;
            {
                const float lx = incx[0] - ibx, ly = incy[0] - iby;
                const float dp = sqrtf(d0x * d0x + d0y * d0y);
                const float nx_ = d0x + lx, ny_ = d0y + ly;
                const float dc = sqrtf(nx_ * nx_ + ny_ * ny_);
                const float den = dp + dc;
                if (den > 0.0f) imp += -(2.0f * (d0x * lx + d0y * ly) + (lx * lx + ly * ly)) / den;
            }
            {
                const float lx = incx[1] - ibx, ly = incy[1] - iby;
                const float dp = sqrtf(d1x * d1x + d1y * d1y);
                const float nx_ = d1x + lx, ny_ = d1y + ly;
                const float dc = sqrtf(nx_ * nx_ + ny_ * ny_);
                const float den = dp + dc;
                if (den > 0.0f) imp += -(2.0f * (d1x * lx + d1y * ly) + (lx * lx + ly * ly)) / den;
            }
            r += c.prox_mult * imp;
        }
        {
            const float dp = sqrtf(dgx * dgx + dgy * dgy);
            const float nx_ = dgx + ibx, ny_ = dgy + iby;
            const float dc = sqrtf(nx_ * nx_ + ny_ * ny_);
            const float den = dp + dc;
            float imp = 0.0f;
            if (den > 0.0f) imp = -(2.0f * (dgx * ibx + dgy * iby) + (ibx * ibx + iby * iby)) / den;
            r += imp * c.move_mult;
        }
        if (TEAMS) { /* the same terms for red, in the same order */
            if (c.prox_mult != 0.0f)
                r_red += c.prox_mult * (distance_drop(d2x, d2y, incx[2] - ibx, incy[2] - iby) + distance_drop(d3x, d3y, incx[3] - ibx, incy[3] - iby));
            r_red += distance_drop(dhx, dgy, ibx, iby) * c.move_mult;
        }
    }

    const bool run_islands = run_pair || run_multi;
    if (run_contacts || run_islands) {
        /* park what the contact path needs with a dynamic body index (and what it does not need at
           all until it is over) in the lane's scratch: pre-update velocities for the arbiter
           pre-step, poses for the narrow phase */
#pragma unroll
        for (int i = 0; i < 5; i++) {
            /* (island modes keep the pre-update velocities in the bias fields until the body's island is solved) */
            float *pb = W.body + i * SCR;
            pb[(run_islands ? BF_BX : BF_VX) * BODY_FS] = E.vx[i]; pb[(run_islands ? BF_BY : BF_VY) * BODY_FS] = E.vy[i];
            pb[(run_islands ? BF_BW : BF_W) * BODY_FS] = E.w[i];
            W.geom[(GF_PX + i) * SCR] = E.px[i]; W.geom[(GF_PY + i) * SCR] = E.py[i];
        }
#pragma unroll
        for (int i = 0; i < 4; i++) {
            W.geom[(GF_CS + i) * SCR] = cs[i]; W.geom[(GF_SN + i) * SCR] = sn[i]; W.geom[(GF_ANG + i) * SCR] = E.ang[i];
        }
    }

    /* light mode: the one agent that may touch a wall; its pre-update velocity feeds the arbiter pre-step */
    const int l_idx = run_light ? ctz32(m_as) : 0, l_i = l_idx >> 3;
    float l_ovx = 0.0f, l_ovy = 0.0f, l_ow = 0.0f;
    if (run_light) { l_ovx = sel4(E.vx, l_i); l_ovy = sel4(E.vy, l_i); l_ow = sel4(E.w, l_i); }

    /* ---- cpBodyUpdateVelocity (gravity 0, damping 1) + the reference's custom velocity functions
       (game/entities.py:19-28 agent, :69-77 ball): friction multiplier, max_velocity clamp.
       (Chipmunk runs the arbiter pre-step before this; it only reads the parked old velocities.) */
#pragma unroll
    for (int i = 0; i < 5; i++) {
        const bool ag = i < 4;
        float vx = E.vx[i], vy = E.vy[i];
        if (ag) { vx = vx + (Fx[i] * c.agent_minv) * DT; vy = vy + (Fy[i] * c.agent_minv) * DT; }
        const float fr = ag ? c.agent_friction : c.ball_friction;
        vx *= fr; vy *= fr;
        if (ag) E.w[i] = (E.w[i] + (Tq[i] * c.agent_iinv) * DT) * fr;
        const float l2 = vx * vx + vy * vy;
        if (l2 > c.max_velocity * c.max_velocity) { const float s_ = c.max_velocity * rsqrt_f(l2); vx *= s_; vy *= s_; }
        E.vx[i] = vx; E.vy[i] = vy;
    }
    if (run_islands) {
        /* the islands fetch and return their bodies by (dynamic) index */
#pragma unroll
        for (int i = 0; i < 5; i++) {
            float *pb = W.body + i * SCR;
            pb[BF_VX * BODY_FS] = E.vx[i]; pb[BF_VY * BODY_FS] = E.vy[i]; pb[BF_W * BODY_FS] = E.w[i];
        }
    }

    if (run_light) {
        /* ---- light mode: exactly one candidate pair, agent l_i x static segment.  The same arithmetic as
           the general path below (narrow phase, arbiter cache, pre-step, warm start, 10 iterations, cache
           write-out) for a single dynamic body and at most two contacts, entirely in registers. */
        const uint32_t *oc = A.cache[cur] + cache_slot(e, 0);
        uint32_t *nc_ = A.cache[cur ^ 1] + cache_slot(e, 0);
        Manifold m;
        const Seg g = get_segment(l_idx & 7);
        collide_segment_box(g, mk(sel4(E.px, l_i), sel4(E.py, l_i)), sel4(cs, l_i), sel4(sn, l_i), m);
        n_contacts = m.count;
        if (m.count > 0) {
            /* cpArbiterUpdate: accumulated impulses of equal-key contacts, first-contact state */
            bool first = true;
            float jn0 = 0.0f, jt0 = 0.0f, jn1 = 0.0f, jt1 = 0.0f;
            auto lookup = [&](uint32_t info, uint32_t wjn, uint32_t wjt) {
                if ((int)(info & 63u) != l_idx) return;
                if (((info >> 10) & 3u) == 0u) first = false;
                const int key = (int)((info >> 6) & 15u);
                if (key == m.key[0]) { jn0 = u2f(wjn); jt0 = u2f(wjt); }
                if (m.count > 1 && key == m.key[1]) { jn1 = u2f(wjn); jt1 = u2f(wjt); }
            };
#pragma unroll
            for (int j = 0; j < 4; j++)
                if (j < old_count) lookup(pc[3 * j], pc[3 * j + 1], pc[3 * j + 2]);
            for (int j = 4; j < old_count; j++) lookup(oc[3 * j], oc[3 * j + 1], oc[3 * j + 2]);
            const bool two = m.count > 1;
            const float nx = m.n.x, ny = m.n.y;
            const V2 tng = vperp(m.n);
            const float mb = c.agent_minv, ib = c.agent_iinv;
            const float u = ((l_idx & 7) < 6) ? U_AGENT_WALL : U_AGENT_GOALLINE;
            /* contact records: lever arm of the agent (static side: none), cpArbiterPreStep */
            const float rn0 = vcross(m.p2[0], m.n), rt0 = vcross(m.p2[0], tng);
            const float rn1 = two ? vcross(m.p2[1], m.n) : 0.0f, rt1 = two ? vcross(m.p2[1], tng) : 0.0f;
            const float nM0 = 1.0f / (mb + ib * rn0 * rn0), tM0 = 1.0f / (mb + ib * rt0 * rt0);
            const float nM1 = 1.0f / (mb + ib * rn1 * rn1), tM1 = 1.0f / (mb + ib * rt1 * rt1);
            const float bias0 = -BIAS_COEF_OVER_DT * fminf(0.0f, vdot(m.p2[0] - m.p1[0], m.n) + SLOP);
            const float bias1 = two ? -BIAS_COEF_OVER_DT * fminf(0.0f, vdot(m.p2[1] - m.p1[1], m.n) + SLOP) : 0.0f;
            const float bnc0 = (l_ovx * nx + l_ovy * ny + l_ow * rn0) * E_AGENT_SEG;
            const float bnc1 = (l_ovx * nx + l_ovy * ny + l_ow * rn1) * E_AGENT_SEG;
            float vx = sel4(E.vx, l_i), vy = sel4(E.vy, l_i), w = sel4(E.w, l_i), bx = 0.0f, by = 0.0f, bw = 0.0f;
            /* cpArbiterApplyCachedImpulse (skipped in an arbiter's first step) */
            if (!first) {
                { const float jx = nx * jn0 - ny * jt0, jy = ny * jn0 + nx * jt0;
                  vx += jx * mb; vy += jy * mb; w += ib * (rn0 * jn0 + rt0 * jt0); }
                if (two) { const float jx = nx * jn1 - ny * jt1, jy = ny * jn1 + nx * jt1;
                  vx += jx * mb; vy += jy * mb; w += ib * (rn1 * jn1 + rt1 * jt1); }
            }
            /* cpArbiterApplyImpulse x 10 */
            float jb0 = 0.0f, jb1 = 0.0f;
#if defined(__CUDACC__)
#pragma unroll 1
#endif
            for (int it = 0; it < SOLVER_ITERS; it++) {
                {
                    const float vrn = vx * nx + vy * ny + w * rn0;
                    const float vrt = vy * nx - vx * ny + w * rt0;
                    const float vbn = bx * nx + by * ny + bw * rn0;
                    const float jbN = fmaxf(jb0 + (bias0 - vbn) * nM0, 0.0f);
                    const float jnN = fmaxf(jn0 - (bnc0 + vrn) * nM0, 0.0f);
                    const float jtMax = u * jnN;
                    const float jtN = fminf(fmaxf(jt0 - vrt * tM0, -jtMax), jtMax);
                    const float djb = jbN - jb0, djn = jnN - jn0, djt = jtN - jt0;
                    jb0 = jbN; jn0 = jnN; jt0 = jtN;
                    const float jx = nx * djn - ny * djt, jy = ny * djn + nx * djt;
                    bx += nx * djb * mb; by += ny * djb * mb; bw += ib * rn0 * djb;
                    vx += jx * mb; vy += jy * mb; w += ib * (rn0 * djn + rt0 * djt);
                }
                if (two) {
                    const float vrn = vx * nx + vy * ny + w * rn1;
                    const float vrt = vy * nx - vx * ny + w * rt1;
                    const float vbn = bx * nx + by * ny + bw * rn1;
                    const float jbN = fmaxf(jb1 + (bias1 - vbn) * nM1, 0.0f);
                    const float jnN = fmaxf(jn1 - (bnc1 + vrn) * nM1, 0.0f);
                    const float jtMax = u * jnN;
                    const float jtN = fminf(fmaxf(jt1 - vrt * tM1, -jtMax), jtMax);
                    const float djb = jbN - jb1, djn = jnN - jn1, djt = jtN - jt1;
                    jb1 = jbN; jn1 = jnN; jt1 = jtN;
                    const float jx = nx * djn - ny * djt, jy = ny * djn + nx * djt;
                    bx += nx * djb * mb; by += ny * djb * mb; bw += ib * rn1 * djb;
                    vx += jx * mb; vy += jy * mb; w += ib * (rn1 * djn + rt1 * djt);
                }
            }
#pragma unroll
            for (int k = 0; k < 4; k++)
                if (k == l_i) { E.vx[k] = vx; E.vy[k] = vy; E.w[k] = w; E.vbx[k] = bx; E.vby[k] = by; E.wb[k] = bw; }
            /* this step's contacts open the arbiter cache of the next step (age 0) */
            nc_[0] = (uint32_t)l_idx | ((uint32_t)m.key[0] << 6); nc_[1] = f2u(jn0); nc_[2] = f2u(jt0);
            new_count = 1;
            if (two) {
                nc_[3] = (uint32_t)l_idx | ((uint32_t)m.key[1] << 6); nc_[4] = f2u(jn1); nc_[5] = f2u(jt1);
                new_count = 2;
            }
        }
        /* then the untouched arbiters younger than collision_persistence (3) */
        auto age_entry = [&](uint32_t info, uint32_t wjn, uint32_t wjt) {
            const uint32_t age = (info >> 10) & 3u;
            if ((m.count > 0 && (int)(info & 63u) == l_idx) || age >= 2u) return;
            if (new_count >= MAX_CACHE) { overflow++; return; }
            nc_[3 * new_count] = (info & 1023u) | ((age + 1u) << 10);
            nc_[3 * new_count + 1] = wjn; nc_[3 * new_count + 2] = wjt;
            new_count++;
        };
#pragma unroll
        for (int j = 0; j < 4; j++)
            if (j < old_count) age_entry(pc[3 * j], pc[3 * j + 1], pc[3 * j + 2]);
        for (int j = 4; j < old_count; j++) age_entry(oc[3 * j], oc[3 * j + 1], oc[3 * j + 2]);
    }

    else if (run_islands) {
        /* ---- islands of one or two dynamic bodies: the bodies in registers, their contacts in the lane's slots.  Cached
           arbiter entries: the first four are in pc[], the rest in global memory. */
        const uint32_t *oc = A.cache[cur] + cache_slot(e, 0);
        uint32_t *nc_ = A.cache[cur ^ 1] + cache_slot(e, 0);
        uint64_t touched = 0ull;
        uint32_t solved = 0u; /* bodies whose bias fields hold bias velocities (not the parked pre-update velocities any more) */
        const float *G = W.geom;
        /* cpArbiterUpdate for the arbiter `pair` with the manifold keys k0, k1 (k1 < 0: one contact): accumulated
           impulses of equal-key contacts, first-contact state */
        bool first; float cjn0, cjt0, cjn1, cjt1;
        auto cache_lookup = [&](int pair, int k0, int k1) {
            first = true; cjn0 = cjt0 = cjn1 = cjt1 = 0.0f;
            auto one = [&](uint32_t info, uint32_t wjn, uint32_t wjt) {
                if ((int)(info & 63u) != pair) return;
                if (((info >> 10) & 3u) == 0u) first = false;
                const int key = (int)((info >> 6) & 15u);
                if (key == k0) { cjn0 = u2f(wjn); cjt0 = u2f(wjt); }
                if (k1 >= 0 && key == k1) { cjn1 = u2f(wjn); cjt1 = u2f(wjt); }
            };
#pragma unroll
            for (int j = 0; j < 4; j++)
                if (j < old_count) one(pc[3 * j], pc[3 * j + 1], pc[3 * j + 2]);
            for (int j = 4; j < old_count; j++) one(oc[3 * j], oc[3 * j + 1], oc[3 * j + 2]);
        };

        /* ---- pair class: exactly one candidate pair that joins two dynamic bodies -- agent i x agent j (a = i, b = j) or
           ball x agent (a = ball, b = agent), at most two contacts -- and at most one agent x segment candidate beside it.
           The wall arbiter comes first in arbiter order.  If its agent is one of the pair's bodies and both manifolds have
           contacts, the four contacts are ONE island of two bodies (slots 0-1 wall, 2-3 pair); otherwise the wall agent is a
           single-body island of its own and goes through the multi class's loop below. */
        bool aa = false, wall_merged = false;
        int ia_ = 0, ib_ = 1, pair = 0, wl_idx = 0;
        Manifold m;
        m.count = 0;
        V2 r1_off = mk(0.0f, 0.0f), r2_off = mk(0.0f, 0.0f);
        uint32_t loop_as = run_multi ? m_as : 0u, loop_bw = run_multi ? m_bw : 0u; /* candidates of the single-body loop */
        if (run_pair) {
            aa = m_aa != 0u;
            const int idx = aa ? ctz32(m_aa) : ctz32(m_ba);
            ia_ = aa ? ((idx < 3) ? 0 : (idx < 5) ? 1 : 2) : BALL;
            ib_ = aa ? ((idx < 3) ? idx + 1 : (idx < 5) ? idx - 1 : 3) : idx;
            pair = (aa ? PAIR_AGENT_AGENT : PAIR_BALL_AGENT) + idx;
            const V2 off = mk(G[(GF_PX + ib_) * SCR] - G[(GF_PX + ia_) * SCR], G[(GF_PY + ib_) * SCR] - G[(GF_PY + ia_) * SCR]); /* centre b - centre a */
            if (aa) { collide_box_box(G[(GF_CS + (ia_ & 3)) * SCR], G[(GF_SN + (ia_ & 3)) * SCR], G[(GF_CS + ib_) * SCR], G[(GF_SN + ib_) * SCR], off, m); r2_off = off; }
            else { const V2 cb = vneg(off); collide_ball_box(cb, G[(GF_CS + ib_) * SCR], G[(GF_SN + ib_) * SCR], m); r1_off = cb; }
            if (m_as != 0u) {
                wl_idx = ctz32(m_as);
                const int wa = wl_idx >> 3;
                wall_merged = m.count > 0 && (wa == ia_ || wa == ib_);
                if (!wall_merged) loop_as = m_as;
            }
        }

        if ((loop_as | loop_bw) != 0u) {
            /* ---- single-body islands -- one dynamic body against the static one, at most two arbiters (four contacts) --
               solved one after the other, bodies and arbiters in ascending order (the canonical arbiter order restricted
               to them): all of a multi env, the separate wall agent of a pair env */
            uint32_t bodies = ((loop_as & 0xffu) ? 1u : 0u) | ((loop_as & 0xff00u) ? 2u : 0u) | ((loop_as & 0xff0000u) ? 4u : 0u) |
                              ((loop_as & 0xff000000u) ? 8u : 0u) | (loop_bw ? 16u : 0u);
#if defined(__CUDACC__)
#pragma unroll 1
#endif
            while (bodies) {
                const int b = ctz32(bodies);
                bodies &= bodies - 1u;
                const bool ag = b < 4;
                uint32_t segs = ag ? ((loop_as >> (8 * b)) & 255u) : loop_bw;
                float *pb = W.body + b * SCR;
                const V2 pos = mk(G[(GF_PX + b) * SCR], G[(GF_PY + b) * SCR]);
                const float bcs = G[(GF_CS + (b & 3)) * SCR], bsn = G[(GF_SN + (b & 3)) * SCR];
                const float obx = pb[BF_BX * BODY_FS], oby = pb[BF_BY * BODY_FS], obw = pb[BF_BW * BODY_FS]; /* pre-update velocity */
                const float mb = ag ? c.agent_minv : c.ball_minv, ibm = ag ? c.agent_iinv : c.ball_iinv;
                const float e_ = ag ? E_AGENT_SEG : E_BALL_WALL;
                uint32_t firsts = 0u;
                int cnt = 0;
#if defined(__CUDACC__)
#pragma unroll 1
#endif
                while (segs) {
                    const int sg = ctz32(segs);
                    segs &= segs - 1u;
                    const Seg g = get_segment(sg);
                    Manifold mw;
                    if (ag) collide_segment_box(g, pos, bcs, bsn, mw);
                    else collide_ball_segment(g, pos, mw);
                    if (mw.count == 0) continue;
                    const int wpair = ag ? 8 * b + sg : PAIR_BALL_WALL + sg;
                    const bool two = mw.count > 1;
                    touched |= 1ull << wpair;
                    cache_lookup(wpair, mw.key[0], two ? mw.key[1] : -1);
                    /* stored with the dynamic body second (add_contacts): a ball x wall manifold (ball first) is flipped */
                    const V2 n_ = ag ? mw.n : vneg(mw.n), tng = vperp(n_);
                    const float u_ = ag ? ((sg < 6) ? U_AGENT_WALL : U_AGENT_GOALLINE) : U_BALL_WALL;
#pragma unroll
                    for (int i = 0; i < 2; i++) {
                        if ((i == 0 || two) && cnt < ISL_SLOTS) {
                            float *q = W.isl + cnt * ISL_FIELDS * SCR;
                            const V2 r2 = ag ? mw.p2[i] : mw.p1[i];
                            const float rn = vcross(r2, n_), rt = vcross(r2, tng);
                            q[IF_NX * SCR] = n_.x; q[IF_NY * SCR] = n_.y; q[IF_RN2 * SCR] = rn; q[IF_RT2 * SCR] = rt;
                            q[IF_NM * SCR] = 1.0f / (mb + ibm * rn * rn); q[IF_TM * SCR] = 1.0f / (mb + ibm * rt * rt);
                            q[IF_BIAS * SCR] = -BIAS_COEF_OVER_DT * fminf(0.0f, vdot(mw.p2[i] - mw.p1[i], mw.n) + SLOP);
                            q[IF_BNC * SCR] = (obx * n_.x + oby * n_.y + obw * rn) * e_;
                            q[IF_JN * SCR] = (i == 0) ? cjn0 : cjn1; q[IF_JT * SCR] = (i == 0) ? cjt0 : cjt1; q[IF_JB * SCR] = 0.0f;
                            q[IF_U * SCR] = u_;
                            q[IF_INFO * SCR] = u2f((uint32_t)wpair | ((uint32_t)mw.key[i] << 6));
                            if (first) firsts |= 1u << cnt;
                            cnt++;
                        }
                    }
                }
                solved |= 1u << b;
                float vx = pb[BF_VX * BODY_FS], vy = pb[BF_VY * BODY_FS], w = pb[BF_W * BODY_FS], bx = 0.0f, by = 0.0f, bw = 0.0f;
                /* cpArbiterApplyCachedImpulse (skipped for arbiters in their first step) */
                for (int k = 0; k < cnt; k++) {
                    if (!((firsts >> k) & 1u)) {
                        const float *q = W.isl + k * ISL_FIELDS * SCR;
                        const float nx = q[IF_NX * SCR], ny = q[IF_NY * SCR], jn = q[IF_JN * SCR], jt = q[IF_JT * SCR];
                        const float jx = nx * jn - ny * jt, jy = ny * jn + nx * jt;
                        vx += jx * mb; vy += jy * mb; w += ibm * (q[IF_RN2 * SCR] * jn + q[IF_RT2 * SCR] * jt);
                    }
                }
                /* cpArbiterApplyImpulse x 10 */
#if defined(__CUDACC__)
#pragma unroll 1
#endif
                for (int it = 0; it < SOLVER_ITERS; it++) {
#if defined(__CUDACC__)
#pragma unroll 1
#endif
                    for (int k = 0; k < cnt; k++) {
                        float *q = W.isl + k * ISL_FIELDS * SCR;
                        const float nx = q[IF_NX * SCR], ny = q[IF_NY * SCR], rn = q[IF_RN2 * SCR], rt = q[IF_RT2 * SCR];
                        const float nM = q[IF_NM * SCR], jbO = q[IF_JB * SCR], jnO = q[IF_JN * SCR], jtO = q[IF_JT * SCR];
                        const float vrn = vx * nx + vy * ny + w * rn;
                        const float vrt = vy * nx - vx * ny + w * rt;
                        const float vbn = bx * nx + by * ny + bw * rn;
                        const float jbN = fmaxf(jbO + (q[IF_BIAS * SCR] - vbn) * nM, 0.0f);
                        const float jnN = fmaxf(jnO - (q[IF_BNC * SCR] + vrn) * nM, 0.0f);
                        const float jtMax = q[IF_U * SCR] * jnN;
                        const float jtN = fminf(fmaxf(jtO - vrt * q[IF_TM * SCR], -jtMax), jtMax);
                        const float djb = jbN - jbO, djn = jnN - jnO, djt = jtN - jtO;
                        q[IF_JB * SCR] = jbN; q[IF_JN * SCR] = jnN; q[IF_JT * SCR] = jtN;
                        const float jx = nx * djn - ny * djt, jy = ny * djn + nx * djt;
                        bx += nx * djb * mb; by += ny * djb * mb; bw += ibm * rn * djb;
                        vx += jx * mb; vy += jy * mb; w += ibm * (rn * djn + rt * djt);
                    }
                }
                pb[BF_VX * BODY_FS] = vx; pb[BF_VY * BODY_FS] = vy; pb[BF_W * BODY_FS] = w;
                pb[BF_BX * BODY_FS] = bx; pb[BF_BY * BODY_FS] = by; pb[BF_BW * BODY_FS] = bw;
                /* this step's contacts open the arbiter cache of the next step (age 0) */
                for (int k = 0; k < cnt; k++) {
                    const float *q = W.isl + k * ISL_FIELDS * SCR;
                    nc_[3 * new_count] = f2u(q[IF_INFO * SCR]); nc_[3 * new_count + 1] = f2u(q[IF_JN * SCR]); nc_[3 * new_count + 2] = f2u(q[IF_JT * SCR]);
                    new_count++;
                }
                n_contacts += cnt;
            }
        }

        if (run_pair && m.count > 0) {
            /* ---- the pair's island: two bodies in registers; slots 2-3 its own (<= 2) contacts, slots 0-1 the (<= 2)
               contacts of the wall arbiter of one of its agents when there is one (wall_merged) */
            const bool two = m.count > 1;
            float *pa = W.body + ia_ * SCR, *pb = W.body + ib_ * SCR;
            const float ma = aa ? c.agent_minv : c.ball_minv, iam = aa ? c.agent_iinv : c.ball_iinv;
            const float mb = c.agent_minv, ibm = c.agent_iinv;
            /* pre-update velocities: parked in the bias fields */
            const float oax = pa[BF_BX * BODY_FS], oay = pa[BF_BY * BODY_FS], oaw = pa[BF_BW * BODY_FS];
            const float obx = pb[BF_BX * BODY_FS], oby = pb[BF_BY * BODY_FS], obw = pb[BF_BW * BODY_FS];
            /* the wall arbiter first (arbiter order) */
            int wcnt = 0;
            bool wfirst = true, wall_on_a = false;
            if (wall_merged) {
                const int wa = wl_idx >> 3, sg = wl_idx & 7;
                wall_on_a = wa == ia_;
                const Seg g = get_segment(sg);
                Manifold mw;
                collide_segment_box(g, mk(G[(GF_PX + wa) * SCR], G[(GF_PY + wa) * SCR]), G[(GF_CS + wa) * SCR], G[(GF_SN + wa) * SCR], mw);
                if (mw.count > 0) {
                    const bool wtwo = mw.count > 1;
                    touched |= 1ull << wl_idx;
                    cache_lookup(wl_idx, mw.key[0], wtwo ? mw.key[1] : -1);
                    wfirst = first;
                    const V2 tng = vperp(mw.n);
                    const float ovx_ = wall_on_a ? oax : obx, ovy_ = wall_on_a ? oay : oby, ow_ = wall_on_a ? oaw : obw;
                    const float u_ = (sg < 6) ? U_AGENT_WALL : U_AGENT_GOALLINE;
#pragma unroll
                    for (int i = 0; i < 2; i++) {
                        if (i == 0 || wtwo) {
                            float *q = W.isl + i * ISL_FIELDS * SCR;
                            const float rn = vcross(mw.p2[i], mw.n), rt = vcross(mw.p2[i], tng);
                            q[IF_NX * SCR] = mw.n.x; q[IF_NY * SCR] = mw.n.y; q[IF_RN2 * SCR] = rn; q[IF_RT2 * SCR] = rt;
                            q[IF_NM * SCR] = 1.0f / (c.agent_minv + c.agent_iinv * rn * rn); q[IF_TM * SCR] = 1.0f / (c.agent_minv + c.agent_iinv * rt * rt);
                            q[IF_BIAS * SCR] = -BIAS_COEF_OVER_DT * fminf(0.0f, vdot(mw.p2[i] - mw.p1[i], mw.n) + SLOP);
                            q[IF_BNC * SCR] = (ovx_ * mw.n.x + ovy_ * mw.n.y + ow_ * rn) * E_AGENT_SEG;
                            q[IF_JN * SCR] = (i == 0) ? cjn0 : cjn1; q[IF_JT * SCR] = (i == 0) ? cjt0 : cjt1; q[IF_JB * SCR] = 0.0f;
                            q[IF_U * SCR] = u_;
                            q[IF_INFO * SCR] = u2f((uint32_t)wl_idx | ((uint32_t)mw.key[i] << 6));
                        }
                    }
                    wcnt = mw.count;
                }
            }
            touched |= 1ull << pair;
            solved |= (1u << ia_) | (1u << ib_);
            cache_lookup(pair, m.key[0], two ? m.key[1] : -1);
            const float e_ = aa ? E_AGENT_AGENT : E_BALL_AGENT, u = aa ? U_AGENT_AGENT : U_BALL_AGENT;
            const float nx = m.n.x, ny = m.n.y;
            const V2 tng = vperp(m.n);
#pragma unroll
            for (int i = 0; i < 2; i++) {
                if (i == 0 || two) {
                    float *q = W.isl + (2 + i) * ISL_FIELDS * SCR;
                    const V2 r1 = m.p1[i] - r1_off, r2 = m.p2[i] - r2_off;
                    const float rn1 = vcross(r1, m.n), rt1 = vcross(r1, tng), rn2 = vcross(r2, m.n), rt2 = vcross(r2, tng);
                    q[IF_RN1 * SCR] = rn1; q[IF_RT1 * SCR] = rt1; q[IF_RN2 * SCR] = rn2; q[IF_RT2 * SCR] = rt2;
                    q[IF_NM * SCR] = 1.0f / (ma + iam * rn1 * rn1 + mb + ibm * rn2 * rn2);
                    q[IF_TM * SCR] = 1.0f / (ma + iam * rt1 * rt1 + mb + ibm * rt2 * rt2);
                    q[IF_BIAS * SCR] = -BIAS_COEF_OVER_DT * fminf(0.0f, vdot(m.p2[i] - m.p1[i], m.n) + SLOP);
                    float vn = 0.0f;
                    vn -= oax * nx + oay * ny + oaw * rn1;
                    vn += obx * nx + oby * ny + obw * rn2;
                    q[IF_BNC * SCR] = vn * e_;
                    q[IF_JN * SCR] = (i == 0) ? cjn0 : cjn1; q[IF_JT * SCR] = (i == 0) ? cjt0 : cjt1; q[IF_JB * SCR] = 0.0f;
                }
            }
            float avx = pa[BF_VX * BODY_FS], avy = pa[BF_VY * BODY_FS], aw = pa[BF_W * BODY_FS], abx = 0.0f, aby = 0.0f, abw = 0.0f;
            float bvx = pb[BF_VX * BODY_FS], bvy = pb[BF_VY * BODY_FS], bw_ = pb[BF_W * BODY_FS], bbx = 0.0f, bby = 0.0f, bbw = 0.0f;
            /* one contact of the wall arbiter against the agent it belongs to (warm = cpArbiterApplyCachedImpulse, else
               cpArbiterApplyImpulse), the same arithmetic as in the single-body loop above */
            auto wall_contact = [&](int k, bool warm, float &vx, float &vy, float &w, float &bx, float &by, float &bw) {
                float *q = W.isl + k * ISL_FIELDS * SCR;
                const float wnx = q[IF_NX * SCR], wny = q[IF_NY * SCR], rn = q[IF_RN2 * SCR], rt = q[IF_RT2 * SCR];
                const float jbO = q[IF_JB * SCR], jnO = q[IF_JN * SCR], jtO = q[IF_JT * SCR];
                if (warm) {
                    const float jx = wnx * jnO - wny * jtO, jy = wny * jnO + wnx * jtO;
                    vx += jx * c.agent_minv; vy += jy * c.agent_minv; w += c.agent_iinv * (rn * jnO + rt * jtO);
                    return;
                }
                const float nM = q[IF_NM * SCR];
                const float vrn = vx * wnx + vy * wny + w * rn;
                const float vrt = vy * wnx - vx * wny + w * rt;
                const float vbn = bx * wnx + by * wny + bw * rn;
                const float jbN = fmaxf(jbO + (q[IF_BIAS * SCR] - vbn) * nM, 0.0f);
                const float jnN = fmaxf(jnO - (q[IF_BNC * SCR] + vrn) * nM, 0.0f);
                const float jtMax = q[IF_U * SCR] * jnN;
                const float jtN = fminf(fmaxf(jtO - vrt * q[IF_TM * SCR], -jtMax), jtMax);
                const float djb = jbN - jbO, djn = jnN - jnO, djt = jtN - jtO;
                q[IF_JB * SCR] = jbN; q[IF_JN * SCR] = jnN; q[IF_JT * SCR] = jtN;
                const float jx = wnx * djn - wny * djt, jy = wny * djn + wnx * djt;
                bx += wnx * djb * c.agent_minv; by += wny * djb * c.agent_minv; bw += c.agent_iinv * rn * djb;
                vx += jx * c.agent_minv; vy += jy * c.agent_minv; w += c.agent_iinv * (rn * djn + rt * djt);
            };
            /* cpArbiterApplyCachedImpulse (skipped in an arbiter's first step), wall arbiter first */
            if (!wfirst) {
                for (int k = 0; k < wcnt; k++) {
                    if (wall_on_a) wall_contact(k, true, avx, avy, aw, abx, aby, abw);
                    else wall_contact(k, true, bvx, bvy, bw_, bbx, bby, bbw);
                }
            }
            if (!first) {
#pragma unroll
                for (int i = 0; i < 2; i++) {
                    if (i == 0 || two) {
                        const float *q = W.isl + (2 + i) * ISL_FIELDS * SCR;
                        const float jn = q[IF_JN * SCR], jt = q[IF_JT * SCR];
                        const float jx = nx * jn - ny * jt, jy = ny * jn + nx * jt;
                        avx -= jx * ma; avy -= jy * ma; aw -= iam * (q[IF_RN1 * SCR] * jn + q[IF_RT1 * SCR] * jt);
                        bvx += jx * mb; bvy += jy * mb; bw_ += ibm * (q[IF_RN2 * SCR] * jn + q[IF_RT2 * SCR] * jt);
                    }
                }
            }
            /* cpArbiterApplyImpulse x 10 */
#if defined(__CUDACC__)
#pragma unroll 1
#endif
            for (int it = 0; it < SOLVER_ITERS; it++) {
                for (int k = 0; k < wcnt; k++) {
                    if (wall_on_a) wall_contact(k, false, avx, avy, aw, abx, aby, abw);
                    else wall_contact(k, false, bvx, bvy, bw_, bbx, bby, bbw);
                }
#pragma unroll
                for (int i = 0; i < 2; i++) {
                    if (i == 0 || two) {
                        float *q = W.isl + (2 + i) * ISL_FIELDS * SCR;
                        const float rn1 = q[IF_RN1 * SCR], rt1 = q[IF_RT1 * SCR], rn2 = q[IF_RN2 * SCR], rt2 = q[IF_RT2 * SCR];
                        const float nM = q[IF_NM * SCR], jbO = q[IF_JB * SCR], jnO = q[IF_JN * SCR], jtO = q[IF_JT * SCR];
                        float vrn = bvx * nx + bvy * ny + bw_ * rn2;
                        float vrt = bvy * nx - bvx * ny + bw_ * rt2;
                        float vbn = bbx * nx + bby * ny + bbw * rn2;
                        vrn -= avx * nx + avy * ny + aw * rn1;
                        vrt -= avy * nx - avx * ny + aw * rt1;
                        vbn -= abx * nx + aby * ny + abw * rn1;
                        const float jbN = fmaxf(jbO + (q[IF_BIAS * SCR] - vbn) * nM, 0.0f);
                        const float jnN = fmaxf(jnO - (q[IF_BNC * SCR] + vrn) * nM, 0.0f);
                        const float jtMax = u * jnN;
                        const float jtN = fminf(fmaxf(jtO - vrt * q[IF_TM * SCR], -jtMax), jtMax);
                        const float djb = jbN - jbO, djn = jnN - jnO, djt = jtN - jtO;
                        q[IF_JB * SCR] = jbN; q[IF_JN * SCR] = jnN; q[IF_JT * SCR] = jtN;
                        const float jx = nx * djn - ny * djt, jy = ny * djn + nx * djt;
                        bbx += nx * djb * mb; bby += ny * djb * mb; bbw += ibm * rn2 * djb;
                        bvx += jx * mb; bvy += jy * mb; bw_ += ibm * (rn2 * djn + rt2 * djt);
                        abx -= nx * djb * ma; aby -= ny * djb * ma; abw -= iam * rn1 * djb;
                        avx -= jx * ma; avy -= jy * ma; aw -= iam * (rn1 * djn + rt1 * djt);
                    }
                }
            }
            pa[BF_VX * BODY_FS] = avx; pa[BF_VY * BODY_FS] = avy; pa[BF_W * BODY_FS] = aw;
            pa[BF_BX * BODY_FS] = abx; pa[BF_BY * BODY_FS] = aby; pa[BF_BW * BODY_FS] = abw;
            pb[BF_VX * BODY_FS] = bvx; pb[BF_VY * BODY_FS] = bvy; pb[BF_W * BODY_FS] = bw_;
            pb[BF_BX * BODY_FS] = bbx; pb[BF_BY * BODY_FS] = bby; pb[BF_BW * BODY_FS] = bbw;
            /* this step's contacts open the arbiter cache of the next step (age 0): wall arbiter, then the pair's */
            for (int k = 0; k < wcnt; k++) {
                const float *q = W.isl + k * ISL_FIELDS * SCR;
                nc_[3 * new_count] = f2u(q[IF_INFO * SCR]); nc_[3 * new_count + 1] = f2u(q[IF_JN * SCR]); nc_[3 * new_count + 2] = f2u(q[IF_JT * SCR]);
                new_count++;
            }
#pragma unroll
            for (int i = 0; i < 2; i++) {
                if (i == 0 || two) {
                    const float *q = W.isl + (2 + i) * ISL_FIELDS * SCR;
                    nc_[3 * new_count] = (uint32_t)pair | ((uint32_t)m.key[i] << 6); nc_[3 * new_count + 1] = f2u(q[IF_JN * SCR]); nc_[3 * new_count + 2] = f2u(q[IF_JT * SCR]);
                    new_count++;
                }
            }
            n_contacts += wcnt + m.count;
        }

        /* then the untouched arbiters younger than collision_persistence (3) */
        auto age_entry = [&](uint32_t info, uint32_t wjn, uint32_t wjt) {
            const uint32_t age = (info >> 10) & 3u;
            if (((touched >> (info & 63u)) & 1ull) || age >= 2u) return;
            if (new_count >= MAX_CACHE) { overflow++; return; }
            nc_[3 * new_count] = (info & 1023u) | ((age + 1u) << 10);
            nc_[3 * new_count + 1] = wjn; nc_[3 * new_count + 2] = wjt;
            new_count++;
        };
#pragma unroll
        for (int j = 0; j < 4; j++)
            if (j < old_count) age_entry(pc[3 * j], pc[3 * j + 1], pc[3 * j + 2]);
        for (int j = 4; j < old_count; j++) age_entry(oc[3 * j], oc[3 * j + 1], oc[3 * j + 2]);
        /* the env back from the scratch (bias fields of unsolved bodies still hold the parked pre-update velocities) */
#pragma unroll
        for (int i = 0; i < 5; i++) {
            const float *pb = W.body + i * SCR;
            const bool sv = (solved >> i) & 1u;
            E.vx[i] = pb[BF_VX * BODY_FS]; E.vy[i] = pb[BF_VY * BODY_FS]; E.w[i] = pb[BF_W * BODY_FS];
            E.vbx[i] = sv ? pb[BF_BX * BODY_FS] : 0.0f; E.vby[i] = sv ? pb[BF_BY * BODY_FS] : 0.0f;
            if (i < 4) E.wb[i] = sv ? pb[BF_BW * BODY_FS] : 0.0f;
            E.px[i] = W.geom[(GF_PX + i) * SCR]; E.py[i] = W.geom[(GF_PY + i) * SCR];
        }
#pragma unroll
        for (int i = 0; i < 4; i++) E.ang[i] = W.geom[(GF_ANG + i) * SCR];
    }

    if (run_contacts) {
        CacheIO cio;
        W.nc = 0; W.overflow = 0; W.touched = 0ull; W.head = NIL; W.tail = NIL; W.n_ovf = 0;
        cio.oldc = A.cache[cur] + cache_slot(e, 0); cio.newc = A.cache[cur ^ 1] + cache_slot(e, 0);
        cio.n = A.n; cio.e = e; cio.old_count = old_count;
        /* preload the cached arbiter entries: independent loads, one memory round trip */
#pragma unroll
        for (int j = 0; j < OLD_FAST; j++) {
            if (j < old_count) {
                W.old[j * SCR] = u2f(cio.oldc[3 * j]);
                W.old[(OLD_FAST + j) * SCR] = u2f(cio.oldc[3 * j + 1]);
                W.old[(2 * OLD_FAST + j) * SCR] = u2f(cio.oldc[3 * j + 2]);
            }
        }

        /* ---- narrow phase in canonical arbiter order = ascending pair id: agent x segment
           (agent-major), agent x agent, ball x agent, ball x wall.  One loop per pair type (each lane
           walks its own candidates of that type), so a warp only pays for a collide routine as many
           times as its busiest lane needs it. */
        const float *G = W.geom;
#pragma unroll 1
        for (int phase = 0; phase < 4; phase++) { /* warp-uniform: one pair type at a time, one add_contacts site */
            uint32_t todo = phase == 0 ? m_as : phase == 1 ? m_aa : phase == 2 ? m_ba : m_bw;
#pragma unroll 1
            while (todo) {
                const int idx = ctz32(todo);
                todo &= todo - 1;
                Manifold m;
                int pair, a, b; float e_; V2 r1_off = mk(0.0f, 0.0f), r2_off = mk(0.0f, 0.0f);
                if (phase == 0) {
                    const int i = idx >> 3;
                    const Seg g = get_segment(idx & 7);
                    collide_segment_box(g, mk(G[(GF_PX + i) * SCR], G[(GF_PY + i) * SCR]), G[(GF_CS + i) * SCR], G[(GF_SN + i) * SCR], m);
                    pair = idx; a = STATIC_BODY; b = i; e_ = E_AGENT_SEG;
                } else if (phase == 1) {
                    const int i = (idx < 3) ? 0 : (idx < 5) ? 1 : 2;
                    const int j = (idx < 3) ? idx + 1 : (idx < 5) ? idx - 1 : 3;
                    const V2 off = mk(G[(GF_PX + j) * SCR] - G[(GF_PX + i) * SCR], G[(GF_PY + j) * SCR] - G[(GF_PY + i) * SCR]);
                    collide_box_box(G[(GF_CS + i) * SCR], G[(GF_SN + i) * SCR], G[(GF_CS + j) * SCR], G[(GF_SN + j) * SCR], off, m);
                    pair = PAIR_AGENT_AGENT + idx; a = i; b = j; e_ = E_AGENT_AGENT; r2_off = off;
                } else if (phase == 2) {
                    const V2 cb = mk(G[(GF_PX + 4) * SCR] - G[(GF_PX + idx) * SCR], G[(GF_PY + 4) * SCR] - G[(GF_PY + idx) * SCR]);
                    collide_ball_box(cb, G[(GF_CS + idx) * SCR], G[(GF_SN + idx) * SCR], m);
                    pair = PAIR_BALL_AGENT + idx; a = BALL; b = idx; e_ = E_BALL_AGENT; r1_off = cb;
                } else {
                    const Seg g = get_segment(idx);
                    collide_ball_segment(g, mk(G[(GF_PX + 4) * SCR], G[(GF_PY + 4) * SCR]), m);
                    pair = PAIR_BALL_WALL + idx; a = BALL; b = STATIC_BODY; e_ = E_BALL_WALL;
                }
                if (m.count) add_contacts(W, cio, pair, a, b, e_, m, r1_off, r2_off);
            }
        }
        n_contacts = W.nc; overflow = W.overflow;

        if (W.nc > 0) {
            /* ---- cpArbiterPreStep with the (parked) velocities from BEFORE the velocity update */
#pragma unroll 1
            for (int p = W.head; p != NIL;) {
                if (p >= 0) { float *cp = W.pool + p; prestep_contact<CON_FS>(cp, W.body, c); p = (int)f2u(cp[CF_NEXT * CON_FS]); }
                else { float *cp = &W.ovf[-1 - p][0]; prestep_contact<1>(cp, W.body, c); p = (int)f2u(cp[CF_NEXT]); }
            }
#pragma unroll
            for (int i = 0; i < 5; i++) {
                float *pb = W.body + i * SCR;
                pb[BF_VX * BODY_FS] = E.vx[i]; pb[BF_VY * BODY_FS] = E.vy[i]; pb[BF_W * BODY_FS] = E.w[i];
                pb[BF_BX * BODY_FS] = 0.0f; pb[BF_BY * BODY_FS] = 0.0f; pb[BF_BW * BODY_FS] = 0.0f;
            }
            /* ---- cpArbiterApplyCachedImpulse */
#pragma unroll 1
            for (int p = W.head; p != NIL;) {
                if (p >= 0) { float *cp = W.pool + p; warmstart_contact<CON_FS>(cp, W.body, c); p = (int)f2u(cp[CF_NEXT * CON_FS]); }
                else { float *cp = &W.ovf[-1 - p][0]; warmstart_contact<1>(cp, W.body, c); p = (int)f2u(cp[CF_NEXT]); }
            }
            /* ---- cpArbiterApplyImpulse x 10, contacts in arbiter order */
            BodyCache bc; bc.cur = -1;
            bc.vx = bc.vy = bc.w = bc.bx = bc.by = bc.bw = 0.0f;
#if defined(__CUDACC__)
#pragma unroll 1
#endif
            for (int it = 0; it < SOLVER_ITERS; it++) {
#pragma unroll 1
                for (int p = W.head; p != NIL;) {
                    if (p >= 0) { float *cp = W.pool + p; const int nx_ = (int)f2u(cp[CF_NEXT * CON_FS]); solve_contact<CON_FS>(cp, W.body, c, bc); p = nx_; }
                    else { float *cp = &W.ovf[-1 - p][0]; const int nx_ = (int)f2u(cp[CF_NEXT]); solve_contact<1>(cp, W.body, c, bc); p = nx_; }
                }
            }
            bc_flush(bc, W.body);
#pragma unroll
            for (int i = 0; i < 5; i++) {
                const float *pb = W.body + i * SCR;
                E.vx[i] = pb[BF_VX * BODY_FS]; E.vy[i] = pb[BF_VY * BODY_FS]; E.w[i] = pb[BF_W * BODY_FS];
                E.vbx[i] = pb[BF_BX * BODY_FS]; E.vby[i] = pb[BF_BY * BODY_FS];
            }
#pragma unroll
            for (int i = 0; i < 4; i++) E.wb[i] = W.body[i * SCR + BF_BW * BODY_FS];
        }

        /* ---- arbiter cache for the next step: this step's contacts (age 0), then the untouched
           arbiters younger than collision_persistence (3) */
        for (int p = W.head; p != NIL && new_count < MAX_CACHE;) {
            int fs; const float *cp = contact_ptr(W, p, fs);
            p = (int)f2u(cp[CF_NEXT * fs]);
            cio.newc[3 * new_count] = (f2u(cp[CF_META * fs]) >> 6) & 1023u; /* pair | key<<6, age 0 */
            cio.newc[3 * new_count + 1] = f2u(cp[CF_JN * fs]); cio.newc[3 * new_count + 2] = f2u(cp[CF_JT * fs]);
            new_count++;
        }
        for (int j = 0; j < old_count; j++) {
            const uint32_t info = old_info_at(W, cio, j);
            const uint32_t age = (info >> 10) & 3u;
            if (((W.touched >> (info & 63u)) & 1ull) || age >= 2u) continue;
            if (new_count >= MAX_CACHE) { overflow++; continue; }
            cio.newc[3 * new_count] = (info & 1023u) | ((age + 1u) << 10);
            cio.newc[3 * new_count + 1] = f2u(old_jn_at(W, cio, j)); cio.newc[3 * new_count + 2] = f2u(old_jt_at(W, cio, j));
            new_count++;
        }
        /* poses back from the scratch */
#pragma unroll
        for (int i = 0; i < 5; i++) { E.px[i] = W.geom[(GF_PX + i) * SCR]; E.py[i] = W.geom[(GF_PY + i) * SCR]; }
#pragma unroll
        for (int i = 0; i < 4; i++) E.ang[i] = W.geom[(GF_ANG + i) * SCR];
    }
    if (age_only) {
        /* nothing can touch this step, but the env still carries arbiters of contacts that ended
           less than collision_persistence (3) steps ago: age them (cpSpaceArbiterSetFilter) */
        const uint32_t *oc = A.cache[cur] + cache_slot(e, 0);
        uint32_t *nc_ = A.cache[cur ^ 1] + cache_slot(e, 0);
        for (int j = 0; j < old_count; j++) {
            const uint32_t info = oc[3 * j];
            const uint32_t age = (info >> 10) & 3u;
            if (age >= 2u) continue;
            nc_[3 * new_count] = (info & 1023u) | ((age + 1u) << 10);
            nc_[3 * new_count + 1] = oc[3 * j + 1]; nc_[3 * new_count + 2] = oc[3 * j + 2];
            new_count++;
        }
    }

    MSOC_CHECK(new_count >= 0 && new_count <= MAX_CACHE && old_count <= MAX_CACHE, CHK_CACHE_COUNT);
    MSOC_CHECK(E.px[4] == E.px[4] && E.vx[0] == E.vx[0] && E.ang[3] == E.ang[3], CHK_FINITE_STATE);
    E.flags = (E.flags & ~(FLAG_CACHE_MASK | FLAG_INJECT)) | (uint32_t)new_count;

    /* ---- goal test (game/game.py:401-412), strict inequalities */
    int goal = 0;
    const float bx = E.px[4], by = E.py[4];
    if (bx < FIELD_L && GOAL_Y_BOT < by && by < GOAL_Y_TOP) { goal = -1; E.score_r++; }
    else if (bx > FIELD_R && GOAL_Y_BOT < by && by < GOAL_Y_TOP) { goal = +1; E.score_b++; }

    /* ---- goal / alive terms of the reward (game/game.py:362-373) */
    if (goal > 0) r += c.goal_reward;
    if (goal < 0) r -= c.conceded_penalty;
    r -= c.alive_penalty;
    if (TEAMS) {
        if (goal < 0) r_red += c.goal_reward;
        if (goal > 0) r_red -= c.conceded_penalty;
        r_red -= c.alive_penalty;
    }

    /* ---- soft reset on goal (game/game.py:421-422, :120-127): positions re-spawned in the current
       mode, velocities zeroed, agent angles 0/pi; ball angular velocity, biases, counters kept */
    if (goal != 0) {
        uint32_t sc = A.spawn_count[e];
        float px[5], py[5];
        sc = spawn_positions((int)((E.flags & FLAG_MODE_MASK) >> FLAG_MODE_SHIFT), A.seed[e], gidx, sc, px, py);
        A.spawn_count[e] = sc;
#pragma unroll
        for (int i = 0; i < 5; i++) { E.px[i] = px[i]; E.py[i] = py[i]; E.vx[i] = 0.0f; E.vy[i] = 0.0f; }
#pragma unroll
        for (int i = 0; i < 4; i++) { E.w[i] = 0.0f; E.ang[i] = (i < 2) ? 0.0f : PI_F; }
    }

    /* ---- truncation at max_steps (game/game.py:424-433): reward replaced by the terminal bonus */
    bool done = false;
    if (c.max_steps > 0 && E.steps >= c.max_steps) {
        done = true;
        r = c.score_diff_mult * (float)(E.score_b - E.score_r);
        if (TEAMS) r_red = c.score_diff_mult * (float)(E.score_r - E.score_b);
    }
    E.ep_return += r;
    out.reward = r; out.reward_r = r_red; out.done = done ? 1 : 0; out.goal = (int8_t)goal;
    out.fresh_episode = false; out.finished_return = 0.0f; out.score_dirty = goal != 0;
    out.n_contacts = n_contacts; out.overflow = overflow;
    out.score_b = E.score_b; out.score_r = E.score_r;
    if (done) {
        out.finished_return = E.ep_return;
        E.ep_return = 0.0f;
        if (step_flags & 1u) { /* marl_vecenv.py:45-53: auto-reset, full-random mode, no re-seed */
            uint32_t sc = A.spawn_count[e];
            env_full_reset(E, 2, A.seed[e], gidx, sc);
            A.spawn_count[e] = sc;
            out.fresh_episode = true; out.score_dirty = true;
        }
    }
    return true;
}

} /* namespace msoc */
