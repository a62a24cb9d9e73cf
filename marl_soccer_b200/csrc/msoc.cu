/*
 * msoc.cu -- B200 (sm_100a) kernels and the C-ABI (include/msoc.h) of the batched 2v2 soccer
 * simulator.  Replaces the reference's per-env Python/pymunk update loop
 * (soccer_simulation/marl_vecenv.py:30-68 -> soccer_env.py:100-154 -> game/game.py:378-437 ->
 * pymunk Space.step) with one fused device step per vectorised step: two launches, see "The fused step".
 *
 * Data layout: one 128-byte record per env in each of three rotating buffers (msoc::Arrays in step_core.cuh);
 * one thread owns one env while it is stepped, one warp a batch of 32 envs (consecutive in the streaming kernel,
 * listed in the contact kernel).  The stacked observations (N,4,66) are never read back: once a warp has stored
 * the new states, the three buffers hold the poses behind the three frames of the stack, and the warp rebuilds
 * the observations of its envs from them -- four lanes per env (one per agent), eight envs at a time, staged in
 * shared memory in the layout of the output and written as whole 1 056-byte blocks by bulk asynchronous copies, so
 * that every DRAM sector is written exactly once and in full.
 *
 * There is no CPU fallback in this library: every entry point needs a CUDA device.
 */
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <atomic>
#include <string>
#include <vector>

#include "../../include/msoc.h"
#include "step_core.cuh"
#include "render_core.cuh"

using namespace msoc;

#ifdef MSOC_CHECKS
__device__ unsigned int g_msoc_check_bits;
#endif

/* ------------------------------------------------------------------------------------ errors */
static thread_local std::string g_last_error;
static std::atomic<uint64_t> g_launches{0};

static int fail(int code, const char *what, cudaError_t ce = cudaSuccess)
{
    char buf[512];
    if (ce != cudaSuccess) snprintf(buf, sizeof buf, "%s: %s", what, cudaGetErrorString(ce));
    else snprintf(buf, sizeof buf, "%s", what);
    g_last_error = buf;
    return code;
}
#define CUDA_TRY(expr)                                                        \
    do {                                                                      \
        cudaError_t _e = (expr);                                              \
        if (_e != cudaSuccess) return fail(MSOC_ERR_CUDA, #expr, _e);         \
    } while (0)

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

/* ------------------------------------------------------------------------------------ handle */
constexpr int MAX_CHUNKS = 8; /* pipeline stages of the host-buffer step */
/* control block in device memory (ints): two sets of list counters that alternate between steps, the step counters
   that select the ping-pong halves, one set of list counters per pipeline chunk of the host-buffer step */
enum { CTL_LIGHT = 0, CTL_HEAVY = 1, CTL_NEXT_BATCH = 2, CTL_PAIR = 4, CTL_MULTI = 5, CTL_WORDS = 8 };
enum { CTL_STEP_FAST = 16, CTL_STEP_CONTACT = 17, CTL_LAST_COUNTS = 20 /* light, heavy, pair, multi of the last step */, CTL_CHUNK0 = 24, CTL_TOTAL = CTL_CHUNK0 + CTL_WORDS * MAX_CHUNKS };

struct msoc_handle {
    int device;
    int64_t n;
    uint64_t global_offset;
    SimCfg cfg;
    Arrays A;
    int sm_count, blocks_per_sm; /* persistent grid of the contact kernel */
    int blocks_per_sm_teams;     /* the same for its TEAMS instance (msoc_step_teams) */
    int heavy_lanes_override; /* MSOC_HEAVY_LANES (experiments): 0 = choose by batch size */
    void *slab;
    /* internal I/O buffers of the host-buffer API */
    float *d_obs, *d_act, *d_rew;
    uint8_t *d_done, *d_mask;
    int8_t *d_goal;
    int32_t *d_score;
    double *d_stats; /* 8 doubles, msoc_stats layout */
    int *d_ctl;      /* CTL_TOTAL ints */
    int *d_list;     /* n ints: contact lists of the step in flight (light from the front of a range, heavy from its back) */
    int *d_list2;    /* n ints: pair class from the front, multi class from the back */
    float *d_frames; /* (N,4,22) newest frames, msoc_step_host_frames; allocated on first use */
    void *d_inject;  /* Arrays::inject, allocated by the first msoc_set_state */
    cudaStream_t pipe_stream;          /* second lane of the chunked host-buffer step */
    cudaEvent_t ev_pipe_fork, ev_pipe_join;
    void *d_stage; size_t stage_bytes; /* get/set_state staging */
};

constexpr int WARPS_PER_BLOCK = 4;
constexpr int BLOCK = WARPS_PER_BLOCK * 32; /* reset kernel */

/* ------------------------------------------------------------------ observation blocks */
constexpr int ENV_STRIDE = SCRATCH_WORDS | 1; /* floats of per-lane solver scratch in the contact kernel; odd: no bank conflicts */
constexpr int OBS_ENVS = 8;                     /* envs whose observations a warp builds at a time */
constexpr int BLOCK_WORDS = OBS_ENVS * 4 * OBS;  /* floats of staged observation blocks: 8 x (4 x 66) */
constexpr int REC_F4 = 7;                        /* float4s of a record that a frame is made of */
constexpr int RECS_WORDS = OBS_ENVS * 3 * REC_F4 * 4; /* floats of staged records: 8 envs x 3 buffers x 7 float4 */
constexpr int STAGE_WORDS = BLOCK_WORDS + RECS_WORDS; /* per warp: 8 448 + 2 688 bytes, both 16-byte multiples */

/* ---------------------------------------------------------------------------- the fused step */
struct StepParams {
    Arrays A;
    SimCfg cfg;
    const float *actions; /* (N,4,3) */
    float *obs_out;       /* (N,4,66) */
    float *frames_out;    /* (N,4,22) or null */
    float *reward;        /* (N,2); (N,4), 16-byte aligned, in the TEAMS instances (msoc_step_teams) */
    uint8_t *done;        /* (N) */
    int8_t *goal;         /* (N) */
    int32_t *score;       /* (N,2) or null */
    double *stats;        /* 8 */
    int *ctl;             /* the handle's control block */
    int *list;            /* N slots: envs that need the contact path -- light from the front of [e0, e1), heavy from its back */
    int *list2;           /* N slots: pair class from the front of [e0, e1), multi class from its back */
    int64_t e0, e1;       /* the envs this launch steps */
    uint64_t global_offset;
    uint32_t flags;
    int heavy_lanes;      /* envs per heavy warp-batch (MSOC_HEAVY_LANES, experiments) or 0: chosen by the contact kernel */
    int chunk;            /* -1: a whole step (list counters alternate with the step counter, the contact kernel advances it);
                             >= 0: one pipeline chunk of a host-buffer step (its own pre-zeroed counters, nobody advances) */
};

#ifdef MSOC_TIMELINE /* debug build only (tools/timeline.py): when did every batch of every step kernel run? */
__device__ unsigned long long g_tl[1 << 18]; /* records of 4 words: kernel id, start, end (globaltimer ns), sm id */
__device__ unsigned int g_tl_n;
extern "C" int msoc_debug_timeline(unsigned long long *out, unsigned int *n) {
    cudaMemcpyFromSymbol(n, g_tl_n, sizeof(unsigned int)); unsigned int z = 0; cudaMemcpyToSymbol(g_tl_n, &z, sizeof z);
    return (int)cudaMemcpyFromSymbol(out, g_tl, sizeof g_tl);
}
__device__ __forceinline__ unsigned long long gtime() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
__device__ __forceinline__ void tl_record(int kid, unsigned long long t0) {
    const unsigned int i = atomicAdd(&g_tl_n, 1u);
    unsigned int smid; asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    if (i < (1u << 16)) { g_tl[4 * i] = (unsigned long long)kid; g_tl[4 * i + 1] = t0; g_tl[4 * i + 2] = gtime(); g_tl[4 * i + 3] = smid; }
}
#define MSOC_TL_BEGIN() const unsigned long long tl0 = gtime()
#define MSOC_TL_END(kid) do { if (lane == 0) tl_record(kid, tl0); } while (0)
#else
#define MSOC_TL_BEGIN() do { } while (0)
#define MSOC_TL_END(kid) do { } while (0)
#endif
/* Per-thread tallies for the per-rollout statistics. */
struct Tally { int done, goals_b, goals_r, contacts, overflow, nonfinite; float ret; };
__device__ __forceinline__ void tally_clear(Tally &T) { T.done = T.goals_b = T.goals_r = T.contacts = T.overflow = T.nonfinite = 0; T.ret = 0.0f; }

__device__ __forceinline__ int *step_ctl(const StepParams &P, int step) { return P.chunk < 0 ? P.ctl + CTL_WORDS * (step & 1) : P.ctl + CTL_CHUNK0 + CTL_WORDS * P.chunk; }

/* Loads env e (the record of buffer step % 3, or the injected record of a flagged env) and its actions, steps it.  On
   success (always, except for the contact-free mode, which declines envs that need the contact path) the per-env
   outputs and the new state are written; the observation follows in obs_tile once the whole warp has stored. */
template <bool TEAMS>
__device__ __forceinline__ bool step_one_env(const int MODE, const int ALLOWED, const StepParams &P, int step, int64_t e, Work &W, int &load, Tally &T)
{
    float act[12];
    const float4 *a4 = reinterpret_cast<const float4 *>(P.actions + e * 12);
    const float4 x0 = __ldg(a4), x1 = __ldg(a4 + 1), x2 = __ldg(a4 + 2);
    act[0] = x0.x; act[1] = x0.y; act[2] = x0.z; act[3] = x0.w;
    act[4] = x1.x; act[5] = x1.y; act[6] = x1.z; act[7] = x1.w;
    act[8] = x2.x; act[9] = x2.y; act[10] = x2.z; act[11] = x2.w;
    /* soccer_env.py:116-117 raises on non-finite actions; a device-resident caller gets a counter instead (the clip
       turns NaN into -1) */
    bool finite = true;
#pragma unroll
    for (int k = 0; k < 12; k++) finite = finite && (fabsf(act[k]) <= 3.0e38f);
    Env E;
    const float4 *rec = P.A.pose[buf_cur(step)] + e * POSE_F4;
    if ((ALLOWED & (1 << MODE_FULL)) && MODE == MODE_FULL) { /* the only kernel that sees injected states */
        if (__float_as_uint(rec[7].z) & FLAG_INJECT) rec = P.A.inject + e * POSE_F4;
    }
    load_env(P.A, rec, e, E);
    StepOut out;
    if (!env_step<TEAMS>(MODE, ALLOWED, E, act, P.cfg, P.A, cache_half(step), e, P.global_offset + (uint64_t)e, P.flags, W, out, load)) return false;
    if (TEAMS) reinterpret_cast<float4 *>(P.reward)[e] = make_float4(out.reward, out.reward, out.reward_r, out.reward_r);
    else reinterpret_cast<float2 *>(P.reward)[e] = make_float2(out.reward, out.reward);
    P.done[e] = out.done;
    P.goal[e] = out.goal;
    if (P.score != nullptr) reinterpret_cast<int2 *>(P.score)[e] = make_int2(out.score_b, out.score_r);
    store_env(P.A, buf_next(step), e, E, out.score_dirty);
    if (out.fresh_episode) { /* a fresh episode has no history but its first frame (soccer_env.py:92-96) */
        store_env_record(P.A.pose[buf_cur(step)] + e * POSE_F4, E);
        store_env_record(P.A.pose[buf_prev(step)] + e * POSE_F4, E);
    }
    T.nonfinite += finite ? 0 : 1;
    T.done += out.done; T.goals_b += out.goal > 0; T.goals_r += out.goal < 0;
    T.contacts += out.n_contacts; T.overflow += out.overflow; T.ret += out.finished_return;
    return true;
}

/* ---- bulk asynchronous copies (the TMA engine, PTX cp.async.bulk): shared memory -> global memory */
__device__ __forceinline__ void bulk_store(void *gdst, const void *ssrc, uint32_t bytes)
{
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"((uint32_t)__cvta_generic_to_shared(ssrc)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
/* until the engine has READ the shared-memory sources of all committed groups (they may then be overwritten) */
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
/* orders this thread's shared-memory writes before later bulk copies of any thread it then synchronises with */
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

/* Stacked observations [frame(t-2) | frame(t-1) | frame(t)] (soccer_env.py:130-140) of the warp's envs whose bit is set
   in `mask` (lane l owns env `my_env`; its new state is stored), eight envs at a time:
     1. the warp fetches the 8 x 3 records (buffers (step+2)%3, step%3 -- L1/L2 hits, this warp read or prefetched
        them -- and (step+1)%3, just written by sibling lanes: read from L2) with 16-byte loads, 168 in all, the loads of
        the next eight envs in flight while the current ones are worked on, and parks them in shared memory;
     2. lane = (env, agent) rebuilds its agent's three frames and puts them where they belong in the env's 4 x 66 block;
     3. the blocks leave as bulk asynchronous copies, one per env (1 056 contiguous, 32-byte aligned bytes = 33 whole
        sectors; nothing is ever read back or written twice).
   frames_out (or null): the newest frames once more, compact (N,4,22), for the host path. */
struct RecLoad { float4 v[6]; };
/* which record word lane `lane` fetches in round r: slot r*32 + lane in [buffer][env][float4] order, 168 used */
__device__ __forceinline__ void fetch_slot(int r, int lane, int &k, int &e8, int &f)
{
    const int sl = r * 32 + lane;
    k = sl / (OBS_ENVS * REC_F4);
    const int rem = sl - k * (OBS_ENVS * REC_F4);
    e8 = rem / REC_F4; f = rem - e8 * REC_F4;
}
__device__ __forceinline__ void obs_fetch(const Arrays &A, int step, uint32_t mask, int g, int my_env, int lane, RecLoad &R)
{
    const uint32_t m8 = (mask >> (8 * g)) & 0xffu;
#pragma unroll
    for (int r = 0; r < 6; r++) {
        int k, e8, f;
        fetch_slot(r, lane, k, e8, f);
        const int env = __shfl_sync(0xffffffffu, my_env, (8 * g + e8) & 31);
        R.v[r] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        if ((r < 5 || lane < 3 * OBS_ENVS * REC_F4 - 160) && ((m8 >> e8) & 1u)) {
            const int b = k == 0 ? buf_prev(step) : k == 1 ? buf_cur(step) : buf_next(step);
            const float4 *p = A.pose[b] + (int64_t)env * POSE_F4 + f;
            R.v[r] = k == 2 ? __ldcg(p) : *p;
        }
    }
}
__device__ __forceinline__ void obs_tile(const Arrays &A, const SimCfg &cfg, float *obs_out, float *frames_out, int step, float *s_stage,
                                         uint32_t lane_mask, int64_t my_env64, int lane)
{
    const int a = lane & 3, el = lane >> 2;
    float4 *recs4 = reinterpret_cast<float4 *>(s_stage + BLOCK_WORDS);
    float2 *mine = reinterpret_cast<float2 *>(s_stage) + lane * 33; /* row (el, a) of the staged blocks */
    __syncwarp(); /* the siblings' stores of the new records are ordered before the loads below */
    /* the envs of the lanes in lane_mask, compacted: the streaming kernel's warps have ~23 of 32 (the others were declined),
       which is three groups of eight instead of four */
    uint32_t mask = lane_mask;
    int my_env = (int)my_env64; /* a handle holds fewer than 2^31 envs */
    if (lane_mask != 0xffffffffu) {
        int *s_idx = reinterpret_cast<int *>(s_stage);
        if ((lane_mask >> lane) & 1u) s_idx[__popc(lane_mask & ((1u << lane) - 1u))] = my_env;
        __syncwarp();
        const int cnt = __popc(lane_mask);
        my_env = lane < cnt ? s_idx[lane] : 0;
        mask = (1u << cnt) - 1u; /* cnt < 32 here */
        __syncwarp();
    }
    int g = __ffs((int)((mask & 0xffu ? 1u : 0u) | (mask & 0xff00u ? 2u : 0u) | (mask & 0xff0000u ? 4u : 0u) | (mask & 0xff000000u ? 8u : 0u))) - 1;
    RecLoad R;
    obs_fetch(A, step, mask, g, my_env, lane, R);
#pragma unroll 1
    while (true) {
        const uint32_t m8 = (mask >> (8 * g)) & 0xffu;
        /* the staging areas are free: every lane has waited for its own bulk copies, then the warp synchronised */
#pragma unroll
        for (int r = 0; r < 6; r++)
            if (r < 5 || lane < 3 * OBS_ENVS * REC_F4 - 160) recs4[r * 32 + lane] = R.v[r];
        __syncwarp();
        /* next group with work, its loads in flight from here on */
        int gn = g + 1;
        while (gn < 4 && ((mask >> (8 * gn)) & 0xffu) == 0u) gn++;
        if (gn < 4) obs_fetch(A, step, mask, gn, my_env, lane, R);
        const int env = __shfl_sync(0xffffffffu, my_env, 8 * g + el);
        if ((m8 >> el) & 1u) {
            MSOC_CHECK(env >= 0 && env < A.n, CHK_OBS_ENV);
#pragma unroll
            for (int k = 0; k < 3; k++) {
                float o[22];
                frame_of_record(recs4 + (k * OBS_ENVS + el) * REC_F4, a, cfg, o);
#pragma unroll
                for (int i = 0; i < 11; i++) mine[k * 11 + i] = make_float2(o[2 * i], o[2 * i + 1]);
            }
        }
        fence_async_smem();
        __syncwarp();
        if (a == 0 && ((m8 >> el) & 1u)) /* one lane per env */
            bulk_store(obs_out + (int64_t)env * (4 * OBS), s_stage + el * (4 * OBS), 4 * OBS * sizeof(float));
        bulk_commit();
        if (frames_out != nullptr) {
            float2 *fr2 = reinterpret_cast<float2 *>(frames_out);
            const float2 *stage2 = reinterpret_cast<const float2 *>(s_stage);
#pragma unroll
            for (int it = 0; it < 11; it++) { /* 8 x 4 x 11 = 352 float2: the third frame of every row */
                const int idx = it * 32 + lane;
                const int row = idx / 11, j = idx - row * 11;
                const int env2 = __shfl_sync(0xffffffffu, my_env, 8 * g + (row >> 2));
                if ((m8 >> (row >> 2)) & 1u) fr2[(int64_t)env2 * 44 + (row & 3) * 11 + j] = stage2[row * 33 + 22 + j];
            }
        }
        bulk_wait_read();
        __syncwarp();
        if (gn >= 4) break;
        g = gn;
    }
}

/* The fused step is two launches on the caller's stream.
   msoc_step_fast_kernel     streams over ALL envs, thread t of block b steps env e0 + b*128 + t in contact-free
                             mode and its warp writes the observation rows.  No contact code is compiled into
                             it: few registers, small shared memory, small instruction footprint -> many
                             resident warps to hide the HBM latency.  Envs whose broad phase finds a candidate
                             pair (~27 % in the benchmark mix) write nothing and are appended, one atomic per
                             warp and class, to the list of their work class (step_core.cuh LOAD_*): light
                             (exactly one agent x wall pair, the bulk), pair (exactly one agent x agent or
                             ball x agent pair, at most one agent x wall pair beside it), multi (only wall candidates, several), heavy (anything else).
   msoc_step_contact_kernel  every warp of a persistent grid pulls batches of listed envs of ONE class -- heavy
                             batches first, then multi, pair, light: longest first -- and every thread steps one
                             env in the mode of its class: the register-only single-body solver (light), islands
                             of one or two bodies with their contacts in the lane's shared-memory slots (pair,
                             multi), or the general Chipmunk path (heavy): narrow phase over all candidate pairs,
                             arbiter cache, 10-iteration impulse solver with bodies and contacts in shared
                             memory.  The warp then writes the rows.
   The divergent, latency-bound contact work therefore always runs on warps of similar work, and the few long
   heavy batches start at once on their own warps while all other warps stream through the rest.  (Separate kernels
   per class on separate streams were measured to run one after the other, not side by side: profiles/.)

   Which half of the ping-pong state is current is a step counter in DEVICE memory (so a captured CUDA graph of any
   number of steps replays correctly): the fast kernel reads ctl[CTL_STEP_FAST] and copies it to ctl[CTL_STEP_CONTACT]
   for the contact kernel of the same step; the contact kernel, which only starts when the fast kernel is complete
   and is complete before the next fast kernel starts, writes the incremented counter back. */
#ifndef MSOC_FAST_BLOCK
#define MSOC_FAST_BLOCK 128
#endif
constexpr int FAST_BLOCK = MSOC_FAST_BLOCK; /* envs (= threads) per block of the fast kernel */
constexpr size_t FAST_SMEM_BYTES = (size_t)(FAST_BLOCK / 32) * STAGE_WORDS * sizeof(float);
#ifndef MSOC_FAST_MIN_BLOCKS
#define MSOC_FAST_MIN_BLOCKS 4
#endif

/* warp reduce of the per-rollout statistics (marl-soccer.ipynb:411-429), one atomic per warp and counter */
__device__ __forceinline__ void flush_tally(const Tally &T, double *stats, int lane)
{
    int nd = T.done, gb = T.goals_b, gr = T.goals_r, nc = T.contacts, ov = T.overflow, nf = T.nonfinite;
    float ret = T.ret;
    if (!__any_sync(0xffffffffu, (nd | gb | gr | nc | ov | nf) != 0)) return; /* the common case of the streaming kernel */
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        nd += __shfl_xor_sync(0xffffffffu, nd, o); gb += __shfl_xor_sync(0xffffffffu, gb, o);
        gr += __shfl_xor_sync(0xffffffffu, gr, o); nc += __shfl_xor_sync(0xffffffffu, nc, o);
        ov += __shfl_xor_sync(0xffffffffu, ov, o);
        nf += __shfl_xor_sync(0xffffffffu, nf, o);
        ret += __shfl_xor_sync(0xffffffffu, ret, o);
    }
    if (lane == 0) {
        if (nd) { atomicAdd(stats + 0, (double)nd); atomicAdd(stats + 1, (double)ret); }
        if (gb) atomicAdd(stats + 2, (double)gb);
        if (gr) atomicAdd(stats + 3, (double)gr);
        if (nc) atomicAdd(stats + 5, (double)nc);
        if (ov) atomicAdd(stats + 6, (double)ov);
        if (nf) atomicAdd(stats + 7, (double)nf);
    }
}

/* TEAMS (both step kernels): the step of msoc_step_teams, red's reward beside blue's (env_step) */
template <bool TEAMS>
__global__ void __launch_bounds__(FAST_BLOCK, MSOC_FAST_MIN_BLOCKS) msoc_step_fast_kernel(const __grid_constant__ StepParams P)
{
    extern __shared__ __align__(16) float s_dyn[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    float *s_warp = s_dyn + warp * STAGE_WORDS;
    cudaGridDependencySynchronize(); /* launched programmatically behind the previous kernel of the stream */
    const int step = P.ctl[CTL_STEP_FAST];
    int *ctl = step_ctl(P, step);
    if (blockIdx.x == 0) {
        if (P.chunk < 0 && tid < CTL_WORDS) P.ctl[CTL_WORDS * ((step & 1) ^ 1) + tid] = 0; /* the next step's list counters */
        if (tid == 0) {
            P.ctl[CTL_STEP_CONTACT] = step;
            atomicAdd(P.stats + 4, (double)(P.e1 - P.e0)); /* every env of the range is stepped by one of the two kernels */
        }
    }
    MSOC_TL_BEGIN();
    const int64_t my_env = P.e0 + (int64_t)blockIdx.x * FAST_BLOCK + tid;
    const bool have = my_env < P.e1;
    Tally T; tally_clear(T);
    Work W; /* never touched in contact-free mode */
    W.ovf = nullptr; W.body = W.pool = W.geom = W.old = W.isl = nullptr; W.pool_count = nullptr;
    bool ok = false;
    int load = 0;
    if (have) {
        /* the oldest of the three records the observation is rebuilt from is not needed by the step: start pulling it */
        asm volatile("prefetch.global.L2 [%0];" ::"l"(P.A.pose[buf_prev(step)] + my_env * POSE_F4));
        ok = step_one_env<TEAMS>(MODE_FAST, 1 << MODE_FAST, P, step, my_env, W, load, T);
    }
    const uint32_t mask = __ballot_sync(0xffffffffu, ok);
    /* list slots of the declined envs, by work class: lanes 0..3 each fetch the base of one class (one atomic per warp and
       class that occurs); the atomics are in flight while the observations are built */
    const bool declined = have && !ok;
    const uint32_t mdec = __ballot_sync(0xffffffffu, declined);
    uint32_t mclass = 0u; /* the warp's declined lanes of my class */
    int base = 0;
    if (mdec != 0u) {
        const uint32_t b0 = __ballot_sync(0xffffffffu, declined && (load & 1)), b1 = __ballot_sync(0xffffffffu, declined && (load & 2));
        auto class_mask = [&](int cl) { return mdec & ((cl & 1) ? b0 : ~b0) & ((cl & 2) ? b1 : ~b1); };
        mclass = class_mask(load);
        const uint32_t of_lane = class_mask(lane & 3); /* lane c < 4 speaks for class c */
        if (lane < N_LOADS && of_lane != 0u) {
            const int word = lane == LOAD_LIGHT ? CTL_LIGHT : lane == LOAD_HEAVY ? CTL_HEAVY : lane == LOAD_PAIR ? CTL_PAIR : CTL_MULTI;
            base = atomicAdd(ctl + word, __popc(of_lane));
        }
    }
    if (mask != 0u) obs_tile(P.A, P.cfg, P.obs_out, P.frames_out, step, s_warp, mask, my_env, lane);
    if (mdec != 0u) {
        base = __shfl_sync(0xffffffffu, base, declined ? load : 0);
        if (declined) {
            const int rank = base + __popc(mclass & ((1u << lane) - 1u));
            int *lst = (load == LOAD_LIGHT || load == LOAD_HEAVY) ? P.list : P.list2;
            const bool front = load == LOAD_LIGHT || load == LOAD_PAIR;
            lst[front ? P.e0 + rank : P.e1 - 1 - rank] = (int)my_env;
        }
    }
    flush_tally(T, P.stats, lane);
    if ((blockIdx.x & 15) == 0 && warp == 0) MSOC_TL_END(0);
}

/* Per-warp scratch of 32 x ENV_STRIDE floats: during the contact solve it holds the lanes' solver bodies (30 fields,
   field-major with stride 32: conflict-free), the warp's pool of 32 x CON_FAST contact records (15 fields, field-major;
   an env takes as many records as it has contacts; in the pair / multi modes the same words are the lanes' own island
   slots), the parked poses and the preloaded arbiter cache entries; afterwards the staged observation blocks. */
static_assert(STAGE_WORDS <= 32 * ENV_STRIDE, "the observation staging must fit the per-warp solver scratch");
#ifndef MSOC_HEAVY_BLOCK
#define MSOC_HEAVY_BLOCK 64 /* threads per block of the contact kernel */
#endif
constexpr int HEAVY_BLOCK = MSOC_HEAVY_BLOCK;
#ifndef MSOC_HEAVY_MIN_BLOCKS
#define MSOC_HEAVY_MIN_BLOCKS 4 /* register cap 255: no spills with all four modes compiled in; at 168 registers (5 or 6 blocks) the spills cost more than the extra warps bring */
#endif
constexpr int HEAVY_MIN_BLOCKS = MSOC_HEAVY_MIN_BLOCKS;

constexpr int HEAVY_WARP_WORDS = (32 * ENV_STRIDE + 3) & ~3; /* 16-byte aligned per-warp scratch */
constexpr size_t STEP_SMEM_BYTES = (size_t)(HEAVY_BLOCK / 32) * HEAVY_WARP_WORDS * sizeof(float);

/* All four contact classes in ONE persistent kernel (concurrent kernels with different register / shared-memory shapes
   were measured to run one after the other on this part, not side by side): every warp pulls batches from one counter
   over the combined batch space [heavy | multi | pair | light], i.e. longest batches first, so that the few long
   latency-bound heavy batches start at once on their own warps while all the other warps stream through the rest. */
template <int MODES, bool TEAMS>
__device__ __forceinline__ void contact_body(const StepParams &P, int *s_pool_count)
{
    extern __shared__ __align__(16) float s_dyn[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    float *s_warp = s_dyn + warp * HEAVY_WARP_WORDS;
    cudaGridDependencySynchronize(); /* launched programmatically behind the streaming kernel: wait until it is complete */
    const int step = P.ctl[CTL_STEP_CONTACT];
    int *ctl = step_ctl(P, step);
    /* this step's fast kernel is complete and the next one starts after this kernel: advance the step counter */
    if (P.chunk < 0 && blockIdx.x == 0 && tid == 0) {
        P.ctl[CTL_STEP_FAST] = (step + 1) % 6;
        P.ctl[CTL_LAST_COUNTS + 0] = ctl[CTL_LIGHT]; P.ctl[CTL_LAST_COUNTS + 1] = ctl[CTL_HEAVY];
        P.ctl[CTL_LAST_COUNTS + 2] = ctl[CTL_PAIR]; P.ctl[CTL_LAST_COUNTS + 3] = ctl[CTL_MULTI];
    }
    /* final: the fast kernel has finished */
    const int n_heavy = (MODES & (1 << MODE_FULL)) ? ctl[CTL_HEAVY] : 0, n_multi = (MODES & (1 << MODE_MULTI)) ? ctl[CTL_MULTI] : 0;
    const int n_pair = (MODES & (1 << MODE_PAIR)) ? ctl[CTL_PAIR] : 0, n_light = (MODES & (1 << MODE_LIGHT)) ? ctl[CTL_LIGHT] : 0;
    MSOC_CHECK(step >= 0 && step < 6, CHK_STEP_COUNTER);
    MSOC_CHECK(n_heavy >= 0 && n_light >= 0 && (int64_t)n_heavy + n_light <= P.e1 - P.e0, CHK_LIST_COUNT);
    MSOC_CHECK(n_multi >= 0 && n_pair >= 0 && (int64_t)n_multi + n_pair <= P.e1 - P.e0, CHK_LIST_COUNT);
    /* Envs per heavy batch.  A heavy batch is bound by its latency (the warp walks the union of its lanes' divergent
       contact work: 24 us median / 65 us worst for one env, ~110 us median for 32): as few envs per warp as still gives every heavy batch a warp of
       its own at once; wider batches once there are several times more heavy envs than warps (throughput). */
    int heavy_lanes = P.heavy_lanes;
    if (heavy_lanes == 0) {
        const int n_warps_ = gridDim.x * (HEAVY_BLOCK / 32);
        heavy_lanes = 1;
        while (heavy_lanes < 32 && heavy_lanes * n_warps_ < n_heavy) heavy_lanes *= 2;
        if (heavy_lanes >= 8) heavy_lanes = heavy_lanes >= 16 ? 32 : 16; /* several rounds of batches per warp anyway: throughput
                                                                             (measured: 512 Ki envs 0.282 ms with 16, 0.295 with 8) */
    }
    const int b_heavy = (n_heavy + heavy_lanes - 1) / heavy_lanes;
    const int b_multi = b_heavy + (n_multi + 31) / 32, b_pair = b_multi + (n_pair + 31) / 32;
    const int batches = b_pair + (n_light + 31) / 32;

    Tally T; tally_clear(T);
    float ovf_store[MAXC - CON_FAST][CON_FIELDS]; /* local memory, touched only by envs with more than CON_FAST contacts */
    Work W;
    W.ovf = ovf_store;
    W.body = s_warp + lane;
    W.pool = s_warp + BODY_FIELDS * 5 * 32; /* shared by the warp's lanes */
    W.pool_count = s_pool_count + warp;
    W.geom = s_warp + (BODY_FIELDS * 5 + CON_FIELDS * CON_FAST) * 32 + lane;
    W.old = s_warp + (BODY_FIELDS * 5 + CON_FIELDS * CON_FAST + GEOM_WORDS) * 32 + lane;
    W.isl = s_warp + BODY_FIELDS * 5 * 32 + lane; /* island modes: their contact slots, in the (then idle) contact pool */
    /* A warp's first batch is its own number (so the heavy batches, numbered first, each start at once on a warp of their
       own); the following ones are handed out by the batch counter.  (Claiming batches ahead of time and pulling their
       state into the L2 while the current one is stepped was measured slower: batches waiting behind a long one cost
       more than the latency that is hidden.) */
    const int n_warps = gridDim.x * (HEAVY_BLOCK / 32);
    int b = blockIdx.x * (HEAVY_BLOCK / 32) + warp;
#pragma unroll 1
    while (b < batches) {
        int mode, idx, count, lanes = 32;
        const int *slot;
        if (b < b_heavy)      { mode = MODE_FULL;  lanes = heavy_lanes; idx = b * lanes + lane;  count = n_heavy; slot = P.list + (P.e1 - 1 - idx); }
        else if (b < b_multi) { mode = MODE_MULTI; idx = (b - b_heavy) * 32 + lane; count = n_multi; slot = P.list2 + (P.e1 - 1 - idx); }
        else if (b < b_pair)  { mode = MODE_PAIR;  idx = (b - b_multi) * 32 + lane; count = n_pair;  slot = P.list2 + (P.e0 + idx); }
        else                  { mode = MODE_LIGHT; idx = (b - b_pair) * 32 + lane;  count = n_light; slot = P.list + (P.e0 + idx); }
        const bool have = lane < lanes && idx < count;
        const int64_t my_env = have ? (int64_t)*slot : 0;
        MSOC_CHECK(!have || (my_env >= P.e0 && my_env < P.e1), CHK_LIST_ENV);
        MSOC_TL_BEGIN();
        bool ok = false;
        int load = 0;
        if (lane == 0) *W.pool_count = 0; /* the warp's contact pool is empty */
        __syncwarp();
        if (have) {
            asm volatile("prefetch.global.L2 [%0];" ::"l"(P.A.pose[buf_prev(step)] + my_env * POSE_F4));
            ok = step_one_env<TEAMS>(mode, MODES, P, step, my_env, W, load, T);
        }
        const uint32_t mask = __ballot_sync(0xffffffffu, ok);
        /* (obs_tile starts with a __syncwarp: the solver scratch of every lane is dead before it is reused) */
        if (mask != 0u) obs_tile(P.A, P.cfg, P.obs_out, P.frames_out, step, s_warp, mask, my_env, lane);
        MSOC_TL_END(mode == MODE_FULL ? 2 : mode == MODE_LIGHT ? 1 : 3);
        if (lane == 0) b = n_warps + atomicAdd(ctl + CTL_NEXT_BATCH, 1);
        b = __shfl_sync(0xffffffffu, b, 0);
    }
    flush_tally(T, P.stats, lane);
}

template <bool TEAMS>
__global__ void __launch_bounds__(HEAVY_BLOCK, HEAVY_MIN_BLOCKS) msoc_step_contact_kernel(const __grid_constant__ StepParams P)
{
    __shared__ int s_pool_count[HEAVY_BLOCK / 32];
    contact_body<(1 << MODE_FULL) | (1 << MODE_LIGHT) | (1 << MODE_PAIR) | (1 << MODE_MULTI), TEAMS>(P, s_pool_count);
}

/* after a chunked host-buffer step (whose contact kernels do not): advances the step counter, sums the chunks' class counts */
__global__ void msoc_advance_kernel(int *ctl)
{
    if (threadIdx.x == 0) ctl[CTL_STEP_FAST] = (ctl[CTL_STEP_FAST] + 1) % 6;
    if (threadIdx.x < 4) {
        const int word = threadIdx.x == 0 ? CTL_LIGHT : threadIdx.x == 1 ? CTL_HEAVY : threadIdx.x == 2 ? CTL_PAIR : CTL_MULTI;
        int sum = 0;
        for (int c = 0; c < MAX_CHUNKS; c++) sum += ctl[CTL_CHUNK0 + CTL_WORDS * c + word];
        ctl[CTL_LAST_COUNTS + threadIdx.x] = sum;
    }
}

/* ------------------------------------------------------------------------------------- reset */
struct ResetParams {
    Arrays A;
    SimCfg cfg;
    const uint8_t *mask; /* N or null */
    float *obs_out;      /* (N,4,66) or null */
    const int *ctl;
    uint64_t global_offset, seed;
    int mode, has_seed;
};

__global__ void __launch_bounds__(BLOCK) msoc_reset_kernel(const __grid_constant__ ResetParams P)
{
    __shared__ __align__(16) float s_stage[WARPS_PER_BLOCK][STAGE_WORDS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t block_base = (int64_t)blockIdx.x * BLOCK;
    const int64_t e = block_base + threadIdx.x;
    if (block_base + warp * 32 >= P.A.n) return;
    const int step = P.ctl[CTL_STEP_FAST];
    const bool doit = (e < P.A.n) && (P.mask == nullptr || P.mask[e] != 0);
    if (doit) {
        const uint64_t gidx = P.global_offset + (uint64_t)e;
        uint64_t seed; uint32_t sc;
        if (P.has_seed) { seed = P.seed + gidx; sc = 0; P.A.seed[e] = seed; } /* marl_vecenv.py:23: seed + i */
        else { seed = P.A.seed[e]; sc = P.A.spawn_count[e]; }
        Env E;
        env_full_reset(E, P.mode, seed, gidx, sc);
        P.A.spawn_count[e] = sc;
        /* all three buffers: the observation history of a fresh episode is its first frame (soccer_env.py:92-96).
           The state the next step starts from is buffer step % 3. */
        store_env(P.A, buf_cur(step), e, E, true);
        store_env_record(P.A.pose[buf_prev(step)] + e * POSE_F4, E);
        store_env_record(P.A.pose[buf_next(step)] + e * POSE_F4, E);
    }
    const uint32_t m = __ballot_sync(0xffffffffu, doit);
    if (P.obs_out != nullptr && m != 0u) obs_tile(P.A, P.cfg, P.obs_out, nullptr, step, s_stage[warp], m, e, lane);
}

/* ------------------------------------------------------------------- state save / load (msoc_env_state) */
/* Records of a list of envs as msoc_env_state (include/msoc.h) in device memory, and back.  The state array is large and
   touched once, so both kernels are built around it: a warp takes a group of eight consecutive entries (8 x 808 = 6 464
   bytes, a 16-byte multiple), staged in shared memory in the layout of the array and moved between shared and global
   memory as coalesced 16-byte accesses -- every sector of the array is read or written once and in full.  Four lanes
   serve one env: lane q of the env reads / writes float4 q and q + 4 of each of its 128-byte records, so that every
   warp access of a record covers whole sectors.  The bias block and the arbiter-cache entries are touched only when the
   record's flags say they exist: an env without contacts costs its two records, score, seed and spawn count. */
enum { CHK_STATES = CHK_RENDER + 1 }; /* staging slots, cache counts read from a record, the step counter */
constexpr int STATE_ENVS = 8;                                 /* envs per warp group */
constexpr int STATE_WORDS = (int)(sizeof(msoc_env_state) / 4); /* 202 */
constexpr int STATE_GROUP_U4 = STATE_ENVS * STATE_WORDS / 4;  /* 404 */
constexpr int STATE_BLOCK = 128;
static_assert(sizeof(msoc_env_state) == 808 && (STATE_ENVS * sizeof(msoc_env_state)) % 16 == 0, "msoc_env_state layout");
/* word offsets in msoc_env_state */
enum : int {
    SW_POS = offsetof(msoc_env_state, pos) / 4, SW_VEL = offsetof(msoc_env_state, vel) / 4,
    SW_ANG = offsetof(msoc_env_state, ang) / 4, SW_ANGVEL = offsetof(msoc_env_state, angvel) / 4,
    SW_VBIAS = offsetof(msoc_env_state, vbias) / 4, SW_RET = offsetof(msoc_env_state, ep_return) / 4,
    SW_STEPS = offsetof(msoc_env_state, steps) / 4, SW_SCORE = offsetof(msoc_env_state, score) / 4,
    SW_MODE = offsetof(msoc_env_state, mode) / 4, SW_SPAWN = offsetof(msoc_env_state, spawn_count) / 4,
    SW_CCOUNT = offsetof(msoc_env_state, cache_count) / 4, SW_SEED = offsetof(msoc_env_state, seed) / 4,
    SW_CINFO = offsetof(msoc_env_state, cache_info) / 4, SW_HVALID = offsetof(msoc_env_state, hist_valid) / 4,
    SW_HPOS = offsetof(msoc_env_state, hist_pos) / 4, SW_HVEL = offsetof(msoc_env_state, hist_vel) / 4,
    SW_HANG = offsetof(msoc_env_state, hist_ang) / 4, SW_HANGVEL = offsetof(msoc_env_state, hist_angvel) / 4,
};
/* the bias block (4 float4 per env in Arrays::bias: vbias of the five bodies, then wbias) is words SW_VBIAS.. in order */
static_assert(offsetof(msoc_env_state, wbias) == offsetof(msoc_env_state, vbias) + 40 && offsetof(msoc_env_state, cache_jn) == offsetof(msoc_env_state, cache_info) + 128,
              "msoc_env_state layout");

struct StateParams {
    Arrays A;
    const int *ctl;
    const int64_t *idx; /* n env indices or null: envs 0..n-1 */
    int64_t n;
    uint8_t *states;    /* n x 808 bytes, 16-byte aligned */
};

/* the group of entries [t0, t0 + count) between global and shared memory, 16-byte accesses (8 at an odd-count end) */
__device__ __forceinline__ void group_store(uint8_t *g, const uint32_t *s, int count, int lane)
{
    const int valid = count * (int)sizeof(msoc_env_state);
    const uint4 *s4 = reinterpret_cast<const uint4 *>(s);
#pragma unroll
    for (int i = 0; i < (STATE_GROUP_U4 + 31) / 32; i++) {
        const int k = i * 32 + lane, off = k * 16;
        if (off + 16 <= valid) reinterpret_cast<uint4 *>(g)[k] = s4[k];
        else if (off < valid) reinterpret_cast<uint2 *>(g + off)[0] = reinterpret_cast<const uint2 *>(s4 + k)[0];
    }
}
__device__ __forceinline__ void group_load(uint32_t *s, const uint8_t *g, int count, int lane)
{
    const int valid = count * (int)sizeof(msoc_env_state);
    uint4 *s4 = reinterpret_cast<uint4 *>(s);
#pragma unroll
    for (int i = 0; i < (STATE_GROUP_U4 + 31) / 32; i++) {
        const int k = i * 32 + lane, off = k * 16;
        if (off + 16 <= valid) s4[k] = __ldcs(reinterpret_cast<const uint4 *>(g) + k);
        else if (off < valid) reinterpret_cast<uint2 *>(s4 + k)[0] = __ldcs(reinterpret_cast<const uint2 *>(g + off));
    }
}

/* the state's float4 f of a record (store_env_record order) -> its words of msoc_env_state */
__device__ __forceinline__ void put_state_f4(uint32_t *w, int f, float4 v)
{
    if (f < 5) {
        w[SW_POS + 2 * f] = __float_as_uint(v.x); w[SW_POS + 2 * f + 1] = __float_as_uint(v.y);
        w[SW_VEL + 2 * f] = __float_as_uint(v.z); w[SW_VEL + 2 * f + 1] = __float_as_uint(v.w);
    } else if (f < 7) {
        const int o = f == 5 ? SW_ANG : SW_ANGVEL;
        w[o] = __float_as_uint(v.x); w[o + 1] = __float_as_uint(v.y); w[o + 2] = __float_as_uint(v.z); w[o + 3] = __float_as_uint(v.w);
    } else {
        const uint32_t flags = __float_as_uint(v.z);
        w[SW_ANGVEL + 4] = __float_as_uint(v.x); w[SW_STEPS] = __float_as_uint(v.y); w[SW_RET] = __float_as_uint(v.w);
        w[SW_MODE] = (flags & FLAG_MODE_MASK) >> FLAG_MODE_SHIFT; w[SW_CCOUNT] = flags & FLAG_CACHE_MASK;
    }
}
/* float4 f < 7 of a record -> history pose k (what a frame is made of: the ball velocity r[4].zw is not part of it) */
__device__ __forceinline__ void put_hist_f4(uint32_t *w, int k, int f, float4 v)
{
    if (f < 5) {
        w[SW_HPOS + 10 * k + 2 * f] = __float_as_uint(v.x); w[SW_HPOS + 10 * k + 2 * f + 1] = __float_as_uint(v.y);
        if (f < 4) { w[SW_HVEL + 8 * k + 2 * f] = __float_as_uint(v.z); w[SW_HVEL + 8 * k + 2 * f + 1] = __float_as_uint(v.w); }
    } else {
        const int o = (f == 5 ? SW_HANG : SW_HANGVEL) + 4 * k;
        w[o] = __float_as_uint(v.x); w[o + 1] = __float_as_uint(v.y); w[o + 2] = __float_as_uint(v.z); w[o + 3] = __float_as_uint(v.w);
    }
}
/* Angles: kept bit for bit when |a| <= float(pi) (the threshold of msoc_set_state's host wrap), otherwise wrapped with
   the step's own range reduction -- which may differ in the last bit from the host's double-precision atan2 wrap. */
__device__ __forceinline__ float state_angle(uint32_t bits)
{
    const float a = __uint_as_float(bits);
    return (a > PI_F || a < -PI_F) ? wrap_angle(a) : a;
}
/* float4 f of the record of the state in w (store_env_record order; the flags word is the caller's) */
__device__ __forceinline__ float4 get_state_f4(const uint32_t *w, int f, uint32_t flags)
{
    if (f < 5) return make_float4(__uint_as_float(w[SW_POS + 2 * f]), __uint_as_float(w[SW_POS + 2 * f + 1]),
                                  __uint_as_float(w[SW_VEL + 2 * f]), __uint_as_float(w[SW_VEL + 2 * f + 1]));
    if (f == 5) return make_float4(state_angle(w[SW_ANG]), state_angle(w[SW_ANG + 1]), state_angle(w[SW_ANG + 2]), state_angle(w[SW_ANG + 3]));
    if (f == 6) return make_float4(__uint_as_float(w[SW_ANGVEL]), __uint_as_float(w[SW_ANGVEL + 1]), __uint_as_float(w[SW_ANGVEL + 2]), __uint_as_float(w[SW_ANGVEL + 3]));
    return make_float4(__uint_as_float(w[SW_ANGVEL + 4]), __uint_as_float(w[SW_STEPS]), __uint_as_float(flags), __uint_as_float(w[SW_RET]));
}
/* float4 f < 7 of the record of history pose k (pose_pack order, ball velocity 0) */
__device__ __forceinline__ float4 get_hist_f4(const uint32_t *w, int k, int f)
{
    if (f < 4) return make_float4(__uint_as_float(w[SW_HPOS + 10 * k + 2 * f]), __uint_as_float(w[SW_HPOS + 10 * k + 2 * f + 1]),
                                  __uint_as_float(w[SW_HVEL + 8 * k + 2 * f]), __uint_as_float(w[SW_HVEL + 8 * k + 2 * f + 1]));
    if (f == 4) return make_float4(__uint_as_float(w[SW_HPOS + 10 * k + 8]), __uint_as_float(w[SW_HPOS + 10 * k + 9]), 0.0f, 0.0f);
    const int o = SW_HANG + 4 * k;
    if (f == 5) return make_float4(state_angle(w[o]), state_angle(w[o + 1]), state_angle(w[o + 2]), state_angle(w[o + 3]));
    const int p = SW_HANGVEL + 4 * k;
    return make_float4(__uint_as_float(w[p]), __uint_as_float(w[p + 1]), __uint_as_float(w[p + 2]), __uint_as_float(w[p + 3]));
}
/* same bits in the part of float4 f that a frame is made of */
__device__ __forceinline__ bool same_pose_f4(int f, float4 a, float4 b)
{
    bool same = __float_as_uint(a.x) == __float_as_uint(b.x) && __float_as_uint(a.y) == __float_as_uint(b.y);
    if (f != 4) same = same && __float_as_uint(a.z) == __float_as_uint(b.z) && __float_as_uint(a.w) == __float_as_uint(b.w);
    return same;
}
/* group index and validity of the env of lane group el */
__device__ __forceinline__ int64_t state_env(const StateParams &P, int64_t t, bool &ok)
{
    const int64_t e = P.idx != nullptr ? P.idx[t] : t;
    ok = e >= 0 && e < P.A.n;
    MSOC_CHECK(P.idx != nullptr || ok, CHK_STATES);
    return e;
}

/* Save: the bytes msoc_get_state returns -- the state (the injected record of a flagged env), the pose of the oldest
   record as history 0 and the current record as history 1 (hist_valid = 1), cache entries, zeros after cache_count;
   an out-of-range index gives an all-zero entry. */
__global__ void __launch_bounds__(STATE_BLOCK) msoc_save_states_kernel(const __grid_constant__ StateParams P)
{
    __shared__ __align__(16) uint32_t s_stage[STATE_BLOCK / 32][STATE_ENVS * STATE_WORDS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, el = lane >> 2, q = lane & 3;
    const int64_t t0 = ((int64_t)blockIdx.x * (STATE_BLOCK / 32) + warp) * STATE_ENVS;
    if (t0 >= P.n) return; /* warp-uniform */
    const int count = P.n - t0 < STATE_ENVS ? (int)(P.n - t0) : STATE_ENVS;
    uint32_t *stage = s_stage[warp];
    const int step = P.ctl[CTL_STEP_FAST];
    MSOC_CHECK(step >= 0 && step < 6, CHK_STATES);
    bool ok = false;
    const int64_t e = el < count ? state_env(P, t0 + el, ok) : 0;
    const int f0 = q, f1 = q + 4;
    float4 c0 = make_float4(0.0f, 0.0f, 0.0f, 0.0f), c1 = c0, p0 = c0, p1 = c0;
    if (ok) {
        const float4 *cur = P.A.pose[buf_cur(step)] + e * POSE_F4, *prev = P.A.pose[buf_prev(step)] + e * POSE_F4;
        c0 = cur[f0]; c1 = cur[f1]; p0 = prev[f0];
        if (f1 < 7) p1 = prev[f1];
    }
    /* zero the staging area: out-of-range entries, the cache tail and the padding stay zero */
    uint4 *stage4 = reinterpret_cast<uint4 *>(stage);
#pragma unroll
    for (int i = 0; i < (STATE_GROUP_U4 + 31) / 32; i++)
        if (i * 32 + lane < STATE_GROUP_U4) stage4[i * 32 + lane] = make_uint4(0u, 0u, 0u, 0u);
    /* lane 4 el + 3 holds float4 7 of the env's current record: flags */
    const uint32_t cflags = __shfl_sync(0xffffffffu, __float_as_uint(c1.z), lane | 3);
    float4 s0 = c0, s1 = c1;
    if (ok && (cflags & FLAG_INJECT) != 0u && P.A.inject != nullptr) {
        const float4 *inj = P.A.inject + e * POSE_F4;
        s0 = inj[f0]; s1 = inj[f1];
    }
    const uint32_t flags = __shfl_sync(0xffffffffu, __float_as_uint(s1.z), lane | 3);
    __syncwarp();
    if (ok) {
        uint32_t *w = stage + el * STATE_WORDS;
        put_state_f4(w, f0, s0); put_state_f4(w, f1, s1);
        put_hist_f4(w, 0, f0, p0); put_hist_f4(w, 1, f0, c0);
        if (f1 < 7) { put_hist_f4(w, 0, f1, p1); put_hist_f4(w, 1, f1, c1); }
        if (q == 0) {
            const int2 sc = P.A.score[e];
            w[SW_SCORE] = (uint32_t)sc.x; w[SW_SCORE + 1] = (uint32_t)sc.y;
            w[SW_HVALID] = 1u;
        } else if (q == 1) {
            const uint64_t sd = P.A.seed[e];
            w[SW_SEED] = (uint32_t)sd; w[SW_SEED + 1] = (uint32_t)(sd >> 32);
            w[SW_SPAWN] = P.A.spawn_count[e];
        }
        if (flags & FLAG_HAS_BIAS) {
            const float4 b = P.A.bias[4 * e + q];
            w[SW_VBIAS + 4 * q] = __float_as_uint(b.x); w[SW_VBIAS + 4 * q + 1] = __float_as_uint(b.y);
            if (q < 3) { w[SW_VBIAS + 4 * q + 2] = __float_as_uint(b.z); w[SW_VBIAS + 4 * q + 3] = __float_as_uint(b.w); }
        }
        /* cache entries j < count: 3 words each, contiguous per env (cache_slot), read as 16-byte chunks */
        const uint32_t cnt = flags & FLAG_CACHE_MASK;
        MSOC_CHECK(cnt <= (uint32_t)MAX_CACHE, CHK_STATES);
        const int nw = 3 * (int)(cnt < (uint32_t)MAX_CACHE ? cnt : (uint32_t)MAX_CACHE);
        const uint4 *c4 = reinterpret_cast<const uint4 *>(P.A.cache[cache_half(step)] + cache_slot(e, 0));
        for (int c = q; 4 * c < nw; c += 4) {
            const uint4 v = c4[c];
            const uint32_t vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int i = 0; i < 4; i++) {
                const int word = 4 * c + i, j = word / 3;
                MSOC_CHECK(word >= nw || j < MAX_CACHE, CHK_STATES);
                if (word < nw) w[SW_CINFO + MAX_CACHE * (word - 3 * j) + j] = vv[i];
            }
        }
    }
    __syncwarp();
    MSOC_CHECK(t0 + count <= P.n, CHK_STATES);
    group_store(P.states + t0 * (int64_t)sizeof(msoc_env_state), stage, count, lane);
}

/* Load: what msoc_set_state did -- cache count clamped to MSOC_MAX_CACHE; hist_valid = 1 installs both history poses,
   hist_valid = 0 keeps the emitted ones; a state whose pose differs from the newest emitted one goes to Arrays::inject
   and its record is flagged FLAG_INJECT; the has-bias flag follows the bias values.  Out-of-range entries are skipped. */
__global__ void __launch_bounds__(STATE_BLOCK) msoc_load_states_kernel(const __grid_constant__ StateParams P)
{
    __shared__ __align__(16) uint32_t s_stage[STATE_BLOCK / 32][STATE_ENVS * STATE_WORDS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, el = lane >> 2, q = lane & 3;
    const int64_t t0 = ((int64_t)blockIdx.x * (STATE_BLOCK / 32) + warp) * STATE_ENVS;
    if (t0 >= P.n) return; /* warp-uniform */
    const int count = P.n - t0 < STATE_ENVS ? (int)(P.n - t0) : STATE_ENVS;
    uint32_t *stage = s_stage[warp];
    const int step = P.ctl[CTL_STEP_FAST];
    MSOC_CHECK(step >= 0 && step < 6, CHK_STATES);
    MSOC_CHECK(t0 + count <= P.n, CHK_STATES);
    group_load(stage, P.states + t0 * (int64_t)sizeof(msoc_env_state), count, lane);
    bool ok = false;
    const int64_t e = el < count ? state_env(P, t0 + el, ok) : 0;
    __syncwarp();
    const uint32_t *w = stage + el * STATE_WORDS;
    const int f0 = q, f1 = q + 4;
    const uint32_t hist_valid = w[SW_HVALID];
    /* the bias words of this lane's float4 of the bias block; any non-zero value in the env sets the has-bias flag */
    float4 b = make_float4(__uint_as_float(w[SW_VBIAS + 4 * q]), __uint_as_float(w[SW_VBIAS + 4 * q + 1]), 0.0f, 0.0f);
    if (q < 3) { b.z = __uint_as_float(w[SW_VBIAS + 4 * q + 2]); b.w = __uint_as_float(w[SW_VBIAS + 4 * q + 3]); }
    const bool my_bias = b.x != 0.0f || b.y != 0.0f || b.z != 0.0f || b.w != 0.0f;
    const uint32_t group = 0xfu << (lane & ~3);
    const bool any_bias = (__ballot_sync(0xffffffffu, ok && my_bias) & group) != 0u;
    const uint32_t ccount = w[SW_CCOUNT];
    const uint32_t cnt = ccount > (uint32_t)MAX_CACHE ? (uint32_t)MAX_CACHE : ccount;
    const uint32_t flags = cnt | ((w[SW_MODE] & 3u) << FLAG_MODE_SHIFT) | (any_bias ? FLAG_HAS_BIAS : 0u);
    const float4 n0 = get_state_f4(w, f0, flags), n1 = get_state_f4(w, f1, flags);
    float4 *rec = P.A.pose[buf_cur(step)] + (ok ? e : 0) * POSE_F4;
    /* the pose behind the newest emitted frame: the caller's history pose 1, or what the current record holds */
    float4 h0 = make_float4(0.0f, 0.0f, 0.0f, 0.0f), h1 = h0;
    if (ok) {
        if (hist_valid) { h0 = get_hist_f4(w, 1, f0); if (f1 < 7) h1 = get_hist_f4(w, 1, f1); }
        else { h0 = rec[f0]; if (f1 < 7) h1 = rec[f1]; }
    }
    const bool my_same = same_pose_f4(f0, h0, n0) && (f1 >= 7 || same_pose_f4(f1, h1, n1));
    const bool same = (__ballot_sync(0xffffffffu, !ok || my_same) & group) == group;
    if (!ok) return; /* no warp-wide operation follows */
    if (hist_valid) {
        float4 *prev = P.A.pose[buf_prev(step)] + e * POSE_F4;
        prev[f0] = get_hist_f4(w, 0, f0);
        if (f1 < 7) prev[f1] = get_hist_f4(w, 0, f1);
    }
    if (any_bias) P.A.bias[4 * e + q] = b;
    if (q == 0) P.A.score[e] = make_int2((int)w[SW_SCORE], (int)w[SW_SCORE + 1]);
    else if (q == 1) { P.A.seed[e] = (uint64_t)w[SW_SEED] | ((uint64_t)w[SW_SEED + 1] << 32); P.A.spawn_count[e] = w[SW_SPAWN]; }
    /* cache entries j < cnt of the current parity, as whole 16-byte chunks where the chunk lies inside them */
    const int nw = 3 * (int)cnt;
    uint32_t *cw = P.A.cache[cache_half(step)] + cache_slot(e, 0);
    for (int c = q; 4 * c < nw; c += 4) {
        uint32_t vv[4];
#pragma unroll
        for (int i = 0; i < 4; i++) { const int word = 4 * c + i, j = word / 3; vv[i] = word < nw ? w[SW_CINFO + MAX_CACHE * (word - 3 * j) + j] : 0u; }
        if (4 * c + 4 <= nw) reinterpret_cast<uint4 *>(cw)[c] = make_uint4(vv[0], vv[1], vv[2], vv[3]);
        else {
#pragma unroll
            for (int i = 0; i < 4; i++)
                if (4 * c + i < nw) cw[4 * c + i] = vv[i];
        }
    }
    if (same) {
        rec[f0] = n0; rec[f1] = n1;
    } else {
        float4 *inj = P.A.inject + e * POSE_F4;
        inj[f0] = n0; inj[f1] = n1;
        if (hist_valid) { rec[f0] = h0; if (f1 < 7) rec[f1] = h1; } /* otherwise the record already holds that pose */
        if (f1 == 7) rec[7] = make_float4(0.0f, n1.y, __uint_as_float(FLAG_INJECT), 0.0f);
    }
}

/* rows of the internal observation buffer of a list of envs, packed */
__global__ void msoc_gather_obs_kernel(const float *obs, const int64_t *idx, int64_t n, float *out)
{
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * 4 * OBS) return;
    const int64_t k = t / (4 * OBS);
    out[t] = obs[idx[k] * 4 * OBS + (t - k * 4 * OBS)];
}

__global__ void msoc_init_kernel(Arrays A, uint64_t seed)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= A.n) return;
    A.seed[e] = seed;
    A.spawn_count[e] = 0;
}

/* ------------------------------------------------------------------ rollout: policy inputs */
/* One pass over one team's observation rows (528 contiguous bytes per env): normalised + clipped bf16 policy input
   (padded rows), raw bf16 copy for the rollout buffer, per-feature sum / sum of squares for the running normaliser.
   Thread (x, y): float2 x of the 132 floats of env y (+ 4 per iteration), so a thread always sees the same two features.
   TEAM 0 reads rows 0, 1 (blue) as they are.  TEAM 1 reads rows 2, 3 (red) and first mirrors them about x = 400
   (include/msoc.h, msoc_team_inputs): a frame has an even length, so a thread's two features sit at the same even
   offset g of every frame it sees, and its mirror is two fixed sign flips plus, at g = 2, the angle map. */
constexpr int PI_X = 66, PI_Y = 4, PI_PAD = 72;
template <int TEAM>
__global__ void __launch_bounds__(PI_X * PI_Y) msoc_policy_inputs_kernel(const float *__restrict__ obs, int64_t n, const float *__restrict__ shift,
                                                                         const float *__restrict__ inv_std, __nv_bfloat162 *__restrict__ x_out,
                                                                         __nv_bfloat162 *__restrict__ raw_out, double *moments)
{
    __shared__ float s_red[PI_Y][PI_X][4];
    const int x = threadIdx.x, y = threadIdx.y;
    const int row = x >= 33 ? 1 : 0, f = 2 * x - 66 * row; /* features f, f + 1 of agent `row` */
    const float sh0 = shift[f], sh1 = shift[f + 1], is0 = inv_std[f], is1 = inv_std[f + 1];
    /* the mirror of features g, g + 1 of a frame: negated are the x components 0, 3 (omega), 4, 7, 10, 13, 16, 19 */
    const int g = f % FRAME;
    const uint32_t neg0 = (g == 0 || g == 4 || g == 10 || g == 16) ? 0x80000000u : 0u;
    const uint32_t neg1 = (g == 2 || g == 6 || g == 12 || g == 18) ? 0x80000000u : 0u;
    float s0 = 0.0f, s1 = 0.0f, q0 = 0.0f, q1 = 0.0f;
    for (int64_t e = (int64_t)blockIdx.x * PI_Y + y; e < n; e += (int64_t)gridDim.x * PI_Y) {
        float2 v = reinterpret_cast<const float2 *>(obs + e * (4 * OBS) + TEAM * (2 * OBS))[x];
        if (TEAM == 1) {
            v.x = g == 2 ? (v.x >= 0.0f ? 1.0f - v.x : -1.0f - v.x) : __uint_as_float(__float_as_uint(v.x) ^ neg0);
            v.y = __uint_as_float(__float_as_uint(v.y) ^ neg1);
        }
        const float a = fminf(fmaxf(fmaf(v.x, is0, sh0), -10.0f), 10.0f), b = fminf(fmaxf(fmaf(v.y, is1, sh1), -10.0f), 10.0f);
        x_out[((2 * e + row) * PI_PAD + f) >> 1] = __floats2bfloat162_rn(a, b);
        if (raw_out != nullptr) raw_out[(e * (2 * OBS) + 2 * x) >> 1] = __floats2bfloat162_rn(v.x, v.y);
        s0 += v.x; s1 += v.y; q0 = fmaf(v.x, v.x, q0); q1 = fmaf(v.y, v.y, q1);
    }
    if (moments == nullptr) return;
    s_red[y][x][0] = s0; s_red[y][x][1] = s1; s_red[y][x][2] = q0; s_red[y][x][3] = q1;
    __syncthreads();
    if (y == 0) {
        double t0 = 0.0, t1 = 0.0, u0 = 0.0, u1 = 0.0;
        for (int k = 0; k < PI_Y; k++) { t0 += s_red[k][x][0]; t1 += s_red[k][x][1]; u0 += s_red[k][x][2]; u1 += s_red[k][x][3]; }
        atomicAdd(moments + f, t0); atomicAdd(moments + f + 1, t1);
        atomicAdd(moments + OBS + f, u0); atomicAdd(moments + OBS + f + 1, u1);
    }
}

/* ------------------------------------------------------------------------------------ render */
/* RGB images of a list of envs (render_core.cuh).  The output is write-only: n H W 3 bytes against 96 bytes of record
   per env.  A block takes a tile of the flat pixel stream (a multiple of 32 pixels, at most RENDER_MAX_SPAN images):
   the scenes of the tile's images are set up once, in shared memory; then every thread colours 32-pixel segments, and
   each warp stages its 32 consecutive segments (3 072 contiguous bytes) in shared memory and writes them with
   coalesced 16-byte stores -- every output byte once, nothing read back. */
struct RenderParams {
    Arrays A;
    const int *ctl;
    const int64_t *idx; /* n env indices or null: envs 0..n-1 */
    uint8_t *out;       /* 16-byte aligned */
    int64_t total_px, tile_px, tiles;
    RenderGeom G;
};

__global__ void __launch_bounds__(RENDER_BLOCK) msoc_render_kernel(const __grid_constant__ RenderParams P)
{
    __shared__ RenderScene s_scene[RENDER_MAX_SPAN];
    __shared__ __align__(16) uint32_t s_stage[RENDER_BLOCK / 32][32 * RENDER_SEG_WORDS];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int step = P.ctl[CTL_STEP_FAST];
    const int64_t hw = (int64_t)P.G.H * P.G.W;
    uint32_t *stage = s_stage[warp];
#pragma unroll 1
    for (int64_t tile = blockIdx.x; tile < P.tiles; tile += gridDim.x) {
        const int64_t g_begin = tile * P.tile_px;
        const int64_t g_end = g_begin + P.tile_px < P.total_px ? g_begin + P.tile_px : P.total_px;
        const int64_t i0 = g_begin / hw;
        const int span = (int)((g_end - 1) / hw - i0 + 1);
        __syncthreads(); /* the previous tile's scenes are no longer read */
        for (int k = tid; k < span; k += RENDER_BLOCK) {
            const int64_t e = P.idx != nullptr ? P.idx[i0 + k] : i0 + k;
            const bool ok = e >= 0 && e < P.A.n;
            MSOC_CHECK(P.idx != nullptr || ok, CHK_RENDER);
            render_scene(P.G, ok ? render_record(P.A, step, e) : nullptr, s_scene[k]);
        }
        __syncthreads();
        const int base_off = (int)(g_begin - i0 * hw); /* pixel offset of the tile in image i0 */
#pragma unroll 1
        for (int s = 0; s < RENDER_SEGS_PER_THREAD; s++) {
            const int64_t warp_g0 = g_begin + (int64_t)(s * RENDER_BLOCK + warp * 32) * RENDER_SEG;
            if (warp_g0 >= g_end) break; /* warp-uniform */
            const int64_t g0 = warp_g0 + (int64_t)lane * RENDER_SEG;
            uint32_t w[RENDER_SEG_WORDS];
            if (g0 < g_end) {
                const int o = base_off + (int)(g0 - g_begin);
                const int img = o / (int)hw, rem = o - img * (int)hw;
                const int row = rem / P.G.W, col = rem - row * P.G.W;
                const int count = g_end - g0 < RENDER_SEG ? (int)(g_end - g0) : RENDER_SEG;
                uint32_t wm, bm, rm, ym, zm;
                render_segment_masks(P.G, s_scene, img, row, col, count, wm, bm, rm, ym, zm);
                render_pack(wm, bm, rm, ym, zm, w);
                uint4 *st4 = reinterpret_cast<uint4 *>(stage + lane * RENDER_SEG_WORDS);
#pragma unroll
                for (int i = 0; i < RENDER_SEG_WORDS / 4; i++) st4[i] = make_uint4(w[4 * i], w[4 * i + 1], w[4 * i + 2], w[4 * i + 3]);
            }
            __syncwarp();
            /* the warp's bytes [warp_g0 * 3, +3072) clipped to the tile (the rest belongs to the next tile's block, and
               the idle lanes staged nothing), as 16-byte stores, bytes at a ragged end */
            const int64_t byte0 = warp_g0 * 3;
            const int64_t valid = (g_end - warp_g0) * 3 < 32 * RENDER_SEG * 3 ? (g_end - warp_g0) * 3 : 32 * RENDER_SEG * 3;
            const uint4 *src = reinterpret_cast<const uint4 *>(stage);
#pragma unroll
            for (int i = 0; i < RENDER_SEG_WORDS / 4; i++) {
                const int off = (i * 32 + lane) * 16;
                if (off + 16 <= valid) {
                    MSOC_CHECK(byte0 + off + 16 <= P.total_px * 3, CHK_RENDER);
                    __stcs(reinterpret_cast<uint4 *>(P.out + byte0 + off), src[i * 32 + lane]);
                } else if (off < valid) {
                    const uint8_t *sb = reinterpret_cast<const uint8_t *>(src + i * 32 + lane);
                    for (int b = 0; b < valid - off; b++) P.out[byte0 + off + b] = sb[b];
                }
            }
            __syncwarp();
        }
    }
}

/* msoc_policy_inputs / msoc_team_inputs after their argument checks */
template <int TEAM>
static int launch_policy_inputs(const float *d_obs, int64_t n_envs, const float *d_shift, const float *d_inv_std, void *d_x_out,
                                void *d_raw_out, double *d_moments, void *stream)
{
    int dev = 0, sms = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int64_t want = (n_envs + PI_Y - 1) / PI_Y, cap = (int64_t)sms * 7; /* 7 blocks of 264 threads per SM; a thread sums n / (4 * grid) rows in fp32 */
    msoc_policy_inputs_kernel<TEAM><<<(unsigned)(want < cap ? want : cap), dim3(PI_X, PI_Y), 0, (cudaStream_t)stream>>>(
        d_obs, n_envs, d_shift, d_inv_std, (__nv_bfloat162 *)d_x_out, (__nv_bfloat162 *)d_raw_out, d_moments);
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    return MSOC_OK;
}

/* ---------------------------------------------------------------------------------- C-ABI */
extern "C" {

const char *msoc_last_error(void) { return g_last_error.c_str(); }
int msoc_version(void) { return MSOC_VERSION; }
uint64_t msoc_launch_count(void) { return g_launches.load(); }
/* Bits of the failed kernel checks since the last call (see MSOC_CHECK in step_core.cuh); -1 in a build without
   -DMSOC_CHECKS.  Synchronises the device. */
int msoc_debug_errors(void)
{
#ifdef MSOC_CHECKS
    unsigned int bits = 0, zero = 0;
    if (cudaDeviceSynchronize() != cudaSuccess) return -2;
    if (cudaMemcpyFromSymbol(&bits, g_msoc_check_bits, sizeof bits) != cudaSuccess) return -2;
    cudaMemcpyToSymbol(g_msoc_check_bits, &zero, sizeof zero);
    return (int)bits;
#else
    return -1;
#endif
}
int64_t msoc_num_envs(const msoc_handle *h) { return h ? h->n : 0; }

static size_t align_up(size_t x) { return (x + 255) & ~(size_t)255; }

static int grid_for(int64_t n) { return (int)((n + BLOCK - 1) / BLOCK); }

static void fill_cfg(const msoc_config *c, SimCfg &s)
{
    s.max_velocity = c->max_velocity;
    s.agent_minv = 1.0f / c->agent_mass; s.ball_minv = 1.0f / c->ball_mass;
    s.agent_iinv = 1.0f / c->agent_moment; s.ball_iinv = 1.0f / c->ball_moment;
    s.agent_friction = c->agent_friction; s.ball_friction = c->ball_friction;
    s.force_max = c->action_force_max; s.torque_max = c->action_torque_max;
    s.max_ang_vel = c->max_angular_velocity;
    s.prox_mult = c->ball_proximity_multiplier; s.move_mult = c->move_ball_to_goal_multiplier;
    s.goal_reward = c->goal_scored_reward; s.conceded_penalty = c->goal_conceded_penalty;
    s.alive_penalty = c->alive_penalty; s.score_diff_mult = c->score_difference_multiplier;
    s.max_steps = c->max_steps; s.pad = 0;
    cfg_derive(s);
}

int msoc_reset(msoc_handle *h, const uint8_t *d_mask, int mode, int has_seed, uint64_t seed, float *d_obs_out, void *stream);
int msoc_destroy(msoc_handle *h);

int msoc_create(const msoc_config *cfg, int64_t n_envs, int device, uint64_t seed, uint64_t global_env_offset,
                msoc_handle **out)
{
    if (!cfg || !out || n_envs <= 0) return fail(MSOC_ERR_INVALID, "msoc_create: bad argument");
    if (n_envs > 0x7fffffff) return fail(MSOC_ERR_INVALID, "msoc_create: at most 2^31 - 1 envs per handle");
    if (!(cfg->agent_mass > 0.0f) || !(cfg->ball_mass > 0.0f) || !(cfg->agent_moment > 0.0f) || !(cfg->ball_moment > 0.0f))
        return fail(MSOC_ERR_INVALID, "msoc_create: masses and moments must be positive");
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev <= 0)
        return fail(MSOC_ERR_CUDA, "msoc_create: no CUDA device (this library has no CPU fallback)", ce);
    if (device < 0 || device >= ndev) return fail(MSOC_ERR_INVALID, "msoc_create: bad device index");
    DeviceGuard guard(device);

    msoc_handle *h = new msoc_handle();
    memset(h, 0, sizeof *h);
    h->device = device; h->n = n_envs; h->global_offset = global_env_offset;
    fill_cfg(cfg, h->cfg);
    if (const char *hl = getenv("MSOC_HEAVY_LANES")) {
        const int v = atoi(hl);
        if (v == 1 || v == 2 || v == 4 || v == 8 || v == 16 || v == 32) h->heavy_lanes_override = v;
    }
    /* every failure below goes through msoc_destroy, which releases whatever exists so far */
    auto bail = [&](int code, const char *what, cudaError_t e) { msoc_destroy(h); return fail(code, what, e); };

    const size_t n = (size_t)n_envs;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += align_up(bytes); return o; };
    size_t o_pose[3], o_cache[2];
    for (int k = 0; k < 3; k++) o_pose[k] = take(n * POSE_F4 * sizeof(float4));
    const size_t o_iscore = take(n * sizeof(int2));
    const size_t o_bias = take(n * 4 * sizeof(float4));
    const size_t o_seed = take(n * sizeof(uint64_t)), o_sc = take(n * sizeof(uint32_t));
    for (int k = 0; k < 2; k++) o_cache[k] = take(n * MAX_CACHE * 3 * sizeof(uint32_t));
    const size_t o_obs = take(n * 4 * OBS * sizeof(float)), o_act = take(n * 12 * sizeof(float));
    const size_t o_rew = take(n * 2 * sizeof(float)), o_done = take(n), o_goal = take(n), o_mask = take(n);
    const size_t o_score = take(n * 2 * sizeof(int32_t));
    const size_t o_stats = take(8 * sizeof(double));
    const size_t o_ctl = take(CTL_TOTAL * sizeof(int));
    const size_t o_list = take(n * sizeof(int)), o_list2 = take(n * sizeof(int));
    const size_t total = off;

    ce = cudaMalloc(&h->slab, total);
    if (ce != cudaSuccess) return bail(MSOC_ERR_ALLOC, "msoc_create: cudaMalloc", ce);
    ce = cudaMemset(h->slab, 0, total);
    if (ce != cudaSuccess) return bail(MSOC_ERR_CUDA, "msoc_create: cudaMemset", ce);
    char *base = (char *)h->slab;
    Arrays &A = h->A;
    A.n = n_envs;
    for (int k = 0; k < 3; k++) A.pose[k] = (float4 *)(base + o_pose[k]);
    for (int k = 0; k < 2; k++) A.cache[k] = (uint32_t *)(base + o_cache[k]);
    A.score = (int2 *)(base + o_iscore);
    A.bias = (float4 *)(base + o_bias);
    A.inject = nullptr;
    A.seed = (uint64_t *)(base + o_seed); A.spawn_count = (uint32_t *)(base + o_sc);
    h->d_obs = (float *)(base + o_obs); h->d_act = (float *)(base + o_act); h->d_rew = (float *)(base + o_rew);
    h->d_done = (uint8_t *)(base + o_done); h->d_goal = (int8_t *)(base + o_goal); h->d_mask = (uint8_t *)(base + o_mask);
    h->d_score = (int32_t *)(base + o_score);
    h->d_stats = (double *)(base + o_stats);
    h->d_ctl = (int *)(base + o_ctl);
    h->d_list = (int *)(base + o_list); h->d_list2 = (int *)(base + o_list2);

    ce = cudaFuncSetAttribute(msoc_step_contact_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)STEP_SMEM_BYTES);
    if (ce == cudaSuccess)
        ce = cudaFuncSetAttribute(msoc_step_fast_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FAST_SMEM_BYTES);
    if (ce == cudaSuccess)
        ce = cudaFuncSetAttribute(msoc_step_contact_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)STEP_SMEM_BYTES);
    if (ce == cudaSuccess)
        ce = cudaFuncSetAttribute(msoc_step_fast_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FAST_SMEM_BYTES);
    if (ce != cudaSuccess) return bail(MSOC_ERR_CUDA, "msoc_create: smem attribute", ce);
    cudaDeviceGetAttribute(&h->sm_count, cudaDevAttrMultiProcessorCount, device);
    ce = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&h->blocks_per_sm, msoc_step_contact_kernel<false>, HEAVY_BLOCK, STEP_SMEM_BYTES);
    if (ce == cudaSuccess)
        ce = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&h->blocks_per_sm_teams, msoc_step_contact_kernel<true>, HEAVY_BLOCK, STEP_SMEM_BYTES);
    if (ce != cudaSuccess || h->blocks_per_sm < 1 || h->blocks_per_sm_teams < 1 || h->sm_count < 1)
        return bail(MSOC_ERR_CUDA, "msoc_create: occupancy query", ce);
    if (ce == cudaSuccess) ce = cudaStreamCreateWithFlags(&h->pipe_stream, cudaStreamNonBlocking);
    if (ce == cudaSuccess) ce = cudaEventCreateWithFlags(&h->ev_pipe_fork, cudaEventDisableTiming);
    if (ce == cudaSuccess) ce = cudaEventCreateWithFlags(&h->ev_pipe_join, cudaEventDisableTiming);
    if (ce != cudaSuccess) return bail(MSOC_ERR_CUDA, "msoc_create: stream/event", ce);
    msoc_init_kernel<<<(unsigned)((n_envs + 255) / 256), 256>>>(A, seed);
    g_launches++;
    /* Game.__init__ -> setup_field -> reset(): first spawn in the default random mode */
    int rc = msoc_reset(h, nullptr, MSOC_MODE_RANDOM, 0, 0, h->d_obs, nullptr);
    if (rc != MSOC_OK) { msoc_destroy(h); return rc; }
    ce = cudaDeviceSynchronize();
    if (ce != cudaSuccess) return bail(MSOC_ERR_CUDA, "msoc_create: init", ce);
    *out = h;
    return MSOC_OK;
}

int msoc_destroy(msoc_handle *h)
{
    if (!h) return MSOC_OK;
    DeviceGuard guard(h->device);
    cudaDeviceSynchronize();
    if (h->d_stage) cudaFree(h->d_stage);
    if (h->d_frames) cudaFree(h->d_frames);
    if (h->d_inject) cudaFree(h->d_inject);
    if (h->ev_pipe_fork) cudaEventDestroy(h->ev_pipe_fork);
    if (h->ev_pipe_join) cudaEventDestroy(h->ev_pipe_join);
    if (h->pipe_stream) cudaStreamDestroy(h->pipe_stream);
    if (h->slab) cudaFree(h->slab);
    delete h;
    return MSOC_OK;
}

int msoc_reset(msoc_handle *h, const uint8_t *d_mask, int mode, int has_seed, uint64_t seed, float *d_obs_out, void *stream)
{
    if (!h) return fail(MSOC_ERR_INVALID, "msoc_reset: null handle");
    if (mode < 0 || mode > 2) return fail(MSOC_ERR_INVALID, "msoc_reset: bad mode");
    DeviceGuard guard(h->device);
    ResetParams P;
    P.A = h->A; P.cfg = h->cfg; P.mask = d_mask; P.obs_out = d_obs_out; P.ctl = h->d_ctl;
    P.global_offset = h->global_offset; P.seed = seed; P.mode = mode; P.has_seed = has_seed;
    msoc_reset_kernel<<<grid_for(h->n), BLOCK, 0, (cudaStream_t)stream>>>(P);
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    return MSOC_OK;
}

/* the two launches of one step over the envs [e0, e1), both on `st` */
static int launch_step(msoc_handle *h, StepParams &P, int64_t e0, int64_t e1, int chunk, cudaStream_t st, bool teams = false)
{
    P.e0 = e0; P.e1 = e1; P.chunk = chunk;
    const int64_t m = e1 - e0;
    P.heavy_lanes = h->heavy_lanes_override; /* 0: the contact kernel chooses by the number of heavy envs */
    /* Both kernels are launched programmatically dependent on whatever kernel precedes them in the stream: their grids
       are set up while that kernel drains and their blocks wait in cudaGridDependencySynchronize() until it is complete
       (a few microseconds of launch latency per step, which is what small batches are made of). */
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t lf = {};
    lf.gridDim = dim3((unsigned)((m + FAST_BLOCK - 1) / FAST_BLOCK));
    lf.blockDim = dim3(FAST_BLOCK);
    lf.dynamicSmemBytes = FAST_SMEM_BYTES;
    lf.stream = st;
    lf.attrs = at; lf.numAttrs = 1;
    CUDA_TRY(cudaLaunchKernelEx(&lf, teams ? msoc_step_fast_kernel<true> : msoc_step_fast_kernel<false>, P));
    g_launches++;
    /* one persistent grid for all contact classes, right behind the streaming kernel */
    const int64_t resident = (int64_t)h->sm_count * (teams ? h->blocks_per_sm_teams : h->blocks_per_sm);
    const int64_t blocks_max = (m + HEAVY_BLOCK - 1) / HEAVY_BLOCK;
    cudaLaunchConfig_t lc = {};
    lc.gridDim = dim3((unsigned)(blocks_max < resident ? blocks_max : resident));
    lc.blockDim = dim3(HEAVY_BLOCK);
    lc.dynamicSmemBytes = STEP_SMEM_BYTES;
    lc.stream = st;
    lc.attrs = at; lc.numAttrs = 1;
    CUDA_TRY(cudaLaunchKernelEx(&lc, teams ? msoc_step_contact_kernel<true> : msoc_step_contact_kernel<false>, P));
    g_launches++;
    return MSOC_OK;
}

static void fill_step_params(msoc_handle *h, StepParams &P, const float *d_actions, float *d_obs_out, float *d_frames_out,
                             float *d_reward, uint8_t *d_done, int8_t *d_goal, int32_t *d_score, uint32_t flags)
{
    P.A = h->A; P.cfg = h->cfg; P.actions = d_actions; P.obs_out = d_obs_out; P.frames_out = d_frames_out;
    P.reward = d_reward; P.done = d_done; P.goal = d_goal; P.score = d_score; P.stats = h->d_stats;
    P.global_offset = h->global_offset; P.flags = flags;
    P.ctl = h->d_ctl; P.list = h->d_list; P.list2 = h->d_list2;
}

int msoc_step(msoc_handle *h, const float *d_actions, float *d_obs_out, float *d_reward,
              uint8_t *d_done, int8_t *d_goal, int32_t *d_score, uint32_t flags, void *stream)
{
    if (!h || !d_actions || !d_obs_out || !d_reward || !d_done || !d_goal)
        return fail(MSOC_ERR_INVALID, "msoc_step: null argument");
    DeviceGuard guard(h->device);
    StepParams P;
    fill_step_params(h, P, d_actions, d_obs_out, nullptr, d_reward, d_done, d_goal, d_score, flags);
    return launch_step(h, P, 0, h->n, -1, (cudaStream_t)stream);
}

int msoc_step_teams(msoc_handle *h, const float *d_actions, float *d_obs_out, float *d_reward,
                    uint8_t *d_done, int8_t *d_goal, int32_t *d_score, uint32_t flags, void *stream)
{
    if (!h || !d_actions || !d_obs_out || !d_reward || !d_done || !d_goal)
        return fail(MSOC_ERR_INVALID, "msoc_step_teams: null argument");
    if ((uintptr_t)d_reward & 15u) return fail(MSOC_ERR_INVALID, "msoc_step_teams: d_reward must be 16-byte aligned");
    DeviceGuard guard(h->device);
    StepParams P;
    fill_step_params(h, P, d_actions, d_obs_out, nullptr, d_reward, d_done, d_goal, d_score, flags);
    return launch_step(h, P, 0, h->n, -1, (cudaStream_t)stream, true);
}

/* Host-buffer step: the envs are cut into chunks that alternate between two stream lanes, so that the H2D copy and the
   kernels of one chunk run while the D2H copies of the previous one are still on the wire. */
static int step_host_impl(msoc_handle *h, const float *h_actions, float *h_obs, float *h_frames, float *h_reward, uint8_t *h_done,
                          int8_t *h_goal, int32_t *h_score, uint32_t flags, void *stream)
{
    if (!h || !h_actions) return fail(MSOC_ERR_INVALID, "msoc_step_host: null argument");
    DeviceGuard guard(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (h_frames && !h->d_frames) {
        cudaError_t ce = cudaMalloc(&h->d_frames, (size_t)h->n * 4 * FRAME * sizeof(float));
        if (ce != cudaSuccess) return fail(MSOC_ERR_ALLOC, "msoc_step_host_frames: cudaMalloc", ce);
    }
    StepParams P;
    fill_step_params(h, P, h->d_act, h->d_obs, h_frames ? h->d_frames : nullptr, h->d_rew, h->d_done, h->d_goal, h->d_score, flags);
    /* chunks of at least 64 Ki envs, at most MAX_CHUNKS */
    int chunks = (int)(h->n / 65536);
    if (chunks < 1) chunks = 1;
    if (chunks > MAX_CHUNKS) chunks = MAX_CHUNKS;
    const int64_t per = ((h->n + chunks - 1) / chunks + 127) & ~(int64_t)127;
    auto copies_back = [&](int64_t e0, int64_t m, cudaStream_t s) -> int {
        if (h_obs) CUDA_TRY(cudaMemcpyAsync(h_obs + e0 * 4 * OBS, h->d_obs + e0 * 4 * OBS, (size_t)m * 4 * OBS * sizeof(float), cudaMemcpyDeviceToHost, s));
        if (h_frames) CUDA_TRY(cudaMemcpyAsync(h_frames + e0 * 4 * FRAME, h->d_frames + e0 * 4 * FRAME, (size_t)m * 4 * FRAME * sizeof(float), cudaMemcpyDeviceToHost, s));
        if (h_reward) CUDA_TRY(cudaMemcpyAsync(h_reward + e0 * 2, h->d_rew + e0 * 2, (size_t)m * 2 * sizeof(float), cudaMemcpyDeviceToHost, s));
        if (h_done) CUDA_TRY(cudaMemcpyAsync(h_done + e0, h->d_done + e0, (size_t)m, cudaMemcpyDeviceToHost, s));
        if (h_goal) CUDA_TRY(cudaMemcpyAsync(h_goal + e0, h->d_goal + e0, (size_t)m, cudaMemcpyDeviceToHost, s));
        if (h_score) CUDA_TRY(cudaMemcpyAsync(h_score + e0 * 2, h->d_score + e0 * 2, (size_t)m * 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
        return MSOC_OK;
    };
    if (chunks == 1) {
        CUDA_TRY(cudaMemcpyAsync(h->d_act, h_actions, (size_t)h->n * 12 * sizeof(float), cudaMemcpyHostToDevice, st));
        int rc = launch_step(h, P, 0, h->n, -1, st);
        if (rc != MSOC_OK) return rc;
        rc = copies_back(0, h->n, st);
        if (rc != MSOC_OK) return rc;
        CUDA_TRY(cudaStreamSynchronize(st));
        return MSOC_OK;
    }
    CUDA_TRY(cudaMemsetAsync(h->d_ctl + CTL_CHUNK0, 0, CTL_WORDS * MAX_CHUNKS * sizeof(int), st));
    /* A whole step expects the list counters of its parity to be zero: the streaming kernel of the previous whole step
       clears them, and the chunks of this step do not.  Clear both sets, so that a device step or a graph replay may
       follow on the same handle.  (Words 16.. hold the step counters and the last class counts.) */
    CUDA_TRY(cudaMemsetAsync(h->d_ctl, 0, 2 * CTL_WORDS * sizeof(int), st));
    CUDA_TRY(cudaEventRecord(h->ev_pipe_fork, st));
    CUDA_TRY(cudaStreamWaitEvent(h->pipe_stream, h->ev_pipe_fork, 0));
    for (int c = 0; c < chunks; c++) {
        const int64_t e0 = c * per, e1 = (e0 + per < h->n) ? e0 + per : h->n;
        if (e0 >= e1) break;
        cudaStream_t s = (c & 1) ? h->pipe_stream : st;
        CUDA_TRY(cudaMemcpyAsync(h->d_act + e0 * 12, h_actions + e0 * 12, (size_t)(e1 - e0) * 12 * sizeof(float), cudaMemcpyHostToDevice, s));
        int rc = launch_step(h, P, e0, e1, c, s);
        if (rc != MSOC_OK) return rc;
        rc = copies_back(e0, e1 - e0, s);
        if (rc != MSOC_OK) return rc;
    }
    CUDA_TRY(cudaEventRecord(h->ev_pipe_join, h->pipe_stream));
    CUDA_TRY(cudaStreamWaitEvent(st, h->ev_pipe_join, 0));
    msoc_advance_kernel<<<1, 32, 0, st>>>(h->d_ctl);
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaStreamSynchronize(st));
    return MSOC_OK;
}

int msoc_step_host(msoc_handle *h, const float *h_actions, float *h_obs, float *h_reward, uint8_t *h_done,
                   int8_t *h_goal, int32_t *h_score, uint32_t flags, void *stream)
{
    return step_host_impl(h, h_actions, h_obs, nullptr, h_reward, h_done, h_goal, h_score, flags, stream);
}

int msoc_step_host_frames(msoc_handle *h, const float *h_actions, float *h_frames, float *h_reward, uint8_t *h_done,
                          int8_t *h_goal, int32_t *h_score, uint32_t flags, void *stream)
{
    if (!h_frames) return fail(MSOC_ERR_INVALID, "msoc_step_host_frames: null frame buffer");
    return step_host_impl(h, h_actions, nullptr, h_frames, h_reward, h_done, h_goal, h_score, flags, stream);
}

int msoc_reset_host(msoc_handle *h, const uint8_t *h_mask, int mode, int has_seed, uint64_t seed, float *h_obs, void *stream)
{
    if (!h) return fail(MSOC_ERR_INVALID, "msoc_reset_host: null handle");
    DeviceGuard guard(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    const size_t n = (size_t)h->n;
    if (h_mask) CUDA_TRY(cudaMemcpyAsync(h->d_mask, h_mask, n, cudaMemcpyHostToDevice, st));
    int rc = msoc_reset(h, h_mask ? h->d_mask : nullptr, mode, has_seed, seed, h->d_obs, stream);
    if (rc != MSOC_OK) return rc;
    if (h_obs) CUDA_TRY(cudaMemcpyAsync(h_obs, h->d_obs, n * 4 * OBS * sizeof(float), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return MSOC_OK;
}

int msoc_read_counters(msoc_handle *h, int32_t *h_score, int32_t *h_steps, void *stream)
{
    if (!h) return fail(MSOC_ERR_INVALID, "msoc_read_counters: null handle");
    DeviceGuard guard(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    int step = 0;
    CUDA_TRY(cudaMemcpyAsync(&step, h->d_ctl + CTL_STEP_FAST, sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (h_steps) {
        std::vector<float4> tmp((size_t)h->n);
        CUDA_TRY(cudaMemcpy2DAsync(tmp.data(), sizeof(float4), h->A.pose[step % 3] + 7, POSE_F4 * sizeof(float4), sizeof(float4), (size_t)h->n, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        for (int64_t i = 0; i < h->n; i++) { int32_t v; memcpy(&v, &tmp[(size_t)i].y, 4); h_steps[i] = v; }
    }
    if (h_score) {
        CUDA_TRY(cudaMemcpyAsync(h_score, h->A.score, (size_t)h->n * sizeof(int2), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
    }
    return MSOC_OK;
}

static int ensure_stage(msoc_handle *h, size_t bytes)
{
    if (h->stage_bytes >= bytes) return MSOC_OK;
    if (h->d_stage) cudaFree(h->d_stage);
    h->d_stage = nullptr; h->stage_bytes = 0;
    cudaError_t ce = cudaMalloc(&h->d_stage, bytes);
    if (ce != cudaSuccess) return fail(MSOC_ERR_ALLOC, "state staging cudaMalloc", ce);
    h->stage_bytes = bytes;
    return MSOC_OK;
}

static int check_idx(const msoc_handle *h, const int64_t *idx, int64_t n, const char *who)
{
    if (!h || !idx || n <= 0) return fail(MSOC_ERR_INVALID, who);
    for (int64_t i = 0; i < n; i++)
        if (idx[i] < 0 || idx[i] >= h->n) return fail(MSOC_ERR_INVALID, "env index out of range");
    return MSOC_OK;
}

static int launch_states(msoc_handle *h, bool save, const int64_t *d_idx, int64_t n, void *d_states, cudaStream_t st)
{
    StateParams P;
    P.A = h->A; P.ctl = h->d_ctl; P.idx = d_idx; P.n = n; P.states = (uint8_t *)d_states;
    const int64_t envs_per_block = (STATE_BLOCK / 32) * STATE_ENVS;
    const unsigned grid = (unsigned)((n + envs_per_block - 1) / envs_per_block);
    if (save) msoc_save_states_kernel<<<grid, STATE_BLOCK, 0, st>>>(P);
    else msoc_load_states_kernel<<<grid, STATE_BLOCK, 0, st>>>(P);
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    return MSOC_OK;
}

/* Arrays::inject: records of injected states whose pose differs from the newest emitted frame's */
static int ensure_inject(msoc_handle *h, cudaStream_t st, const char *who)
{
    if (h->d_inject) return MSOC_OK;
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    CUDA_TRY(cudaStreamIsCapturing(st, &cs));
    if (cs != cudaStreamCaptureStatusNone)
        return fail(MSOC_ERR_INVALID, "msoc_load_states: the first load on a handle allocates and cannot be captured; load once before capturing");
    cudaError_t ce = cudaMalloc(&h->d_inject, (size_t)h->n * POSE_F4 * sizeof(float4));
    if (ce != cudaSuccess) return fail(MSOC_ERR_ALLOC, who, ce);
    h->A.inject = (float4 *)h->d_inject;
    return MSOC_OK;
}

int msoc_get_state(msoc_handle *h, const int64_t *h_idx, int64_t n, msoc_env_state *h_out)
{
    int rc = check_idx(h, h_idx, n, "msoc_get_state: bad argument");
    if (rc != MSOC_OK) return rc;
    if (!h_out) return fail(MSOC_ERR_INVALID, "msoc_get_state: null output");
    DeviceGuard guard(h->device);
    const size_t ib = align_up((size_t)n * sizeof(int64_t)), sb = (size_t)n * sizeof(msoc_env_state);
    rc = ensure_stage(h, ib + sb);
    if (rc != MSOC_OK) return rc;
    int64_t *d_idx = (int64_t *)h->d_stage;
    msoc_env_state *d_s = (msoc_env_state *)((char *)h->d_stage + ib);
    CUDA_TRY(cudaDeviceSynchronize());
    CUDA_TRY(cudaMemcpy(d_idx, h_idx, (size_t)n * sizeof(int64_t), cudaMemcpyHostToDevice));
    rc = launch_states(h, true, d_idx, n, d_s, nullptr);
    if (rc != MSOC_OK) return rc;
    CUDA_TRY(cudaMemcpy(h_out, d_s, sb, cudaMemcpyDeviceToHost));
    return MSOC_OK;
}

static float wrap_host(float x)
{
    double a = (double)x;
    if (a > 3.14159274101257324 || a < -3.14159274101257324) a = atan2(sin(a), cos(a));
    return (float)a;
}

int msoc_set_state(msoc_handle *h, const int64_t *h_idx, int64_t n, const msoc_env_state *h_in)
{
    int rc = check_idx(h, h_idx, n, "msoc_set_state: bad argument");
    if (rc != MSOC_OK) return rc;
    if (!h_in) return fail(MSOC_ERR_INVALID, "msoc_set_state: null input");
    DeviceGuard guard(h->device);
    CUDA_TRY(cudaDeviceSynchronize());
    rc = ensure_inject(h, nullptr, "msoc_set_state: cudaMalloc");
    if (rc != MSOC_OK) return rc;
    const size_t ib = align_up((size_t)n * sizeof(int64_t)), sb = (size_t)n * sizeof(msoc_env_state);
    rc = ensure_stage(h, ib + sb);
    if (rc != MSOC_OK) return rc;
    int64_t *d_idx = (int64_t *)h->d_stage;
    msoc_env_state *d_s = (msoc_env_state *)((char *)h->d_stage + ib);
    /* wrap angles on the host in double (the reference keeps them unwrapped) */
    std::vector<msoc_env_state> tmp(h_in, h_in + n);
    for (auto &S : tmp)
        for (int i = 0; i < 4; i++) {
            S.ang[i] = wrap_host(S.ang[i]);
            for (int k = 0; k < 2; k++) S.hist_ang[k][i] = wrap_host(S.hist_ang[k][i]);
        }
    CUDA_TRY(cudaMemcpy(d_idx, h_idx, (size_t)n * sizeof(int64_t), cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(d_s, tmp.data(), sb, cudaMemcpyHostToDevice));
    rc = launch_states(h, false, d_idx, n, d_s, nullptr);
    if (rc != MSOC_OK) return rc;
    CUDA_TRY(cudaDeviceSynchronize());
    return MSOC_OK;
}

static int check_states_args(const msoc_handle *h, const int64_t *d_idx, int64_t n, const void *d_states, const char *who)
{
    if (!h) return fail(MSOC_ERR_INVALID, who);
    if (n < 0) return fail(MSOC_ERR_INVALID, "states: negative count");
    if (n == 0) return MSOC_OK;
    if (!d_states || ((uintptr_t)d_states & 15u) != 0u) return fail(MSOC_ERR_INVALID, "states: the state array must be a 16-byte aligned device pointer");
    if (!d_idx && n > h->n) return fail(MSOC_ERR_INVALID, "states: more entries than envs");
    return MSOC_OK;
}

int msoc_save_states(msoc_handle *h, const int64_t *d_idx, int64_t n, msoc_env_state *d_out, void *stream)
{
    int rc = check_states_args(h, d_idx, n, d_out, "msoc_save_states: null handle");
    if (rc != MSOC_OK || n == 0) return rc;
    DeviceGuard guard(h->device);
    return launch_states(h, true, d_idx, n, d_out, (cudaStream_t)stream);
}

int msoc_load_states(msoc_handle *h, const int64_t *d_idx, int64_t n, const msoc_env_state *d_in, void *stream)
{
    int rc = check_states_args(h, d_idx, n, d_in, "msoc_load_states: null handle");
    if (rc != MSOC_OK || n == 0) return rc;
    DeviceGuard guard(h->device);
    rc = ensure_inject(h, (cudaStream_t)stream, "msoc_load_states: cudaMalloc");
    if (rc != MSOC_OK) return rc;
    return launch_states(h, false, d_idx, n, (void *)d_in, (cudaStream_t)stream);
}

int msoc_get_obs_host(msoc_handle *h, const int64_t *h_idx, int64_t n, float *h_obs)
{
    int rc = check_idx(h, h_idx, n, "msoc_get_obs_host: bad argument");
    if (rc != MSOC_OK) return rc;
    if (!h_obs) return fail(MSOC_ERR_INVALID, "msoc_get_obs_host: null output");
    DeviceGuard guard(h->device);
    const size_t ib = align_up((size_t)n * sizeof(int64_t)), ob = (size_t)n * 4 * OBS * sizeof(float);
    rc = ensure_stage(h, ib + ob);
    if (rc != MSOC_OK) return rc;
    int64_t *d_idx = (int64_t *)h->d_stage;
    float *d_o = (float *)((char *)h->d_stage + ib);
    CUDA_TRY(cudaDeviceSynchronize());
    CUDA_TRY(cudaMemcpy(d_idx, h_idx, (size_t)n * sizeof(int64_t), cudaMemcpyHostToDevice));
    msoc_gather_obs_kernel<<<(unsigned)((n * 4 * OBS + 255) / 256), 256>>>(h->d_obs, d_idx, n, d_o);
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpy(h_obs, d_o, ob, cudaMemcpyDeviceToHost));
    return MSOC_OK;
}

static int check_render_args(const msoc_handle *h, int64_t n, int height, int width, const char *who)
{
    if (!h) return fail(MSOC_ERR_INVALID, who);
    if (n < 0) return fail(MSOC_ERR_INVALID, "render: negative image count");
    if (height < 1 || height > RENDER_MAX_SIDE || width < 1 || width > RENDER_MAX_SIDE)
        return fail(MSOC_ERR_INVALID, "render: height and width must be in [1, 4096]");
    return MSOC_OK;
}

static int launch_render(msoc_handle *h, const int64_t *d_idx, int64_t n, int height, int width, uint8_t *d_out, cudaStream_t st)
{
    RenderParams P;
    P.A = h->A; P.ctl = h->d_ctl; P.idx = d_idx; P.out = d_out;
    render_geom(height, width, P.G);
    P.total_px = n * height * width;
    P.tile_px = render_tile_px((int64_t)height * width);
    P.tiles = (P.total_px + P.tile_px - 1) / P.tile_px;
    const int64_t grid_cap = (int64_t)h->sm_count * 64; /* tiles beyond that are taken grid-stride */
    msoc_render_kernel<<<(unsigned)(P.tiles < grid_cap ? P.tiles : grid_cap), RENDER_BLOCK, 0, st>>>(P);
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    return MSOC_OK;
}

int msoc_render(msoc_handle *h, const int64_t *d_idx, int64_t n, int height, int width, uint8_t *d_out, void *stream)
{
    int rc = check_render_args(h, n, height, width, "msoc_render: null handle");
    if (rc != MSOC_OK || n == 0) return rc;
    if (!d_out || ((uintptr_t)d_out & 15u) != 0u) return fail(MSOC_ERR_INVALID, "msoc_render: output must be a 16-byte aligned device pointer");
    if (!d_idx && n > h->n) return fail(MSOC_ERR_INVALID, "msoc_render: more images than envs");
    DeviceGuard guard(h->device);
    return launch_render(h, d_idx, n, height, width, d_out, (cudaStream_t)stream);
}

int msoc_render_host(msoc_handle *h, const int64_t *h_idx, int64_t n, int height, int width, uint8_t *h_out)
{
    int rc = check_render_args(h, n, height, width, "msoc_render_host: null handle");
    if (rc != MSOC_OK || n == 0) return rc;
    if (!h_out) return fail(MSOC_ERR_INVALID, "msoc_render_host: null output");
    if (h_idx) {
        rc = check_idx(h, h_idx, n, "msoc_render_host: bad argument");
        if (rc != MSOC_OK) return rc;
    } else if (n > h->n) {
        return fail(MSOC_ERR_INVALID, "msoc_render_host: more images than envs");
    }
    DeviceGuard guard(h->device);
    const size_t ib = align_up((size_t)n * sizeof(int64_t)), ob = (size_t)n * height * width * 3;
    rc = ensure_stage(h, ib + ob);
    if (rc != MSOC_OK) return rc;
    int64_t *d_idx = h_idx ? (int64_t *)h->d_stage : nullptr;
    uint8_t *d_o = (uint8_t *)h->d_stage + ib;
    CUDA_TRY(cudaDeviceSynchronize());
    if (h_idx) CUDA_TRY(cudaMemcpy(d_idx, h_idx, (size_t)n * sizeof(int64_t), cudaMemcpyHostToDevice));
    rc = launch_render(h, d_idx, n, height, width, d_o, nullptr);
    if (rc != MSOC_OK) return rc;
    CUDA_TRY(cudaMemcpy(h_out, d_o, ob, cudaMemcpyDeviceToHost));
    return MSOC_OK;
}

int msoc_device_buffers(msoc_handle *h, msoc_buffers *out)
{
    if (!h || !out) return fail(MSOC_ERR_INVALID, "msoc_device_buffers: null argument");
    out->obs = h->d_obs; out->actions = h->d_act; out->reward = h->d_rew; out->done = h->d_done;
    out->goal = h->d_goal; out->score = h->d_score; out->mask = h->d_mask; out->stats = h->d_stats;
    return MSOC_OK;
}

int msoc_stats_device(msoc_handle *h, double *d_out, int reset, void *stream)
{
    if (!h || !d_out) return fail(MSOC_ERR_INVALID, "msoc_stats_device: null argument");
    DeviceGuard guard(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaMemcpyAsync(d_out, h->d_stats, 8 * sizeof(double), cudaMemcpyDeviceToDevice, st));
    if (reset) CUDA_TRY(cudaMemsetAsync(h->d_stats, 0, 8 * sizeof(double), st));
    return MSOC_OK;
}

int msoc_policy_inputs(const float *d_obs, int64_t n_envs, const float *d_shift, const float *d_inv_std, void *d_x_out,
                       void *d_raw_out, double *d_moments, void *stream)
{
    if (!d_obs || !d_shift || !d_inv_std || !d_x_out || n_envs <= 0) return fail(MSOC_ERR_INVALID, "msoc_policy_inputs: bad argument");
    return launch_policy_inputs<0>(d_obs, n_envs, d_shift, d_inv_std, d_x_out, d_raw_out, d_moments, stream);
}

int msoc_team_inputs(const float *d_obs, int64_t n_envs, int team, const float *d_shift, const float *d_inv_std,
                     void *d_x_out, void *d_raw_out, double *d_moments, void *stream)
{
    if (team != 0 && team != 1) return fail(MSOC_ERR_INVALID, "msoc_team_inputs: team must be 0 (blue) or 1 (red)");
    if (!d_obs || !d_shift || !d_inv_std || !d_x_out || n_envs <= 0) return fail(MSOC_ERR_INVALID, "msoc_team_inputs: bad argument");
    return team == 0 ? launch_policy_inputs<0>(d_obs, n_envs, d_shift, d_inv_std, d_x_out, d_raw_out, d_moments, stream)
                     : launch_policy_inputs<1>(d_obs, n_envs, d_shift, d_inv_std, d_x_out, d_raw_out, d_moments, stream);
}

int msoc_last_class_counts(msoc_handle *h, int32_t h_out[4], void *stream)
{
    if (!h || !h_out) return fail(MSOC_ERR_INVALID, "msoc_last_class_counts: null argument");
    DeviceGuard guard(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaMemcpyAsync(h_out, h->d_ctl + CTL_LAST_COUNTS, 4 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return MSOC_OK;
}

int msoc_stats_read(msoc_handle *h, msoc_stats *h_out, int reset, void *stream)
{
    if (!h || !h_out) return fail(MSOC_ERR_INVALID, "msoc_stats_read: null argument");
    DeviceGuard guard(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaMemcpyAsync(h_out, h->d_stats, 8 * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (reset) CUDA_TRY(cudaMemsetAsync(h->d_stats, 0, 8 * sizeof(double), st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return MSOC_OK;
}

} /* extern "C" */
