/*
 * msoc.h -- C-ABI of the B200-native batched 2v2 soccer simulator.
 *
 * The reference (sdace9719/marl-soccer) is pure Python and has NO FFI for this
 * path; its boundary is two duck-typed classes.  Each entry point below names
 * the reference interface it replaces (paths relative to the reference's
 * soccer_simulation/).  The Python host layer (marl_soccer_b200/soccer_env.py,
 * marl_vecenv.py) binds these with ctypes; INTEGRATION.md shows the stub.
 *
 * Conventions: every function returns 0 on success or a negative msoc_status;
 * msoc_last_error() describes the last failure on the calling thread.  All
 * `d_` pointers are DEVICE pointers on the handle's device, `h_` pointers are
 * HOST pointers.  `stream` is a cudaStream_t passed as void* (NULL = default
 * stream); calls are stream-ordered and asynchronous unless stated otherwise.
 * A handle is not re-entrant (the reference env is not thread-safe either).
 */
#ifndef MSOC_H
#define MSOC_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MSOC_VERSION 2
#define MSOC_N_AGENTS 4
#define MSOC_ACT_DIM 3
#define MSOC_FRAME 22   /* soccer_env.py:39 _frame_size */
#define MSOC_STACK 3    /* soccer_env.py:37 _stack_size */
#define MSOC_OBS 66
#define MSOC_MAX_CACHE 32 /* warm-start cache entries kept per env */

typedef enum {
    MSOC_OK = 0,
    MSOC_ERR_INVALID = -1, /* bad argument */
    MSOC_ERR_CUDA = -2,    /* CUDA runtime error, see msoc_last_error() */
    MSOC_ERR_ALLOC = -3
} msoc_status;

/* Spawn modes: game/game.py:109-114 */
#define MSOC_MODE_RANDOM 0      /* _apply_random_positions, game/game.py:154 */
#define MSOC_MODE_FIXED 1       /* _apply_fixed_positions, game/game.py:129 */
#define MSOC_MODE_FULL_RANDOM 2 /* _apply_full_random_positions, game/game.py:192 */

/* step flags */
#define MSOC_STEP_AUTO_RESET 1u /* marl_vecenv.py:45-53: reset finished envs in full-random mode */
#define MSOC_STEP_GENERAL_PATH 2u /* debugging / tests: every env that touches something goes through the general contact
                                     path (no light / pair / multi class); same simulation, slower */

/* config.json keys (config.json:1-22; readers: soccer_env.py:63-64, game/entities.py:11-17,62-67,
   game/game.py:27,262-264,330-372,430).  Absent keys take the reference's defaults in the
   Python layer before this struct is filled. */
typedef struct msoc_config {
    float max_velocity;
    float agent_mass, ball_mass;
    float agent_moment, ball_moment; /* literals 100 / 10 in game/entities.py:11,62 */
    float agent_friction, ball_friction;
    float action_force_max, action_torque_max;
    float max_angular_velocity;
    float ball_proximity_multiplier, move_ball_to_goal_multiplier;
    float goal_scored_reward, goal_conceded_penalty, alive_penalty, score_difference_multiplier;
    int32_t max_steps;
    int32_t reserved;
} msoc_config;

/* One env's complete simulator state, host side, for injection / extraction
   (parity tests, checkpointing, render pull-back of one env; replaces pymunk
   Body property access, e.g. game/game.py:131-152, :267-275).
   cache_info packs a warm-start entry: bits 0-5 pair id, 6-9 feature key, 10-11 age.
   Pair ids: agent i x segment s (setup_field order, game/game.py:50-68): i*8+s;
   agents i<j: 32+{01,02,03,12,13,23}; ball x agent i: 38+i; ball x wall s: 42+s. */
typedef struct msoc_env_state {
    float pos[5][2];   /* agent_0..3, ball */
    float vel[5][2];
    float ang[4];      /* agents; stored wrapped to [-pi, pi] */
    float angvel[5];
    float vbias[5][2]; /* Chipmunk v_bias carried to the next position update */
    float wbias[4];
    float ep_return;   /* running blue return of the current episode */
    int32_t steps;
    int32_t score[2];  /* blue, red */
    int32_t mode;
    uint32_t spawn_count;
    uint32_t cache_count;
    uint64_t seed;
    uint32_t cache_info[MSOC_MAX_CACHE];
    float cache_jn[MSOC_MAX_CACHE];
    float cache_jt[MSOC_MAX_CACHE];
    /* Observation history (the 3-frame deques of soccer_env.py:69,92-96,134-137).  The simulator does not keep
       emitted frames; it keeps the POSES they were made from and rebuilds the stack every step (bit-identical:
       same arithmetic, same fp32 inputs).  hist_*[0] is the pose behind frame t-2, hist_*[1] behind frame t-1
       (the newest emitted frame; normally the state itself).  msoc_get_state always fills them (hist_valid = 1).
       msoc_set_state with hist_valid = 0 leaves the emitted history alone, like poking the bodies of the
       reference's Game (the next observation still shows the frames emitted before the poke); with
       hist_valid = 1 it installs both poses (checkpoint restore, parity injection). */
    uint32_t hist_valid;
    uint32_t reserved0;
    float hist_pos[2][5][2];
    float hist_vel[2][4][2];
    float hist_ang[2][4];
    float hist_angvel[2][4];
} msoc_env_state;

/* Per-rollout statistics accumulated on the device since the last msoc_stats_read(.., reset=1)
   (replaces the trainer-side bookkeeping of marl-soccer.ipynb:411-429). */
typedef struct msoc_stats {
    double episodes;          /* episodes finished (steps reached max_steps) */
    double episode_return_sum; /* sum of blue returns of the finished episodes */
    double goals_blue, goals_red;
    double env_steps;
    double contacts;          /* contacts solved */
    double contact_overflow;  /* contacts dropped because an env exceeded MSOC_MAX_CONTACTS */
    double nonfinite_actions; /* env-steps whose action block held a NaN/Inf (soccer_env.py:116-117 raises; the
                                 device path clips -- NaN acts as -1 -- and counts) */
} msoc_stats;

typedef struct msoc_handle msoc_handle;

const char *msoc_last_error(void);
int msoc_version(void);

/* Replaces: SoccerEnv.__init__ x n_envs inside SyncMultiAgentVecEnv.__init__
   (soccer_env.py:19-73, marl_vecenv.py:8-16).  Allocates struct-of-arrays state for n_envs
   independent envs on `device` and spawns them once in MSOC_MODE_RANDOM (Game.__init__ ->
   setup_field -> reset, game/game.py:43,74).  global_env_offset is the global index of local
   env 0; the Philox spawn stream is keyed by (seed, global index) so results do not depend on
   how envs are sharded over GPUs. */
int msoc_create(const msoc_config *cfg, int64_t n_envs, int device, uint64_t seed,
                uint64_t global_env_offset, msoc_handle **out);
int msoc_destroy(msoc_handle *h);
int64_t msoc_num_envs(const msoc_handle *h);

/* Replaces: SoccerEnv.reset / SyncMultiAgentVecEnv.reset (soccer_env.py:81-98, marl_vecenv.py:18-28,
   Game.reset game/game.py:76-118).  d_mask: N bytes, non-zero = reset that env; NULL = all.
   has_seed: env i is re-seeded with seed + global_index(i) (marl_vecenv.py:23) and its spawn
   counter restarts.  d_obs_out (N,4,66) f32 receives 3 copies of frame 0 for the reset envs
   (soccer_env.py:92-96); rows of other envs are left untouched. */
int msoc_reset(msoc_handle *h, const uint8_t *d_mask, int mode, int has_seed, uint64_t seed,
               float *d_obs_out, void *stream);

/* Replaces: SyncMultiAgentVecEnv.step -> SoccerEnv.step -> Game.step -> Space.step(1/60)
   (marl_vecenv.py:30-68, soccer_env.py:100-154, game/game.py:378-437).
     d_actions (N,4,3) f32 in [-1,1] (clipped, soccer_env.py:119)
     d_obs_out (N,4,66) f32  new stacked observation [frame t-2 | frame t-1 | frame t] per agent; write-only: the
                             history lives in the handle as poses (see msoc_env_state), not in this buffer
     d_reward  (N,2) f32     blue agents' reward (red is always 0.0, soccer_env.py:141-146)
     d_done    (N) u8        truncation flag (soccer_env.py:148)
     d_goal    (N) i8        +1 blue scored, -1 red scored, 0 none (info["goal_scored_by"])
     d_score   (N,2) i32     info["score"] of this step = (blue, red) after the goal test and before
                             any auto-reset (game/game.py:415); may be NULL
   flags: MSOC_STEP_AUTO_RESET, MSOC_STEP_GENERAL_PATH.
   Stream semantics: asynchronous; everything is ordered after the work already enqueued on `stream`, and work
   enqueued on `stream` afterwards sees the complete step.  One step is two kernel launches on `stream` (a streaming
   contact-free kernel over all envs, then one persistent contact kernel over the envs it declined).  Which half of the ping-pong state
   is current is a counter in device memory that the kernels advance themselves, so a CUDA graph may capture any
   number of consecutive steps and be replayed any number of times. */
int msoc_step(msoc_handle *h, const float *d_actions, float *d_obs_out,
              float *d_reward, uint8_t *d_done, int8_t *d_goal, int32_t *d_score, uint32_t flags,
              void *stream);

/* msoc_step with a reward for both teams (self-play that trains on red's experience too; the reference has no red
   reward).  Arguments, outputs, flags, stream semantics and graph capture are those of msoc_step, except:
     d_reward  (N,4) f32, 16-byte aligned   columns 0, 1: blue's reward, bit for bit what msoc_step writes;
                                            columns 2, 3: red's reward (the same for both red agents)
   Red's reward is blue's reward on the field mirrored about x = 400 (msoc_team_inputs): in exact arithmetic, red's
   reward of (S, actions) is blue's reward of M(S) with the mirrored actions.  Term by term, from the positions at the
   start of the step and the step's displacement (before any soft reset), like blue's:
     term            blue                                          red
     proximity       ball_proximity_multiplier x decrease of the   the same for agents 2, 3
                     distance of agents 0, 1 to the ball
     ball to goal    move_ball_to_goal_multiplier x decrease of    the same to (10, 300)
                     the ball's distance to (790, 300)
     goals           +goal_scored_reward blue scores,              +goal_scored_reward red scores,
                     -goal_conceded_penalty red scores             -goal_conceded_penalty blue scores
     alive           -alive_penalty                                -alive_penalty
     truncation      the step's reward becomes                     score_difference_multiplier x (red - blue)
                     score_difference_multiplier x (blue - red)
   Red's episode return is not kept by the handle (msoc_env_state.ep_return and msoc_stats stay blue's).  A misaligned
   d_reward gives MSOC_ERR_INVALID, as do msoc_step's null arguments. */
int msoc_step_teams(msoc_handle *h, const float *d_actions, float *d_obs_out,
                    float *d_reward, uint8_t *d_done, int8_t *d_goal, int32_t *d_score, uint32_t flags,
                    void *stream);

/* Same call with HOST buffers (the NumPy drop-in path, marl_vecenv.py:62-68): copies actions
   H2D, steps, copies obs/reward/done/goal D2H and synchronises; NULL output pointers are skipped.  Large batches are
   cut into up to 8 chunks on two internal streams so that the H2D copy and the kernels of one chunk overlap the D2H
   copies of the previous one.  Pinned host memory is used as given.  Host-buffer steps, device steps (msoc_step,
   msoc_step_teams), replays of captured graphs of them, resets and state loads may be interleaved on one handle in any
   order: each step continues from the state the previous call left. */
int msoc_step_host(msoc_handle *h, const float *h_actions, float *h_obs, float *h_reward,
                   uint8_t *h_done, int8_t *h_goal, int32_t *h_score, uint32_t flags, void *stream);
/* The same step, but only the NEWEST frame comes back: h_frames (N,4,22) f32 = 352 B per env instead of 1 056.  The
   caller owns the 3-frame stack exactly as soccer_env.py:130-140 does (append the new frame; after a truncation with
   MSOC_STEP_AUTO_RESET the new frame is frame 0 of the next episode and fills all three slots, soccer_env.py:92-96). */
int msoc_step_host_frames(msoc_handle *h, const float *h_actions, float *h_frames, float *h_reward,
                          uint8_t *h_done, int8_t *h_goal, int32_t *h_score, uint32_t flags, void *stream);
int msoc_reset_host(msoc_handle *h, const uint8_t *h_mask, int mode, int has_seed, uint64_t seed,
                    float *h_obs, void *stream);

/* Device pointers of per-env counters kept in the state (valid for the handle's lifetime):
   score (N,2) i32 = info["score"] (game/game.py:415), steps (N) i32. Synchronous gather. */
int msoc_read_counters(msoc_handle *h, int32_t *h_score /* N*2 */, int32_t *h_steps /* N */, void *stream);

/* State injection / extraction for a list of local env indices (host arrays); synchronous.  msoc_set_state wraps the
   agent angles on the host in double precision.  Both run the kernels of msoc_save_states / msoc_load_states. */
int msoc_get_state(msoc_handle *h, const int64_t *h_idx, int64_t n, msoc_env_state *h_out);
int msoc_set_state(msoc_handle *h, const int64_t *h_idx, int64_t n, const msoc_env_state *h_in);

/* Device-side checkpointing, branching and cloning of envs: msoc_env_state records in DEVICE memory, n x 808 bytes.
   Records of the envs d_idx[0..n) (NULL: envs 0..n-1) as msoc_env_state, into device memory; stream-ordered,
   no allocation, no host wait, capturable.  d_out 16-byte aligned.  An out-of-range device index gives an all-zero
   record (hist_valid = 0).  The bytes equal what msoc_get_state returns for the same env. */
int msoc_save_states(msoc_handle *h, const int64_t *d_idx, int64_t n, msoc_env_state *d_out, void *stream);
/* Installs d_in[k] into env d_idx[k], with the semantics of msoc_set_state; out-of-range entries are skipped, duplicate
   destinations are undefined.  The observation buffer is not written (as msoc_set_state).  The first call on a handle
   may allocate the injection side array; if it is missing while `stream` is capturing, returns MSOC_ERR_INVALID.
   Graphs of msoc_step / msoc_reset captured before that allocation do not see the side array: call msoc_load_states or
   msoc_set_state once before capturing any graph on a handle whose states will be loaded.
   d_in 16-byte aligned.  Agent angles (ang, hist_ang) are taken bit for bit when |a| <= 3.14159274101257324 (float(pi),
   the threshold of msoc_set_state's host wrap); larger ones are wrapped into [-pi, pi] on the device in single
   precision, which may differ in the last bit from the double-precision host wrap of msoc_set_state.
   Both calls: n == 0 is a no-op; a null handle, n < 0, NULL d_idx with n > the env count and a null or misaligned state
   pointer give MSOC_ERR_INVALID. */
int msoc_load_states(msoc_handle *h, const int64_t *d_idx, int64_t n, const msoc_env_state *d_in, void *stream);

/* Device pointers of the handle's INTERNAL I/O buffers (the ones the *_host entry points use), so that a
   device-resident caller can wrap them zero-copy (e.g. as torch tensors through
   __cuda_array_interface__) and pass them to msoc_step / msoc_reset.  Valid until msoc_destroy. */
typedef struct msoc_buffers {
    float *obs;      /* (N,4,66) */
    float *actions;  /* (N,4,3)  */
    float *reward;   /* (N,2)    */
    uint8_t *done;   /* (N)      */
    int8_t *goal;    /* (N)      */
    int32_t *score;  /* (N,2)    */
    uint8_t *mask;   /* (N) scratch for masked resets */
    double *stats;   /* 8 live accumulators (msoc_stats layout) */
} msoc_buffers;
int msoc_device_buffers(msoc_handle *h, msoc_buffers *out);

/* Rows of the handle's INTERNAL observation buffer (the last stacked observation the *_host entry points produced,
   per env 4 x 66 floats) for a list of envs; synchronous. */
int msoc_get_obs_host(msoc_handle *h, const int64_t *h_idx, int64_t n, float *h_obs);

/* RGB images of envs, drawn on the device (no counterpart in the reference's batched path; the picture is the one of
   marl_soccer_b200/renderer.py scene(): field, lines, agents with their noses, ball).  Each image shows the state
   msoc_get_state returns: after a step the state behind the newest observation frame, after an auto-reset the first
   state of the new episode, after msoc_set_state the injected state.
     d_out  (n, height, width, 3) uint8, HWC, images contiguous; 16-byte aligned; every byte is written once
   Pixel (r, c) shows the point ((c + 0.5) 800 / width, (r + 0.5) 600 / height) of the 800 x 600 screen (y down), so
   the two axes scale independently.  The handle's state is not changed, nothing is allocated and the host does not
   wait: the call can be captured in a CUDA graph behind msoc_step. */
/* RGB images (n, height, width, 3) uint8 of the envs d_idx[0..n) (NULL: envs 0..n-1), stream-ordered, capturable.
   An out-of-range device index yields an all-zero image and reads/writes nothing else. 1 <= height, width <= 4096. */
int msoc_render(msoc_handle *h, const int64_t *d_idx, int64_t n, int height, int width, uint8_t *d_out, void *stream);
/* Same with host index list and host output; validates indices (MSOC_ERR_INVALID), synchronous. */
int msoc_render_host(msoc_handle *h, const int64_t *h_idx, int64_t n, int height, int width, uint8_t *h_out);

/* Statistics: d_out receives 8 doubles (msoc_stats layout) on the device, stream-ordered, ready to
   be all-reduced with NCCL; reset != 0 zeroes the accumulators afterwards. */
int msoc_stats_device(msoc_handle *h, double *d_out, int reset, void *stream);
int msoc_stats_read(msoc_handle *h, msoc_stats *h_out, int reset, void *stream);

/* Rollout half of the trainer (marl-soccer.ipynb:366-431), the immediate caller of msoc_step: what the loop does with the
   blue agents' observations before the policy runs, as ONE pass over them instead of five torch passes.
     d_obs      (N,4,66) f32   the stacked observation msoc_step wrote; rows 0,1 of every env (the trainable agents) are read
     d_shift, d_inv_std (66) f32   normaliser in multiply-add form: x' = clip(x * inv_std + shift, -10, 10)
                                   (shift = -mean / (std + 1e-8), inv_std = 1 / (std + 1e-8); marl-soccer.ipynb:385)
     d_x_out    (2N,72) bf16   normalised policy input, rows padded from 66 to 72 columns (columns 66..71 are not written:
                               allocate zeroed); row 2e + a = agent a of env e
     d_raw_out  (N,2,66) bf16  the raw observation for the rollout buffer (marl-soccer.ipynb:403), or NULL
     d_moments  (2,66) f64     per-feature sum and sum of squares of the raw rows are ADDED here (running mean / variance
                               of the normaliser, marl-soccer.ipynb:264-296, :431), or NULL
   Runs on the current device, asynchronous on `stream`. */
int msoc_policy_inputs(const float *d_obs, int64_t n_envs, const float *d_shift, const float *d_inv_std, void *d_x_out,
                       void *d_raw_out, double *d_moments, void *stream);

/* The same pass over either team's rows, for a policy that plays red as if it were blue (self-play against frozen
   snapshots; no counterpart in the reference, whose red agents play U(-1, 1)).  team 0 is msoc_policy_inputs: rows 0, 1
   of every env.  team 1 reads rows 2, 3 (bytes 528..1055 of the env's 1056-byte block) and applies the mirror M below
   to each of their three 22-float frames BEFORE the normalise, clip, bf16 and pad steps; d_raw_out and d_moments
   receive the mirrored rows.  Output layout, NULL rules and the stream are those of msoc_policy_inputs (row 2e + a of
   d_x_out = agent 2 + a of env e).  A team other than 0 or 1, a NULL d_obs / d_shift / d_inv_std / d_x_out or
   n_envs <= 0 gives MSOC_ERR_INVALID.
   The field is symmetric about x = 400 and red's frames are built from red's own side (mate a ^ 1, opponents 0 and 1,
   own goal at x = 790), so M turns a red frame into the frame a blue agent sees on the mirrored field (x -> 800 - x,
   theta -> pi - theta):
     index                               feature                                mirrored
     0, 1                                vx, vy / max_velocity                  -x, x
     2                                   angle / pi                             x >= 0 ? 1 - x : -1 - x  (fp32; +0 and -0 -> 1)
     3                                   omega / max_angular_velocity           -x
     4, 7, 10, 13, 16, 19                unit-x to mate, opp 0, opp 1, ball,    -x
                                         own goal, opp goal
     5, 6, 8, 9, 11, 12, 14, 15, 17, 18, 20, 21   unit-y, distances             x
   The negations are exact sign flips.  An action (a0, a1, a2) a mirrored policy returns (body-frame force x, y and
   torque) is red's action (a0, -a1, -a2). */
int msoc_team_inputs(const float *d_obs, int64_t n_envs, int team, const float *d_shift, const float *d_inv_std,
                     void *d_x_out, void *d_raw_out, double *d_moments, void *stream);

/* Work classes of the last step (instrumentation for tests and bench.py; no counterpart in the reference): how many envs
   the streaming kernel handed to the contact kernel as light (exactly one agent x wall candidate pair), heavy (the
   general path), pair (exactly one agent x agent / ball x agent pair, at most one wall pair beside it) and multi (several
   wall pairs), in this order.
   The rest of the envs were contact-free.  Stream-ordered read, then synchronises `stream`. */
int msoc_last_class_counts(msoc_handle *h, int32_t h_out[4], void *stream);

/* Launch accounting for bench.py: number of kernels this library has launched. */
uint64_t msoc_launch_count(void);

/* Debug aid: bit set of the kernels' own bounds / invariant checks that failed since the last call (list entries
   inside the stepped range, contact-pool and overflow slots, arbiter-cache counts, env indices of the observation
   builder, the device-side step counter, non-NaN state, render and state save / load indices).  Only the checked build (libmsoc_checked.so, compiled with
   -DMSOC_CHECKS by marl_soccer_b200/build.py) evaluates them; the product build returns -1. */
int msoc_debug_errors(void);

#ifdef __cplusplus
}
#endif
#endif /* MSOC_H */
