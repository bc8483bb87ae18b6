/*
 * navgym_b200.h — C ABI of libnavgym_b200.so, the sm_100a implementation of nav-gym's
 * NavGym-v0 per-step hot path.
 *
 * Plain C types only (pointers, sizes, one POD argument block); no torch / C++ types cross
 * this boundary.  All *_dev pointers are CUDA device pointers; `stream` is a cudaStream_t
 * passed as void* (NULL = legacy default stream).  Every launcher is asynchronous with
 * respect to the host unless its name ends in _host; return value 0 = success, otherwise a
 * cudaError_t (text via navgym_error_string()).  There is NO CPU fallback: with no device
 * every call fails.
 *
 * Citations are relative to /root/reference/nav_gym/src/nav_gym_env/ (the reference) and
 * name the interface each entry point replaces.
 */
#ifndef NAVGYM_B200_H
#define NAVGYM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NAVGYM_NUM_BEAMS 512   /* keti_robot.py:48 n_angles */
#define NAVGYM_OBS_TAIL 7      /* prev_pose(2) pose(2) vel(2) yaw(1), env.py:455 */
#define NAVGYM_HIT_NONE (-32768)
#define NAVGYM_MAX_DISC 64     /* per-env capacity of the kernel's staging buffers */
#define NAVGYM_MAX_SEG 128
#define NAVGYM_SCHED_BUCKETS 32

/* Observation row formats (navgym_step_args_t / navgym_her_args_t .obs_format).
 *   NAVGYM_OBS_F32  float32 rows of obs_stride floats: [S*512 scans | 7 tail fields], obs_stride >= S*512 + 7.
 *   NAVGYM_OBS_F16  rows of obs_stride HALVES (2-byte units): [S*512 scans as float16, round-to-nearest
 *                   of the float32 value | the 7 tail fields as float32 (14 halves) | padding, never
 *                   written].  obs_stride must be even and >= S*512 + 14 and the row base 4-byte
 *                   aligned, so that the tail is aligned float32; S*512 + 16 halves gives 16-byte
 *                   aligned rows.  The obs / obs_host pointers of every entry point stay `float *`:
 *                   pass the row storage cast to it.
 * Anything else (an unknown format, an odd or too short stride, a misaligned base) is
 * cudaErrorInvalidValue. */
#define NAVGYM_OBS_F32 0
#define NAVGYM_OBS_F16 1

/* navgym_step_args_t.auto_reset: 0 = off, 1 = same-step (the launch that ends an episode writes
 * the next episode's first observation over its final one), NAVGYM_AUTORESET_NEXT_STEP = the
 * launch after the one that ends an episode starts the next (see navgym_step_batch). */
#define NAVGYM_AUTORESET_NEXT_STEP 2

/* rows of the structure-of-arrays float64 state block state[NAVGYM_NS][num_envs] */
enum {
    NAVGYM_S_PX = 0, NAVGYM_S_PY, NAVGYM_S_TH,   /* robot pose (keti_robot.py:56-58) */
    NAVGYM_S_GX, NAVGYM_S_GY,                    /* goal */
    NAVGYM_S_PPX, NAVGYM_S_PPY, NAVGYM_S_PYAW,   /* pose / yaw fields of prev_obs (env.py:726) */
    NAVGYM_S_PV, NAVGYM_S_PW,                    /* prev_action (env.py:725) */
    NAVGYM_NS
};

/* One occupancy map of the pool (reference map_info dict, map_generator.py:113-122). */
typedef struct {
    int32_t W, H;            /* cells */
    int64_t edt_offset;      /* element offset of this map's float EDT ([H][W]) in edt_pool */
    double ox, oy, res;      /* origin [m], resolution [m/cell] */
    int64_t spawn_offset;    /* first row of this map's spawn tuples in spawn_pool */
    int32_t spawn_count;     /* 0 = map has no spawn pool */
    int32_t _pad;
} navgym_map_t;

/* Argument block of the fused step / reset kernels.  Layouts:
 *   state   f64 [NAVGYM_NS][num_envs]         steps    i32 [num_envs]
 *   actions f32 [num_envs][2]                 map_id   i32 [num_envs]
 *   discs   f32 [num_envs][max_disc][3] (x,y,r)   ndisc i32 [num_envs]
 *   segs    f32 [num_envs][max_seg][4] (ax,ay,bx,by)  nseg i32 [num_envs]
 *           (max_disc + max_seg <= 256: the kernel parks one beam window per obstacle in shared memory)
 *   noise   f32 [num_envs][2][512] additive, slot 0 = the step's scan, slot 1 = the crash
 *           re-scan (parity traces); NULL -> Philox N(0, noise_std[env]) (production)
 *   obs     f32 [num_envs][obs_stride], first S*512+7 columns written per row (S = num_scan_stack;
 *           the S-1 older scans are carried over from the row's previous contents); with
 *           obs_format = NAVGYM_OBS_F16 the rows are [num_envs][obs_stride] halves instead (see
 *           NAVGYM_OBS_F16 above; the older scans are shifted as float16)
 *   tail64  f64 [num_envs][7]   (the 7 trailing observation fields in float64, env.py:455)
 *   hits    i16 [num_envs][512][2] hit cell minus origin cell of the step's first scan, or
 *           NAVGYM_HIT_NONE; NULL = not recorded
 */
typedef struct {
    /* ---- constants (reference kwargs, __init__.py:6-38) ---- */
    double dt;               /* time_step */
    double dist_thresh;      /* distance_threshold */
    double min_turn_radius;  /* min_turning_radius */
    double r_scale, r_success, r_crash, r_progress, r_forward, r_rotation, r_discomfort;
    float range_max;         /* keti_robot.py:47 */
    float t_stop;            /* march limit in cells (reference: W*H, env.py:337) */
    int32_t cell_rule;       /* 0: float64 cell division (NumPy 1.x), 1: float32 (NumPy 2) */
    int32_t max_disc, max_seg;
    int32_t num_envs;
    int32_t obs_stride;      /* floats per obs row, >= 519 */
    int32_t auto_reset;      /* 1: on done draw a spawn tuple and return the new first obs;
                              * NAVGYM_AUTORESET_NEXT_STEP: draw it in the next launch */
    int32_t max_episode_steps; /* 0 = none (the reference has no time limit) */
    int32_t num_maps;
    int32_t resample_map;    /* 1: auto-reset also draws a new map id */
    uint64_t seed;
    int64_t env_offset;      /* global index of env 0 (multi-GPU sharding) */
    int32_t sched_phase;     /* which third of `sched` is current: step counter mod 3 */
    int32_t num_scan_stack;  /* S of env.py:257-279 (0 or 1 = no stacking): obs row = S*512 + 7 */
    int32_t env_begin;       /* this launch steps environments [env_begin, env_begin + env_count) */
    int32_t env_count;       /* 0 = through num_envs; num_envs stays the SoA stride of all buffers */
    float noise_lo, noise_hi; /* scan_noise_std range resampled at auto-reset */
    /* ---- device pointers ---- */
    const navgym_map_t *maps;
    const float *edt_pool;      /* per-map float EDTs as built by navgym_edt_build */
    const double *spawn_pool;   /* [rows][5] = sx, sy, gx, gy, theta */
    int32_t *map_id;
    const double *lin;          /* [512] beam angle table (env.py:388-390) */
    const float *thr, *dthr;    /* [512] crash / discomfort thresholds (env.py:162-180) */
    double *state;
    int32_t *steps;
    int32_t *episodes;          /* [num_envs] episode counter (RNG stream id) */
    const float *actions;
    const float *discs;
    const int32_t *ndisc;
    const float *segs;
    const int32_t *nseg;
    const float *noise;
    float *noise_std;           /* [num_envs] */
    float *obs;
    double *tail64;
    float *reward;
    uint8_t *done, *is_success, *is_crash, *truncated;
    float *distance;
    int16_t *hits;
    /* optional longest-first launch order, i32 [3][NAVGYM_SCHED_BUCKETS] counts followed by
     * [3][NAVGYM_SCHED_BUCKETS][num_envs] env ids; initialise third 0 with all envs in bucket 0
     * (count = num_envs, list = 0..num_envs-1), everything else zero, and advance sched_phase by
     * one (mod 3) after every navgym_step_batch.  NULL = block i steps env i. */
    int32_t *sched;
    /* optional second destinations of reward / done (NULL = none): device-visible addresses the
     * kernel also stores to, e.g. mapped pinned host memory -- the host-buffer entry points
     * below point them at reward_host / done_host so that a group needs one D2H copy (its
     * observation rows) instead of three. */
    float *reward_mirror;
    uint8_t *done_mirror;
    /* optional pedestrian geometry of the NEXT episode (same layouts as discs / ndisc / segs /
     * nseg; discs_reset == NULL = none): the first scan after an auto-reset is taken against it
     * instead of the ended episode's pedestrians. */
    const float *discs_reset;
    const int32_t *ndisc_reset;
    const float *segs_reset;
    const int32_t *nseg_reset;
    /* row format of obs (and of obs_host in the host-buffer entry points): NAVGYM_OBS_F32 (0, the
     * zero-initialised default) or NAVGYM_OBS_F16; obs_stride counts elements of that format */
    int32_t obs_format;
    int32_t _pad;
} navgym_step_args_t;

/* navgym_step_batch, navgym_reset_obs_batch, navgym_reset_envs and navgym_export_env return
 * cudaErrorInvalidValue, and launch nothing, for an argument block with
 *   - obs rows that NAVGYM_OBS_F32 / NAVGYM_OBS_F16 above do not allow (format, stride, alignment);
 *   - env_begin < 0, env_begin > num_envs, env_count < 0 or env_begin + env_count > num_envs;
 *   - max_disc + max_seg > 256 counting the obstacle buffers given (discs, segs; for
 *     navgym_reset_envs also discs_reset, segs_reset on their own).
 * The three launchers return 0 without launching when num_envs <= 0 or when the range is empty
 * (env_begin == num_envs). */

/* ---- fused hot path: NavGymEnv.step (env.py:591-728) over num_envs environments ------ */
int navgym_step_batch(const navgym_step_args_t *args, void *stream);
/* Next-step auto-reset (auto_reset = NAVGYM_AUTORESET_NEXT_STEP, Gymnasium's default).  `done` is
 * then an INPUT as well.  For every environment e of the launch range:
 *   - done[e] == 0 on entry: the step of auto_reset = 0, crash rollback and re-scan included.  The
 *     row of an episode that ends now is its final observation, and its goal is still
 *     state[NAVGYM_S_GX / S_GY];
 *   - done[e] != 0 on entry: actions[e] is not read (a NaN action changes nothing), and the
 *     environment starts its next episode bit for bit as navgym_reset_envs with mask[e] = 1 starts
 *     it: the draw keyed by (env_offset + e, episodes[e]), episodes[e] += 1, steps[e] = 0, the
 *     first observation in every stack slot, tail64, state, map_id, noise_std, the scan taken
 *     against discs_reset / segs_reset when discs_reset != NULL, else against discs / segs.
 *     Unlike navgym_reset_envs it also writes the step outputs: reward = 0, done = is_success =
 *     is_crash = truncated = 0, distance = the distance from the new pose to the new goal (float64
 *     rounded to float32, as the step computes it), the mirrors alike; hits of that scan; and the
 *     environment's entry in the next launch order.
 * navgym_reset_obs_batch and navgym_reset_envs do not write done: a caller that resets
 * environments through them clears their done bytes, or the next step starts yet another episode.
 * Setting done[e] = 1 has the next step start a new episode for e.  Each draw depends only on
 * the environment's own episodes[e]: for the same per-episode actions every episode's sequence of
 * (episode, step) records is the one of auto_reset = 0 followed by navgym_reset_envs(mask = done)
 * after every step, whatever the sharding.  The host-buffer entry points below launch through
 * navgym_step_batch and so follow the same contract: the final row lands in obs_host at the
 * ending step, the next episode's first row one step later. */
/* The same step for a caller whose buffers live on the HOST (the reference's own calling
 * convention: numpy in, numpy out).  actions_host f32 [num_envs][2], obs_host f32
 * [num_envs][obs_stride] (rows of args->obs_format, like obs), reward_host f32 [num_envs],
 * done_host u8 [num_envs] must be pinned
 * (cudaHostAlloc / cudaHostRegister).  The batch is stepped as `chunks` launches over consecutive
 * environment ranges on prioritised streams, each followed by the device-to-host copy of its
 * rows, so the copies of early chunks overlap the raycast of later ones; args->actions, obs,
 * reward, done are the device staging buffers.  Ordered after prior work on `stream`; returns
 * when every result has landed on the host. */
typedef struct navgym_host_pipe navgym_host_pipe_t;
navgym_host_pipe_t *navgym_host_pipe_create(int chunks, int num_envs, int longest_first);
void navgym_host_pipe_destroy(navgym_host_pipe_t *pipe);
int navgym_step_batch_host(navgym_host_pipe_t *pipe, const navgym_step_args_t *args, void *stream,
                           const float *actions_host, float *obs_host, float *reward_host,
                           uint8_t *done_host);
/* Asynchronous form for hosts that keep several groups of environments in flight (group g =
 * the pipe's g-th env range; EnvPool-style): submit enqueues H2D(actions of the group) -> step
 * -> D2H(its rows) on the group's stream and returns at once; wait blocks until that group's
 * results are on the host.  While the host consumes group A's observations group B is stepping,
 * so the PCIe transfer of one group hides behind the raycast of the other.  The caller must not
 * submit a group again before waiting for it, and must have synchronised prior work that
 * touches the state (reset) before the first submit. */
int navgym_step_batch_host_submit(navgym_host_pipe_t *pipe, const navgym_step_args_t *args, int group,
                                  const float *actions_host, float *obs_host, float *reward_host,
                                  uint8_t *done_host);
int navgym_step_batch_host_wait(navgym_host_pipe_t *pipe, int group);
/* the pipe's number of groups, and group g's env range [begin, end) */
int navgym_host_pipe_groups(const navgym_host_pipe_t *pipe);
int navgym_host_pipe_group_bounds(const navgym_host_pipe_t *pipe, int group, int *begin, int *end);
/* The whole host-side rollout loop in C (the reference's `while True: obs, r, d, info =
 * env.step(policy(obs))` smoke loop, env.py:1318-1355, for a batch): every group is primed with
 * the policy's step-0 actions, then `steps` times round each group is waited for, `policy` is
 * called with the group's env range -- its rows of obs_host / reward_host / done_host hold the
 * results of step `step - 1` -- to write the group's next actions into actions_host, and the
 * group is submitted again.  No per-group work in the caller's language; the PCIe transfers of
 * one group hide behind the raycast of the others.  Returns when all `steps` steps of every
 * group have landed (also on error: nothing stays in flight). */
typedef void (*navgym_policy_fn)(void *user, int group, int env_begin, int env_end, int64_t step,
                                 const float *obs_host, const float *reward_host,
                                 const uint8_t *done_host, float *actions_host);
int navgym_host_rollout(navgym_host_pipe_t *pipe, const navgym_step_args_t *args, int64_t steps,
                        navgym_policy_fn policy, void *user, float *actions_host, float *obs_host,
                        float *reward_host, uint8_t *done_host);
/* navgym_step_batch_host, navgym_step_batch_host_submit and navgym_host_rollout return
 * cudaErrorInvalidValue for
 *   - a NULL pipe, or args->num_envs other than the pipe's;
 *   - a NULL args->actions (the device staging buffer of the actions);
 *   - an argument block that navgym_step_batch rejects (see above; the pipe sets env_begin,
 *     env_count, sched and sched_phase of each group itself);
 *   - obs_host rows that args->obs_format does not allow (float16: a 4-byte aligned base);
 *   - submit: a group outside [0, groups); rollout: a NULL policy or steps < 0.
 * A rejected call enqueues nothing and leaves the pipe as it was.  So does a submit that fails
 * (a failed copy or graph capture): a group's schedule phase and cached graphs change only once
 * its step has been enqueued. */
/* built-in policy: step s plays row (s mod rows) of a host action bank f32 [rows][num_envs][2] */
typedef struct {
    const float *actions;
    int32_t rows, num_envs;
} navgym_action_bank_t;
void navgym_policy_action_bank(void *user, int group, int env_begin, int env_end, int64_t step,
                               const float *obs_host, const float *reward_host,
                               const uint8_t *done_host, float *actions_host);
/* first observation of an episode, NavGymEnv.reset's tail (env.py:822-831) */
int navgym_reset_obs_batch(const navgym_step_args_t *args, void *stream);
/* Masked device reset: new episodes for chosen environments, exactly as the step's auto-reset
 * starts them, for callers that step with auto_reset = 0 so that they can read each ended
 * episode's final observation row (and its goal, state[NAVGYM_S_GX / S_GY]) first.  One launch;
 * mask u8 [num_envs] on the device.  For every environment e of the launch range [env_begin,
 * env_begin + count) (count = env_count, 0 = through num_envs) with mask[e] != 0:
 *   1. the next episode is drawn as the auto-reset of navgym_step_batch draws it: Philox key
 *      (env_offset + e, episodes[e], 0x5eed, 0xfffffff0) with `seed`; a new map when
 *      resample_map && num_maps > 1; a spawn row (start, goal, theta) of that map's pool;
 *      noise_std = noise_lo + (noise_hi - noise_lo) * u01; then episodes[e] += 1, steps[e] = 0.
 *      A map without a spawn pool keeps the pose and goal in `state` (and its map): the
 *      auto-reset would restart from the pose before the ending step instead, so for such maps
 *      the two are not equivalent;
 *   2. the first observation is written as the auto-reset pass writes it: the obs row in
 *      obs_format (all S stack slots hold the new scan), tail64, the state rows (previous pose =
 *      pose, previous action 0, previous yaw = yaw), map_id, noise_std.  The scan is taken
 *      against discs_reset / segs_reset when discs_reset != NULL, else against discs / segs, with
 *      the same noise as the auto-reset pass (Philox, or slot 0 of `noise`);
 *   3. hits are not written (they keep the step's first scan, as with auto-reset).
 * Whatever the mask, reward, done, is_success, is_crash, truncated, distance, the mirrors and
 * sched are not written (the step already filed every environment into the next launch order),
 * and environments with mask[e] == 0 are not written at all.  auto_reset and actions are not
 * read.  After navgym_step_batch with auto_reset = 0 and then this call with mask = done, every
 * buffer above holds what the step with auto_reset = 1 would have left, bit for bit (pools with
 * spawn rows).  Each draw depends only on the environment's own episodes[e], so the result does
 * not depend on how the masked set is split across calls or env_offset shards.
 * cudaErrorInvalidValue: mask == NULL, or an argument block rejected as above. */
int navgym_reset_envs(const navgym_step_args_t *args, const uint8_t *mask, void *stream);

/* ---- host export of one environment (ros_env.py:69-176 reads a NavGymEnv's attributes; the
 * single-env drop-in returns numpy per step, env.py:728): everything it needs from environment
 * `env`, packed into one float64 row out_dev[navgym_export_env_len(S)] so that ONE device-to-host
 * copy fetches it: state[NAVGYM_NS] | tail64[7] | reward done is_success is_crash truncated
 * distance steps map_id episode noise_std | the S*512 scan columns of its observation row. */
int navgym_export_env_len(int num_scan_stack);
int navgym_export_env(const navgym_step_args_t *args, int env, double *out_dev, void *stream);

/* ---- HER batch API: compute_rewards / compute_terminals / compute_info (env.py:464-589) on
 * `count` stored observation rows obs[count][obs_stride] (float32, the layout of env.py:455;
 * with obs_format = NAVGYM_OBS_F16 the float16-scan rows above, obs cast to float *, obs_stride
 * in halves) with goals[count][2]; any output pointer may be NULL. */
typedef struct {
    double dist_thresh;
    double r_scale, r_success, r_crash, r_progress, r_forward, r_rotation, r_discomfort;
    int32_t count, obs_stride;
    int32_t num_scan_stack, _pad;
    const float *obs, *goals;
    const float *thr, *dthr;   /* [512] */
    float *reward;
    uint8_t *done, *is_success, *is_crash;
    float *distance;
    int32_t obs_format;        /* NAVGYM_OBS_F32 (0) or NAVGYM_OBS_F16 */
    int32_t _pad2;
} navgym_her_args_t;
int navgym_compute_rewards(const navgym_her_args_t *args, void *stream);

/* ---- pedestrian geometry, and scripted pedestrians: emit the geometry the robot's lidar sees
 * (leg discs env.py:398-402, box footprints env.py:404-414, or one trunk disc each) into the discs /
 * segs buffers of navgym_step_args_t -- with advance = 1 after moving every pedestrian one time
 * step as a waypoint walker (BASELINE configs C3 / C4), with advance = 0 for poses the caller
 * moved itself (the policy-driven pedestrians of env.py:617-662: navgym_peds_move below).
 *   peds f32 [num_envs][max_ped][NAVGYM_PED_F] (16-byte aligned, as is segs: cudaErrorMisalignedAddress otherwise):
 *     0 x, 1 y, 2 theta, 3 speed | 4 ax, 5 ay, 6 bx, 7 by (the two waypoints) | 8 target (0/1),
 *     9..11 distance travelled in the base frame (x, y, theta; leg gait, env.py:237-255) |
 *     12 has_legs (0/1), 13 trunk radius, 14..15 unused */
#define NAVGYM_PED_F 16
typedef struct {
    int32_t num_envs, max_ped, max_disc, max_seg;
    int32_t advance;      /* 0: only emit geometry for the current poses */
    int32_t trunk_mode;   /* 1: one disc of radius peds[..][13] per pedestrian */
    float dt;
    int32_t _pad;
    float *peds;
    const int32_t *nped;  /* [num_envs] or NULL = max_ped everywhere */
    float *discs;
    int32_t *ndisc;
    float *segs;
    int32_t *nseg;
} navgym_peds_args_t;
int navgym_peds_advance(const navgym_peds_args_t *args, void *stream);

/* ---- lidar of the simulated pedestrians: _convert_obs(human, [robot] + other humans,
 * add_scan_noise=False, lidar_legs=False) (env.py:683-693, 808-815) for every pedestrian of
 * every environment in one launch.  Agent n = (environment n / agents_per_env, slot n %
 * agents_per_env); each casts K beams lin[k] + float32(theta) from float32(x, y) through its
 * environment's map (env.py:386-426), min-merges the closed footprints of the other agents
 * (segs of its environment, minus its own [skip_first, +skip_count)), clips to [0, range_max]
 * (env.py:435).  No noise.  ranges[n][k] of slots >= nagent[env] are left untouched. */
typedef struct {
    int32_t num_envs, agents_per_env;
    int32_t num_beams;           /* K (human.py:16: 512) */
    int32_t max_seg;             /* segment slots per environment */
    int32_t cell_rule, _pad;
    float range_max;             /* metres (human.py:15: 6.0) */
    float t_stop;                /* march cut-off in cells, as navgym_step_args_t.t_stop */
    const navgym_map_t *maps;
    const float *edt_pool;
    const int32_t *map_id;       /* [num_envs] */
    const int32_t *nagent;       /* [num_envs] live slots, or NULL = agents_per_env */
    const double *pose;          /* [num_envs][agents_per_env][3] x, y, theta */
    const double *lin;           /* [K] beam angles before the heading is added */
    const float *segs;           /* [num_envs][max_seg][4] ax, ay, bx, by */
    const int32_t *nseg;         /* [num_envs] */
    const int32_t *skip;         /* [num_envs][agents_per_env][2] first, count; or NULL */
    float *ranges;               /* [num_envs][agents_per_env][K] out */
    /* crowd mode (segs == NULL): the other agents' footprints are built in the kernel from
     * `pose` (every other live agent of the environment, footprint agent_fp) and the robot
     * (robot_state = navgym_step_args_t.state of the same batch, footprint robot_fp =
     * KetiRobot.threshold_footprint), float64 transform then float32 as env.py:404-414;
     * footprints farther than range_max cannot change a clipped scan and are skipped. */
    const double *robot_state;
    const uint8_t *env_mask;     /* [num_envs] or NULL: scan only environments with mask != 0 */
    double robot_fp[8], agent_fp[8];  /* 4 vertices (x, y) each, body frame */
} navgym_scan_args_t;
int navgym_agent_scan_batch(const navgym_scan_args_t *args, void *stream);
int navgym_sizeof_scan_args(void);

/* ---- pedestrian route following (env.py:633-645 waypoints, :666-680 new goal on arrival).
 * The reference plans an A* path on the 0.25 m cost map (env.py:312-332, 343-354) per
 * pedestrian and walks its waypoints (spaced > 2 m, popped within 1 m).  On the device each
 * map carries num_goals geodesic distance fields over that cost map (one per candidate goal,
 * u16 cells, 65535 = unreachable); following a field downhill is a shortest path, so the
 * waypoint 2 m further along it is found without a path object, and a new goal is a new field
 * id.  One thread per pedestrian:
 *   1. within 0.5 m of its goal: draw a new goal (Philox; reachable from here, farther than
 *      min_goal_dist) -- kept as is when none of 4 draws qualifies, like the reference when
 *      its planner fails;
 *   2. waypoint missing or within 1 m: advance it along the field until > 2 m away (or the goal);
 *   3. emit the waypoint (world) and the local goal the policy sees (env.py:641-645). */
typedef struct {
    int32_t W, H;             /* planning grid */
    int32_t num_goals, _pad;
    int64_t field_offset;     /* into fields, u16 elements: [num_goals][H][W] */
    int64_t goal_offset;      /* into goals, rows of 2 doubles */
    int64_t free_offset;      /* into free_xy, rows of 2 doubles: centres of free cost-map cells */
    int64_t free_count;
    double ox, oy, res;
} navgym_plan_map_t;
typedef struct {
    int32_t num_envs, max_ped;
    int32_t step;             /* RNG stream position: advance by one per call */
    int32_t _pad;
    uint64_t seed;
    int64_t env_offset;       /* global id of environment 0 (multi-GPU shards) */
    double min_goal_dist;     /* env.py:669: 10 m */
    const navgym_plan_map_t *maps;
    const uint16_t *fields;
    const double *goals;
    const int32_t *map_id;    /* [num_envs] */
    const int32_t *nped;      /* [num_envs] or NULL */
    const double *pose;       /* [num_envs][max_ped][3] */
    int32_t *goal_id;         /* [num_envs][max_ped] in/out */
    double *waypoint;         /* [num_envs][max_ped][2] in/out, NaN = none yet */
    float *goal_local;        /* [num_envs][max_ped][2] out */
    /* respawn (env.py:785-806).  Every call draws, for every pedestrian slot, the pedestrian of
     * the environment's NEXT episode into the cand_* arrays: a free cost-map cell at least
     * min_robot_dist from where the robot will start (up to 6 draws), heading U[0, 2 pi),
     * preferred speed U[v_pref_lo, v_pref_hi], legs with probability has_legs_ratio, a goal
     * field.  "Where the robot will start" is the spawn tuple navgym_step_batch draws on auto-reset
     * (same Philox stream: robot_seed, global env id, episodes[e]; robot_maps / spawn_pool /
     * num_maps / resample_map as in navgym_step_args_t) when cand_next_spawn != 0, else the
     * robot's current pose (robot_state = navgym_step_args_t.state).  cand_rows (layout of
     * navgym_peds_args_t.peds) feed navgym_peds_advance for navgym_step_args_t.discs_reset /
     * segs_reset.  Environments with respawn[e] != 0 (NULL = none) first ADOPT the candidates
     * drawn by the previous call: odometry, velocity and previous action zeroed, route reset. */
    const uint8_t *respawn;
    const double *free_xy;
    const double *robot_state;
    double min_robot_dist, v_pref_lo, v_pref_hi, has_legs_ratio;
    double *pose_rw;          /* == pose */
    double *v_pref;           /* [num_envs][max_ped] */
    uint8_t *has_legs;        /* [num_envs][max_ped] */
    double *dist_travelled;   /* [num_envs][max_ped][3] */
    double *vel;              /* [num_envs][max_ped][2] */
    float *prev_action;       /* [num_envs][max_ped][2] */
    double *cand_pose;        /* [num_envs][max_ped][3]; NULL = no candidates, no respawn */
    double *cand_v_pref;
    uint8_t *cand_legs;
    int32_t *cand_goal;
    float *cand_rows;         /* [num_envs][max_ped][NAVGYM_PED_F] */
    const navgym_map_t *robot_maps;
    const double *spawn_pool;
    const int32_t *episodes;
    uint64_t robot_seed;
    int32_t num_maps, resample_map;
    int32_t cand_next_spawn, _pad2;
} navgym_plan_args_t;
int navgym_peds_plan(const navgym_plan_args_t *args, void *stream);

/* env.py:655-662 + 237-255 for every pedestrian: clip the policy mean to [0, 1] x [-1, 1] (kept
 * as the next `speed` input), scale by the preferred speed, Human.set_vel (human.py:32-41,
 * float64), leg-gait odometry in the base frame, and the pedestrian rows of
 * navgym_peds_args_t.peds (pose, odometry, has_legs) the geometry kernel reads. */
typedef struct {
    int32_t num_envs, max_ped;
    double dt;
    const int32_t *nped;
    const float *mean;        /* [num_envs][max_ped][2] policy output */
    const double *v_pref;
    const uint8_t *has_legs;
    double *pose;             /* in/out */
    double *vel;              /* out: world velocity (vx, vy) */
    double *dist_travelled;   /* in/out */
    float *prev_action;       /* out */
    float *rows;              /* [num_envs][max_ped][NAVGYM_PED_F] out */
} navgym_move_args_t;
int navgym_peds_move(const navgym_move_args_t *args, void *stream);
int navgym_sizeof_move_args(void);
int navgym_sizeof_plan_args(void);
int navgym_sizeof_plan_map(void);

/* ---- the pedestrian policy, natively: HumanPolicy's deterministic action mean
 * (human_policy.py:38-55, the only output env.py:649-656 uses) for n pedestrians,
 *   mean = (sigmoid(actor1(a)), tanh(actor2(a))),  a = relu(act_fc2([relu(act_fc1(feat)), goal, speed])),
 *   feat = the convolutional front end (human_policy.py:24-25, 45-47 fed as in env.py:627-629,
 *          647) on the pedestrian's newest scan[512] (metres): clip to [0, 6], / 6 - 0.5 (float64,
 *          then float32) -> conv1d(1 -> 32, k 5, stride 2, pad 1) with act_fea_cv1's weight
 *          summed over its three input frames (env.py:647 feeds the same scan to all three; the
 *          fold is done here from the reference-shaped weight) -> relu -> conv1d(32 -> 32, k 3,
 *          stride 2, pad 1) -> relu -> 4096 features, channel-major like `.view(N, -1)`.
 * Three launches, no library GEMM, every contraction on the tcgen05 tensor cores in the "f16x3"
 * scheme (hi/lo f16 splits of both operands, three MMAs per K step: float32-grade results): the
 * front end (features leave as two f16 halves), act_fc1 with TMA-fed operands and TMEM
 * accumulators, act_fc2 with the heads in its epilogue.  Parameters are float32 device pointers
 * in torch's state_dict layout; they are copied / pre-split into the caller's workspace by navgym_policy_create, so
 * changing the weights means creating a new policy.  workspace: device memory, 1024-byte
 * aligned, navgym_policy_workspace_bytes(max_n) bytes (the feature halves dominate: 16 KB per
 * pedestrian), owned by the caller and kept alive for the policy's lifetime. */
typedef struct {
    int32_t max_n, _pad;
    const float *cv1_w, *cv1_b;   /* act_fea_cv1: [32][3][5], [32] */
    const float *cv2_w, *cv2_b;   /* act_fea_cv2: [32][32][3], [32] */
    const float *fc1_w, *fc1_b;   /* act_fc1: [256][4096], [256] */
    const float *fc2_w, *fc2_b;   /* act_fc2: [128][260], [128] */
    const float *a1_w, *a1_b;     /* actor1: [128], [1] */
    const float *a2_w, *a2_b;     /* actor2: [128], [1] */
    void *workspace;
    uint64_t workspace_bytes;
} navgym_policy_params_t;
typedef struct navgym_policy navgym_policy_t;
size_t navgym_policy_workspace_bytes(int max_n);
int navgym_sizeof_policy_params(void);
navgym_policy_t *navgym_policy_create(const navgym_policy_params_t *params, void *stream); /* NULL on failure */
void navgym_policy_destroy(navgym_policy_t *policy);
/* scan f32 [n][512] metres (clipped to [0, 6] and centred inside, env.py:627-629), goal f32
 * [n][2] (env.py:641-645), speed f32 [n][2] (the previous clipped mean) -> mean f32 [n][2]. */
int navgym_policy_mean(navgym_policy_t *policy, const float *scan, const float *goal,
                       const float *speed, int n, float *mean, void *stream);
/* byte offsets inside the workspace of {features hi, features lo, scales, total, act_fc1 output
 * hi, lo (f16 pairs times scales[6])} (tests compare the intermediate results against a float32
 * reference) */
void navgym_policy_workspace_layout(int max_n, uint64_t *out6);

/* ---- inner native boundary: range_libc --------------------------------------------- */
/* PyOMap(bool[H,W]) + PyRayMarching(omap, max_range) (env.py:337-340): exact Euclidean
 * distance transform of occ_dev (u8, non-zero = occupied, [H][W], row = y) into dist_dev.
 * W <= 12000 and H <= 32767 cells (cudaErrorInvalidValue otherwise). */
int navgym_edt_build(const uint8_t *occ_dev, int H, int W, float *dist_dev, int32_t *scratch_dev,
                     void *stream);
/* PyRayMarching.calc_range_many(ins f32[N,3], outs f32[N]) (env.py:425), ranges in cells. */
int navgym_calc_range_many(const float *dist_dev, int W, int H, const float *ins_dev,
                           float *outs_dev, int N, float max_range, float t_stop,
                           int16_t *hits_dev, void *stream);

/* Host-buffer drop-ins with the lifetime of the reference's Python objects. */
typedef struct navgym_raymarching navgym_raymarching_t;
navgym_raymarching_t *navgym_raymarching_create_host(const uint8_t *occ_host, int H, int W,
                                                     float max_range);
int navgym_raymarching_calc_range_many_host(navgym_raymarching_t *rm, const float *ins_host,
                                            float *outs_host, int N);
const float *navgym_raymarching_edt_dev(const navgym_raymarching_t *rm);
int navgym_raymarching_edt_host(const navgym_raymarching_t *rm, float *out_host); /* [H][W] */
void navgym_raymarching_destroy(navgym_raymarching_t *rm);

/* ---- inner native boundary: pymap2d ------------------------------------------------ */
/* render_contours_in_lidar(ranges, angles, flat, lidar_xy) (env.py:430-431) with the polygons
 * already flattened to closed segments segs[S][4], then CMap2D.render_agents_in_lidar
 * (env.py:432) with agents reduced to discs[D][3]; in-place min into ranges[K]. */
int navgym_render_in_lidar_host(float *ranges_host, const float *headings_host, int K,
                                const float *segs_host, int S, const float *discs_host, int D,
                                float ox, float oy);

/* ---- reset path (host only) --------------------------------------------------------- */
/* 4-connected BFS distance in cells over blocked[H][W] (non-zero = blocked), -1 where
 * unreachable: the uniform-cost stand-in for pyastar2d.astar_path (env.py:343-354) used to
 * precompute spawn pools. */
void navgym_grid_bfs(const uint8_t *blocked, int H, int W, int sr, int sc, int32_t *dist);

/* ---- misc -------------------------------------------------------------------------- */
const char *navgym_error_string(int code);
int navgym_device_count(void);
int navgym_abi_version(void);
/* 1: the march samples trunc(fmaf(dx, t, x0)) (canonical); 0: this build rounds dx * t and the
 * sum separately (-DNAVGYM_MARCH_NO_FMA; range_libc's own rounding is unknown, see DESIGN.md) */
int navgym_march_is_fused(void);
int navgym_sizeof_step_args(void);   /* layout check for FFI bindings */
int navgym_sizeof_map(void);
int navgym_sizeof_her_args(void);
int navgym_sizeof_peds_args(void);
/* kernels launched by this library since load (for bench.py's gpu_launches) */
uint64_t navgym_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif
