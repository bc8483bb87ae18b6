// navgym_b200.cu — sm_100a kernels + C ABI for nav-gym's NavGym-v0 per-step hot path.
//
// Written from scratch for B200; the reference (leekwoon/nav-gym) has no GPU code.  What each
// piece replaces (paths relative to /root/reference/nav_gym/src/nav_gym_env/):
//   step_kernel          NavGymEnv.step            env.py:591-728 (robot branch)
//     kinematics         KetiRobot.set_vel         keti_robot.py:64-93
//     scan               NavGymEnv._compute_scan   env.py:385-441
//       march            range_libc calc_range_many (third party, call site env.py:425)
//       segments/discs   pymap2d render_contours_in_lidar / render_agents_in_lidar
//                                                  (third party, call sites env.py:430-432)
//     observation        _convert_obs              env.py:443-462
//     reward/done/info   compute_rewards/terminals/info   env.py:464-589
//     rollback           env.py:707-723
//   edt_*_kernel         range_libc PyOMap + PyRayMarching ctor   env.py:337-340
//
// Floating-point contract (DESIGN.md): compiled with -fmad=false; every arithmetic step that
// feeds an integer result (cells, hit cells, flags) is a single IEEE rounding, spelled with
// __f*_rn intrinsics where it matters, fmaf only where the contract says fused.
//
// One translation unit; the kernels live in the files included below:
//   device_helpers.cuh      cell mapping, canonical beam direction / march / segment / disc, Philox
//   step_kernel.cuh         the fused step: one CTA = one environment, 2 warps, pass loop
//   her_kernel.cuh          compute_rewards / terminals / info on stored observations
//   pedestrian_kernels.cuh  pedestrians' lidar, routes, motion, geometry
//   native_kernels.cuh      EDT build, calc_range_many, render_in_lidar
//   host_pipe.inl           host-buffer entry points (chunked / asynchronous, CUDA-graph replay)
// and this file holds the C ABI (include/navgym_b200.h) around them.
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <math_constants.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <mutex>
#include <type_traits>

#include "../../include/navgym_b200.h"

#define NB NAVGYM_NUM_BEAMS
#define OBS_DIM (NB + NAVGYM_OBS_TAIL)
#define HIT_NONE NAVGYM_HIT_NONE
#define EDT_INF_G 32768

static unsigned long long g_launches = 0;

#include "device_helpers.cuh"
#include "step_kernel.cuh"
#include "her_kernel.cuh"
#include "pedestrian_kernels.cuh"
#include "native_kernels.cuh"
#include "policy_gemm.cuh"

// ------------------------------------------------------------------ C ABI
// SM count of the current device (a B200's 148 when the query fails).
static int sm_count()
{
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0)
        return 148;
    return sms;
}

// Launch shape of the fused kernel: one 64-thread CTA per environment of the launch.
template <int MODE, int FMT>
static void launch_step_fmt(const navgym_step_args_t &a, const uint8_t *mask, int count, bool coop, cudaStream_t st)
{
    if constexpr (MODE == MODE_MASKED_RESET) {
        if (coop) reset_envs_kernel<true, FMT><<<count, NAVGYM_CTA_THREADS, 0, st>>>(a, mask);
        else reset_envs_kernel<false, FMT><<<count, NAVGYM_CTA_THREADS, 0, st>>>(a, mask);
    } else {
        if (coop) step_kernel<MODE, true, FMT><<<count, NAVGYM_CTA_THREADS, 0, st>>>(a);
        else step_kernel<MODE, false, FMT><<<count, NAVGYM_CTA_THREADS, 0, st>>>(a);
    }
}

// The obstacle windows of an environment are parked in NB / 2 shared-memory slots.
static bool obstacle_slots_ok(int max_disc, int max_seg, const void *discs, const void *segs)
{
    return (discs ? max_disc : 0) + (segs ? max_seg : 0) <= NB / 2;
}

// MODE_STEP / MODE_RESET / MODE_MASKED_RESET (step_kernel.cuh) over the launch's env range, which
// step_args_ok has accepted; `mask` is read by the masked reset only.  A step with auto_reset ==
// NAVGYM_AUTORESET_NEXT_STEP runs MODE_NEXT_STEP.  An empty range launches nothing.
template <int MODE>
static cudaError_t launch_step(const navgym_step_args_t &a, cudaStream_t st, const uint8_t *mask = nullptr)
{
    const int count = a.env_count > 0 ? a.env_count : a.num_envs - a.env_begin;
    if (count == 0) return cudaSuccess;
    // tail regime B (see step_kernel) while the launch is at most ~2.4 waves of CTAs (measured
    // crossover on B200: 5120 envs -2 %, 6144 envs +2 %)
    static const int coop_max = (int)(2.4 * sm_count() * NAVGYM_CTAS_PER_SM);
    const bool coop = count <= coop_max, f16 = a.obs_format == NAVGYM_OBS_F16;
    if (MODE == MODE_STEP && a.auto_reset == NAVGYM_AUTORESET_NEXT_STEP) {
        if (f16) launch_step_fmt<MODE_NEXT_STEP, NAVGYM_OBS_F16>(a, mask, count, coop, st);
        else launch_step_fmt<MODE_NEXT_STEP, NAVGYM_OBS_F32>(a, mask, count, coop, st);
    } else if (f16) {
        launch_step_fmt<MODE, NAVGYM_OBS_F16>(a, mask, count, coop, st);
    } else {
        launch_step_fmt<MODE, NAVGYM_OBS_F32>(a, mask, count, coop, st);
    }
    g_launches++;
    return cudaGetLastError();
}

// Observation rows (include/navgym_b200.h NAVGYM_OBS_*): a known format, a stride that holds S
// scans and the tail, and for float16 rows an even stride and a 4-byte aligned base (the tail is
// stored as float32).  `obs` is the row storage the call reads or writes.
static bool obs_rows_ok(int format, int stride, int num_scan_stack, const void *obs)
{
    const int scans = (num_scan_stack > 1 ? num_scan_stack : 1) * NB;
    if (format == NAVGYM_OBS_F32) return stride >= scans + NAVGYM_OBS_TAIL;
    if (format == NAVGYM_OBS_F16)
        return stride % 2 == 0 && stride >= scans + 2 * NAVGYM_OBS_TAIL && ((uintptr_t)obs & 3) == 0;
    return false;
}

// What every entry point taking a navgym_step_args_t rejects (include/navgym_b200.h): malformed
// obs rows, an env range outside [0, num_envs), a negative env_count, too many obstacle slots.
static bool step_args_ok(const navgym_step_args_t *a)
{
    return obs_rows_ok(a->obs_format, a->obs_stride, a->num_scan_stack, a->obs) && a->env_begin >= 0 &&
           a->env_begin <= a->num_envs && a->env_count >= 0 && a->env_count <= a->num_envs - a->env_begin &&
           obstacle_slots_ok(a->max_disc, a->max_seg, a->discs, a->segs);
}

#define CK(x) do { cudaError_t _e = (x); if (_e != cudaSuccess) return (int)_e; } while (0)

extern "C" {

#ifdef NAVGYM_PROFILE
int navgym_debug_read_prof(unsigned long long *out, int reset)
{
    cudaError_t e = cudaMemcpyFromSymbol(out, g_prof, sizeof(unsigned long long) * 16);
    if (!e && reset) { unsigned long long z[16] = {0}; e = cudaMemcpyToSymbol(g_prof, z, sizeof(z)); }
    return (int)e;
}
#endif

int navgym_abi_version(void) { return 1; }
int navgym_march_is_fused(void)
{
#ifdef NAVGYM_MARCH_NO_FMA
    return 0;
#else
    return 1;
#endif
}
int navgym_sizeof_step_args(void) { return (int)sizeof(navgym_step_args_t); }
int navgym_sizeof_map(void) { return (int)sizeof(navgym_map_t); }
int navgym_sizeof_her_args(void) { return (int)sizeof(navgym_her_args_t); }
int navgym_sizeof_peds_args(void) { return (int)sizeof(navgym_peds_args_t); }
uint64_t navgym_launch_count(void) { return g_launches; }
const char *navgym_error_string(int code) { return cudaGetErrorString((cudaError_t)code); }
int navgym_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

int navgym_step_batch(const navgym_step_args_t *args, void *stream)
{
    if (args->num_envs <= 0) return 0;
    if (!step_args_ok(args)) return (int)cudaErrorInvalidValue;
    return (int)launch_step<MODE_STEP>(*args, (cudaStream_t)stream);
}

#include "host_pipe.inl"

int navgym_reset_obs_batch(const navgym_step_args_t *args, void *stream)
{
    if (args->num_envs <= 0) return 0;
    if (!step_args_ok(args)) return (int)cudaErrorInvalidValue;
    return (int)launch_step<MODE_RESET>(*args, (cudaStream_t)stream);
}

int navgym_reset_envs(const navgym_step_args_t *args, const uint8_t *mask, void *stream)
{
    if (args->num_envs <= 0) return 0;
    // (the masked reset may scan the next episode's geometry alone)
    if (!mask || !step_args_ok(args) || !obstacle_slots_ok(args->max_disc, args->max_seg, args->discs_reset, args->segs_reset))
        return (int)cudaErrorInvalidValue;
    return (int)launch_step<MODE_MASKED_RESET>(*args, (cudaStream_t)stream, mask);
}

int navgym_export_env_len(int num_scan_stack)
{
    return NAVGYM_EXPORT_HEAD + (num_scan_stack > 1 ? num_scan_stack : 1) * NB;
}

int navgym_export_env(const navgym_step_args_t *args, int env, double *out_dev, void *stream)
{
    if (!step_args_ok(args) || env < 0 || env >= args->num_envs || !out_dev) return (int)cudaErrorInvalidValue;
    export_env_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(*args, env, out_dev);
    g_launches++;
    return (int)cudaGetLastError();
}

int navgym_compute_rewards(const navgym_her_args_t *args, void *stream)
{
    if (args->count <= 0) return 0;
    if (!obs_rows_ok(args->obs_format, args->obs_stride, args->num_scan_stack, args->obs))
        return (int)cudaErrorInvalidValue;
    // warps stride over the rows: at most one full wave of CTAs
    static const int sms = sm_count();
    const int warps_per_cta = NAVGYM_HER_THREADS / 32;
    const int want = (args->count + warps_per_cta - 1) / warps_per_cta;
    const int ctas = want < sms * HER_CTAS_PER_SM ? want : sms * HER_CTAS_PER_SM;
    if (args->obs_format == NAVGYM_OBS_F16)
        her_kernel<NAVGYM_OBS_F16><<<ctas, NAVGYM_HER_THREADS, 0, (cudaStream_t)stream>>>(*args);
    else
        her_kernel<NAVGYM_OBS_F32><<<ctas, NAVGYM_HER_THREADS, 0, (cudaStream_t)stream>>>(*args);
    g_launches++;
    return (int)cudaGetLastError();
}

int navgym_peds_advance(const navgym_peds_args_t *args, void *stream)
{
    if (args->num_envs <= 0) return 0;
    // rows of 16 floats are moved as four 16-byte words, box segments stored as float4
    if (((uintptr_t)args->peds & 15) || ((uintptr_t)args->segs & 15)) return (int)cudaErrorMisalignedAddress;
    peds_advance_kernel<<<(args->num_envs + 3) / 4, 128, 0, (cudaStream_t)stream>>>(*args);  // a warp per environment
    g_launches++;
    return (int)cudaGetLastError();
}

int navgym_sizeof_scan_args(void) { return (int)sizeof(navgym_scan_args_t); }
int navgym_sizeof_plan_args(void) { return (int)sizeof(navgym_plan_args_t); }
int navgym_sizeof_plan_map(void) { return (int)sizeof(navgym_plan_map_t); }
int navgym_sizeof_move_args(void) { return (int)sizeof(navgym_move_args_t); }

// ---- the pedestrian policy as one native pipeline (include/navgym_b200.h, navgym_policy_*)
size_t navgym_policy_workspace_bytes(int max_n) { return policy_ws_layout(max_n).total; }
int navgym_sizeof_policy_params(void) { return (int)sizeof(navgym_policy_params_t); }

navgym_policy_t *navgym_policy_create(const navgym_policy_params_t *p, void *stream)
{
    if (!p || p->max_n <= 0 || !p->workspace || !p->cv1_w || !p->cv1_b || !p->cv2_w || !p->cv2_b || !p->fc1_w ||
        !p->fc1_b || !p->fc2_w || !p->fc2_b || !p->a1_w || !p->a1_b || !p->a2_w || !p->a2_b)
        return nullptr;
    const policy_ws_t L = policy_ws_layout(p->max_n);
    if (p->workspace_bytes < L.total || ((uintptr_t)p->workspace & 1023)) return nullptr;
    navgym_policy_t *pol = new navgym_policy_t();
    pol->max_n = p->max_n;
    pol->ws = (uint8_t *)p->workspace;
    pol->L = L;
    cudaGetDevice(&pol->device);
    pol->sms = sm_count();
    const uint64_t np = ((uint64_t)p->max_n + 127) / 128 * 128;
    cudaStream_t st = (cudaStream_t)stream;
    bool ok = cudaMemsetAsync(pol->ws + L.fh, 0, (size_t)np * 4096 * 2, st) == cudaSuccess &&
              cudaMemsetAsync(pol->ws + L.fl, 0, (size_t)np * 4096 * 2, st) == cudaSuccess;
    ok = ok && cudaMemsetAsync(pol->ws + L.hh, 0, (size_t)np * 256 * 2, st) == cudaSuccess &&
         cudaMemsetAsync(pol->ws + L.hl, 0, (size_t)np * 256 * 2, st) == cudaSuccess;
    ok = ok && policy_make_map(&pol->tm_fh, pol->ws + L.fh, np, pg::BM, 4096) == 0 &&
         policy_make_map(&pol->tm_fl, pol->ws + L.fl, np, pg::BM, 4096) == 0 &&
         policy_make_map(&pol->tm_wh, pol->ws + L.wh, 256, pg::Fc1::WBOX, 4096) == 0 &&
         policy_make_map(&pol->tm_wl, pol->ws + L.wl, 256, pg::Fc1::WBOX, 4096) == 0 &&
         policy_make_map(&pol->tm_hh, pol->ws + L.hh, np, pg::BM, 256) == 0 &&
         policy_make_map(&pol->tm_hl, pol->ws + L.hl, np, pg::BM, 256) == 0 &&
         policy_make_map(&pol->tm_w2h, pol->ws + L.w2h, 128, 128, 256) == 0 &&
         policy_make_map(&pol->tm_w2l, pol->ws + L.w2l, 128, 128, 256) == 0;
    ok = ok && cudaFuncSetAttribute(dense_umma_kernel<pg::Fc1, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, pg::Fc1::SMEM_BYTES) == cudaSuccess &&
         cudaFuncSetAttribute(dense_umma_kernel<pg::Fc2, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, pg::Fc2::SMEM_BYTES) == cudaSuccess &&
         cudaFuncSetAttribute(policy_features_umma2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, pf::SMEM_BYTES) == cudaSuccess;
    if (ok) {
        policy_prepare_kernel<<<1, 1024, 0, st>>>(*p, pol->ws, L);
        g_launches++;
        ok = cudaGetLastError() == cudaSuccess;
    }
    if (!ok) { delete pol; return nullptr; }
    return pol;
}

void navgym_policy_destroy(navgym_policy_t *pol) { delete pol; }

int navgym_policy_mean(navgym_policy_t *pol, const float *scan, const float *goal, const float *speed, int n,
                       float *mean, void *stream)
{
    if (!pol) return (int)cudaErrorInvalidValue;
    if (n <= 0) return 0;
    if (n > pol->max_n || !scan || !goal || !speed || !mean) return (int)cudaErrorInvalidValue;
    cudaStream_t st = (cudaStream_t)stream;
    uint8_t *ws = pol->ws;
    const policy_ws_t &L = pol->L;
    const float *scales = (const float *)(ws + L.scales);
    // front end (both convolutions), act_fc1, then act_fc2 + heads: all on the tensor cores
    policy_features_umma2_kernel<<<n < pol->sms ? n : pol->sms, pf::THREADS, pf::SMEM_BYTES, st>>>(
        scan, n, (const uint4 *)(ws + L.conv1_img), (const uint4 *)(ws + L.conv2_img), (const float *)(ws + L.b2), scales,
        (__half *)(ws + L.fh), (__half *)(ws + L.fl));
    const int tiles = (n + pg::BM - 1) / pg::BM, grid = tiles < pol->sms ? tiles : pol->sms;
    dense_umma_kernel<pg::Fc1, 0><<<grid, pg::THREADS, pg::Fc1::SMEM_BYTES, st>>>(
        pol->tm_fh, pol->tm_fl, pol->tm_wh, pol->tm_wl, (const float *)(ws + L.fc1_b), scales, n, tiles,
        (__half *)(ws + L.hh), (__half *)(ws + L.hl), nullptr, nullptr, nullptr);
    dense_umma_kernel<pg::Fc2, 1><<<grid, pg::THREADS, pg::Fc2::SMEM_BYTES, st>>>(
        pol->tm_hh, pol->tm_hl, pol->tm_w2h, pol->tm_w2l, (const float *)(ws + L.fc2_tab), scales, n, tiles,
        nullptr, nullptr, goal, speed, mean);
    g_launches += 3;
    return (int)cudaGetLastError();
}

/* test hook: byte offsets of the intermediate buffers inside the workspace */
void navgym_policy_workspace_layout(int max_n, uint64_t *out /* [6]: fh, fl, scales, total, hh, hl */)
{
    const policy_ws_t L = policy_ws_layout(max_n);
    out[0] = L.fh; out[1] = L.fl; out[2] = L.scales; out[3] = L.total; out[4] = L.hh; out[5] = L.hl;
}

int navgym_peds_move(const navgym_move_args_t *args, void *stream)
{
    const int n = args->num_envs * args->max_ped;
    if (n <= 0) return 0;
    if (!args->mean || !args->v_pref || !args->has_legs || !args->pose || !args->vel || !args->dist_travelled ||
        !args->prev_action || !args->rows)
        return (int)cudaErrorInvalidValue;
    peds_move_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(*args);
    g_launches++;
    return (int)cudaGetLastError();
}

int navgym_peds_plan(const navgym_plan_args_t *args, void *stream)
{
    const int n = args->num_envs * args->max_ped;
    if (n <= 0) return 0;
    if (!args->maps || !args->fields || !args->goals || !args->pose || !args->goal_id || !args->waypoint || !args->goal_local)
        return (int)cudaErrorInvalidValue;
    if (args->cand_pose && (!args->free_xy || !args->robot_state || !args->pose_rw || !args->v_pref || !args->has_legs ||
                            !args->dist_travelled || !args->vel || !args->prev_action || !args->cand_v_pref ||
                            !args->cand_legs || !args->cand_goal || !args->cand_rows))
        return (int)cudaErrorInvalidValue;
    const int lo = args->num_humans_lo, hi = args->num_humans_hi;
    if (lo < 0 || lo > hi || hi > args->max_ped) return (int)cudaErrorInvalidValue;
    // per-episode counts: the launch reads nped / cand_nped_prev and writes the other two
    if (hi > 0 && (!args->nped || !args->cand_pose || !args->cand_nped_prev || !args->cand_nped || !args->nped_out ||
                   (const void *)args->nped_out == (const void *)args->nped ||
                   (const void *)args->cand_nped == (const void *)args->cand_nped_prev))
        return (int)cudaErrorInvalidValue;
    if (hi > 0)
        peds_plan_kernel<true><<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(*args);
    else
        peds_plan_kernel<false><<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(*args);
    g_launches++;
    return (int)cudaGetLastError();
}

int navgym_agent_scan_batch(const navgym_scan_args_t *args, void *stream)
{
    if (args->num_envs <= 0 || args->agents_per_env <= 0) return 0;
    if (args->num_beams <= 0 || !args->pose || !args->lin || !args->ranges) return (int)cudaErrorInvalidValue;
    // crowd mode: one thread per other agent stages its footprint in a fixed shared-memory list
    const bool crowd = !args->segs && args->robot_state;
    if (crowd && args->agents_per_env > NAVGYM_SCAN_AGENTS) return (int)cudaErrorInvalidValue;
    if (crowd || !args->segs || args->max_seg <= NAVGYM_SCAN_SEGS)
        agent_scan_kernel<<<args->num_envs * args->agents_per_env, 128, 0, (cudaStream_t)stream>>>(*args);
    else   // longer segment lists: every segment against every beam, straight from global memory
        agent_scan_generic_kernel<<<args->num_envs * args->agents_per_env, 128, 0, (cudaStream_t)stream>>>(*args);
    g_launches++;
    return (int)cudaGetLastError();
}

int navgym_edt_build(const uint8_t *occ_dev, int H, int W, float *dist_dev, int32_t *scratch_dev, void *stream)
{
    // W: one row of int32 in the default 48 KB of dynamic shared memory; H: hit cells travel as
    // (y << 16 | x) through the march
    if (H <= 0 || W <= 0 || W > 12000 || H > 32767) return (int)cudaErrorInvalidValue;
    cudaStream_t st = (cudaStream_t)stream;
    edt_columns_kernel<<<(W + 127) / 128, 128, 0, st>>>(occ_dev, H, W, scratch_dev);
    edt_rows_kernel<<<H, 256, (size_t)W * sizeof(int32_t), st>>>(scratch_dev, H, W, dist_dev);
    g_launches += 2;
    return (int)cudaGetLastError();
}

int navgym_calc_range_many(const float *dist_dev, int W, int H, const float *ins_dev, float *outs_dev,
                           int N, float max_range, float t_stop, int16_t *hits_dev, void *stream)
{
    if (N <= 0) return 0;
    calc_range_many_kernel<<<(N + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
        dist_dev, W, H, ins_dev, outs_dev, N, max_range, t_stop, hits_dev);
    g_launches++;
    return (int)cudaGetLastError();
}

// Scratch of the host-buffer natives: one grow-only device buffer and one pinned staging buffer
// per device, reused from call to call (the reference calls these natives 1 + num_humans times per
// step: a cudaMalloc / cudaFree pair and four pageable copies per call cost several times the
// kernel).  Calls are serialised by a mutex, like the GIL-holding originals.
struct host_scratch {
    float *dev = nullptr, *pin = nullptr;
    size_t cap = 0;
};
static std::mutex g_scratch_mutex;
static host_scratch g_scratch[64];
static cudaError_t scratch_for(size_t nfloats, host_scratch *&out)
{
    int dev = 0;
    cudaError_t err = cudaGetDevice(&dev);
    if (err) return err;
    if (dev < 0 || dev >= 64) return cudaErrorInvalidDevice;
    host_scratch &s = g_scratch[dev];
    if (s.cap < nfloats) {
        if (s.dev) cudaFree(s.dev);
        if (s.pin) cudaFreeHost(s.pin);
        s.dev = s.pin = nullptr;
        s.cap = 0;
        size_t cap = 4096;
        while (cap < nfloats) cap *= 2;
        err = cudaMalloc(&s.dev, cap * sizeof(float));
        if (!err) err = cudaMallocHost(&s.pin, cap * sizeof(float));
        if (err) {
            if (s.dev) cudaFree(s.dev);
            s.dev = nullptr;
            return err;
        }
        s.cap = cap;
    }
    out = &s;
    return cudaSuccess;
}

int navgym_render_in_lidar_host(float *ranges_host, const float *headings_host, int K,
                                const float *segs_host, int S, const float *discs_host, int D,
                                float ox, float oy)
{
    if (K <= 0) return 0;
    if (S < 0 || D < 0) return (int)cudaErrorInvalidValue;
    std::lock_guard<std::mutex> lock(g_scratch_mutex);
    const size_t nf = (size_t)2 * K + (size_t)4 * S + (size_t)3 * D;
    host_scratch *sc = nullptr;
    CK(scratch_for(nf, sc));
    // one staged copy in: [ranges | headings | segments | discs]
    float *r = sc->dev, *hd = r + K, *sg = hd + K, *dc = sg + 4 * (size_t)S;
    memcpy(sc->pin, ranges_host, K * sizeof(float));
    memcpy(sc->pin + K, headings_host, K * sizeof(float));
    if (S) memcpy(sc->pin + 2 * (size_t)K, segs_host, (size_t)4 * S * sizeof(float));
    if (D) memcpy(sc->pin + 2 * (size_t)K + 4 * (size_t)S, discs_host, (size_t)3 * D * sizeof(float));
    CK(cudaMemcpyAsync(sc->dev, sc->pin, nf * sizeof(float), cudaMemcpyHostToDevice, 0));
    render_in_lidar_kernel<<<(K + 127) / 128, 128>>>(r, hd, K, sg, S, dc, D, ox, oy);
    g_launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(sc->pin, r, K * sizeof(float), cudaMemcpyDeviceToHost, 0));
    CK(cudaStreamSynchronize(0));
    memcpy(ranges_host, sc->pin, K * sizeof(float));
    return 0;
}

struct navgym_raymarching {
    int H, W;
    float max_range;
    float *dist;
};

navgym_raymarching_t *navgym_raymarching_create_host(const uint8_t *occ_host, int H, int W, float max_range)
{
    uint8_t *occ = nullptr;
    int32_t *scratch = nullptr;
    float *dist = nullptr;
    size_t n = (size_t)H * W;
    if (cudaMalloc(&occ, n) != cudaSuccess) return nullptr;
    if (cudaMalloc(&scratch, n * sizeof(int32_t)) != cudaSuccess) { cudaFree(occ); return nullptr; }
    if (cudaMalloc(&dist, n * sizeof(float)) != cudaSuccess) { cudaFree(occ); cudaFree(scratch); return nullptr; }
    cudaError_t err = cudaMemcpy(occ, occ_host, n, cudaMemcpyHostToDevice);
    if (!err) err = (cudaError_t)navgym_edt_build(occ, H, W, dist, scratch, nullptr);
    if (!err) err = cudaDeviceSynchronize();
    cudaFree(occ);
    cudaFree(scratch);
    if (err) { cudaFree(dist); return nullptr; }
    navgym_raymarching_t *rm = new navgym_raymarching_t{H, W, max_range, dist};
    return rm;
}

int navgym_raymarching_calc_range_many_host(navgym_raymarching_t *rm, const float *ins_host,
                                            float *outs_host, int N)
{
    if (!rm) return (int)cudaErrorInvalidValue;
    if (N <= 0) return 0;
    std::lock_guard<std::mutex> lock(g_scratch_mutex);
    host_scratch *sc = nullptr;
    CK(scratch_for((size_t)4 * N, sc));
    memcpy(sc->pin, ins_host, (size_t)3 * N * sizeof(float));
    CK(cudaMemcpyAsync(sc->dev, sc->pin, (size_t)3 * N * sizeof(float), cudaMemcpyHostToDevice, 0));
    const int lerr = navgym_calc_range_many(rm->dist, rm->W, rm->H, sc->dev, sc->dev + 3 * (size_t)N, N,
                                            rm->max_range, rm->max_range, nullptr, nullptr);
    if (lerr) return lerr;
    CK(cudaMemcpyAsync(sc->pin + 3 * (size_t)N, sc->dev + 3 * (size_t)N, (size_t)N * sizeof(float),
                       cudaMemcpyDeviceToHost, 0));
    CK(cudaStreamSynchronize(0));
    memcpy(outs_host, sc->pin + 3 * (size_t)N, (size_t)N * sizeof(float));
    return 0;
}

// Reset-path host helper (no device work): 4-connected BFS distance over a grid, the
// uniform-cost equivalent of pyastar2d.astar_path (reference env.py:343-354).
void navgym_grid_bfs(const uint8_t *blocked, int H, int W, int sr, int sc, int32_t *dist)
{
    size_t n = (size_t)H * W;
    for (size_t i = 0; i < n; i++) dist[i] = -1;
    if (sr < 0 || sc < 0 || sr >= H || sc >= W || blocked[(size_t)sr * W + sc]) return;
    int32_t *queue = new int32_t[n];
    size_t head = 0, tail = 0;
    queue[tail++] = sr * W + sc;
    dist[(size_t)sr * W + sc] = 0;
    const int dr[4] = {1, -1, 0, 0}, dc[4] = {0, 0, 1, -1};
    while (head < tail) {
        int32_t cur = queue[head++];
        int r = cur / W, c = cur % W;
        for (int k = 0; k < 4; k++) {
            int nr = r + dr[k], nc = c + dc[k];
            if (nr < 0 || nc < 0 || nr >= H || nc >= W) continue;
            size_t ni = (size_t)nr * W + nc;
            if (blocked[ni] || dist[ni] >= 0) continue;
            dist[ni] = dist[cur] + 1;
            queue[tail++] = (int32_t)ni;
        }
    }
    delete[] queue;
}

const float *navgym_raymarching_edt_dev(const navgym_raymarching_t *rm) { return rm ? rm->dist : nullptr; }

int navgym_raymarching_edt_host(const navgym_raymarching_t *rm, float *out_host)
{
    if (!rm) return (int)cudaErrorInvalidValue;
    return (int)cudaMemcpy(out_host, rm->dist, (size_t)rm->H * rm->W * sizeof(float), cudaMemcpyDeviceToHost);
}

void navgym_raymarching_destroy(navgym_raymarching_t *rm)
{
    if (!rm) return;
    cudaFree(rm->dist);
    delete rm;
}

}  // extern "C"
