// her_kernel.cuh -- part of navgym_b200.cu (included there; one translation unit).
// compute_rewards / compute_terminals / compute_info on stored observations (env.py:464-589).
// ------------------------------------------------------------------ HER batch API
// compute_rewards / compute_terminals / compute_info on a batch of stored observations
// (env.py:464-589: the reference's hindsight-relabelling entry points).  Observation row
// [scan(512) | prev_pose(2) pose(2) vel(2) yaw(1)], goals given separately.
//
// HBM-bound: 2095 algorithmic bytes per row (2076 row + 8 goal in, 11 out) against ~250 instructions;
// with float16 scans (FMT = NAVGYM_OBS_F16) 1075 (a 1056-byte row).
// One warp per row at a time, warps striding over the rows: lane l owns 16 beams, whose thresholds
// stay in its registers for every row the warp handles -- beams l + 32 i of float32 rows, the two
// beams of half2 words l + 32 i of float16 rows; the row loads of a lane are independent streaming
// loads (128 contiguous bytes per warp and load; rows are consumed once and should not displace
// anything in L2), 32 warps per SM keep 64 KB (float16: 32 KB) in flight.  The discomfort ratio
// min_k (scan_k - thr_k) / (dthr_k - thr_k + 1e-6) -- 512 float64 divisions -- is only evaluated for
// rows that are in discomfort (a warp-uniform branch), from the row already in registers; the two
// goal distances are taken by lanes 0 and 1 side by side.  Crash, discomfort and the minimum do not
// depend on which lane holds which beam, so both formats give the results of the float32 values.
#define NAVGYM_HER_THREADS 256
constexpr int HER_CTAS_PER_SM = 4;
template <int FMT>
__device__ __forceinline__ int her_beam(int lane, int i)
{
    return FMT == NAVGYM_OBS_F16 ? 2 * (lane + 32 * (i >> 1)) + (i & 1) : lane + 32 * i;
}

template <int FMT>
__global__ void __launch_bounds__(NAVGYM_HER_THREADS, HER_CTAS_PER_SM) her_kernel(const navgym_her_args_t a)
{
    constexpr int BPL = NB / 32;
    const int lane = threadIdx.x & 31;
    const int warps_per_cta = blockDim.x >> 5;
    const int stride = (int)gridDim.x * warps_per_cta;
    const unsigned FULL = 0xffffffffu;
    const int SS = a.num_scan_stack > 1 ? a.num_scan_stack : 1;
    float thr[BPL], dthr[BPL];
#pragma unroll
    for (int i = 0; i < BPL; i++) {
        thr[i] = a.thr[her_beam<FMT>(lane, i)];
        dthr[i] = a.dthr[her_beam<FMT>(lane, i)];
    }
    for (int n = blockIdx.x * warps_per_cta + (threadIdx.x >> 5); n < a.count; n += stride) {
        using Row = ObsRow<FMT, const float>;
        const typename Row::E *o = Row(a.obs, (size_t)n, a.obs_stride).p + (size_t)(SS - 1) * NB;   // the newest scan
        float v[BPL];
        if constexpr (FMT == NAVGYM_OBS_F16) {
#pragma unroll
            for (int i = 0; i < BPL / 2; i++) {
                const float2 f = __half22float2(__ldcs(reinterpret_cast<const __half2 *>(o) + lane + 32 * i));
                v[2 * i] = f.x;
                v[2 * i + 1] = f.y;
            }
        } else {
#pragma unroll
            for (int i = 0; i < BPL; i++) v[i] = __ldcs(o + lane + 32 * i);
        }
        // lanes 0..5: prev_pose(2) pose(2) vel(2); lanes 6, 7: the goal
        float tv = 0.0f;
        if (lane < 6) tv = __ldcs(Row::tail_after(o) + lane);
        else if (lane < 8) tv = __ldcs(a.goals + 2 * (size_t)n + (lane - 6));
        bool c_any = false, d_any = false;
#pragma unroll
        for (int i = 0; i < BPL; i++) {
            c_any |= v[i] < thr[i];
            d_any |= v[i] < dthr[i];
        }
        const int crash = __any_sync(FULL, c_any);
        const int discomf = __any_sync(FULL, d_any) && !crash;
        double mn = CUDART_INF;
        if (discomf) {
#pragma unroll
            for (int i = 0; i < BPL; i++) {   // (fully unrolled: v / thr / dthr stay in registers)
                const float den = __fadd_rn(__fsub_rn(dthr[i], thr[i]), 1e-6f);
                mn = fmin(mn, __ddiv_rn(__dsub_rn((double)v[i], (double)thr[i]), (double)den));
            }
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) mn = fmin(mn, __shfl_xor_sync(FULL, mn, off));
        }
        // lane 0: distance from pose to the goal; lane 1: from prev_pose
        const double gx = (double)__shfl_sync(FULL, tv, 6), gy = (double)__shfl_sync(FULL, tv, 7);
        const double qx = (double)__shfl_sync(FULL, tv, lane == 0 ? 2 : 0);
        const double qy = (double)__shfl_sync(FULL, tv, lane == 0 ? 3 : 1);
        const double pv = (double)__shfl_sync(FULL, tv, 4), pw = (double)__shfl_sync(FULL, tv, 5);
        const double ddx = __dsub_rn(gx, qx), ddy = __dsub_rn(gy, qy);
        const double dq = sqrt(__dadd_rn(__dmul_rn(ddx, ddx), __dmul_rn(ddy, ddy)));
        const double dist = __shfl_sync(FULL, dq, 0), pdist = __shfl_sync(FULL, dq, 1);
        if (lane == 0) {
            const int success = dist < a.dist_thresh;
            double r_s = success ? __dmul_rn(__dmul_rn(1.0, a.r_success), a.r_scale) : 0.0;
            double r_c = crash ? __dmul_rn(__dmul_rn(-1.0, a.r_crash), a.r_scale) : 0.0;
            double r_p = __dmul_rn(__dmul_rn(__dsub_rn(pdist, dist), a.r_progress), a.r_scale);
            double r_f = __dmul_rn(__dmul_rn(pv, a.r_forward), a.r_scale);
            double r_r = __dmul_rn(__dmul_rn(__dmul_rn(-1.0, __dmul_rn(pw, pw)), a.r_rotation), a.r_scale);
            double r_d = discomf ? __dmul_rn(__dmul_rn(-__dsub_rn(1.0, mn), a.r_discomfort), a.r_scale) : 0.0;
            if (a.reward)
                a.reward[n] = (float)__dadd_rn(__dadd_rn(__dadd_rn(__dadd_rn(__dadd_rn(r_s, r_c), r_p), r_f), r_r), r_d);
            if (a.done) a.done[n] = (uint8_t)(success || crash);
            if (a.is_success) a.is_success[n] = (uint8_t)success;
            if (a.is_crash) a.is_crash[n] = (uint8_t)crash;
            if (a.distance) a.distance[n] = (float)dist;
        }
    }
}
