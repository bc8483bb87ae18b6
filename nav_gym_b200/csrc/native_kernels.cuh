// native_kernels.cuh -- part of navgym_b200.cu (included there; one translation unit).
// range_libc / pymap2d stand-ins: exact EDT build, calc_range_many, render_*_in_lidar.
// ------------------------------------------------------------------ EDT build kernels
// Pass 1: per column, distance to the nearest occupied cell of that column (coalesced in x).
__global__ void edt_columns_kernel(const uint8_t *__restrict__ occ, int H, int W, int32_t *__restrict__ g)
{
    int x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= W) return;
    int last = -1;
    for (int y = 0; y < H; y++) {
        if (occ[(size_t)y * W + x]) last = y;
        g[(size_t)y * W + x] = last < 0 ? EDT_INF_G : y - last;
    }
    last = -1;
    for (int y = H - 1; y >= 0; y--) {
        if (occ[(size_t)y * W + x]) last = y;
        int dn = last < 0 ? EDT_INF_G : last - y;
        size_t i = (size_t)y * W + x;
        if (dn < g[i]) g[i] = dn;
    }
}

// Pass 2: per row, exact integer minimisation d2(x) = min_q (x-q)^2 + g(q)^2 with the row in
// shared memory; the search window is |x-q| < g(x) (a farther q cannot beat q = x).
__global__ void edt_rows_kernel(const int32_t *__restrict__ g, int H, int W, float *__restrict__ dist)
{
    extern __shared__ int32_t row[];
    const int y = blockIdx.x;
    for (int x = threadIdx.x; x < W; x += blockDim.x) row[x] = g[(size_t)y * W + x];
    __syncthreads();
    for (int x = threadIdx.x; x < W; x += blockDim.x) {
        int gx = row[x];
        int best = gx * gx;  // <= 2^30
        int lo = max(0, x - gx + 1), hi = min(W - 1, x + gx - 1);
        for (int q = lo; q <= hi; q++) {
            int dq = x - q, gq = row[q];
            int v = dq * dq + gq * gq;
            best = min(best, v);
        }
        dist[(size_t)y * W + x] = __fsqrt_rn((float)best);
    }
}

// ------------------------------------------------------------------ stand-alone natives
__global__ void calc_range_many_kernel(const float *__restrict__ dist, int W, int H,
                                       const float *__restrict__ ins, float *__restrict__ outs, int N,
                                       float max_range, float t_stop, int16_t *__restrict__ hits)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    float x0 = ins[3 * i], y0 = ins[3 * i + 1], h = ins[3 * i + 2];
    double s, c;
    dir_sincos((double)h, s, c);
    int hx, hy;
    outs[i] = march(dist, W, H, x0, y0, (float)c, (float)s, max_range, t_stop, hx, hy);
    if (hits) { hits[2 * i] = (int16_t)hx; hits[2 * i + 1] = (int16_t)hy; }
}

__global__ void render_in_lidar_kernel(float *__restrict__ ranges, const float *__restrict__ headings,
                                       int K, const float *__restrict__ segs, int S,
                                       const float *__restrict__ discs, int D, float ox, float oy)
{
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= K) return;
    double s, c;
    dir_sincos((double)headings[k], s, c);
    float dx = (float)c, dy = (float)s, r = ranges[k];
    for (int i = 0; i < S; i++)
        r = fminf(r, seg_hit(ox, oy, dx, dy, segs[4 * i], segs[4 * i + 1], segs[4 * i + 2], segs[4 * i + 3]));
    for (int i = 0; i < D; i++)
        r = fminf(r, disc_hit(ox, oy, dx, dy, discs[3 * i], discs[3 * i + 1], discs[3 * i + 2]));
    ranges[k] = r;
}

// ------------------------------------------------------------------ host export of one env
// Everything the single-environment drop-in reads back per step (SURVEY 8f row 4), packed into
// one float64 row so that the host needs ONE device-to-host copy:
//   [0..NS) state rows | [NS..NS+7) tail64 | reward done is_success is_crash truncated distance
//   steps map_id episode noise_std | S*512 scan values (float32 or float16 -> float64, exact)
#define NAVGYM_EXPORT_HEAD (NAVGYM_NS + NAVGYM_OBS_TAIL + 10)
__global__ void export_env_kernel(const navgym_step_args_t a, int e, double *out)
{
    const int B = a.num_envs;
    const int SS = a.num_scan_stack > 1 ? a.num_scan_stack : 1;
    for (int i = threadIdx.x; i < NAVGYM_EXPORT_HEAD + SS * NB; i += blockDim.x) {
        double v = 0.0;
        if (i < NAVGYM_NS) v = a.state[(size_t)i * B + e];
        else if (i < NAVGYM_NS + NAVGYM_OBS_TAIL) v = a.tail64 ? a.tail64[(size_t)e * 7 + (i - NAVGYM_NS)] : 0.0;
        else if (i < NAVGYM_EXPORT_HEAD) {
            switch (i - NAVGYM_NS - NAVGYM_OBS_TAIL) {
            case 0: v = (double)a.reward[e]; break;
            case 1: v = (double)a.done[e]; break;
            case 2: v = (double)a.is_success[e]; break;
            case 3: v = (double)a.is_crash[e]; break;
            case 4: v = a.truncated ? (double)a.truncated[e] : 0.0; break;
            case 5: v = (double)a.distance[e]; break;
            case 6: v = (double)a.steps[e]; break;
            case 7: v = (double)a.map_id[e]; break;
            case 8: v = a.episodes ? (double)a.episodes[e] : 0.0; break;
            case 9: v = a.noise_std ? (double)a.noise_std[e] : 0.0; break;
            }
        } else v = (double)obs_scan_at(a.obs, a.obs_format, e, a.obs_stride, i - NAVGYM_EXPORT_HEAD);
        out[i] = v;
    }
}
