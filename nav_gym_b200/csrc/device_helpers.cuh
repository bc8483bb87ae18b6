// device_helpers.cuh -- part of navgym_b200.cu (included there; one translation unit).
// Device helpers shared by every kernel: cell mapping, the canonical beam direction, the
// canonical march / segment / disc arithmetic (DESIGN.md section 2), Philox.
// ------------------------------------------------------------------ small device helpers
__device__ __forceinline__ int xy_to_cell(float x32, double origin, double res, int dim, int rule)
{
    // batch_xy_to_ij, env.py:1235-1253 (rule 0: NumPy-1.x float64 division; 1: NumPy-2 float32)
    float c;
    if (rule == 0)
        c = (float)__ddiv_rn(__dsub_rn((double)x32, origin), res);
    else
        c = __fdiv_rn(__fsub_rn(x32, (float)origin), (float)res);
    if (c >= (float)dim) c = (float)(dim - 1);
    if (c < 0.0f) c = 0.0f;
    return __float2int_rz(c);
}

// cos / sin of a beam heading, canonical form (DESIGN.md "beam direction"): Cody-Waite
// reduction by pi/2 in two fma steps, fdlibm kernel polynomials in Horner/fma form, quadrant
// fix-up.  A fixed sequence of IEEE operations, so the direction depends on the heading bits
// only (the CPU oracle evaluates the same sequence) — and ~5x fewer instructions than the
// full-range sincos() of the CUDA math library.
__device__ __forceinline__ void dir_sincos(double x, double &sn, double &cs)
{
    const double k = rint(__dmul_rn(x, 6.36619772367581382433e-01));
    double r = fma(-k, 1.57079632679489655800e+00, x);
    r = fma(-k, 6.12323399573676603587e-17, r);
    const double z = __dmul_rn(r, r);
    double ps = fma(z, 1.58969099521155010221e-10, -2.50507602534068634195e-08);
    ps = fma(z, ps, 2.75573137070700676789e-06);
    ps = fma(z, ps, -1.98412698298579493134e-04);
    ps = fma(z, ps, 8.33333333332248946124e-03);
    ps = fma(z, ps, -1.66666666666666324348e-01);
    const double s = fma(__dmul_rn(r, z), ps, r);
    double pc = fma(z, -1.13596475577881948265e-11, 2.08757232129817482790e-09);
    pc = fma(z, pc, -2.75573143513906633035e-07);
    pc = fma(z, pc, 2.48015872894767294178e-05);
    pc = fma(z, pc, -1.38888888888741095749e-03);
    pc = fma(z, pc, 4.16666666666666019037e-02);
    const double c = fma(__dmul_rn(z, z), pc, fma(z, -0.5, 1.0));
    const int n = __double2int_rn(k) & 3;
    const double a = (n & 1) ? c : s, b = (n & 1) ? s : c;
    sn = (n & 2) ? -a : a;
    cs = ((n + 1) & 2) ? -b : b;
}

// Sample position of the march, x0 + dx * t (range_libc RayMarching::calc_range).  The real
// range_libc is built -O3 -march=native -ffast-math, where the compiler is free to contract the
// multiply-add; its source is absent ("parity unpinned"), so which form its binary uses is
// unknown.  Canonical: fused (one rounding).  -DNAVGYM_MARCH_NO_FMA builds the separately
// rounded form -- the oracle has the matching switch (-DNVO_MARCH_NO_FMA) and both pairs are
// parity-tested, so the real package can be matched by flipping one flag.
__device__ __forceinline__ float march_pos(float d, float t, float o)
{
#ifdef NAVGYM_MARCH_NO_FMA
    return __fadd_rn(__fmul_rn(d, t), o);
#else
    return __fmaf_rn(d, t, o);
#endif
}

// range_libc RayMarching::calc_range, canonical form (oracle/navgym_oracle.c nvo_calc_range).
__device__ __forceinline__ float march(const float *__restrict__ dist, int W, int H, float x0,
                                       float y0, float dx, float dy, float max_range,
                                       float t_stop, int &hx, int &hy)
{
    float t = 0.0f;
    hx = HIT_NONE;
    hy = HIT_NONE;
    while (t < t_stop) {
        int px = __float2int_rz(march_pos(dx, t, x0));
        int py = __float2int_rz(march_pos(dy, t, y0));
        if ((unsigned)px >= (unsigned)W || (unsigned)py >= (unsigned)H) break;
        float d = __ldg(dist + (size_t)py * W + px);
        if (d <= 0.0f) {
            float xd = __fsub_rn((float)px, x0);
            float yd = __fsub_rn((float)py, y0);
            hx = (int)xd;
            hy = (int)yd;
            return __fsqrt_rn(__fadd_rn(__fmul_rn(xd, xd), __fmul_rn(yd, yd)));
        }
        t = __fadd_rn(t, fmaxf(__fmul_rn(d, 0.999f), 1.0f));
    }
    return max_range;
}

__device__ __forceinline__ float seg_hit(float ox, float oy, float dx, float dy, float ax,
                                         float ay, float bx, float by)
{
    float ex = __fsub_rn(bx, ax), ey = __fsub_rn(by, ay);
    float wx = __fsub_rn(ax, ox), wy = __fsub_rn(ay, oy);
    float den = __fsub_rn(__fmul_rn(dx, ey), __fmul_rn(dy, ex));
    if (den == 0.0f) return CUDART_INF_F;
    float tn = __fsub_rn(__fmul_rn(wx, ey), __fmul_rn(wy, ex));
    float un = __fsub_rn(__fmul_rn(wx, dy), __fmul_rn(wy, dx));
    float t = __fdiv_rn(tn, den);
    float u = __fdiv_rn(un, den);
    if (t >= 0.0f && u >= 0.0f && u <= 1.0f) return t;
    return CUDART_INF_F;
}

__device__ __forceinline__ float disc_hit(float ox, float oy, float dx, float dy, float X,
                                          float Y, float r)
{
    float cx = __fsub_rn(X, ox), cy = __fsub_rn(Y, oy);
    float b = __fadd_rn(__fmul_rn(dx, cx), __fmul_rn(dy, cy));
    float c = __fsub_rn(__fadd_rn(__fmul_rn(cx, cx), __fmul_rn(cy, cy)), __fmul_rn(r, r));
    float q = __fsub_rn(__fmul_rn(b, b), c);
    if (q < 0.0f) return CUDART_INF_F;
    float s = __fsqrt_rn(q);
    float t = __fsub_rn(b, s);
    if (t < 0.0f) t = __fadd_rn(b, s);
    if (t < 0.0f) return CUDART_INF_F;
    return t;
}

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k)
{
#pragma unroll
    for (int i = 0; i < 10; i++) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += 0x9E3779B9u;
        k.y += 0xBB67AE85u;
    }
    return c;
}

__device__ __forceinline__ float u01(uint32_t x) { return ((float)(x >> 8) + 0.5f) * (1.0f / 16777216.0f); }

// The draw that starts environment `env`'s next episode (global id, episode = its episode counter
// BEFORE the new episode): one Philox call keyed (env, episode, 0x5eed, 0xfffffff0) with `seed`.
// A new map when resample_map && num_maps > 1, and a spawn row of that map's pool: spawn(row, map)
// is called with the row (start x, y, goal x, y, theta) and the drawn map, or no_pool() when that
// map has no spawn pool.  Returns the new episode's scan-noise std.  The step kernel's auto-reset
// and the masked reset (navgym_reset_envs) both draw through here, so the two cannot disagree on
// where an episode starts (peds_plan spells the same draw out for the pedestrians' next-episode
// candidates).  The argument-block fields are taken by reference and the outcomes handed to
// callbacks, so the auto-reset branch compiles to the code it had when it spelled the draw out.
template <typename Spawn, typename NoPool>
__device__ __forceinline__ float draw_episode(const navgym_map_t *const &maps, const double *const &spawn_pool,
                                              const int32_t &num_maps, const int32_t &resample_map,
                                              const uint64_t &seed, uint32_t env, uint32_t episode, int map,
                                              const float &noise_lo, const float &noise_hi, Spawn &&spawn,
                                              NoPool &&no_pool)
{
    const uint4 rnd = philox4x32_10(make_uint4(env, episode, 0x5eedu, 0xfffffff0u),
                                    make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    int nmap = map;
    if (resample_map && num_maps > 1) nmap = (int)(((uint64_t)rnd.y * (uint64_t)num_maps) >> 32);
    const navgym_map_t m2 = maps[nmap];
    if (m2.spawn_count > 0) {
        const long long row = m2.spawn_offset + (long long)(((uint64_t)rnd.x * (uint64_t)m2.spawn_count) >> 32);
        spawn(spawn_pool + row * 5, nmap);
    } else {
        no_pool();
    }
    return noise_lo + (noise_hi - noise_lo) * u01(rnd.z);
}

// The observation row layouts (include/navgym_b200.h NAVGYM_OBS_*), the one place that knows
// them.  Element i < S*512 of p is a scan value; the 7 tail fields follow the S scans.
//   F32: float[obs_stride].
//   F16: __half[obs_stride]: float16 scans (round-to-nearest of the float32 value), the tail as
//        float32 in the 14 halves after them (4-byte aligned: even stride, aligned base).
// F = float for rows that are written, const float for rows that are only read; the row storage
// is passed as F * in either format (the C ABI's obs pointers).  A stored scan value moves from
// slot to slot of the stack as `p[dst] = p[src]` in both formats: float16 rounding is idempotent,
// so a shifted float16 history equals the rounded float32 history.
template <int FMT, typename F = float> struct ObsRow;
template <typename F> struct ObsRow<NAVGYM_OBS_F32, F> {
    using E = F;   // element type
    E *p;          // the scans, then the tail
    __device__ __forceinline__ ObsRow(F *obs, size_t row, int stride) : p(obs + row * stride) {}
    __device__ __forceinline__ float scan(int i) const { return p[i]; }
    __device__ __forceinline__ void set_scan(int i, float v) const { p[i] = v; }
    __device__ __forceinline__ void set_tail(int S, int f, float v) const { p[S * NB + f] = v; }
    // the tail, from the row's last scan
    static __device__ __forceinline__ F *tail_after(E *last_scan) { return last_scan + NB; }
};
template <typename F> struct ObsRow<NAVGYM_OBS_F16, F> {
    using E = typename std::conditional<std::is_const<F>::value, const __half, __half>::type;
    E *p;
    __device__ __forceinline__ ObsRow(F *obs, size_t row, int stride) : p(reinterpret_cast<E *>(obs) + row * stride) {}
    __device__ __forceinline__ float scan(int i) const { return __half2float(p[i]); }
    __device__ __forceinline__ void set_scan(int i, float v) const { p[i] = __float2half_rn(v); }
    __device__ __forceinline__ void set_tail(int S, int f, float v) const { reinterpret_cast<F *>(p + S * NB)[f] = v; }
    static __device__ __forceinline__ F *tail_after(E *last_scan) { return reinterpret_cast<F *>(last_scan + NB); }
};

// Scan value i of a row of either format (runtime format: debug / export paths only).
__device__ __forceinline__ float obs_scan_at(const float *obs, int format, size_t row, int stride, int i)
{
    if (format == NAVGYM_OBS_F16) return ObsRow<NAVGYM_OBS_F16, const float>(obs, row, stride).scan(i);
    return ObsRow<NAVGYM_OBS_F32, const float>(obs, row, stride).scan(i);
}
