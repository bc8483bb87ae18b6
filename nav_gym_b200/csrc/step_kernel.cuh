// step_kernel.cuh -- part of navgym_b200.cu (included there; one translation unit).
// The fused step kernel: NavGymEnv.step (env.py:591-728) for one environment per CTA.
// ------------------------------------------------------------------ fused step kernel
// Optional per-phase cycle accounting (tools/phase_prof.py builds with -DNAVGYM_PROFILE).
#ifdef NAVGYM_PROFILE
__device__ unsigned long long g_prof[16];
#define PROF_DECL long long _pt = clock64(); unsigned long long _g_begin; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(_g_begin));
#define PROF_MARK(i) do { if (tid == 0) { long long _n = clock64(); atomicAdd(&g_prof[i], (unsigned long long)(_n - _pt)); _pt = _n; } } while (0)
#else
#define PROF_DECL
#define PROF_MARK(i)
#endif

#define NAVGYM_CTA_THREADS 64  // one CTA of 2 warps = one environment
#define NAVGYM_CTAS_PER_SM 16  // resident CTAs the register budget is tuned for (64 registers)

struct EnvSmem {
    int scan[NB];          // float bits of the ranges [m] (non-negative floats order like ints)
    float2 dir[NB];        // beam directions (cos, sin) of the current pass
    double red[4];         // per-warp partial minima (NAVGYM_CTA_THREADS / 32 <= 4)
    // per-environment scalars parked here between the phases that need them, so the march
    // loop runs with a small register footprint
    double px, py, th, gx, gy, ppx, ppy, pyaw, pv, pw, act_v, act_w;
    double th_spec, yaw_spec;  // heading warp 1 assumed for the final pose, and its yaw
    int map, steps, episode, next_pass;
    int n_vis_seg, n_vis_disc;  // visible box segments / discs listed by the obstacle phase
    short alive[NB];       // beams still marching after the head phase: one list per warp, NB / 2 entries each
    float noise_std;
    // per-pass scan setup
    float lx, ly, lt, res32, max_range, t_stop;
    int ci, cj, W, H;
    long long edt_off;
#ifdef NAVGYM_PROFILE
    int prof_iters_a[8], prof_rounds_b[8], prof_alive, prof_cyc_b[8], prof_walk[8];   // per warp: tail iterations / cooperative rounds
#endif
};

// EDT value of an in-map cell through the read-only L1/L2 path (element 0 when !valid).  Kept a
// function: the same load written out at the three call sites compiles to a different schedule.
__device__ __forceinline__ float edt_at(const float *__restrict__ dist, int cx, int cy, int W, bool valid)
{
    return __ldg(dist + (valid ? (unsigned)(cy * W + cx) : 0u));
}

#ifndef NAVGYM_PROFILE
// 16 resident CTAs x (sizeof(EnvSmem) + 1 KB the system reserves per CTA) must fit the 132 KB
// shared-memory configuration: 64 bytes more and the driver picks the 164 KB one, taking 32 KB
// from the L1 the EDT gathers go through.
static_assert(sizeof(EnvSmem) <= 132 * 1024 / 16 - 1024, "EnvSmem outgrew the 132 KB carve-out at 16 CTAs/SM");
#endif
enum { PASS_STEP = 0, PASS_RESCAN = 1, PASS_RESET = 2, PASS_END = 3 };
constexpr int HEAD_STEPS = 4;  // samples every beam marches in the lockstep head phase
// ... in launches too large for tail regime B (COOP = false): throughput-bound, where two more
// lockstep samples (four gathers in flight per thread) beat the tail's one per lane
// (32 768 envs: 0.478 -> 0.468 ms; at 4096 envs the length makes no difference)
constexpr int HEAD_STEPS_LARGE = 6;

// Angular window of beams that can see an obstacle spanning bearings [phi0, phi0 + width].
// Beam k looks along lin[k] + theta with lin[k] = ANGLE_MIN + k * step (env.py:388-390).
__device__ __forceinline__ void beam_window(float phi0, float width, float theta, int &k0, int &cnt)
{
    const float step = 0.012271843f, amin = -3.141592f;
    float rel = phi0 - theta - amin;
    rel -= 6.2831853f * floorf(rel * 0.15915494f);
    k0 = (int)floorf(rel / step) - 2;
    cnt = (int)ceilf(width / step) + 5;
    if (cnt > NB) cnt = NB;
}

__device__ __forceinline__ void normal4(uint64_t seed, uint32_t env, uint32_t episode, uint32_t step,
                                        uint32_t slot, uint32_t group, float (&z)[4])
{
    uint4 r = philox4x32_10(make_uint4(env, episode, step, (slot << 16) | group),
                            make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    float r0 = sqrtf(-2.0f * __logf(u01(r.x))), r1 = sqrtf(-2.0f * __logf(u01(r.z)));
    float s0, c0, s1, c1;
    __sincosf(6.283185307179586f * u01(r.y), &s0, &c0);
    __sincosf(6.283185307179586f * u01(r.w), &s1, &c1);
    z[0] = r0 * c0; z[1] = r0 * s0; z[2] = r1 * c1; z[3] = r1 * s1;
}

// theta mod 2 pi with the sign of the divisor (numpy's float64 `%`, keti_robot.py:93).  One step
// turns by far less than 2 pi, so |x| < 4 pi in practice: there fmod is the identity or one
// exact subtraction (Sterbenz), bit-identical to the library call kept for anything larger.
__device__ __forceinline__ double wrap_2pi(double x)
{
    const double twopi = 6.283185307179586;
    double r;
    const double ax = fabs(x);
    if (ax < twopi) r = x;
    else if (ax < 2.0 * twopi) r = x < 0 ? __dadd_rn(x, twopi) : __dsub_rn(x, twopi);
    else r = fmod(x, twopi);
    if (r != 0 && r < 0) r = __dadd_rn(r, twopi);
    return r;
}

// Heading after this step's action (keti_robot.py:86-93); warps 0 and 1 both evaluate it.
__device__ __forceinline__ double turned_heading(double th0, double w, double dt, double &th1)
{
    th1 = __dadd_rn(th0, __dmul_rn(w, dt));
    return wrap_2pi(th1);
}

// Per-pass scan setup from the pose in shared memory: float32 lidar pose, origin cell
// (env.py:386, 419), map geometry.  Run by one thread.
__device__ __forceinline__ void pass_setup(EnvSmem &sm, const navgym_map_t &m, const navgym_step_args_t &a)
{
    sm.lx = (float)sm.px; sm.ly = (float)sm.py; sm.lt = (float)sm.th;
    sm.ci = xy_to_cell(sm.lx, m.ox, m.res, m.H, a.cell_rule);
    sm.cj = xy_to_cell(sm.ly, m.oy, m.res, m.W, a.cell_rule);
    sm.W = m.W; sm.H = m.H; sm.edt_off = m.edt_offset;
    sm.res32 = (float)m.res;
    sm.max_range = (float)((double)m.W * (double)m.H);
    sm.t_stop = fminf(fminf(a.t_stop, sm.max_range), 8.0e6f);
}

// Tail phase.  Two regimes:
//  A  dealing: every warp has its own list of the beams it marched through the head phase and
//     that are still alive; the entries are dealt to its lanes with ballot ranks (no atomics, no
//     cross-warp traffic): a lane whose beam ends takes the warp's next undealt entry; one beam
//     per lane, one EDT gather per lane and round trip.
//  B  cooperative: once the warp's entries are all dealt and at most COOP_ENTER beams are
//     still marching, the idle lanes stop idling: the L live beams are regrouped onto G = 32 / L
//     (power of two) lanes each, and lane j of a group fetches the cell the beam would sample
//     at t + j -- a guess at where the march goes next (along a wall the step is max(0.999 d, 1)
//     ~ 1..2 cells).  The group then WALKS the true march in registers: the next sample's cell
//     is computed with the canonical arithmetic and looked up among the fetched cells (shuffles;
//     an EDT value depends on the cell alone, so a match is exactly the value the march would
//     load); the walk goes on until a sample's cell was not fetched, and the next fetch starts
//     there.  Sample 0 of a fetch is the beam's own next sample, so every round trip advances
//     the beam at least as far as regime A would -- and the dependent-gather chain of a scan's
//     longest beams (max 226 samples on the bench world, one L2 round trip each) shrinks 3-5x
//     (oracle/analysis/coop_march.py).  The sequence of t values and hit cells is bit-identical.
constexpr int COOP_ENTER = 1;
constexpr int COOP_LOG2_WIDTH = 5;   // at most 2^5 lanes fetch ahead for one beam
template <bool COOP>
__device__ __forceinline__ void march_tail_dealt(EnvSmem &sm, const float *__restrict__ dist, float x0, float y0,
                                                 int W, int H, float t_stop, int n_alive, int warp, int lane)
{
    // every warp deals from its own survivor list
    const short *list = sm.alive + warp * (NB / 2);
    const unsigned FULL = 0xffffffffu;
    int next_j = 32;                       // warp-uniform: entries dealt so far
    int idx = lane;
    int kb = idx < n_alive ? (int)list[idx] : -1;
    float t = __int_as_float(sm.scan[kb >= 0 ? kb : 0]);
    float2 dd = sm.dir[kb >= 0 ? kb : 0];
    unsigned live = __ballot_sync(FULL, kb >= 0);
    if (!live) return;
    // ---- regime A.  The warp's dealing state (next_j, live) and with it the switch to regime B
    // only change in an iteration in which some beam ended: all of that sits behind one
    // warp-uniform test of the ballot.
    bool to_b = COOP && !(next_j < n_alive) && __popc(live) <= COOP_ENTER;
    while (!to_b) {
        const int cx = __float2int_rz(march_pos(dd.x, t, x0));
        const int cy = __float2int_rz(march_pos(dd.y, t, y0));
        const bool inb = ((unsigned)cx < (unsigned)W) & ((unsigned)cy < (unsigned)H);
        const float d = edt_at(dist, cx, cy, W, inb & (kb >= 0));
        const bool hit = inb & (d <= 0.0f);
        t = __fadd_rn(t, fmaxf(__fmul_rn(d, 0.999f), 1.0f));
        const bool fin = (kb >= 0) & (!inb | hit | !(t < t_stop));
        const unsigned fm = __ballot_sync(FULL, fin);
#ifdef NAVGYM_PROFILE
        if (lane == 0) sm.prof_iters_a[warp]++;
#endif
        if (fm) {
            if (fin) {
                // absolute hit cell, (y << 16 | x), or -1 for "no hit"
                sm.scan[kb] = hit ? (cy << 16 | cx) : -1;
                idx = (next_j + __popc(fm & ((1u << lane) - 1u)));
                kb = -1;
                if (idx < n_alive) {
                    kb = list[idx];
                    t = __int_as_float(sm.scan[kb]);
                    dd = sm.dir[kb];
                }
            }
            next_j += __popc(fm);
            live = __ballot_sync(FULL, kb >= 0);
            if (!live) return;
            to_b = COOP && !(next_j < n_alive) && __popc(live) <= COOP_ENTER;
        }
    }
    // ---- regime B: `live` marks the lanes that hold a marching beam (kb, t, dd)
#ifdef NAVGYM_PROFILE
    const long long prof_b0 = clock64();
#endif
    while (live) {
        const int L = __popc(live);        // <= COOP_ENTER
        const int lg = min(L > 8 ? 1 : L > 4 ? 2 : L > 2 ? 3 : L > 1 ? 4 : 5, COOP_LOG2_WIDTH);   // G = 32 / L, a power of two
        const int G = 1 << lg;             // lanes per beam
        const int g = lane >> lg, j = lane & (G - 1), base = lane & ~(G - 1);
        const bool act = g < L;
        const int owner = act ? (int)__fns(live, 0, g + 1) : 0;
        const int bk = __shfl_sync(FULL, kb, owner);
        float bt = __shfl_sync(FULL, t, owner);
        const float bdx = __shfl_sync(FULL, dd.x, owner), bdy = __shfl_sync(FULL, dd.y, owner);
        bool fin = !act;                   // group-uniform
        int res = -1;
        const int regroup_at = L > 1 ? (32 >> (lg + 1)) : 0;   // unfinished beams that fit twice the lanes
        for (;;) {
            // fetch: lane j guesses the sample at t + j (j = 0: the beam's own next sample)
            const float tj = __fadd_rn(bt, (float)j);
            const int fx = __float2int_rz(march_pos(bdx, tj, x0));
            const int fy = __float2int_rz(march_pos(bdy, tj, y0));
            const bool finb = ((unsigned)fx < (unsigned)W) & ((unsigned)fy < (unsigned)H);
            const int fcell = finb ? (fy << 16 | fx) : -2;
            const float fd = edt_at(dist, fx, fy, W, finb & !fin);
            // walk the true march through the fetched cells
            const float t0 = bt;
            bool walking = !fin;
#pragma unroll 1
            for (int it = 0; it < G; it++) {
                const int wx = __float2int_rz(march_pos(bdx, bt, x0));
                const int wy = __float2int_rz(march_pos(bdy, bt, y0));
                const bool winb = ((unsigned)wx < (unsigned)W) & ((unsigned)wy < (unsigned)H);
                const int wcell = wy << 16 | wx;
                // the guess nearest to t (one candidate finds all but ~2 % of what three would)
                const int l0 = base + min(__float2int_rn(__fsub_rn(bt, t0)), G - 1);
                const int c0 = __shfl_sync(FULL, fcell, l0);
                const float d = __shfl_sync(FULL, fd, l0);
                const float tn = __fadd_rn(bt, fmaxf(__fmul_rn(d, 0.999f), 1.0f));
                if (walking) {
                    if (!winb) { fin = true; res = -1; walking = false; }
                    else if (c0 != wcell) walking = false;      // not fetched: the next fetch starts here
                    else if (d <= 0.0f) { fin = true; res = wcell; walking = false; }
                    else {
                        bt = tn;
                        if (!(tn < t_stop)) { fin = true; res = -1; walking = false; }
                    }
                }
#ifdef NAVGYM_PROFILE
                if (lane == 0) sm.prof_walk[warp]++;
#endif
                if (!__any_sync(FULL, walking)) break;
            }
#ifdef NAVGYM_PROFILE
            if (lane == 0) sm.prof_rounds_b[warp]++;
#endif
            const unsigned un = __ballot_sync(FULL, !fin & (j == 0));
            if (__popc(un) <= regroup_at) break;
        }
        if (act & fin & (j == 0)) sm.scan[bk] = res;
        // the group's first lane now holds the beam
        kb = (act & !fin & (j == 0)) ? bk : -1;
        t = bt;
        dd = make_float2(bdx, bdy);
        live = __ballot_sync(FULL, kb >= 0);
    }
#ifdef NAVGYM_PROFILE
    if (lane == 0) sm.prof_cyc_b[warp] += (int)(clock64() - prof_b0);
#endif
}

// One scan's occupancy-grid march (env.py:425-426) for the beams of head rounds [r_begin, r_end)
// (round r = this thread's beams BEAM(4 r .. 4 r + 3)): beam directions, lockstep head phase,
// survivor list, tail phase.  Leaves every beam's hit cell, (y << 16 | x) or -1, in sm.scan and
// its direction in sm.dir; ends on a CTA barrier.  Scan set-up is read from sm (pass_setup).
template <bool COOP>
__device__ __forceinline__ void march_scan(EnvSmem &sm, const navgym_step_args_t &a, const int r_begin, const int r_end,
                                           const int tid)
{
    constexpr int TPB = NAVGYM_CTA_THREADS;
    const unsigned FULL = 0xffffffffu;
    const int lane = tid & 31, warp = tid >> 5;
#define BEAM(i) (tid + TPB * (i))
    const int W = sm.W, H = sm.H, ci = sm.ci, cj = sm.cj;
    const float x0 = (float)ci, y0 = (float)cj;
    const float t_stop = sm.t_stop;
    const float *dist = a.edt_pool + sm.edt_off;
    asm volatile("" : "+l"(dist));  // keep base + offset folded into one register pair
    // xy_to_cell clips ci against H and cj against W (the reference's quirk, env.py:1245-1248):
    // on a non-square map the origin can still lie outside [0, W) x [0, H), where
    // calc_range's first sample returns "no hit" for every beam
    const bool o_in = ((unsigned)ci < (unsigned)W) & ((unsigned)cj < (unsigned)H);
    const float d0 = o_in ? __ldg(dist + cj * W + ci) : 1.0f;
    const float t1 = fmaxf(__fmul_rn(d0, 0.999f), 1.0f);  // == 0.0f + first step
    const bool degenerate = !o_in | (d0 <= 0.0f) | !(t1 < t_stop);
    constexpr int HB = 4;   // beams in flight per thread in the head phase
    int n_mine = 0;   // warp-uniform: survivors in this warp's list
#pragma unroll 1
    for (int r = r_begin; r < r_end; r++) {
        float th_[HB], dxh[HB], dyh[HB];
        // beam directions (env.py:388-390, 420-424)
#pragma unroll
        for (int j = 0; j < HB; j++) {
            const int k = BEAM(r * HB + j);
            const float h = (float)__dadd_rn(a.lin[k], (double)sm.lt);
            double sd, cd;
            dir_sincos((double)h, sd, cd);
            dxh[j] = (float)cd;
            dyh[j] = (float)sd;
            sm.dir[k] = make_float2(dxh[j], dyh[j]);
            th_[j] = t1;
            if (degenerate) { sm.scan[k] = (o_in & (d0 <= 0.0f)) ? (cj << 16 | ci) : -1; th_[j] = CUDART_NAN_F; }
        }
        // An ended beam is marked by t = NaN: its sample position converts to cell (0, 0) (a valid
        // load of element 0, like the idle lanes of the tail), its next t is NaN again, which fails
        // "t < t_stop" and so counts as ended -- only the store of the hit cell asks whether the beam
        // was still alive (one compare instead of a predicate carried through the whole step:
        // 99 instead of 119 instructions per four samples).
#pragma unroll 1
        for (int st = 0; st < (COOP ? HEAD_STEPS : HEAD_STEPS_LARGE); st++) {
            float dv[HB];
            int cx[HB], cy[HB];
            bool inb[HB];
#pragma unroll
            for (int j = 0; j < HB; j++) {
                cx[j] = __float2int_rz(march_pos(dxh[j], th_[j], x0));
                cy[j] = __float2int_rz(march_pos(dyh[j], th_[j], y0));
                inb[j] = ((unsigned)cx[j] < (unsigned)W) & ((unsigned)cy[j] < (unsigned)H);
                dv[j] = edt_at(dist, cx[j], cy[j], W, inb[j]);
            }
#pragma unroll
            for (int j = 0; j < HB; j++) {
                const bool hit = inb[j] & (dv[j] <= 0.0f);
                const float tn = __fadd_rn(th_[j], fmaxf(__fmul_rn(dv[j], 0.999f), 1.0f));   // NaN for an ended beam
                const bool fin = !inb[j] | hit | !(tn < t_stop);
                if (fin & (th_[j] == th_[j])) sm.scan[BEAM(r * HB + j)] = hit ? (cy[j] << 16 | cx[j]) : -1;
                th_[j] = fin ? CUDART_NAN_F : tn;
            }
        }
        // survivors: park t in the scan slot and append the beam to the compact list
#pragma unroll
        for (int j = 0; j < HB; j++) {
            const int k = BEAM(r * HB + j);
            const bool alive = th_[j] == th_[j];
            if (alive) sm.scan[k] = __float_as_int(th_[j]);
            const unsigned mk = __ballot_sync(FULL, alive);
            if (alive) sm.alive[warp * (NB / 2) + n_mine + __popc(mk & ((1u << lane) - 1u))] = (short)k;
            n_mine += __popc(mk);
        }
    }
    // A warp compacts and deals its own survivors (its beams are 32-beam sectors alternating with
    // the other warp's, so the lists are about equally long): no atomic on a shared counter, and no
    // CTA barrier between the head and the tail phase -- only the warp's own stores to wait for.
    __syncwarp();
    {
        const int n_alive = n_mine;
#ifdef NAVGYM_PROFILE
        if (tid == 0) sm.prof_alive += n_alive;
#endif
        march_tail_dealt<COOP>(sm, dist, x0, y0, W, H, t_stop, n_alive, warp, lane);
    }
    __syncthreads();
#undef BEAM
}

// One CTA of 2 warps = one environment.  Thread t of the CTA owns beams t + 64 i, i = 0 .. 7:
// the lanes of a warp work on neighbouring beams, whose EDT gathers share sectors.
// A scan marches in two phases (see the march section below): a lockstep head phase, four
// samples per beam with four beams per thread in flight, then a tail phase in which the beams
// still alive are dealt to lanes as lanes fall free (ballot-rank dealing, one beam per lane at a
// time; the last beam of a warp is marched by all its lanes together).  The three scans a step
// may need (the step's scan, the crash re-scan env.py:718, the auto-reset first scan) run
// through ONE copy of the scan code inside a CTA-uniform pass loop.
constexpr float RISK_MARGIN = 0.25f;  // [m] clearance under which the next step may end the episode
// What one CTA of the fused kernel does to its environment:
//   MODE_STEP          one step (navgym_step_batch), auto-reset included;
//   MODE_RESET         the first observation of an episode from the pose in `state`
//                      (navgym_reset_obs_batch);
//   MODE_MASKED_RESET  a new episode drawn exactly as the step's auto-reset draws it, then its
//                      first observation as the auto-reset pass writes it (navgym_reset_envs):
//                      no hits recorded, no launch-order filing.
// NEXT (next-step auto-reset, step_kernel<MODE_NEXT_STEP>) runs MODE_STEP with auto-reset off, or
// MODE_MASKED_RESET extended to write what a step writes: outputs (0, and the distance from the new
// pose to the new goal), hits and the launch-order filing.  Neither doubles the cost class of a
// risky environment: no step of this mode runs a reset scan after its own.
enum { MODE_STEP = 0, MODE_RESET = 1, MODE_MASKED_RESET = 2, MODE_NEXT_STEP = 3 };
template <int MODE, bool COOP, int FMT, bool NEXT = false>
__device__ __forceinline__ void step_body(const navgym_step_args_t &a, EnvSmem &sm, const int e, const int tid,
                                          int *sched_cnt, int *sched_list)
{
    constexpr bool IS_RESET_KERNEL = MODE != MODE_STEP;   // both reset modes: no action, a new episode
    constexpr bool MASKED = MODE == MODE_MASKED_RESET;
    constexpr int TPB = NAVGYM_CTA_THREADS;  // threads of the CTA
    constexpr int BPL = NB / TPB;            // beams per lane
    const int lane = tid & 31, warp = tid >> 5;
    const int B = a.num_envs;
    const long long t_begin = clock64();
    const unsigned FULL = 0xffffffffu;
    double *S = a.state;
#define ST(f) S[(size_t)(f) * B + e]
#define BEAM(i) (tid + TPB * (i))

    PROF_DECL
#ifdef NAVGYM_PROFILE
    if (tid < 8) { sm.prof_iters_a[tid] = 0; sm.prof_rounds_b[tid] = 0; sm.prof_cyc_b[tid] = 0; sm.prof_walk[tid] = 0; }
    if (tid == 0) sm.prof_alive = 0;
#endif
    // ---------------- prologue (warp 0): state (lane f holds row f), kinematics ----------
    // Every global load the prologue needs is issued up front (they only depend on e), the map
    // descriptor as soon as the map id is back, so one L2 round trip overlaps the next and the
    // float64 kinematics.  Warp 1 meanwhile evaluates the yaw the epilogue will need (the same
    // heading arithmetic as warp 0): for every environment that neither rolls back nor resets,
    // the float64 sincos + atan2 of the final heading leave the critical path.
    if (warp == 1) {
        double th = ST(NAVGYM_S_TH);
        if (!IS_RESET_KERNEL) {
            double th1;
            th = turned_heading(th, (double)a.actions[2 * (size_t)e + 1], a.dt, th1);
        }
        double sn, cn;
        sincos(th, &sn, &cn);
        const double yaw = atan2(sn, cn);  // utils.py:5-9
        if (lane == 0) { sm.th_spec = th; sm.yaw_spec = yaw; }
    }
    if (warp == 0) {
        double sv = lane < NAVGYM_NS ? ST(lane) : 0.0;
        int steps = a.steps[e];
        int map0 = a.map_id[e];
        const int episode0 = a.episodes ? a.episodes[e] : 0;
        float noise_std0 = a.noise_std ? a.noise_std[e] : 0.0f;
        float2 av = make_float2(0.f, 0.f);
        if (!IS_RESET_KERNEL) av = *reinterpret_cast<const float2 *>(a.actions + 2 * (size_t)e);
        // masked reset: the next episode's spawn row (and map), drawn before the map descriptor is read
        const double *spawn = nullptr;
        if (MASKED)
            noise_std0 = draw_episode(a.maps, a.spawn_pool, a.num_maps, a.resample_map, a.seed,
                                      (uint32_t)(a.env_offset + e), (uint32_t)episode0, map0, a.noise_lo, a.noise_hi,
                                      [&](const double *sp, int nmap) { spawn = sp; map0 = nmap; }, [] {});
        const navgym_map_t m0 = a.maps[map0];
        double px = __shfl_sync(FULL, sv, NAVGYM_S_PX), py = __shfl_sync(FULL, sv, NAVGYM_S_PY);
        double th0 = __shfl_sync(FULL, sv, NAVGYM_S_TH), th = th0;
        double gx = 0.0, gy = 0.0;
        if (MASKED) {   // without a spawn pool the pose and goal in `state` stay
            gx = __shfl_sync(FULL, sv, NAVGYM_S_GX);
            gy = __shfl_sync(FULL, sv, NAVGYM_S_GY);
            if (spawn) { px = spawn[0]; py = spawn[1]; gx = spawn[2]; gy = spawn[3]; th = spawn[4]; }
        }
        double act_v = 0, act_w = 0;
        if (!IS_RESET_KERNEL) {
            double v = (double)av.x, w = (double)av.y;
            if (a.min_turn_radius > 0) {  // env.py:595-600
                double lim = __dmul_rn(fabs(w), a.min_turn_radius);
                if (v >= 0) v = v > lim ? v : lim;
                else v = v < -lim ? v : -lim;
            }
            act_v = a.min_turn_radius > 0 ? v : (double)av.x;  // env.py:725 (the clamp edits `action`)
            act_w = (double)av.y;
            double th1;
            th = turned_heading(th0, w, a.dt, th1);
            double s_, c_;
            sincos(lane == 0 ? th0 : th1, &s_, &c_);  // lanes 0 / 1 in parallel
            double s0 = __shfl_sync(FULL, s_, 0), c0 = __shfl_sync(FULL, c_, 0);
            double s1 = __shfl_sync(FULL, s_, 1), c1 = __shfl_sync(FULL, c_, 1);
            // keti_robot.py:64-93
            double rx = __dadd_rn(__dmul_rn(0.14474, c0), px);
            double ry = __dadd_rn(__dmul_rn(0.14474, s0), py);
            rx = __dadd_rn(rx, __dmul_rn(__dmul_rn(c1, v), a.dt));
            ry = __dadd_rn(ry, __dmul_rn(__dmul_rn(s1, v), a.dt));
            px = __dadd_rn(__dmul_rn(-0.14474, c1), rx);
            py = __dadd_rn(__dmul_rn(-0.14474, s1), ry);
            steps += 1;  // env.py:592
        } else {
            steps = 0;
        }
        // a host-side reset starts a new episode: a new noise / spawn stream (the in-kernel
        // auto-reset advances the same counter)
        const int episode1 = episode0 + (IS_RESET_KERNEL ? 1 : 0);
        if (!MASKED && lane == NAVGYM_S_GX) sm.gx = sv;
        if (!MASKED && lane == NAVGYM_S_GY) sm.gy = sv;
        if (!IS_RESET_KERNEL) {
            if (lane == NAVGYM_S_PPX) sm.ppx = sv;
            if (lane == NAVGYM_S_PPY) sm.ppy = sv;
            if (lane == NAVGYM_S_PYAW) sm.pyaw = sv;
            if (lane == NAVGYM_S_PV) sm.pv = sv;
            if (lane == NAVGYM_S_PW) sm.pw = sv;
        }
        if (lane == 0) {
            sm.px = px; sm.py = py; sm.th = th;
            sm.act_v = act_v; sm.act_w = act_w;
            sm.map = map0;
            sm.steps = steps;
            sm.episode = episode1;
            sm.noise_std = noise_std0;
            if (IS_RESET_KERNEL) { sm.ppx = px; sm.ppy = py; sm.pyaw = 0; sm.pv = 0; sm.pw = 0; }
            if (MASKED) { sm.gx = gx; sm.gy = gy; }
            pass_setup(sm, m0, a);  // first pass: the map descriptor is already here
        }
    }
    int nd = a.discs ? min(a.ndisc[e], a.max_disc) : 0;
    int ns = a.segs ? min(a.nseg[e], a.max_seg) : 0;
    if (MASKED && a.discs_reset != nullptr) {   // the first scan sees the next episode's pedestrians, if given
        nd = min(a.ndisc_reset[e], a.max_disc);
        ns = a.segs_reset ? min(a.nseg_reset[e], a.max_seg) : 0;
    }
    int pass = IS_RESET_KERNEL ? PASS_RESET : PASS_STEP;
    const ObsRow<FMT> orow(a.obs, (size_t)e, a.obs_stride);   // the row format is a template parameter

    long long t_pass = t_begin;  // start of the pass that produces the returned observation
    float margin = CUDART_INF_F; // its smallest clearance over the crash thresholds [m]
    for (bool first = true;; first = false) {
        // ---- per-pass setup; the first pass was set up by the prologue
        __syncthreads();
        if (!first) {
            t_pass = clock64();
            if (tid == 0) pass_setup(sm, a.maps[sm.map], a);
            __syncthreads();
        }
        margin = CUDART_INF_F;
        PROF_MARK(0);
        const float lx = sm.lx, ly = sm.ly, lt = sm.lt;
        PROF_MARK(1);
        // ---- occupancy-grid march (env.py:425-426).
        // Every beam of a scan starts on the origin cell, so that first sample (t = 0) is taken
        // once per environment: either the origin is occupied (all beams end there) or all
        // beams advance by the same first step.  The march then runs in two phases:
        //  head: every thread marches its own beams HEAD_STEPS samples, HB beams at a
        //        time in lockstep — almost every beam is still alive that early, and the HB
        //        independent EDT gathers per thread hide the L2 latency by ILP;
        //  tail: the surviving beams are compacted into a list and dealt out dynamically (a
        //        lane takes the next survivor whenever its beam ends), so lanes stay busy on
        //        the long-tailed remainder instead of idling until the slowest beam ends.
        // The loops only find each beam's hit cell (packed into sm.scan); ranges are computed
        // afterwards with all lanes active.
        {
            march_scan<COOP>(sm, a, 0, BPL / 4, tid);
            const int ci = sm.ci, cj = sm.cj;
            // ranges (env.py:426), all lanes active: sqrt(di^2 + dj^2) * resolution
            const bool rec = (!MASKED || NEXT) && pass == (IS_RESET_KERNEL ? PASS_RESET : PASS_STEP) && a.hits;
            const float max_range = sm.max_range, res32 = sm.res32;
#pragma unroll
            for (int i = 0; i < BPL; i++) {
                const int k = BEAM(i);
                const int cell = sm.scan[k];
                float rc = max_range;
                int rel = (int)0x80008000;
                if (cell != -1) {
                    const int hx = (cell & 0xffff) - ci, hy = (cell >> 16) - cj;
                    const float xd = (float)hx, yd = (float)hy;
                    rc = __fsqrt_rn(__fadd_rn(__fmul_rn(xd, xd), __fmul_rn(yd, yd)));
                    rel = (hx & 0xffff) | (hy << 16);
                }
                sm.scan[k] = __float_as_int(__fmul_rn(rc, res32));
                if (rec) reinterpret_cast<int *>(a.hits)[(size_t)e * NB + k] = rel;
            }
        }
        PROF_MARK(3);
        // ---- pedestrians: segments (env.py:430-431) and discs (env.py:432), min-merged.
        // Two steps.  (A) lanes across obstacles: every thread loads one obstacle and works out the
        // angular window of beams that can see it (or that it is out of sight) -- all obstacle
        // loads of the environment are in flight together, and the window trigonometry runs 32
        // obstacles wide; the windows are parked in the survivor list's shared memory (free since
        // the tail phase).  (B) one warp per visible obstacle, lanes across the beams of its window.
        // (One warp per obstacle for both steps walked the list through one global-memory round
        // trip per obstacle and computed every window 32 times over.)
        if (ns + nd > 0) {
            if (tid == 0) { sm.n_vis_seg = 0; sm.n_vis_disc = 0; }
            __syncthreads();
            // (the first scan after an auto-reset or of a masked reset sees the next episode's pedestrians, if given)
            const bool nxt = MODE != MODE_RESET && pass == PASS_RESET && a.discs_reset != nullptr;
            const float *discs = (nxt ? a.discs_reset : a.discs) + (size_t)e * a.max_disc * 3;
            const float *segs = (nxt ? a.segs_reset : a.segs) + (size_t)e * a.max_seg * 4;
            // The visible obstacles are listed in the survivor list's shared memory (free since the tail
            // phase), segments from the front and discs from the back of its NB / 2 words:
            // index (8 bits) | k0 + 2 (10 bits) << 8 | cnt (10 bits) << 18.
            int *vis = reinterpret_cast<int *>(sm.alive);
            const int n_obs = min(ns + nd, NB / 2);         // (host: max_seg + max_disc <= NB / 2)
            for (int o0 = 0; o0 < n_obs; o0 += TPB) {
                const int o = o0 + tid;
                int k0 = 0, cnt = 0;
                if (o < ns) {
                    const float4 sg = *reinterpret_cast<const float4 *>(segs + 4 * o);
                    const float ax = sg.x, ay = sg.y, bx = sg.z, by = sg.w;
                    float da2 = (ax - lx) * (ax - lx) + (ay - ly) * (ay - ly);
                    float db2 = (bx - lx) * (bx - lx) + (by - ly) * (by - ly);
                    // out of sight: every point of the segment is farther than range_max (its
                    // nearer end minus its length still is), so any hit would be clipped to
                    // range_max two phases on -- the same value as no hit (env.py:435)
                    const float len2 = (bx - ax) * (bx - ax) + (by - ay) * (by - ay);
                    const float reach = a.range_max * 1.001f + sqrtf(len2) + 0.01f;
                    if (!(fminf(da2, db2) > reach * reach)) {
                        float pa = atan2f(ay - ly, ax - lx), pb = atan2f(by - ly, bx - lx);
                        float dl = pb - pa;
                        dl -= 6.2831853f * rintf(dl * 0.15915494f);
                        if (fabsf(dl) > 3.0f || da2 < 1e-6f || db2 < 1e-6f) { k0 = 0; cnt = NB; }
                        else beam_window(dl >= 0 ? pa : pb, fabsf(dl), lt, k0, cnt);
                    }
                } else if (o < n_obs) {
                    const int q = o - ns;
                    const float X = discs[3 * q], Y = discs[3 * q + 1], Rd = discs[3 * q + 2];
                    const float cx = X - lx, cy = Y - ly;
                    const float dc = sqrtf(cx * cx + cy * cy);
                    if (!(dc > a.range_max * 1.001f + fabsf(Rd) + 0.01f)) {   // else out of sight (see the segments)
                        if (dc <= Rd * 1.05f + 1e-3f) { k0 = 0; cnt = NB; }
                        else {
                            const float half = asinf(fminf(Rd / dc, 1.0f)) * 1.01f + 1e-4f;
                            beam_window(atan2f(cy, cx) - half, 2.0f * half, lt, k0, cnt);
                        }
                    }
                }
                // list the visible ones (the order within a list does not matter: hits are min-merged)
                const bool is_seg = o < ns;
                const unsigned ms_ = __ballot_sync(FULL, cnt > 0 && is_seg), md_ = __ballot_sync(FULL, cnt > 0 && !is_seg);
                int bs = 0, bd = 0;
                if (lane == 0) {
                    if (ms_) bs = atomicAdd(&sm.n_vis_seg, __popc(ms_));
                    if (md_) bd = atomicAdd(&sm.n_vis_disc, __popc(md_));
                }
                bs = __shfl_sync(FULL, bs, 0);
                bd = __shfl_sync(FULL, bd, 0);
                if (cnt > 0) {
                    const int word = (is_seg ? o : o - ns) | ((k0 + 2) & 0x3ff) << 8 | cnt << 18;   // k0 in [-2, 510], cnt <= NB = 512
                    const unsigned below = (1u << lane) - 1u;
                    if (is_seg) vis[bs + __popc(ms_ & below)] = word;
                    else vis[NB / 2 - 1 - (bd + __popc(md_ & below))] = word;
                }
            }
            __syncthreads();
            // hits: 16 lanes per visible obstacle across the beams of its window (a window is typically
            // a dozen beams wide), segments first, then discs
            {
                const int grp = tid >> 4, l16 = tid & 15;
                constexpr int NG = TPB / 16;
                const int nvs = sm.n_vis_seg, nvd = sm.n_vis_disc;
                for (int i = grp; i < nvs; i += NG) {
                    const int w = vis[i];
                    const int cnt = w >> 18, k0 = ((w >> 8) & 0x3ff) - 2;
                    const float4 sg = *reinterpret_cast<const float4 *>(segs + 4 * (w & 0xff));
                    for (int j = l16; j < cnt; j += 16) {
                        const int k = (k0 + j) & (NB - 1);
                        const float tt = seg_hit(lx, ly, sm.dir[k].x, sm.dir[k].y, sg.x, sg.y, sg.z, sg.w);
                        if (tt < CUDART_INF_F) atomicMin(&sm.scan[k], __float_as_int(tt));
                    }
                }
                // (8 lanes per disc: a leg's window is 6-8 beams)
                for (int i = tid >> 3; i < nvd; i += TPB / 8) {
                    const int w = vis[NB / 2 - 1 - i];
                    const int cnt = w >> 18, k0 = ((w >> 8) & 0x3ff) - 2;
                    const int q = w & 0xff;
                    const float X = discs[3 * q], Y = discs[3 * q + 1], Rd = discs[3 * q + 2];
                    for (int j = tid & 7; j < cnt; j += 8) {
                        const int k = (k0 + j) & (NB - 1);
                        const float tt = disc_hit(lx, ly, sm.dir[k].x, sm.dir[k].y, X, Y, Rd);
                        if (tt < CUDART_INF_F) atomicMin(&sm.scan[k], __float_as_int(tt));
                    }
                }
            }
            __syncthreads();
        }
        PROF_MARK(4);
        // ---- clip + noise (env.py:435-440), thresholds, observation row
        bool c_any = false, d_any = false;
        {
            const int nslot = pass == PASS_RESCAN ? 1 : 0;
            const float noise_std = sm.noise_std;
            const int steps = sm.steps, episode = sm.episode;
            const int SS = a.num_scan_stack > 1 ? a.num_scan_stack : 1;
            constexpr int G = 4;
            // Production noise: one Philox4x32-10 call + two Box-Muller pairs per group of four
            // CONSECUTIVE beams 4q .. 4q + 3, keyed (seed; global env, episode, step, scan slot,
            // q) -- a function of the beam index alone, whatever the launch shape.  The unit
            // normals are staged in sm.dir (the beam directions are not needed any more).
            const bool philox = !a.noise && noise_std > 0.0f;   // CTA-uniform
            float *zs = reinterpret_cast<float *>(sm.dir);
            if (philox) {
                for (int q = tid; q < NB / 4; q += TPB) {
                    float z[4];
                    normal4(a.seed, (uint32_t)(a.env_offset + e), (uint32_t)episode, (uint32_t)steps,
                            (uint32_t)pass, (uint32_t)q, z);
                    *reinterpret_cast<float4 *>(zs + 4 * q) = make_float4(z[0], z[1], z[2], z[3]);
                }
                __syncthreads();
            }
#pragma unroll 1
            for (int g = 0; g < BPL / G; g++) {
#pragma unroll
                for (int j = 0; j < G; j++) {
                    const int k = BEAM(G * g + j);
                    float v = fminf(fmaxf(__int_as_float(sm.scan[k]), 0.0f), a.range_max);
                    if (v != a.range_max) {
                        if (a.noise) v = __fadd_rn(v, a.noise[((size_t)e * 2 + nslot) * NB + k]);
                        else if (philox) v = __fadd_rn(v, noise_std * zs[k]);
                    }
                    sm.scan[k] = __float_as_int(v);
                    if (SS == 1) {
                        orow.set_scan(k, v);
                    } else {
                        // _stack_scan (env.py:257-279): [pads = current scan | previous scans,
                        // oldest first | current scan]; the previous observation row still holds
                        // them one slot to the right
                        const int hist = pass == PASS_RESET ? 0 : min(steps, SS - 1);
                        for (int j = 0; j < SS - 1; j++) {
                            if (j < SS - 1 - hist) orow.set_scan(j * NB + k, v);
                            else if (pass == PASS_STEP) orow.p[j * NB + k] = orow.p[(j + 1) * NB + k];   // stored value, either format
                        }
                        orow.set_scan((SS - 1) * NB + k, v);
                    }
                    const float thr_k = a.thr[k];
                    c_any |= v < thr_k;
                    d_any |= v < a.dthr[k];
                    margin = fminf(margin, v - thr_k);
                }
            }
        }

        PROF_MARK(5);
        if (pass == PASS_STEP) {
            // ---- reward / done / info on this observation (env.py:464-589)
            int crash, discomf;
            crash = __syncthreads_or(c_any);
            discomf = __syncthreads_or(d_any) && !crash;
            double mn = CUDART_INF;
            if (discomf) {
                for (int i = 0; i < BPL; i++) {
                    const int k = BEAM(i);
                    const float thr_k = a.thr[k], dthr_k = a.dthr[k];
                    const float den = __fadd_rn(__fsub_rn(dthr_k, thr_k), 1e-6f);
                    mn = fmin(mn, __ddiv_rn(__dsub_rn((double)__int_as_float(sm.scan[k]), (double)thr_k), (double)den));
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) mn = fmin(mn, __shfl_xor_sync(FULL, mn, o));
                if (lane == 0) sm.red[warp] = mn;
                __syncthreads();
            }
            if (warp == 0) {
                if (discomf) mn = fmin(fmin(mn, sm.red[0]), sm.red[1]);
                // lanes 0 / 1: distance to goal from pose / prev_pose
                const double gx = sm.gx, gy = sm.gy;
                const double qx = lane == 0 ? sm.px : sm.ppx, qy = lane == 0 ? sm.py : sm.ppy;
                const double ddx = __dsub_rn(gx, qx), ddy = __dsub_rn(gy, qy);
                const double dq = sqrt(__dadd_rn(__dmul_rn(ddx, ddx), __dmul_rn(ddy, ddy)));
                const double dist_g = __shfl_sync(FULL, dq, 0), pdist = __shfl_sync(FULL, dq, 1);
                const int steps_now = sm.steps;
                __syncwarp();  // every lane has read sm.ppx / sm.ppy / sm.steps before lane 0 may rewrite them below
                const int success = dist_g < a.dist_thresh;
                const int trunc = a.max_episode_steps > 0 && steps_now >= a.max_episode_steps && !(success || crash);
                const int done = success || crash || trunc;
                if (lane == 0) {
                    const double pv = sm.pv, pw = sm.pw;
                    double r_s = success ? __dmul_rn(__dmul_rn(1.0, a.r_success), a.r_scale) : 0.0;
                    double r_c = crash ? __dmul_rn(__dmul_rn(-1.0, a.r_crash), a.r_scale) : 0.0;
                    double r_p = __dmul_rn(__dmul_rn(__dsub_rn(pdist, dist_g), a.r_progress), a.r_scale);
                    double r_f = __dmul_rn(__dmul_rn(pv, a.r_forward), a.r_scale);
                    double r_r = __dmul_rn(__dmul_rn(__dmul_rn(-1.0, __dmul_rn(pw, pw)), a.r_rotation), a.r_scale);
                    double r_d = 0.0;
                    if (discomf) r_d = __dmul_rn(__dmul_rn(-__dsub_rn(1.0, mn), a.r_discomfort), a.r_scale);
                    double rew = __dadd_rn(__dadd_rn(__dadd_rn(__dadd_rn(__dadd_rn(r_s, r_c), r_p), r_f), r_r), r_d);
                    a.reward[e] = (float)rew;
                    a.done[e] = (uint8_t)done;
                    if (a.reward_mirror) a.reward_mirror[e] = (float)rew;
                    if (a.done_mirror) a.done_mirror[e] = (uint8_t)done;
                    a.is_success[e] = (uint8_t)success;
                    a.is_crash[e] = (uint8_t)crash;
                    if (a.truncated) a.truncated[e] = (uint8_t)trunc;
                    a.distance[e] = (float)dist_g;
                    int next = PASS_END;
                    if (done && !NEXT && a.auto_reset) {
                        // auto-reset: draw a spawn tuple (and a map) for the next episode
                        sm.noise_std = draw_episode(
                            a.maps, a.spawn_pool, a.num_maps, a.resample_map, a.seed, (uint32_t)(a.env_offset + e),
                            (uint32_t)sm.episode, sm.map, a.noise_lo, a.noise_hi,
                            [&](const double *sp, int nmap) {
                                sm.px = sp[0]; sm.py = sp[1]; sm.gx = sp[2]; sm.gy = sp[3]; sm.th = sp[4];
                                sm.map = nmap;
                            },
                            [&] {  // no pool: restart from the rolled-back pose
                                sm.px = sm.ppx; sm.py = sm.ppy; sm.th = sm.pyaw;
                            });
                        sm.episode += 1;
                        sm.steps = 0;
                        sm.ppx = sm.px; sm.ppy = sm.py; sm.pv = 0; sm.pw = 0; sm.act_v = 0; sm.act_w = 0;
                        next = PASS_RESET;
                    } else if (crash) {  // env.py:707-717: back to the pose / yaw of prev_obs
                        sm.px = sm.ppx; sm.py = sm.ppy; sm.th = sm.pyaw;
                        next = PASS_RESCAN;
                    }
                    sm.next_pass = next;
                }
            }
            __syncthreads();
            pass = sm.next_pass;
            if (pass == PASS_RESET && a.discs_reset != nullptr) {
                nd = min(a.ndisc_reset[e], a.max_disc);
                ns = a.segs_reset ? min(a.nseg_reset[e], a.max_seg) : 0;
            }
            if (pass != PASS_END) continue;
        }
        break;
    }

    PROF_MARK(6);
    // File this environment under its cost class for the next step: the cycles its last scan
    // took (an auto-reset first scan is taken at the pose the next step starts from), doubled
    // when the next step is likely to end the episode and run a second scan -- the robot is
    // within one step of a crash threshold, of the goal, or of the step limit.  Such
    // environments then start first instead of stretching the end of the launch.  The slot in
    // the class list is claimed here and filled in at the very end, so the atomic's round trip
    // overlaps the epilogue.
    int sched_pos = 0, sched_b = 0;
    if (sched_cnt) {
        bool risky = margin < RISK_MARGIN;
        if (tid == 0) {
            const double gx = sm.gx - sm.px, gy = sm.gy - sm.py;
            risky |= gx * gx + gy * gy < (a.dist_thresh + RISK_MARGIN) * (a.dist_thresh + RISK_MARGIN);
            risky |= a.max_episode_steps > 0 && sm.steps + 1 >= a.max_episode_steps;
        }
        risky = __syncthreads_or(risky) && !NEXT && a.auto_reset;
        if (tid == 0) {
            const long long kc = ((clock64() - t_pass) << (risky ? 1 : 0)) >> 13;
            sched_b = NAVGYM_SCHED_BUCKETS - 1 - (int)(kc > NAVGYM_SCHED_BUCKETS - 1 ? NAVGYM_SCHED_BUCKETS - 1 : kc);
            sched_pos = atomicAdd(&sched_cnt[sched_b], 1);
        }
    }
    // ---------------- epilogue (warp 0): observation tail + state (env.py:455, 725-727) ---
    if (warp == 0) {
        double yaw;
        if (sm.th_spec == sm.th) {
            yaw = sm.yaw_spec;  // warp 1 had the final heading right
        } else {
            double sn, cn;
            sincos(sm.th, &sn, &cn);
            yaw = atan2(sn, cn);  // utils.py:5-9
        }
        double tv = 0.0;
        switch (lane) {
        case 0: tv = sm.ppx; break;
        case 1: tv = sm.ppy; break;
        case 2: tv = sm.px; break;
        case 3: tv = sm.py; break;
        case 4: tv = sm.pv; break;
        case 5: tv = sm.pw; break;
        case 6: tv = yaw; break;
        }
        if (lane < 7) {
            orow.set_tail(a.num_scan_stack > 1 ? a.num_scan_stack : 1, lane, (float)tv);
            if (a.tail64) a.tail64[(size_t)e * 7 + lane] = tv;
        }
        double nv = 0.0;
        switch (lane) {
        case NAVGYM_S_PX: nv = sm.px; break;
        case NAVGYM_S_PY: nv = sm.py; break;
        case NAVGYM_S_TH: nv = sm.th; break;
        case NAVGYM_S_GX: nv = sm.gx; break;
        case NAVGYM_S_GY: nv = sm.gy; break;
        case NAVGYM_S_PPX: nv = sm.px; break;
        case NAVGYM_S_PPY: nv = sm.py; break;
        case NAVGYM_S_PYAW: nv = yaw; break;
        case NAVGYM_S_PV: nv = sm.act_v; break;
        case NAVGYM_S_PW: nv = sm.act_w; break;
        }
        if (lane < NAVGYM_NS) ST(lane) = nv;
        if (lane == 0) {
            a.steps[e] = sm.steps;
            a.map_id[e] = sm.map;
            if (a.episodes) a.episodes[e] = sm.episode;
            if (a.noise_std) a.noise_std[e] = sm.noise_std;
            if (MASKED && NEXT) {   // the outputs of a launch that started a new episode
                const double ddx = __dsub_rn(sm.gx, sm.px), ddy = __dsub_rn(sm.gy, sm.py);
                const double dist_g = sqrt(__dadd_rn(__dmul_rn(ddx, ddx), __dmul_rn(ddy, ddy)));
                a.reward[e] = 0.0f;
                a.done[e] = 0;
                if (a.reward_mirror) a.reward_mirror[e] = 0.0f;
                if (a.done_mirror) a.done_mirror[e] = 0;
                a.is_success[e] = 0;
                a.is_crash[e] = 0;
                if (a.truncated) a.truncated[e] = 0;
                a.distance[e] = (float)dist_g;
            }
        }
    }
    if (sched_cnt && tid == 0) sched_list[(size_t)sched_b * B + sched_pos] = e;
    PROF_MARK(7);
#ifdef NAVGYM_PROFILE
    if (tid == 0 && a.tail64) {  // CTA timeline (global ns clock, SM id) for tail analysis
        unsigned long long t_end;
        unsigned smid;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_end));
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        a.tail64[(size_t)e * 7 + 0] = (double)_g_begin;
        a.tail64[(size_t)e * 7 + 1] = (double)t_end;
        a.tail64[(size_t)e * 7 + 2] = (double)smid;
        a.tail64[(size_t)e * 7 + 3] = (double)blockIdx.x;
        a.tail64[(size_t)e * 7 + 4] = (double)sm.prof_alive + 4096.0 * (double)max(sm.prof_cyc_b[0], sm.prof_cyc_b[1]) + 4096.0 * 16777216.0 * (double)max(sm.prof_walk[0], sm.prof_walk[1]);
        a.tail64[(size_t)e * 7 + 5] = (double)max(sm.prof_iters_a[0], sm.prof_iters_a[1]);
        a.tail64[(size_t)e * 7 + 6] = (double)max(sm.prof_rounds_b[0], sm.prof_rounds_b[1]);
    }
#endif
#undef ST
#undef BEAM
}

// Launch order.  With a schedule buffer, teams take environments in descending order of the
// cycles they cost in the previous step (they change slowly from step to step): position p of
// the order is the p-th entry of the concatenated cost-class lists, NAVGYM_SCHED_BUCKETS classes,
// class 0 = most expensive (a warp-wide prefix scan over the class counts finds it).
__device__ __forceinline__ int sched_lookup(const navgym_step_args_t &a, const int pos, int *&sched_cnt, int *&sched_list)
{
    const int B = a.num_envs, lane = threadIdx.x & 31;
    const int cur = a.sched_phase, nxt = (a.sched_phase + 1) % 3, clr = (a.sched_phase + 2) % 3;
    int *cnt = a.sched;                                   // [3][NBK]
    int *lst = a.sched + 3 * NAVGYM_SCHED_BUCKETS;        // [3][NBK][B]
    const int c = cnt[cur * NAVGYM_SCHED_BUCKETS + lane];
    int incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    const unsigned m = __ballot_sync(0xffffffffu, pos < incl);
    const int b = m ? __ffs(m) - 1 : 31;
    const int excl = __shfl_sync(0xffffffffu, incl - c, b);
    sched_cnt = cnt + nxt * NAVGYM_SCHED_BUCKETS;
    sched_list = lst + (size_t)nxt * NAVGYM_SCHED_BUCKETS * B;
    if (blockIdx.x == 0 && threadIdx.x < NAVGYM_SCHED_BUCKETS) cnt[clr * NAVGYM_SCHED_BUCKETS + threadIdx.x] = 0;
    return lst[((size_t)cur * NAVGYM_SCHED_BUCKETS + b) * B + (pos - excl)];
}

// One CTA (2 warps) = one environment; CTA b of the launch takes the b-th environment of the
// launch order.  COOP selects tail regime B (march_tail_dealt): it shortens the launch's slowest
// environments at the price of ~4 % more gathers and instructions, which pays while a launch is
// at most ~2 waves of CTAs (4096 envs: -16 %) and costs beyond (32768 envs: +7 %).  FMT is the
// observation row format (NAVGYM_OBS_F32 / F16, ObsRow): it only changes the row stores.
// MODE_NEXT_STEP (auto_reset == NAVGYM_AUTORESET_NEXT_STEP): an environment whose done byte is
// set on entry starts its next episode instead of stepping; the others step with auto-reset off.
// Every thread of the CTA reads the byte before the first barrier of the body, and only this CTA
// writes it, after that barrier: the choice is CTA-uniform.
template <int MODE, bool COOP, int FMT>
__global__ void __launch_bounds__(NAVGYM_CTA_THREADS, NAVGYM_CTAS_PER_SM) step_kernel(const navgym_step_args_t a)
{
    static_assert(MODE == MODE_STEP || MODE == MODE_RESET || MODE == MODE_NEXT_STEP,
                  "the masked reset is reset_envs_kernel");
    __shared__ EnvSmem sm;
    int e = a.env_begin + (int)blockIdx.x;
    int *sched_cnt = nullptr, *sched_list = nullptr;
    if ((MODE == MODE_STEP || MODE == MODE_NEXT_STEP) && a.sched) e = sched_lookup(a, (int)blockIdx.x, sched_cnt, sched_list);
    if constexpr (MODE == MODE_NEXT_STEP) {
        if (a.done[e]) step_body<MODE_MASKED_RESET, COOP, FMT, true>(a, sm, e, (int)threadIdx.x, sched_cnt, sched_list);
        else step_body<MODE_STEP, COOP, FMT, true>(a, sm, e, (int)threadIdx.x, sched_cnt, sched_list);
    } else {
        step_body<MODE, COOP, FMT>(a, sm, e, (int)threadIdx.x, sched_cnt, sched_list);
    }
}

// The masked reset (navgym_reset_envs): CTA b takes environment env_begin + b in index order and
// returns at once when its mask byte is 0; `sched` is neither read nor written.
template <bool COOP, int FMT>
__global__ void __launch_bounds__(NAVGYM_CTA_THREADS, NAVGYM_CTAS_PER_SM)
reset_envs_kernel(const navgym_step_args_t a, const uint8_t *__restrict__ mask)
{
    __shared__ EnvSmem sm;
    const int e = a.env_begin + (int)blockIdx.x;
    if (!mask[e]) return;
    step_body<MODE_MASKED_RESET, COOP, FMT>(a, sm, e, (int)threadIdx.x, nullptr, nullptr);
}
