// pedestrian_kernels.cuh -- part of navgym_b200.cu (included there; one translation unit).
// The pedestrians of env.py:617-693 on the device: their lidar, route following, motion, and
// the geometry the robot's lidar sees.
// ------------------------------------------------------------------ pedestrian lidar
// The scan every simulated pedestrian takes of its surroundings (env.py:683-693): map raycast
// from its own pose + the closed footprints of the robot and the other pedestrians, clipped,
// no noise.  One CTA per agent, threads across beams; the same canonical march / segment
// arithmetic as the robot's scan.
// World-frame closed footprint of an agent at (x, y, th) as 4 segments (env.py:408-414):
// float64 rotation + translation, vertices rounded to float32.
__device__ __forceinline__ void footprint_segments(double x, double y, double th, const double *fp, float4 *out)
{
    const double c = cos(th), s = sin(th);
    float wx[4], wy[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        wx[i] = (float)(c * fp[2 * i] - s * fp[2 * i + 1] + x);
        wy[i] = (float)(s * fp[2 * i] + c * fp[2 * i + 1] + y);
    }
#pragma unroll
    for (int i = 0; i < 4; i++) out[i] = make_float4(wx[i], wy[i], wx[(i + 1) & 3], wy[(i + 1) & 3]);
}

#define NAVGYM_SCAN_AGENTS 127  // crowd mode: agents per environment (+ the robot = one thread each)
// Fallback for beam tables of more than NB entries: one thread per beam, every segment tested
// against every beam.
__global__ void __launch_bounds__(128) agent_scan_generic_kernel(const navgym_scan_args_t a)
{
    const int n = blockIdx.x;
    const int e = n / a.agents_per_env, slot = n - e * a.agents_per_env;
    if (a.env_mask && !a.env_mask[e]) return;
    const int live = a.nagent ? min(a.nagent[e], a.agents_per_env) : a.agents_per_env;
    if (slot >= live) return;
    const double *p = a.pose + (size_t)n * 3;
    const float lx = (float)p[0], ly = (float)p[1], lt = (float)p[2];  // env.py:386
    const navgym_map_t m = a.maps[a.map_id[e]];
    const float *dist = a.edt_pool + m.edt_offset;
    const int ci = xy_to_cell(lx, m.ox, m.res, m.H, a.cell_rule);
    const int cj = xy_to_cell(ly, m.oy, m.res, m.W, a.cell_rule);
    const float max_range = (float)((double)m.W * (double)m.H);
    const float t_stop = a.t_stop > 0.0f ? fminf(a.t_stop, max_range) : max_range;
    const float res32 = (float)m.res;
    int ns = 0, s0 = -1, s1 = -1;
    const float4 *segs = nullptr;
    if (a.segs) {
        ns = a.nseg ? min(a.nseg[e], a.max_seg) : 0;
        segs = reinterpret_cast<const float4 *>(a.segs) + (size_t)e * a.max_seg;
        if (a.skip) { s0 = a.skip[2 * (size_t)n]; s1 = s0 + a.skip[2 * (size_t)n + 1]; }
    }
    for (int k = threadIdx.x; k < a.num_beams; k += blockDim.x) {
        const float h = (float)__dadd_rn(a.lin[k], (double)lt);
        double sd, cd;
        dir_sincos((double)h, sd, cd);
        const float dx = (float)cd, dy = (float)sd;
        int hx, hy;
        float r = __fmul_rn(march(dist, m.W, m.H, (float)ci, (float)cj, dx, dy, max_range, t_stop, hx, hy), res32);
        for (int s = 0; s < ns; s++) {
            if (s >= s0 && s < s1) continue;
            const float4 sg = segs[s];
            r = fminf(r, seg_hit(lx, ly, dx, dy, sg.x, sg.y, sg.z, sg.w));
        }
        a.ranges[(size_t)n * a.num_beams + k] = fminf(fmaxf(r, 0.0f), a.range_max);
    }
}

// Beams that can see a segment: a conservative angular window (bearing of the segment's ends
// +- 2 beams; beam k of an evenly spaced table looks along amin + k step + theta), as beam indices
// [k0, k0 + cnt) -- and the same window 2 pi lower, [k1, k1 + cnt): a lidar of less than 360
// degrees has no beam at most of those indices, a full one wraps around.  Beams outside cannot hit,
// so testing only the window equals the all-beams loop bit for bit.  Segments wholly beyond
// `reach_max` get an empty window: a hit would be clipped to range_max afterwards -- the same
// value as no hit (env.py:435).
__device__ __forceinline__ int4 segment_window(const float4 sg, float lx, float ly, float lt, float amin, float step,
                                               int K, float reach_max)
{
    const float ax = sg.x, ay = sg.y, bx = sg.z, by = sg.w;
    const float da2 = (ax - lx) * (ax - lx) + (ay - ly) * (ay - ly);
    const float db2 = (bx - lx) * (bx - lx) + (by - ly) * (by - ly);
    const float len2 = (bx - ax) * (bx - ax) + (by - ay) * (by - ay);
    const float reach = reach_max * 1.001f + sqrtf(len2) + 0.01f;
    if (fminf(da2, db2) > reach * reach) return make_int4(0, 0, 0, 0);
    const float pa = atan2f(ay - ly, ax - lx), pb = atan2f(by - ly, bx - lx);
    float dl = pb - pa;
    dl -= 6.2831853f * rintf(dl * 0.15915494f);
    if (fabsf(dl) > 3.0f || da2 < 1e-6f || db2 < 1e-6f) return make_int4(0, 0, K, 0);
    float rel = (dl >= 0 ? pa : pb) - lt - amin;
    rel -= 6.2831853f * floorf(rel * 0.15915494f);
    const int cnt = (int)ceilf(fabsf(dl) / step) + 5;
    if (cnt >= K) return make_int4(0, 0, K, 0);
    return make_int4((int)floorf(rel / step) - 2, (int)floorf((rel - 6.2831853f) / step) - 2, cnt, 0);
}

// One CTA per agent, threads across beams.  The segments the agent can see (crowd mode: the
// footprints of the robot and the other agents in range, built here; else the environment's list
// minus the agent's own) are staged in shared memory with their beam windows, so a beam only
// evaluates the few segments whose window covers it; the first march sample, on the origin cell,
// is shared by all beams (as in the robot's scan).  Requires an evenly spaced, ascending beam
// table (np.linspace: what the reference builds, env.py:388-390, and what pymap2d's renderers
// assume); more than NAVGYM_SCAN_SEGS listed segments fall back to agent_scan_generic_kernel.
#define NAVGYM_SCAN_SEGS (4 * (NAVGYM_SCAN_AGENTS + 1))
constexpr int AGENT_MIN_CTAS = 12;   // 40 registers: the kernel waits on its EDT gathers, 48 resident warps beat 36 (0.406 -> 0.350 ms for 40 960 agents)
__device__ __forceinline__ void agent_scan_one(const navgym_scan_args_t &a, const int n, float4 *near_segs, int4 *near_win, int &n_near)
{
    const int e = n / a.agents_per_env, slot = n - e * a.agents_per_env;
    if (a.env_mask && !a.env_mask[e]) return;
    const int live = a.nagent ? min(a.nagent[e], a.agents_per_env) : a.agents_per_env;
    if (slot >= live) return;
    const int K = a.num_beams;
    const double *p = a.pose + (size_t)n * 3;
    const float lx = (float)p[0], ly = (float)p[1], lt = (float)p[2];  // env.py:386
    const navgym_map_t m = a.maps[a.map_id[e]];
    const float *dist = a.edt_pool + m.edt_offset;
    const int W = m.W, H = m.H;
    const int ci = xy_to_cell(lx, m.ox, m.res, m.H, a.cell_rule);
    const int cj = xy_to_cell(ly, m.oy, m.res, m.W, a.cell_rule);
    const float x0 = (float)ci, y0 = (float)cj;
    const float max_range = (float)((double)m.W * (double)m.H);
    const float t_stop = a.t_stop > 0.0f ? fminf(a.t_stop, max_range) : max_range;
    const float res32 = (float)m.res;
    const float amin = (float)a.lin[0];
    const float bstep = K > 1 ? (float)((a.lin[K - 1] - a.lin[0]) / (double)(K - 1)) : 1.0f;
    if (threadIdx.x == 0) n_near = 0;
    __syncthreads();
    if (a.segs) {
        const int ns = a.nseg ? min(a.nseg[e], a.max_seg) : 0;
        const float4 *segs = reinterpret_cast<const float4 *>(a.segs) + (size_t)e * a.max_seg;
        int s0 = -1, s1 = -1;
        if (a.skip) { s0 = a.skip[2 * (size_t)n]; s1 = s0 + a.skip[2 * (size_t)n + 1]; }
        for (int s = threadIdx.x; s < ns; s += blockDim.x) {   // host: max_seg <= NAVGYM_SCAN_SEGS
            if (s >= s0 && s < s1) continue;
            const float4 sg = segs[s];
            const int4 w = segment_window(sg, lx, ly, lt, amin, bstep, K, a.range_max);
            if (w.z > 0) {
                const int at = atomicAdd(&n_near, 1);
                near_segs[at] = sg;
                near_win[at] = w;
            }
        }
    } else if (a.robot_state) {
        // crowd mode: thread 0 = the robot, thread 1 + j = agent j of this environment
        const int o = threadIdx.x;
        if (o <= live && o != slot + 1) {  // host: agents_per_env <= NAVGYM_SCAN_AGENTS
            double ox, oy, oth;
            const double *fp;
            if (o == 0) {
                const size_t B = (size_t)a.num_envs;
                ox = a.robot_state[NAVGYM_S_PX * B + e]; oy = a.robot_state[NAVGYM_S_PY * B + e];
                oth = a.robot_state[NAVGYM_S_TH * B + e];
                fp = a.robot_fp;
            } else {
                const double *q = a.pose + ((size_t)e * a.agents_per_env + (o - 1)) * 3;
                ox = q[0]; oy = q[1]; oth = q[2];
                fp = a.agent_fp;
            }
            float reach = 0.0f;  // farthest footprint vertex from the body origin
#pragma unroll
            for (int i = 0; i < 4; i++) reach = fmaxf(reach, hypotf((float)fp[2 * i], (float)fp[2 * i + 1]));
            const float dc = hypotf((float)ox - lx, (float)oy - ly);
            if (dc <= a.range_max + reach + 0.01f) {
                float4 sg[4];
                footprint_segments(ox, oy, oth, fp, sg);
                const int at = atomicAdd(&n_near, 4);
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    near_segs[at + i] = sg[i];
                    near_win[at + i] = segment_window(sg[i], lx, ly, lt, amin, bstep, K, a.range_max);
                }
            }
        }
    }
    __syncthreads();
    const int ns = n_near;
    // every beam starts on the origin cell: that sample is the same for all of them
    const bool o_in = ((unsigned)ci < (unsigned)W) & ((unsigned)cj < (unsigned)H);
    const float d0 = o_in ? __ldg(dist + cj * W + ci) : 1.0f;
    const float t1 = fmaxf(__fmul_rn(d0, 0.999f), 1.0f);
    for (int k = threadIdx.x; k < K; k += blockDim.x) {
        const float h = (float)__dadd_rn(a.lin[k], (double)lt);
        double sd, cd;
        dir_sincos((double)h, sd, cd);
        const float dx = (float)cd, dy = (float)sd;
        float rc = max_range;
        if (o_in & (d0 <= 0.0f)) {
            rc = 0.0f;
        } else if (o_in) {
            float t = t1;
            while (t < t_stop) {
                const int px = __float2int_rz(march_pos(dx, t, x0));
                const int py = __float2int_rz(march_pos(dy, t, y0));
                if ((unsigned)px >= (unsigned)W || (unsigned)py >= (unsigned)H) break;
                const float d = __ldg(dist + (unsigned)(py * W + px));
                if (d <= 0.0f) {
                    const float xd = (float)(px - ci), yd = (float)(py - cj);
                    rc = __fsqrt_rn(__fadd_rn(__fmul_rn(xd, xd), __fmul_rn(yd, yd)));
                    break;
                }
                t = __fadd_rn(t, fmaxf(__fmul_rn(d, 0.999f), 1.0f));
            }
        }
        float r = __fmul_rn(rc, res32);
        for (int s = 0; s < ns; s++) {
            const int4 w = near_win[s];
            if ((unsigned)(k - w.x) < (unsigned)w.z || (unsigned)(k - w.y) < (unsigned)w.z) {
                const float4 sg = near_segs[s];
                r = fminf(r, seg_hit(lx, ly, dx, dy, sg.x, sg.y, sg.z, sg.w));
            }
        }
        a.ranges[(size_t)n * K + k] = fminf(fmaxf(r, 0.0f), a.range_max);
    }
}

// One CTA per agent; CTAs of unmasked environments / dead slots exit at once.  (Round 2 tried one CTA
// per 128 consecutive agents that lists the masked ones and scans them in turn for the ~1 % masked
// launches: an environment's agents are consecutive, so its ten scans ran one after the other in one
// CTA and the crowd step lost 0.23 ms; the full grid costs 25-44 us.)
__global__ void __launch_bounds__(128, AGENT_MIN_CTAS) agent_scan_kernel(const navgym_scan_args_t a)
{
    __shared__ float4 near_segs[NAVGYM_SCAN_SEGS];
    __shared__ int4 near_win[NAVGYM_SCAN_SEGS];
    __shared__ int n_near;
    agent_scan_one(a, (int)blockIdx.x, near_segs, near_win, n_near);
}

// ------------------------------------------------------------------ pedestrian routes
// (include/navgym_b200.h, navgym_plan_args_t.)  One thread per pedestrian.
__device__ __forceinline__ int plan_cell(double v, double origin, double res, int dim)
{
    int c = (int)floor((v - origin) / res);
    return c < 0 ? 0 : (c >= dim ? dim - 1 : c);
}

// From cell (cx, cy) walk the field downhill until the cell centre is more than 2 m from the
// starting point (sx, sy) or the goal cell is reached.  Returns false on an unreachable cell.
__device__ __forceinline__ bool plan_advance(const uint16_t *f, const navgym_plan_map_t &m, int cx, int cy,
                                             double sx, double sy, double &wx, double &wy, bool &is_goal)
{
    unsigned d = f[cy * m.W + cx];
    is_goal = false;
    if (d == 65535u) return false;
    for (int it = 0; it < 64; it++) {
        if (d == 0u) { is_goal = true; break; }
        int bx = cx, by = cy;
        unsigned bd = d;
        if (cx > 0 && f[cy * m.W + cx - 1] < bd) { bd = f[cy * m.W + cx - 1]; bx = cx - 1; by = cy; }
        if (cx + 1 < m.W && f[cy * m.W + cx + 1] < bd) { bd = f[cy * m.W + cx + 1]; bx = cx + 1; by = cy; }
        if (cy > 0 && f[(cy - 1) * m.W + cx] < bd) { bd = f[(cy - 1) * m.W + cx]; bx = cx; by = cy - 1; }
        if (cy + 1 < m.H && f[(cy + 1) * m.W + cx] < bd) { bd = f[(cy + 1) * m.W + cx]; bx = cx; by = cy + 1; }
        if (bd >= d) break;  // local minimum that is not the goal: cannot happen on a BFS field
        cx = bx; cy = by; d = bd;
        wx = m.ox + (cx + 0.5) * m.res;
        wy = m.oy + (cy + 0.5) * m.res;
        if ((wx - sx) * (wx - sx) + (wy - sy) * (wy - sy) > 4.0) return true;
    }
    wx = m.ox + (cx + 0.5) * m.res;
    wy = m.oy + (cy + 0.5) * m.res;
    return true;
}

__global__ void peds_plan_kernel(const navgym_plan_args_t a)
{
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= a.num_envs * a.max_ped) return;
    const int e = n / a.max_ped, slot = n - e * a.max_ped;
    if (a.nped && slot >= a.nped[e]) return;
    const navgym_plan_map_t m = a.maps[a.map_id[e]];
    if (a.respawn && a.respawn[e] && a.cand_pose) {
        // env.py:785-806: the pedestrian drawn for this episode by the previous call
        for (int i = 0; i < 3; i++) a.pose_rw[3 * (size_t)n + i] = a.cand_pose[3 * (size_t)n + i];
        a.v_pref[n] = a.cand_v_pref[n];
        a.has_legs[n] = a.cand_legs[n];
        a.goal_id[n] = a.cand_goal[n];
        a.waypoint[2 * (size_t)n] = CUDART_NAN;
        a.waypoint[2 * (size_t)n + 1] = CUDART_NAN;
        for (int i = 0; i < 3; i++) a.dist_travelled[3 * (size_t)n + i] = 0.0;
        a.vel[2 * (size_t)n] = a.vel[2 * (size_t)n + 1] = 0.0;
        a.prev_action[2 * (size_t)n] = a.prev_action[2 * (size_t)n + 1] = 0.0f;
    }
    const double px = a.pose[3 * (size_t)n], py = a.pose[3 * (size_t)n + 1], th = a.pose[3 * (size_t)n + 2];
    const int cx = plan_cell(px, m.ox, m.res, m.W), cy = plan_cell(py, m.oy, m.res, m.H);
    const size_t fsz = (size_t)m.W * m.H;
    int g = a.goal_id[n];
    const double *goals = a.goals + 2 * m.goal_offset;
    double gx = goals[2 * g], gy = goals[2 * g + 1];
    double wx = a.waypoint[2 * (size_t)n], wy = a.waypoint[2 * (size_t)n + 1];
    // 1. arrived (env.py:666-668): a new goal, if one qualifies
    if ((px - gx) * (px - gx) + (py - gy) * (py - gy) < 0.25) {
        const uint4 r = philox4x32_10(make_uint4((uint32_t)(a.env_offset + e), (uint32_t)slot, (uint32_t)a.step, 0x9ed5u),
                                      make_uint2((uint32_t)a.seed, (uint32_t)(a.seed >> 32)));
        const uint32_t draws[4] = {r.x, r.y, r.z, r.w};
        for (int i = 0; i < 4; i++) {
            const int c = (int)(((uint64_t)draws[i] * (uint64_t)m.num_goals) >> 32);
            const double qx = goals[2 * c], qy = goals[2 * c + 1];
            const double dd = (qx - px) * (qx - px) + (qy - py) * (qy - py);
            if (c != g && dd > a.min_goal_dist * a.min_goal_dist &&
                a.fields[m.field_offset + c * fsz + (size_t)cy * m.W + cx] != 65535u) {
                g = c; gx = qx; gy = qy;
                wx = CUDART_NAN;
                break;
            }
        }
        a.goal_id[n] = g;
    }
    const uint16_t *f = a.fields + m.field_offset + g * fsz;
    // 2. / 3. the waypoint: first one from here, later ones from the previous waypoint
    bool is_goal = (wx == gx) & (wy == gy);
    if (wx != wx) {
        if (!plan_advance(f, m, cx, cy, px, py, wx, wy, is_goal)) { wx = gx; wy = gy; is_goal = true; }
        if (is_goal) { wx = gx; wy = gy; }
    }
    for (int it = 0; it < 8 && !is_goal && (px - wx) * (px - wx) + (py - wy) * (py - wy) < 1.0; it++) {
        const double sx = wx, sy = wy;
        if (!plan_advance(f, m, plan_cell(sx, m.ox, m.res, m.W), plan_cell(sy, m.oy, m.res, m.H), sx, sy, wx, wy, is_goal)) {
            is_goal = true;
        }
        if (is_goal) { wx = gx; wy = gy; }
    }
    a.waypoint[2 * (size_t)n] = wx;
    a.waypoint[2 * (size_t)n + 1] = wy;
    // env.py:641-645: the goal in the pedestrian's frame
    const double c = cos(th), s = sin(th);
    a.goal_local[2 * (size_t)n] = (float)((wx - px) * c + (wy - py) * s);
    a.goal_local[2 * (size_t)n + 1] = (float)(-(wx - px) * s + (wy - py) * c);

    // ---- the pedestrian of this slot in the environment's next episode
    if (a.cand_pose) {
        const size_t B = (size_t)a.num_envs;
        const uint32_t ge = (uint32_t)(a.env_offset + e);
        double rx = a.robot_state[NAVGYM_S_PX * B + e], ry = a.robot_state[NAVGYM_S_PY * B + e];
        int nmap = a.map_id[e];
        if (a.cand_next_spawn && a.robot_maps) {
            // the spawn tuple step_kernel draws on auto-reset and navgym_reset_envs draws
            // (draw_episode in device_helpers.cuh: keep in step with it -- spelled out here because
            // routing this kernel through the helper changes its register allocation)
            const uint4 rnd = philox4x32_10(make_uint4(ge, (uint32_t)(a.episodes ? a.episodes[e] : 0), 0x5eedu, 0xfffffff0u),
                                            make_uint2((uint32_t)a.robot_seed, (uint32_t)(a.robot_seed >> 32)));
            int cand_map = nmap;
            if (a.resample_map && a.num_maps > 1) cand_map = (int)(((uint64_t)rnd.y * (uint64_t)a.num_maps) >> 32);
            const navgym_map_t m2 = a.robot_maps[cand_map];
            if (m2.spawn_count > 0) {
                const long long row = m2.spawn_offset + (long long)(((uint64_t)rnd.x * (uint64_t)m2.spawn_count) >> 32);
                rx = a.spawn_pool[row * 5];
                ry = a.spawn_pool[row * 5 + 1];
                nmap = cand_map;
            }
        }
        const navgym_plan_map_t mc = a.maps[nmap];
        const uint2 key = make_uint2((uint32_t)a.seed, (uint32_t)(a.seed >> 32));
        const uint4 r0 = philox4x32_10(make_uint4(ge, (uint32_t)slot, (uint32_t)a.step, 0x5b0au), key);
        const uint4 r1 = philox4x32_10(make_uint4(ge, (uint32_t)slot, (uint32_t)a.step, 0x5b0bu), key);
        const uint4 r2 = philox4x32_10(make_uint4(ge, (uint32_t)slot, (uint32_t)a.step, 0x5b0cu), key);
        // spawn (env.py:786-797): a free, goal-connected cost-map cell at least min_robot_dist
        // from the robot's start; of 8 draws the first that qualifies, else the farthest -- and
        // if even that one is too close (or the map has no free cell) the slot sits the episode
        // out, parked outside the map with zero preferred speed where no lidar sees it
        const uint32_t draws[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
        double sx = mc.ox - 1000.0, sy = mc.oy - 1000.0, best = -1.0;
        for (int i = 0; i < 8 && mc.free_count > 0; i++) {
            const long long row = mc.free_offset + (long long)(((uint64_t)draws[i] * (uint64_t)mc.free_count) >> 32);
            const double qx = a.free_xy[2 * row], qy = a.free_xy[2 * row + 1];
            const double dd = (qx - rx) * (qx - rx) + (qy - ry) * (qy - ry);
            if (dd > best) { best = dd; sx = qx; sy = qy; }
            if (dd >= a.min_robot_dist * a.min_robot_dist) break;
        }
        const bool parked = best < a.min_robot_dist * a.min_robot_dist;
        if (parked) { sx = mc.ox - 1000.0; sy = mc.oy - 1000.0; }
        const double cth = 6.283185307179586 * (double)u01(r2.x);
        const bool legs = (double)u01(r2.z) < a.has_legs_ratio;
        // goal (env.py:370-381): a goal field that reaches the spawn cell, farther than
        // min_goal_dist; up to 5 draws, else the farthest reachable one drawn
        int cgoal = (int)(((uint64_t)r2.w * (uint64_t)mc.num_goals) >> 32);
        if (!parked) {
            const uint4 r3 = philox4x32_10(make_uint4(ge, (uint32_t)slot, (uint32_t)a.step, 0x5b0du), key);
            const uint32_t gd[5] = {r2.w, r3.x, r3.y, r3.z, r3.w};
            const int scx = plan_cell(sx, mc.ox, mc.res, mc.W), scy = plan_cell(sy, mc.oy, mc.res, mc.H);
            const size_t csz = (size_t)mc.W * mc.H;
            const double *cg = a.goals + 2 * mc.goal_offset;
            double gbest = -1.0;
            for (int i = 0; i < 5; i++) {
                const int c = (int)(((uint64_t)gd[i] * (uint64_t)mc.num_goals) >> 32);
                if (a.fields[mc.field_offset + c * csz + (size_t)scy * mc.W + scx] == 65535u) continue;
                const double dd = (cg[2 * c] - sx) * (cg[2 * c] - sx) + (cg[2 * c + 1] - sy) * (cg[2 * c + 1] - sy);
                if (dd > gbest) { gbest = dd; cgoal = c; }
                if (dd > a.min_goal_dist * a.min_goal_dist) break;
            }
        }
        a.cand_pose[3 * (size_t)n] = sx;
        a.cand_pose[3 * (size_t)n + 1] = sy;
        a.cand_pose[3 * (size_t)n + 2] = cth;
        a.cand_v_pref[n] = parked ? 0.0 : a.v_pref_lo + (a.v_pref_hi - a.v_pref_lo) * (double)u01(r2.y);
        a.cand_legs[n] = legs;
        a.cand_goal[n] = cgoal;
        float *q = a.cand_rows + (size_t)n * NAVGYM_PED_F;
        q[0] = (float)sx; q[1] = (float)sy; q[2] = (float)cth;
        q[9] = 0.0f; q[10] = 0.0f; q[11] = 0.0f;
        q[12] = legs ? 1.0f : 0.0f;
    }
}

// ------------------------------------------------------------------ pedestrian motion
// (include/navgym_b200.h, navgym_move_args_t.)  One thread per pedestrian.
__global__ void peds_move_kernel(const navgym_move_args_t a)
{
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= a.num_envs * a.max_ped) return;
    const int e = n / a.max_ped, slot = n - e * a.max_ped;
    if (a.nped && slot >= a.nped[e]) return;
    // env.py:655-661
    const float m0 = fminf(fmaxf(a.mean[2 * (size_t)n], 0.0f), 1.0f);
    const float m1 = fminf(fmaxf(a.mean[2 * (size_t)n + 1], -1.0f), 1.0f);
    a.prev_action[2 * (size_t)n] = m0;
    a.prev_action[2 * (size_t)n + 1] = m1;
    const double factor = a.v_pref[n];
    const double v = (double)m0 * factor, w = (double)m1 * factor;
    // human.py:32-41
    double x = a.pose[3 * (size_t)n], y = a.pose[3 * (size_t)n + 1];
    const double th0 = a.pose[3 * (size_t)n + 2];
    const double vx = v * cos(th0), vy = v * sin(th0);
    const double th1 = th0 + w * a.dt;
    x = x + cos(th1) * v * a.dt;
    y = y + sin(th1) * v * a.dt;
    const double twopi = 6.283185307179586;
    double th = fmod(th1, twopi);
    if (th != 0 && th < 0) th += twopi;
    a.pose[3 * (size_t)n] = x;
    a.pose[3 * (size_t)n + 1] = y;
    a.pose[3 * (size_t)n + 2] = th;
    a.vel[2 * (size_t)n] = vx;
    a.vel[2 * (size_t)n + 1] = vy;
    // env.py:237-255: rotation rate from the previous observation's yaw, world velocity into
    // the base frame (pose2d inverse_pose2d / apply_tf_to_vel written out), integrated
    const double prev_yaw = atan2(sin(th0), cos(th0));
    const double vrot = (th - prev_yaw) / a.dt;
    const double c = cos(th), s = sin(th);
    double *d = a.dist_travelled + 3 * (size_t)n;
    d[0] += (c * vx + s * vy) * a.dt;
    d[1] += (-s * vx + c * vy) * a.dt;
    d[2] += vrot * a.dt;
    float *q = a.rows + (size_t)n * NAVGYM_PED_F;
    q[0] = (float)x; q[1] = (float)y; q[2] = (float)th;
    q[9] = (float)d[0]; q[10] = (float)d[1]; q[11] = (float)d[2];
    q[12] = a.has_legs[n] ? 1.0f : 0.0f;
}

// ------------------------------------------------------------------ scripted pedestrians
// Pedestrian motion + geometry for the batched simulator (SURVEY §8f row 2, scripted stand-in
// for the reference's CNN-driven humans whose weights are absent): each pedestrian walks
// between two waypoints at its preferred speed with Human.set_vel's unicycle update
// (human.py:32-41), turning at <= 1 rad/s toward the current target, and its leg-gait odometry
// advances as in _update_dist_travelled (env.py:237-255).  Emits what the robot's lidar sees:
// two leg discs (pymap2d CSimAgent "legs") for legged pedestrians, the 0.44 x 0.38 m box
// footprint (human.py:5-10) as four segments otherwise (env.py:398-414), or one trunk disc
// per pedestrian in trunk mode.  One warp per environment, one lane per pedestrian (the
// trigonometry of all pedestrians of an environment runs side by side; a thread per environment
// walked them one after the other); the slots of the disc / segment lists are handed out in
// pedestrian order by a warp prefix sum, so the lists are those of the sequential loop.
__global__ void __launch_bounds__(128) peds_advance_kernel(const navgym_peds_args_t a)
{
    const int e = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (e >= a.num_envs) return;
    const int P = a.nped ? min(a.nped[e], a.max_ped) : a.max_ped;
    float *pp = a.peds + (size_t)e * a.max_ped * NAVGYM_PED_F;
    float *discs = a.discs + (size_t)e * a.max_disc * 3;
    float *segs = a.segs ? a.segs + (size_t)e * a.max_seg * 4 : nullptr;
    int nd = 0, ns = 0;   // warp-uniform running totals
    for (int p0 = 0; p0 < P; p0 += 32) {
        const int p = p0 + lane;
        const bool live = p < P;
        // the pedestrian's row as four 16-byte loads: {x, y, theta, speed} {waypoint a, waypoint b}
        // {target, distance travelled x, y, theta} {has_legs, trunk radius, -, -}
        float4 *q4 = reinterpret_cast<float4 *>(pp + (live ? p : 0) * NAVGYM_PED_F);
        float4 r0 = q4[0], r2 = q4[2];
        const float4 r1 = q4[1], r3 = q4[3];
        float x = r0.x, y = r0.y, th = r0.z;
        if (live && a.advance) {
            const float v = r0.w;
            float tgt = r2.x;
            float gx = tgt > 0.5f ? r1.z : r1.x, gy = tgt > 0.5f ? r1.w : r1.y;
            if ((gx - x) * (gx - x) + (gy - y) * (gy - y) < 0.25f) {  // reached: turn back
                tgt = 1.0f - tgt;
                gx = tgt > 0.5f ? r1.z : r1.x;
                gy = tgt > 0.5f ? r1.w : r1.y;
            }
            float err = atan2f(gy - y, gx - x) - th;
            err -= 6.2831853f * rintf(err * 0.15915494f);
            const float w = fminf(fmaxf(err / a.dt, -1.0f), 1.0f);
            const float vx = v * cosf(th), vy = v * sinf(th);  // human.py:35-36 (old heading)
            const float thn = th + w * a.dt;
            x += cosf(thn) * v * a.dt;
            y += sinf(thn) * v * a.dt;
            // leg gait odometry in the base frame (env.py:251-255)
            const float c = cosf(thn), s_ = sinf(thn);
            r2.y += (c * vx + s_ * vy) * a.dt;
            r2.z += (-s_ * vx + c * vy) * a.dt;
            r2.w += w * a.dt;
            th = thn - 6.2831853f * floorf(thn * 0.15915494f);
            r0.x = x; r0.y = y; r0.z = th; r2.x = tgt;
            q4[0] = r0;
            q4[2] = r2;
        }
        // what this pedestrian contributes: 1 trunk disc | 2 leg discs | 4 box segments
        const bool legs = r3.x > 0.5f;
        const int want_d = !live ? 0 : (a.trunk_mode ? 1 : (legs ? 2 : 0));
        const int want_s = (!live || a.trunk_mode || legs || !segs) ? 0 : 4;
        int pre_d = want_d, pre_s = want_s;   // inclusive warp prefix sums
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int ud = __shfl_up_sync(0xffffffffu, pre_d, o), us = __shfl_up_sync(0xffffffffu, pre_s, o);
            if (lane >= o) { pre_d += ud; pre_s += us; }
        }
        const int at_d = nd + pre_d - want_d, at_s = ns + pre_s - want_s;
        // items of one kind have one size, so "fits after everything before it" is the
        // sequential loop's "fits at the running count"
        const bool put_d = want_d && at_d + want_d <= a.max_disc, put_s = want_s && at_s + want_s <= a.max_seg;
        const float c = cosf(th), s_ = sinf(th);
        if (put_d && a.trunk_mode) {
            discs[3 * at_d] = x; discs[3 * at_d + 1] = y; discs[3 * at_d + 2] = r3.y;
        } else if (put_d) {  // legs (SURVEY App. B.3)
            const float front = 0.3f * cosf(r2.y * (2.0f / 0.3f) + r2.w);
            const float side = 0.1f * cosf(r2.z * (2.0f / 0.1f) + r2.w) + 0.1f;
            discs[3 * at_d] = x + c * front - s_ * side; discs[3 * at_d + 1] = y + s_ * front + c * side;
            discs[3 * at_d + 2] = 0.03f;
            discs[3 * at_d + 3] = x - c * front + s_ * side; discs[3 * at_d + 4] = y - s_ * front - c * side;
            discs[3 * at_d + 5] = 0.03f;
        }
        if (put_s) {  // box footprint, closed
            const float fx[4] = {0.22f, -0.22f, -0.22f, 0.22f}, fy[4] = {0.19f, 0.19f, -0.19f, -0.19f};
            float wx[4], wy[4];
#pragma unroll
            for (int i = 0; i < 4; i++) { wx[i] = c * fx[i] - s_ * fy[i] + x; wy[i] = s_ * fx[i] + c * fy[i] + y; }
#pragma unroll
            for (int i = 0; i < 4; i++)
                *reinterpret_cast<float4 *>(segs + 4 * (at_s + i)) = make_float4(wx[i], wy[i], wx[(i + 1) & 3], wy[(i + 1) & 3]);
        }
        nd += __popc(__ballot_sync(0xffffffffu, put_d)) * (a.trunk_mode ? 1 : 2);
        ns += __popc(__ballot_sync(0xffffffffu, put_s)) * 4;
    }
    if (lane == 0) {
        a.ndisc[e] = nd;
        if (a.nseg) a.nseg[e] = ns;
    }
}
