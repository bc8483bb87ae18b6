"""Policy-driven pedestrians on the device (SURVEY 8f row 2; reference env.py:617-693).

The reference moves every pedestrian with a small CNN policy (human_policy.py:19-71) fed with
the pedestrian's own 512-beam 180 deg / 6 m lidar scan, its local goal and its previous action,
then re-scans the world from each pedestrian's new pose.  Here the same pipeline runs batched
over [num_envs, max_ped] on the GPU:

  agent_scans()            navgym_agent_scan_batch: every pedestrian's scan in one launch
  HumanPolicy              the reference architecture in torch, which holds the weights (its
                           pretrained weights, human_policy.pth, are not distributed: load
                           them with load_state_dict when available, else random-init)
  NativePolicy             HumanPolicy's action mean through the library's own kernels
  PedestrianSim            device state + the per-step sequence of env.py:617-693

Everything on the per-step path is a kernel of the library, the policy forward included
(NativePolicy: both convolutions, act_fc1 and act_fc2 on the tcgen05 tensor cores, DESIGN 4.3);
torch owns the device memory.  Nothing here touches the CPU oracle.
"""
import ctypes as C
import operator

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib
from .robot import Human, KetiRobot, beam_table


class HumanPolicy(nn.Module):
    """Actor / critic of human_policy.py:19-71 with the reference's parameter names and
    construction order, so that its state_dict loads here and `torch.manual_seed(s);
    HumanPolicy()` draws the same initial weights as the reference class does."""

    def __init__(self, frames=3, action_space=2):
        super().__init__()
        self.logstd = nn.Parameter(torch.zeros(action_space))
        self.act_fea_cv1 = nn.Conv1d(frames, 32, kernel_size=5, stride=2, padding=1)
        self.act_fea_cv2 = nn.Conv1d(32, 32, kernel_size=3, stride=2, padding=1)
        self.act_fc1 = nn.Linear(128 * 32, 256)
        self.act_fc2 = nn.Linear(256 + 2 + 2, 128)
        self.actor1 = nn.Linear(128, 1)
        self.actor2 = nn.Linear(128, 1)
        self.crt_fea_cv1 = nn.Conv1d(frames, 32, kernel_size=5, stride=2, padding=1)
        self.crt_fea_cv2 = nn.Conv1d(32, 32, kernel_size=3, stride=2, padding=1)
        self.crt_fc1 = nn.Linear(128 * 32, 256)
        self.crt_fc2 = nn.Linear(256 + 2 + 2, 128)
        self.critic = nn.Linear(128, 1)

    def mean(self, x, goal, speed):
        """The deterministic action mean, the only output env.py:652-656 uses.
        x [N, frames, 512] preprocessed scans, goal [N, 2] local goal, speed [N, 2]."""
        a = F.relu(self.act_fea_cv1(x))
        a = F.relu(self.act_fea_cv2(a))
        a = F.relu(self.act_fc1(a.reshape(a.shape[0], -1)))
        a = F.relu(self.act_fc2(torch.cat((a, goal, speed), dim=-1)))
        return torch.cat((torch.sigmoid(self.actor1(a)), torch.tanh(self.actor2(a))), dim=-1)

    def forward(self, x, goal, speed):
        """(value, sampled action, log-prob, mean) as the reference's forward."""
        mean = self.mean(x, goal, speed)
        logstd = self.logstd.expand_as(mean)
        std = torch.exp(logstd)
        action = torch.normal(mean, std)
        logprob = (-(action - mean).pow(2) / (2 * std.pow(2)) - 0.5 * np.log(2 * np.pi) - logstd).sum(-1, keepdim=True)
        v = F.relu(self.crt_fea_cv1(x))
        v = F.relu(self.crt_fea_cv2(v))
        v = F.relu(self.crt_fc1(v.reshape(v.shape[0], -1)))
        v = self.critic(F.relu(self.crt_fc2(torch.cat((v, goal, speed), dim=-1))))
        return v, action, logprob, mean


def preprocess_scan(scan):
    """env.py:627-629, 648: clip to the pedestrian lidar's 6 m and centre -- in float64, as the
    reference does before its `.float()`."""
    return (torch.clamp(scan.double(), 0.0, Human.range_max) / Human.range_max - 0.5).float()


def footprint_polygons(pose, footprint):
    """Closed world-frame footprints as segments (env.py:404-414): pose [..., 3] float64 ->
    float32 [..., 4, 4] rows (ax, ay, bx, by)."""
    fp = torch.as_tensor(footprint, dtype=torch.float64, device=pose.device)  # [4, 2]
    c, s = torch.cos(pose[..., 2:3]), torch.sin(pose[..., 2:3])
    wx = c * fp[:, 0] - s * fp[:, 1] + pose[..., 0:1]
    wy = s * fp[:, 0] + c * fp[:, 1] + pose[..., 1:2]
    pts = torch.stack((wx, wy), dim=-1).to(torch.float32)                     # [..., 4, 2]
    return torch.cat((pts, torch.roll(pts, -1, dims=-2)), dim=-1)


def human_set_vel(pose, action, dt):
    """Human.set_vel (human.py:32-41) on float64 tensors: pose [..., 3], action [..., 2] =
    (linvel, rotvel) -> (new pose, world velocity (vx, vy) = linvel * (cos, sin)(old theta))."""
    x, y, th = pose[..., 0], pose[..., 1], pose[..., 2]
    v, w = action[..., 0], action[..., 1]
    vel = torch.stack((v * torch.cos(th), v * torch.sin(th)), dim=-1)
    th1 = th + w * dt
    x = x + torch.cos(th1) * v * dt
    y = y + torch.sin(th1) * v * dt
    return torch.stack((x, y, torch.remainder(th1, 2 * np.pi)), dim=-1), vel


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


class NativePolicy(object):
    """HumanPolicy.mean (human_policy.py:38-55) through the library's own kernels
    (navgym_policy_create / navgym_policy_mean): convolutional front end -> act_fc1 -> act_fc2 +
    heads, every contraction on the tcgen05 tensor cores (f16x3 operand split, float32-grade).  No torch op
    and no library GEMM runs in `mean`; torch only owns the workspace memory.  The weights are
    copied (pre-split) at construction: build a new NativePolicy after changing them."""

    def __init__(self, policy, max_n, device):
        self.lib = _lib.load()
        self.device, self.max_n = torch.device(device), int(max_n)
        nbytes = int(self.lib.navgym_policy_workspace_bytes(self.max_n))
        self.workspace = torch.empty(nbytes + 1024, dtype=torch.uint8, device=self.device)
        off = (-self.workspace.data_ptr()) % 1024
        self._ws = self.workspace[off:off + nbytes]
        f = lambda t: t.detach().to(self.device, torch.float32).contiguous()
        self._w = [f(t) for t in (policy.act_fea_cv1.weight, policy.act_fea_cv1.bias, policy.act_fea_cv2.weight,
                                  policy.act_fea_cv2.bias, policy.act_fc1.weight, policy.act_fc1.bias,
                                  policy.act_fc2.weight, policy.act_fc2.bias, policy.actor1.weight, policy.actor1.bias,
                                  policy.actor2.weight, policy.actor2.bias)]
        assert tuple(self._w[0].shape) == (32, 3, 5) and tuple(self._w[4].shape) == (256, 4096)
        p = _lib.PolicyParams()
        p.max_n = self.max_n
        for name, t in zip(('cv1_w', 'cv1_b', 'cv2_w', 'cv2_b', 'fc1_w', 'fc1_b', 'fc2_w', 'fc2_b',
                            'a1_w', 'a1_b', 'a2_w', 'a2_b'), self._w):
            setattr(p, name, _ptr(t))
        p.workspace, p.workspace_bytes = _ptr(self._ws), nbytes
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream(self.device).cuda_stream
            self.handle = self.lib.navgym_policy_create(C.byref(p), C.c_void_p(stream))
        if not self.handle:
            raise RuntimeError('navgym_policy_create failed (needs an sm_100a device and a driver with TMA support)')

    def mean(self, scan, goal, speed, out=None):
        """scan f32 [n, 512] raw metres, goal / speed f32 [n, 2] -> mean f32 [n, 2] (into `out`)."""
        n = int(scan.shape[0])
        for t in (scan, goal, speed):
            assert t.dtype == torch.float32 and t.is_contiguous() and t.is_cuda
        if out is None:
            out = torch.empty(n, 2, dtype=torch.float32, device=self.device)
        assert out.dtype == torch.float32 and out.is_contiguous() and out.numel() == 2 * n
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream(self.device).cuda_stream
            _lib.check(self.lib.navgym_policy_mean(self.handle, _ptr(scan), _ptr(goal), _ptr(speed), n, _ptr(out),
                                                   C.c_void_p(stream)), 'policy_mean')
        return out

    def intermediates(self, n):
        """(features hi, features lo) f16 [n, 4096] put back into torch's channel-major order (the
        kernels keep them position-major, [pos][channel]), act_fc1 output f32 [n, 256] (re-assembled
        from the f16 pairs the tensor-core act_fc2 reads), scales f32 [8] (feature scale, 1 /
        (feature scale x fc1 weight scale), conv1 output scale, 1 / (conv1 output scale x conv2
        weight scale), -, -, act_fc1 output scale, 1 / (that x fc2 weight scale)): copies / views of
        the workspace (tests)."""
        L = (C.c_uint64 * 6)()
        self.lib.navgym_policy_workspace_layout(self.max_n, L)
        w = self._ws
        unperm = lambda t: t.view(torch.float16).reshape(n, 128, 32).permute(0, 2, 1).reshape(n, 4096)
        fh, fl = unperm(w[L[0]:L[0] + n * 8192]), unperm(w[L[1]:L[1] + n * 8192])
        scales = w[L[2]:L[2] + 32].view(torch.float32)
        hh = w[L[4]:L[4] + n * 512].view(torch.float16).reshape(n, 256)
        hl = w[L[5]:L[5] + n * 512].view(torch.float16).reshape(n, 256)
        h = ((hh.double() + hl.double()) / float(scales[6])).float()
        return fh, fl, h, scales

    def __del__(self):
        h, self.handle = getattr(self, 'handle', None), None
        if h:
            self.lib.navgym_policy_destroy(h)


class AgentScanner(object):
    """navgym_agent_scan_batch bound to one MapPool: scans of [num_envs, agents_per_env] agents
    with the pedestrian lidar (human.py:11-16) against the map and the other agents' closed
    footprints."""

    def __init__(self, pool, num_envs, agents_per_env, max_seg, map_id, agent=Human, cell_rule='numpy1'):
        self.lib = _lib.load()
        self.pool, self.device = pool, pool.device
        self.B, self.P, self.K = int(num_envs), int(agents_per_env), int(agent.n_angles)
        self.lin = torch.from_numpy(beam_table(agent)).to(self.device)
        self.ranges = torch.zeros(self.B, self.P, self.K, dtype=torch.float32, device=self.device)
        a = _lib.ScanArgs()
        a.num_envs, a.agents_per_env, a.num_beams, a.max_seg = self.B, self.P, self.K, int(max_seg)
        a.cell_rule = {'numpy1': 0, 'numpy2': 1}[cell_rule]
        a.range_max = float(agent.range_max)
        res = float(pool.maps[0]['resolution'])
        a.t_stop = float(agent.range_max) / res + 2.0  # farther samples are clipped anyway
        a.maps, a.edt_pool = _ptr(pool.maps_dev), _ptr(pool.edt_pool)
        self.map_id = map_id
        a.map_id, a.lin, a.ranges = _ptr(map_id), _ptr(self.lin), _ptr(self.ranges)
        self.args = a

    def scan(self, pose, segs, nseg, skip=None, nagent=None):
        """pose f64 [B, P, 3]; segs f32 [B, max_seg, 4]; nseg i32 [B]; skip i32 [B, P, 2] (each
        agent's own segments) -> ranges f32 [B, P, K] (owned by the scanner, overwritten)."""
        a = self.args
        assert pose.dtype == torch.float64 and pose.is_contiguous() and tuple(pose.shape) == (self.B, self.P, 3)
        assert segs.dtype == torch.float32 and segs.is_contiguous() and segs.shape[1] == a.max_seg
        self._keep = (pose, segs, nseg, skip, nagent)
        a.pose, a.segs, a.nseg, a.skip, a.nagent = _ptr(pose), _ptr(segs), _ptr(nseg), _ptr(skip), _ptr(nagent)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        _lib.check(self.lib.navgym_agent_scan_batch(C.byref(a), C.c_void_p(stream)), 'agent_scan_batch')
        return self.ranges


class PedestrianSim(object):
    """The reference's pedestrians for a whole BatchedNavGym, on the device.

    Per step, in the reference's order (env.py:617-693):
        sim.act()            respawn for episodes that just ended -> route following
                             (navgym_peds_plan) -> policy (NativePolicy) -> clip, Human.set_vel, leg
                             odometry (navgym_peds_move) -> the geometry the robot's lidar sees
                             (navgym_peds_advance: discs for legs, boxes otherwise)
        env.step(actions)    the robot's fused step, scanning against that geometry
        sim.observe()        every pedestrian's own scan from its new pose, robot included
                             (navgym_agent_scan_batch, crowd mode): the next policy input
    `sim.step(actions)` does the three.

    State, all [num_envs, max_ped, ...] device tensors: pose f64 (x, y, theta), vel f64 (vx, vy),
    v_pref f64, has_legs bool, dist_travelled f64 (x, y, theta in the base frame), prev_action f32
    (the clipped policy mean, the policy's `speed` input), scan f32 [.., 512], goal_id i32,
    waypoint f64, goal_local f32.

    The policy forward runs through the library's own kernels (NativePolicy: both convolutions,
    act_fc1 and act_fc2 on the tcgen05 tensor cores with hi/lo f16 operand splits, float32-grade:
    the mean matches the reference's CPU forward to ~1e-5).

    Auto-reset: every act() also draws the pedestrians of each environment's NEXT episode (at
    least 4 m from where the robot's auto-reset will put it -- the same Philox draw the step
    kernel makes) and hands their geometry to the robot's step as discs_reset / segs_reset, so the
    first observation of a new episode already sees the new pedestrians; the next act() adopts
    them for the environments whose episode ended.  Over an auto_reset=False env, step and read
    the final observations, then sim.reset_envs(env.done) does the same for those environments.

    Pedestrian counts: `nped` (int32 [num_envs], None = max_ped) fixes each environment's count
    for the sim's whole life.  `num_humans_range=(lo, hi)` instead draws every episode's count
    uniformly from lo..hi (inclusive), as NavGym-v0 draws num_humans: at reset(), with each
    auto-reset and with each reset_envs().  sim.nped (= env.nped) then always holds the current
    episodes' counts, and sim.cand_nped those of the next episodes, whose pedestrians the
    candidates are (None without a range).  Slots at or beyond an environment's count are not
    simulated, scanned or emitted.
    """

    def __init__(self, env, max_ped, nped=None, policy=None, v_pref_range=(0.0, 0.6), has_legs_ratio=0.5,
                 num_goals=32, min_goal_dist=10.0, min_robot_dist=4.0, seed=0, num_humans_range=None):
        from . import maps as M
        if env.args.auto_reset == _lib.AUTORESET_NEXT_STEP:
            # act() respawns the pedestrians of an env in the launch that ends its episode
            raise ValueError("PedestrianSim does not drive an auto_reset='next_step' env")
        self.env, self.device = env, env.device
        self.B, self.P = env.B, int(max_ped)
        if self.P > 127:  # navgym_agent_scan_batch, crowd mode: one thread per other agent
            raise ValueError('at most 127 pedestrians per environment')
        if num_humans_range is not None:
            if nped is not None:
                raise ValueError('give nped or num_humans_range, not both')
            lo, hi = (operator.index(v) for v in num_humans_range)
            if not 0 <= lo <= hi <= self.P:
                raise ValueError('num_humans_range=(%d, %d): need 0 <= lo <= hi <= max_ped = %d' % (lo, hi, self.P))
        self.dt = float(env.args.dt)
        self.lib = _lib.load()
        dev, f64, f32, i32 = self.device, torch.float64, torch.float32, torch.int32
        B, P = self.B, self.P
        self.nped = None if nped is None else torch.as_tensor(nped, dtype=i32).to(dev)
        self.cand_nped = self._counts = self._counts_out = None
        if num_humans_range is not None:
            # [nped; cand_nped], which navgym_peds_plan reads, and the two it writes in their
            # place: _plan copies the second pair over the first after each launch
            self._counts = torch.zeros(2, B, dtype=i32, device=dev)
            self._counts_out = torch.zeros(2, B, dtype=i32, device=dev)
            self.nped, self.cand_nped = self._counts[0], self._counts[1]
        if policy is None:
            policy = HumanPolicy()
        self.policy = policy.to(dev).eval()
        self.native = NativePolicy(self.policy, self.B * self.P, dev)
        # ---- planning fields + free-cell pools per map (kept on the MapPool: a pool that is
        # reused for another episode / another sim does not rebuild them)
        cache = getattr(env.pool, '_plan_cache', None)
        if cache is None:
            cache = env.pool._plan_cache = {}
        if int(num_goals) not in cache:
            rng = np.random.RandomState(int(seed) + 77)
            pm = (_lib.PlanMapT * len(env.pool.maps))()
            fl, gl, xl = [], [], []
            foff = goff = xoff = 0
            for i, m in enumerate(env.pool.maps):
                fields, goals, cm = M.goal_fields(m, num_goals, rng)
                # spawn cells (env.py:786-797): free cost-map cells connected to the goals'
                # component, so that a spawned pedestrian always has a route (ADVICE r1: a
                # pedestrian in a disconnected pocket walked at its goal through walls)
                r, c = np.where((cm['data'] == 0) & (fields[0] != 65535))
                xy = np.column_stack([(c + 0.5) * cm['resolution'] + cm['origin'][0],
                                      (r + 0.5) * cm['resolution'] + cm['origin'][1]]).astype(np.float64)
                pm[i] = _lib.PlanMapT(cm['width'], cm['height'], num_goals, 0, foff, goff, xoff, len(xy),
                                      float(cm['origin'][0]), float(cm['origin'][1]), float(cm['resolution']))
                fl.append(fields.reshape(-1))
                gl.append(goals)
                xl.append(xy.reshape(-1, 2))
                foff += fields.size
                goff += num_goals
                xoff += len(xy)
            xy_all = np.concatenate(xl) if sum(len(x) for x in xl) else np.zeros((1, 2))
            cache[int(num_goals)] = (
                torch.from_numpy(np.frombuffer(bytes(pm), dtype=np.uint8).copy()).to(dev),
                torch.from_numpy(np.concatenate(fl).view(np.int16)).to(dev),
                torch.from_numpy(np.concatenate(gl)).to(dev),
                torch.from_numpy(xy_all).to(dev))
        self.plan_maps, self.fields, self.goals, self.free_xy = cache[int(num_goals)]
        self.num_goals = int(num_goals)
        # ---- state
        self.pose = torch.zeros(B, P, 3, dtype=f64, device=dev)
        self.vel = torch.zeros(B, P, 2, dtype=f64, device=dev)
        self.v_pref = torch.zeros(B, P, dtype=f64, device=dev)
        self.has_legs = torch.zeros(B, P, dtype=torch.bool, device=dev)
        self.dist_travelled = torch.zeros(B, P, 3, dtype=f64, device=dev)
        self.prev_action = torch.zeros(B, P, 2, dtype=f32, device=dev)
        self.goal_id = torch.zeros(B, P, dtype=i32, device=dev)
        self.waypoint = torch.full((B, P, 2), float('nan'), dtype=f64, device=dev)
        self.goal_local = torch.zeros(B, P, 2, dtype=f32, device=dev)
        self._all = torch.ones(B, dtype=torch.uint8, device=dev)
        # ---- geometry for the robot's lidar goes through the env's pedestrian rows
        env.attach_pedestrians(torch.zeros(B, P, _lib.PED_F, dtype=f32, device=dev), self.nped)
        env.peds_scripted = False  # the sim moves them; env.step only emits their geometry
        env.crowd = self           # export_env reads the float64 state from here
        a = _lib.PlanArgs()
        a.num_envs, a.max_ped, a.step, a.seed = B, P, 0, int(seed)
        a.env_offset, a.min_goal_dist = int(env.args.env_offset), float(min_goal_dist)
        a.maps, a.fields, a.goals = _ptr(self.plan_maps), _ptr(self.fields), _ptr(self.goals)
        a.map_id, a.nped, a.pose = _ptr(env.map_id), _ptr(self.nped), _ptr(self.pose)
        a.goal_id, a.waypoint, a.goal_local = _ptr(self.goal_id), _ptr(self.waypoint), _ptr(self.goal_local)
        a.free_xy, a.robot_state = _ptr(self.free_xy), _ptr(env.state)
        a.min_robot_dist, a.has_legs_ratio = float(min_robot_dist), float(has_legs_ratio)
        a.v_pref_lo, a.v_pref_hi = float(v_pref_range[0]), float(v_pref_range[1])
        a.pose_rw, a.v_pref, a.has_legs = _ptr(self.pose), _ptr(self.v_pref), _ptr(self.has_legs)
        a.dist_travelled, a.vel, a.prev_action = _ptr(self.dist_travelled), _ptr(self.vel), _ptr(self.prev_action)
        # ---- the next episode's pedestrians (candidates) and their geometry
        self.cand_pose = torch.zeros(B, P, 3, dtype=f64, device=dev)
        self.cand_v_pref = torch.zeros(B, P, dtype=f64, device=dev)
        self.cand_legs = torch.zeros(B, P, dtype=torch.bool, device=dev)
        self.cand_goal = torch.zeros(B, P, dtype=i32, device=dev)
        self.cand_rows = torch.zeros(B, P, _lib.PED_F, dtype=f32, device=dev)
        a.cand_pose, a.cand_v_pref, a.cand_legs = _ptr(self.cand_pose), _ptr(self.cand_v_pref), _ptr(self.cand_legs)
        a.cand_goal, a.cand_rows = _ptr(self.cand_goal), _ptr(self.cand_rows)
        if num_humans_range is not None:
            a.num_humans_lo, a.num_humans_hi = lo, hi
            a.cand_nped_prev, a.cand_nped = _ptr(self.cand_nped), _ptr(self._counts_out[1])
            a.nped_out = _ptr(self._counts_out[0])
        ea = env.args
        a.robot_maps, a.spawn_pool, a.episodes = ea.maps, ea.spawn_pool, ea.episodes
        a.robot_seed, a.num_maps, a.resample_map = ea.seed, ea.num_maps, ea.resample_map
        self.cand_discs = torch.zeros_like(env._pdiscs)
        self.cand_segs = torch.zeros_like(env._psegs)
        self.cand_nd = torch.zeros_like(env._pnd)
        self.cand_ns = torch.zeros_like(env._pns)
        cp = _lib.PedsArgs()
        for f, _t in _lib.PedsArgs._fields_:
            setattr(cp, f, getattr(env._pargs, f))
        cp.advance = 0
        cp.peds, cp.discs, cp.ndisc = _ptr(self.cand_rows), _ptr(self.cand_discs), _ptr(self.cand_nd)
        cp.segs, cp.nseg = _ptr(self.cand_segs), _ptr(self.cand_ns)
        if self.cand_nped is not None:
            cp.nped = _ptr(self.cand_nped)  # the reset scan sees the next episode's count
        self.cand_pargs = cp
        # (the step reads them only on auto-reset; navgym_reset_envs reads them in sim.reset_envs)
        ea.discs_reset, ea.ndisc_reset = _ptr(self.cand_discs), _ptr(self.cand_nd)
        ea.segs_reset, ea.nseg_reset = _ptr(self.cand_segs), _ptr(self.cand_ns)
        self._pending = None  # u8 [B]: environments sim.reset_envs restarted, respawned at the next act()
        self.plan_args = a
        self._mean = torch.zeros(B, P, 2, dtype=f32, device=dev)
        mv = _lib.MoveArgs()
        mv.num_envs, mv.max_ped, mv.dt = B, P, self.dt
        mv.nped, mv.mean, mv.v_pref, mv.has_legs = _ptr(self.nped), _ptr(self._mean), _ptr(self.v_pref), _ptr(self.has_legs)
        mv.pose, mv.vel, mv.dist_travelled = _ptr(self.pose), _ptr(self.vel), _ptr(self.dist_travelled)
        mv.prev_action, mv.rows = _ptr(self.prev_action), _ptr(env.peds)
        self.move_args = mv
        # ---- lidar of the pedestrians, crowd mode: footprints built in the kernel
        self.scanner = AgentScanner(env.pool, B, P, 0, env.map_id,
                                    cell_rule='numpy2' if env.args.cell_rule else 'numpy1')
        sa = self.scanner.args
        sa.pose, sa.nagent, sa.robot_state = _ptr(self.pose), _ptr(self.nped), _ptr(env.state)
        sa.robot_fp = (C.c_double * 8)(*np.asarray(KetiRobot.threshold_footprint, np.float64).reshape(-1))
        sa.agent_fp = (C.c_double * 8)(*np.asarray(Human.footprint, np.float64).reshape(-1))
        self.scan = self.scanner.ranges
        self.reset()

    def _call(self, fn, args, what):
        with torch.cuda.device(self.device):
            _lib.check(fn(C.byref(args), self.env._stream()), what)

    def _plan(self, respawn, next_spawn=True):
        a = self.plan_args
        self._respawn = respawn  # keep the tensor alive while the launch reads it
        a.respawn = _ptr(respawn)
        a.cand_next_spawn = int(bool(next_spawn))
        self._call(self.lib.navgym_peds_plan, a, 'peds_plan')
        if self._counts is not None:
            with torch.cuda.device(self.device):
                self._counts.copy_(self._counts_out)  # same stream, before anything reads the counts
        a.step += 1
        self._call(self.lib.navgym_peds_advance, self.cand_pargs, 'peds_advance')  # candidates' geometry

    def _scan(self, env_mask=None):
        self._mask = env_mask
        self.scanner.args.env_mask = _ptr(env_mask)
        self._call(self.lib.navgym_agent_scan_batch, self.scanner.args, 'agent_scan_batch')

    # ---- episode start (env.py:785-815) ------------------------------------------------
    def reset(self):
        """Spawn every environment's pedestrians (env.py:785-806) around the robots' current poses
        and take their first scans."""
        self._pending = None
        self._plan(None, next_spawn=False)  # draw them ...
        self._plan(self._all)               # ... adopt them, and draw the next episode's
        rows = self.env.peds
        rows[..., 0:3] = self.pose.float()
        rows[..., 9:12] = 0.0
        rows[..., 12] = self.has_legs.float()
        self.env._peds_emit(advance=False)
        self.observe()

    # ---- env.py:617-662 + 664-681 + 237-255 ---------------------------------------------
    @torch.no_grad()
    def act(self):
        env = self.env
        respawn = env.done if env.args.auto_reset else None
        if self._pending is not None:
            respawn = self._pending if respawn is None else respawn | self._pending
            self._pending = None
        self._plan(respawn)
        if respawn is not None:
            self._scan(respawn)  # first scans of the respawned pedestrians (env.py:808-815)
        goal, speed = self.goal_local.reshape(-1, 2), self.prev_action.reshape(-1, 2)
        # three launches of the library, straight into the move kernel's input
        self.native.mean(self.scan.reshape(self.B * self.P, -1), goal, speed, out=self._mean)
        self._call(self.lib.navgym_peds_move, self.move_args, 'peds_move')
        env._peds_emit(advance=False)

    # ---- masked reset (BatchedNavGym.reset_envs for an env this sim drives) ------------------
    @torch.no_grad()
    def reset_envs(self, envs):
        """New episodes for the environments `envs` (a bool / uint8 [B] device tensor such as
        env.done, or env ids), exactly as auto-reset starts them: the robot's new episode
        (navgym_reset_envs) with its first scan against the next episode's pedestrians, those
        pedestrians adopted at the next act(), and the current pedestrians' scans of these
        environments retaken with the robot at its new pose.  After `sim.step(actions)` on an
        auto_reset=False env, `sim.reset_envs(env.done)` leaves the robot's and the pedestrians'
        state as an auto_reset=True run would have, bit for bit.  Returns env.obs."""
        env = self.env
        mask = env.env_mask(envs)
        env._reset_envs(mask)
        self._pending = mask.clone() if self._pending is None else self._pending | mask
        self._scan(mask)
        return env.obs

    # ---- env.py:683-693 -------------------------------------------------------------------
    def observe(self):
        """Every pedestrian's scan from its current pose: the map, the robot's threshold
        footprint and the other pedestrians' footprints (lidar_legs=False), no noise."""
        self._scan(None)
        return self.scan

    def step(self, actions):
        self.act()
        out = self.env.step(actions)
        self.observe()
        return out
