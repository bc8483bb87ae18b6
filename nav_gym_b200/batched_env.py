"""BatchedNavGym — thousands of NavGym-v0 environments stepped in lockstep on one B200.

Host-side mirror of the reference's NavGymEnv.step contract (env.py:591-728) for a batch:
``step(actions[B,2]) -> obs[B,519], reward[B], done[B], info`` with every tensor resident on
the device.  All arithmetic happens in the hand-written sm_100a kernels of
csrc/ (navgym_b200.cu and the kernels it includes), reached through the C ABI of include/navgym_b200.h via ctypes; torch is
used only for device memory and streams.  There is no CPU fallback.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import NB, NS, OBS_DIM
from .robot import KetiRobot, beam_table, closed_segments

DEFAULT_REWARD = dict(reward_scale=15., reward_success_factor=1, reward_crash_factor=1,
                      reward_progress_factor=0.001, reward_forward_factor=0.0,
                      reward_rotation_factor=0.005, reward_discomfort_factor=0.01)


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


_THRESHOLDS = {}


def scan_thresholds(device):
    """_make_scan_threshold / _make_scan_discomfort_threshold (env.py:162-180): the inflated
    footprints rendered into a 25 m scan from the origin at heading 0, on the GPU."""
    lib = _lib.require_device()
    key = str(torch.device(device))
    if key in _THRESHOLDS:  # constants of the robot model: rendered once per device
        return [t.copy() for t in _THRESHOLDS[key]]
    head = beam_table().astype(np.float32)  # float32(lin + float32(0))
    out = []
    for fp in (KetiRobot.threshold_footprint, KetiRobot.discomfort_threshold_footprint):
        ranges = np.full(NB, KetiRobot.range_max, np.float32)
        segs = np.ascontiguousarray(closed_segments(fp))
        with torch.cuda.device(torch.device(device)):
            _lib.check(lib.navgym_render_in_lidar_host(
                ranges.ctypes.data_as(C.c_void_p), head.ctypes.data_as(C.c_void_p), NB,
                segs.ctypes.data_as(C.c_void_p), len(segs), None, 0, 0.0, 0.0), 'render_in_lidar_host')
        out.append(np.clip(ranges, 0, KetiRobot.range_max))
    _THRESHOLDS[key] = [t.copy() for t in out]
    return out


class MapPool(object):
    """Occupancy maps resident in HBM as exact float32 Euclidean distance transforms, [H][W]
    row-major per map (what range_libc's PyRayMarching holds per map, env.py:337-340), plus
    optional per-map spawn pools of (start, goal, theta) tuples for device-side auto-reset."""

    def __init__(self, maps, device, spawn_pools=None):
        lib = _lib.require_device()
        self.device = torch.device(device)
        self.maps = maps
        n = len(maps)
        self.spawn_arrays = [None] * n if spawn_pools is None else [
            None if p is None else np.asarray(p, np.float64).reshape(-1, 5) for p in spawn_pools]
        self.num_maps = n
        self.offsets = []
        off = 0
        for m in maps:
            if not (0 < int(m['width']) <= 12000 and 0 < int(m['height']) <= 32767):
                raise ValueError('map of %d x %d cells: at most 12000 wide and 32767 high' % (int(m['width']), int(m['height'])))
            self.offsets.append(off)
            off += int(m['height']) * int(m['width'])
        self.edt_pool = torch.empty(off, dtype=torch.float32, device=self.device)
        carr = (_lib.MapT * n)()
        soff = 0
        spawn_rows = []
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            for i, m in enumerate(maps):
                H, W = int(m['height']), int(m['width'])
                occ = torch.from_numpy(np.ascontiguousarray(np.asarray(m['data']) >= 0.1).astype(np.uint8))
                occ = occ.to(self.device)
                scratch = torch.empty(H * W, dtype=torch.int32, device=self.device)
                dist = self.edt_pool[self.offsets[i]:self.offsets[i] + H * W]
                _lib.check(lib.navgym_edt_build(_ptr(occ), H, W, _ptr(dist), _ptr(scratch),
                                                C.c_void_p(stream)), 'edt_build')
                cnt = 0
                if self.spawn_arrays[i] is not None and len(self.spawn_arrays[i]):
                    spawn_rows.append(self.spawn_arrays[i])
                    cnt = len(self.spawn_arrays[i])
                carr[i] = _lib.MapT(W, H, self.offsets[i], float(m['origin'][0]), float(m['origin'][1]),
                                    float(m['resolution']), soff, cnt, 0)
                soff += cnt
            torch.cuda.synchronize(self.device)
        raw = np.frombuffer(bytes(carr), dtype=np.uint8).copy()
        self.maps_dev = torch.from_numpy(raw).to(self.device)
        self.spawn_pool = None
        if spawn_rows:
            self.spawn_pool = torch.from_numpy(np.concatenate(spawn_rows)).to(self.device)

    def edt(self, i):
        m = self.maps[i]
        H, W = int(m['height']), int(m['width'])
        return self.edt_pool[self.offsets[i]:self.offsets[i] + H * W].view(H, W)


def filter_spawn_pool(map_info, pool, device='cuda:0', chunk=16384, map_pool=None):
    """Drop spawn tuples whose noise-free first scan already violates the discomfort threshold
    (the reference re-samples such spawns, env.py:779-783)."""
    pool = np.asarray(pool, np.float64).reshape(-1, 5)
    if not len(pool):
        return pool
    mp = map_pool if map_pool is not None else MapPool([map_info], device)
    keep = []
    for s in range(0, len(pool), chunk):
        p = pool[s:s + chunk]
        env = BatchedNavGym(len(p), mp, device=device)
        env.set_state(p[:, 0:2], p[:, 2:4], p[:, 4])
        obs = env.reset()
        ok = ~(obs[:, :NB] < env.dthr[None, :]).any(dim=1)
        keep.append(ok.cpu().numpy())
    return pool[np.concatenate(keep)]


class BatchedNavGym(object):
    def __init__(self, num_envs, maps, device='cuda:0', map_id=None, spawn_pools=None,
                 time_step=0.2, distance_threshold=0.5, min_turning_radius=0.0,
                 max_disc=0, max_seg=0, seed=0, env_offset=0, auto_reset=False,
                 max_episode_steps=0, resample_map=False, scan_noise_std_range=(0.0, 0.05),
                 cell_rule='numpy1', early_stop=True, record_hits=False, longest_first=True,
                 num_scan_stack=1, obs_dtype=torch.float32, **reward):
        # auto_reset: False (off), True (same-step: the ending launch writes the next episode's first
        # observation over the final one) or 'next_step' (the next launch starts the new episode)
        if isinstance(auto_reset, str):
            if auto_reset != 'next_step':
                raise ValueError("auto_reset must be True, False or 'next_step', not %r" % (auto_reset,))
            auto_reset = _lib.AUTORESET_NEXT_STEP
        else:
            auto_reset = 1 if auto_reset else 0
        self.next_step_reset = auto_reset == _lib.AUTORESET_NEXT_STEP
        self.lib = _lib.require_device()
        self.device = torch.device(device)
        self.B = B = int(num_envs)
        self.pool = maps if isinstance(maps, MapPool) else MapPool(maps, self.device, spawn_pools)
        dev = self.device
        rp = dict(DEFAULT_REWARD)
        rp.update(reward)
        if max_disc > _lib.MAX_DISC or max_seg > _lib.MAX_SEG:
            raise ValueError('max_disc <= %d and max_seg <= %d' % (_lib.MAX_DISC, _lib.MAX_SEG))
        self.max_disc, self.max_seg = int(max_disc), int(max_seg)
        f32, f64, i32, u8 = torch.float32, torch.float64, torch.int32, torch.uint8
        self.state = torch.zeros(NS, B, dtype=f64, device=dev)
        self.steps = torch.zeros(B, dtype=i32, device=dev)
        self.episodes = torch.zeros(B, dtype=i32, device=dev)
        mid = np.zeros(B, np.int32) if map_id is None else np.asarray(map_id, np.int32)
        self.map_id = torch.from_numpy(mid).to(dev)
        self.noise_std = torch.zeros(B, dtype=f32, device=dev)
        self.num_scan_stack = S = max(int(num_scan_stack), 1)
        # Observation rows: float32 [scans | 7 tail fields], or with obs_dtype=torch.float16 the
        # S*512 scans in float16 followed by the tail as float32 in 14 halves and 2 halves of padding
        # (1056-byte rows for S = 1; obs_parts() splits either format)
        if obs_dtype == torch.float32:
            obs_format, self.obs_dim = _lib.OBS_F32, S * NB + 7
        elif obs_dtype == torch.float16:
            obs_format, self.obs_dim = _lib.OBS_F16, S * NB + 16
        else:
            raise ValueError('obs_dtype must be torch.float32 or torch.float16, not %r' % (obs_dtype,))
        self.obs_dtype = obs_dtype
        self.obs = torch.zeros(B, self.obs_dim, dtype=obs_dtype, device=dev)
        self.tail64 = torch.zeros(B, 7, dtype=f64, device=dev)
        self.reward = torch.zeros(B, dtype=f32, device=dev)
        self.done = torch.zeros(B, dtype=u8, device=dev)
        self.is_success = torch.zeros(B, dtype=u8, device=dev)
        self.is_crash = torch.zeros(B, dtype=u8, device=dev)
        self.truncated = torch.zeros(B, dtype=u8, device=dev)
        self.distance = torch.zeros(B, dtype=f32, device=dev)
        self.hits = torch.zeros(B, NB, 2, dtype=torch.int16, device=dev) if record_hits else None
        self.lin = torch.from_numpy(beam_table()).to(dev)
        thr, dthr = scan_thresholds(dev)
        self.scan_threshold, self.scan_discomfort_threshold = thr, dthr
        self.thr = torch.from_numpy(thr).to(dev)
        self.dthr = torch.from_numpy(dthr).to(dev)
        self.early_stop = bool(early_stop)
        t_stop = KetiRobot.range_max / 0.05 + 2.0 if early_stop else 3.0e38
        if early_stop:
            res = min(float(m['resolution']) for m in self.pool.maps)
            t_stop = KetiRobot.range_max / res + 2.0
        a = _lib.StepArgs()
        a.dt, a.dist_thresh, a.min_turn_radius = time_step, distance_threshold, min_turning_radius
        a.r_scale = rp['reward_scale']
        a.r_success, a.r_crash = rp['reward_success_factor'], rp['reward_crash_factor']
        a.r_progress, a.r_forward = rp['reward_progress_factor'], rp['reward_forward_factor']
        a.r_rotation, a.r_discomfort = rp['reward_rotation_factor'], rp['reward_discomfort_factor']
        a.range_max, a.t_stop = KetiRobot.range_max, t_stop
        a.cell_rule = {'numpy1': 0, 'numpy2': 1}[cell_rule]
        a.max_disc, a.max_seg = self.max_disc, self.max_seg
        a.num_envs, a.obs_stride, a.num_scan_stack = B, self.obs_dim, S
        a.obs_format = obs_format
        a.auto_reset, a.max_episode_steps = auto_reset, int(max_episode_steps)
        a.num_maps, a.resample_map = self.pool.num_maps, int(resample_map)
        a.seed, a.env_offset = int(seed), int(env_offset)
        a.noise_lo, a.noise_hi = scan_noise_std_range
        a.maps, a.edt_pool = _ptr(self.pool.maps_dev), _ptr(self.pool.edt_pool)
        a.spawn_pool = _ptr(self.pool.spawn_pool)
        a.map_id, a.lin, a.thr, a.dthr = _ptr(self.map_id), _ptr(self.lin), _ptr(self.thr), _ptr(self.dthr)
        a.state, a.steps, a.episodes = _ptr(self.state), _ptr(self.steps), _ptr(self.episodes)
        a.noise_std = _ptr(self.noise_std)
        a.obs, a.tail64, a.reward = _ptr(self.obs), _ptr(self.tail64), _ptr(self.reward)
        a.done, a.is_success, a.is_crash = _ptr(self.done), _ptr(self.is_success), _ptr(self.is_crash)
        a.truncated, a.distance, a.hits = _ptr(self.truncated), _ptr(self.distance), _ptr(self.hits)
        self.sched = None
        if longest_first:
            self.sched = self._make_sched(np.arange(B, dtype=np.int32))
            a.sched, a.sched_phase = _ptr(self.sched), 0
        self.args = a
        self._keep = None
        self._act_dev = None
        self._pipe = None
        self.peds = None

    # -------------------------------------------------------------------------------------
    def set_state(self, start, goal, theta, noise_std=None):
        """start/goal [B,2], theta [B] (numpy or tensors); prev fields are set by reset()."""
        t = lambda x: torch.as_tensor(np.asarray(x) if not torch.is_tensor(x) else x,
                                      dtype=torch.float64, device=self.device)
        s, g = t(start), t(goal)
        self.state[_lib.S_PX], self.state[_lib.S_PY] = s[:, 0], s[:, 1]
        self.state[_lib.S_TH] = t(theta)
        self.state[_lib.S_GX], self.state[_lib.S_GY] = g[:, 0], g[:, 1]
        if noise_std is not None:
            self.noise_std.copy_(torch.as_tensor(noise_std, dtype=torch.float32, device=self.device))

    def _geom(self, discs, ndisc, segs, nseg, noise, actions=None):
        a = self.args
        keep = []

        def dev(x, dtype):
            if x is None:
                return None
            if not torch.is_tensor(x):
                x = torch.from_numpy(np.ascontiguousarray(x))
            x = x.to(device=self.device, dtype=dtype).contiguous()
            keep.append(x)
            return x
        d, nd = dev(discs, torch.float32), dev(ndisc, torch.int32)
        s, ns = dev(segs, torch.float32), dev(nseg, torch.int32)
        nz = dev(noise, torch.float32)
        if d is not None:
            assert d.numel() == self.B * self.max_disc * 3 and nd.numel() == self.B
        if s is not None:
            assert s.numel() == self.B * self.max_seg * 4 and ns.numel() == self.B
        if nz is not None:
            assert nz.numel() == self.B * 2 * NB
        a.discs, a.ndisc, a.segs, a.nseg, a.noise = _ptr(d), _ptr(nd), _ptr(s), _ptr(ns), _ptr(nz)
        if actions is not None:
            act = dev(actions, torch.float32)
            assert act.numel() == self.B * 2
            a.actions = _ptr(act)
        self._keep = keep

    def reset_from_spawn_pool(self, rng=None, noise_std_range=None):
        """Draw every env's (start, goal, theta) from its map's spawn pool (host RNG), set the
        per-episode scan noise std (reference env_param 'scan_noise_std', __init__.py:36) and
        compute the first observations."""
        rng = np.random if rng is None else rng
        pools = self.pool.spawn_arrays
        mid = self.map_id.cpu().numpy()
        rows = np.zeros((self.B, 5))
        for i in np.unique(mid):
            sel = np.where(mid == i)[0]
            if pools[i] is None or not len(pools[i]):
                raise ValueError('map %d has no spawn pool' % i)
            rows[sel] = pools[i][rng.randint(len(pools[i]), size=len(sel))]
        lo, hi = (self.args.noise_lo, self.args.noise_hi) if noise_std_range is None else noise_std_range
        self.set_state(rows[:, 0:2], rows[:, 2:4], rows[:, 4],
                       noise_std=rng.uniform(lo, hi, self.B).astype(np.float32))
        return self.reset()

    def _make_sched(self, envs):
        """longest-first schedule buffer (include/navgym_b200.h) for the given env ids"""
        nbk = _lib.SCHED_BUCKETS
        sched = np.zeros(3 * nbk + 3 * nbk * self.B, np.int32)
        sched[0] = len(envs)
        sched[3 * nbk:3 * nbk + len(envs)] = envs
        return torch.from_numpy(sched).to(self.device)

    def step_host(self, actions_host, obs_host, reward_host, done_host, chunks=2):
        """The same step for callers that live on the host (the reference's calling
        convention): pinned host actions in, pinned host obs (rows of the env's obs_dtype and
        width, like env.obs) / reward / done out, through the
        C ABI's navgym_step_batch_host: `chunks` launches over consecutive env ranges on
        prioritised streams, each followed by the D2H copy of its rows, so the copies of early
        chunks overlap the raycast of later ones (PCIe is the end-to-end bound: 2.1 KB per
        env-step).  Returns when all results have landed."""
        self._check_host_tensors('step_host', actions_host, obs_host, reward_host, done_host)
        self._geom(*self._obstacles(None, None, None, None, advance=True), None)
        self._make_pipe(1 if self.peds is not None else chunks)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.navgym_step_batch_host(
                self._pipe[0], C.byref(self.args), self._stream(), _ptr(actions_host), _ptr(obs_host),
                _ptr(reward_host), _ptr(done_host)), 'step_host')
        return obs_host, reward_host, done_host

    # ---- asynchronous host API: several env groups in flight (EnvPool style) ----------------
    def host_groups(self, groups, actions_host, obs_host, reward_host, done_host):
        """Split the batch into `groups` consecutive env ranges for submit_host / wait_host,
        bind the pinned [B, ...] host tensors they read / write, and return the ranges'
        (begin, end) bounds."""
        if self.peds is not None:
            raise NotImplementedError('async host groups with device pedestrians')
        self._check_host_tensors('host_groups', actions_host, obs_host, reward_host, done_host)
        self._make_pipe(groups, fresh=True)
        self._geom(None, None, None, None, None)
        self._host_bufs = (actions_host, obs_host, reward_host, done_host)
        self._host_ptrs = tuple(_ptr(t) for t in self._host_bufs)
        self._args_ref = C.byref(self.args)
        torch.cuda.synchronize(self.device)
        bounds = []
        for g in range(self.lib.navgym_host_pipe_groups(self._pipe[0])):
            b0, b1 = C.c_int(), C.c_int()
            _lib.check(self.lib.navgym_host_pipe_group_bounds(self._pipe[0], g, C.byref(b0), C.byref(b1)), 'group_bounds')
            bounds.append((b0.value, b1.value))
        return bounds

    def _check_host_tensors(self, what, actions_host, obs_host, reward_host, done_host):
        """The host-buffer calls' [B, ...] host tensors: ValueError unless pinned and contiguous,
        AssertionError for a dtype or shape other than the env's."""
        for t in (actions_host, obs_host, reward_host, done_host):
            if not t.is_pinned() or not t.is_contiguous():
                raise ValueError('%s needs contiguous pinned host tensors' % what)
        assert obs_host.dtype == self.obs_dtype and tuple(obs_host.shape) == (self.B, self.obs_dim)
        assert actions_host.dtype == torch.float32 and actions_host.numel() == 2 * self.B
        assert reward_host.dtype == torch.float32 and done_host.dtype == torch.uint8

    def _make_pipe(self, groups, fresh=False):
        """(Re)create the host pipe -- its streams, events and schedule buffers live on the env's
        device (the C side switches to it on every call; here the device is made current so that
        the creation itself lands there)."""
        if self._pipe is None or self._pipe[1] != groups or fresh:
            with torch.cuda.device(self.device):
                if self._pipe is not None:
                    self.lib.navgym_host_pipe_destroy(self._pipe[0])
                    self._pipe = None
                h = self.lib.navgym_host_pipe_create(groups, self.B, int(self.sched is not None))
            if not h:
                raise RuntimeError('navgym_host_pipe_create failed')
            self._pipe = (C.c_void_p(h), groups)
            self._act_dev = torch.empty(self.B, 2, dtype=torch.float32, device=self.device)
        self.args.actions = _ptr(self._act_dev)

    def submit_host(self, group):
        """Enqueue one step of env group `group` (its rows of the bound host tensors are read /
        written); returns immediately."""
        p = self._host_ptrs
        err = self.lib.navgym_step_batch_host_submit(self._pipe[0], self._args_ref, group, p[0], p[1], p[2], p[3])
        if err:
            _lib.check(err, 'step_host_submit')

    def wait_host(self, group):
        """Block until the results of the last submit_host(group) are on the host."""
        err = self.lib.navgym_step_batch_host_wait(self._pipe[0], group)
        if err:
            _lib.check(err, 'step_host_wait')

    def rollout_host(self, steps, policy, user=None):
        """`steps` lockstep steps of every env group bound by host_groups(), the group rotation
        done in C (navgym_host_rollout): per group and step the results land in the bound host
        tensors, `policy` writes the group's next actions into the bound actions tensor, and the
        group is resubmitted while the others are stepping / copying.

        policy: a C function pointer of type _lib.POLICY_FN (e.g. the library's
        navgym_policy_action_bank with `user` = a _lib.ActionBank), or a Python callable
        policy(group, env_begin, env_end, step) that reads / writes the bound tensors' rows
        [env_begin:env_end] (called with the GIL held: convenient, not fast)."""
        if callable(policy) and not isinstance(policy, (C._CFuncPtr,)):
            fn = policy
            policy = _lib.POLICY_FN(lambda u, g, b0, b1, s, o, r, d, a: fn(g, b0, b1, s))
        self._policy_keep = (policy, user)
        p = self._host_ptrs
        uptr = None if user is None else C.cast(C.pointer(user), C.c_void_p)
        err = self.lib.navgym_host_rollout(self._pipe[0], self._args_ref, int(steps),
                                           C.cast(policy, C.c_void_p), uptr, p[0], p[1], p[2], p[3])
        if err:
            _lib.check(err, 'host_rollout')

    def __del__(self):
        p, self._pipe = getattr(self, '_pipe', None), None
        if p is not None:
            self.lib.navgym_host_pipe_destroy(p[0])

    # ---- host export of one environment (SURVEY 8f row 4) --------------------------------
    def export_env(self, i):
        """Copy environment `i` back to the attribute surface ros_env.py and render read from a
        NavGymEnv (ros_env.py:69-176): map_info, robot.{px,py,theta,gx,gy,...}, humans[...],
        prev_obs (the dict form of its last observation row), num_scan_stack, steps_since_reset,
        plus the step's reward / done / info scalars.  One kernel packs the robot's side into a
        float64 row (navgym_export_env) and ONE device-to-host copy fetches it (a second one for
        the pedestrians, if any); synchronises the device -- a debugging / single-env aid, not
        part of the batched step path."""
        from types import SimpleNamespace
        from .robot import Human
        n_out = self.lib.navgym_export_env_len(self.num_scan_stack)
        if getattr(self, '_export_dev', None) is None:
            self._export_dev = torch.empty(n_out, dtype=torch.float64, device=self.device)
            self._export_host = torch.empty(n_out, dtype=torch.float64).pin_memory()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.navgym_export_env(C.byref(self.args), int(i), _ptr(self._export_dev),
                                                  self._stream()), 'export_env')
            self._export_host.copy_(self._export_dev, non_blocking=True)
            ped_host = None
            crowd = getattr(self, 'crowd', None)
            if crowd is not None:  # policy-driven pedestrians: float64 state of the PedestrianSim
                P = crowd.P
                packed = torch.cat([crowd.pose[i].reshape(-1), crowd.vel[i].reshape(-1),
                                    crowd.waypoint[i].reshape(-1), crowd.has_legs[i].double(),
                                    crowd.prev_action[i].reshape(-1).double(), crowd.v_pref[i],
                                    (crowd.nped[i:i + 1] if crowd.nped is not None else
                                     torch.full((1,), P, device=self.device)).double()])
                ped_host = packed.cpu()
            elif self.peds is not None:
                P = self.peds.shape[1]
                nn_ = self.nped[i:i + 1] if getattr(self, 'nped', None) is not None else torch.full((1,), P, device=self.device)
                ped_host = torch.cat([self.peds[i].reshape(-1).double(), nn_.double()]).cpu()
            torch.cuda.current_stream(self.device).synchronize()
        x = self._export_host.numpy().copy()
        st, tail = x[:NS], x[NS:NS + 7].copy()
        sc = x[NS + 7:NS + 17]
        m = self.pool.maps[int(sc[7])]
        robot = KetiRobot(float(st[_lib.S_PX]), float(st[_lib.S_PY]), float(st[_lib.S_TH]),
                          float(st[_lib.S_GX]), float(st[_lib.S_GY]), self.args.dt)
        robot.v, robot.r = float(st[_lib.S_PV]), float(st[_lib.S_PW])
        robot.vx, robot.vy = robot.v * np.cos(robot.theta), robot.v * np.sin(robot.theta)
        humans = []
        if ped_host is not None and crowd is not None:
            q = ped_host.numpy()
            n = int(q[-1])
            pose, vel, wp = q[:3 * P].reshape(P, 3), q[3 * P:5 * P].reshape(P, 2), q[5 * P:7 * P].reshape(P, 2)
            legs, act, vp = q[7 * P:8 * P], q[8 * P:10 * P].reshape(P, 2), q[10 * P:11 * P]
            for j in range(n):
                h = Human(float(pose[j, 0]), float(pose[j, 1]), float(pose[j, 2]), float(wp[j, 0]), float(wp[j, 1]), self.args.dt)
                h.vx, h.vy, h.has_legs, h.v_pref = float(vel[j, 0]), float(vel[j, 1]), bool(legs[j]), float(vp[j])
                h.v, h.r = float(act[j, 0] * vp[j]), float(act[j, 1] * vp[j])
                humans.append(h)
        elif ped_host is not None:
            q = ped_host.numpy()
            n = int(q[-1])
            for row in q[:-1].reshape(P, _lib.PED_F)[:n]:
                tgt = row[6:8] if row[8] > 0.5 else row[4:6]
                h = Human(float(row[0]), float(row[1]), float(row[2]), float(tgt[0]), float(tgt[1]), self.args.dt)
                h.v, h.has_legs = float(row[3]), bool(row[12] > 0.5)
                h.vx, h.vy = h.v * np.cos(h.theta), h.v * np.sin(h.theta)
                humans.append(h)
        obs = {'observation': np.concatenate([x[NS + 17:], tail]),
               'achieved_goal': tail[2:4].copy(), 'desired_goal': np.array([robot.gx, robot.gy])}
        return SimpleNamespace(map_info=m, robot=robot, humans=humans, prev_obs=obs,
                               num_scan_stack=self.num_scan_stack, steps_since_reset=int(sc[6]),
                               reward=float(np.float32(sc[0])), done=bool(sc[1]), is_success=bool(sc[2]),
                               is_crash=bool(sc[3]), truncated=bool(sc[4]), distance=float(np.float32(sc[5])),
                               episode=int(sc[8]), noise_std=float(np.float32(sc[9])))

    def obs_parts(self, rows=None):
        """(scans [N, S*512], tail [N, 7] float32) views of observation rows of this env's format:
        env.obs (rows=None) or any [N, width] tensor of the same dtype laid out like it, e.g. pinned
        host rows or a slice of a replay buffer.  float16 rows keep the tail as float32 in the 14
        halves after the scans, seen here through .view(torch.float32); for float32 rows the two
        are plain slices, so code written against obs_parts runs on either format."""
        rows = self.obs if rows is None else rows
        n = self.num_scan_stack * NB
        if rows.dtype != self.obs_dtype:
            raise ValueError('rows of dtype %s, the env keeps %s rows' % (rows.dtype, self.obs_dtype))
        if self.obs_dtype == torch.float16:
            return rows[:, :n], rows[:, n:n + 14].view(torch.float32)
        return rows[:, :n], rows[:, n:n + 7]

    # ---- HER batch API (env.py:491-589) on device tensors ---------------------------------
    def compute_rewards(self, obs, goals, **reward):
        """compute_rewards / compute_terminals / compute_info for stored observations:
        obs float32 [N, >=519] (row layout of env.py:455), or float16 rows in the layout of
        obs_dtype=torch.float16 (float16 scans, float32 tail; an even row stride, a 4-byte aligned
        start), whatever the env's own format; goals float32 [N, 2], both on the device.  Returns
        dict(reward, done, is_success, is_crash, distance) of device tensors."""
        if obs.dtype == torch.float16:
            obs_format = _lib.OBS_F16
            obs = obs.to(device=self.device)
        else:
            obs_format = _lib.OBS_F32
            obs = obs.to(device=self.device, dtype=torch.float32)
        if obs.stride(-1) != 1:
            obs = obs.contiguous()
        goals = goals.to(device=self.device, dtype=torch.float32).contiguous()
        n = obs.shape[0]
        out = dict(reward=torch.empty(n, dtype=torch.float32, device=self.device),
                   done=torch.empty(n, dtype=torch.uint8, device=self.device),
                   is_success=torch.empty(n, dtype=torch.uint8, device=self.device),
                   is_crash=torch.empty(n, dtype=torch.uint8, device=self.device),
                   distance=torch.empty(n, dtype=torch.float32, device=self.device))
        a, h = self.args, _lib.HerArgs()
        h.dist_thresh = a.dist_thresh
        h.r_scale, h.r_success, h.r_crash = a.r_scale, a.r_success, a.r_crash
        h.r_progress, h.r_forward, h.r_rotation, h.r_discomfort = a.r_progress, a.r_forward, a.r_rotation, a.r_discomfort
        for k, v in reward.items():
            setattr(h, {'reward_scale': 'r_scale', 'reward_success_factor': 'r_success',
                        'reward_crash_factor': 'r_crash', 'reward_progress_factor': 'r_progress',
                        'reward_forward_factor': 'r_forward', 'reward_rotation_factor': 'r_rotation',
                        'reward_discomfort_factor': 'r_discomfort'}[k], v)
        h.count, h.obs_stride, h.num_scan_stack = n, obs.stride(0), self.num_scan_stack
        h.obs_format = obs_format
        h.obs, h.goals, h.thr, h.dthr = _ptr(obs), _ptr(goals), _ptr(self.thr), _ptr(self.dthr)
        h.reward, h.done, h.is_success = _ptr(out['reward']), _ptr(out['done']), _ptr(out['is_success'])
        h.is_crash, h.distance = _ptr(out['is_crash']), _ptr(out['distance'])
        with torch.cuda.device(self.device):
            _lib.check(self.lib.navgym_compute_rewards(C.byref(h), self._stream()), 'compute_rewards')
        return out

    # ---- scripted pedestrians on the device ------------------------------------------------
    def attach_pedestrians(self, peds, nped=None, trunk_mode=False):
        """peds float32 [B, P, 16] (layout in include/navgym_b200.h), nped int32 [B] or None.
        From now on step() first advances the pedestrians (reference order: humans move
        env.py:659-662, then the robot :664) and scans against their geometry."""
        peds = torch.as_tensor(peds, dtype=torch.float32).to(self.device).contiguous()
        assert peds.shape[0] == self.B and peds.shape[2] == _lib.PED_F
        P = peds.shape[1]
        self.peds = peds
        self.nped = None if nped is None else torch.as_tensor(nped, dtype=torch.int32).to(self.device)
        need_disc, need_seg = (P, 0) if trunk_mode else (2 * P, 4 * P)
        if need_disc > _lib.MAX_DISC or need_seg > _lib.MAX_SEG:
            raise ValueError('too many pedestrians per environment')
        self.max_disc, self.max_seg = max(need_disc, 1), max(need_seg, 1)
        self.args.max_disc, self.args.max_seg = self.max_disc, self.max_seg
        f32, i32 = torch.float32, torch.int32
        self._pdiscs = torch.zeros(self.B, self.max_disc, 3, dtype=f32, device=self.device)
        self._psegs = torch.zeros(self.B, self.max_seg, 4, dtype=f32, device=self.device)
        self._pnd = torch.zeros(self.B, dtype=i32, device=self.device)
        self._pns = torch.zeros(self.B, dtype=i32, device=self.device)
        p = _lib.PedsArgs()
        p.num_envs, p.max_ped, p.max_disc, p.max_seg = self.B, P, self.max_disc, self.max_seg
        p.trunk_mode, p.dt = int(trunk_mode), self.args.dt
        p.peds, p.nped = _ptr(self.peds), _ptr(self.nped)
        p.discs, p.ndisc, p.segs, p.nseg = _ptr(self._pdiscs), _ptr(self._pnd), _ptr(self._psegs), _ptr(self._pns)
        self._pargs = p
        self.peds_scripted = True  # step() advances them itself; PedestrianSim turns this off
        self._peds_emit(advance=False)

    def _peds_emit(self, advance):
        self._pargs.advance = int(advance)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.navgym_peds_advance(C.byref(self._pargs), self._stream()), 'peds_advance')

    def _obstacles(self, discs, ndisc, segs, nseg, advance):
        """The obstacle buffers a launch reads: the caller's or, with none given, the attached
        pedestrians' geometry, emitted first (`advance`: scripted pedestrians move one step)."""
        if self.peds is None or discs is not None or segs is not None:
            return discs, ndisc, segs, nseg
        self._peds_emit(advance=advance and self.peds_scripted)
        return self._pdiscs, self._pnd, self._psegs, self._pns

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def reset(self, discs=None, ndisc=None, segs=None, nseg=None, noise=None):
        """First observation of an episode from the state set by set_state (env.py:822-831).
        With auto_reset='next_step' also clears done, so that the next step steps every env."""
        self._geom(*self._obstacles(discs, ndisc, segs, nseg, advance=False), noise)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.navgym_reset_obs_batch(C.byref(self.args), self._stream()), 'reset')
            if self.next_step_reset:
                self.done.zero_()
        return self.obs

    def env_mask(self, envs):
        """u8 [B] device mask of `envs`: a bool / uint8 [B] tensor on the env's device (returned
        as is, a bool tensor viewed as uint8: no copy), or a 1-D sequence / integer tensor of env
        ids (a new mask).  ValueError for anything else, or for ids outside [0, B)."""
        if torch.is_tensor(envs) and envs.dtype in (torch.bool, torch.uint8):
            if envs.device != self.device:
                raise ValueError('mask on %s, the env lives on %s' % (envs.device, self.device))
            if envs.dim() != 1 or envs.shape[0] != self.B:
                raise ValueError('mask of shape %s, expected [%d]' % (tuple(envs.shape), self.B))
            m = envs.contiguous()
            return m.view(torch.uint8) if m.dtype == torch.bool else m
        if torch.is_tensor(envs):
            if envs.dtype.is_floating_point or envs.dtype.is_complex:
                raise ValueError('env ids of dtype %s: pass a bool / uint8 mask or integer ids' % envs.dtype)
            if envs.device.type != 'cpu' and envs.device != self.device:
                raise ValueError('env ids on %s, the env lives on %s' % (envs.device, self.device))
            if envs.dim() > 1:
                raise ValueError('env ids must be 1-D')
            ids = envs.reshape(-1).to(device=self.device, dtype=torch.int64)
        else:
            arr = np.asarray(envs)
            if arr.size and arr.dtype.kind not in 'iu':
                raise ValueError('env ids of dtype %s: pass a bool / uint8 mask or integer ids' % arr.dtype)
            if arr.ndim > 1:
                raise ValueError('env ids must be 1-D')
            ids = torch.from_numpy(arr.astype(np.int64).reshape(-1)).to(self.device)
        if ids.numel() and (int(ids.min()) < 0 or int(ids.max()) >= self.B):
            raise ValueError('env ids outside [0, %d)' % self.B)
        m = torch.zeros(self.B, dtype=torch.uint8, device=self.device)
        m[ids] = 1
        return m

    def reset_envs(self, envs):
        """Start new episodes for the environments `envs` only, on the device, exactly as
        auto-reset would have started them (navgym_reset_envs): the same spawn / map / noise draw
        from each env's own episode counter, the same first observation.  Everything else is left
        as it is.  `envs`: a bool / uint8 [B] tensor on the env's device (env.done itself works,
        without a copy or a host sync) or a 1-D sequence / integer tensor of env ids.  Returns
        self.obs.

        Meant for auto_reset=False: step, read the rows of the ended episodes (their final
        observations; their goals are still state[S_GX / S_GY]), then reset_envs(done).  Works with
        auto_reset=True too.  With auto_reset='next_step' it clears done for `envs`, so that the
        next step steps them instead of starting yet another episode.  With scripted pedestrians
        the first scan sees the geometry the last step emitted, not advanced, as auto-reset does.
        An env driven by a PedestrianSim is reset through sim.reset_envs, which also respawns its
        pedestrians."""
        if getattr(self, 'crowd', None) is not None:
            raise ValueError('this env is driven by a PedestrianSim: call sim.reset_envs(envs), which also '
                             'respawns its pedestrians')
        return self._reset_envs(self.env_mask(envs))

    def _reset_envs(self, mask):
        self._reset_mask = mask  # kept alive until the next call; the launch is stream-ordered
        with torch.cuda.device(self.device):
            _lib.check(self.lib.navgym_reset_envs(C.byref(self.args), _ptr(mask), self._stream()), 'reset_envs')
            if self.next_step_reset:   # after the launch: `mask` may be done itself
                self.done.masked_fill_(mask.bool(), 0)
        return self.obs

    def step(self, actions, discs=None, ndisc=None, segs=None, nseg=None, noise=None):
        """One lockstep NavGymEnv.step.  Returned tensors are owned by the env and overwritten
        by the next call (clone to keep).

        With auto_reset='next_step' an env whose last step ended its episode (done set on entry)
        ignores its action and starts the next episode instead: its row is the first observation,
        its reward and flags are 0.  info['autoreset'] (bool [B], a new tensor) marks those envs;
        their transitions are not the policy's and belong in no replay buffer."""
        self._geom(*self._obstacles(discs, ndisc, segs, nseg, advance=True), noise, actions)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.navgym_step_batch(C.byref(self.args), self._stream()), 'step')
            info = dict(is_success=self.is_success, is_crash=self.is_crash, distance=self.distance,
                        episode_step=self.steps, truncated=self.truncated)
            if self.next_step_reset:   # a stepped env has steps >= 1
                info['autoreset'] = self.steps == 0
        if self.sched is not None:
            self.args.sched_phase = (self.args.sched_phase + 1) % 3
        return self.obs, self.reward, self.done, info
