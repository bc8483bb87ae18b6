"""GPU: the pedestrian pipeline on the device against the reference's recorded pipeline
(humans_*.npz) -- the batched pedestrian lidar bit-exactly, the policy forward within float32
summation-order tolerance."""
import numpy as np
import pytest
import torch

import golden_util as gu
from cuda_util import f32_reference

pytestmark = pytest.mark.gpu


def _scanner(G, B, P, max_seg):
    from nav_gym_b200.batched_env import MapPool
    from nav_gym_b200.pedestrians import AgentScanner
    pool = MapPool([gu.map_info(G)], 'cuda:0')
    map_id = torch.zeros(B, dtype=torch.int32, device='cuda:0')
    return AgentScanner(pool, B, P, max_seg, map_id, cell_rule='numpy2')


@pytest.mark.parametrize('name', gu.human_trace_names())
def test_agent_scan_batch_matches_reference_scans(name):
    """Every recorded step becomes one environment of a batch: the pedestrians' scans from their
    recorded poses, against the map and the recorded footprints of the others, equal the scans
    the reference stored -- bit for bit."""
    G = gu.load(name)
    T, P = G['pose_after'].shape[:2]
    per = [gu.human_env_segments(G, t) for t in range(T)]
    S = per[0][0].shape[0]
    segs = torch.from_numpy(np.stack([p[0] for p in per])).cuda()
    skip = torch.from_numpy(np.stack([p[1] for p in per])).cuda()
    nseg = torch.full((T,), S, dtype=torch.int32, device='cuda')
    sc = _scanner(G, T, P, S)
    r = sc.scan(torch.from_numpy(G['pose_after']).cuda().contiguous(), segs, nseg, skip)
    torch.cuda.synchronize()
    assert np.array_equal(r.cpu().numpy(), G['scan_out'])
    # fewer live agents than slots: the dead slots' rows are left alone
    sc.ranges.fill_(-1.0)
    nag = torch.full((T,), P - 1, dtype=torch.int32, device='cuda')
    r = sc.scan(torch.from_numpy(G['pose_after']).cuda().contiguous(), segs, nseg, skip, nag)
    torch.cuda.synchronize()
    r = r.cpu().numpy()
    assert np.array_equal(r[:, :P - 1], G['scan_out'][:, :P - 1]) and (r[:, P - 1] == -1).all()
    # the first scans of the episode (reset, env.py:808-815) from the start poses
    segs0, skip0 = gu.human_env_segments(G, 0)
    from nav_gym_b200.pedestrians import footprint_polygons
    from nav_gym_b200.robot import Human, KetiRobot
    poly = footprint_polygons(torch.from_numpy(G['pose0']), Human.footprint).reshape(-1, 4)
    rob = footprint_polygons(torch.from_numpy(G['robot0']), KetiRobot.threshold_footprint).reshape(-1, 4)
    env_segs = torch.cat((rob, poly)).cuda()[None].contiguous()
    sk = torch.tensor([[4 * (1 + j), 4] for j in range(P)], dtype=torch.int32, device='cuda')[None].contiguous()
    sc1 = _scanner(G, 1, P, env_segs.shape[1])
    r0 = sc1.scan(torch.from_numpy(G['pose0'])[None].cuda().contiguous(), env_segs,
                  torch.tensor([env_segs.shape[1]], dtype=torch.int32, device='cuda'), sk)
    torch.cuda.synchronize()
    got, want = r0[0].cpu().numpy(), G['scan0']
    # footprints rebuilt on the device may differ from the reference's by a float32 ulp, which
    # moves a beam's hit on a footprint edge by ~1e-6 m; map hits stay exact
    assert np.allclose(got, want, rtol=0, atol=2e-5) and (got == want).mean() > 0.97


@pytest.mark.parametrize('name', gu.human_trace_names())
def test_policy_forward_on_device(name):
    from nav_gym_b200.pedestrians import HumanPolicy
    G = gu.load(name)
    torch.manual_seed(1234)
    pol = HumanPolicy().cuda()
    T, P = G['mean'].shape[:2]
    x = torch.from_numpy(G['scan_in']).cuda().reshape(T * P, 1, 512).expand(-1, 3, -1).contiguous()
    with torch.no_grad():
        m = pol.mean(x, torch.from_numpy(G['goal_local']).cuda().reshape(-1, 2),
                     torch.from_numpy(G['speed']).cuda().reshape(-1, 2))
    assert np.allclose(m.cpu().numpy().reshape(T, P, 2), G['mean'], rtol=0, atol=2e-5)


@pytest.mark.parametrize('n', [1, 77, 128, 300, 1029, 19200])
def test_native_policy_stage_by_stage(n):
    """navgym_policy_mean (front end -> tcgen05 act_fc1 in the f16x3 scheme -> act_fc2 + heads)
    against torch float32 / float64 on random scans, one stage at a time: the feature halves
    re-assemble the float32 features, the tensor-core layer equals a float64 product of those
    very features to float32 rounding, the means equal torch's float32 forward.  n covers a
    single row, partial 128-row tiles, several tiles per CTA, and (19 200 = 150 tiles on 148 SMs) a last
    round whose left-over tiles act_fc1 splits along N."""
    import torch.nn.functional as F
    from nav_gym_b200.pedestrians import HumanPolicy, NativePolicy, preprocess_scan
    torch.manual_seed(7)
    pol = HumanPolicy().cuda()
    with torch.no_grad():   # default-init biases are small; make every term count
        pol.act_fc1.bias.uniform_(-0.3, 0.3)
        pol.act_fea_cv2.bias.uniform_(-0.2, 0.2)
    g = torch.Generator(device='cuda').manual_seed(n)
    scan = (8.0 * torch.rand(n, 512, device='cuda', generator=g) - 1.0).contiguous()   # beyond [0, 6] on both sides
    goal = 4.0 * torch.rand(n, 2, device='cuda', generator=g) - 2.0
    speed = torch.rand(n, 2, device='cuda', generator=g)
    nat = NativePolicy(pol, max(n, 5), 'cuda:0')
    got = nat.mean(scan, goal, speed)
    torch.cuda.synchronize()
    fh, fl, h, scales = nat.intermediates(n)
    x3 = preprocess_scan(scan)[:, None, :].expand(-1, 3, -1).contiguous()
    feat = f32_reference(lambda: F.relu(pol.act_fea_cv2(F.relu(pol.act_fea_cv1(x3)))).reshape(n, -1))
    s_f = float(scales[0])
    assert s_f > 0 and np.log2(s_f) == int(np.log2(s_f)) and float(fh.float().abs().max()) < 32768.0
    mine = (fh.double() + fl.double()) / s_f
    assert float((mine - feat.double()).abs().max()) < 4e-6   # conv2 runs in the f16x3 scheme too
    assert float(((fh.double() + fl.double()) / s_f - mine).abs().max()) == 0.0
    # the tensor-core layer on the features the kernel itself produced
    # (12 288 products per output accumulate in the tensor core's float32 adder: a few 1e-6, the
    # size of a float32 GEMM's own rounding -- torch's SGEMM is checked against the same bar)
    with torch.no_grad():
        want_h = torch.relu(mine @ pol.act_fc1.weight.double().t() + pol.act_fc1.bias.double())
        err = float((h.double() - want_h).abs().max())
        sgemm = f32_reference(lambda: torch.relu(mine.float() @ pol.act_fc1.weight.t() + pol.act_fc1.bias))
        err_sgemm = float((sgemm.double() - want_h).abs().max())
    bar = 1e-5 * max(1.0, float(want_h.abs().max()))
    assert err < bar and err_sgemm < bar, (err, err_sgemm)
    want = f32_reference(lambda: pol.mean(x3, goal, speed))
    assert float((got - want).abs().max()) < 1e-5


@pytest.mark.parametrize('name', gu.human_trace_names())
def test_native_policy_reproduces_the_reference_means(name):
    """The reference's recorded policy outputs (humans_*.npz `mean`, minted by running its own
    human_policy.py on the CPU) from its recorded raw scans, through the native pipeline; the
    recorded policy inputs are those raw scans preprocessed."""
    from nav_gym_b200.pedestrians import HumanPolicy, NativePolicy, preprocess_scan
    G = gu.load(name)
    torch.manual_seed(1234)
    pol = HumanPolicy().cuda()
    T, P = G['mean'].shape[:2]
    # the raw scans the policy inputs were made from: scan0, then each step's scan_out
    raw = np.concatenate([G['scan0'][None], G['scan_out'][:-1]]).reshape(T * P, 512)
    x = torch.from_numpy(raw).cuda()
    assert np.array_equal(preprocess_scan(x).cpu().numpy().reshape(T, P, 512), G['scan_in'])
    nat = NativePolicy(pol, T * P, 'cuda:0')
    m = nat.mean(x, torch.from_numpy(G['goal_local']).cuda().reshape(-1, 2).contiguous(),
                 torch.from_numpy(G['speed']).cuda().reshape(-1, 2).contiguous())
    torch.cuda.synchronize()
    assert np.allclose(m.cpu().numpy().reshape(T, P, 2), G['mean'], rtol=0, atol=2e-5)


def _crowd(B=64, P=6, seed=0):
    from nav_gym_b200 import maps
    from nav_gym_b200.batched_env import BatchedNavGym, MapPool, filter_spawn_pool
    from nav_gym_b200.pedestrians import PedestrianSim
    rng = np.random.RandomState(3)
    m = maps.create_indoor_map(3, 100, rng)
    pool = filter_spawn_pool(m, maps.spawn_pool(m, 2048, rng), 'cuda:0')
    mp = MapPool([m], 'cuda:0', spawn_pools=[pool])
    env = BatchedNavGym(B, mp, seed=seed, auto_reset=True)
    env.reset_from_spawn_pool(np.random.RandomState(seed))
    return m, env, PedestrianSim(env, P, seed=seed)


def test_pedestrian_sim_policy_matches_the_float32_forward():
    """PedestrianSim's policy forward (sim.native) on its own scans against torch's float32 forward."""
    m, env, sim = _crowd(B=32, P=8, seed=3)
    from nav_gym_b200.pedestrians import preprocess_scan
    x = sim.scan.reshape(-1, 512)
    goal, speed = sim.goal_local.reshape(-1, 2), torch.rand(32 * 8, 2, device='cuda')
    want = f32_reference(lambda: sim.policy.mean(preprocess_scan(x)[:, None, :].expand(-1, 3, -1).contiguous(), goal, speed))
    got = sim.native.mean(x, goal, speed)
    assert float((got - want).abs().max()) < 1e-5


def test_native_pedestrian_sim_follows_the_reference_step_order():
    """One PedestrianSim step against a by-hand evaluation of env.py:617-693 on the same state:
    policy mean (the native forward, against torch's float32 forward) from the previous scan /
    local goal / previous action, Human.set_vel with the preferred-speed factor, leg odometry,
    and the new scans from the new poses."""
    from nav_gym_b200.pedestrians import human_set_vel, preprocess_scan
    m, env, sim = _crowd(B=16, P=5, seed=1)
    g = torch.Generator(device='cuda'); g.manual_seed(0)
    for t in range(3):
        pose0, scan0, prev_a = sim.pose.clone(), sim.scan.clone(), sim.prev_action.clone()
        dist0 = sim.dist_travelled.clone()
        act = torch.rand(16, 2, device='cuda', generator=g) * torch.tensor([0.5, 1.28], device='cuda') + torch.tensor([0, -0.64], device='cuda')
        sim.step(act)
        torch.cuda.synchronize()
        done = env.done.bool()
        # waypoints: 1 m .. a few m ahead, and the local goal is that point in the old frame
        wp = sim.waypoint
        rel = wp - pose0[..., :2]
        c, s = torch.cos(pose0[..., 2]), torch.sin(pose0[..., 2])
        loc = torch.stack((rel[..., 0] * c + rel[..., 1] * s, -rel[..., 0] * s + rel[..., 1] * c), -1)
        assert torch.allclose(loc.float(), sim.goal_local, atol=1e-5)
        x = preprocess_scan(scan0).reshape(-1, 1, 512).expand(-1, 3, -1).contiguous()
        mean = f32_reference(lambda: sim.policy.mean(x, sim.goal_local.reshape(-1, 2), prev_a.reshape(-1, 2))).reshape(16, 5, 2)
        clipped = torch.minimum(torch.maximum(mean, torch.tensor([0., -1.], device='cuda')), torch.tensor([1., 1.], device='cuda'))
        assert torch.allclose(clipped, sim.prev_action, atol=1e-5)
        pose1, vel1 = human_set_vel(pose0, sim.prev_action.double() * sim.v_pref[..., None], 0.2)
        assert torch.allclose(pose1, sim.pose, atol=1e-12) and torch.allclose(vel1, sim.vel, atol=1e-12)
        yaw0 = torch.atan2(torch.sin(pose0[..., 2]), torch.cos(pose0[..., 2]))
        vrot = (pose1[..., 2] - yaw0) / 0.2
        c, s = torch.cos(pose1[..., 2]), torch.sin(pose1[..., 2])
        base = torch.stack((c * vel1[..., 0] + s * vel1[..., 1], -s * vel1[..., 0] + c * vel1[..., 1], vrot), -1)
        assert torch.allclose(dist0 + base * 0.2, sim.dist_travelled, atol=1e-12)
        assert not done.any()  # (a respawn would break the by-hand bookkeeping above)
        # the robot's lidar saw them: every non-legged pedestrian contributes 4 segments, legged 2 discs
        legs = sim.has_legs.sum(1)
        assert torch.equal(env._pnd.long(), 2 * legs) and torch.equal(env._pns.long(), 4 * (5 - legs))
        # scans: finite, in [0, 6], and a pedestrian close to another one sees it
        assert float(sim.scan.min()) >= 0 and float(sim.scan.max()) <= 6.0


def test_pedestrian_sim_scans_match_oracle_and_routes_descend():
    """The scans PedestrianSim stores equal the oracle's pedestrian scan of the same poses and
    footprints; waypoints lie on free cost-map cells 1-3.5 m from where they were issued, and
    following them brings a pedestrian walking at its waypoint to its goal."""
    from oracle import oracle as orc
    from test_pedestrians import oracle_human_scan
    m, env, sim = _crowd(B=8, P=4, seed=2)
    torch.cuda.synchronize()
    dist = orc.edt(np.asarray(m['data']) >= 0.1)
    from nav_gym_b200.pedestrians import footprint_polygons
    from nav_gym_b200.robot import Human, KetiRobot
    # crowd the pedestrians around the robot so that they see each other and it
    g = torch.Generator(device='cuda'); g.manual_seed(5)
    rob = env.state[:3].t().contiguous()
    sim.pose[..., :2] = rob[:, None, :2] + (torch.rand(8, 4, 2, device='cuda', generator=g, dtype=torch.float64) - 0.5) * 8
    sim.observe()
    torch.cuda.synchronize()
    segs = torch.cat((footprint_polygons(rob, KetiRobot.threshold_footprint),
                      footprint_polygons(sim.pose, Human.footprint).reshape(8, -1, 4)), 1).cpu().numpy()
    pose = sim.pose.cpu().numpy()
    scan = sim.scan.cpu().numpy()
    seen = 0
    for e in range(8):
        for i in range(4):
            keep = np.ones(20, bool)
            keep[4 * (1 + i):4 * (2 + i)] = False
            want = oracle_human_scan(dist, m, pose[e, i], segs[e][keep], cell_rule=0)
            bare = oracle_human_scan(dist, m, pose[e, i], np.zeros((0, 4), np.float32), cell_rule=0)
            seen += int((want != bare).sum())
            assert np.array_equal(want, scan[e, i]), (e, i)
    assert seen > 100  # the footprints did shape the scans
    # route following: teleport each pedestrian onto its waypoint, repeatedly
    sim.reset()
    fields = sim.fields.cpu().numpy().view(np.uint16).reshape(sim.num_goals, 200, 200)
    goals = sim.goals.cpu().numpy()
    d_prev, gid_prev, changes = None, None, 0
    for it in range(300):
        sim._plan(None)
        torch.cuda.synchronize()
        wp = sim.waypoint.cpu().numpy()
        p = sim.pose.cpu().numpy()
        gid = sim.goal_id.cpu().numpy()
        step_len = np.hypot(*(wp - p[..., :2]).transpose(2, 0, 1))
        cx, cy = (wp[..., 0] / 0.25).astype(int), (wp[..., 1] / 0.25).astype(int)
        d_now = fields[gid, cy, cx].astype(np.int64)
        assert (d_now < 65535).all()
        if gid_prev is None:
            assert (step_len < 3.6).all()         # the first waypoint is ~2 m down the field
        else:
            same = gid == gid_prev
            assert (d_now[same] <= d_prev[same]).all()      # never uphill
            new = ~same
            changes += int(new.sum())
            # a new goal is drawn on arrival only, and lies farther than min_goal_dist
            assert (np.hypot(*(goals[gid_prev] - p[..., :2]).transpose(2, 0, 1))[new] < 0.5).all()
            assert (np.hypot(*(goals[gid] - p[..., :2]).transpose(2, 0, 1))[new] > 10.0).all()
        d_prev, gid_prev = d_now, gid.copy()
        sim.pose[..., :2] = torch.from_numpy(wp).cuda()
    assert changes >= 8  # 32 pedestrians walking 2 m a call for 300 calls: many arrivals


def test_auto_reset_first_scan_sees_the_next_episodes_pedestrians():
    """When an episode ends inside the fused step, the new episode's first observation is taken
    against the pedestrians drawn for it (candidates of the preceding act()), which the next
    act() then adopts: at least 4 m from the robot's new start, and the scan equals the
    oracle's scan of the new pose with exactly that geometry."""
    from oracle import oracle as orc
    m, env, sim = _crowd(B=256, P=4, seed=4)
    env.args.noise_lo = env.args.noise_hi = 0.0
    env.noise_std.zero_()
    g = torch.Generator(device='cuda'); g.manual_seed(1)
    checked = 0
    dist = orc.edt(np.asarray(m['data']) >= 0.1)
    for t in range(60):
        act = torch.rand(256, 2, device='cuda', generator=g) * torch.tensor([0.5, 1.28], device='cuda') + torch.tensor([0, -0.64], device='cuda')
        sim.act()
        cand_pose = sim.cand_pose.clone()
        cd, cnd = sim.cand_discs.clone(), sim.cand_nd.clone()
        cs, cns = sim.cand_segs.clone(), sim.cand_ns.clone()
        env.step(act)
        sim.observe()
        torch.cuda.synchronize()
        done = env.done.bool().cpu().numpy()
        if t < 3:
            continue  # (noise of the episodes that started before it was switched off)
        for e in np.where(done)[0][:4]:
            st = env.state[:, e].cpu().numpy()
            rob = st[:3]
            d = np.hypot(*(cand_pose[e, :, :2].cpu().numpy() - rob[:2]).T)
            assert (d >= 4.0 - 1e-9).all()
            ob = orc.OracleBatch([m], np.zeros(1, np.int32), rob[None, :2], st[None, 3:5], rob[None, 2:3],
                                 max_disc=env.max_disc, max_seg=env.max_seg)
            ob.reset_obs(cd[e][None].cpu().numpy(), cnd[e][None].cpu().numpy(), cs[e][None].cpu().numpy(),
                         cns[e][None].cpu().numpy())
            assert np.array_equal(ob.obs[0, :512], env.obs[e, :512].cpu().numpy())
            checked += 1
        # the next act() adopts exactly those pedestrians
        if done.any() and checked >= 3:
            sim._plan(env.done)
            torch.cuda.synchronize()
            for e in np.where(done)[0]:
                assert torch.equal(sim.pose[e], cand_pose[e])
            break
    assert checked >= 3


def test_respawn_follows_the_map_drawn_at_auto_reset():
    """Two different maps, resample_map: when an episode ends the robot may move to the other map,
    and the pedestrians adopted for the new episode stand on free cost-map cells of THAT map, at
    least 4 m from the robot's new start."""
    from nav_gym_b200 import maps
    from nav_gym_b200.batched_env import BatchedNavGym, MapPool, filter_spawn_pool
    from nav_gym_b200.pedestrians import PedestrianSim
    rng = np.random.RandomState(8)
    ms = [maps.create_indoor_map(3, 100, rng), maps.create_outdoor_map(10, 0.7, rng)]
    pools = [filter_spawn_pool(ms[0], maps.spawn_pool(ms[0], 1024, rng), 'cuda:0'),
             filter_spawn_pool(ms[1], maps.spawn_pool(ms[1], 1024, rng, min_goal_dist=5, max_goal_dist=15), 'cuda:0')]
    mp = MapPool(ms, 'cuda:0', spawn_pools=pools)
    B, P = 256, 3
    env = BatchedNavGym(B, mp, seed=3, auto_reset=True, resample_map=True,
                        map_id=rng.randint(0, 2, B).astype(np.int32))
    env.reset_from_spawn_pool(np.random.RandomState(1))
    sim = PedestrianSim(env, P, seed=3)
    cms = [maps.cost_map(m) for m in ms]
    g = torch.Generator(device='cuda'); g.manual_seed(2)
    moved = checked = 0
    for t in range(50):
        act = torch.rand(B, 2, device='cuda', generator=g) * torch.tensor([0.5, 1.28], device='cuda') + torch.tensor([0, -0.64], device='cuda')
        map_before = env.map_id.clone()
        sim.act()
        env.step(act)
        sim.observe()
        torch.cuda.synchronize()
        done = env.done.bool()
        if not done.any():
            continue
        sim._plan(env.done)            # what the next act() does first: adopt the new pedestrians
        torch.cuda.synchronize()
        pose = sim.pose.cpu().numpy()
        rob = env.state[:2].t().cpu().numpy()
        mid = env.map_id.cpu().numpy()
        moved += int((env.map_id != map_before)[done].sum())
        for e in np.where(done.cpu().numpy())[0]:
            cm = cms[mid[e]]
            c = (pose[e, :, 0] / cm['resolution']).astype(int)
            r = (pose[e, :, 1] / cm['resolution']).astype(int)
            assert (c < cm['width']).all() and (r < cm['height']).all()
            assert (cm['data'][r, c] == 0).all(), (t, e)
            assert (np.hypot(*(pose[e, :, :2] - rob[e]).T) >= 4.0 - 1e-9).all()
            checked += 1
        env.done.zero_()               # consumed: the loop's next act() must not adopt again
    assert checked > 20 and moved > 5


@pytest.mark.parametrize('agent_name', ['Human', 'KetiRobot'])
def test_agent_scan_beam_windows_and_long_segment_lists(agent_name):
    """The pedestrian-lidar kernel evaluates a segment only on the beams of its angular window: against
    the oracle's all-beams loop on segments chosen to stress the window arithmetic -- touching the agent,
    behind it (across the +-pi seam of the bearing), spanning more than half a turn, degenerate (zero
    length), far out of range -- for the 180 degree / 6 m pedestrian lidar and the 360 degree / 25 m one
    (whose windows wrap around the beam table).  The same list padded to more slots than the kernel
    stages in shared memory takes the fallback kernel (every segment against every beam): identical."""
    from oracle import oracle as orc
    import synth
    from nav_gym_b200 import robot as R
    from nav_gym_b200.batched_env import MapPool
    from nav_gym_b200.pedestrians import AgentScanner
    agent = getattr(R, agent_name)
    rng = np.random.RandomState(11)
    m = synth.indoor_map(rng, cells=60, iterations=40)
    occ = np.asarray(m['data']) >= 0.1
    dist = orc.edt(occ)
    B, P, S = 6, 5, 48
    xy = synth.free_poses(rng, m, B * P, 6, dist).reshape(B, P, 2)
    pose = np.concatenate([xy, rng.uniform(0, 2 * np.pi, (B, P, 1))], 2)
    segs = np.zeros((B, S, 4), np.float32)
    for e in range(B):
        for s in range(S):
            i = rng.randint(P)
            c = xy[e, i]
            kind = s % 6
            if kind == 0:      # a short segment somewhere within range
                a = c + rng.uniform(-5, 5, 2); b = a + rng.uniform(-0.6, 0.6, 2)
            elif kind == 1:    # through (or touching) the agent's position
                d = rng.uniform(-1, 1, 2); a = c - d * rng.uniform(0, 1); b = c + d
            elif kind == 2:    # behind the agent, across the bearing seam
                th = pose[e, i, 2] + np.pi; n = np.array([-np.sin(th), np.cos(th)])
                mid = c + 2.0 * np.array([np.cos(th), np.sin(th)]); a = mid + n; b = mid - n
            elif kind == 3:    # long: subtends more than half a turn
                d = rng.uniform(-1, 1, 2); d /= np.linalg.norm(d) + 1e-9
                off = 0.05 * np.array([-d[1], d[0]]); a = c + off - 30 * d; b = c + off + 30 * d
            elif kind == 4:    # zero length
                a = c + rng.uniform(-3, 3, 2); b = a.copy()
            else:              # far out of range
                a = c + np.array([60.0, 45.0]); b = a + rng.uniform(-1, 1, 2)
            segs[e, s] = [a[0], a[1], b[0], b[1]]
    nseg = np.full(B, S, np.int32)
    nseg[1] = 0
    nseg[2] = 7
    lin = R.beam_table(agent)
    want = np.empty((B, P, 512), np.float32)
    res = np.float32(m['resolution'])
    H, W = dist.shape
    for e in range(B):
        for i in range(P):
            lx, ly, lt = np.float32(pose[e, i, 0]), np.float32(pose[e, i, 1]), np.float32(pose[e, i, 2])
            head, dirs = orc.beam_dirs(lt, lin)
            ci = orc.lib().nvo_xy_to_cell(float(lx), float(m['origin'][0]), float(m['resolution']), H, 0)
            cj = orc.lib().nvo_xy_to_cell(float(ly), float(m['origin'][1]), float(m['resolution']), W, 0)
            ins = np.column_stack([np.full(512, ci), np.full(512, cj), head]).astype(np.float32)
            r = np.ascontiguousarray(orc.calc_range_many(dist, ins, float(W * H)) * res, np.float32)
            orc.render_segments(r, dirs, segs[e, :nseg[e]], np.array([lx, ly], np.float32))
            want[e, i] = np.clip(r, 0, np.float32(agent.range_max))
    pool = MapPool([m], 'cuda:0')
    map_id = torch.zeros(B, dtype=torch.int32, device='cuda:0')
    tp = torch.from_numpy(pose).cuda().contiguous()
    for slots in (S, 520):   # 520 > the 512 segments the kernel stages: the fallback kernel
        padded = np.zeros((B, slots, 4), np.float32)
        padded[:, :S] = segs
        sc = AgentScanner(pool, B, P, slots, map_id, agent=agent, cell_rule='numpy1')
        got = sc.scan(tp, torch.from_numpy(padded).cuda().contiguous(), torch.from_numpy(nseg).cuda()).cpu().numpy()
        assert np.array_equal(got, want), (agent_name, slots, int((got != want).sum()))
    assert np.isfinite(want).all() and want.max() <= agent.range_max
