"""The pedestrian policy forward (navgym_policy_mean: policy_features_umma2_kernel -> act_fc1 ->
act_fc2 + heads, csrc/policy_gemm.cuh) against a float64 evaluation of the same policy, stage by
stage: features, h = relu(act_fc1), means.

The kernels run in the f16x3 scheme (float32 operands as f16 hi/lo halves times power-of-two scales
that policy_prepare_kernel picks from the weights).  Their error bars scale with the data: a stage
Q passes when max|Q_native - Q_f64| <= max(k x max|Q_torch_f32 - Q_f64|, floor), with k = 10 for
the features and the means and FC1_FACTOR = 30 for act_fc1's output (see there), the floor being
2^-20 max|Q_f64| for features and h and 1e-6 for the means.  Losing one of the three hi/lo
products, or one half, costs ~2^-13 relative: far above the bar.

Covered: act_fc1's tile schedule (whole tiles in rounds, the leftover tiles of a last round split
along N in 4, 2 or 1 parts, accumulators reused inside a launch), the front end's distribution of
pedestrians over CTAs and groups, reuse of one workspace across batch sizes, exact power-of-two
invariance of the scale choice, weight sets far from PyTorch's default init, and edge scans."""
import copy
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from cuda_util import f32_reference

BM = 128                      # rows per act_fc1 tile (pg::BM)
FEAT_FLOOR = 2.0 ** -20       # features and h: relative to max|Q_f64|
MEAN_FLOOR = 1e-6
# act_fc1 adds 3 x 256 MMAs (K 16 each) into one float32 accumulator per output, and the tensor
# core rounds each of those sums toward zero: its error grows with the step count and leans toward
# zero.  Measured on a B200 it is 10-12x SGEMM's; a numpy emulation with a truncating accumulator
# gives the same (rounding to nearest would give ~1x).  Dropping the fh x wl product costs ~100x.
FC1_FACTOR = 30.0
SENTINEL = -7.25


# ---------------------------------------------------------------- act_fc1's work list
def fc1_schedule(n, sms):
    """Python mirror of dense_umma_kernel's work list (policy_gemm.cuh, `item()`) for act_fc1 at
    n rows on `sms` SMs: grid, whole rounds, leftover tiles, their split along N, and the most
    work items any CTA gets."""
    tiles = -(-n // BM)
    grid = min(tiles, sms)
    rounds = tiles // grid
    rem = tiles - rounds * grid
    split = 1
    if rem > 0:   # Fc1: WBOX 64 < BN 256, so leftover tiles are split
        split = 4 if rem * 4 <= grid else (2 if rem * 2 <= grid else 1)
    return dict(n=n, tiles=tiles, grid=grid, rounds=rounds, rem=rem, split=split,
                items=rounds + (1 if rem > 0 else 0))


SCHEDULE_CASES = ('grid_below_sms', 'one_round', 'split4_top', 'split2_bottom', 'split2_top',
                  'split1_bottom', 'split1_top', 'two_rounds', 'bench_crowd', 'five_items')


def schedule_sizes(sms):
    """Batch sizes that put act_fc1's work list in every regime for a device with `sms` SMs.  Where
    the size is not a multiple of 128 the last tile is partial (71 rows), and it lies in a
    leftover item."""
    partial = lambda tiles: BM * tiles - 57
    return {
        'grid_below_sms': partial(sms - 1),             # fewer tiles than SMs
        'one_round': BM * sms,                          # exactly one tile per CTA
        'split4_top': partial(sms + sms // 4),          # most leftover tiles that still split in 4
        'split2_bottom': partial(sms + sms // 4 + 1),   # fewest that split in 2
        'split2_top': partial(sms + sms // 2),
        'split1_bottom': partial(sms + sms // 2 + 1),   # leftover tiles, not split
        'split1_top': partial(2 * sms - 1),             # sms - 1 leftover tiles
        'two_rounds': BM * 2 * sms,                     # two whole rounds, nothing left over
        'bench_crowd': 4096 * 10,                       # bench.py's crowd: 4096 envs x 10 pedestrians
        'five_items': partial(4 * sms + 1),             # 4 rounds + 1 tile: 5 items, each accumulator reused twice
    }


def assert_schedule_coverage(sms):
    sched = [fc1_schedule(n, sms) for n in schedule_sizes(sms).values()]
    assert {s['split'] for s in sched if s['rem'] > 0} == {1, 2, 4}, sched
    assert any(s['rem'] == 0 and s['rounds'] >= 2 for s in sched), sched
    assert any(s['grid'] < sms for s in sched), sched
    assert any(s['items'] >= 3 for s in sched) and any(s['items'] >= 5 for s in sched), sched
    assert any(s['rem'] > 0 and s['n'] % BM for s in sched), sched   # a partial tile inside a leftover item


def test_schedule_sizes_cover_every_regime():
    """CPU: the size picker reaches every act_fc1 schedule regime on devices of 148, 132 and 160
    SMs, and gives the sizes worked out by hand for the B200's 148."""
    for sms in (148, 132, 160):
        assert_schedule_coverage(sms)
    sizes = schedule_sizes(148)
    assert [sizes[k] for k in SCHEDULE_CASES] == [18759, 18944, 23623, 23751, 28359, 28487, 37703, 37888, 40960, 75847]
    bench = fc1_schedule(40960, 148)
    assert (bench['tiles'], bench['rem'], bench['split'], bench['items']) == (320, 24, 4, 3)


# ---------------------------------------------------------------- policies, inputs, references
def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _policy(seed=7):
    from nav_gym_b200.pedestrians import HumanPolicy
    torch.manual_seed(seed)
    return HumanPolicy().cuda().eval()


def _inputs(n, seed, scans=None):
    """Random scans beyond [0, 6] m on both sides (the given edge scans first), goals, speeds."""
    g = torch.Generator(device='cuda').manual_seed(seed)
    scan = 8.0 * torch.rand(n, 512, device='cuda', generator=g) - 1.0
    if scans is not None:
        scan[:scans.shape[0]] = scans
    goal = 4.0 * torch.rand(n, 2, device='cuda', generator=g) - 2.0
    speed = torch.rand(n, 2, device='cuda', generator=g)
    return scan.contiguous(), goal.contiguous(), speed.contiguous()


def _edge_scans(pol):
    """Scans at the edges of the front end's input range: all 0 m, all 6 m, beyond 6 m, negative,
    +inf; alternating 0 / 6 m; a single 0 m beam in 6 m at every beam; and, for the first and the
    last conv1 window, inputs at +-0.5 with the signs of each conv1 channel's (frame-folded)
    weights, which drives that channel to its bound (the rest of the scan at 3 m, input 0)."""
    rows = [torch.full((512,), v) for v in (0.0, 6.0, 7.5, -1.0, float('inf'))]
    alt = torch.zeros(512)
    alt[1::2] = 6.0
    rows += [alt, 6.0 - alt]
    onehot = torch.full((512, 512), 6.0)
    onehot.fill_diagonal_(0.0)
    w1f = pol.act_fea_cv1.weight.detach().sum(1).cpu()   # [32, 5]
    win = []
    for c in range(32):
        first, last = torch.full((512,), 3.0), torch.full((512,), 3.0)
        first[0:4] = 6.0 * (w1f[c, 1:5] > 0)   # conv1 output 0 reads inputs -1 (padding) .. 3
        last[507:512] = 6.0 * (w1f[c] > 0)     # conv1 output 254 reads inputs 507 .. 511
        win += [first, last]
    return torch.cat((torch.stack(rows), onehot, torch.stack(win))).cuda()


def _x3(scan, dtype):
    """The policy input: the preprocessed scan (float32, as the reference feeds it) in 3 identical frames."""
    from nav_gym_b200.pedestrians import preprocess_scan
    return preprocess_scan(scan).to(dtype)[:, None, :].expand(-1, 3, -1).contiguous()


def _stages(pol, x, goal, speed):
    """(features, h = relu(act_fc1), means): HumanPolicy.mean's sequence, keeping the stages."""
    feat = F.relu(pol.act_fea_cv2(F.relu(pol.act_fea_cv1(x)))).reshape(x.shape[0], -1)
    h = F.relu(pol.act_fc1(feat))
    a = F.relu(pol.act_fc2(torch.cat((h, goal, speed), dim=-1)))
    return feat, h, torch.cat((torch.sigmoid(pol.actor1(a)), torch.tanh(pol.actor2(a))), dim=-1)


def _references(pol, scan, goal, speed):
    """The three stages in float64 (a double copy of the policy) and in torch float32 (TF32 off)."""
    pol64 = copy.deepcopy(pol).double()
    with torch.no_grad():
        r64 = _stages(pol64, _x3(scan, torch.float64), goal.double(), speed.double())
    r32 = f32_reference(lambda: _stages(pol, _x3(scan, torch.float32), goal, speed))
    return r64, r32


def _native(pol, scan, goal, speed, max_n=None, pad=BM):
    """navgym_policy_mean into a sentinel-filled buffer `pad` rows longer than n; (features as
    float64 from the kernel's hi + lo halves, h, means, scales, the untouched tail)."""
    from nav_gym_b200.pedestrians import NativePolicy
    n = scan.shape[0]
    nat = NativePolicy(pol, max_n or n, 'cuda:0')
    buf = torch.full((n + pad, 2), SENTINEL, device='cuda')
    nat.mean(scan, goal, speed, out=buf[:n])
    torch.cuda.synchronize()
    fh, fl, h, scales = nat.intermediates(n)
    s_f = float(scales[0])
    feat = (fh.double() + fl.double()) / s_f
    return dict(nat=nat, feat=feat, h=h, mean=buf[:n], tail=buf[n:], scales=scales.clone())


def _err(a, b):
    return float((a.double() - b.double()).abs().max())


def _check_stages(got, r64, r32, record=None):
    """Each stage within max(k x torch float32's error, floor) of float64; returns the ratios."""
    ratios = {}
    for name, nat, q64, q32 in (('features', got['feat'], r64[0], r32[0]), ('h', got['h'], r64[1], r32[1]),
                                ('mean', got['mean'], r64[2], r32[2])):
        e_nat, e_f32 = _err(nat, q64), _err(q32, q64)
        floor = MEAN_FLOOR if name == 'mean' else FEAT_FLOOR * float(q64.abs().max())
        bar = max((FC1_FACTOR if name == 'h' else 10.0) * e_f32, floor)
        ratios[name] = e_nat / e_f32 if e_f32 > 0 else float('inf') if e_nat > 0 else 0.0
        if record is not None:
            record('%s_err_native' % name, e_nat)
            record('%s_err_f32' % name, e_f32)
        assert e_nat <= bar, (name, e_nat, e_f32, bar)
    return ratios


def _check_h_per_tile(pol, got):
    """act_fc1 on the features the kernel itself produced, against a float64 product, tile by tile:
    each 128-row tile within max(FC1_FACTOR x SGEMM's error on that tile, 2^-20 x the tile's max|h|), so
    that one wrong tile or split part cannot hide behind the others."""
    feat, h = got['feat'], got['h'].double()
    n = feat.shape[0]
    with torch.no_grad():
        want = torch.relu(feat @ pol.act_fc1.weight.double().t() + pol.act_fc1.bias.double())
    sgemm = f32_reference(lambda: torch.relu(feat.float() @ pol.act_fc1.weight.t() + pol.act_fc1.bias)).double()
    tiles = -(-n // BM)
    pad = lambda t: F.pad(t, (0, 0, 0, tiles * BM - n)).reshape(tiles, -1)
    e_nat = pad((h - want).abs()).max(1).values
    e_sg = pad((sgemm - want).abs()).max(1).values
    top = pad(want.abs()).max(1).values
    bar = torch.maximum(FC1_FACTOR * e_sg, FEAT_FLOOR * top)
    bad = torch.nonzero(e_nat > bar).flatten().tolist()
    assert not bad, [(t, float(e_nat[t]), float(e_sg[t]), float(top[t])) for t in bad[:8]]


# ---------------------------------------------------------------- 1. act_fc1's tile schedule
@pytest.mark.gpu
@pytest.mark.parametrize('case', SCHEDULE_CASES)
def test_tile_schedule_against_float64(case):
    """Every row at a batch size that puts act_fc1's work list in one regime (see schedule_sizes):
    features, h (per 128-row tile) and means against float64, and nothing written past row n."""
    sms = _sms()
    assert_schedule_coverage(sms)
    n = schedule_sizes(sms)[case]
    pol = _policy()
    with torch.no_grad():   # default-init biases are small; make every term count
        pol.act_fc1.bias.uniform_(-0.3, 0.3)
        pol.act_fea_cv2.bias.uniform_(-0.2, 0.2)
    scan, goal, speed = _inputs(n, seed=n)
    got = _native(pol, scan, goal, speed)
    assert bool((got['tail'] == SENTINEL).all())
    r64, r32 = _references(pol, scan, goal, speed)
    _check_stages(got, r64, r32)
    _check_h_per_tile(pol, got)


# ---------------------------------------------------------------- 3. the front end's distribution
FRONT_CASES = ('1', '2', '3', 'sms-1', 'sms', 'sms+1', '2sms', '3sms-1', '3sms', '3sms+1')


@pytest.mark.gpu
@pytest.mark.parametrize('case', FRONT_CASES)
def test_front_end_distribution(case):
    """The persistent front end hands pedestrians to CTAs round robin and to a CTA's 3 groups in
    turn (`my_count`): sizes around 1, 2 and 3 pedestrians per CTA.  Every pedestrian's features
    within the bar of float64."""
    sms = _sms()
    n = {'1': 1, '2': 2, '3': 3, 'sms-1': sms - 1, 'sms': sms, 'sms+1': sms + 1, '2sms': 2 * sms,
         '3sms-1': 3 * sms - 1, '3sms': 3 * sms, '3sms+1': 3 * sms + 1}[case]
    pol = _policy()
    scan, goal, speed = _inputs(n, seed=100 + n)
    got = _native(pol, scan, goal, speed)
    r64, r32 = _references(pol, scan, goal, speed)
    per_ped = (got['feat'] - r64[0]).abs().max(1).values
    bar = max(10.0 * _err(r32[0], r64[0]), FEAT_FLOOR * float(r64[0].abs().max()))
    bad = torch.nonzero(per_ped > bar).flatten().tolist()
    assert not bad, (bad[:8], float(per_ped.max()), bar)


@pytest.mark.gpu
def test_front_end_is_batch_invariant():
    """One pedestrian's feature halves are the same bits wherever it lands: alone (n = 1) and at
    several rows of the five-item batch, the last row included."""
    from nav_gym_b200.pedestrians import NativePolicy
    sms = _sms()
    big = schedule_sizes(sms)['five_items']
    pol = _policy()
    scan, goal, speed = _inputs(big, seed=11)
    nat = NativePolicy(pol, big, 'cuda:0')
    nat.mean(scan[:1].contiguous(), goal[:1].contiguous(), speed[:1].contiguous())
    torch.cuda.synchronize()
    fh1, fl1, _, _ = nat.intermediates(1)
    fh1, fl1 = fh1.clone(), fl1.clone()
    rows = [0, 1, sms - 1, sms, 3 * sms, big // 2, big - 1]
    for r in rows:
        scan[r], goal[r], speed[r] = scan[0], goal[0], speed[0]
    nat.mean(scan, goal, speed)
    torch.cuda.synchronize()
    fh, fl, _, _ = nat.intermediates(big)
    for r in rows:
        assert torch.equal(fh[r], fh1[0]) and torch.equal(fl[r], fl1[0]), r


# ---------------------------------------------------------------- 4. one workspace, many batch sizes
@pytest.mark.gpu
def test_workspace_reuse_across_batch_sizes():
    """One NativePolicy called with shrinking and growing n (rows past n in the last tile hold an
    earlier call's data) gives the same bits as a fresh NativePolicy for each call; two identical
    calls agree; n = 0 writes nothing; n > max_n raises."""
    from nav_gym_b200.pedestrians import NativePolicy
    pol = _policy()
    max_n = 40960
    nat = NativePolicy(pol, max_n, 'cuda:0')
    for i, n in enumerate((40960, 77, 40959, 1, 300, 40960)):
        scan, goal, speed = _inputs(n, seed=1000 + i)
        got = nat.mean(scan, goal, speed).clone()
        torch.cuda.synchronize()
        fh, _, h, _ = nat.intermediates(n)
        fh, h = fh.clone(), h.clone()
        fresh = NativePolicy(pol, n, 'cuda:0')
        want = fresh.mean(scan, goal, speed)
        torch.cuda.synchronize()
        wfh, _, wh, _ = fresh.intermediates(n)
        assert torch.equal(got, want) and torch.equal(fh, wfh) and torch.equal(h, wh), (i, n)
        del fresh
    again = nat.mean(scan, goal, speed)
    torch.cuda.synchronize()
    assert torch.equal(again, got)
    buf = torch.full((4, 2), SENTINEL, device='cuda')
    nat.mean(scan[:0], goal[:0], speed[:0], out=buf[:0])
    torch.cuda.synchronize()
    assert bool((buf == SENTINEL).all())
    scan, goal, speed = _inputs(max_n + 1, seed=2000)
    with pytest.raises(RuntimeError):
        nat.mean(scan, goal, speed)


# ---------------------------------------------------------------- 5. power-of-two rescaling
def _rescaled(pol, a, b, c, d):
    """The same function with every layer rescaled by powers of two that cancel through the ReLUs."""
    p = copy.deepcopy(pol)
    k = a + b + c + d
    with torch.no_grad():
        p.act_fea_cv1.weight.mul_(2.0 ** a); p.act_fea_cv1.bias.mul_(2.0 ** a)
        p.act_fea_cv2.weight.mul_(2.0 ** b); p.act_fea_cv2.bias.mul_(2.0 ** (a + b))
        p.act_fc1.weight.mul_(2.0 ** c); p.act_fc1.bias.mul_(2.0 ** (a + b + c))
        p.act_fc2.weight[:, :256].mul_(2.0 ** d); p.act_fc2.weight[:, 256:].mul_(2.0 ** k)
        p.act_fc2.bias.mul_(2.0 ** k)
        p.actor1.weight.mul_(2.0 ** -k); p.actor2.weight.mul_(2.0 ** -k)
    return p


def _raw_h(nat, n):
    """act_fc1's output as the f16 (hi, lo) pairs act_fc2 reads."""
    L = (C.c_uint64 * 6)()
    nat.lib.navgym_policy_workspace_layout(nat.max_n, L)
    w = nat._ws
    return (w[L[4]:L[4] + n * 512].view(torch.float16).reshape(n, 256).clone(),
            w[L[5]:L[5] + n * 512].view(torch.float16).reshape(n, 256).clone())


@pytest.mark.gpu
@pytest.mark.parametrize('abcd', [(9, -6, 5, -7), (-11, 8, -10, 12)])
def test_power_of_two_rescaling_is_exact(abcd):
    """Rescaling the layers by powers of two shifts every bound and scale policy_prepare_kernel
    picks by an exact power of two: feature halves, act_fc1's output halves and the means are the
    same bits, and the scales differ by exactly the expected powers."""
    a, b, c, d = abcd
    pol = _policy()
    with torch.no_grad():
        pol.act_fc1.bias.uniform_(-0.3, 0.3)
        pol.act_fea_cv2.bias.uniform_(-0.2, 0.2)
    n = 1029
    scan, goal, speed = _inputs(n, seed=5, scans=_edge_scans(pol))
    one = _native(pol, scan, goal, speed)
    two = _native(_rescaled(pol, a, b, c, d), scan, goal, speed)
    f1, f2 = one['nat'].intermediates(n), two['nat'].intermediates(n)
    assert torch.equal(f1[0], f2[0]) and torch.equal(f1[1], f2[1])
    h1, h2 = _raw_h(one['nat'], n), _raw_h(two['nat'], n)
    assert torch.equal(h1[0], h2[0]) and torch.equal(h1[1], h2[1])
    assert torch.equal(one['mean'], two['mean'])
    # scales: 0 feature, 1 act_fc1 descale, 2 conv1 output, 3 conv2 descale, 6 h, 7 act_fc2 descale
    shift = {0: -(a + b), 1: a + b + c, 2: -a, 3: a + b, 6: -(a + b + c), 7: a + b + c + d}
    s1, s2 = one['scales'].cpu().double(), two['scales'].cpu().double()
    for i, e in shift.items():
        assert float(s2[i]) == float(s1[i]) * 2.0 ** e, (i, float(s1[i]), float(s2[i]), e)


# ---------------------------------------------------------------- 6. weight regimes
def _regime(name):
    """A policy whose weights are far from PyTorch's default init in one way ('mostly_dead' gets its
    act_fc1 bias from _kill_most_of_h once the inputs are known)."""
    pol = _policy(seed=21)
    layers = [pol.act_fea_cv1, pol.act_fea_cv2, pol.act_fc1, pol.act_fc2, pol.actor1, pol.actor2]
    with torch.no_grad():
        if name == 'student_t':   # heavy tails: max / median ~ 10^3 per large tensor
            g = torch.Generator().manual_seed(3)
            for m in layers:
                std = (3.0 * m.weight[0].numel()) ** -0.5   # std of the default uniform init
                for t in (m.weight, m.bias):
                    z = torch.randn(t.shape, generator=g, dtype=torch.float64)
                    chi2 = torch.randn((2,) + tuple(t.shape), generator=g, dtype=torch.float64).pow(2).sum(0)
                    t.copy_((z / (chi2 / 2.0).sqrt() * std).float())   # Student-t, 2 degrees of freedom
        elif name in ('times_37.5', 'over_300'):
            f = 37.5 if name == 'times_37.5' else 1.0 / 300.0
            for t in pol.parameters():
                t.mul_(f)
        elif name == 'dead_channels':
            pol.act_fea_cv1.weight[5].zero_()
            pol.act_fea_cv1.bias[5] = -0.1
            pol.act_fc1.weight[17].zero_()
        elif name == 'fc1_zero':      # h = relu(fc1 bias); the weight scale hits its 2^100 clamp
            pol.act_fc1.weight.zero_()
        else:
            assert name in ('default', 'mostly_dead')
    return pol


def _kill_most_of_h(pol, scan, goal, speed):
    """Shift act_fc1's bias by each output's 95th percentile on these inputs: ~95 % of h is 0 and
    the survivors are small next to the bias, far below the bound s_h2 is chosen from."""
    r64, _ = _references(pol, scan, goal, speed)
    with torch.no_grad():
        z = r64[0] @ pol.act_fc1.weight.double().t() + pol.act_fc1.bias.double()
        pol.act_fc1.bias.sub_(torch.quantile(z, 0.95, dim=0).float())


REGIMES = ('default', 'student_t', 'times_37.5', 'over_300', 'mostly_dead', 'dead_channels', 'fc1_zero')


@pytest.mark.gpu
@pytest.mark.parametrize('regime', REGIMES)
def test_weight_regimes_against_float64(regime, record_property):
    """Features, h (also per tile) and means against float64 for weights far from init scale,
    heavy-tailed, saturating the heads, tiny, with mostly dead ReLUs, dead channels and an all-zero
    act_fc1: the scales policy_prepare_kernel picks keep float32-grade results in each."""
    n = 1029
    pol = _regime(regime)
    scan, goal, speed = _inputs(n, seed=9, scans=_edge_scans(pol))
    if regime == 'mostly_dead':
        _kill_most_of_h(pol, scan, goal, speed)
    got = _native(pol, scan, goal, speed)
    assert bool((got['tail'] == SENTINEL).all())
    r64, r32 = _references(pol, scan, goal, speed)
    if regime == 'mostly_dead':
        dead = float((r64[1] == 0).double().mean())
        assert 0.9 < dead < 0.99, dead
    if regime == 'fc1_zero':
        assert float(got['scales'][1]) * float(got['scales'][0]) == 2.0 ** -100 or float(got['scales'][1]) == 0.0
    ratios = _check_stages(got, r64, r32, record_property)
    for k, v in ratios.items():
        record_property('%s_ratio' % k, v)
    _check_h_per_tile(pol, got)


# ---------------------------------------------------------------- 7. edge scans
@pytest.mark.gpu
def test_edge_scans():
    """Clipping at exactly 0 and 6 m, out-of-range and infinite ranges, single-beam contrasts at
    every beam, and each conv1 channel driven to its bound in the first and last window (where
    the kernel's padding columns act): the tensor-core front end against float64 convolutions."""
    pol = _policy()
    with torch.no_grad():
        pol.act_fea_cv2.bias.uniform_(-0.2, 0.2)
    scan = _edge_scans(pol).contiguous()
    n = scan.shape[0]
    goal, speed = torch.zeros(n, 2, device='cuda'), torch.zeros(n, 2, device='cuda')
    got = _native(pol, scan, goal, speed)
    r64, r32 = _references(pol, scan, goal, speed)
    e_f32 = _err(r32[0], r64[0])
    bar = max(10.0 * e_f32, FEAT_FLOOR * float(r64[0].abs().max()))
    assert _err(got['feat'], r64[0]) <= bar, (_err(got['feat'], r64[0]), e_f32, bar)
