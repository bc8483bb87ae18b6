"""Adapters that drive the CUDA path (through the C ABI) with the golden_util.replay protocol."""
import numpy as np
import torch

import golden_util as gu
from nav_gym_b200.batched_env import BatchedNavGym


def f32_reference(fn):
    """Run fn with TF32 off everywhere (cuDNN / cuBLAS would round operands to TF32)."""
    old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad():
            return fn()
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old


class CudaStepper(object):
    def __init__(self, maps, map_id, start, goal, theta, max_disc=0, max_seg=0, early_stop=True,
                 cell_rule='numpy1', **kw):
        B = len(map_id)
        self.env = BatchedNavGym(B, maps, device='cuda:0', map_id=map_id, max_disc=max_disc,
                                 max_seg=max_seg, early_stop=early_stop, cell_rule=cell_rule,
                                 record_hits=True, **kw)
        self.env.set_state(start, goal, theta)
        self.early_stop = early_stop

    def reset_obs(self, discs=None, ndisc=None, segs=None, nseg=None, noise=None):
        if noise is None:
            noise = np.zeros((self.env.B, 2, gu.NB), np.float32)
        self.env.reset(discs, ndisc, segs, nseg, noise)
        torch.cuda.synchronize()

    def step(self, actions, discs=None, ndisc=None, segs=None, nseg=None, noise=None):
        if noise is None:
            noise = np.zeros((self.env.B, 2, gu.NB), np.float32)
        self.env.step(actions, discs, ndisc, segs, nseg, noise)
        torch.cuda.synchronize()

    def __getattr__(self, k):
        if k in ('obs', 'tail64', 'reward', 'done', 'is_success', 'is_crash', 'distance', 'hits',
                 'state', 'steps'):
            return getattr(self.env, k).cpu().numpy()
        raise AttributeError(k)


def golden_stepper(G, early_stop, cell_rule='numpy2'):
    md, ms = gu.geom_dims(G)
    S = int(G['num_scan_stack']) if 'num_scan_stack' in G else 1
    return CudaStepper([gu.map_info(G)], np.zeros(1, np.int32), G['start'][None, :2], G['goal'][None],
                       G['start'][2:3], max_disc=md, max_seg=ms, early_stop=early_stop,
                       cell_rule=cell_rule, num_scan_stack=S,
                       min_turning_radius=float(G['min_turning_radius']) if 'min_turning_radius' in G else 0.0,
                       **gu.env_kwargs(G))
