"""The warp-pair rollout kernel addresses the table of step t+1 from the unclipped state of step t, through a table with an
8-cell border (rtd3_env.cu, kHalo).  These cases drive states onto both walls and to the farthest border cells, start from
states in [99, 100) (cell 99, which only a state can reach), put NaN / inf actions inside chunks and at chunk boundaries,
and use maps that do not fit the border (the state-addressed path): the rollout must equal repeated `step` bit for bit."""
import numpy as np
import pytest
import torch

from oracle import env_oracle as eo

pytestmark = pytest.mark.gpu

W = 100
EDGE_STARTS = np.array([0.0, 98.9999, 98.99995, 99.0, 99.5, 99.99999], np.float32)


def diagonal_map(speed=1.0):
    """Uniform map with angle 1/8: rot = pi/4, |cos|+|sin| = sqrt(2), so saturated actions move a state 5*sqrt(2)*speed
    along one axis per step - at speed 1 from 98.9999 to 106.07 (border cell 106) and from 0 to -7.07 (border cell -8)."""
    return np.full((W, W), speed, np.float32), np.full((W, W), 0.125, np.float32)


def edge_workload(n, T, seed):
    """Start states on and beyond the walls and actions that stay saturated at +-7.5 (clipped to +-5) for long stretches."""
    rs = np.random.RandomState(seed)
    start = rs.uniform(0, 100, (n, 2)).astype(np.float32)
    start[: n // 2, 0] = EDGE_STARTS[np.arange(n // 2) % len(EDGE_STARTS)]
    start[: n // 2, 1] = EDGE_STARTS[(np.arange(n // 2) // len(EDGE_STARTS)) % len(EDGE_STARTS)]
    start = np.minimum(start, np.float32(99.99999))
    hold = 40                                                   # steps per saturated stretch
    signs = rs.choice([-7.5, 7.5], (T // hold + 1, 2, n)).astype(np.float32)
    planes = np.repeat(signs, hold, axis=0)[:T]
    free = rs.uniform(0, 1, (T // hold + 1, 1, n)) < 0.25        # a quarter of the stretches: uniform actions instead
    free = np.repeat(free, hold, axis=0)[:T] & np.ones((1, 2, 1), bool)
    planes[free] = rs.uniform(-7.5, 7.5, free.sum()).astype(np.float32)
    return start, planes


def put_nonfinite(planes, n, T):
    """NaN / inf actions: whole first chunks for some lanes (they keep a start state in [99, 100) into a fast chunk), and single
    ones inside chunks and on both sides of chunk boundaries for others."""
    last_warp = (n // 32 - 1) * 32
    for lane, steps in ((1, 32), (2, 40), (3, 64), (last_warp + 5, 32)):
        if lane < n:
            planes[:min(steps, T), :, lane] = np.nan
    for t, axis, lane in ((5, 0, n // 2), (16, 1, 0), (31, 0, n - 1), (32, 1, n - 1), (63, 0, n // 3), (64, 1, n // 3),
                          (97, 0, 7), (500, 1, n // 2 + 1), (999, 0, n - 2)):
        if t < T:
            planes[t, axis, lane] = np.nan if t % 2 else np.inf


def rollout_vs_steps(pkg, maps, start, planes, env=None, env_ref=None):
    n = start.shape[0]
    env = env or pkg.Environment(num_envs=n, seed=3, maps=maps)
    env_ref = env_ref or pkg.Environment(num_envs=n, seed=3, maps=maps)
    s0 = torch.from_numpy(start).cuda()
    env.robot_state = s0
    env_ref.robot_state = s0
    p = torch.from_numpy(planes).cuda()
    traj = env.rollout(p.permute(0, 2, 1))
    steps = torch.stack([env_ref.step(p[t].t()).clone() for t in range(p.shape[0])])
    bad = (traj != steps) & ~(torch.isnan(traj) & torch.isnan(steps))
    assert not bool(bad.any()), "first mismatch (t, env, axis) %s" % (torch.nonzero(bad)[:3].tolist(),)
    assert torch.equal(env.robot_state, env_ref.robot_state)
    return traj


@pytest.mark.parametrize("T", [1, 31, 32, 33, 97, 1000])
@pytest.mark.parametrize("n", [32, 4096, 8192])
def test_rollout_saturated_edges_equal_steps(pkg, n, T):
    start, planes = edge_workload(n, T, seed=n + T)
    put_nonfinite(planes, n, T)
    traj = rollout_vs_steps(pkg, diagonal_map(), start, planes)
    if T >= 97:                                                 # the workload does reach both walls on both axes
        lo = float(np.float32(98.9999))
        for axis in (0, 1):
            assert bool((traj[..., axis] == 0).any()) and bool((traj[..., axis] == lo).any())


@pytest.mark.parametrize("n,T", [(4096, 97), (8192, 33)])
def test_rollout_synthetic_map_equal_steps(pkg, n, T):
    start, planes = edge_workload(n, T, seed=7)
    put_nonfinite(planes, n, T)
    rollout_vs_steps(pkg, eo.synthetic_maps(0), start, planes)


@pytest.mark.parametrize("n", [4096, 8192])
def test_rollout_maps_that_do_not_fit(pkg, n):
    """Speed 2 moves a state up to 14.1 per step, beyond the border; a map with NaN / inf cells has dead cells (which fit)
    next to fast ones."""
    T = 97
    start, planes = edge_workload(n, T, seed=11)
    rollout_vs_steps(pkg, diagonal_map(2.0), start, planes)
    speed, angle = diagonal_map(1.0)
    speed[10:20, :] = np.nan
    angle[:, 50:60] = np.inf
    speed[70:80, 70:80] = 1.6                                   # 5 * 1.6 * sqrt(2) = 11.3: does not fit either
    rollout_vs_steps(pkg, (speed, angle), start, planes)
    speed[70:80, 70:80] = 1.0                                   # only non-finite cells left: fits
    rollout_vs_steps(pkg, (speed, angle), start, planes)


def test_set_map_switches_fit(pkg):
    """One Environment, maps switched fit -> no fit -> fit: the fit flag follows every set_maps."""
    n, T = 4096, 97
    start, planes = edge_workload(n, T, seed=13)
    put_nonfinite(planes, n, T)
    env = pkg.Environment(num_envs=n, seed=3, maps=diagonal_map(1.0))
    ref = pkg.Environment(num_envs=n, seed=3, maps=diagonal_map(1.0))
    for speed in (1.0, 2.0, 1.0):
        maps = diagonal_map(speed)
        env.set_maps(*maps)
        ref.set_maps(*maps)
        rollout_vs_steps(pkg, maps, start, planes, env, ref)


def test_rollout_host_equals_rollout_4096x1000(pkg):
    """The host-buffer rollout runs the same kernel in graph-captured time slices."""
    n, T = 4096, 1000
    maps = diagonal_map(1.0)
    start, planes = edge_workload(n, T, seed=17)
    put_nonfinite(planes, n, T)
    env = pkg.Environment(num_envs=n, seed=3, maps=maps)
    ref = pkg.Environment(num_envs=n, seed=3, maps=maps)
    env.robot_state = torch.from_numpy(start).cuda()
    ref.robot_state = torch.from_numpy(start).cuda()
    h_act = torch.from_numpy(planes).pin_memory()
    out = env.rollout_host(h_act)
    traj = ref.rollout(h_act.cuda())
    assert torch.equal(out.cuda().permute(0, 2, 1), traj)
    assert torch.equal(env.robot_state, ref.robot_state)
