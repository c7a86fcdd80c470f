"""Map bank: K maps per Environment and a map index per env (rtd3_env_set_maps / rtd3_env_set_map_index).  The reference for
every bank result is the single-map kernels run on each map's sub-batch: the envs of map k gathered into an
`Environment(maps=map k)` and stepped with the same actions.  Those kernels are pinned to repeated `step` bit for bit
(test_rollout_halo_gpu.py, test_env_gpu.py), so the bank must match them bit for bit - in every rollout variant, in the
uniform-warp (staged table) and the mixed-warp (per-lane global table) regime."""
import numpy as np
import pytest
import torch

from oracle import env_oracle as eo
from test_rollout_halo_gpu import diagonal_map, edge_workload, put_nonfinite

pytestmark = pytest.mark.gpu

W = 100


def nonfinite_map():
    """Dead (non-finite) cells next to cells that fit the halo border."""
    speed, angle = diagonal_map(1.0)
    speed[10:20, :] = np.nan
    angle[:, 50:60] = np.inf
    return speed, angle


def bank_maps():
    """Map 0 fits (synthetic), 1 fits and reaches the border cells, 2 does not fit (speed 2), 3 has non-finite cells."""
    return [eo.synthetic_maps(0), diagonal_map(1.0), diagonal_map(2.0), nonfinite_map()]


def stack(maps):
    return np.stack([m[0] for m in maps]), np.stack([m[1] for m in maps])


def assignment(kind, n, K, seed=0):
    rs = np.random.RandomState(seed + n)
    if kind == "contiguous":
        return (np.arange(n) * K // n).astype(np.int32)
    if kind == "warp_random":                                    # one random map per aligned block of 32 envs
        return np.repeat(rs.randint(0, K, (n + 31) // 32), 32)[:n].astype(np.int32)
    if kind == "per_env":
        return rs.randint(0, K, n).astype(np.int32)
    if kind == "last":
        return np.full(n, K - 1, np.int32)
    raise ValueError(kind)


def workload(n, T, seed):
    start, planes = edge_workload(n, T, seed)
    if n >= 32:
        put_nonfinite(planes, n, T)
    else:
        for t, axis, lane in ((0, 0, 0), (5, 1, n - 1), (16, 0, n // 2), (31, 1, 0)):
            if t < T:
                planes[t, axis, lane] = np.nan if t % 2 else np.inf
    return start, planes


def reference_rollout(pkg, maps, index, start, planes):
    """Per map k: the envs with index == k as their own single-map Environment."""
    T, n = planes.shape[0], start.shape[0]
    traj = np.empty((T, 2, n), np.float32)
    final = np.empty((n, 2), np.float32)
    for k in np.unique(index):
        sel = np.nonzero(index == k)[0]
        env = pkg.Environment(num_envs=len(sel), seed=3, maps=maps[k])
        env._state.copy_(torch.from_numpy(np.ascontiguousarray(start[sel].T)).cuda())
        p = torch.from_numpy(np.ascontiguousarray(planes[:, :, sel])).cuda()
        traj[:, :, sel] = env.rollout(p.permute(0, 2, 1)).permute(0, 2, 1).cpu().numpy()
        final[sel] = env._state.t().cpu().numpy()
    return traj, final


def bank_rollout(env, start, planes):
    env._state.copy_(torch.from_numpy(np.ascontiguousarray(start.T)).cuda())
    p = torch.from_numpy(planes).cuda()
    traj = env.rollout(p.permute(0, 2, 1)).permute(0, 2, 1).cpu().numpy()
    return traj, env._state.t().cpu().numpy()


def check_rollout(pkg, maps, index, n, T, seed, env=None):
    start, planes = workload(n, T, seed)
    if env is None:
        env = pkg.Environment(num_envs=n, seed=3, maps=stack(maps), map_index=torch.from_numpy(index).cuda())
    got = bank_rollout(env, start, planes)
    want = reference_rollout(pkg, maps, index, start, planes)
    for g, w, what in zip(got, want, ("trajectory", "final state")):
        bad = np.nonzero(g != w)
        assert bad[0].size == 0, "%s differs, first at %s" % (what, [b[:3].tolist() for b in bad])
    return env


# pair kernel, one pair per CTA: 32, 100, 4096; two pairs per CTA: 6000; TMA shallow: 65536; cp.async kernel: 1, 31, 4097.
# Every env on map K-1 ("last"): one size per variant.
ROLLOUT_CASES = [(n, kind) for n in (32, 100, 4096, 6000, 65536, 1, 31, 4097) for kind in ("contiguous", "warp_random", "per_env")]
ROLLOUT_CASES += [(n, "last") for n in (100, 6000, 65536, 31)]


@pytest.mark.parametrize("n,kind", ROLLOUT_CASES)
def test_bank_rollout_equals_single_map_sub_batches(pkg, n, kind):
    T = 40 if n >= 65536 else 97
    maps = bank_maps()
    check_rollout(pkg, maps, assignment(kind, n, len(maps)), n, T, seed=n)


@pytest.mark.parametrize("kind", ["contiguous", "per_env"])
def test_bank_rollout_single_warp_tma_kernel(pkg, kind):
    maps = bank_maps()
    pkg._lib.lib().rtd3_env_force_plain_rollout(2)
    try:
        check_rollout(pkg, maps, assignment(kind, 4096, len(maps)), 4096, 97, seed=5)
    finally:
        pkg._lib.lib().rtd3_env_force_plain_rollout(0)


@pytest.mark.parametrize("n", [4096, 6000, 4097])
def test_bank_rollout_warps_mixing_fit_nofit_and_nonfinite_maps(pkg, n):
    """Warp 0 alternates a fitting map with the one that does not fit, warp 1 a border-reaching map with the non-finite one;
    the CTA's first env is on map 0, so warp 1 is mixed without containing the staged map at all."""
    maps = bank_maps()
    index = (np.arange(n) * 4 // n).astype(np.int32)
    index[0:32] = np.where(np.arange(32) % 2 == 0, 0, 2)
    index[32:64] = np.where(np.arange(32) % 3 == 0, 1, 3)
    index[64:96] = 2
    check_rollout(pkg, maps, index, n, 1000 if n == 4096 else 97, seed=21)


def test_bank_rollout_host(pkg):
    """rollout_host replays cached graphs: an index change in place, an index of another map and a bank that reallocates."""
    n, T = 4096, 200
    maps = bank_maps()
    start, planes = workload(n, T, seed=17)
    idx = assignment("warp_random", n, 4)
    env = pkg.Environment(num_envs=n, seed=3, maps=stack(maps), map_index=torch.from_numpy(idx).cuda())
    h_act = torch.from_numpy(planes).pin_memory()

    def run_and_check(maps, idx):
        env._state.copy_(torch.from_numpy(np.ascontiguousarray(start.T)).cuda())
        out = env.rollout_host(h_act).numpy()
        traj, final = reference_rollout(pkg, maps, idx, start, planes)
        assert np.array_equal(out, traj)
        assert np.array_equal(env._state.t().cpu().numpy(), final)

    run_and_check(maps, idx)
    idx = assignment("per_env", n, 4)
    env.set_map_index(idx)
    run_and_check(maps, idx)
    maps = maps + [eo.synthetic_maps(k) for k in (1, 2, 3, 4)]   # K 4 -> 8 reallocates the bank
    idx = assignment("contiguous", n, 8)
    env.set_maps(*stack(maps), index=idx)
    run_and_check(maps, idx)


# ---- step / dynamics --------------------------------------------------------------------------------------------------------------
def _step_inputs(n, seed):
    rs = np.random.RandomState(seed)
    state = rs.uniform(0, 100, (n, 2)).astype(np.float32)
    state[:8] = np.array([[0, 0], [98.9999, 99.99999], [99.5, 0.5], [50, 99]], np.float32).repeat(2, axis=0)
    act = rs.uniform(-7.5, 7.5, (n, 2)).astype(np.float32)
    return state, act


@pytest.mark.parametrize("variant", [0, 1, 2])
@pytest.mark.parametrize("n", [5003, 300000])
def test_bank_step_and_dynamics(pkg, n, variant):
    """Step (every variant: SMEM falls back to the read-only path with a bank) and dynamics, bank against per-map sub-batches
    bit for bit and against the oracle per map to 1e-5.  Dynamics over 2n rows: row j uses env j % n's map."""
    maps = bank_maps()
    idx = assignment("per_env", n, 4, seed=1)
    env = pkg.Environment(num_envs=n, seed=3, maps=stack(maps), map_index=idx)
    env.step_variant = variant
    state, act = _step_inputs(n, seed=n)
    act_nan = act.copy()
    act_nan[::97, 0] = np.nan
    env.robot_state = torch.from_numpy(state).cuda()
    got_step = env.step(torch.from_numpy(act_nan).cuda()).cpu().numpy()
    rows_s = np.concatenate([state, state[::-1]])
    rows_a = np.concatenate([act, act[::-1]])
    got_dyn = env.dynamics(torch.from_numpy(rows_s).cuda(), torch.from_numpy(rows_a).cuda()).cpu().numpy()
    row_map = np.concatenate([idx, idx])
    for k in range(len(maps)):
        sel = np.nonzero(idx == k)[0]
        ref = pkg.Environment(num_envs=len(sel), seed=3, maps=maps[k])
        ref.step_variant = variant
        ref.robot_state = torch.from_numpy(state[sel]).cuda()
        want = ref.step(torch.from_numpy(act_nan[sel]).cuda()).cpu().numpy()
        assert np.array_equal(got_step[sel], want), (k, variant)
        rsel = np.nonzero(row_map == k)[0]
        want_d = ref.dynamics(torch.from_numpy(rows_s[rsel]).cuda(), torch.from_numpy(rows_a[rsel]).cuda()).cpu().numpy()
        assert np.array_equal(got_dyn[rsel], want_d, equal_nan=True), (k, variant)
        if np.isfinite(maps[k][0]).all() and np.isfinite(maps[k][1]).all():    # the reference raises on non-finite cells
            o = eo.step_batch(maps[k][0], maps[k][1], state[sel].astype(np.float64), act[sel].astype(np.float64))
            ok = ~np.isnan(act_nan[sel, 0])
            np.testing.assert_allclose(got_step[sel][ok], o[ok], rtol=1e-5, atol=1e-5)
            od = eo.dynamics_batch(maps[k][0], maps[k][1], rows_s[rsel].astype(np.float64), rows_a[rsel].astype(np.float64))
            np.testing.assert_allclose(got_dyn[rsel], od, rtol=1e-5, atol=1e-5)


# ---- index handling ---------------------------------------------------------------------------------------------------------------
def test_set_map_index_switches_between_calls_and_modes(pkg):
    n, T = 4096, 97
    maps = bank_maps()
    a = assignment("contiguous", n, 4)
    env = check_rollout(pkg, maps, a, n, T, seed=31)
    assert env.num_maps == 4 and torch.equal(env.map_index.cpu(), torch.from_numpy(a))
    b = assignment("per_env", n, 4)
    env.set_map_index(torch.from_numpy(b).long().cuda())
    check_rollout(pkg, maps, b, n, T, seed=32, env=env)
    env.set_maps(*maps[2])                                       # bank -> single map
    assert env.map_index is None and env.num_maps == 1 and env.dynamics_speed.shape == (W, W)
    check_rollout(pkg, [maps[2]], np.zeros(n, np.int32), n, T, seed=33, env=env)
    env.set_maps(*stack(maps), index=b)                          # and back
    assert env.dynamics_speed.shape == (4, W, W)
    check_rollout(pkg, maps, b, n, T, seed=34, env=env)
    env.set_map_index(None)                                      # no index: every env on map 0
    check_rollout(pkg, maps, np.zeros(n, np.int32), n, T, seed=35, env=env)


def test_captured_graph_follows_index_contents(pkg):
    n, T = 4096, 97
    maps = bank_maps()
    a, b = assignment("contiguous", n, 4), assignment("per_env", n, 4)
    env = pkg.Environment(num_envs=n, seed=3, maps=stack(maps), map_index=a)
    start, planes = workload(n, T, seed=41)
    p = torch.from_numpy(planes).cuda().permute(0, 2, 1)
    s0 = torch.from_numpy(np.ascontiguousarray(start.T)).cuda()
    env._state.copy_(s0)
    env.rollout(p)                                               # warm-up outside the capture
    g = torch.cuda.CUDAGraph()
    with pkg._lib.capture(g):
        traj = env.rollout(p)
    for idx in (a, b):
        env.set_map_index(idx)                                   # same length: written in place
        env._state.copy_(s0)
        g.replay()
        torch.cuda.synchronize()
        want, final = reference_rollout(pkg, maps, idx, start, planes)
        assert np.array_equal(traj.permute(0, 2, 1).cpu().numpy(), want)
        assert np.array_equal(env._state.t().cpu().numpy(), final)


def test_index_input_checks(pkg):
    n = 64
    maps = bank_maps()
    env = pkg.Environment(num_envs=n, seed=3, maps=stack(maps))
    assert torch.equal(env.map_index.cpu(), torch.arange(n, dtype=torch.int32) * 4 // n)   # default: contiguous blocks
    before = env.map_index
    for bad in (np.full(n, 4), np.full(n, -1), np.zeros(n - 1, np.int64), np.zeros((n, 1), np.int64), np.zeros(n, np.float32),
                torch.zeros(n, dtype=torch.bool)):
        with pytest.raises(ValueError):
            env.set_map_index(bad)
    with pytest.raises(ValueError):
        env.set_maps(*stack(maps), index=np.full(n, 4))
    with pytest.raises(ValueError):
        pkg.Environment(num_envs=n, seed=3, maps=stack(maps), map_index=np.zeros(n + 1, np.int32))
    assert torch.equal(env.map_index, before) and env.num_maps == 4
    with pytest.raises(ValueError):
        env.set_maps(np.zeros((2, W, W), np.float32), np.zeros((3, W, W), np.float32))


def test_k1_bank_equals_set_map(pkg):
    n, T = 4096, 97
    maps = bank_maps()
    s, a = maps[1]
    env = pkg.Environment(num_envs=n, seed=3, maps=(s[None], a[None]))
    assert env.map_index is None and env.num_maps == 1 and env.dynamics_speed.shape == (W, W)
    check_rollout(pkg, [maps[1]], np.zeros(n, np.int32), n, T, seed=51, env=env)
    env.set_maps(s[None], a[None], index=np.zeros(n, np.int32))  # the bank kernels with K = 1
    check_rollout(pkg, [maps[1]], np.zeros(n, np.int32), n, T, seed=52, env=env)
    state, act = _step_inputs(n, seed=53)
    ref = pkg.Environment(num_envs=n, seed=3, maps=maps[1])
    for e in (env, ref):
        e.robot_state = torch.from_numpy(state).cuda()
    assert torch.equal(env.step(torch.from_numpy(act).cuda()), ref.step(torch.from_numpy(act).cuda()))


# ---- fused tick ---------------------------------------------------------------------------------------------------------------------
def _tick_build(pkg, n, idx, fused, noise, graph=False, check_interval=1, hidden=64):
    from test_tick_gpu import _demo_path
    env = pkg.Environment(num_envs=n, seed=5, maps=stack(bank_maps()), map_index=idx)
    robot = pkg.Robot(env.goal_state, hidden=hidden, layers=2, seed=3, buffer_size=max(40000, 140 * n))
    robot.td3_agent.actor_network.load_flat(np.random.RandomState(0).normal(0, 0.05, robot.td3_agent.actor_network.count()).astype(np.float32))
    robot.episodes_per_update = 10 ** 9
    robot.demo_grid_min_points = 64
    robot.set_demonstration_states(_demo_path(400))
    tr = pkg.BatchedTrainer(env, robot, noise=noise, graph=graph, check_interval=check_interval, fused=fused)
    return env, robot, tr


def _same(snaps):
    (a, rows_a, tab_a) = snaps[0]
    for (b, rows_b, tab_b) in snaps[1:]:
        for k in a:
            assert torch.equal(a[k], b[k]), k
        assert rows_a == rows_b and rows_a > 0 and np.array_equal(tab_a, tab_b)


def test_bank_fused_tick_equals_hook_by_hook(pkg):
    from test_tick_gpu import _snapshot
    n = 2048
    idx = assignment("per_env", n, 4)
    snaps = []
    for fused in (False, True):
        env, robot, tr = _tick_build(pkg, n, idx, fused, "mt19937")
        for _ in range(60):
            tr.tick()
        snaps.append(_snapshot(env, robot, tr))
    _same(snaps)


def test_bank_tick_graph_and_multi_tick_kernel_equal_eager_ticks(pkg):
    """f16 forward, Philox noise: eager fused ticks, the 8-tick graph and rtd3_tick_run_f16 over 64 ticks."""
    from test_tick_gpu import _snapshot
    n = 2048
    idx = assignment("warp_random", n, 4)
    snaps = []
    for graph, multi in ((False, False), (True, False), (False, True)):
        env, robot, tr = _tick_build(pkg, n, idx, True, "philox", graph=graph, check_interval=8)
        robot.td3_agent.precision = "f16"
        tr.multi_tick_kernel = multi
        assert tr._multi_tick_ok() == multi
        tr.run(64)
        snaps.append(_snapshot(env, robot, tr))
        if graph:
            assert tr._graph_k is not None
    _same(snaps)


def test_bank_tick_graph_recaptures_after_set_maps(pkg):
    """A captured tick holds the bank and index addresses: a set_maps that reallocates the bank must force a recapture."""
    from test_tick_gpu import _snapshot
    n = 512
    idx = assignment("per_env", n, 4)
    more = stack(bank_maps() + [eo.synthetic_maps(k) for k in (5, 6, 7, 8)])
    idx8 = assignment("per_env", n, 8, seed=9)
    snaps = []
    for graph in (False, True):
        env, robot, tr = _tick_build(pkg, n, idx, True, "philox", graph=graph, check_interval=4)
        tr.multi_tick_kernel = False
        tr.run(24)
        env.set_maps(*more, index=idx8)
        tr.run(24)
        snaps.append(_snapshot(env, robot, tr))
    _same(snaps)


# ---- batched planner ----------------------------------------------------------------------------------------------------------------
def test_bank_planner_equals_single_map_envs(pkg):
    """The planner's P*n virtual envs v = p*n + i use index[v % n] = env i's map: per map, the envs of that map plan exactly
    what a single-map Environment with the same seed and N plans for them."""
    n = 96
    maps = bank_maps()
    idx = assignment("per_env", n, 4, seed=2)
    env = pkg.Environment(num_envs=n, seed=11, maps=stack(maps), map_index=idx)
    states, actions = env.get_demonstration()
    for k in range(len(maps)):
        ref = pkg.Environment(num_envs=n, seed=11, maps=maps[k])
        rs, ra = ref.get_demonstration()
        sel = torch.from_numpy(np.nonzero(idx == k)[0]).cuda()
        assert torch.equal(states[sel], rs[sel]) and torch.equal(actions[sel], ra[sel]), k
