"""Device Perlin maps (rtd3_perlin_maps, perlin_maps_device, Environment.set_perlin_maps / map_seeds) against the host's
perlin_maps: the fields before normalisation and `angle` bit for bit; `speed` bit for bit against the host restatement that
rounds a float64 exp once to float32, and within a few ulp of perlin_maps itself, whose float32 exp depends on the host CPU."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

W = 100
SEEDS = [0, 1, 7, 1707366464, 2 ** 32 - 1, 2 ** 32, 2 ** 40 + 7, 2 ** 63 - 1]
SPEED_ULP = 4   # numpy's float32 exp against the rounded-once float64 exp; the most measured on an AVX-512 host


def host_fields(pkg, seed):
    """perlin_maps's float32 cells before normalisation: speed n(5) + 0.5 n(10) + 0.25 n(20), angle n(5)."""
    P = pkg.environment._PerlinNoise
    n1, n2, n3 = P(5, seed), P(10, seed), P(20, seed)
    speed = np.zeros((W, W), np.float32)
    angle = np.zeros((W, W), np.float32)
    for col in range(W):
        for row in range(W):
            q = [col / W, row / W]
            a = n1(q)
            speed[col, row] = a + 0.5 * n2(q) + 0.25 * n3(q)
            angle[col, row] = a
    return speed, angle


def normalise(cells):
    return (cells - np.min(cells)) / (np.max(cells) - np.min(cells))


def speed_rounded_once(cells):
    """perlin_maps's speed with exp evaluated in float64 and rounded once to float32 (numpy's float32 order otherwise)."""
    x = -10 * (normalise(cells) - 0.5)
    e = np.exp(x.astype(np.float64)).astype(np.float32)
    return (1 / (1 + e)).astype(np.float32)


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def ulps(a, b):
    return np.abs(bits(a).astype(np.int64) - bits(b).astype(np.int64))


def device_maps(pkg, seeds, raw=False):
    L = pkg._lib.lib()
    L.rtd3_perlin_set_raw_fields(1 if raw else 0)
    try:
        speed, angle = pkg.perlin_maps_device(seeds)
        torch.cuda.synchronize()
    finally:
        L.rtd3_perlin_set_raw_fields(0)
    return speed.cpu().numpy(), angle.cpu().numpy()


def check_against_host(pkg, seed, speed, angle, raw=None):
    """Returns the largest ulp distance of `speed` from perlin_maps."""
    fs, fa = host_fields(pkg, seed)
    if raw is not None:
        assert np.array_equal(bits(raw[0]), bits(fs)), seed
        assert np.array_equal(bits(raw[1]), bits(fa)), seed
    ref_speed, ref_angle = pkg.environment.perlin_maps(seed)
    assert np.array_equal(bits(angle), bits(ref_angle)), seed
    assert np.array_equal(bits(angle), bits(normalise(fa))), seed
    assert np.array_equal(bits(speed), bits(speed_rounded_once(fs))), seed
    worst = int(ulps(speed, ref_speed).max())
    assert worst <= SPEED_ULP, (seed, worst)
    return worst


# ---- exactness ----------------------------------------------------------------------------------------------------------------------
def test_fields_and_maps_match_the_host(pkg):
    raw_s, raw_a = device_maps(pkg, SEEDS, raw=True)
    speed, angle = device_maps(pkg, SEEDS)
    worst = {}
    for k, seed in enumerate(SEEDS):
        worst[seed] = check_against_host(pkg, seed, speed[k], angle[k], raw=(raw_s[k], raw_a[k]))
    print("speed: largest distance from perlin_maps in ulp, per seed:", worst)


def test_a_map_depends_only_on_its_seed(pkg):
    s = 2 ** 40 + 7
    rs = np.random.RandomState(3)
    others = rs.randint(0, 2 ** 63, size=36, dtype=np.int64)
    alone = device_maps(pkg, [s])
    among = device_maps(pkg, np.concatenate([others[:17], [s], others[17:]]))
    again = device_maps(pkg, torch.from_numpy(np.concatenate([others[:17], [s], others[17:]])).cuda())
    for q in range(2):
        assert np.array_equal(bits(alone[q][0]), bits(among[q][17]))
        assert np.array_equal(bits(among[q]), bits(again[q]))


def test_many_seeds(pkg):
    K = 4096
    seeds = np.random.RandomState(11).randint(0, 2 ** 63, size=K, dtype=np.int64)
    speed, angle = device_maps(pkg, seeds)
    assert speed.shape == (K, W, W) and angle.shape == (K, W, W)
    assert np.isfinite(speed).all() and np.isfinite(angle).all()
    assert (angle.min(axis=(1, 2)) == 0).all() and (angle.max(axis=(1, 2)) == 1).all()
    assert (speed > 0).all() and (speed < 1).all()
    for k in (0, 1234, 2047, K - 1):
        check_against_host(pkg, int(seeds[k]), speed[k], angle[k])


# ---- Environment ---------------------------------------------------------------------------------------------------------------------
def _trainer(pkg, env):
    from test_tick_gpu import _demo_path
    robot = pkg.Robot(env.goal_state, hidden=64, layers=2, seed=3, buffer_size=max(40000, 140 * env.num_envs))
    robot.td3_agent.actor_network.load_flat(np.random.RandomState(0).normal(0, 0.05, robot.td3_agent.actor_network.count()).astype(np.float32))
    robot.episodes_per_update = 10 ** 9
    robot.demo_grid_min_points = 64
    robot.set_demonstration_states(_demo_path(400))
    return robot, pkg.BatchedTrainer(env, robot, noise="mt19937", fused=True)


def _workload(n, T, seed):
    rs = np.random.RandomState(seed)
    start = rs.uniform(0, 99, (2, n)).astype(np.float32)
    planes = rs.uniform(-7.5, 7.5, (T, 2, n)).astype(np.float32)
    return torch.from_numpy(start).cuda(), torch.from_numpy(planes).cuda()


def _same_dynamics(pkg, env, ref, seed):
    n = env.num_envs
    start, planes = _workload(n, 97, seed)
    for e in (env, ref):
        e._state.copy_(start)
    assert torch.equal(env.step(planes[0].t()), ref.step(planes[0].t()))
    trajs = [e.rollout(planes.permute(0, 2, 1)) for e in (env, ref)]
    assert torch.equal(trajs[0], trajs[1]) and torch.equal(env._state, ref._state)


@pytest.mark.parametrize("seeds", [[5, 2 ** 33 + 1, 77, 1707366464, 9, 2 ** 62, 3, 123456789], [1707366464]])
def test_environment_map_seeds_equal_the_same_maps_given(pkg, seeds):
    from test_tick_gpu import _snapshot
    n, K = 4096, len(seeds)
    speed, angle = pkg.perlin_maps_device(seeds)
    host = (speed.cpu().numpy(), angle.cpu().numpy())
    env = pkg.Environment(num_envs=n, seed=5, map_seeds=np.array(seeds, np.int64))
    ref = pkg.Environment(num_envs=n, seed=5, maps=host)
    assert env.num_maps == ref.num_maps == K
    assert torch.equal(env.map_seeds, torch.tensor(seeds, dtype=torch.int64)) and ref.map_seeds is None
    if K == 1:
        assert env.map_index is None and ref.map_index is None and env.dynamics_speed.shape == (W, W)
    else:
        assert torch.equal(env.map_index, ref.map_index)
    for a, b in ((env.dynamics_speed, host[0]), (env.dynamics_angle, host[1])):
        assert isinstance(a, np.ndarray) and np.array_equal(bits(a), bits(b[0] if K == 1 else b))
    _same_dynamics(pkg, env, ref, seed=21)

    snaps = []
    for e in (env, ref):
        robot, tr = _trainer(pkg, e)
        for _ in range(60):
            tr.tick()
        snaps.append(_snapshot(e, robot, tr))
    (a, rows_a, tab_a), (b, rows_b, tab_b) = snaps
    for k in a:
        assert torch.equal(a[k], b[k]), k
    assert rows_a == rows_b and rows_a > 0 and np.array_equal(tab_a, tab_b)

    env.set_maps(*host)
    assert env.map_seeds is None and env.num_maps == K


def test_set_perlin_maps_switches_banks(pkg):
    n = 4096
    env = pkg.Environment(num_envs=n, seed=5, map_seeds=[1, 2, 3])
    idx = np.random.RandomState(0).randint(0, 5, n)
    env.set_perlin_maps(torch.tensor([4, 5, 6, 7, 8]).cuda(), index=idx)   # a larger bank, a given index
    ref = pkg.Environment(num_envs=n, seed=5, maps=tuple(t.cpu().numpy() for t in pkg.perlin_maps_device([4, 5, 6, 7, 8])),
                          map_index=idx)
    assert env.map_seeds.tolist() == [4, 5, 6, 7, 8] and env.num_maps == 5
    assert torch.equal(env.map_index.cpu(), torch.from_numpy(idx).int())
    _same_dynamics(pkg, env, ref, seed=22)
    env.set_dynamics()
    assert env.map_seeds is None and env.num_maps == 1


# ---- graph capture -------------------------------------------------------------------------------------------------------------------
def test_captured_generation_follows_the_seeds_tensor(pkg):
    """rtd3_perlin_maps + rtd3_env_set_maps captured once; new seeds written into the same tensor take effect at replay."""
    lib = pkg._lib
    L = lib.lib()
    n, K = 4096, 6
    first, second = [11, 12, 13, 14, 15, 16], [2 ** 50 + 3, 0, 99, 1707366464, 2 ** 63 - 1, 5]
    env = pkg.Environment(num_envs=n, seed=5, map_seeds=first)           # allocates a bank of K maps
    seeds = torch.tensor(first, dtype=torch.int64, device="cuda")
    speed = torch.empty((K, W, W), dtype=torch.float32, device="cuda")
    angle = torch.empty_like(speed)
    g = torch.cuda.CUDAGraph()
    with lib.capture(g):
        lib.check(L.rtd3_perlin_maps(lib.ptr(seeds), K, lib.ptr(speed), lib.ptr(angle), lib.stream_ptr()), "perlin_maps")
        lib.check(L.rtd3_env_set_maps(env._handle, lib.ptr(speed), lib.ptr(angle), K, lib.stream_ptr()), "env_set_maps")
    seeds.copy_(torch.tensor(second, dtype=torch.int64))
    g.replay()
    torch.cuda.synchronize()
    want = pkg.perlin_maps_device(second)
    assert torch.equal(speed, want[0]) and torch.equal(angle, want[1])
    ref = pkg.Environment(num_envs=n, seed=5, map_seeds=second)
    _same_dynamics(pkg, env, ref, seed=23)


# ---- argument checks -----------------------------------------------------------------------------------------------------------------
def test_bad_seeds_raise(pkg):
    n = 64
    env = pkg.Environment(num_envs=n, seed=5, map_seeds=[1, 2])
    before = env.dynamics_speed.copy()
    bad_inputs = ([-1], [3, -2], [1.5], np.array([1.0, 2.0]), [[1, 2]], np.zeros((2, 2), np.int64), [], torch.zeros(0, dtype=torch.int64).cuda(),
                  torch.tensor([-4]).cuda(), torch.tensor([0.5]).cuda(), np.zeros(65537, np.int64))
    for bad in bad_inputs:
        with pytest.raises(ValueError):
            pkg.perlin_maps_device(bad)
        with pytest.raises(ValueError):
            env.set_perlin_maps(bad)
        with pytest.raises(ValueError):
            pkg.Environment(num_envs=n, seed=5, map_seeds=bad)
    with pytest.raises(ValueError):
        env.set_perlin_maps([1, 2, 3], index=np.full(n, 3))
    with pytest.raises(ValueError):
        pkg.Environment(num_envs=n, seed=5, maps=pkg.synthetic_maps(0), map_seeds=[1])
    assert env.map_seeds.tolist() == [1, 2] and env.num_maps == 2 and np.array_equal(env.dynamics_speed, before)
