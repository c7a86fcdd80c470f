"""Robot.evaluate: the reference's test phase (robot-learning.py:104-117) for every env of an Environment, on the GPU.

Pinned bit for bit against the host driver loop (`DriverLoop` in testing mode, one env), against the scheduler's test branch of
the fused tick kernels (batched, fp32 and f16), between its two paths (the persistent f16 kernel and the per-step graphs), and
between every env of a map bank and the same env evaluated on its map alone."""
import types

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ENV_SEED = 1707366464


def _maps(pkg, seed=0, turn=0.05):
    """Benchmark maps with the flow angle scaled down (at most 18 degrees of turn), so that the homing actor reaches most goals."""
    speed, angle = pkg.synthetic_maps(seed)
    return speed, (angle * turn).astype(np.float32)


def make_env(pkg, n, maps=None, seed=ENV_SEED, **kw):
    env = pkg.Environment(num_envs=n, seed=seed, maps=maps, **kw)
    env.reset()
    return env


def set_actor(robot, actor):
    """'zero': residual 0, the action is state - goal (away from the goal); 'homing': residual = -2 base, so the action is
    goal - state clipped to +-5; 'random': the seeded initialisation."""
    agent = robot.td3_agent
    H, L = agent.hidden, agent.layers
    if actor == "random":
        return
    flat = agent.flat(0)
    flat.zero_()
    if actor == "homing":
        net = agent.actor_network
        w1 = net.layer_1.weight
        w1[0, 0], w1[1, 0], w1[2, 1], w1[3, 1] = 1.0, -1.0, 1.0, -1.0      # relu(x), relu(-x), relu(y), relu(-y)
        for k in range(2, L + 1):
            w = getattr(net, "layer_%d" % k).weight
            for j in range(4):
                w[j, j] = 1.0
        wo = net.output_layer.weight
        wo[0, 0], wo[0, 1], wo[1, 2], wo[1, 3] = -2.0, 2.0, -2.0, 2.0
    agent.sync_transposed()


def make_robot(pkg, n=4, hidden=64, layers=2, precision="f16", actor="random", seed=3):
    torch.manual_seed(1)
    goal = torch.full((n, 2), 50.0, dtype=torch.float64, device="cuda")
    robot = pkg.Robot(goal, hidden=hidden, layers=layers, seed=seed, buffer_size=max(10000, n))
    robot.td3_agent.precision = precision
    set_actor(robot, actor)
    return robot


def clone_env(pkg, env, maps=None, **kw):
    """A second environment with the same goals, regions and current states (and the same maps unless `maps` is given)."""
    e = pkg.Environment(num_envs=env.num_envs, seed=ENV_SEED, maps=maps if maps is not None else (env._speed_dev.cpu(), env._angle_dev.cpu()), **kw)
    assert torch.equal(e._goal, env._goal)
    if maps is None and env.map_index is not None:
        e.set_map_index(env.map_index)
    e._state.copy_(env._state)
    return e


def run(robot, env, T=None, record=False, persistent=True):
    robot.eval_kernel = persistent
    r = robot.evaluate(env, max_steps=T, record=record)
    torch.cuda.synchronize()
    r = {k: v.clone() for k, v in r.items()}
    r["state"] = env._state.clone()
    return r


def assert_same(a, b, what=""):
    assert a.keys() == b.keys()
    for k in a:
        assert torch.equal(a[k], b[k]), (what, k)


# ---- against the reference's test branch --------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", [1707366464, 11, 29])
def test_single_env_equals_the_driver_loop_in_testing_mode(pkg, env_golden, seed):
    """N = 1, the reference's 3 x 200 fp32 actor: success, test ticks, best distance and final state as the host driver loop."""
    maps = (env_golden["speed"], env_golden["angle"])
    loop = pkg.DriverLoop.from_seed(seed, maps=maps)
    loop.mode = "testing"
    np.random.seed(seed)
    env = pkg.Environment(maps=maps)
    env.reset()
    assert np.array_equal(env.goal_state, loop.environment.goal_state)
    torch.manual_seed(5)
    robot = pkg.Robot(env.goal_state)
    robot.td3_agent.params.copy_(loop.robot.td3_agent.params)
    robot.td3_agent.sync_transposed()
    assert (robot.td3_agent.hidden, robot.td3_agent.layers, robot.td3_agent.precision) == (200, 3, "fp32")
    loop.run()
    r = robot.evaluate(env)
    assert bool(r["success"][0]) == loop.success
    assert int(r["steps"][0]) == loop.test_ticks
    assert float(r["best_distance"][0]) == loop.test_best_distance
    assert np.array_equal(env.robot_state, loop.environment.robot_state)


def _scheduler_twin(pkg, maps, n, T, precision, hidden, actor, form):
    env = make_env(pkg, n, maps)
    torch.manual_seed(1)
    robot = pkg.Robot(env.goal_state, hidden=hidden, layers=2, seed=3, buffer_size=max(20000, 8 * n))
    robot.td3_agent.precision = precision
    robot.episodes_per_update = 1 << 30
    set_actor(robot, actor)
    K = 8
    tr = pkg.BatchedTrainer(env, robot, noise="philox", fused=True, scheduler=True, graph=form == "multi", check_interval=K if form == "multi" else 1)
    tr.multi_tick_kernel = form == "multi"
    start = env._state.clone()                                       # the trainer's constructor has reset the envs
    tr.mode.fill_(1)
    tr.test_timeout_ticks = T
    if form == "multi":
        assert tr._multi_tick_ok()
        tr.run(T)
    else:
        for _ in range(T):
            tr.tick()
    assert tr.all_finished()
    return env, robot, tr, start


@pytest.mark.parametrize("precision,form", [("fp32", "eager"), ("f16", "eager"), ("f16", "multi")])
@pytest.mark.parametrize("actor", ["random", "homing"])
def test_batched_equals_the_scheduler_test_branch(pkg, precision, form, actor):
    n, T = 512, 96
    maps = _maps(pkg)
    env_t, robot_t, tr, start = _scheduler_twin(pkg, maps, n, T, precision, 128, actor, form)
    env = make_env(pkg, n, maps)
    env._state.copy_(start)
    robot = make_robot(pkg, hidden=128, precision=precision, actor=actor)
    robot.td3_agent.params.copy_(robot_t.td3_agent.params)
    robot.td3_agent.sync_transposed()
    assert robot.td3_agent._f16_ok(n) == (precision == "f16")
    r = run(robot, env, T)
    assert torch.equal(r["success"], tr.test_success.bool())
    assert torch.equal(r["steps"], tr.test_ticks)
    assert torch.equal(r["best_distance"], tr.test_best_distance)
    assert torch.equal(r["state"], env_t._state)


# ---- the two paths ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [128, 129, 4096, 20000, 65536])
@pytest.mark.parametrize("T", [1, 17, 1000])
@pytest.mark.parametrize("actor", ["zero", "homing", "random"])
def test_persistent_kernel_equals_per_step_path(pkg, n, T, actor):
    maps = _maps(pkg)
    robot = make_robot(pkg, hidden=256, actor=actor)
    env = make_env(pkg, n, maps)
    twin = clone_env(pkg, env)
    a = run(robot, env, T, persistent=True)
    assert robot._eval_work is not None
    b = run(robot, twin, T, persistent=False)
    assert_same(a, b, (n, T, actor))
    stopped_early = (a["steps"] < T)
    assert torch.equal(stopped_early, a["success"] & (a["steps"] < T))
    assert bool((a["steps"] >= 1).all() and (a["steps"] <= T).all())
    if actor == "homing" and T == 1000:
        assert a["success"].any() and len(torch.unique(a["steps"])) > 1     # tiles finish at different times


@pytest.mark.parametrize("n", [1, 127])
def test_below_one_tile_f16_evaluates_with_the_fp32_forward(pkg, n):
    maps = _maps(pkg)
    env = make_env(pkg, n, maps)
    twin = clone_env(pkg, env)
    r16 = make_robot(pkg, precision="f16", actor="random")
    r32 = make_robot(pkg, precision="fp32", actor="random")
    assert not r16.td3_agent._f16_ok(n)
    a = run(r16, env, 300)
    assert r16._eval_work is None                                     # the persistent kernel was not used
    b = run(r32, twin, 300)
    assert_same(a, b)


# ---- map banks -------------------------------------------------------------------------------------------------------------
def _bank(pkg, K, seed=0):
    s, a = zip(*[_maps(pkg, seed + k, turn=0.05 * (k + 1)) for k in range(K)])
    return np.stack(s), np.stack(a)


@pytest.mark.parametrize("bank", ["k8_contiguous", "k8_random", "k1_bank", "map_seeds"])
@pytest.mark.parametrize("persistent", [True, False])
def test_every_env_of_a_bank_equals_its_map_alone(pkg, bank, persistent):
    n, T = 1000, 400
    robot = make_robot(pkg, hidden=128, actor="homing" if persistent else "random")
    if bank == "map_seeds":
        env = make_env(pkg, n, map_seeds=[3, 17, 250, 4])
        speed, angle = env._speed_dev.cpu().numpy(), env._angle_dev.cpu().numpy()
    else:
        K = 1 if bank == "k1_bank" else 8
        speed, angle = _bank(pkg, K)
        index = None
        if bank == "k8_random":
            index = torch.from_numpy(np.random.RandomState(4).randint(0, K, n))
        env = make_env(pkg, n, (speed, angle), map_index=index)
    index = env.map_index.cpu().numpy() if env.map_index is not None else np.zeros(n, np.int64)
    start = env._state.clone()
    r = run(robot, env, T, persistent=persistent)
    for k in range(speed.shape[0]):
        alone = make_env(pkg, n, (speed[k], angle[k]))
        alone._state.copy_(start)
        ra = run(robot, alone, T, persistent=persistent)
        sel = torch.from_numpy(index == k).cuda()
        for key in r:
            got = r[key][..., sel]
            assert torch.equal(got, ra[key][..., sel]), (bank, k, key)


# ---- record ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("persistent", [True, False])
def test_record(pkg, persistent):
    n, T = 3000, 200
    maps = _maps(pkg)
    robot = make_robot(pkg, hidden=128, actor="homing")
    env = make_env(pkg, n, maps)
    start = env._state.clone()
    twin = clone_env(pkg, env)
    a = run(robot, env, T, record=True, persistent=persistent)
    b = run(robot, twin, T, record=False, persistent=persistent)
    traj = a.pop("trajectory")
    assert traj.shape == (T, n, 2) and traj.permute(0, 2, 1).is_contiguous()
    assert_same(a, b)
    assert torch.equal(traj[-1].t(), a["state"])
    steps = a["steps"].long()
    assert a["success"].any() and (steps < T).any()
    rows = torch.arange(T, device="cuda")[:, None]
    final = a["state"].t()[None].expand(T, n, 2)
    after = (rows >= steps[None] - 1)
    assert torch.equal(traj[after], final[after])                    # from the stop on: the final state
    for t in (1, 7, 30, 150):                                        # row t-1 = the state after t steps
        e = make_env(pkg, n, maps)
        e._state.copy_(start)
        rt = run(robot, e, t, persistent=persistent)
        assert torch.equal(traj[t - 1].t(), rt["state"]), t


# ---- the robot is untouched ------------------------------------------------------------------------------------------------
def _tensors(obj, prefix, out, skip=()):
    for k, v in vars(obj).items():
        if k in skip:
            continue
        if isinstance(v, torch.Tensor):
            out[prefix + k] = v.clone()
        elif isinstance(v, dict):
            for kk, vv in v.items():
                if isinstance(vv, torch.Tensor):
                    out["%s%s.%s" % (prefix, k, kk)] = vv.clone()
    return out


def snapshot(robot, tr=None):
    out = _tensors(robot, "robot.", {}, skip=("_eval_graphs", "_eval_work"))
    _tensors(robot.memory, "memory.", out)
    _tensors(robot._bank, "bank.", out)
    _tensors(robot.td3_agent, "td3.", out, skip=("params_t", "params_u", "params_h", "_graphs", "_scratch", "_coop_scratch"))
    if tr is not None:
        _tensors(tr, "trainer.", out, skip=("_graph", "_graph_k"))
    out["counts"] = (robot.num_updates, len(robot.memory), tr.ticks if tr is not None else 0)
    return out


def assert_snapshots_equal(a, b):
    assert a.keys() == b.keys()
    for k in a:
        if isinstance(a[k], torch.Tensor):
            assert torch.equal(a[k], b[k]), k
        else:
            assert a[k] == b[k], k


def _trainer(pkg, n, maps, precision):
    env = make_env(pkg, n, maps)
    torch.manual_seed(1)
    robot = pkg.Robot(env.goal_state, hidden=128, layers=2, seed=3, buffer_size=20000)
    robot.td3_agent.precision = precision
    robot.episodes_per_update = 8
    tr = pkg.BatchedTrainer(env, robot, noise="philox", fused=True, graph=True, check_interval=8)
    return env, robot, tr


@pytest.mark.parametrize("precision", ["fp32", "f16"])
def test_evaluation_leaves_the_robot_and_training_untouched(pkg, precision):
    maps = _maps(pkg)
    n = 32                                  # one warp: the replay rows land in one order in both runs (one ring atomic per tick)
    runs = []
    for with_eval in (False, True):
        env, robot, tr = _trainer(pkg, n, maps, precision)
        held_out = make_env(pkg, 2048, _maps(pkg, 9), seed=77)
        for block in range(16):
            tr.run(8)
            if with_eval:
                before = snapshot(robot, tr)
                for persistent in (True, False):
                    robot.eval_kernel = persistent
                    held_out.reset()
                    robot.evaluate(held_out, max_steps=40)
                    robot.evaluate(held_out, max_steps=7, record=True)
                torch.cuda.synchronize()
                assert_snapshots_equal(before, snapshot(robot, tr))
        assert robot.num_updates > 0
        runs.append((snapshot(robot, tr), env._state.clone()))
    assert_snapshots_equal(runs[0][0], runs[1][0])
    assert torch.equal(runs[0][1], runs[1][1])


@pytest.mark.parametrize("m", [1024, 65536])
def test_robot_and_environment_sizes_may_differ(pkg, m):
    robot = make_robot(pkg, n=4096, hidden=128, actor="homing")
    env = make_env(pkg, m, _maps(pkg))
    twin = clone_env(pkg, env)
    a = run(robot, env, 300, persistent=True)
    b = run(robot, twin, 300, persistent=False)
    assert_same(a, b)
    assert a["success"].shape == (m,)


# ---- staleness -------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["fp32", "f16"])
def test_results_follow_maps_index_and_weights(pkg, precision):
    n, T = 600, 120
    maps0, maps1 = _maps(pkg, 0), _maps(pkg, 1)
    robot = make_robot(pkg, hidden=128, precision=precision, actor="homing")
    for persistent in (True, False):
        env = make_env(pkg, n, maps0)
        start = env._state.clone()

        def again(e):
            e._state.copy_(start)
            return run(robot, e, T, persistent=persistent)

        again(env)
        env.set_maps(*maps1)                                         # graph cache: the bank moved or was rebuilt
        got = again(env)
        assert_same(got, again(make_env(pkg, n, maps1)))
        bank = tuple(np.stack([a, b]) for a, b in zip(maps0, maps1))
        env.set_maps(*bank, index=torch.zeros(n, dtype=torch.int32))
        again(env)
        idx = torch.from_numpy(np.random.RandomState(2).randint(0, 2, n))
        env.set_map_index(idx)                                       # same index length: only the contents changed
        got = again(env)
        assert_same(got, again(make_env(pkg, n, bank, map_index=idx)))
    # a learner update between two evaluations
    rows = 2000
    rs = np.random.RandomState(0)
    cu = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).cuda()
    robot.memory.push(cu(rs.uniform(0, 99, (rows, 2))), cu(rs.uniform(-5, 5, (rows, 2))), cu(rs.normal(size=rows)),
                      cu(rs.uniform(0, 99, (rows, 2))), torch.zeros(rows, dtype=torch.bool, device="cuda"))
    env = make_env(pkg, n, maps0)
    start = env._state.clone()
    for persistent in (True, False):
        env._state.copy_(start)
        first = run(robot, env, T, persistent=persistent)
    robot.td3_agent.actor_lr = 1e-2                                  # a step large enough to move the evaluation
    robot.td3_agent.td3_update(robot.memory)
    fresh = make_robot(pkg, hidden=128, precision=precision)
    fresh.td3_agent.params.copy_(robot.td3_agent.params)
    fresh.td3_agent.sync_transposed()
    for persistent in (True, False):
        env._state.copy_(start)
        got = run(robot, env, T, persistent=persistent)
        env._state.copy_(start)
        assert_same(got, run(fresh, env, T, persistent=persistent))
    assert not all(torch.equal(first[k], got[k]) for k in ("best_distance", "state"))


# ---- argument errors -------------------------------------------------------------------------------------------------------
def test_argument_errors(pkg):
    robot = make_robot(pkg)
    env = make_env(pkg, 8, _maps(pkg))
    for bad in (0, -1, 1.5, True, "10", 1 << 30):
        with pytest.raises(ValueError):
            robot.evaluate(env, max_steps=bad)
    with pytest.raises(ValueError):
        robot.evaluate(types.SimpleNamespace(device=torch.device("cpu"), num_envs=8))
    if torch.cuda.device_count() > 1:
        with torch.cuda.device(1):
            other = make_env(pkg, 8, _maps(pkg), device="cuda:1")
        with pytest.raises(ValueError):
            robot.evaluate(other)
