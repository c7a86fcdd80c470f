"""Robot.evaluate(environment, episodes=E): E test episodes of every env in one call.

Pinned bit for bit against the loop a user would write without it, run on a twin Environment built from the same seeds:
    for e in range(E): env.reset(); r[e] = robot.evaluate(env, max_steps, record)
results, start states, trajectories, and the environment afterwards (final states, the float64 reset state, every MT19937
word and position of the env bank, numpy's global stream for a single env), for both paths (the persistent f16 kernel and the
per-step graphs), every forward precision, streams that wrap during the E draws and every map configuration."""
import functools

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ENV_SEED = 1707366464


@functools.lru_cache(maxsize=None)
def _maps(seed=0, turn=0.05):
    """Benchmark maps with the flow angle scaled down (at most 18 degrees of turn), so that the homing actor reaches most goals."""
    import rtd3_b200
    speed, angle = rtd3_b200.synthetic_maps(seed)
    return speed, (angle * turn).astype(np.float32)


def make_env(pkg, n, maps=None, seed=ENV_SEED, **kw):
    return pkg.Environment(num_envs=n, seed=seed, maps=maps if maps is not None or "map_seeds" in kw else _maps(), **kw)


def set_actor(robot, actor):
    """'zero': residual 0, the action is state - goal (away from the goal); 'homing': residual = -2 base, so the action is
    goal - state clipped to +-5; 'random': the seeded initialisation."""
    agent = robot.td3_agent
    if actor == "random":
        return
    agent.flat(0).zero_()
    if actor == "homing":
        net = agent.actor_network
        w1 = net.layer_1.weight
        w1[0, 0], w1[1, 0], w1[2, 1], w1[3, 1] = 1.0, -1.0, 1.0, -1.0      # relu(x), relu(-x), relu(y), relu(-y)
        for k in range(2, agent.layers + 1):
            w = getattr(net, "layer_%d" % k).weight
            for j in range(4):
                w[j, j] = 1.0
        wo = net.output_layer.weight
        wo[0, 0], wo[0, 1], wo[1, 2], wo[1, 3] = -2.0, 2.0, -2.0, 2.0
    agent.sync_transposed()


def make_robot(pkg, hidden=64, layers=2, precision="f16", actor="random", seed=3):
    torch.manual_seed(1)
    goal = torch.full((4, 2), 50.0, dtype=torch.float64, device="cuda")
    robot = pkg.Robot(goal, hidden=hidden, layers=layers, seed=seed, buffer_size=10000)
    robot.td3_agent.precision = precision
    set_actor(robot, actor)
    return robot


_ROBOTS = {}


def robot_for(pkg, hidden, layers, precision, actor):
    """Evaluation leaves a Robot untouched, so one per configuration serves every test."""
    key = (hidden, layers, precision, actor)
    if key not in _ROBOTS:
        _ROBOTS[key] = make_robot(pkg, hidden, layers, precision, actor)
    return _ROBOTS[key]


def env_state(env):
    b = env._bank
    return {"state": env._state.clone(), "state64": env._state64.clone(), "mt": b.mt.clone(), "pos": b.pos.clone(),
            "has_gauss": b.has_gauss.clone(), "gauss": b.gauss.clone()}


def episodes(robot, env, E, T, record=False, persistent=True):
    robot.eval_kernel = persistent
    r = robot.evaluate(env, max_steps=T, record=record, episodes=E)
    torch.cuda.synchronize()
    return {k: v.clone() for k, v in r.items()}, env_state(env)


def loop(robot, env, E, T, record=False, persistent=True):
    """The reference form: E rounds of reset + evaluate."""
    robot.eval_kernel = persistent
    rs = []
    for _ in range(E):
        env.reset()
        start = env._state.t().clone()
        r = {k: v.clone() for k, v in robot.evaluate(env, max_steps=T, record=record).items()}
        r["start"] = start
        rs.append(r)
    torch.cuda.synchronize()
    return {k: torch.stack([r[k] for r in rs]) for k in rs[0]}, env_state(env)


def assert_same(a, b, what=""):
    assert a.keys() == b.keys(), what
    for k in a:
        assert a[k].shape == b[k].shape and a[k].dtype == b[k].dtype, (what, k)
        assert torch.equal(a[k], b[k]), (what, k)


def check_against_loop(robot, make, E, T, record=False, persistent=True, what=""):
    got, got_env = episodes(robot, make(), E, T, record, persistent)
    ref, ref_env = loop(robot, make(), E, T, record, persistent)
    n = got["success"].shape[-1]
    assert got["success"].shape == (E, n) and got["start"].shape == (E, n, 2)
    assert_same(got, ref, what)
    assert_same(got_env, ref_env, what)
    return got


# ---- the persistent path ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("hidden", [256, 64])
@pytest.mark.parametrize("n", [128, 129, 4096, 20000])
@pytest.mark.parametrize("E", [1, 2, 7, 16])
@pytest.mark.parametrize("T", [1, 17, 1000])
@pytest.mark.parametrize("actor", ["zero", "homing", "random"])
def test_persistent_episodes_equal_the_reset_loop(pkg, hidden, n, E, T, actor):
    robot = robot_for(pkg, hidden, 2, "f16", actor)
    assert robot.td3_agent._f16_ok(n)
    got = check_against_loop(robot, lambda: make_env(pkg, n), E, T, what=(hidden, n, E, T, actor))
    assert bool((got["steps"] >= 1).all() and (got["steps"] <= T).all())
    if E > 1:
        assert not torch.equal(got["start"][0], got["start"][1])          # every episode has its own start
    if actor == "homing" and T == 1000:
        assert got["success"].any() and len(torch.unique(got["steps"])) > 1


@pytest.mark.parametrize("n,E", [(4096, 7), (129, 16)])
@pytest.mark.parametrize("actor", ["homing", "random"])
def test_persistent_episodes_equal_the_per_step_path_behind_the_f16_forward(pkg, n, E, actor):
    robot = robot_for(pkg, 256, 2, "f16", actor)
    a, a_env = episodes(robot, make_env(pkg, n), E, 1000, persistent=True)
    b, b_env = episodes(robot, make_env(pkg, n), E, 1000, persistent=False)
    assert_same(a, b)
    assert_same(a_env, b_env)


# ---- the per-step path -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 127, 4096])
@pytest.mark.parametrize("E", [1, 7])
@pytest.mark.parametrize("actor", ["homing", "random"])
def test_per_step_fp32_reference_actor_equals_the_reset_loop(pkg, n, E, actor):
    robot = robot_for(pkg, 200, 3, "fp32", actor)
    check_against_loop(robot, lambda: make_env(pkg, n), E, 300, what=(n, E, actor))


@pytest.mark.parametrize("persistent", [True, False])
def test_per_step_tf32_equals_the_reset_loop(pkg, persistent):
    robot = robot_for(pkg, 128, 2, "tf32", "random")
    assert robot.td3_agent._tc_ok(4096) and not robot.td3_agent._f16_ok(4096)
    check_against_loop(robot, lambda: make_env(pkg, 4096), 5, 200, persistent=persistent)


def test_f16_below_one_tile_uses_the_fp32_forward_for_every_episode(pkg):
    """N = 100 < 128 rows: evaluate on N rows takes the fp32 forward, so the E x N = 400 rows of 4 episodes must too."""
    n, E, T = 100, 4, 300
    r16 = make_robot(pkg, 128, 2, "f16", "random")
    r32 = make_robot(pkg, 128, 2, "fp32", "random")
    assert not r16.td3_agent._f16_ok(n) and not r16.td3_agent._tc_ok(n) and r16.td3_agent._f16_ok(E * n)
    got = check_against_loop(r16, lambda: make_env(pkg, n), E, T)
    assert r16._eval_work is None                                      # the persistent kernel was not used
    b, _ = episodes(r32, make_env(pkg, n), E, T)
    assert_same(got, b)


# ---- streams that wrap during the E draws ----------------------------------------------------------------------------------
@pytest.mark.parametrize("persistent", [True, False])
def test_streams_that_wrap_at_the_first_a_middle_and_the_last_draw(pkg, persistent):
    n, E, T = 1024, 9, 200
    # a reset takes 4 words; a stream at position p wraps at draw d (0-based) when p + 4 d + 4 > 624
    wrap_at = lambda d: 621 - 4 * d
    choices = torch.tensor([wrap_at(0), wrap_at(E // 2), wrap_at(E - 1), 0, 622, 623, 624, 100, 620, wrap_at(E - 1) - 1], dtype=torch.int32)
    g = torch.Generator().manual_seed(4)
    pos = choices[torch.randint(0, len(choices), (n,), generator=g)].cuda()
    pos[:32] = wrap_at(E // 2)                                          # a warp whose lanes all wrap at one draw
    pos[32:64:2] = wrap_at(0)                                           # a warp with a wrap at the first draw on every other lane

    def make():
        env = make_env(pkg, n)
        env._bank.pos.copy_(pos)
        return env
    robot = robot_for(pkg, 128, 2, "f16", "homing")
    check_against_loop(robot, make, E, T, persistent=persistent)


# ---- map banks -------------------------------------------------------------------------------------------------------------
def _bank(K, seed=0):
    s, a = zip(*[_maps(seed + k, turn=0.05 * (k + 1)) for k in range(K)])
    return np.stack(s), np.stack(a)


@pytest.mark.parametrize("bank", ["k8_contiguous", "k8_random", "map_seeds"])
@pytest.mark.parametrize("persistent", [True, False])
def test_map_banks_equal_the_reset_loop(pkg, bank, persistent):
    n, E, T = 1000, 5, 300
    if bank == "map_seeds":
        make = lambda: make_env(pkg, n, map_seeds=[3, 17, 250, 4])
    else:
        index = torch.from_numpy(np.random.RandomState(4).randint(0, 8, n)) if bank == "k8_random" else None
        make = lambda: make_env(pkg, n, _bank(8), map_index=index)
    robot = robot_for(pkg, 128, 2, "f16", "homing" if persistent else "random")
    check_against_loop(robot, make, E, T, persistent=persistent, what=bank)


@pytest.mark.parametrize("persistent", [True, False])
def test_a_short_map_index_applies_to_every_episode(pkg, persistent):
    """An index of length m < n set through the C ABI: env i steps on map index[i % m] in every episode."""
    n, m, E, T = 1000, 37, 4, 300
    idx = torch.from_numpy(np.random.RandomState(6).randint(0, 8, m)).int().cuda()

    def short():
        env = make_env(pkg, n, _bank(8), map_index=torch.zeros(n, dtype=torch.int32))
        pkg._lib.check(pkg._lib.lib().rtd3_env_set_map_index(env._handle, pkg._lib.ptr(idx), m, pkg._lib.stream_ptr(env.device)),
                       "env_set_map_index")
        return env
    full = lambda: make_env(pkg, n, _bank(8), map_index=idx[torch.arange(n, device="cuda") % m])
    robot = robot_for(pkg, 128, 2, "f16", "homing" if persistent else "random")
    got, got_env = episodes(robot, short(), E, T, persistent=persistent)
    ref, ref_env = loop(robot, full(), E, T, persistent=persistent)
    assert_same(got, ref)
    assert_same(got_env, ref_env)


# ---- record ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("persistent", [True, False])
def test_record_equals_the_stacked_loop_trajectories(pkg, persistent):
    n, E, T = 3000, 3, 200
    robot = robot_for(pkg, 128, 2, "f16", "homing")
    got = check_against_loop(robot, lambda: make_env(pkg, n), E, T, record=True, persistent=persistent)
    traj = got["trajectory"]
    assert traj.shape == (E, T, n, 2) and traj.transpose(-1, -2).is_contiguous()
    assert got["success"].any() and (got["steps"] < T).any()


# ---- a single env on numpy's global stream ---------------------------------------------------------------------------------
@pytest.mark.parametrize("E", [1, 6])
def test_single_env_advances_numpy_global_stream_by_e_resets(pkg, E):
    robot = make_robot(pkg, 200, 3, "fp32", "random")
    out = []
    for form in ("episodes", "loop"):
        np.random.seed(11)
        env = pkg.Environment(maps=_maps())
        assert env._numpy_global
        np.random.uniform(size=150)                                     # start mid-stream: the draws cross a twist
        r, st = (episodes if form == "episodes" else loop)(robot, env, E, 300)
        out.append((r, st, np.random.get_state()))
    (a, a_env, a_np), (b, b_env, b_np) = out
    assert_same(a, b)
    assert_same(a_env, b_env)
    assert a_np[0] == b_np[0] and np.array_equal(a_np[1], b_np[1]) and a_np[2:] == b_np[2:]


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


def snapshot(robot, tr):
    out = _tensors(robot, "robot.", {}, skip=("_eval_graphs", "_eval_work"))
    _tensors(robot.memory, "memory.", out)
    _tensors(robot._bank, "bank.", out)
    _tensors(robot.td3_agent, "td3.", out, skip=("params_t", "params_u", "params_h", "_graphs", "_scratch"))
    _tensors(tr, "trainer.", out, skip=("_graph", "_graph_k"))
    out["counts"] = (robot.num_updates, len(robot.memory), tr.ticks)
    return out


@pytest.mark.parametrize("precision", ["fp32", "f16"])
def test_episodes_leave_the_robot_and_training_untouched(pkg, precision):
    env = make_env(pkg, 32)
    env.reset()
    torch.manual_seed(1)
    robot = pkg.Robot(env.goal_state, hidden=128, layers=2, seed=3, buffer_size=20000)
    robot.td3_agent.precision = precision
    robot.episodes_per_update = 8
    tr = pkg.BatchedTrainer(env, robot, noise="philox", fused=True, graph=True, check_interval=8)
    held_out = make_env(pkg, 2048, _maps(9), seed=77)
    for block in range(4):
        tr.run(8)
        before = snapshot(robot, tr)
        for persistent in (True, False):
            robot.eval_kernel = persistent
            robot.evaluate(held_out, max_steps=40, episodes=3)
            robot.evaluate(held_out, max_steps=7, record=True, episodes=2)
        torch.cuda.synchronize()
        after = snapshot(robot, tr)
        assert before.keys() == after.keys()
        for k in before:
            assert (torch.equal(before[k], after[k]) if isinstance(before[k], torch.Tensor) else before[k] == after[k]), k
    assert robot.num_updates > 0

