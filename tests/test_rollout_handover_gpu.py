"""The warp-pair rollout kernel hands each 32-step chunk over between its chain warps and the helper warp (rtd3_env.cu): the chain
warp probes the next chunk's barriers and careful flag before the end of a chunk, and between two fast chunks it carries the table
address of the next step across the boundary instead of taking it from the state.  These cases put every transition at every
place a chunk boundary can sit - fast -> careful -> fast, a careful first chunk, NaN / inf at the first and the last step of a
chunk, a wall reached at the last step of a chunk, start states in cell 99, ragged last chunks, maps that do not fit, uniform and
mixed bank warps, both sides of the one / two tiles per CTA switch, all three trajectory destinations, and long back-to-back
sequences with launch overlap and from a replayed graph.  The rollout must equal repeated `step` and the cp.async rollout kernel
bit for bit."""
import numpy as np
import pytest
import torch

from oracle import env_oracle as eo

pytestmark = pytest.mark.gpu

U = 32                   # kPairU of rtd3_env.cu: steps per chunk
W = 100


@pytest.fixture(scope="module")
def switch(pkg):
    """The last batch with one tile per CTA and the first with two (a multiple of 4: the pair kernel's TMA tiles need one)."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    return {"switch_lo": 32 * sms, "switch_hi": 32 * sms + 4}


@pytest.fixture
def plain_kernel(pkg):
    """Runs the body with every rollout on the cp.async kernel."""
    L = pkg._lib.lib()

    class Ctx:
        def __enter__(self):
            L.rtd3_env_force_plain_rollout(1)

        def __exit__(self, *exc):
            L.rtd3_env_force_plain_rollout(0)
    return Ctx


def diagonal_map(speed=1.0):
    """rot = pi/4 everywhere: a saturated action moves a state 5*sqrt(2)*speed along each axis per step (fits at speed 1)."""
    return np.full((W, W), speed, np.float32), np.full((W, W), 0.125, np.float32)


def axis_map(speed=1.5):
    """rot = 0 everywhere: an action moves a state by speed * action along its own axis, up to 7.5 cells at speed 1.5 (fits)."""
    return np.full((W, W), speed, np.float32), np.zeros((W, W), np.float32)


def workload(n, T, seed, lo=0.0, hi=99.99999):
    rs = np.random.RandomState(seed)
    start = rs.uniform(lo, hi, (n, 2)).astype(np.float32)
    planes = rs.uniform(-7.5, 7.5, (T, 2, n)).astype(np.float32)
    return start, planes


def env_of(pkg, n, maps, index=None):
    idx = None if index is None else torch.from_numpy(index.astype(np.int32)).cuda()
    return pkg.Environment(num_envs=n, seed=3, maps=maps, map_index=idx)


def launch(pkg, env, act, traj, n, T):
    lib = pkg._lib
    lib.check(lib.lib().rtd3_env_rollout(env._handle, lib.ptr(env._state[0]), lib.ptr(env._state[1]), lib.ptr(act),
                                         lib.ptr(traj), n, T, lib.stream_ptr(torch.device("cuda", 0))), "env_rollout")


def rollout(pkg, env, start, planes, traj):
    """rtd3_env_rollout with the trajectory in device memory, in pinned host memory or not recorded; returns (traj, state)."""
    T, _, n = planes.shape
    env.robot_state = torch.from_numpy(start).cuda()
    p = torch.from_numpy(planes).cuda()
    out = None
    if traj == "device":
        out = torch.empty((T, 2, n), dtype=torch.float32, device="cuda")
    elif traj == "host":
        out = torch.full((T, 2, n), -1.0, dtype=torch.float32).pin_memory()
    launch(pkg, env, p, out, n, T)
    torch.cuda.synchronize()
    return (out.cuda() if out is not None else None), env._state.clone()


def same(a, b):
    return bool(((a == b) | (torch.isnan(a) & torch.isnan(b))).all())


def check(pkg, plain_kernel, start, planes, maps, index=None, traj="device"):
    """The pair kernel against repeated `step` and against the cp.async kernel, trajectory and final state."""
    n = start.shape[0]
    got, state = rollout(pkg, env_of(pkg, n, maps, index), start, planes, traj)
    ref = env_of(pkg, n, maps, index)
    ref.robot_state = torch.from_numpy(start).cuda()
    p = torch.from_numpy(planes).cuda()
    steps = []
    for t in range(p.shape[0]):
        ref.step(p[t].t())
        steps.append(ref._state.clone())
    steps = torch.stack(steps)
    assert torch.equal(state, ref._state)
    if got is not None:
        bad = ~((got == steps) | (torch.isnan(got) & torch.isnan(steps)))
        assert not bool(bad.any()), "first mismatch (t, axis, env) %s" % (torch.nonzero(bad)[:3].tolist(),)
    with plain_kernel():
        plain, plain_state = rollout(pkg, env_of(pkg, n, maps, index), start, planes, "device")
    assert torch.equal(state, plain_state)
    if got is not None:
        assert same(got, plain)
    return got


@pytest.mark.parametrize("T", [1, 31, 32, 33, 63, 64, 65, 97, 1000, 1024])
@pytest.mark.parametrize("n", [36, 4096, "switch_lo", "switch_hi"])
def test_chunk_counts(pkg, plain_kernel, switch, n, T):
    """Ragged last chunks, exactly one chunk, one step past a chunk, long runs of carried chunks."""
    n = switch.get(n, n)
    check(pkg, plain_kernel, *workload(n, T, seed=n + T), maps=eo.synthetic_maps(0))


@pytest.mark.parametrize("where", ["middle_chunk", "first_chunk", "first_step", "last_step"])
@pytest.mark.parametrize("bad", [np.nan, np.inf])
@pytest.mark.parametrize("n", [4096, "switch_hi"])
def test_nonfinite_actions(pkg, plain_kernel, switch, n, bad, where):
    """One env's non-finite actions make its tile's chunk careful: fast -> careful -> fast around it, the next fast chunk
    addressed from the state again.  Only in the middle chunk, only in the first, or only at the first or last step of a chunk
    (chunk 1 and chunk 2)."""
    n = switch.get(n, n)
    T = 130
    start, planes = workload(n, T, seed=21)
    lanes = [0, 17, n - 1]                                      # chain warps 0 and 1 of the first tile, the last env
    if where == "middle_chunk":
        for t in range(U, 2 * U, 7):
            planes[t, 0, lanes] = bad
    elif where == "first_chunk":
        planes[0:U, 1, lanes] = bad
    elif where == "first_step":
        planes[U, 0, lanes] = bad
        planes[2 * U, 1, lanes] = bad
    else:
        planes[U - 1, 1, lanes] = bad
        planes[2 * U - 1, 0, lanes] = bad
    check(pkg, plain_kernel, start, planes, maps=diagonal_map())


@pytest.mark.parametrize("n", [36, 4096, "switch_hi"])
def test_start_states_in_cell_99(pkg, plain_kernel, switch, n):
    """States in [99, 100) enter the first chunk, and - kept there through a careful first chunk - the next fast one."""
    n = switch.get(n, n)
    T = 97
    start, planes = workload(n, T, seed=9, lo=99.0, hi=99.99999)
    planes[0:U, :, 1::5] = np.nan
    check(pkg, plain_kernel, start, planes, maps=diagonal_map())


@pytest.mark.parametrize("n", [36, 4096, "switch_hi"])
def test_wall_reached_at_last_step_of_a_chunk(pkg, plain_kernel, switch, n):
    """Zero actions hold the states near a wall; a saturated push at the last step of a chunk takes the unclipped state up to
    7.5 cells past the wall, so the next chunk's carried first address is a border cell of the halo table."""
    n = switch.get(n, n)
    T = 3 * U + 5
    rs = np.random.RandomState(31)
    start = np.where(rs.uniform(size=(n, 2)) < 0.5, rs.uniform(98.0, 98.9999, (n, 2)), rs.uniform(0.0, 1.0, (n, 2)))
    start = start.astype(np.float32)
    planes = np.zeros((T, 2, n), np.float32)
    push = np.where(start > 50, 7.5, -7.5).astype(np.float32).T  # towards the nearer wall on each axis
    for t in (U - 1, 2 * U - 1):
        planes[t] = push
    planes[3 * U:] = rs.uniform(-7.5, 7.5, (T - 3 * U, 2, n))
    traj = check(pkg, plain_kernel, start, planes, maps=axis_map())
    hi_wall = float(np.float32(98.9999))
    for t in (U - 1, 2 * U - 1):
        assert bool((traj[t] == hi_wall).any()) and bool((traj[t] == 0).any())


@pytest.mark.parametrize("n", [4096, "switch_hi"])
def test_map_that_does_not_fit(pkg, plain_kernel, switch, n):
    n = switch.get(n, n)
    start, planes = workload(n, 97, seed=41)
    check(pkg, plain_kernel, start, planes, maps=diagonal_map(2.0))


@pytest.mark.parametrize("kind", ["uniform", "mixed"])
@pytest.mark.parametrize("n", [4096, "switch_hi"])
def test_bank(pkg, plain_kernel, switch, n, kind):
    """Uniform warps (a map per 16 envs: each chain warp on one map) run the fast path on the staged map next to warps on other
    maps; mixed warps step every lane on its own map."""
    n = switch.get(n, n)
    maps = [eo.synthetic_maps(0), eo.synthetic_maps(1), diagonal_map(1.0)]
    bank = np.stack([m[0] for m in maps]), np.stack([m[1] for m in maps])
    ids = np.arange(n)
    index = (ids // 16) % 3 if kind == "uniform" else (ids // 3) % 3
    start, planes = workload(n, 97, seed=43)
    planes[40, 0, 5] = np.nan
    check(pkg, plain_kernel, start, planes, maps=bank, index=index)


@pytest.mark.parametrize("traj", [None, "device", "host"])
@pytest.mark.parametrize("n", [36, 4096, "switch_hi"])
def test_trajectory_destinations(pkg, plain_kernel, switch, n, traj):
    n = switch.get(n, n)
    start, planes = workload(n, 129, seed=47)
    planes[70, 1, n // 2] = np.inf
    check(pkg, plain_kernel, start, planes, maps=eo.synthetic_maps(0), traj=traj)


def back_to_back(pkg, n, T, launches, graph):
    """`launches` rollouts on one stream with no synchronisation in between, each continuing from the state the one before left;
    eagerly or captured into a CUDA graph and replayed.  Returns every trajectory and the final state."""
    env = env_of(pkg, n, eo.synthetic_maps(0))
    gen = torch.Generator(device="cuda").manual_seed(53)
    acts = torch.rand((launches, T, 2, n), device="cuda", generator=gen) * 15 - 7.5
    acts[launches // 2, T // 2, 0, 7] = float("nan")
    env.robot_state = torch.from_numpy(workload(n, 1, seed=59)[0]).cuda()
    trajs = torch.empty((launches, T, 2, n), device="cuda")
    if not graph:
        for k in range(launches):
            launch(pkg, env, acts[k], trajs[k], n, T)
    else:
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        g = torch.cuda.CUDAGraph()
        with torch.cuda.stream(s), torch.cuda.graph(g, stream=s):
            for k in range(launches):
                launch(pkg, env, acts[k], trajs[k], n, T)
        torch.cuda.current_stream().wait_stream(s)
        g.replay()
    torch.cuda.synchronize()
    return trajs, env._state.clone()


@pytest.mark.parametrize("graph", [False, True])
@pytest.mark.parametrize("n,T", [(4096, 65), (4096, 96), ("switch_hi", 33)])
def test_back_to_back_launches_with_overlap(pkg, plain_kernel, switch, n, T, graph):
    n = switch.get(n, n)
    L = pkg._lib.lib()
    L.rtd3_env_set_launch_overlap(1)
    trajs, state = back_to_back(pkg, n, T, 64, graph)
    with plain_kernel():
        ref_trajs, ref_state = back_to_back(pkg, n, T, 64, False)
    assert same(trajs, ref_trajs)
    assert torch.equal(state, ref_state)
