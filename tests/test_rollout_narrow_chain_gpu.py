"""The warp-pair rollout kernel steps each 32-env tile with several narrow chain warps of kChainLanes envs each (rtd3_env.cu).
These cases put the edges of a tile, of a chain warp and of the one-tile / two-tiles-per-CTA switch at every place a batch can
put them, NaN / inf actions and map changes inside one chain warp, and both trajectory destinations the kernel writes (none,
pinned host memory).  The rollout must equal repeated `step` and the cp.async rollout kernel bit for bit."""
import numpy as np
import pytest
import torch

from oracle import env_oracle as eo

pytestmark = pytest.mark.gpu

CHAIN_LANES = 16         # kChainLanes of rtd3_env.cu: envs per chain warp


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def workload(n, T, seed, lo=0.0, hi=99.99999):
    rs = np.random.RandomState(seed)
    start = rs.uniform(lo, hi, (n, 2)).astype(np.float32)
    planes = rs.uniform(-7.5, 7.5, (T, 2, n)).astype(np.float32)
    return start, planes


def bank(index):
    maps = [eo.synthetic_maps(0), eo.synthetic_maps(1), (np.full((100, 100), 1.0, np.float32), np.full((100, 100), 0.125, np.float32))]
    return (np.stack([m[0] for m in maps]), np.stack([m[1] for m in maps])), torch.from_numpy(index.astype(np.int32)).cuda()


def env_of(pkg, n, maps, index):
    return pkg.Environment(num_envs=n, seed=3, maps=maps, map_index=index)


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
    L = pkg._lib.lib()
    pkg._lib.check(L.rtd3_env_rollout(env._handle, pkg._lib.ptr(env._state[0]), pkg._lib.ptr(env._state[1]), pkg._lib.ptr(p),
                                      pkg._lib.ptr(out), n, T, pkg._lib.stream_ptr(torch.device("cuda", 0))))
    torch.cuda.synchronize()
    return (out.cuda() if out is not None else None), env._state.clone()


def same(a, b):
    return bool(((a == b) | (torch.isnan(a) & torch.isnan(b))).all())


def check(pkg, start, planes, maps=None, index=None, traj="device"):
    n = start.shape[0]
    maps = maps if maps is not None else eo.synthetic_maps(0)
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
    L = pkg._lib.lib()
    L.rtd3_env_force_plain_rollout(1)                          # the cp.async kernel
    try:
        plain, plain_state = rollout(pkg, env_of(pkg, n, maps, index), start, planes, "device")
    finally:
        L.rtd3_env_force_plain_rollout(0)
    assert torch.equal(state, plain_state)
    if got is not None:
        assert same(got, plain)


def switch_sizes():
    """The last batch with one tile per CTA and the first with two (a multiple of 4: the pair kernel's TMA tiles need one)."""
    return [32 * sms(), 32 * sms() + 4]


@pytest.mark.parametrize("T", [1, 31, 33, 1000])
@pytest.mark.parametrize("n", [1, 4, 7, 9, 12, 17, 20, 28, 31, 33, 36, 4100, "switch_lo", "switch_hi"])
def test_tiles_split_unevenly_across_chain_warps(pkg, n, T):
    n = {"switch_lo": switch_sizes()[0], "switch_hi": switch_sizes()[1]}.get(n, n)
    check(pkg, *workload(n, T, seed=n + T))


@pytest.mark.parametrize("n", [36, 4096, "switch_hi"])
def test_nonfinite_actions_in_one_tile_and_one_chain_warp(pkg, n):
    """NaN in a tile whose neighbour stays finite, and inf only in the envs of one chain warp of another tile: those tiles run
    the state-addressed path for the chunks concerned, their chain warps with finite actions included."""
    n = switch_sizes()[1] if n == "switch_hi" else n
    T = 97
    start, planes = workload(n, T, seed=5)
    planes[40, 0, 3] = np.nan                                   # tile 0, chain warp 0; tile 1 stays finite
    w = (n // 32 - 1) * 32 + CHAIN_LANES                        # chain warp 1 of the last full tile
    planes[64:72, 1, w:w + CHAIN_LANES] = np.inf
    planes[90, :, w + 1] = -np.inf
    check(pkg, start, planes)


@pytest.mark.parametrize("n,T", [(36, 33), (4096, 33), (4096, 1000)])
def test_start_states_in_cell_99(pkg, n, T):
    check(pkg, *workload(n, T, seed=9, lo=99.0, hi=99.99999))


@pytest.mark.parametrize("n", [64, 4096, "switch_hi"])
def test_bank_maps_inside_and_between_chain_warps(pkg, n):
    """Maps that differ between the lanes of one chain warp (the mixed-map path), and maps that are uniform per chain warp but
    differ between the chain warps of one tile: a warp on the staged map runs the fast path next to warps on other maps."""
    n = switch_sizes()[1] if n == "switch_hi" else n
    T = 97
    start, planes = workload(n, T, seed=13)
    env_ids = np.arange(n)
    check(pkg, start, planes, *bank((env_ids // 3) % 3))
    check(pkg, start, planes, *bank(((env_ids % 32) // CHAIN_LANES) % 3))


@pytest.mark.parametrize("traj", [None, "host"])
@pytest.mark.parametrize("n", [36, 4096, "switch_hi"])
def test_trajectory_none_and_pinned_host(pkg, n, traj):
    n = switch_sizes()[1] if n == "switch_hi" else n
    start, planes = workload(n, 97, seed=17)
    planes[50, 0, n - 1] = np.nan
    check(pkg, start, planes, traj=traj)
