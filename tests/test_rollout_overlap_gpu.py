"""Rollout launches overlap the previous kernel of the stream (programmatic dependent launch, rtd3_env_set_launch_overlap):
a launch stages its table before it waits for that kernel and reads state, actions and the map index after.  Every sequence
below runs back to back on one stream with the overlap on and off; final states and every trajectory must be bit-identical."""
import numpy as np
import pytest
import torch

from oracle import env_oracle as eo

pytestmark = pytest.mark.gpu


def _roll(pkg, env, act, traj):
    """One rtd3_env_rollout launch on the current stream: act / traj are [T,2,n] planes."""
    lib = pkg._lib
    T, _, n = act.shape
    lib.check(lib.lib().rtd3_env_rollout(env._handle, lib.ptr(env._state[0]), lib.ptr(env._state[1]), lib.ptr(act),
                                         lib.ptr(traj), n, T, lib.stream_ptr(env.device)), "env_rollout")


def _actions(n, T, seed, k=1):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    return [torch.rand((T, 2, n), device="cuda", generator=gen) * 15 - 7.5 for _ in range(k)]


def _env(pkg, n, maps=None):
    env = pkg.Environment(num_envs=n, seed=11, maps=maps if maps is not None else eo.synthetic_maps(0))
    env.reset()
    return env


def _both(pkg, seq):
    """seq() -> list of tensors, run with the overlap on and off; the outputs must match bit for bit."""
    L = pkg._lib.lib()
    out = {}
    try:
        for on in (0, 1):
            L.rtd3_env_set_launch_overlap(on)
            res = seq()
            torch.cuda.synchronize()
            out[on] = [r.clone() for r in res]
    finally:
        L.rtd3_env_set_launch_overlap(1)
    assert len(out[0]) == len(out[1])
    for k, (a, b) in enumerate(zip(out[0], out[1])):
        assert torch.equal(a, b), k


def _chain(pkg, n, T, launches=6):
    """Launch k+1's actions are launch k's trajectory (states, clipped to +-5 as actions), no synchronisation in between."""
    def seq():
        env = _env(pkg, n)
        first = _actions(n, T, 5)[0]
        trajs = [torch.empty((T, 2, n), device="cuda") for _ in range(launches)]
        _roll(pkg, env, first, trajs[0])
        for k in range(1, launches):
            _roll(pkg, env, trajs[k - 1], trajs[k])
        return trajs + [env._state]
    return seq


# 4096: one chain/helper pair per CTA (the bench size); 8192: two pairs per CTA; 65536: single-warp TMA kernel, shallow ring;
# 4095 (odd): the cp.async kernel.  T = 77 leaves a ragged last chunk in every kernel.
@pytest.mark.parametrize("n", [4096, 8192, 65536, 4095])
@pytest.mark.parametrize("T", [200, 77])
def test_chained_trajectories(pkg, n, T):
    _both(pkg, _chain(pkg, n, T))


@pytest.mark.parametrize("n", [4096, 4095])
def test_torch_op_rewrites_state_between_launches(pkg, n):
    T = 96

    def seq():
        env = _env(pkg, n)
        acts = _actions(n, T, 7, 4)
        trajs = [torch.empty((T, 2, n), device="cuda") for _ in acts]
        for k, (a, t) in enumerate(zip(acts, trajs)):
            _roll(pkg, env, a, t)
            env._state.mul_(0.5).add_(10.0 * k)          # a torch kernel writes the state the next launch reads
        return trajs + [env._state]
    _both(pkg, seq)


@pytest.mark.parametrize("n", [4096, 8192])
def test_map_changes_directly_before_a_rollout(pkg, n):
    """set_map, set_maps (K = 3, with an index) and set_map_index on the stream right before a launch, each with new content."""
    T = 64
    maps = [eo.synthetic_maps(s) for s in range(4)]
    bank = (np.stack([m[0] for m in maps[1:]]), np.stack([m[1] for m in maps[1:]]))

    def seq():
        env = _env(pkg, n)
        acts = _actions(n, T, 9, 7)
        trajs = [torch.empty((T, 2, n), device="cuda") for _ in acts]
        _roll(pkg, env, acts[0], trajs[0])
        env.set_maps(*maps[1])                           # K = 1: the single-map kernel, table rebuilt just before
        _roll(pkg, env, acts[1], trajs[1])
        _roll(pkg, env, acts[2], trajs[2])
        idx = torch.arange(n, device="cuda", dtype=torch.int32) // 64 % 3
        env.set_maps(*bank, index=idx)                   # K = 3 with an index: the bank kernel
        _roll(pkg, env, acts[3], trajs[3])
        env.set_map_index((idx + 1) % 3)                 # new index, same bank
        _roll(pkg, env, acts[4], trajs[4])
        env.set_map_index(None)                          # back to map 0 of the bank, single-map kernel
        _roll(pkg, env, acts[5], trajs[5])
        env.set_maps(*maps[0])
        _roll(pkg, env, acts[6], trajs[6])
        return trajs + [env._state]
    _both(pkg, seq)


@pytest.mark.parametrize("n", [4096, 4095])
def test_captured_graph_replay(pkg, n):
    """The chained sequence captured into a CUDA graph, replayed twice, then one eager launch after the replays."""
    T, launches = 64, 4

    def seq():
        env = _env(pkg, n)
        first = _actions(n, T, 13)[0]
        trajs = [torch.empty((T, 2, n), device="cuda") for _ in range(launches)]
        tail = torch.empty((T, 2, n), device="cuda")
        outs = []
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        g = torch.cuda.CUDAGraph()
        with torch.cuda.stream(s), torch.cuda.graph(g, stream=s):
            _roll(pkg, env, first, trajs[0])
            for k in range(1, launches):
                _roll(pkg, env, trajs[k - 1], trajs[k])
        torch.cuda.current_stream().wait_stream(s)
        for _ in range(2):
            g.replay()
            outs += [t.clone() for t in trajs] + [env._state.clone()]
        _roll(pkg, env, trajs[-1], tail)
        return outs + [tail, env._state]
    _both(pkg, seq)


@pytest.mark.parametrize("mode", ["graph_in", "graph", "zero_copy", "hybrid"])
def test_rollout_host(pkg, mode):
    """Host trajectories: the kernel's TMA stores cross PCIe (graph_in, zero_copy, hybrid) or the copy engine brings them back."""
    n, T = 4096, 120

    def seq():
        env = _env(pkg, n)
        h_act = [a.cpu().pin_memory() for a in _actions(n, T, 17, 3)]
        h_traj = [torch.empty((T, 2, n)).pin_memory() for _ in h_act]
        for a, t in zip(h_act, h_traj):
            env.rollout_host(a, t, chunks=4, mode=mode)
        torch.cuda.synchronize()
        return [t.clone() for t in h_traj] + [env._state]
    _both(pkg, seq)
