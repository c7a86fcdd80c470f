"""Round-2 learner plumbing on the GPU: `rtd3_td3_update` (the epoch loop behind one C-ABI call), the in-kernel target-policy
smoothing noise (Philox4x32-10, pinned to oracle/philox.py), and the drop-in nits of Environment / Robot."""
import numpy as np
import pytest
import torch

from oracle import philox
from oracle import td3_oracle as to

pytestmark = pytest.mark.gpu


def synthetic_replay(pkg, n=4000, seed=0, capacity=None):
    g = torch.Generator(device="cuda").manual_seed(seed)
    s = torch.rand((n, 2), device="cuda", generator=g) * 98.9999
    a = torch.rand((n, 2), device="cuda", generator=g) * 10 - 5
    s2 = (s + a).clamp(0, 98.9999)
    r = -torch.linalg.norm(s2 - torch.tensor([80., 20.], device="cuda"), dim=1)
    rb = pkg.ReplayBuffer(capacity or n, seed=seed)
    rb.push(s, a, r, s2, (torch.arange(n, device="cuda") % 50) == 49)
    return rb


def make_agent(pkg, H, L, B, E, seed=0):
    torch.manual_seed(seed)
    return pkg.TD3(pkg.Residual_Actor_Network(H, L), pkg.Residual_Critic_Network(H, L), pkg.Residual_Critic_Network(H, L), batch_size=B, num_epochs=E)


def test_target_noise_matches_the_philox_oracle(pkg):
    L = pkg._lib.lib()
    rows, seed, counter = 300, 0x7d3, 12345678901
    out = torch.empty((rows, 2), dtype=torch.float32, device="cuda")
    pkg._lib.check(L.rtd3_td3_target_noise(seed, counter, pkg._lib.ptr(out), rows, pkg._lib.stream_ptr()))
    ref = np.array([philox.normal2(seed, counter, row) for row in range(rows)])
    np.testing.assert_allclose(out.cpu().numpy(), ref.astype(np.float32), rtol=2e-6, atol=2e-7)
    big = torch.empty((1 << 18, 2), dtype=torch.float32, device="cuda")
    pkg._lib.check(L.rtd3_td3_target_noise(seed, 7, pkg._lib.ptr(big), big.shape[0], pkg._lib.stream_ptr()))
    z = big.double()
    assert abs(float(z.mean())) < 5e-3 and abs(float(z.var()) - 1) < 1e-2
    assert abs(float((z[:, 0] * z[:, 1]).mean())) < 5e-3


@pytest.mark.parametrize("H,L,B", [(200, 3, 100), (256, 2, 256)])
def test_update_with_kernel_noise_equals_update_with_that_noise_injected(pkg, H, L, B):
    """td3_update(noise=None) generates the smoothing noise in the critic kernels; injecting the same normals (rtd3_td3_target_noise
    for steps counter .. counter+E-1) must give bit-identical parameters and losses - and both equal the numpy oracle to 1e-3."""
    E = 6
    rb = synthetic_replay(pkg)
    idx = torch.randint(0, len(rb), (E + 3, B), device="cuda", dtype=torch.int32)
    a1, a2 = make_agent(pkg, H, L, B, E), make_agent(pkg, H, L, B, E)
    assert torch.equal(a1.params, a2.params)
    a1.noise_seed = a2.noise_seed = 99
    noise = torch.empty((E, B, 2), dtype=torch.float32, device="cuda")
    for e in range(E):
        pkg._lib.check(pkg._lib.lib().rtd3_td3_target_noise(99, e, pkg._lib.ptr(noise[e]), B, pkg._lib.stream_ptr()))
    c1, l1 = a1.td3_update(rb, idx=idx)                    # noise generated in the kernels, steps 0..E-1
    c2, l2 = a2.td3_update(rb, idx=idx, noise=noise)
    # parameters bit-identical; the reported losses are sums of per-CTA partial sums added atomically (order varies run to run)
    assert torch.equal(a1.params, a2.params)
    torch.testing.assert_close(c1, c2, rtol=1e-6, atol=0)
    torch.testing.assert_close(l1, l2, rtol=1e-6, atol=0)
    assert int(a1._noise_counter.item()) == E and a1._noise_steps == E
    c1b, _ = a1.td3_update(rb, idx=idx)                    # the replayed graph draws FRESH noise (device counter)
    for e in range(E):
        pkg._lib.check(pkg._lib.lib().rtd3_td3_target_noise(99, E + e, pkg._lib.ptr(noise[e]), B, pkg._lib.stream_ptr()))
    c2b, _ = a2.td3_update(rb, idx=idx, noise=noise)
    assert torch.equal(a1.params, a2.params)
    torch.testing.assert_close(c1b, c2b, rtol=1e-6, atol=0)
    assert int(a1._noise_counter.item()) == 2 * E


def test_update_entry_point_vs_oracle_and_eager_steps(pkg):
    """rtd3_td3_update == the step-by-step calls (train_critic / train_actor / soft_update) bit for bit, and the numpy oracle to 1e-3."""
    H, L, B, E = 64, 2, 48, 6
    rb = synthetic_replay(pkg, 1000)
    rs = np.random.RandomState(1)
    idx = torch.from_numpy(rs.randint(0, 1000, (E + 3, B)).astype(np.int32)).cuda()
    noise = torch.from_numpy(rs.normal(size=(E, B, 2)).astype(np.float32)).cuda()
    a1, a2 = make_agent(pkg, H, L, B, E, seed=3), make_agent(pkg, H, L, B, E, seed=3)
    closs, aloss = a1.td3_update(rb, idx=idx, noise=noise, use_graph=False)
    k = 0
    cl, al = [], []
    for e in range(E):
        cl.append(a2.train_critic(rb, noise=noise[e], idx=idx[k])); k += 1
        if e % 2 == 0:
            al.append(a2.train_actor(rb, idx=idx[k])); k += 1
            for t, s in ((a2.target_actor, a2.actor_network), (a2.target_critic_network_1, a2.critic_network_1),
                         (a2.target_critic_network_2, a2.critic_network_2)):
                a2.soft_update(t, s, a2.tau)
    assert torch.equal(a1.params, a2.params)
    np.testing.assert_allclose(closs.cpu().numpy(), np.asarray(cl, dtype=np.float32), rtol=1e-6)    # (atomically summed partial losses)
    np.testing.assert_allclose(aloss.cpu().numpy(), np.asarray(al, dtype=np.float32), rtol=1e-6)
    # oracle
    a3 = make_agent(pkg, H, L, B, E, seed=3)
    orc = to.TD3Oracle(a3.flat(0).cpu().numpy(), a3.flat(1).cpu().numpy(), a3.flat(2).cpu().numpy(), hidden=H, layers=L)
    ro = to.ReplayOracle(1000)
    ro.s[:], ro.a[:], ro.r[:], ro.s2[:] = rb.s.cpu().numpy(), rb.a.cpu().numpy(), rb.r.cpu().numpy(), rb.s2.cpu().numpy()
    ro.done[:] = rb.notdone.cpu().numpy() < 0.5
    ro.size = 1000
    oc, oa = orc.td3_update(ro, list(idx.cpu().numpy()), list(noise.cpu().numpy()), E)
    np.testing.assert_allclose(closs.cpu().numpy(), np.asarray(oc), rtol=1e-3)
    np.testing.assert_allclose(aloss.cpu().numpy(), np.asarray(oa), rtol=1e-3)


def test_update_entry_point_argument_errors(pkg):
    L = pkg._lib.lib()
    a = pkg._lib.Td3UpdateArgs()
    assert L.rtd3_td3_update(None, None, None) == -1
    ag = make_agent(pkg, 64, 2, 16, 2)
    assert L.rtd3_td3_update(ag._handle, pkg._lib.ctypes.byref(a), None) == -1 and b"null learner state" in L.rtd3_last_error()


def test_scratch_growth_keeps_captured_graphs_valid(pkg):
    """B = 64 graph captured, then B = 256 grows the row scratch, then the B = 64 graph is replayed: its (retired) scratch is still
    alive, so the replay equals a fresh agent's run."""
    E = 4
    rb = synthetic_replay(pkg, 2000)
    idx64 = torch.randint(0, 2000, (E + 2, 64), device="cuda", dtype=torch.int32)
    idx256 = torch.randint(0, 2000, (E + 2, 256), device="cuda", dtype=torch.int32)
    a1, a2 = make_agent(pkg, 128, 2, 64, E, seed=5), make_agent(pkg, 128, 2, 64, E, seed=5)
    for ag in (a1, a2):
        ag.td3_update(rb, idx=idx64)
    a1.td3_update(rb, idx=idx256)
    junk = [torch.full((1 << 20,), 7.0, device="cuda") for _ in range(4)]      # would land in a freed scratch
    a2.td3_update(rb, idx=idx256, use_graph=False)
    a1.td3_update(rb, idx=idx64)
    a2.td3_update(rb, idx=idx64, use_graph=False)
    assert torch.equal(a1.params, a2.params)
    del junk


def test_single_env_robot_state_is_returned_by_reference(pkg):
    np.random.seed(3)
    env = pkg.Environment()
    s0 = env.reset()
    assert s0 is env.robot_state and s0.dtype == np.float64
    s1 = env.step(np.array([1.0, -2.0]))
    assert s1 is env.robot_state and s1 is not s0
    assert env.robot_state is s1                                    # stable between state changes
    probe = env.get_random_robot_init_state()
    assert env.robot_state is s1 and not np.array_equal(probe, s1)  # a draw that does not move the robot
    env.robot_state = np.array([10.0, 20.0])
    assert np.array_equal(env.robot_state, [10.0, 20.0])


def test_check_if_stuck_matches_the_reference_logic(pkg):
    """Robot.check_if_stuck against a list-based restatement of robot.py:509-538, single env and batched."""
    rs = np.random.RandomState(0)
    path = np.cumsum(rs.uniform(-1.2, 1.2, (60, 2)), axis=0) + 50
    prev, exp = [], []
    for s in path.astype(np.float32):
        stuck = False
        if len(prev) >= 5:
            if all(np.linalg.norm(s.astype(np.float64) - p.astype(np.float64)) < 2 for p in prev[-5:]):
                stuck = True
                prev.clear()
            else:
                prev.pop(0)
        prev.append(s)
        exp.append(stuck)
    robot = pkg.Robot(np.array([80.0, 20.0]), hidden=32, layers=2)
    got = [robot.check_if_stuck(s) for s in path]
    assert got == exp and any(exp)
    goals = torch.tensor([[80.0, 20.0]] * 3, device="cuda", dtype=torch.float64)
    rb = pkg.Robot(goals, hidden=32, layers=2)
    got_b = [rb.check_if_stuck(torch.from_numpy(np.stack([s, s + 30, s])).cuda().float()).cpu().numpy() for s in path]
    assert [bool(g[0]) for g in got_b] == exp and [bool(g[2]) for g in got_b] == exp


def test_multi_tick_launch_refuses_a_ring_it_could_corrupt(pkg):
    """K ticks x n envs must fit in the replay ring for rtd3_tick_run_f16 (CTAs drift apart by up to K ticks): the entry point
    reports it, and BatchedTrainer.run falls back to the three-launch tick, whose rows are then bit-identical to the eager ticks."""
    n, K = 256, 8
    def build(cap):
        torch.manual_seed(4)                                 # the networks draw their initial weights from torch's generator
        env = pkg.Environment(num_envs=n, seed=11)
        robot = pkg.Robot(env.goal_state, hidden=64, layers=2, seed=5, buffer_size=cap)
        robot.td3_agent.precision = "f16"
        robot.episodes_per_update = 1 << 30
        return env, robot, pkg.BatchedTrainer(env, robot, noise="philox", graph=True, check_interval=K, fused=True)
    env, robot, tr = build(n * K - 1)
    assert not tr._multi_tick_ok()
    robot.td3_agent.prepare_forward(n)
    t = tr._tick_state()
    L = pkg._lib.lib()
    rc = L.rtd3_tick_run_f16(env._handle, pkg._lib.ctypes.byref(t), 64, 2, pkg._lib.ptr(robot.td3_agent.params), pkg._lib.ptr(robot.td3_agent.params_h),
                             pkg._lib.TICK_NOISE_PHILOX, K, 0, pkg._lib.stream_ptr())
    assert rc == -1 and b"replay ring smaller" in L.rtd3_last_error()
    tr.run(3 * K)                                            # wraps the ring inside the run, three-launch ticks in a graph
    env2, robot2, tr2 = build(n * K - 1)
    tr2._use_graph = False
    for _ in range(3 * K):
        tr2.tick()
    assert torch.equal(env._state, env2._state) and int(robot.memory._total_dev) == int(robot2.memory._total_dev)
    key = lambda rb: torch.sort(rb.s[:, 0] * 1000 + rb.r)[0]
    assert torch.equal(key(robot.memory), key(robot2.memory))
    env3, robot3, tr3 = build(n * K)
    assert tr3._multi_tick_ok()


@pytest.mark.parametrize("H,L,B,E", [(256, 2, 256, 6), (200, 3, 100, 6), (64, 2, 48, 5), (128, 4, 33, 4), (32, 2, 700, 3)])
def test_step_kernel_update_vs_oracle_and_graph_replay(pkg, H, L, B, E):
    """td3_update on the step kernels (cluster kernels up to one wave of clusters, row tiles above) against the numpy oracle (losses
    1e-3), and two graph-replayed updates against the same two run without a graph (parameters bit for bit)."""
    rb = synthetic_replay(pkg, 3000)
    rs = np.random.RandomState(2)
    n_idx = E + (E + 1) // 2
    idx = torch.from_numpy(rs.randint(0, 3000, (n_idx, B)).astype(np.int32)).cuda()
    noise = torch.from_numpy(rs.normal(size=(E, B, 2)).astype(np.float32)).cuda()
    a_graph, a_eager = make_agent(pkg, H, L, B, E, seed=7), make_agent(pkg, H, L, B, E, seed=7)
    c1, l1 = a_graph.td3_update(rb, idx=idx, noise=noise)
    c2, l2 = a_eager.td3_update(rb, idx=idx, noise=noise, use_graph=False)
    assert torch.equal(a_graph.params, a_eager.params)
    torch.testing.assert_close(c1, c2, rtol=1e-6, atol=0)             # (atomically summed partial losses)
    torch.testing.assert_close(l1, l2, rtol=1e-6, atol=0)
    a3 = make_agent(pkg, H, L, B, E, seed=7)
    orc = to.TD3Oracle(a3.flat(0).cpu().numpy(), a3.flat(1).cpu().numpy(), a3.flat(2).cpu().numpy(), hidden=H, layers=L)
    ro = to.ReplayOracle(3000)
    ro.s[:], ro.a[:], ro.r[:], ro.s2[:] = rb.s.cpu().numpy(), rb.a.cpu().numpy(), rb.r.cpu().numpy(), rb.s2.cpu().numpy()
    ro.done[:] = rb.notdone.cpu().numpy() < 0.5
    ro.size = 3000
    oc, oa = orc.td3_update(ro, list(idx.cpu().numpy()), list(noise.cpu().numpy()), E)
    np.testing.assert_allclose(c1.cpu().numpy(), np.asarray(oc), rtol=1e-3)
    np.testing.assert_allclose(l1.cpu().numpy(), np.asarray(oa), rtol=1e-3)
    # a second, graph-replayed update keeps agreeing
    c1b, _ = a_graph.td3_update(rb, idx=idx, noise=noise)
    c2b, _ = a_eager.td3_update(rb, idx=idx, noise=noise, use_graph=False)
    assert torch.equal(a_graph.params, a_eager.params)
    assert torch.equal(a_graph.steps, a_eager.steps) and torch.equal(a_graph.beta_pows, a_eager.beta_pows)
    torch.testing.assert_close(c1b, c2b, rtol=1e-6, atol=0)


@pytest.mark.parametrize("H,L,B", [(256, 2, 256), (200, 3, 100), (256, 2, 37), (64, 2, 261), (128, 1, 64)])
def test_cluster_step_kernels_vs_row_tile_kernels(pkg, H, L, B):
    """The cluster step kernels (csrc/rtd3_cluster.cu: 4 CTAs share 8 batch rows and split every layer's columns) against the row-tile
    kernels on the same minibatch: gradients of all three networks, losses, Q-values and targets.  The two differ in summation order
    only - a different split of every reduction - so the bar is float32 round-off of chained 256-term sums over O(100) inputs (1e-4;
    measured <= 8e-5 on the three-layer shape), not the 1e-3 of the parity bar.
    Ragged batches (37, 261 rows: a last cluster with 5 valid rows; 261 rows = 33 clusters, all the device holds at once - larger
    batches stay on the row tiles), 13 column groups per CTA (H = 200) and a single hidden layer
    (the head straight from the first layer) are the cluster plan's edge cases."""
    L_ = pkg._lib.lib()
    rb = synthetic_replay(pkg)
    idx = torch.randint(0, len(rb), (B,), device="cuda", dtype=torch.int32)
    noise = torch.randn((B, 2), device="cuda")
    out = {}
    prev = L_.rtd3_debug_cluster_mode(2)
    try:
        for mode in (2, 0):
            L_.rtd3_debug_cluster_mode(mode)
            ag = make_agent(pkg, H, L, B, 1, seed=5)
            assert L_.rtd3_td3_cluster_supported(ag._handle, B) == (1 if mode == 2 else 0)
            ag.sync_transposed()
            loss2 = torch.zeros(2, device="cuda"); loss1 = torch.zeros(1, device="cuda")
            q = torch.zeros((2, B), device="cuda"); y = torch.zeros(B, device="cuda")
            ag._critic_step(rb, idx, noise, loss2, q, y, apply=False)          # critic gradients stay in ag.grads
            ag._actor_step(rb, idx, loss1)                                     # + the actor's (no optimiser step in between)
            out[mode] = (ag.grads.clone(), torch.cat([loss2, loss1]), q.clone(), y.clone())
    finally:
        L_.rtd3_debug_cluster_mode(prev)
    (g1, l1, q1, y1), (g0, l0, q0, y0) = out[2], out[0]
    torch.testing.assert_close(y1, y0, rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(q1, q0, rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(l1, l0, rtol=1e-4, atol=0)
    scale = float(g0.abs().max())
    assert float((g1 - g0).abs().max()) <= 1e-4 * scale
