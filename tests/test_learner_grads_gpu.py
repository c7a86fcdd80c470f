"""The learner's gradients against a float64 reference, and its optimiser bit for bit against the oracle.

Gradients (oracle/td3_float64.py): each float32 gradient element g must satisfy |g - g64| <= tau * M, where g64 is the float64
gradient of the same step on the same float32 parameters and rows, and M the same backward pass on magnitudes.  Elements with M == 0
must be exactly 0.  Batches are drawn from kink-safe rows only (no pre-activation of a differentiated network within 2^-16 * |z|_abs
of zero), with duplicate rows and rows with `done` set.  Q-values, targets and critic losses share the bar (with their own M); the
actor loss is checked against tau * mean |Q|_abs.
  - The raw fp32 step kernels (`_critic_step(apply=False)`, `_actor_step`) at every dispatch boundary: the cluster kernels, the row
    tiles R = 2 / 4 / 8 / 16 (boundaries at 2, 4 and 16 times the SM count) and the weight-gradient batch split above 512 rows.
  - The production update paths (fused optimiser at B <= 512, unfused above, TF32), with and without the
    CUDA graph.  They expose no gradients, but one epoch from a fresh agent leaves adam_m = RN(0.1f * g), so g = adam_m / 0.1f to one
    ulp.  The actor step of an update reads critic 1 after the critics' Adam step, so its reference uses the final critic 1.
  - Controls: every fp32 case also checks that the bar REJECTS a subtly wrong reference (a dropped row, one `done` flipped, max
    instead of min of the twin targets, the smoothing noise unclipped, the actor gradient through critic 2).

Measured on a B200 (1000 W power limit), worst |x - x64| / M over the cases of this file:
  fp32 step kernels, gradients: cluster 1.5e-7 (the 4-wide net; 1.5e-8 at H >= 64), R=2 1.5e-7 (same), R=4 6.5e-9,
    R=4 with the batch split 1.5e-8, R=8 split 3.9e-8, R=16 split 1.6e-8; Q 7.5e-8, y 3.7e-8, critic loss 2.1e-8, actor loss 7e-9
  update paths, gradients from adam_m: fused 7.6e-9, unfused 8.4e-9, TF32 3.3e-3 (H = 256, B = 8192; 1.5e-4 at
    H = 128, B = 1041)
  controls (fp32), smallest distance from the kernel's gradient: 9.3e-7 (one `done` flipped, H = 200, L = 3, B = 2368)
TAU_FP32 = 2^-21 sits between the two: far below the 2^-15 that fp32 summation-error arithmetic allows, because the magnitude sums
M are loose by the networks' cancellation.  TF32 operands resolve only the actor-through-critic-2 control (2.4e-2); max instead of min
(1.1e-2) and the unclipped noise (1.5e-4) are within TF32's error at B = 8192.  tests/test_tc_exact_gpu.py closes that gap: on dyadic
vectors where nothing rounds (oracle/exact_grid.py) the TF32 critic step, actor step and update epoch must equal the float64 reference
bit for bit, and tests/test_exact_grid.py checks that every one of these controls changes that reference.

Optimiser: the Adam / Polyak kernel, element for element against oracle/td3_oracle.py's adam_step / soft_update (pinned to
torch.optim.Adam), with lr a Python float as in torch, and the Adam step of the fused and TF32 update paths against the
same formula on the device's own moments; the kernels that rebuild the derived weight copies from the whole arena against their layouts.
"""
import numpy as np
import pytest
import torch

from oracle import td3_float64 as t64
from oracle import td3_oracle as to

pytestmark = pytest.mark.gpu
F32 = np.float32
TAU_FP32 = 2.0 ** -21      # 4.8e-7: 3.3x the worst measured 1.46e-7, below the weakest control (9.3e-7)
TAU_TF32 = 2.0 ** -6       # 1.6e-2: 4.7x the worst measured 3.3e-3


# ---------------------------------------------------------------------------------------------------- set-up
def make_nets(rs, H, L):
    """Six networks: kaiming init plus noise (non-zero biases, targets != online); the actors' heads scaled so that actions are O(1),
    inside +-max_action, where the target-action clip and the noise clip both matter."""
    nets = []
    for k in range(6):
        i, o = (2, 2) if k % 3 == 0 else (4, 1)
        w = to.kaiming_uniform_params(rs, i, H, L, o) + rs.normal(0, 0.01, to.param_count(i, H, L, o)).astype(F32)
        if o == 2:
            w[-(2 * H + 2):] *= F32(0.02 if H >= 32 else 0.002)
        nets.append(w.astype(F32))
    return nets


def make_replay(pkg, rs, n):
    s = rs.uniform(0, 98.9999, (n, 2)).astype(F32)
    a = rs.uniform(-5, 5, (n, 2)).astype(F32)
    s2 = np.clip(s + a, 0, 98.9999).astype(F32)
    r = (-np.linalg.norm(s2 - np.array([80, 20], F32), axis=1)).astype(F32)
    d = (np.arange(n) % 7) == 3
    rb = pkg.ReplayBuffer(n, seed=1)
    rb.push(*(torch.from_numpy(x).cuda() for x in (s, a, r, s2, d)))
    return rb, (s, a, r, s2, d)


def make_agent(pkg, nets, H, L, B, **kw):
    agent = pkg.TD3(pkg.Residual_Actor_Network(H, L), pkg.Residual_Critic_Network(H, L), pkg.Residual_Critic_Network(H, L), batch_size=B, **kw)
    for k, w in enumerate(nets):
        agent.flat(k).copy_(torch.from_numpy(w).cuda())
    agent.sync_transposed()
    return agent


def noise_for(rs, B):
    noise = rs.normal(size=(B, 2)).astype(F32)
    noise[::2, 0] = 4.0       # beyond noise_clip / policy_noise = 2.5: the clip matters (one sign: a duplicated row must not cancel)
    return noise


def worst(x, ref, M):
    """max |x - ref| / M over M > 0; asserts x == 0 exactly where M == 0."""
    x, ref, M = (np.asarray(v, np.float64).ravel() for v in (x, ref, M))
    assert (x[M == 0] == 0).all(), "an element with a zero bound is not exactly zero"
    pos = M > 0
    return float((np.abs(x[pos] - ref[pos]) / M[pos]).max()) if pos.any() else 0.0


def rejects(x, ref, M, tau):
    x, ref, M = (np.asarray(v, np.float64).ravel() for v in (x, ref, M))
    return bool((np.abs(x - ref) > tau * M).any())


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def row_tile(B):
    """csrc/rtd3_td3.cu: pick_tile - rows per CTA of the row-tile step kernels."""
    n = sms()
    return 2 if B <= 2 * n else 4 if B <= 4 * n else 8 if B <= 16 * n else 16


def cluster_max_batch(pkg, agent):
    L_ = pkg._lib.lib()
    return max(b for b in range(1, 4097) if L_.rtd3_td3_cluster_supported(agent._handle, b))


# ---------------------------------------------------------------------------------------------------- (a) the fp32 step kernels
def _batch_cases():
    # (H, L, B, path): B given as an int, or as a function of the device (SM count / the cluster kernels' capacity)
    n = lambda k, d=0: ("sms", k, d)
    return [
        (256, 2, 256, "cluster"), (256, 2, 256, "rows"), (200, 3, 100, "cluster"), (200, 3, 100, "rows"), (256, 2, 1, "cluster"),
        (256, 2, 1, "rows"), (64, 2, 37, "cluster"), (256, 2, ("cmax", 0), "cluster"), (256, 2, ("cmax", 1), "rows"),
        (256, 2, n(2), "rows"), (256, 2, n(2, 1), "rows"), (200, 3, 512, "rows"), (200, 3, 513, "rows"), (256, 2, 600, "rows"),
        (256, 2, n(4), "rows"), (256, 2, n(4, 1), "rows"), (200, 3, n(16), "rows"), (256, 2, n(16, 1), "rows"), (256, 2, 8192, "rows"),
        (4, 1, 7, "cluster"), (4, 1, 7, "rows"), (100, 2, 1000, "rows"), (128, 4, 64, "cluster"), (128, 4, 300, "rows"),
    ]


def _case_id(c):
    H, L, B, path = c
    b = B if isinstance(B, int) else ("%dxSM%+d" % (B[1], B[2]) if B[0] == "sms" else "cmax%+d" % B[1])
    return "H%d-L%d-B%s-%s" % (H, L, b, path)


def _critic_actor_grads(agent, rb, idx_c, idx_a, noise):
    B = idx_c.numel()
    loss2 = torch.zeros(2, device="cuda")
    q = torch.zeros((2, B), device="cuda")
    y = torch.zeros((B,), device="cuda")
    loss1 = torch.zeros(1, device="cuda")
    agent.grads.zero_()
    agent._critic_step(rb, idx_c, noise, loss2, q, y, apply=False)
    gc = agent.grads.clone()
    agent.grads.zero_()
    agent._actor_step(rb, idx_a, loss1)
    ga = agent.grads.clone()
    agent.grads.zero_()
    torch.cuda.synchronize()
    return (gc.cpu().numpy(), ga.cpu().numpy(), loss2.cpu().numpy(), float(loss1.cpu()[0]), q.cpu().numpy(), y.cpu().numpy())


def net_grad(agent, g, k):
    return g[agent._off[k]:agent._off[k] + agent._cnt[k]]


@pytest.mark.parametrize("case", _batch_cases(), ids=_case_id)
def test_step_kernel_gradients_vs_float64(pkg, case):
    H, L, B, path = case
    L_ = pkg._lib.lib()
    rs = np.random.RandomState(H * 7 + L)
    nets = make_nets(rs, H, L)
    if not isinstance(B, int):
        if B[0] == "sms":
            B = B[1] * sms() + B[2]
        else:
            probe = make_agent(pkg, nets, H, L, 1)
            B = cluster_max_batch(pkg, probe) + B[1]
    rb, (s, a, r, s2, d) = make_replay(pkg, rs, max(4 * B, 4096))
    ref = t64.Learner64(nets, H, L)
    idx_c, excl_c = t64.draw_usable(rs, ref.usable_rows(s, a, "critic"), B)
    idx_a, excl_a = t64.draw_usable(rs, ref.usable_rows(s, a, "actor"), B)
    assert d[idx_c].any() or B < 8
    noise = noise_for(rs, B)
    prev = L_.rtd3_debug_cluster_mode(2)
    try:
        if path == "rows":
            L_.rtd3_debug_cluster_mode(0)
        agent = make_agent(pkg, nets, H, L, B)
        cl = bool(L_.rtd3_td3_cluster_supported(agent._handle, B))
        assert cl == (path == "cluster"), (B, cl)
        gc, ga, loss2, loss1, q, y = _critic_actor_grads(agent, rb, torch.from_numpy(idx_c).cuda(), torch.from_numpy(idx_a).cuda(),
                                                         torch.from_numpy(noise).cuda())
    finally:
        L_.rtd3_debug_cluster_mode(prev)
    taken = "cluster" if cl else "R=%d" % row_tile(B)
    rc = ref.critic_step(s[idx_c], a[idx_c], r[idx_c], s2[idx_c], d[idx_c], noise)
    ra = ref.actor_step(s[idx_a])
    ratios = {"c1": worst(net_grad(agent, gc, 1), rc["g"][0], rc["M"][0]), "c2": worst(net_grad(agent, gc, 2), rc["g"][1], rc["M"][1]),
              "actor": worst(net_grad(agent, ga, 0), ra["g"], ra["M"]), "q": worst(q, rc["q"], rc["Mq"]), "y": worst(y, rc["y"], rc["My"]),
              "closs": worst(loss2, rc["loss"], rc["Mloss"]), "aloss": abs(loss1 - ra["loss"]) / ra["Mloss"]}
    print("\n[grad-ratio] B=%d path=%s split=%s excluded=%.3f/%.3f %s" % (B, taken, B > 512, excl_c, excl_a,
                                                                        " ".join("%s=%.3g" % kv for kv in ratios.items())))
    assert float(np.abs(gc[:agent._off[1]]).max()) == 0.0 and float(np.abs(ga[agent._off[1]:]).max()) == 0.0
    for k, v in ratios.items():
        assert v <= TAU_FP32, (k, v)
    # (c) the bar is sharp: it rejects each subtly wrong reference
    g_c = [net_grad(agent, gc, 1), net_grad(agent, gc, 2)]
    drop = ["drop_row"] if 1 < B <= 1 / (4 * TAU_FP32) else []
    for control in ["flip_done", "max_target", "noise_unclipped"] + drop:
        bad = ref.critic_step(s[idx_c], a[idx_c], r[idx_c], s2[idx_c], d[idx_c], noise, control=control)
        assert any(rejects(g_c[c], bad["g"][c], rc["M"][c], TAU_FP32) for c in (0, 1)), control
    for control in ["critic2"] + drop:
        assert rejects(net_grad(agent, ga, 0), ref.actor_step(s[idx_a], control=control)["g"], ra["M"], TAU_FP32), control


# ---------------------------------------------------------------------------------------------------- (b) the update paths
UPDATE_CASES = [
    ("fused", 256, 2, 256), ("fused", 200, 3, 100), ("unfused", 256, 2, 600), ("unfused", 200, 3, 1041), ("tf32", 128, 2, 1041),
    ("tf32", 256, 2, 8192),
]


def _update_agent(pkg, nets, H, L, B, path):
    agent = make_agent(pkg, nets, H, L, B, num_epochs=1)
    if path == "tf32":
        agent.precision = "tf32"
        assert agent._tc_learner_ok(B)
    return agent


@pytest.mark.parametrize("use_graph", [True, False], ids=["graph", "eager"])
@pytest.mark.parametrize("path,H,L,B", UPDATE_CASES, ids=["%s-H%d-L%d-B%d" % c for c in UPDATE_CASES])
def test_update_path_gradients_vs_float64(pkg, path, H, L, B, use_graph):
    rs = np.random.RandomState(B + H)
    nets = make_nets(rs, H, L)
    rb, (s, a, r, s2, d) = make_replay(pkg, rs, max(4 * B, 4096))
    ref = t64.Learner64(nets, H, L)
    idx_c, _ = t64.draw_usable(rs, ref.usable_rows(s, a, "critic"), B)
    noise = noise_for(rs, B)
    noise_t = torch.from_numpy(noise[None]).cuda()
    # the actor step differentiates through critic 1 AFTER the critics' Adam step: rows kink-safe for that critic
    dry = _update_agent(pkg, nets, H, L, B, path)
    dry.td3_update(rb, noise=noise_t, idx=torch.from_numpy(np.stack([idx_c, idx_c])).cuda(), use_graph=use_graph)
    c1_after = dry.flat(1).cpu().numpy()
    ref_after = t64.Learner64([nets[0], c1_after] + nets[2:], H, L)
    idx_a, _ = t64.draw_usable(rs, ref_after.usable_rows(s, a, "actor"), B)
    agent = _update_agent(pkg, nets, H, L, B, path)
    agent.td3_update(rb, noise=noise_t, idx=torch.from_numpy(np.stack([idx_c, idx_a])).cuda(), use_graph=use_graph)
    torch.cuda.synchronize()
    assert agent.steps.cpu().tolist() == [1, 1]
    m = agent.adam_m.cpu().numpy()
    g = (m.astype(np.float64) / np.float64(F32(0.1)))              # adam_m = RN(0.1f * g) after one step from zero moments
    c1_final = agent.flat(1).cpu().numpy()
    assert np.array_equal(c1_final, c1_after) or path in ("unfused", "tf32")   # atomics: the split / TF32 reductions may differ in a bit
    rc = ref.critic_step(s[idx_c], a[idx_c], r[idx_c], s2[idx_c], d[idx_c], noise)
    ra = ref.actor_step(s[idx_a], critic=c1_final)
    tau = TAU_TF32 if path == "tf32" else TAU_FP32
    ratios = {"c1": worst(net_grad(agent, g, 1), rc["g"][0], rc["M"][0]), "c2": worst(net_grad(agent, g, 2), rc["g"][1], rc["M"][1]),
              "actor": worst(net_grad(agent, g, 0), ra["g"], ra["M"])}
    print("\n[grad-ratio] update path=%s B=%d graph=%s %s" % (path, B, use_graph, " ".join("%s=%.3g" % kv for kv in ratios.items())))
    for k, v in ratios.items():
        assert v <= tau, (k, v)
    g_c = [net_grad(agent, g, 1), net_grad(agent, g, 2)]
    # TF32 resolves only the critic-2 control (see the module docstring)
    for control in ("max_target", "noise_unclipped", "flip_done") if path != "tf32" else ():
        bad = ref.critic_step(s[idx_c], a[idx_c], r[idx_c], s2[idx_c], d[idx_c], noise, control=control)
        assert any(rejects(g_c[c], bad["g"][c], rc["M"][c], tau) for c in (0, 1)), control
    assert rejects(net_grad(agent, g, 0), ref_after.actor_step(s[idx_a], control="critic2")["g"], ra["M"], tau)


# ---------------------------------------------------------------------------------------------------- (d) Adam and Polyak bit for bit
def special_grads(rs, n):
    """Normal values of several scales, with 0, +-1e-30, subnormals and +-1e20 spread through the arena."""
    g = (rs.normal(size=n) * 10.0 ** rs.randint(-6, 2, n)).astype(F32)
    pool = np.array([0.0, 1e-30, -1e-30, 1e-40, -3e-42, 1.4e-45, -1.4e-45, 1e20, -1e20], F32)
    pick = rs.randint(0, 6, n) == 0
    g[pick] = pool[rs.randint(0, pool.size, int(pick.sum()))]
    return g


def bits(x):
    return np.asarray(x, F32).view(np.int32)


def derived_copies(agent, params):
    """The transposed arena (params_t) and the tensor-core operand copies [u | v] (params_u) the optimiser keeps in step."""
    H, L = agent.hidden, agent.layers
    pt, total = params.copy(), params.size
    u, v = params.copy(), params.copy()
    for k in range(6):
        i = 2 if k % 3 == 0 else 4
        for l in range(L - 1):
            o = agent._off[k] + i * H + H + l * (H * H + H)
            W = params[o:o + H * H].reshape(H, H)
            pt[o:o + H * H] = W.T.reshape(-1)
            Wr = ((W.view(np.uint32) + np.uint32(0x1000)) & np.uint32(0xffffe000)).view(F32)     # TF32, round half away
            u[o:o + H * H] = Wr.T.reshape(H // 4, 4, H).transpose(0, 2, 1).reshape(-1)
            v[o:o + H * H] = Wr.reshape(H // 4, 4, H).transpose(0, 2, 1).reshape(-1)
    return pt, np.concatenate([u, v])


@pytest.mark.parametrize("H,L", [(64, 2), (128, 3), (32, 4)])
def test_sync_kernels_bit_exact(pkg, H, L):
    """The kernels that rebuild the derived copies from the whole arena (after weights were written from outside the optimiser):
    params_t, [u | v] and the fp16 hidden weights (W_l[n][k] at ((net*(L-1) + l-1)*H*H + ((k/8)*H + n)*8 + k%8) bit-equal to their
    layouts, for parameters of every scale, zeros and subnormals included."""
    rs = np.random.RandomState(H + L)
    agent = make_agent(pkg, make_nets(rs, H, L), H, L, 16)
    params = special_grads(rs, agent.params.numel())
    agent.params.copy_(torch.from_numpy(params))
    agent.sync_transposed()
    agent._sync_chunk_major()
    agent._sync_half(force=True)
    torch.cuda.synchronize()
    pt, puv = derived_copies(agent, params)
    assert np.array_equal(bits(agent.params_t.cpu().numpy()), bits(pt))
    uv = agent.params_u.cpu().numpy()
    assert np.array_equal(bits(uv), bits(puv)), int((uv != puv).sum())
    ph = []
    for k in range(6):
        i = 2 if k % 3 == 0 else 4
        for l in range(L - 1):
            o = agent._off[k] + i * H + H + l * (H * H + H)
            W = np.clip(params[o:o + H * H], -65504, 65504).astype(np.float16).reshape(H, H // 8, 8)
            ph.append(W.transpose(1, 0, 2).reshape(-1))
    assert np.array_equal(agent.params_h.cpu().numpy().view(np.uint16), np.concatenate(ph).view(np.uint16))


@pytest.mark.parametrize("lr", [1e-5, 3e-4, 1e-3])
def test_adam_polyak_kernel_bit_exact_vs_oracle(pkg, lr):
    """60 steps of both optimisers through rtd3_td3_adam_polyak with chosen gradients: moments, parameters, targets, clocks and every
    derived copy bit-equal to the oracle.  A third of the parameters start at exactly 0, where a step is never absorbed by the
    parameter it is added to, so a one-ulp difference of the step size shows."""
    H, L, B = 64, 2, 16
    rs = np.random.RandomState(int(lr * 1e6))
    nets = make_nets(rs, H, L)
    for w in nets[:3]:
        w[rs.randint(0, 3, w.size) == 0] = 0.0
    rb, _ = make_replay(pkg, rs, 256)
    agent = make_agent(pkg, nets, H, L, B, actor_lr=lr, critic_lr=lr)
    agent._sync_chunk_major()
    assert agent.params_u is not None and not agent._u_stale
    idx = torch.arange(B, dtype=torch.int32, device="cuda")
    noise = torch.zeros((B, 2), device="cuda")
    p = [w.copy() for w in nets]
    st = [to.AdamState(w.size) for w in nets[:3]]
    for t in range(1, 61):
        loss2, loss1 = torch.zeros(2, device="cuda"), torch.zeros(1, device="cuda")
        agent._critic_step(rb, idx, noise, loss2, apply=False)          # the step kernels advance the Adam clocks
        agent._actor_step(rb, idx, loss1)
        G = np.zeros(agent.grads.numel(), F32)
        for k in range(3):
            gk = special_grads(rs, agent._cnt[k])
            G[agent._off[k]:agent._off[k] + agent._cnt[k]] = gk
            to.adam_step(p[k], gk, st[k], lr=lr)
            to.soft_update(p[k + 3], p[k], agent.tau)
        agent.grads.copy_(torch.from_numpy(G))
        agent._adam(nets=0b111, polyak=0b111)
        torch.cuda.synchronize()
        params = agent.params.cpu().numpy()
        m, v = agent.adam_m.cpu().numpy(), agent.adam_v.cpu().numpy()
        for k in range(6):
            sl = slice(agent._off[k], agent._off[k] + agent._cnt[k])
            assert np.array_equal(bits(params[sl]), bits(p[k])), ("params", k, t, int((params[sl] != p[k]).sum()))
            if k < 3:
                assert np.array_equal(bits(m[sl]), bits(st[k].m)), ("m", k, t)
                assert np.array_equal(bits(v[sl]), bits(st[k].v)), ("v", k, t)
        assert agent.steps.cpu().tolist() == [t, t]
        bp = agent.beta_pows.cpu().numpy()
        exp = [1.0, 1.0]
        for _ in range(t):
            exp = [exp[0] * 0.9, exp[1] * 0.999]
        assert bp.tolist() == exp + exp
        assert float(agent.grads.abs().max()) == 0.0
        pt, puv = derived_copies(agent, params)
        assert np.array_equal(bits(agent.params_t.cpu().numpy()), bits(pt)), ("params_t", t)
        uv, total, n_online = agent.params_u.cpu().numpy(), params.size, params.size // 2
        assert np.array_equal(bits(uv[:total]), bits(puv[:total])), ("params_u", t, int((uv[:total] != puv[:total]).sum()))
        # the input-gradient copy v of the online networks (the target networks run forward only: their v copy is not kept)
        assert np.array_equal(bits(uv[total:total + n_online]), bits(puv[total:total + n_online])), \
            ("params_v", t, int((uv[total:total + n_online] != puv[total:total + n_online]).sum()))


ADAM_PATHS = [("fused", 256, 2, 256), ("tf32", 128, 2, 1041)]


@pytest.mark.parametrize("path,H,L,B", ADAM_PATHS, ids=[c[0] for c in ADAM_PATHS])
def test_update_path_adam_step_bit_exact(pkg, path, H, L, B):
    """The Adam step inside the fused and TF32 updates, from the device's own state: p_t == p_{t-1} +
    (float32(-lr / bc1_t) * m_t) / (sqrt(v_t) / float32(sqrt(bc2_t)) + 1e-8f) bit for bit, at t = 4 and 5 with lr = 1e-5 (steps at which
    a step size formed from a float32 lr is one ulp off).  A third of the online parameters are set to 0 before the step, so the
    step is not absorbed."""
    rs = np.random.RandomState(5)
    nets = make_nets(rs, H, L)
    rb, (s, a, _, _, _) = make_replay(pkg, rs, 4096)
    agent = _update_agent(pkg, nets, H, L, B, path)
    idx = torch.from_numpy(rs.randint(0, 4096, (2, B)).astype(np.int32)).cuda()
    noise = torch.from_numpy(noise_for(rs, B)[None]).cuda()
    half = agent.params.numel() // 2
    checked = 0
    for t in range(1, 6):
        if t >= 4:
            zero = torch.from_numpy(rs.randint(0, 3, half) == 0).cuda()
            for k in range(3):
                sl = slice(agent._off[k], agent._off[k] + agent._cnt[k])
                agent.flat(k).masked_fill_(zero[sl], 0.0)
            prev = agent.params[:half].cpu().numpy()
        agent.td3_update(rb, noise=noise, idx=idx)
        if t < 4:
            continue
        torch.cuda.synchronize()
        assert agent.steps.cpu().tolist() == [t, t]
        m, v, p = agent.adam_m.cpu().numpy(), agent.adam_v.cpu().numpy(), agent.params[:half].cpu().numpy()
        for k, lr in ((0, agent.actor_lr), (1, agent.critic_lr), (2, agent.critic_lr)):
            sl = slice(agent._off[k], agent._off[k] + agent._cnt[k])
            step = F32(-lr / (1 - 0.9 ** t))
            denom = np.sqrt(v[sl]) / F32(np.sqrt(1 - 0.999 ** t)) + F32(1e-8)
            exp = prev[sl] + (step * m[sl]) / denom
            bad = bits(p[sl]) != bits(exp)
            exp32 = prev[sl] + (F32(-F32(lr) / (1 - 0.9 ** t)) * m[sl]) / denom
            assert not bad.any(), (path, t, k, int(bad.sum()), "at p=0:", int((bad & (prev[sl] == 0)).sum()),
                                   "max ulps:", int(np.abs(bits(p[sl]).astype(np.int64) - bits(exp)).max()),
                                   "vs float32-lr formula:", int((bits(p[sl]) != bits(exp32)).sum()),
                                   "m==0:", int((bad & (m[sl] == 0)).sum()), "changed:", int((bad & (p[sl] != prev[sl])).sum()))
            checked += int((prev[sl] == 0).sum())
    assert checked > 0
