"""The tensor-core paths on exact-arithmetic vectors (oracle/exact_grid.py): the TF32 and f16 forwards and the TF32 learner steps equal
the float64 reference bit for bit, and so do the fp32 forward, step kernels and updates on the same vectors.

On these vectors every operand is exact in TF32 and fp16 and every partial sum is exact in fp32 (tests/test_exact_grid.py checks
the premise and that each structural mistake changes the reference), so any difference is a kernel mistake, not rounding.  The
outputs no longer reveal which kernel ran, so the TF32 forward is called through its C entry point and the other calls assert the
path the precision selects."""
import numpy as np
import pytest
import torch

from oracle import exact_grid as eg
from oracle import td3_float64 as t64
from oracle import td3_oracle as to

pytestmark = pytest.mark.gpu

HS = (64, 96, 128, 160, 192, 224, 256)
SEED = 11                                     # tests/test_exact_grid.py checks these vector sets


def agent_on_grid(pkg, vs, H, L):
    torch.manual_seed(0)
    agent = pkg.TD3(pkg.Residual_Actor_Network(H, L), pkg.Residual_Critic_Network(H, L), pkg.Residual_Critic_Network(H, L))
    for k in range(6):
        agent.flat(k).copy_(torch.from_numpy(vs["nets"][k]).cuda())
    agent.sync_transposed()
    return agent


def tf32_arena(pkg, vs, H, L):
    """The six networks in the learner's arena layout (16 B aligned slots: actor, critic 1, critic 2, then the targets) and its
    chunk-major operand copy -> (params, params_u, slot offsets)."""
    sa, sc = ((to.param_count(i, H, L, o) + 3) // 4 * 4 for i, o in ((2, 2), (4, 1)))
    offs = [0, sa, sa + sc, sa + 2 * sc, 2 * sa + 2 * sc, 2 * sa + 3 * sc]
    params = torch.zeros((2 * (sa + 2 * sc),), dtype=torch.float32, device="cuda")
    for k in range(6):
        params[offs[k]:offs[k] + vs["nets"][k].size].copy_(torch.from_numpy(vs["nets"][k]))
    params_u = torch.zeros((2 * params.numel(),), dtype=torch.float32, device="cuda")
    pkg._lib.check(pkg._lib.lib().rtd3_tc_sync_weights(H, L, pkg._lib.ptr(params), pkg._lib.ptr(params_u), pkg._lib.stream_ptr()))
    return params, params_u, offs


def tf32_forward(pkg, arena, H, L, k, x):
    params, params_u, offs = arena
    y = torch.empty((x.shape[0], 2 if k % 3 == 0 else 1), dtype=torch.float32, device="cuda")
    pkg._lib.check(pkg._lib.lib().rtd3_mlp_forward_tf32(H, L, 1 if k % 3 == 0 else 0, offs[k], pkg._lib.ptr(params), pkg._lib.ptr(params_u),
                                                        pkg._lib.ptr(x), pkg._lib.ptr(y), x.shape[0], pkg._lib.stream_ptr()))
    return y


def references(vs, f16=False):
    """float64 reference of each of the six networks on its input pool, cast to float32 (the cast is asserted exact)."""
    out = []
    for k, flat in enumerate(vs["nets"]):
        x, dims = (vs["xa"], vs["dims_a"]) if k % 3 == 0 else (vs["xc"], vs["dims_c"])
        ref = eg.forward64(flat, x, dims, f16=f16)
        assert np.array_equal(ref.astype(np.float32).astype(np.float64), ref)
        out.append(torch.from_numpy(ref.astype(np.float32)).cuda())
    return out


def batch(vs, k, B, rs, last=None):
    """B rows drawn from network k's input pool (row `last` of the pool at the end, if given) -> (x on the device, pool index)."""
    pool = vs["xa"] if k % 3 == 0 else vs["xc"]
    idx = rs.randint(0, pool.shape[0] - (last is not None), B)
    if last is not None:
        idx[-1] = last
    return torch.from_numpy(pool[idx]).cuda(), torch.from_numpy(idx).cuda()


def num_sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.mark.parametrize("L", (2, 3, 4))
@pytest.mark.parametrize("H", HS)
def test_tf32_and_fp32_forwards_equal_float64(pkg, H, L):
    """All six networks; B: a ragged last tile (129, 300), one 128-row tile per SM, one tile more than that (the first CTA takes a
    second tile), several tiles per CTA with a ragged last one.  The fp32 FFMA forward runs on the same rows through a TD3 object,
    at every shape but H = 256, L = 4, where its fp32 learner kernels do not fit in shared memory and TD3 refuses to build."""
    vs = eg.forward_set(H, L, SEED)
    arena = tf32_arena(pkg, vs, H, L)
    agent = agent_on_grid(pkg, vs, H, L) if (H, L) != (256, 4) else None
    refs = references(vs)
    n = num_sms() * 128
    rs = np.random.RandomState(H * 10 + L)
    for B in (129, 300, n, n + 1, 3 * n + 77):
        for k in range(6):
            x, idx = batch(vs, k, B, rs)
            out = tf32_forward(pkg, arena, H, L, k, x)
            assert torch.equal(out, refs[k][idx]), ("tf32", B, k, int((out != refs[k][idx]).any(1).sum()))
            if agent is not None:
                assert not agent._tc_ok(B)                                  # precision "fp32": the FFMA forward
                out = agent.forward(k, x)
                assert torch.equal(out, refs[k][idx]), ("fp32", B, k, int((out != refs[k][idx]).any(1).sum()))


@pytest.mark.parametrize("H", HS)
def test_f16_forward_equals_float64(pkg, H):
    """All six networks; B gives every CTA 1, 2 and 3 tiles (the second tile is the first use of the second TMEM accumulator
    buffer, the third reuses the first with its mbarrier phase flipped).  The last row drives one first-layer activation past
    65504: its expected output is the reference with that activation saturated at 65504, the kernel's conversion."""
    vs = eg.forward_set(H, 2, SEED, sat=True)
    agent = agent_on_grid(pkg, vs, H, 2)
    refs = references(vs, f16=True)
    n = num_sms() * 128
    rs = np.random.RandomState(H)
    sat_row = vs["xa"].shape[0] - 1
    agent.precision = "f16"
    for B in (n, 2 * n - 60, 3 * n - 1):
        for k in range(6):
            x, idx = batch(vs, k, B, rs, last=sat_row)
            assert agent._f16_ok(B)
            out = agent.forward(k, x)
            assert torch.equal(out, refs[k][idx]), (B, k, int((out != refs[k][idx]).any(1).sum()))


# ------------------------------------------------------------------------------------------------ learner
LEARNER_SEED = 4                              # tests/test_exact_grid.py checks these vector sets and what their batches cover


def exact32(x):
    """float64 reference -> float32 device tensor; the cast is asserted exact."""
    x = np.asarray(x, np.float64)
    assert np.array_equal(x.astype(np.float32).astype(np.float64), x)
    return torch.from_numpy(x.astype(np.float32)).cuda()


def learner_agent(pkg, ls, B, precision):
    """A 2-layer agent holding the six networks of `ls`, with the hyper-parameters the vectors are built for, critic_lr = 0 (so
    critic 1 is still on the grid when an update's actor step reads it) and its replay rows in a ring."""
    H = ls["H"]
    torch.manual_seed(0)
    agent = pkg.TD3(pkg.Residual_Actor_Network(H, 2), pkg.Residual_Critic_Network(H, 2), pkg.Residual_Critic_Network(H, 2), gamma=eg.GAMMA,
                    policy_noise=eg.POLICY_NOISE, noise_clip=eg.NOISE_CLIP, batch_size=B, critic_lr=0.0)
    assert agent.max_action == eg.MAX_ACTION
    for k in range(6):
        agent.flat(k).copy_(torch.from_numpy(ls["nets"][k]).cuda())
    agent.sync_transposed()
    agent.precision = precision
    agent.tc_min_batch = 1
    rb = pkg.ReplayBuffer(len(ls["s"]), seed=0)
    rb.push(*(torch.from_numpy(ls[k]).cuda() for k in ("s", "a", "r", "s2")), torch.from_numpy(ls["done"]).cuda())
    idx = torch.from_numpy(ls["idx"]).cuda()
    noise = torch.from_numpy(ls["noise"][ls["idx"]]).cuda()
    return agent, rb, idx, noise


def learner64(ls):
    return t64.Learner64(ls["nets"], hidden=ls["H"], layers=2, gamma=eg.GAMMA, policy_noise=eg.POLICY_NOISE, noise_clip=eg.NOISE_CLIP,
                         max_action=eg.MAX_ACTION)


@pytest.mark.parametrize("B", (32, 1024, 8192))
@pytest.mark.parametrize("H", (128, 256))
def test_critic_step_equals_float64(pkg, H, B):
    """TF32 (td3_critic_tc_kernel; B = 32 is one ragged 64-row tile) and fp32 critic steps: both losses, Q of both critics, the targets
    y and both critics' gradients equal the float64 reference; the actor's gradient slot stays exactly zero."""
    ls = eg.learner_set(H, B, LEARNER_SEED)
    s, a, r, s2, done, noise = eg.batch_rows(ls)
    ref = learner64(ls).critic_step(s, a, r, s2, done, noise)
    for prec in ("tf32", "fp32"):
        agent, rb, idx, noise_d = learner_agent(pkg, ls, B, prec)
        assert agent._tc_learner_ok(B) == (prec == "tf32")
        loss2 = torch.zeros(2, device="cuda")
        q = torch.zeros((2, B), device="cuda")
        y = torch.zeros((B,), device="cuda")
        agent.grads.zero_()
        agent._critic_step(rb, idx, noise_d, loss2, q, y, apply=False)
        torch.cuda.synchronize()
        assert torch.equal(y, exact32(ref["y"])), (prec, int((y != exact32(ref["y"])).sum()))
        assert torch.equal(q, exact32(ref["q"])), prec
        assert torch.equal(loss2, exact32(ref["loss"])), (prec, loss2.tolist(), ref["loss"])
        for c in (1, 2):
            g = agent.flat_grad(c)
            assert torch.equal(g, exact32(ref["g"][c - 1])), (prec, c, int((g != exact32(ref["g"][c - 1])).sum()))
        assert float(agent.grads[:agent._off[1]].abs().max()) == 0.0


@pytest.mark.parametrize("B", (32, 1024, 8192))
@pytest.mark.parametrize("H", (128, 256))
def test_actor_step_equals_float64(pkg, H, B):
    """TF32 (td3_actor_tc_kernel) and fp32 actor steps: the loss and the actor's gradient equal the float64 reference; the critics'
    gradient slots stay exactly zero.  Critic 2 is drawn on its own here, so that a step that read it would show."""
    ls = eg.learner_set(H, B, LEARNER_SEED, twin=False)
    ref = learner64(ls).actor_step(eg.batch_rows(ls)[0])
    for prec in ("tf32", "fp32"):
        agent, rb, idx, _ = learner_agent(pkg, ls, B, prec)
        assert agent._tc_learner_ok(B) == (prec == "tf32")
        loss1 = torch.zeros(1, device="cuda")
        agent.grads.zero_()
        agent._actor_step(rb, idx, loss1)
        torch.cuda.synchronize()
        assert float(loss1[0]) == ref["loss"], (prec, float(loss1[0]), ref["loss"])
        g = agent.flat_grad(0)
        assert torch.equal(g, exact32(ref["g"])), (prec, int((g != exact32(ref["g"])).sum()))
        assert float(agent.grads[agent._off[1]:].abs().max()) == 0.0


@pytest.mark.parametrize("use_graph", (True, False))
@pytest.mark.parametrize("prec,B", (("tf32", 1024), ("tf32", 8192), ("fp32", 256), ("fp32", 1024)))
def test_one_update_epoch_equals_the_oracle_optimiser_on_exact_gradients(pkg, prec, B, use_graph):
    """One epoch of td3_update (critic step + Adam on the critics with critic_lr = 0, actor step + Adam + the three Polyak updates):
    adam_m, adam_v, the new actor and the three targets equal oracle/td3_oracle.py's adam_step / soft_update applied to the float64
    gradients; the fp32 rows cover the fused (B <= 512) and the unfused optimiser."""
    H = 256
    ls = eg.learner_set(H, B, LEARNER_SEED)
    agent, rb, idx, noise = learner_agent(pkg, ls, B, prec)
    agent.num_epochs = 1
    assert agent._tc_learner_ok(B) == (prec == "tf32")
    s, a, r, s2, done, nz = eg.batch_rows(ls)
    ref64 = learner64(ls)
    gc = ref64.critic_step(s, a, r, s2, done, nz)["g"]
    ga = ref64.actor_step(s)["g"]
    agent.td3_update(rb, noise=noise[None], idx=torch.stack([idx, idx]), use_graph=use_graph)
    torch.cuda.synchronize()
    p = [np.array(n, np.float32) for n in ls["nets"]]
    for k, g in ((0, ga), (1, gc[0]), (2, gc[1])):
        g32 = exact32(g).cpu().numpy()
        st = to.AdamState(g32.size)
        to.adam_step(p[k], g32, st, lr=agent.actor_lr if k == 0 else 0.0)
        sl = slice(agent._off[k], agent._off[k] + agent._cnt[k])
        assert torch.equal(agent.adam_m[sl].cpu(), torch.from_numpy(st.m)), (k, "m")
        assert torch.equal(agent.adam_v[sl].cpu(), torch.from_numpy(st.v)), (k, "v")
    for k in (3, 4, 5):
        to.soft_update(p[k], p[k - 3], agent.tau)
    for k in range(6):
        assert torch.equal(agent.flat(k).cpu(), torch.from_numpy(p[k])), k
