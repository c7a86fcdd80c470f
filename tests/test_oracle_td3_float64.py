"""Pin oracle/td3_float64.py (float64 learner gradients + magnitude bound M) to the float32 oracle and check the bound itself.

- On the reference's golden weights and rows (tests/golden/td3_golden.npz), the float32 oracle's gradients, Q-values, targets and
  losses (td3_oracle.mlp_backward / train_critic / train_actor) agree with the float64 reference within 2^-12 * M.
- The bound is an upper bound of the error a float32 pass can make: on a tiny net, perturbing every float32 input (all six networks,
  the replay rows and the noise) in its last bit moves the float64 gradient by at most 2^-20 * M.
- Every control of the reference (a subtly wrong learner) moves the gradient by more than the device tests' bar.
"""
import numpy as np
import pytest

from oracle import td3_float64 as t64
from oracle import td3_oracle as to

F32 = np.float32
BAR = 2.0 ** -12


def golden_rows(g, key):
    idx = g[key]
    return g["rep_s"][idx], g["rep_a"][idx], g["rep_r"][idx], g["rep_s2"][idx], g["rep_d"][idx]


def within(x, ref, M, bar):
    x, ref, M = np.asarray(x, np.float64), np.asarray(ref, np.float64), np.asarray(M, np.float64)
    return float((np.abs(x - ref) / np.where(M > 0, M, 1.0)).max()), bool((x[M == 0] == 0).all())


def test_critic_step_vs_float32_oracle(td3_golden):
    g = td3_golden
    nets = [g["w0_" + k] for k in ("actor", "critic1", "critic2", "t_actor", "t_critic1", "t_critic2")]
    ref = t64.Learner64(nets, 200, 3)
    s, a, r, s2, d = golden_rows(g, "idx_critic")
    out = ref.critic_step(s, a, r, s2, d, g["noise_critic"])
    orc = to.TD3Oracle(*nets)
    losses = orc.train_critic(s, a, r, s2, d, g["noise_critic"])             # float32 targets (y) and losses
    y32 = orc.last_targets[:, 0]
    assert within(y32, out["y"], out["My"], BAR)[0] <= BAR
    assert within(losses, out["loss"], out["Mloss"], BAR)[0] <= BAR
    B = s.shape[0]
    for c in (0, 1):
        q32, acts = to.critic_forward(nets[1 + c], s, a)
        g32, _ = to.mlp_backward(nets[1 + c], acts, F32(2.0 / B) * (q32 - orc.last_targets), 4, 200, 3, 1)
        err, zeros = within(g32, out["g"][c], out["M"][c], BAR)
        assert err <= BAR and zeros, (c, err)
        assert within(q32[:, 0], out["q"][c], out["Mq"][c], BAR)[0] <= BAR
        assert (np.abs(out["g"][c]) <= out["M"][c] * (1 + 1e-12)).all()      # the bound bounds the gradient itself
    np.testing.assert_allclose(out["loss"], g["critic_losses"], rtol=1e-3)   # and the reference's own losses


def test_actor_step_vs_float32_oracle(td3_golden):
    g = td3_golden
    nets = [g["w1_" + k] for k in ("actor", "critic1", "critic2", "t_actor", "t_critic1", "t_critic2")]
    ref = t64.Learner64(nets, 200, 3)
    s = golden_rows(g, "idx_actor")[0]
    out = ref.actor_step(s)
    B = s.shape[0]
    act, a_acts = to.actor_forward(nets[0], s)
    q, c_acts = to.critic_forward(nets[1], s, act)
    _, dx = to.mlp_backward(nets[1], c_acts, np.full_like(q, F32(-1.0 / B)), 4, 200, 3, 1)
    g32, _ = to.mlp_backward(nets[0], a_acts, dx[:, 2:4], 2, 200, 3, 2)
    err, zeros = within(g32, out["g"], out["M"], BAR)
    assert err <= BAR and zeros, err
    assert abs(float(-np.mean(q, dtype=F32)) - out["loss"]) <= BAR * out["Mloss"]
    np.testing.assert_allclose(out["loss"], float(g["actor_loss"]), rtol=1e-3)


def test_usable_rows_exclude_a_minority(td3_golden):
    """The kink margin costs rows in proportion to the number of pre-activations checked: on the golden 3 x 200 networks (1200
    pre-activations per row) it excludes 39 % of the rows for the critic step and 32 % for the actor step."""
    g = td3_golden
    nets = [g["w0_" + k] for k in ("actor", "critic1", "critic2", "t_actor", "t_critic1", "t_critic2")]
    for step in ("critic", "actor"):
        u = t64.Learner64(nets, 200, 3).usable_rows(g["rep_s"], g["rep_a"], step)
        assert 0.2 < 1.0 - u.mean() < 0.5, (step, 1.0 - u.mean())


def ulp_perturbed(rs, x):
    x = np.asarray(x, F32)
    return np.where(rs.randint(0, 2, x.shape) == 1, np.nextafter(x, F32(np.inf)), np.nextafter(x, F32(-np.inf))).astype(F32)


@pytest.mark.parametrize("layers", [1, 2])
def test_magnitude_bound_covers_last_bit_perturbations(layers):
    H, B = 4, 3
    rs = np.random.RandomState(11 + layers)
    nets = []
    for k in range(6):
        i, o = (2, 2) if k % 3 == 0 else (4, 1)
        nets.append(to.kaiming_uniform_params(rs, i, H, layers, o) + rs.normal(0, 0.05, to.param_count(i, H, layers, o)).astype(F32))
    n = 64
    s = rs.uniform(0, 10, (n, 2)).astype(F32)
    a = rs.uniform(-5, 5, (n, 2)).astype(F32)
    r = rs.uniform(-50, 0, n).astype(F32)
    s2 = (s + 0.1 * a).astype(F32)
    d = np.arange(n) % 3 == 1
    noise = rs.normal(size=(B, 2)).astype(F32)
    ref = t64.Learner64(nets, H, layers)
    idx_c, _ = t64.draw_usable(rs, ref.usable_rows(s, a, "critic"), B, dup=1)
    idx_a, _ = t64.draw_usable(rs, ref.usable_rows(s, a, "actor"), B, dup=1)
    base_c = ref.critic_step(s[idx_c], a[idx_c], r[idx_c], s2[idx_c], d[idx_c], noise)
    base_a = ref.actor_step(s[idx_a])
    worst = 0.0
    for trial in range(50):
        pn = [ulp_perturbed(rs, x) for x in nets]
        p = t64.Learner64(pn, H, layers)
        c = p.critic_step(ulp_perturbed(rs, s[idx_c]), ulp_perturbed(rs, a[idx_c]), ulp_perturbed(rs, r[idx_c]), ulp_perturbed(rs, s2[idx_c]),
                          d[idx_c], ulp_perturbed(rs, noise))
        ac = p.actor_step(ulp_perturbed(rs, s[idx_a]))
        for x, x0, M in ((c["g"], base_c["g"], base_c["M"]), (c["q"], base_c["q"], base_c["Mq"]), (c["y"], base_c["y"], base_c["My"]),
                         (ac["g"], base_a["g"], base_a["M"])):
            err, _ = within(x, x0, M, 1.0)
            worst = max(worst, err)
    assert 0.0 < worst <= 2.0 ** -20, worst


def test_controls_move_the_reference_beyond_the_bar(td3_golden):
    """Each wrong reference differs from the right one by more than 2^-14 * M somewhere, far above the device tests' fp32 bar
    (2^-21).  (Not the
    unclipped-noise control: the golden target actor's outputs, ~100, are clipped to +-max_action whatever the noise; the device tests
    scale the actor's head to keep them inside.)  The dropped row is the
    closest call, 1.3e-4 * M: the untrained golden critics cancel heavily, so M is large against the gradient itself."""
    g = td3_golden
    nets = [g["w0_" + k] for k in ("actor", "critic1", "critic2", "t_actor", "t_critic1", "t_critic2")]
    ref = t64.Learner64(nets, 200, 3)
    rows = golden_rows(g, "idx_critic")
    base = ref.critic_step(*rows, g["noise_critic"])
    for control in ("drop_row", "flip_done", "max_target"):
        out = ref.critic_step(*rows, g["noise_critic"], control=control)
        assert max(within(out["g"][c], base["g"][c], base["M"][c], 1)[0] for c in (0, 1)) > 2.0 ** -14, control
    s = golden_rows(g, "idx_actor")[0]
    base = ref.actor_step(s)
    for control in ("drop_row", "critic2"):
        assert within(ref.actor_step(s, control=control)["g"], base["g"], base["M"], 1)[0] > 2.0 ** -14, control
