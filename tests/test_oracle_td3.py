"""Pin oracle/td3_oracle.py (replay ring + TD3 learner restatement) against goldens from the unmodified reference.

Tolerance (BASELINE.json north_star): losses and Q-values within 1e-3 relative after one update; replay indices bit-exact.
Parameters: after one Adam step every element has moved by lr * m_hat / (sqrt(v_hat) + eps) ~ +-1e-5, so they are compared
on the update itself.
"""
import os

import numpy as np

from oracle import td3_oracle as to
from oracle.mt19937 import LegacyMT19937

REL = 1e-3


def make_agent(g, stage="w0"):
    return to.TD3Oracle(g[stage + "_actor"], g[stage + "_critic1"], g[stage + "_critic2"], g[stage + "_t_actor"],
                        g[stage + "_t_critic1"], g[stage + "_t_critic2"])


def make_replay(g):
    rb = to.ReplayOracle(10000)
    for k in range(g["rep_s"].shape[0]):
        rb.push(g["rep_s"][k], g["rep_a"][k], g["rep_r"][k], g["rep_s2"][k], g["rep_d"][k])
    return rb


def update_close(new, old, ref_new, ref_old, frac_ok=0.999):
    """The applied update (new-old) agrees with the reference's for >= frac_ok of the elements (near-zero gradients can
    flip the sign of Adam's normalised step), and no element is off by more than one full step (2 * lr)."""
    d, dr = (new - old).astype(np.float64), (ref_new - ref_old).astype(np.float64)
    assert np.abs(d - dr).max() <= 2.05e-5
    return (np.abs(d - dr) <= 2e-6).mean() >= frac_ok


def test_param_counts():
    assert to.param_count(2, 200, 3, 2) == 81402      # SURVEY.md a-6
    assert to.param_count(4, 200, 3, 1) == 81601


def test_replay_ring_and_indices(replay_golden):
    g = replay_golden
    rb = to.ReplayOracle(16)
    for k in range(40):
        rb.push(np.array([k, k]), np.array([k, -k]), float(k), np.array([k, k + 1]), False)
    assert (rb.s == g["ring_states"]).all() and rb.position == int(g["ring_position"]) and len(rb) == 16
    assert rb.sample_indices(LegacyMT19937(0), 17) is None and bool(g["under_filled_is_none"])
    ci = 0
    while "case_%d" % ci in g:
        n, B, seed = [int(v) for v in g["case_%d" % ci]]
        rng = LegacyMT19937(seed)
        rb = to.ReplayOracle(10000)
        for k in range(n):
            rb.push(np.array([k, 0.5]), np.array([1.0, k]), float(-k), np.array([k + 1, 0.25]), k % 50 == 49)
        for rep in range(3):
            idx = rb.sample_indices(rng, B)
            assert (idx == g["idx_%d" % ci][rep]).all()
        s, a, r, s2, d = rb.gather(idx)
        assert (s == g["rows_s_%d" % ci]).all() and (a == g["rows_a_%d" % ci]).all() and (r == g["rows_r_%d" % ci]).all()
        assert (s2 == g["rows_s2_%d" % ci]).all() and (d == g["rows_d_%d" % ci]).all()
        ci += 1
    assert ci == 5


def test_train_critic_one_step(td3_golden):
    g = td3_golden
    ag, rb = make_agent(g), make_replay(g)
    l1, l2 = ag.train_critic(*rb.gather(g["idx_critic"]), g["noise_critic"])
    np.testing.assert_allclose([l1, l2], g["critic_losses"], rtol=REL)
    assert update_close(ag.critic1, g["w0_critic1"], g["w1_critic1"], g["w0_critic1"])
    assert update_close(ag.critic2, g["w0_critic2"], g["w1_critic2"], g["w0_critic2"])
    s, a, _, _, _ = rb.gather(g["idx_critic"])
    q1, _ = to.critic_forward(ag.critic1, s, a)
    q2, _ = to.critic_forward(ag.critic2, s, a)
    np.testing.assert_allclose(q1, g["q1_after_critic"], rtol=REL, atol=1e-3)
    np.testing.assert_allclose(q2, g["q2_after_critic"], rtol=REL, atol=1e-3)
    # actor and targets untouched by the critic step
    assert (ag.actor == g["w1_actor"]).all() and (ag.t_critic1 == g["w1_t_critic1"]).all()


def test_train_actor_and_polyak(td3_golden):
    g = td3_golden
    ag, rb = make_agent(g, "w1"), make_replay(g)
    ag.opt_c1.t = ag.opt_c2.t = 1
    s, _, _, _, _ = rb.gather(g["idx_actor"])
    la = ag.train_actor(s)
    np.testing.assert_allclose(la, float(g["actor_loss"]), rtol=REL)
    assert update_close(ag.actor, g["w1_actor"], g["w2_actor"], g["w1_actor"])
    assert (ag.critic1 == g["w2_critic1"]).all()          # critic-1 gradients from the actor loss are discarded
    ag.polyak_all()
    for k in ("t_actor", "t_critic1", "t_critic2"):
        np.testing.assert_allclose(getattr(ag, k), g["w2_" + k], rtol=0, atol=3e-8)


def test_td3_update_six_epochs(td3_golden):
    g = td3_golden
    ag, rb = make_agent(g, "w2"), make_replay(g)
    # optimiser state carried over from the two previous steps: replay them instead of injecting moments
    ag = make_agent(g)
    ag.train_critic(*rb.gather(g["idx_critic"]), g["noise_critic"])
    ag.train_actor(rb.gather(g["idx_actor"])[0])
    ag.polyak_all()
    c_losses, a_losses = ag.td3_update(rb, list(g["upd_idx"]), list(g["upd_noise"]), 6)
    np.testing.assert_allclose(c_losses, g["upd_critic_losses"], rtol=REL)
    np.testing.assert_allclose(a_losses, g["upd_actor_losses"], rtol=REL)
    for k in ("actor", "critic1", "critic2"):
        np.testing.assert_allclose(getattr(ag, k), g["w3_" + k], rtol=0, atol=2.5e-5)
        assert (np.abs(getattr(ag, k) - g["w3_" + k]) <= 2e-6).mean() > 0.995
    for k in ("t_actor", "t_critic1", "t_critic2"):
        np.testing.assert_allclose(getattr(ag, k), g["w3_" + k], rtol=0, atol=1e-6)


def test_adam_step_bit_exact_vs_torch():
    """oracle adam_step == torch.optim.Adam on CPU, element for element over five steps (exp_avg, exp_avg_sq bit-exact; parameters
    bit-exact but for the rare element where torch's vectorised division rounds the other way: >= 99.99 %).  The CUDA kernels apply
    the same operation order (csrc/rtd3_td3.cuh: adam_element).  torch's results are the stored ones (tests/golden/make_golden.py
    adam): which kernels torch runs, and so how it rounds, depends on the CPU it runs on.  They are a sample of 2048 elements, too
    few for a rate of 1 in 10^4 in one step, so the rate is taken over the five steps together."""
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "adam_golden.npz"))
    st = to.AdamState(g["p0"].size)
    p = g["p0"].copy()
    equal = []
    for step in range(g["grad"].shape[0]):
        to.adam_step(p, g["grad"][step], st, lr=1e-3)
        assert (st.m == g["exp_avg"][step]).all()
        assert (st.v == g["exp_avg_sq"][step]).all()
        tp = g["param"][step]
        equal.append(p == tp)
        assert np.abs(p - tp).max() <= 2.4e-7 * max(1.0, float(np.abs(tp).max()))
        p[...] = tp                                      # continue from torch's parameters: the next step is again element-exact
    assert np.mean(equal) >= 0.9999
