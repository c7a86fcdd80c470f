"""The dyadic test vectors of oracle/exact_grid.py (CPU): the premise holds on every vector set tests/test_tc_exact_gpu.py uses, float32
evaluations in different summation orders equal the float64 reference there, and every structural mistake the GPU tests claim to
reject changes that reference (with bit equality, "changes the reference" is "rejected")."""
import numpy as np
import pytest

from oracle import exact_grid as eg
from oracle import td3_float64 as t64

HS = (64, 96, 128, 160, 192, 224, 256)
SEED = 11                                     # tests/test_tc_exact_gpu.py uses the same


def f32_forward(flat, x, dims, order, f16=False):
    """float32 forward, products summed either by numpy's float32 matmul ("matmul") or one column at a time from the last K to
    the first, bias last ("reverse")."""
    h = np.asarray(x, np.float32)
    layers = eg.unpack64(flat, dims)
    for li, (W, b) in enumerate(layers):
        W, b = W.astype(np.float32), b.astype(np.float32)
        if order == "matmul":
            z = h @ W.T + b
        else:
            z = np.zeros((h.shape[0], W.shape[0]), np.float32)
            for k in range(W.shape[1] - 1, -1, -1):
                z += h[:, k:k + 1] * W[:, k]
            z += b
        if li == len(layers) - 1:
            return z
        h = np.maximum(z, np.float32(0))
        if f16 and li == 0:
            h = np.minimum(h, np.float32(eg.FP16_MAX))


def sets():
    for H in HS:
        for L in (2, 3, 4):
            yield H, L, False
        yield H, 2, True


def nets_and_inputs(vs):
    for k, flat in enumerate(vs["nets"]):
        yield k, flat, (vs["xa"], vs["dims_a"]) if k % 3 == 0 else (vs["xc"], vs["dims_c"])


@pytest.mark.parametrize("H,L,sat", list(sets()))
def test_premise_holds_on_every_vector_set(H, L, sat):
    chk = eg.forward_premise(eg.forward_set(H, L, SEED, sat=sat), f16=sat)
    assert chk.failures == [], chk.failures[:5]


@pytest.mark.parametrize("H,L,sat", [(64, 4, False), (160, 3, False), (256, 2, False), (256, 4, False), (96, 2, True), (256, 2, True)])
def test_float32_in_two_orders_equals_float64(H, L, sat):
    vs = eg.forward_set(H, L, SEED, sat=sat)
    for k, flat, (x, dims) in nets_and_inputs(vs):
        ref = eg.forward64(flat, x, dims, f16=sat)
        for order in ("matmul", "reverse"):
            out = f32_forward(flat, x, dims, order, f16=sat).astype(np.float64)
            assert np.array_equal(out, ref), (k, order, np.abs(out - ref).max())


def test_the_saturation_row_saturates_one_unit_and_changes_the_output():
    vs = eg.forward_set(256, 2, SEED, sat=True)
    for k, flat, (x, dims) in nets_and_inputs(vs):
        (W0, b0), = eg.unpack64(flat, dims)[:1]
        z0 = x[-1].astype(np.float64) @ W0.T + b0
        assert (z0 > eg.FP16_MAX).sum() == 1
        unclamped = eg.forward64(flat, x[-1:], dims)
        assert not np.array_equal(unclamped, eg.forward64(flat, x[-1:], dims, f16=True))


def mutate(flat, dims, layer, what, arg=None):
    """A copy of `flat` with one structural mistake in layer `layer`: "bias" dropped, "kslab" = (k0, k1) K columns zeroed,
    "kswap" = (k0, k1) two K columns swapped."""
    m = np.asarray(flat, np.float64).copy()
    off = sum(i * o + o for i, o in dims[:layer])
    i, o = dims[layer]
    W = m[off:off + i * o].reshape(o, i)
    if what == "bias":
        m[off + i * o:off + i * o + o] = 0.0
    elif what == "kslab":
        W[:, arg[0]:arg[1]] = 0.0
    elif what == "kswap":
        W[:, [arg[0], arg[1]]] = W[:, [arg[1], arg[0]]]
    return m


@pytest.mark.parametrize("H,L,sat", [(64, 4, False), (96, 3, False), (160, 2, False), (256, 3, False), (128, 2, True), (256, 2, True)])
def test_every_mutation_changes_the_reference(H, L, sat):
    """Each mutation is a mistake a kernel could make: a dropped bias of any layer, a dropped K slab (16 columns: one f16 MMA's K; two
    of them are a TF32 MMA pair), the two halves of every packed pair of hidden inputs exchanged (pack_half2_sat), two adjacent
    4-column k-chunks of a hidden weight exchanged, output rows shifted by one."""
    vs = eg.forward_set(H, L, SEED, sat=sat)
    for k, flat, (x, dims) in nets_and_inputs(vs):
        ref = eg.forward64(flat, x, dims, f16=sat)
        changed = lambda m: not np.array_equal(eg.forward64(m, x, dims, f16=sat), ref)
        for layer in range(len(dims)):
            assert changed(mutate(flat, dims, layer, "bias")), (k, layer, "bias")
        for layer in range(1, len(dims) - 1):
            for k0 in range(0, H, 16):
                assert changed(mutate(flat, dims, layer, "kslab", (k0, k0 + 16))), (k, layer, "kslab", k0)
            m = np.asarray(flat, np.float64).copy()
            for k0 in range(0, H, 2):                                        # halves of every packed half2 exchanged
                m = mutate(m, dims, layer, "kswap", (k0, k0 + 1))
            assert changed(m), (k, layer, "pair swap")
            for k0 in range(0, H - 4, 4):
                m = mutate(mutate(mutate(mutate(flat, dims, layer, "kswap", (k0, k0 + 4)), dims, layer, "kswap", (k0 + 1, k0 + 5)),
                                  dims, layer, "kswap", (k0 + 2, k0 + 6)), dims, layer, "kswap", (k0 + 3, k0 + 7))
                assert changed(m), (k, layer, "kchunk swap", k0)
        assert (ref[1:] != ref[:-1]).any(axis=1).mean() > 0.9                     # a shifted output row is wrong on most rows


# ------------------------------------------------------------------------------------------------ learner

LEARNER_SEED = 4                                  # tests/test_tc_exact_gpu.py uses the same
LEARNER_SETS = [(H, B) for H in (128, 256) for B in (32, 1024, 8192)]


def learner64(ls, nets=None):
    return t64.Learner64(ls["nets"] if nets is None else nets, hidden=ls["H"], layers=2, gamma=eg.GAMMA, policy_noise=eg.POLICY_NOISE,
                         noise_clip=eg.NOISE_CLIP, max_action=eg.MAX_ACTION)


@pytest.mark.parametrize("H,B", LEARNER_SETS)
def test_learner_premise_holds_and_the_batch_covers_every_case(H, B):
    ls = eg.learner_set(H, B, LEARNER_SEED)
    chk = eg.learner_premise(ls)
    assert chk.failures == [], chk.failures[:5]
    cov = eg.coverage(ls)
    assert min(cov.values()) > 0, cov


@pytest.mark.parametrize("H,B", LEARNER_SETS)
def test_learner_premise_holds_on_the_actor_step_vectors(H, B):
    chk = eg.learner_premise(eg.learner_set(H, B, LEARNER_SEED, twin=False), critic_step=False)
    assert chk.failures == [], chk.failures[:5]


def critic_outputs(ref):
    return np.concatenate([ref["g"].reshape(-1), ref["q"].reshape(-1), ref["y"], ref["loss"]])


@pytest.mark.parametrize("H,B", [(128, 32), (256, 1024)])
def test_learner_reference_is_exact_in_float32_and_rejects_every_mutation(H, B):
    """The float64 reference's outputs are float32 values, and each mistake changes them: every control of Learner64, a dropped bias
    of each layer of each trained network, critics 1 and 2 swapped, a batch row shifted by one."""
    ls = eg.learner_set(H, B, LEARNER_SEED)
    s, a, r, s2, done, noise = eg.batch_rows(ls)
    L64 = learner64(ls)
    ref_c = critic_outputs(L64.critic_step(s, a, r, s2, done, noise))
    ref_a = L64.actor_step(s)
    for v in (ref_c, ref_a["g"], np.array([ref_a["loss"]])):
        assert np.array_equal(v.astype(np.float32).astype(np.float64), v)
    for control in ("drop_row", "flip_done", "max_target", "noise_unclipped"):
        assert not np.array_equal(critic_outputs(L64.critic_step(s, a, r, s2, done, noise, control=control)), ref_c), control
    assert not np.array_equal(L64.actor_step(s, control="drop_row")["g"], ref_a["g"])
    # critic 2 is critic 1 permuted: the actor gradient through it is the same, so the actor step's vectors draw their own critic 2
    la = eg.learner_set(H, B, LEARNER_SEED, twin=False)
    assert not np.array_equal(learner64(la).actor_step(s, control="critic2")["g"], learner64(la).actor_step(s)["g"])
    la_swapped = [la["nets"][k] for k in (0, 2, 1, 3, 4, 5)]
    assert not np.array_equal(learner64(la, la_swapped).actor_step(s)["g"], learner64(la).actor_step(s)["g"])
    swapped = [ls["nets"][k] for k in (0, 2, 1, 3, 4, 5)]
    assert not np.array_equal(critic_outputs(learner64(ls, swapped).critic_step(s, a, r, s2, done, noise)), ref_c)
    dims = {0: eg.layer_dims(2, H, 2, 2), 1: eg.layer_dims(4, H, 2, 1), 2: eg.layer_dims(4, H, 2, 1)}
    for k in (0, 1, 2):
        for layer in range(3):
            nets = list(ls["nets"])
            nets[k] = mutate(nets[k], dims[k], layer, "bias").astype(np.float32)
            m = learner64(ls, nets)
            changed = (not np.array_equal(m.actor_step(s)["g"], ref_a["g"])) if k == 0 else \
                not np.array_equal(critic_outputs(m.critic_step(s, a, r, s2, done, noise)), ref_c)
            assert changed, (k, layer)
    shift = lambda v: np.roll(v, 1, axis=0)
    assert not np.array_equal(critic_outputs(L64.critic_step(shift(s), shift(a), shift(r), shift(s2), shift(done), shift(noise))), ref_c)
