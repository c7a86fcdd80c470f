"""Dyadic test vectors on which the tensor-core kernels (forwards and TF32 learner) have nothing to round.  TEST INFRASTRUCTURE (never
imported by the package).

The TF32 and f16 forwards (rtd3_tc.cu: mlp_forward_tc_kernel, mlp_forward_f16_kernel and its hf_* pieces) round their operands and
sum in an order of their own.  On the vectors built here neither matters, so a correct kernel returns the float64 result bit for bit
and the tests compare with `torch.equal`.  The vectors satisfy, on every product a kernel forms:

  1. every tensor-core operand (hidden-layer input X and hidden weight W) has at most 11 significant bits, which TF32 and fp16 hold
     exactly; for fp16 it is also 0 or of magnitude in [2^-14, 65504];
  2. all terms of a dot product (bias included) are multiples of one quantum q and sum(|terms|) < 2^21 q, so every partial sum, in
     any order, is a multiple of q that fp32 holds exactly (3 bits of margin for the tensor-core accumulator's alignment);
  3. no pre-activation is exactly 0, so the ReLU-at-zero convention does not enter.

How the grid keeps these: inputs are small integers, first-layer weights are in {-1, 0, 1}, hidden rows have `nnz` entries of +-1
(so an activation grows by a few bits per layer, not by log2(H)), and the bias of layer l is an odd multiple of 2^-(l+2): half the
quantum of the product it is added to, which makes every pre-activation non-zero.  Output weights are in {0, +-1/2, +-1}.

`Premise` checks conditions 1-3 from the data and returns the failures instead of asserting, so that generators can be tuned
against it.  `forward64` is the float64 reference; with `f16=True` the first-layer activations saturate at 65504 as the f16
kernel's `cvt.rn.satfinite` conversion does.

The learner vectors (`learner_set`, layers == 2) follow the same rules with a bit budget for the backward pass: critic 2 is a
hidden-unit permutation of critic 1 with its output bias moved by 2 Q_QUANTUM, r is solved so that y = Q1 - delta with a 3-bit delta,
the critics' output weights are all +-1/4 and the actor's two output rows read disjoint pairs of hidden units.  `learner_premise`
checks every product of the critic and actor steps: dZ.W and dZ^T.H on the tensor cores (2^21), and the column sums, batch
reductions and loss sums that run as plain fp32 adds (2^24: no accumulator alignment there).  The reference is
oracle/td3_float64.Learner64 with GAMMA, POLICY_NOISE, NOISE_CLIP below.

Parameter vectors are flat float32 arrays in torch `parameters()` order, as in oracle/td3_oracle.py.
"""
import numpy as np

from .td3_oracle import layer_dims

BUDGET = 2.0 ** 21                 # sum(|terms|) / q of every dot product
SUM_BUDGET = 2.0 ** 24             # ... of a plain fp32 sum (FFMA chains, shuffles, L2 reduce-adds, atomicAdd) that the learner's loss
                                   # reductions alone may use: no accumulator alignment, only fp32's 24-bit significand
OPERAND_BITS = 11                  # significand of TF32 and fp16 (10 stored bits + the implicit one)
FP16_MAX = 65504.0
FP16_MIN_NORMAL = 2.0 ** -14
SAT_INPUT = 4096.0                 # input 0 of the saturation row: 16 * 4096 + b > 65504 on the saturating unit


def lowbit(x):
    """The largest power of two dividing each entry of the dyadic array x (inf where x == 0)."""
    x = np.abs(np.asarray(x, np.float64))
    m, e = np.frexp(x)
    mi = (m * 2.0 ** 53).astype(np.int64)
    lb = np.ldexp((mi & -mi).astype(np.float64), e - 53)
    return np.where(x == 0, np.inf, lb)


def sig_bits(x):
    """Significant bits of each entry of the dyadic array x (0 for 0)."""
    x = np.abs(np.asarray(x, np.float64))
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(x == 0, 1.0, x / lowbit(x))
    return np.where(x == 0, 0, np.floor(np.log2(r)).astype(np.int64) + 1)


class Premise:
    """Conditions 1-3 on named operands and products; `failures` lists what does not hold."""

    def __init__(self):
        self.failures = []
        self.worst = 0.0              # largest sum(|terms|) / q seen, as a fraction of BUDGET

    def operand(self, name, x, f16=False):
        x = np.asarray(x, np.float64)
        bits = int(sig_bits(x).max(initial=0))
        if bits > OPERAND_BITS:
            self.failures.append("%s: %d significant bits" % (name, bits))
        if f16:
            a = np.abs(x[x != 0])
            if a.size and (a.min() < FP16_MIN_NORMAL or a.max() > FP16_MAX):
                self.failures.append("%s: outside the fp16 normal range (%g .. %g)" % (name, a.min(), a.max()))

    def dot(self, name, A, B, bias=None, budget=BUDGET):
        """The products A [M,K] @ B [K,N] (+ bias [N]).  The quantum of element (i, j) is taken as the finest entry of row i of A
        times the finest entry of column j of B (and the bias's own), a common divisor of all its terms."""
        A, B = np.asarray(A, np.float64), np.asarray(B, np.float64)
        qa = lowbit(A).min(axis=1, initial=np.inf)[:, None]
        qb = lowbit(B).min(axis=0, initial=np.inf)[None, :]
        with np.errstate(invalid="ignore"):
            q = qa * qb
        mag = np.abs(A) @ np.abs(B)
        if bias is not None:
            bias = np.asarray(bias, np.float64)
            q = np.minimum(q, lowbit(bias)[None, :])
            mag = mag + np.abs(bias)[None, :]
        with np.errstate(invalid="ignore", divide="ignore"):
            ratio = np.where(mag == 0, 0.0, mag / q)
        worst = float(ratio.max(initial=0.0))
        self.worst = max(self.worst, worst / budget)
        if not worst < budget:
            self.failures.append("%s: sum|terms|/q = 2^%.2f" % (name, np.log2(worst)))

    def nonzero(self, name, z):
        n = int((np.asarray(z) == 0).sum())
        if n:
            self.failures.append("%s: %d pre-activations are exactly 0" % (name, n))

    def exact32(self, name, x):
        x = np.asarray(x, np.float64)
        if not np.array_equal(x.astype(np.float32).astype(np.float64), x):
            self.failures.append("%s: not exact in float32" % name)


def unpack64(flat, dims):
    out, off = [], 0
    flat = np.asarray(flat, np.float64)
    for i, o in dims:
        W = flat[off:off + i * o].reshape(o, i)
        off += i * o
        out.append((W, flat[off:off + o]))
        off += o
    return out


def forward64(flat, x, dims, f16=False, chk=None, name="net"):
    """float64 forward of the MLP `dims` (ReLU between layers) on x [B,in] -> [B,out].  f16: the first-layer activations saturate at
    65504 (the f16 kernel's conversion) and the hidden operands must lie in fp16's range.  chk: a Premise that receives every
    operand and product the kernels form."""
    h = np.asarray(x, np.float64)
    layers = unpack64(flat, dims)
    for li, (W, b) in enumerate(layers):
        if chk is not None:
            chk.exact32("%s input %d" % (name, li), h)
            if 0 < li < len(layers) - 1:
                chk.operand("%s X%d" % (name, li), h, f16)
                chk.operand("%s W%d" % (name, li), W, f16)
            chk.dot("%s layer %d" % (name, li), h, W.T, b)
        z = h @ W.T + b
        if li == len(layers) - 1:
            if chk is not None:
                chk.exact32("%s output" % name, z)
            return z
        if chk is not None:
            chk.nonzero("%s z%d" % (name, li), z)
        h = np.maximum(z, 0.0)
        if f16 and li == 0:
            h = np.minimum(h, FP16_MAX)


def grid_net(rs, in_dim, H, L, out_dim, nnz=3, sat_unit=None):
    """One network on the grid -> flat float32.  sat_unit: hidden unit whose first-layer weight on input 0 is 16 while every other
    unit's is -1 or 0, so that an input row (SAT_INPUT, 0, ...) drives exactly that unit past fp16's 65504 and no other unit off
    the fp16 grid (the other units see b or a negative pre-activation)."""
    parts = []
    for li, (i, o) in enumerate(layer_dims(in_dim, H, L, out_dim)):
        if li == 0:
            W = rs.randint(-1, 2, (o, i)).astype(np.float64)
            if sat_unit is not None:
                W[:, 0] = -rs.randint(0, 2, o)
                W[sat_unit, 0] = 16.0
            b = (2 * rs.randint(-4, 4, o) + 1) / 4.0
        elif li < L:
            W = np.zeros((o, i))
            for n in range(o):
                cols = rs.choice(i, nnz, replace=False)
                if sat_unit is not None and li == 1:
                    cols = cols[cols != sat_unit]
                W[n, cols] = rs.choice([-1.0, 1.0], cols.size)
            if sat_unit is not None and li == 1:
                W[rs.randint(o), sat_unit] = 1.0        # the saturated unit feeds one hidden unit
            b = (2 * rs.randint(-8, 8, o) + 1) * 2.0 ** -(li + 2)
        else:
            W = rs.choice([-1.0, -0.5, 0.0, 0.5, 1.0], (o, i))
            b = (2 * rs.randint(-4, 4, o) + 1) / 8.0
        parts += [W.reshape(-1), b]
    return np.concatenate(parts).astype(np.float32)


def grid_inputs(rs, n, in_dim, lo=-4, hi=4):
    """n input rows of small integers (a pool the tests index into; the reference runs on the pool only)."""
    return rs.randint(lo, hi + 1, (n, in_dim)).astype(np.float32)


def forward_set(H, L, seed, pool=512, sat=False):
    """The vectors of the forward tests: the six networks of one agent (actor, critic1, critic2, target actor, target critic1,
    target critic2), an actor input pool and a critic input pool.  sat: every network saturates unit 0 on the row pool[-1]
    = (SAT_INPUT, 0, ...) (fp16 forward only, layers == 2).  -> dict(nets, xa, xc, dims_a, dims_c)."""
    rs = np.random.RandomState(seed)
    nnz = 3 if L <= 3 else 2
    su = 0 if sat else None
    nets = [grid_net(rs, 2 if k % 3 == 0 else 4, H, L, 2 if k % 3 == 0 else 1, nnz, su) for k in range(6)]
    xa, xc = grid_inputs(rs, pool, 2), grid_inputs(rs, pool, 4)
    if sat:
        xa[-1] = 0.0
        xc[-1] = 0.0
        xa[-1, 0] = xc[-1, 0] = SAT_INPUT
    return {"nets": nets, "xa": xa, "xc": xc, "dims_a": layer_dims(2, H, L, 2), "dims_c": layer_dims(4, H, L, 1)}


def forward_premise(vs, f16=False):
    """Conditions 1-3 on every product of the six forwards of a forward_set -> Premise."""
    chk = Premise()
    for k, flat in enumerate(vs["nets"]):
        x, dims = (vs["xa"], vs["dims_a"]) if k % 3 == 0 else (vs["xc"], vs["dims_c"])
        chk.exact32("net %d weights" % k, flat.astype(np.float64))
        forward64(flat, x, dims, f16=f16, chk=chk, name="net %d" % k)
    return chk


# ------------------------------------------------------------------------------------------------ learner (layers == 2)
# The hyper-parameters the learner vectors are built for (pass the same to TD3(...) and td3_float64.Learner64): gamma and
# policy_noise are powers of two, so the target and the smoothing noise stay on the grid.
GAMMA, POLICY_NOISE, NOISE_CLIP, MAX_ACTION = 0.5, 0.25, 0.5, 5.0
Q_QUANTUM = 2.0 ** -6              # quantum of every critic output: h1 (1/16) times the output weights (+-1/4)


def _learner_net(rs, in_dim, H, out_dim, b0_den, action_nnz=None, head=None):
    """One 2-layer network of the learner vectors.  First layer: state columns in {-1, 0, 1}; a critic's action columns carry
    `action_nnz` entries of +-1 each (sparse, so the action gradient dA stays within 11 bits); biases odd multiples of 1/b0_den.
    Hidden layer: 3 entries of +-1 per row, biases odd multiples of half the product's quantum.  Head: the actor's two output rows
    read disjoint pairs of hidden units with weights +-1 (`head` = the four units); a critic's output weights are all +-1/4."""
    W0 = rs.randint(-1, 2, (H, in_dim)).astype(np.float64)
    if in_dim == 4:
        W0[:, 2:] = 0.0
        for j in (2, 3):
            W0[rs.choice(H, action_nnz, replace=False), j] = rs.choice([-1.0, 1.0], action_nnz)
    b0 = (2 * rs.randint(-2, 2, H) + 1) / b0_den
    W1 = np.zeros((H, H))
    for n in range(H):
        W1[n, rs.choice(H, 3, replace=False)] = rs.choice([-1.0, 1.0], 3)
    b1 = (2 * rs.randint(-4, 4, H) + 1) / (2.0 * b0_den)
    if out_dim == 2:
        Wo = np.zeros((2, H))
        Wo[0, head[:2]] = rs.choice([-1.0, 1.0], 2)
        Wo[1, head[2:]] = rs.choice([-1.0, 1.0], 2)
        bo = rs.randint(-4, 5, 2) / 4.0
    else:
        Wo = rs.choice([-0.25, 0.25], (1, H))
        bo = rs.randint(-8, 9, 1) / 8.0
    return np.concatenate([W0.reshape(-1), b0, W1.reshape(-1), b1, Wo.reshape(-1), bo]).astype(np.float32)


def permute_critic(flat, H, perm, bo_shift):
    """The same critic with its hidden units of both layers permuted and the output bias moved by bo_shift: the same Q + bo_shift on
    every input, with a different weight layout (so a mix-up of two critics' gradients shows)."""
    (W0, b0), (W1, b1), (Wo, bo) = unpack64(flat, layer_dims(4, H, 2, 1))
    parts = [W0[perm], b0[perm], W1[perm][:, perm], b1[perm], Wo[:, perm], bo + bo_shift]
    return np.concatenate([p.reshape(-1) for p in parts]).astype(np.float32)


def learner_set(H, B, seed, rows=600, twin=True):
    """The vectors of the learner tests: the six networks, `rows` replay rows (s, a, r, s2, done), a batch idx [B] with duplicates
    and, per replay row, the unit normal the critic step reads for it (noise[b] = row_noise[idx[b]], so that every occurrence of a
    row has the same target).  Critic 2 is a hidden-unit permutation of critic 1 with bo + 2^-5, so Q2 = Q1 + 2 Q_QUANTUM; r is
    solved per row so that y = Q1(s, a) - delta, delta in {-2..2} Q_QUANTUM: every Q - y then has at most 3 bits.
    twin=False: critic 2 is drawn on its own instead (for the actor step, which must not read it: as a permutation of critic 1
    it would give the same action gradient; the critic step then leaves the grid).  -> dict(H, nets, s, a, r, s2, done, idx, noise)."""
    rs = np.random.RandomState(seed)
    head = rs.choice(H, 4, replace=False)
    actor = _learner_net(rs, 2, H, 2, 2.0, head=head)
    t_actor = _learner_net(rs, 2, H, 2, 2.0, head=rs.choice(H, 4, replace=False))
    critic1 = _learner_net(rs, 4, H, 1, 8.0, action_nnz=4)
    critic2 = permute_critic(critic1, H, rs.permutation(H), 2 * Q_QUANTUM)
    if not twin:
        critic2 = _learner_net(np.random.RandomState(seed + 1), 4, H, 1, 8.0, action_nnz=4)
    t_critic1, t_critic2 = (_learner_net(rs, 4, H, 1, 8.0, action_nnz=4) for _ in range(2))
    nets = [actor, critic1, critic2, t_actor, t_critic1, t_critic2]
    s = rs.randint(-2, 3, (rows, 2)).astype(np.float64)
    a = rs.randint(-5, 6, (rows, 2)).astype(np.float64)
    s2 = rs.randint(-2, 3, (rows, 2)).astype(np.float64)
    done = rs.rand(rows) < 0.15
    noise = rs.randint(-4, 5, (rows, 2)).astype(np.float64)      # |0.25 z| > noise_clip for |z| >= 3
    dims_a, dims_c = layer_dims(2, H, 2, 2), layer_dims(4, H, 2, 1)
    q1 = forward64(critic1, np.concatenate([s, a], 1), dims_c)[:, 0]
    na = np.clip(forward64(t_actor, s2, dims_a) + np.clip(POLICY_NOISE * noise, -NOISE_CLIP, NOISE_CLIP), -MAX_ACTION, MAX_ACTION)
    xt = np.concatenate([s2, na], 1)
    tq = np.minimum(forward64(t_critic1, xt, dims_c), forward64(t_critic2, xt, dims_c))[:, 0]
    delta = rs.randint(-2, 3, rows) * Q_QUANTUM
    r = q1 - delta - GAMMA * tq * (~done)
    idx = rs.randint(0, rows, B).astype(np.int32)
    idx[B - min(4, B // 2):] = idx[:min(4, B // 2)]                # duplicate rows
    f = lambda v: v.astype(np.float32)
    return {"H": H, "nets": nets, "s": f(s), "a": f(a), "r": f(r), "s2": f(s2), "done": done, "idx": idx, "noise": f(noise)}


def batch_rows(ls):
    """The batch of a learner_set as the kernels read it: (s, a, r, s2, done, noise) [B, ...]."""
    i = ls["idx"]
    return ls["s"][i], ls["a"][i], ls["r"][i], ls["s2"][i], ls["done"][i], ls["noise"][i]


def _fwd(chk, name, flat, x, dims):
    """Forward with every product checked; the learner rounds both hidden activations to TF32 -> (out, h0, h1, z0, z1)."""
    (W0, b0), (W1, b1), (Wo, bo) = unpack64(flat, dims)
    chk.exact32(name + " input", x)
    chk.dot(name + " layer 0", x, W0.T, b0)
    z0 = x @ W0.T + b0
    chk.nonzero(name + " z0", z0)
    h0 = np.maximum(z0, 0)
    chk.operand(name + " h0", h0)
    chk.operand(name + " W1", W1)
    chk.dot(name + " hidden", h0, W1.T, b1)
    z1 = h0 @ W1.T + b1
    chk.nonzero(name + " z1", z1)
    h1 = np.maximum(z1, 0)
    chk.operand(name + " h1", h1)
    chk.dot(name + " output", h1, Wo.T, bo)
    out = h1 @ Wo.T + bo
    chk.exact32(name + " output", out)
    return out, h0, h1


def _bwd(chk, name, flat, x, h0, h1, dout, dims):
    """Backward of a 2-layer net from dL/dout [B,out], every product the kernels form checked: the output-layer sums, dZ1 (a TF32
    operand), dW1 = dZ1^T H0 over the whole batch (tensor cores per 64-row tile, then L2 reduce-adds), dH0 = dZ1 W1, dZ0 (a TF32
    operand) and the first-layer column sums."""
    (W0, _), (W1, _), (Wo, _) = unpack64(flat, dims)
    chk.dot(name + " gWout", dout.T, h1, budget=SUM_BUDGET)
    chk.dot(name + " gbout", dout.T, np.ones((dout.shape[0], 1)), budget=SUM_BUDGET)
    chk.dot(name + " dZ1", dout, Wo)
    dz1 = (dout @ Wo) * (h1 > 0)
    chk.operand(name + " dZ1", dz1)
    chk.dot(name + " gb1", dz1.T, np.ones((dz1.shape[0], 1)), budget=SUM_BUDGET)
    chk.dot(name + " dW1", dz1.T, h0)
    chk.dot(name + " dH0", dz1, W1)
    dz0 = (dz1 @ W1) * (h0 > 0)
    chk.operand(name + " dZ0", dz0)
    chk.dot(name + " gW0", dz0.T, x, budget=SUM_BUDGET)
    chk.dot(name + " gb0", dz0.T, np.ones((dz0.shape[0], 1)), budget=SUM_BUDGET)
    return dz0 @ W0


def _critic_premise(chk, ls, dims_c, dims_a, s, a, r, s2, done, noise):
    nets, B = ls["nets"], s.shape[0]
    ta = _fwd(chk, "target actor", nets[3], s2, dims_a)[0]
    na = np.clip(ta + np.clip(POLICY_NOISE * noise, -NOISE_CLIP, NOISE_CLIP), -MAX_ACTION, MAX_ACTION)
    xt = np.concatenate([s2, na], 1)
    tq = np.minimum(_fwd(chk, "target critic 1", nets[4], xt, dims_c)[0], _fwd(chk, "target critic 2", nets[5], xt, dims_c)[0])
    chk.exact32("r", r)
    y = r[:, None] + GAMMA * tq * (1.0 - done[:, None])
    chk.exact32("y", y)
    x = np.concatenate([s, a], 1)
    for c in (1, 2):
        q, h0, h1 = _fwd(chk, "critic %d" % c, nets[c], x, dims_c)
        diff = q - y
        chk.dot("critic %d loss" % c, (diff * diff / B).T, np.ones((B, 1)), budget=SUM_BUDGET)
        _bwd(chk, "critic %d" % c, nets[c], x, h0, h1, 2.0 * diff / B, dims_c)


def learner_premise(ls, critic_step=True):
    """Conditions 1-3 on every product of the critic step (unless critic_step=False) and the actor step on a learner_set (the TF32
    kernels' dataflow: rtd3_tc_learner.cu) -> Premise."""
    chk = Premise()
    H = ls["H"]
    dims_a, dims_c = layer_dims(2, H, 2, 2), layer_dims(4, H, 2, 1)
    s, a, r, s2, done, noise = (np.asarray(v, np.float64) for v in batch_rows(ls))
    B = s.shape[0]
    nets = ls["nets"]
    if critic_step:
        _critic_premise(chk, ls, dims_c, dims_a, s, a, r, s2, done, noise)
    # actor step
    act, h0a, h1a = _fwd(chk, "actor", nets[0], s, dims_a)
    xc = np.concatenate([s, act], 1)
    q, h0c, h1c = _fwd(chk, "critic 1 (actor step)", nets[1], xc, dims_c)
    chk.dot("actor loss", (q / B).T, np.ones((B, 1)), budget=SUM_BUDGET)
    (W0c, _), (W1c, _), (Woc, _) = unpack64(nets[1], dims_c)
    dout = np.full((B, 1), -1.0 / B)
    dz1c = (dout @ Woc) * (h1c > 0)
    chk.operand("critic 1 dZ1 (actor step)", dz1c)
    chk.dot("critic 1 dH0 (actor step)", dz1c, W1c)
    g = (dz1c @ W1c) * (h0c > 0)
    chk.dot("dA", g, W0c[:, 2:], budget=SUM_BUDGET)
    _bwd(chk, "actor", nets[0], s, h0a, h1a, g @ W0c[:, 2:], dims_a)
    return chk


def coverage(ls):
    """What the batch of a learner_set exercises: counts of done rows, rows with Q1' > Q2' and Q1' < Q2', rows where the noise clip
    acts, rows where the +-max_action clip acts, rows whose target action is inside the clip, duplicate rows."""
    H = ls["H"]
    dims_a, dims_c = layer_dims(2, H, 2, 2), layer_dims(4, H, 2, 1)
    s, a, r, s2, done, noise = (np.asarray(v, np.float64) for v in batch_rows(ls))
    ta = forward64(ls["nets"][3], s2, dims_a)
    e = POLICY_NOISE * noise
    pre = ta + np.clip(e, -NOISE_CLIP, NOISE_CLIP)
    xt = np.concatenate([s2, np.clip(pre, -MAX_ACTION, MAX_ACTION)], 1)
    q1, q2 = (forward64(ls["nets"][k], xt, dims_c)[:, 0] for k in (4, 5))
    return {"done": int(done.sum()), "q1>q2": int((q1 > q2).sum()), "q1<q2": int((q1 < q2).sum()),
            "noise_clip": int((np.abs(e) > NOISE_CLIP).any(1).sum()), "max_clip": int((np.abs(pre) > MAX_ACTION).any(1).sum()),
            "inside": int((np.abs(pre) < MAX_ACTION).all(1).sum()), "duplicates": int(len(ls["idx"]) - len(np.unique(ls["idx"])))}
