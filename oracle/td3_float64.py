"""float64 reference of the residual-TD3 learner's gradients, with an elementwise magnitude bound.  TEST INFRASTRUCTURE.

The float32 kernels are checked against it elementwise: |g - g64| <= tau * M, where g64 is the float64 gradient (torch CPU autograd on
float64 copies of the float32 parameters and rows) and M is the same backward pass run on magnitudes:
  - the forward pass with |W|, |b| and |input| (`|z|_abs`), keeping the ReLU masks of the float64 forward;
  - the backward pass with |W|, those masks, the magnitude activations, and |dL/dout| bounded by
    (2/B)(|q|_abs + |y|_abs) for the critic losses and 1/B for the actor loss.
Every rounding error of a float32 forward / backward is a multiple of u times a term of that magnitude sum, so a correct float32
kernel stays within a small multiple of u*M, and an element with M == 0 (a unit no row activates, an input that is exactly 0) must
come out exactly 0.

The bound holds only where the float32 and float64 passes take the same ReLU branches.  `usable_rows` selects the replay rows on which
no pre-activation of a differentiated network lies within KINK_MARGIN * |z|_abs of zero (target networks are forward-only and
continuous, so their kinks do not matter).  For critic 1 in the actor step the margin uses |actor(s)| as the action's magnitude.

Follows robot.py:312-366 (critic step) and robot.py:369-398 (actor step) as oracle/td3_oracle.py does.  Parameter vectors are the
flat float32 arrays of td3_oracle (torch `parameters()` order).  `control` replaces the reference by a subtly wrong one, to show
that a bar rejects it:
  "drop_row"   the last batch row contributes nothing (the 1/B normalisation stays)
  "flip_done"  `done` of row 0 inverted                                       (critic step)
  "max_target" max instead of min of the twin target Q-values                 (critic step)
  "noise_unclipped"  the target-policy noise is not clipped to +-noise_clip  (critic step)
  "critic2"    the actor gradient taken through critic 2                     (actor step)
"""
import numpy as np
import torch

from .td3_oracle import layer_dims

KINK_MARGIN = 2.0 ** -16


def _t64(x):
    return torch.as_tensor(np.asarray(x, np.float32)).to(torch.float64)


def _forward(flat, x, dims):
    """float64 MLP forward -> (out, [pre-activations of the hidden layers], [layer inputs])."""
    zs, hs, off, h = [], [x], 0, x
    for li, (i, o) in enumerate(dims):
        W = flat[off:off + i * o].view(o, i)
        off += i * o
        b = flat[off:off + o]
        off += o
        z = h @ W.T + b
        if li == len(dims) - 1:
            return z, zs, hs
        zs.append(z)
        h = torch.relu(z)
        hs.append(h)


def _abs_forward(flat, x_abs, dims, zs):
    """The forward pass on magnitudes with the masks of the real pass -> (|out|_abs, [|z|_abs], [|layer input|_abs])."""
    fa = flat.abs()
    za, ha, off, h = [], [x_abs], 0, x_abs
    for li, (i, o) in enumerate(dims):
        W = fa[off:off + i * o].view(o, i)
        off += i * o
        b = fa[off:off + o]
        off += o
        z = h @ W.T + b
        if li == len(dims) - 1:
            return z, za, ha
        za.append(z)
        h = z * (zs[li] > 0)
        ha.append(h)


def _abs_backward(flat, dims, zs, ha, d):
    """The backward pass on magnitudes: |dL/dout| bound d [B,out] -> (M over the flat parameters, |dL/dinput| bound [B,in])."""
    fa = flat.abs()
    M = torch.zeros_like(flat)
    offs, off = [], 0
    for i, o in dims:
        offs.append(off)
        off += i * o + o
    for li in range(len(dims) - 1, -1, -1):
        i, o = dims[li]
        p = offs[li]
        M[p:p + i * o] = (d.T @ ha[li]).reshape(-1)
        M[p + i * o:p + i * o + o] = d.sum(0)
        d = d @ fa[p:p + i * o].view(o, i)
        if li > 0:
            d = d * (zs[li - 1] > 0)
    return M, d


def _near_kink(zs, za):
    """Rows with a pre-activation within KINK_MARGIN * |z|_abs of zero."""
    bad = torch.zeros(zs[0].shape[0], dtype=torch.bool)
    for z, a in zip(zs, za):
        bad |= (z.abs() <= KINK_MARGIN * a).any(1)
    return bad


class Learner64:
    """The six networks of one agent (actor, critic1, critic2, target actor, target critic1, target critic2) as float64 copies."""

    def __init__(self, nets, hidden, layers, gamma=0.99, policy_noise=0.2, noise_clip=0.5, max_action=5.0):
        self.nets = [_t64(n) for n in nets]
        self.H, self.L = hidden, layers
        self.adims = layer_dims(2, hidden, layers, 2)
        self.cdims = layer_dims(4, hidden, layers, 1)
        self.gamma, self.policy_noise, self.noise_clip, self.max_action = gamma, policy_noise, noise_clip, max_action

    # ---- kink-safe rows
    def usable_rows(self, s, a=None, step="critic"):
        """Rows whose differentiated networks keep every pre-activation out of the kink margin: critics 1 and 2 at (s, a) for the
        critic step, the actor at s and critic 1 at (s, actor(s)) for the actor step."""
        s = _t64(s)
        if step == "critic":
            x = torch.cat([s, _t64(a)], 1)
            bad = torch.zeros(s.shape[0], dtype=torch.bool)
            for c in (1, 2):
                _, zs, _ = _forward(self.nets[c], x, self.cdims)
                bad |= _near_kink(zs, _abs_forward(self.nets[c], x.abs(), self.cdims, zs)[1])
            return ~bad.numpy()
        act, zs, _ = _forward(self.nets[0], s, self.adims)
        bad = _near_kink(zs, _abs_forward(self.nets[0], s.abs(), self.adims, zs)[1])
        # critic 1's margin is taken from its own magnitudes at the action the actor gives, |actor(s)|, not from the actor's
        # magnitude sums: a deep untrained actor cancels so heavily (outputs ~100 from sums ~50 000) that those would exclude
        # every row
        x = torch.cat([s, act], 1)
        _, zc, _ = _forward(self.nets[1], x, self.cdims)
        bad |= _near_kink(zc, _abs_forward(self.nets[1], x.abs(), self.cdims, zc)[1])
        return ~bad.numpy()

    # ---- robot.py:312-366
    def critic_step(self, s, a, r, s2, done, noise, control=None):
        """-> dict: g [2][n] gradients of critics 1 and 2, M [2][n]; q [2][B], Mq; y [B], My; loss [2], Mloss (float64 numpy)."""
        s, a, s2, r = _t64(s), _t64(a), _t64(s2), _t64(r).reshape(-1, 1)
        done = np.asarray(done, bool).copy()
        if control == "flip_done":
            done[0] = not done[0]
        notdone = torch.as_tensor(1.0 - done.astype(np.float64)).reshape(-1, 1)
        B = s.shape[0]
        eps = _t64(noise) * self.policy_noise
        if control != "noise_unclipped":
            eps = eps.clamp(-self.noise_clip, self.noise_clip)
        ta, zt, _ = _forward(self.nets[3], s2, self.adims)
        ta_abs = _abs_forward(self.nets[3], s2.abs(), self.adims, zt)[0]
        na = (ta + eps).clamp(-self.max_action, self.max_action)
        na_abs = torch.minimum(ta_abs + eps.abs(), torch.full_like(ta_abs, self.max_action))
        xt, xt_abs = torch.cat([s2, na], 1), torch.cat([s2.abs(), na_abs], 1)
        qt, qt_abs = [], []
        for c in (4, 5):
            q, zs, _ = _forward(self.nets[c], xt, self.cdims)
            qt.append(q)
            qt_abs.append(_abs_forward(self.nets[c], xt_abs, self.cdims, zs)[0])
        tq = torch.maximum(*qt) if control == "max_target" else torch.minimum(*qt)
        y = r + self.gamma * tq * notdone
        y_abs = r.abs() + self.gamma * torch.maximum(*qt_abs) * notdone
        w = torch.ones((B, 1), dtype=torch.float64)
        if control == "drop_row":
            w[-1] = 0.0
        x = torch.cat([s, a], 1)
        out = {"g": [], "M": [], "q": [], "Mq": [], "loss": [], "Mloss": [], "y": y[:, 0].numpy(), "My": y_abs[:, 0].numpy()}
        for c in (1, 2):
            flat = self.nets[c].clone().requires_grad_(True)
            q, zs, _ = _forward(flat, x, self.cdims)
            loss = ((q - y) ** 2 * w).sum() / B                        # nn.MSELoss (mean) of robot.py:356 / 361
            loss.backward()
            q = q.detach()
            q_abs, _, ha = _abs_forward(self.nets[c], x.abs(), self.cdims, [z.detach() for z in zs])
            M, _ = _abs_backward(self.nets[c], self.cdims, [z.detach() for z in zs], ha, (2.0 / B) * (q_abs + y_abs))
            out["g"].append(flat.grad.numpy())
            out["M"].append(M.numpy())
            out["q"].append(q[:, 0].numpy())
            out["Mq"].append(q_abs[:, 0].numpy())
            out["loss"].append(float(loss.detach()))
            out["Mloss"].append(float(((q_abs + y_abs) ** 2).mean()))
        for k in ("g", "M", "q", "Mq"):
            out[k] = np.stack(out[k])
        out["loss"], out["Mloss"] = np.array(out["loss"]), np.array(out["Mloss"])
        return out

    # ---- robot.py:369-398
    def actor_step(self, s, control=None, critic=None):
        """-> dict: g [n] actor gradient, M; loss (= -mean Q), Mloss (= mean |Q|_abs).  `critic`: flat float32 critic 1 to differentiate
        through instead of this agent's (the one the actor step of an update reads after the critics' Adam step)."""
        s = _t64(s)
        B = s.shape[0]
        cnet = self.nets[2] if control == "critic2" else (self.nets[1] if critic is None else _t64(critic))
        flat = self.nets[0].clone().requires_grad_(True)
        act, za, _ = _forward(flat, s, self.adims)
        x = torch.cat([s, act], 1)
        q, zc, _ = _forward(cnet, x, self.cdims)
        w = torch.ones((B, 1), dtype=torch.float64)
        if control == "drop_row":
            w[-1] = 0.0
        loss = -(q * w).sum() / B
        loss.backward()
        za, zc = [z.detach() for z in za], [z.detach() for z in zc]
        act_abs, _, ha_a = _abs_forward(self.nets[0], s.abs(), self.adims, za)
        q_abs, _, ha_c = _abs_forward(cnet, torch.cat([s.abs(), act_abs.detach()], 1), self.cdims, zc)
        _, dx = _abs_backward(cnet, self.cdims, zc, ha_c, torch.full((B, 1), 1.0 / B, dtype=torch.float64))
        M, _ = _abs_backward(self.nets[0], self.adims, za, ha_a, dx[:, 2:4])
        return {"g": flat.grad.numpy(), "M": M.numpy(), "loss": float(loss.detach()), "Mloss": float(q_abs.mean())}


def draw_usable(rs, usable, B, dup=4):
    """B indices into the rows marked usable, drawn with replacement, the first `dup` of them repeated at the end of the batch (a
    minibatch may hold a row twice).  -> (idx int32 [B], fraction of rows excluded)."""
    pool = np.flatnonzero(usable)
    idx = rs.choice(pool, B, replace=True).astype(np.int32)
    k = min(dup, B // 2)
    if k:
        idx[B - k:] = idx[:k]
    return idx, 1.0 - usable.mean()
