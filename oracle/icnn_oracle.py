"""CPU oracle for the ICNN / Brenier-map hot path.  TEST INFRASTRUCTURE ONLY.

This file is a plain-numpy restatement of the reference algorithm.  Only
``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline /
``--impl reference`` legs may import it; the product path
(``vae_song_b200``) never does and fails loudly without its CUDA library.

Parity pinning: the reference ships no tests or golden vectors for this path
(SURVEY.md section 4), so the oracle is pinned against outputs of the reference
itself: ``oracle/make_golden.py`` imports ``{module,model,utils}.py`` of a
reference checkout (``oracle/fetch_ref.find_reference``) unmodified and writes the fixtures
under ``tests/golden/`` which ``tests/test_oracle_golden.py`` checks this file
against (fp64: <=1e-12 relative; fp32 fixtures: fp32 noise floor).

Reference lines restated here:
  * PositiveLinear   module.py:97-114   (exp / clamp(min=1e-2) weight reparam)
  * ICNN.forward     module.py:142-148  (LeakyReLU(0.2), first layer squared)
  * LIDVAE.decode    model.py:818-830   (two autograd.grad Brenier maps + eye(Dx,D) pad)
  * the autograd double-backward of the above (implicit in lipschitz.py:41)

Parameter dict keys (all numpy arrays, dtype = compute dtype):
  A0w [H,d] A0b [H]        <- ICNN.A0.weight / .bias
  A1w [H,d] A1b [H]        <- ICNN.A[0].weight / .bias
  A2w [1,d] A2b [1]        <- ICNN.A[1].weight / .bias
  W0  [H,H]                <- ICNN.W[0].param   (raw, pre-reparam)
  W1  [1,H]                <- ICNN.W[1].param
"""
from __future__ import annotations

import numpy as np

SLOPE = 0.2          # module.py:122  LeakyReLU(0.2)
CLAMP_MIN = 1e-2     # module.py:114
MODE_EXP, MODE_CLAMP = 0, 1

PARAM_KEYS = ("A0w", "A0b", "A1w", "A1b", "A2w", "A2b", "W0", "W1")


def positive(W, mode=MODE_EXP):
    """module.py:110 / :114."""
    if mode == MODE_EXP:
        return np.exp(W)
    return np.maximum(W, W.dtype.type(CLAMP_MIN))


def positive_chain(dP, W, P, mode=MODE_EXP):
    """d/dW of positive(): exp -> dP*P ; clamp -> dP*[W >= 1e-2] (aten clamp_backward)."""
    if mode == MODE_EXP:
        return dP * P
    return dP * (W >= W.dtype.type(CLAMP_MIN))


def _slope(h):
    # torch leaky_relu(_backward): x > 0 ? 1 : negative_slope   (0 takes the 0.2 branch)
    return np.where(h > 0, h.dtype.type(1.0), h.dtype.type(SLOPE))


def random_params(rng, d, H, dtype=np.float64, regime="default"):
    """Seeded ICNN parameters drawn with numpy only (so tests can rebuild them on any box).

    regime="default": PyTorch-default-like ranges (U(+-1/sqrt(fan_in)); exp(W)~1 -> huge outputs,
                      SURVEY.md section 7 'huge dynamic range').
    regime="mixed":   trained-like: small positive weights, wide biases -> LeakyReLU masks of both
                      signs in every layer, O(1) outputs.  This is the regime that exercises kinks.
    """
    u = lambda lo, hi, *s: rng.uniform(lo, hi, size=s)
    if regime == "default":
        bd, bh = 1.0 / np.sqrt(d), 1.0 / np.sqrt(H)
        p = dict(A0w=u(-bd, bd, H, d), A0b=u(-bd, bd, H), A1w=u(-bd, bd, H, d), A1b=u(-bd, bd, H),
                 A2w=u(-bd, bd, 1, d), A2b=u(-bd, bd, 1), W0=u(-bh, bh, H, H), W1=u(-1, 1, 1, H) * bh)
    elif regime == "mixed":
        p = dict(A0w=rng.normal(0, 0.7, (H, d)), A0b=rng.normal(0, 0.5, H),
                 A1w=rng.normal(0, 1.0, (H, d)), A1b=rng.normal(-0.3, 1.0, H),
                 A2w=rng.normal(0, 1.0, (1, d)), A2b=rng.normal(0, 0.5, 1),
                 W0=rng.normal(np.log(1.0 / H), 1.0, (H, H)), W1=rng.normal(np.log(2.0 / H), 1.0, (1, H)))
    elif regime == "clampy":  # raw weights straddling the 1e-2 clamp (is_exp=False path)
        p = dict(A0w=rng.normal(0, 0.7, (H, d)), A0b=rng.normal(0, 0.5, H),
                 A1w=rng.normal(0, 1.0, (H, d)), A1b=rng.normal(-0.5, 1.0, H),
                 A2w=rng.normal(0, 1.0, (1, d)), A2b=rng.normal(0, 0.5, 1),
                 W0=rng.normal(0.01, 0.02, (H, H)), W1=rng.normal(0.01, 0.02, (1, H)))
    else:
        raise ValueError(regime)
    return {k: np.ascontiguousarray(v, dtype=dtype) for k, v in p.items()}


def cast_params(p, dtype):
    return {k: np.ascontiguousarray(v, dtype=dtype) for k, v in p.items()}


def icnn_brenier(z, p, mode=MODE_EXP, kappa=0.0, keep=False, masks=None):
    """psi(z) [B] and xhat = grad_z(psi(z) + kappa*|z|^2) [B,d]   (SURVEY.md Appendix A).

    Forward  module.py:142-148; reverse = what autograd.grad(psi, z, ones) evaluates (model.py:822).
    Returns (psi, xhat, aux) where aux holds the masks (and, if keep, every intermediate).

    masks=(mask1 [B,H] bool, mask2 [B] bool): evaluate the REVERSE sweep with these LeakyReLU branch choices for h1 / h2
    instead of the signs of this evaluation's own pre-activations (the forward value psi is continuous across a kink and
    keeps its own).  Given the masks xhat is linear in everything else, so a kernel whose pre-activation landed on the
    other side of a kink within its rounding error can be checked exactly against "the oracle with the kernel's masks"."""
    dt = z.dtype.type
    P0, P1 = positive(p["W0"], mode), positive(p["W1"], mode)[0]
    h0 = z @ p["A0w"].T + p["A0b"]
    s0 = _slope(h0)
    a0 = h0 * s0
    x1 = a0 * a0
    h1 = x1 @ P0.T + z @ p["A1w"].T + p["A1b"]
    s1 = _slope(h1)
    x2 = h1 * s1
    h2 = x2 @ P1 + z @ p["A2w"][0] + p["A2b"][0]
    s2 = _slope(h2)
    psi = h2 * s2
    if masks is not None:
        s1 = np.where(np.asarray(masks[0], dtype=bool), dt(1.0), dt(SLOPE))
        s2 = np.where(np.asarray(masks[1], dtype=bool), dt(1.0), dt(SLOPE))
    g1 = (s2[:, None] * P1[None, :]) * s1
    gx1 = g1 @ P0
    g0 = gx1 * (dt(2.0) * a0 * s0)
    xhat = g0 @ p["A0w"] + g1 @ p["A1w"] + s2[:, None] * p["A2w"] + dt(2.0 * kappa) * z
    aux = dict(mask1=(h1 > 0), mask2=(h2 > 0), h1=h1, h2=h2)
    if keep:
        aux.update(P0=P0, P1=P1, h0=h0, s0=s0, a0=a0, x1=x1, s1=s1, x2=x2, s2=s2, g1=g1, gx1=gx1, g0=g0)
    return psi, xhat, aux


def icnn_brenier_backward(z, v, p, mode=MODE_EXP, kappa=0.0, gpsi=None, masks=None):
    """Gradients of  L = <v, xhat(z)> (+ <gpsi, psi(z)>)  w.r.t. z and every parameter.

    This is what PyTorch's double-backward through autograd.grad(create_graph=True) produces
    (model.py:822/828 then lipschitz.py:41).  Masks are constants a.e.; A1b/A2b get exact zeros
    on the <v,xhat> path.  Returns (dz [B,d], grads dict keyed like the params).
    masks: see icnn_brenier (the LeakyReLU branch choices of h1 / h2 are then given, not derived)."""
    dt = z.dtype.type
    psi, xhat, a = icnn_brenier(z, p, mode, kappa, keep=True, masks=masks)
    P0, P1, s0, a0, s1, s2, g1, gx1, g0 = (a[k] for k in ("P0", "P1", "s0", "a0", "s1", "s2", "g1", "gx1", "g0"))
    u0 = v @ p["A0w"].T
    u1 = v @ p["A1w"].T
    q1 = u0 * (dt(2.0) * a0 * s0)
    t0 = u0 * (dt(2.0) * gx1 * s0 * s0)
    w1 = u1 + q1 @ P0.T
    g = {}
    g["A0w"] = g0.T @ v + t0.T @ z
    g["A0b"] = t0.sum(0)
    g["A1w"] = g1.T @ v
    g["A1b"] = np.zeros_like(p["A1b"])
    g["A2w"] = (s2[:, None] * v).sum(0, keepdims=True)
    g["A2b"] = np.zeros_like(p["A2b"])
    dP0 = g1.T @ q1
    dP1 = (s2[:, None] * s1 * w1).sum(0)
    dz = t0 @ p["A0w"] + dt(2.0 * kappa) * v
    if gpsi is not None:
        # ordinary first-order backward of psi weighted by gpsi (SURVEY Appendix A last line)
        w = gpsi
        dh2 = w * s2
        dh1 = w[:, None] * g1
        dh0 = w[:, None] * g0
        g["A2w"] = g["A2w"] + (dh2[:, None] * z).sum(0, keepdims=True)
        g["A2b"] = g["A2b"] + dh2.sum(keepdims=True)
        dP1 = dP1 + (dh2[:, None] * a["x2"]).sum(0)
        g["A1w"] = g["A1w"] + dh1.T @ z
        g["A1b"] = g["A1b"] + dh1.sum(0)
        dP0 = dP0 + dh1.T @ a["x1"]
        g["A0w"] = g["A0w"] + dh0.T @ z
        g["A0b"] = g["A0b"] + dh0.sum(0)
        dz = dz + w[:, None] * (xhat - dt(2.0 * kappa) * z)
    g["W0"] = positive_chain(dP0, p["W0"], P0, mode)
    g["W1"] = positive_chain(dP1[None, :], p["W1"], P1[None, :], mode)
    return dz, g


def pad_eye(x1, Dx):
    """x = x1 @ eye(Dx, D).T  (model.py:771-774, :824): zero-pad D -> Dx columns."""
    B, D = x1.shape
    if Dx == D:
        return x1
    out = np.zeros((B, Dx), dtype=x1.dtype)
    out[:, :D] = x1
    return out


def lidvae_decode(z, p0, p1, Dx, mode=MODE_EXP, kappa=0.0):
    """LIDVAE.decode model.py:818-830 -> (y [B,Dx], x1 [B,D], psi0, psi1)."""
    psi0, x1, _ = icnn_brenier(z, p0, mode, kappa)
    x = pad_eye(x1, Dx)
    psi1, y, _ = icnn_brenier(x, p1, mode, kappa)
    return y, x1, psi0, psi1


def lidvae_decode_backward(z, vy, p0, p1, Dx, mode=MODE_EXP, kappa=0.0):
    """Chain of the two double-backwards: dL/dy -> (dz, grads ICNN0, grads ICNN1)."""
    _, x1, _ = icnn_brenier(z, p0, mode, kappa)
    x = pad_eye(x1, Dx)
    dx, g1 = icnn_brenier_backward(x, vy, p1, mode, kappa)
    v1 = np.ascontiguousarray(dx[:, : z.shape[1]])
    dz, g0 = icnn_brenier_backward(z, v1, p0, mode, kappa)
    return dz, g0, g1


# ----------------------------------------------------------------------------- FLOP model
def flops_decode(d, H):
    """SURVEY.md section 8(d): F_dec(d,H) = 4H^2 + 8dH + 2H + 4d per sample (multiply-add = 2)."""
    return 4 * H * H + 8 * d * H + 2 * H + 4 * d


def flops_train(d, H):
    """SURVEY.md section 8(d): F_train(d,H) = 8H^2 + 22dH per sample."""
    return 8 * H * H + 22 * d * H
