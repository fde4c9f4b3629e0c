"""CPU oracle of the Brenier map's exact Jacobian and of the decoder's chain.  TEST INFRASTRUCTURE ONLY (same rules as
icnn_oracle.py, on which it builds): the product path never imports it.

With the LeakyReLU masks fixed the Brenier map x = grad(psi + kappa|z|^2) is affine in z (SURVEY.md Appendix A), so its
Jacobian is exact and closed-form; LIDVAE.decode (model.py:818-830) composes two such maps through x = x1 . M^T.
"""
from __future__ import annotations

import numpy as np

from . import icnn_oracle as io


def icnn_jacobian(z, p, mode=io.MODE_EXP, kappa=0.0, masks=None):
    """d xhat / d z [B,d,d] of icnn_oracle.icnn_brenier: with the LeakyReLU masks fixed xhat is affine in z (gx1 depends on the masks
    only, g0 = gx1 * 2 h0 s0^2), so  J = A0^T diag(2 s0^2 gx1) A0 + 2 kappa I.  `masks` as in icnn_oracle.icnn_brenier; s0 comes from
    this evaluation's h0 (0 takes the 0.2 branch, like torch's leaky_relu_backward)."""
    _, _, a = io.icnn_brenier(z, p, mode, kappa, keep=True, masks=masks)
    w = z.dtype.type(2.0) * a["s0"] * a["s0"] * a["gx1"]
    J = np.einsum("hi,bh,hj->bij", p["A0w"], w, p["A0w"])
    return J + z.dtype.type(2.0 * kappa) * np.eye(z.shape[1], dtype=z.dtype)[None]


def lidvae_decode_jacobian(z, p0, p1, Dx, mode=io.MODE_EXP, kappa=0.0, M=None, masks0=None, masks1=None):
    """Jacobian of icnn_oracle.lidvae_decode (with x = x1 @ M.T; M = eye(Dx, D) by default): J = J2(x) . M . J1(z) -> (J [B,Dx,D],
    J1 [B,D,D], J2 [B,Dx,Dx])."""
    D = z.shape[1]
    M = np.eye(Dx, D, dtype=z.dtype) if M is None else np.asarray(M, dtype=z.dtype)
    _, x1, _ = io.icnn_brenier(z, p0, mode, kappa, masks=masks0)
    J1 = icnn_jacobian(z, p0, mode, kappa, masks=masks0)
    x = x1 @ M.T
    J2 = icnn_jacobian(x, p1, mode, kappa, masks=masks1)
    return J2 @ M @ J1, J1, J2
