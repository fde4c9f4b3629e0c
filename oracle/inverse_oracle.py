"""CPU oracle of the Brenier map's left inverse (csrc/inverse.cu).  TEST INFRASTRUCTURE ONLY (same rules as icnn_oracle.py,
on which it builds): the product path never imports it.

z* = T^{-1}(x) for T = grad(psi + kappa|.|^2) is the minimiser of f(z) = psi(z) + kappa|z|^2 - <x, z>; its gradient is
xhat(z) - x and, with the LeakyReLU masks fixed, its Hessian is jacobian_oracle.icnn_jacobian.  `newton_step` is the step
kernel's state machine written out per row in fp64 on the kernel's state layout (the [N_FIELDS, B] fp64 arrays that follow
the state's 256-byte header), so that the kernel can be checked one step at a time; `brenier_inverse` runs the same
machine to convergence on the fp64 oracle (trial points kept in fp64 instead of being rounded to the fp32 points the
kernels evaluate)."""
from __future__ import annotations

import math

import numpy as np

from . import icnn_oracle as io
from . import jacobian_oracle as jo

ACTIVE, CONVERGED, MAXITER, STALLED, SINGULAR, NONFINITE = range(6)     # B200VAE_INV_*
MAX_HALVINGS, ETA, PIVOT_REL = 12, 0.5, 1e-12
MAX_D = 4
F_Z, F_P = 0, 4
F_T, F_LO, F_HI, F_PHI0, F_TOL, F_RNORM, F_STATUS, F_NSTEP, F_NHALF, F_CROSSED = range(8, 18)
N_FIELDS = 18
HEADER_BYTES = 256


def state_bytes(B):
    return HEADER_BYTES + N_FIELDS * B * 8


def _f32(v):
    return float(np.float32(v))


def _f64(v):
    return float(v)


def _isfinite(*vals):
    return all(math.isfinite(v) for v in vals)


def _newton_dir(J, r):
    """Cholesky solve of J p = -r (J [d][d] lists); None when a pivot is <= PIVOT_REL * max diag or not finite."""
    d = len(r)
    dmax = 0.0
    for i in range(d):
        dmax = max(dmax, J[i][i]) if not math.isnan(J[i][i]) else dmax
    L = [[0.0] * d for _ in range(d)]
    for j in range(d):
        s = J[j][j]
        for k in range(j):
            s -= L[j][k] * L[j][k]
        if not (s > PIVOT_REL * dmax):
            return None
        L[j][j] = math.sqrt(s)
        for i in range(j + 1, d):
            u = J[i][j]
            for k in range(j):
                u -= L[i][k] * L[j][k]
            L[i][j] = u / L[j][j]
    y = [0.0] * d
    for i in range(d):
        u = -r[i]
        for k in range(i):
            u -= L[i][k] * y[k]
        y[i] = u / L[i][i]
    p = [0.0] * d
    for i in reversed(range(d)):
        u = y[i]
        for k in range(i + 1, d):
            u -= L[k][i] * p[k]
        p[i] = u / L[i][i]
    return p


def _norm(v):
    return math.sqrt(sum(a * a for a in v))


def _accept(s, t, r, J, rnd):
    """The kernel's accept(): move to the evaluated point z + t p (t = 0: z itself), then the next direction."""
    if t != 0.0:
        s["z"] = [rnd(z + t * p) for z, p in zip(s["z"], s["p"])]
        s["nstep"] += 1.0
        s["crossed"] = 0.0
    s["rnorm"] = _norm(r)
    if s["rnorm"] <= s["tol"]:
        s["status"] = CONVERGED
        return
    if not (_isfinite(s["rnorm"]) and all(_isfinite(*row) for row in J)):
        s["status"] = NONFINITE
        return
    p = _newton_dir(J, r)
    if p is None:
        s["status"] = SINGULAR
        return
    s["p"] = p
    s["phi0"] = sum(a * b for a, b in zip(r, p))
    s["t"], s["lo"], s["hi"], s["nhalf"] = 1.0, 0.0, 1.0, 0.0


def init(x, z0=None, tol_rel=1e-5, tol_abs=1e-5, rnd=_f32):
    """b200vae_brenier_inverse_init: x [B,d] -> (rows [N_FIELDS,B] fp64, trial [B,d], z [B,d], status [B], err [B])."""
    x = np.asarray(x, dtype=np.float64)
    B, d = x.shape
    z0 = np.zeros((B, d)) if z0 is None else np.asarray(z0, dtype=np.float64)
    rows = np.zeros((N_FIELDS, B))
    fin = np.isfinite(x).all(1) & np.isfinite(z0).all(1)
    rows[F_Z:F_Z + d] = z0.T
    rows[F_HI] = 1.0
    xn = np.sqrt((x * x).sum(1))
    rows[F_TOL] = tol_rel * xn + tol_abs
    rows[F_RNORM] = np.inf
    rows[F_STATUS] = np.where(fin, ACTIVE, NONFINITE)
    trial = np.where(fin[:, None], z0, 0.0)
    return rows, trial, z0.copy(), rows[F_STATUS].astype(np.int32), np.full(B, np.inf)


def newton_step(rows, x, xhat, jac, kappa, final=False, rnd=_f32):
    """One launch of the step kernel: rows [N_FIELDS,B] (not modified), target x [B,d], xhat [B,d] and jac [B,d,d] at the
    rows' trial points -> (rows', trial [B,d], z [B,d], status [B], err [B], active).  rnd rounds a trial point: fp32 like
    the kernel, or identity (_f64) for an all-fp64 solve."""
    rows = np.array(rows, dtype=np.float64, copy=True)
    x, xhat, jac = (np.asarray(a, dtype=np.float64) for a in (x, xhat, jac))
    B, d = x.shape
    trial, z = np.zeros((B, d)), np.zeros((B, d))
    status, err = np.zeros(B, dtype=np.int32), np.zeros(B)
    active = 0
    for b in range(B):
        col = rows[:, b]
        s = dict(z=list(col[F_Z:F_Z + d]), p=list(col[F_P:F_P + d]), t=col[F_T], lo=col[F_LO], hi=col[F_HI],
                 phi0=col[F_PHI0], tol=col[F_TOL], rnorm=col[F_RNORM], status=int(col[F_STATUS]), nstep=col[F_NSTEP],
                 nhalf=col[F_NHALF], crossed=col[F_CROSSED])
        if s["status"] != ACTIVE:     # the kernel leaves a finished row's outputs alone; here they restate its state
            trial[b], z[b], status[b] = col[F_Z:F_Z + d], col[F_Z:F_Z + d], s["status"]
            err[b] = s["rnorm"] / (2.0 * kappa) if kappa > 0 else np.inf
            continue
        r = [float(xhat[b, i]) - float(x[b, i]) for i in range(d)]
        J = [[float(jac[b, i, k]) for k in range(d)] for i in range(d)]
        fin = _isfinite(*r) and all(_isfinite(*row) for row in J)
        if s["t"] == 0.0:
            _accept(s, 0.0, r, J, rnd)
        elif s["crossed"] == 2.0:   # the evaluation at a kink crossing z + hi p: it becomes z
            if fin:
                _accept(s, s["t"], r, J, rnd)
                s["crossed"] = 1.0
            else:
                s["status"] = STALLED
        else:
            bisect = True
            if not fin:
                s["hi"] = s["t"]
            else:
                ph = sum(a * c for a, c in zip(r, s["p"]))
                if _norm(r) <= s["tol"] or (ph <= 0.0 and (s["t"] == 1.0 or ph >= -ETA * abs(s["phi0"]))):
                    _accept(s, s["t"], r, J, rnd)
                    bisect = False
                elif ph <= 0.0:
                    s["lo"] = s["t"]
                else:
                    s["hi"] = s["t"]
            if bisect:
                s["nhalf"] += 1.0
                if s["nhalf"] <= MAX_HALVINGS:
                    s["t"] = 0.5 * (s["lo"] + s["hi"])
                elif s["lo"] == 0.0 and s["crossed"] == 1.0:
                    s["status"] = STALLED
                else:           # cross the kink: the next trial point is z + hi p
                    s["t"] = s["hi"]
                    s["crossed"] = 2.0
        zt = [rnd(zz + s["t"] * pp) for zz, pp in zip(s["z"], s["p"])]
        if s["status"] == ACTIVE and zt == [rnd(zz) for zz in s["z"]]:
            s["status"] = STALLED
        if s["status"] == ACTIVE and final:
            s["status"] = MAXITER
        act = s["status"] == ACTIVE
        trial[b] = zt if act else s["z"]
        z[b] = s["z"]
        col[F_Z:F_Z + d], col[F_P:F_P + d] = s["z"], s["p"]
        col[F_T], col[F_LO], col[F_HI], col[F_PHI0], col[F_RNORM] = s["t"], s["lo"], s["hi"], s["phi0"], s["rnorm"]
        col[F_STATUS], col[F_NSTEP], col[F_NHALF], col[F_CROSSED] = s["status"], s["nstep"], s["nhalf"], s["crossed"]
        status[b] = s["status"]
        err[b] = s["rnorm"] / (2.0 * kappa) if kappa > 0 else np.inf
        active += act
    return rows, trial, z, status, err, active


def brenier_inverse(x, p, mode=io.MODE_EXP, kappa=0.0, z0=None, max_iter=400, tol_rel=1e-13, tol_abs=1e-13):
    """The whole solve in fp64 on icnn_oracle / jacobian_oracle -> (z [B,d], status [B], err_bound [B], rounds)."""
    rows, trial, z, status, err = init(x, z0, tol_rel, tol_abs, rnd=_f64)
    for k in range(max_iter):
        xhat = io.icnn_brenier(trial, p, mode, kappa)[1]
        J = jo.icnn_jacobian(trial, p, mode, kappa)
        rows, trial, z, status, err, active = newton_step(rows, x, xhat, J, kappa, final=(k == max_iter - 1), rnd=_f64)
        if active == 0:
            return z, status, err, k + 1
    return z, status, err, max_iter
