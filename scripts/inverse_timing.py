#!/usr/bin/env python
"""Cost and convergence of the Brenier map's Newton left inverse (ops.icnn_brenier_inverse, LIDVAE.decode_inverse)
-> profiles/r06_inverse.json.

    python scripts/inverse_timing.py [--out profiles/r06_inverse.json] [--reps 5]

(a) one ICNN (d = 2, H = 512 / 1024, B = 5000 / 65536, every precision, utils.trained_like_icnn_ weights, round-trip
    targets x = T(z_true), kappa = 0.1): rounds per row (histogram of the rows' last active round), status counts, the whole
    inverse, time per round against b200vae_icnn_decode_jac alone (the step kernel's share), and the step kernel alone
    on a fresh state (every row active, every row takes a Cholesky);
(b) LIDVAE.decode_inverse on the toy decoder (ICNN(2,512) + ICNN(2,1024), inverse_lipschitz 0.2), B = 5000 / 65536,
    against Newton's method in PyTorch eager -- decode with autograd, D backward passes for the Jacobian,
    torch.linalg.solve, full steps: one iteration, and the whole loop from z = 0 to the same tolerance (at most 100
    iterations; timed once, its iteration count and converged fraction reported).
CUDA events around each call, median; every timed call is preceded by a 512 MB write that evicts the 126 MB L2; every shape
is warmed up first.  The card's name and power limit are read in the same run."""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from jacobian_timing import card, flush_l2, time_ms  # noqa: E402
from vae_song_b200 import _C, model, module, ops, utils  # noqa: E402

KAPPA = 0.1


def rounds_hist(x, kappa, mode, prec, P, cache):
    """Run the inverse with budgets of 1, 2, ... rounds and record the round at which each row finished ("never": MAXITER)."""
    B = x.shape[0]
    z, st, err, rounds = ops.icnn_brenier_inverse(x, kappa, mode, prec, P, cache)
    done_at = torch.full((B,), -1, dtype=torch.int32, device="cuda")
    for k in range(1, rounds + 1):
        _, stk, _, _ = ops.icnn_brenier_inverse(x, kappa, mode, prec, P, cache, max_iter=k) if k < rounds else (z, st, err, k)
        newly = (done_at < 0) & (stk != _C.INV_MAXITER)
        done_at[newly] = k
    h = torch.bincount(done_at.clamp(min=0).long(), minlength=rounds + 1).cpu().tolist()
    hist = {str(k): n for k, n in enumerate(h) if n and k > 0}
    hist["never"] = h[0]             # still active after the last round (MAXITER)
    return hist, st, rounds


def one_icnn(reps):
    out = []
    lib = _C.load()
    B_list, d = (5000, 65536), 2
    for H in (512, 1024):
        for name, prec in _C.PRECISIONS.items():
            torch.manual_seed(0)
            ic = utils.trained_like_icnn_(module.ICNN(d, H, precision=name).cuda(), np.random.default_rng(H))
            P, mode = ic._flat_params(), ic._mode()
            for B in B_list:
                z_true = torch.randn(B, d, device="cuda", generator=torch.Generator("cuda").manual_seed(B))
                cache = {}
                with torch.no_grad():
                    _, x = ops.icnn_brenier_inference(z_true, KAPPA, mode, prec, P, cache)
                hist, st, rounds = rounds_hist(x, KAPPA, mode, prec, P, cache)
                t_inv = time_ms(lambda: ops.icnn_brenier_inverse(x, KAPPA, mode, prec, P, cache), reps)
                ws = cache["ws"]
                t_jac = time_ms(lambda: ops.icnn_decode_jac(z_true, ws, d, H, KAPPA, prec), 3 * reps)
                # the step kernel alone on a fresh state: init + step minus init
                nst = lib.b200vae_brenier_inverse_state_bytes(B, d)
                state = torch.empty(nst, dtype=torch.uint8, device="cuda")
                tr, zz = torch.empty(B, d, device="cuda"), torch.empty(B, d, device="cuda")
                s32, e32 = torch.empty(B, dtype=torch.int32, device="cuda"), torch.empty(B, device="cuda")
                _, xh, jac, _, _ = ops.icnn_decode_jac(z_true, ws, d, H, KAPPA, prec)
                p_ = ops._ptr
                init = lambda: lib.b200vae_brenier_inverse_init(p_(x), None, B, d, 1e-5, 1e-5, p_(state), nst, p_(tr),
                                                                p_(zz), p_(s32), p_(e32), ops._stream())
                step = lambda: lib.b200vae_brenier_newton_step(p_(x), p_(xh), p_(jac), B, d, KAPPA, 0, 0, p_(state), nst,
                                                               p_(tr), p_(zz), p_(s32), p_(e32), ops._stream())
                t_init = time_ms(init, 3 * reps)
                t_init_step = time_ms(lambda: (init(), step()), 3 * reps)
                stc = torch.bincount(st.long(), minlength=6).cpu().tolist()
                zi = ops.icnn_brenier_inverse(x, KAPPA, mode, prec, P, cache)[0]
                conv = st == _C.INV_CONVERGED
                rel = ((zi - z_true).norm(dim=1) / z_true.norm(dim=1).clamp(min=1e-30))[conv]
                per_round = t_inv / rounds
                out.append(dict(precision=name, d=d, H=H, B=B, kappa=KAPPA, rounds=rounds, rows_finished_at_round=hist,
                                status_counts=dict(zip(("active", "converged", "maxiter", "stalled", "singular",
                                                        "nonfinite"), stc)),
                                converged_rel_err_max=float(rel.max()) if rel.numel() else None,
                                inverse_ms=t_inv, per_round_ms=per_round, decode_jac_ms=t_jac,
                                step_share_of_round=(per_round - t_jac) / per_round,
                                step_kernel_fresh_state_ms=t_init_step - t_init, init_ms=t_init))
                print(json.dumps(out[-1]), flush=True)
    return out


def lidvae(precision):
    torch.manual_seed(0)
    m = model.LIDVAE(dataset="pinwheel", icnn_channels=[512, 1024], hidden_channels=[64, 128, 64, 2], inverse_lipschitz=0.2,
                     precision=precision).cuda().eval()
    for i, ic in enumerate((m.decoder[0], m.decoder[1])):
        utils.trained_like_icnn_(ic, np.random.default_rng(10 + i))
    return m


def decoder(reps):
    out = []
    for precision in ("fp32", "f16x3"):
        m = lidvae(precision)
        for B in (5000, 65536):
            z = torch.randn(B, 2, device="cuda", generator=torch.Generator("cuda").manual_seed(B))
            with torch.no_grad():
                y = m.decode(z)
            zi, st, bound = m.decode_inverse(y)
            t_inv = time_ms(lambda: m.decode_inverse(y), reps)

            tol = ops.INVERSE_TOL[_C.PRECISIONS[precision]] * (y.norm(dim=1) + 1)

            def eager_iteration(zc):
                zg = zc.clone().requires_grad_(True)
                yy = m.decode(zg)
                cols = []
                for i in range(yy.shape[1]):
                    e = torch.zeros_like(yy)
                    e[:, i] = 1.0
                    cols.append(torch.autograd.grad(yy, zg, e, retain_graph=i + 1 < yy.shape[1])[0])
                J = torch.stack(cols, 1)
                r = (yy - y).detach()
                return (zc - torch.linalg.solve(J, r.unsqueeze(-1)).squeeze(-1)).detach(), r.norm(dim=1)

            def eager_loop():
                """the loop a user writes today: full Newton steps on the whole decoder from z = 0 until every row's
                residual meets the same tolerance (checked on the host each iteration) or 100 iterations"""
                zc = torch.zeros_like(z)
                for it in range(1, 101):
                    zc, rn = eager_iteration(zc)
                    if bool((rn <= tol).all()):
                        return zc, it
                return zc, 100

            t_it = time_ms(lambda: eager_iteration(z), reps)
            ze, iters = eager_loop()
            t_loop = time_ms(eager_loop, 1, warmup=0)
            with torch.no_grad():
                eager_conv = float(((m.decode(ze) - y).norm(dim=1) <= tol).float().mean())
            stc = torch.bincount(st.long(), minlength=6).cpu().tolist()
            conv = st == _C.INV_CONVERGED
            out.append(dict(precision=precision, B=B, decode_inverse_ms=t_inv,
                            status_counts=dict(zip(("active", "converged", "maxiter", "stalled", "singular", "nonfinite"),
                                                   stc)),
                            converged_max_dist=float((zi - z).norm(dim=1)[conv].max()) if conv.any() else None,
                            bound_median=float(bound.median()),
                            eager_autograd_newton_iteration_ms=t_it, eager_autograd_newton_loop_ms=t_loop,
                            eager_loop_iterations=iters, eager_loop_converged_fraction=eager_conv))
            print(json.dumps(out[-1]), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_inverse.json"))
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("inverse_timing.py measures on the GPU; no CUDA device found")
    flush_l2()
    res = dict(card=card(), method="CUDA events per call, median; L2 overwritten (512 MB) before every timed call; every "
                                   "shape warmed up first",
               icnn=one_icnn(a.reps), decoder=decoder(a.reps))
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
