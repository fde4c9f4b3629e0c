#!/usr/bin/env python
"""Cost of the Brenier map's exact Jacobian (b200vae_icnn_decode_jac, LIDVAE.decode_jacobian) -> profiles/r05_jacobian.json.

    python scripts/jacobian_timing.py [--out profiles/r05_jacobian.json] [--reps 30]

(a) decode kernel vs decode + Jacobian kernel, d = 2, H = 512 / 1024, B = 65536, every precision;
(b) LIDVAE.decode_jacobian vs the autograd route (D torch.autograd.grad calls of decode with one-hot cotangents, which also
    run the parameter-gradient kernels) at B = 65536 and 5000;
(c) the data-based (inverse, local, bi) Lipschitz estimate at 5000 points: Jacobian vs sampled pairs vs all-pairs quantiles.
CUDA events around each call; every timed call is preceded by a 512 MB write that evicts the 126 MB L2, and every shape is
warmed up first.  Reports medians and the card's name / power limit, read in the same run."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from vae_song_b200 import _C, model, ops, utils  # noqa: E402

_FLUSH = None


def flush_l2():
    global _FLUSH
    if _FLUSH is None:
        _FLUSH = torch.empty(512 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda")
    _FLUSH.zero_()


def time_ms(fn, reps, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        flush_l2()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    ts.sort()
    return ts[len(ts) // 2]


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else torch.cuda.get_device_name()


def kernel_pair(reps):
    out = []
    B, d = 65536, 2
    g = torch.Generator("cuda").manual_seed(0)
    for H in (512, 1024):
        for name, prec in _C.PRECISIONS.items():
            P = [torch.randn(H, d, device="cuda", generator=g) * 0.7, torch.randn(H, device="cuda", generator=g) * 0.5,
                 torch.randn(H, d, device="cuda", generator=g), torch.randn(H, device="cuda", generator=g) - 0.3,
                 torch.randn(1, d, device="cuda", generator=g), torch.randn(1, device="cuda", generator=g) * 0.5,
                 torch.randn(H, H, device="cuda", generator=g) - float(torch.log(torch.tensor(float(H)))),
                 torch.randn(1, H, device="cuda", generator=g) - float(torch.log(torch.tensor(H / 2.0)))]
            z = torch.randn(B, d, device="cuda", generator=g)
            ws = ops.icnn_prepare(P, d, H, 0, prec, B, False)
            t_fwd = time_ms(lambda: ops.icnn_decode_fwd(z, ws, d, H, 0, 0.1, prec, True, True, False), reps)
            t_jac = time_ms(lambda: ops.icnn_decode_jac(z, ws, d, H, 0.1, prec), reps)
            out.append(dict(precision=name, d=d, H=H, B=B, decode_ms=t_fwd, decode_jac_ms=t_jac, ratio=t_jac / t_fwd))
            print(json.dumps(out[-1]), flush=True)
    return out


def lidvae(precision):
    torch.manual_seed(0)
    m = model.LIDVAE(dataset="pinwheel", icnn_channels=[512, 1024], hidden_channels=[64, 128, 64, 2], inverse_lipschitz=0.2,
                     precision=precision).cuda().eval()
    with torch.no_grad():          # trained-like scale: exp(W) ~ 1/sqrt(H) instead of ~1 (O(1) outputs, masks of both signs)
        for ic in (m.decoder[0], m.decoder[1]):
            for w in ic.W:
                w.param.sub_(0.5 * float(torch.log(torch.tensor(float(ic.hidden_channel)))))
    return m


def decoder_vs_autograd(reps):
    out = []
    for precision in ("fp32", "f16x3"):
        m = lidvae(precision)
        for B in (65536, 5000):
            z = torch.randn(B, 2, device="cuda")

            def autograd_route():
                zg = z.clone().requires_grad_(True)
                y = m.decode(zg)
                cols = []
                for i in range(y.shape[1]):
                    e = torch.zeros_like(y)
                    e[:, i] = 1.0
                    cols.append(torch.autograd.grad(y, zg, e, retain_graph=i + 1 < y.shape[1])[0])
                return torch.stack(cols, 1)

            t_j = time_ms(lambda: m.decode_jacobian(z), reps)
            t_a = time_ms(autograd_route, max(5, reps // 3))
            out.append(dict(precision=precision, B=B, decode_jacobian_ms=t_j, autograd_ms=t_a, speedup=t_a / t_j))
            print(json.dumps(out[-1]), flush=True)
    return out


def estimators(reps):
    out = []
    for precision in ("fp32", "f16x3"):
        m = lidvae(precision)
        z = torch.randn(5000, 2, device="cuda")
        with torch.no_grad():
            t_j = time_ms(lambda: utils.estimate_local_lipschitz_jacobian(m, z), reps)
            t_s = time_ms(lambda: utils.estimate_local_lipschitz(m.decode, z, num_pairs=5000), reps)
            t_all = time_ms(lambda: utils.estimate_lipschitz_allpairs(m.decode, z, quantile=0.05), max(5, reps // 3))
            vals = dict(jacobian=utils.estimate_local_lipschitz_jacobian(m, z),
                        sampled=utils.estimate_local_lipschitz(m.decode, z, num_pairs=5000))
            r = utils.estimate_lipschitz_allpairs(m.decode, z, quantile=0.05)
            vals["all_pairs"] = (r["inverse_lipschitz"], r["lipschitz"], r["bi_lipschitz"])
        out.append(dict(precision=precision, points=5000, jacobian_ms=t_j, sampled_pairs_ms=t_s, all_pairs_ms=t_all,
                        triples_inverse_local_bi=vals))
        print(json.dumps(out[-1]), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_jacobian.json"))
    ap.add_argument("--reps", type=int, default=30)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("jacobian_timing.py measures on the GPU; no CUDA device found")
    res = dict(card=card(), method="CUDA events per call, median; L2 overwritten (512 MB) before every timed call; "
                                    "every shape warmed up first",
               kernel=kernel_pair(a.reps), decoder=decoder_vs_autograd(a.reps), estimators=estimators(a.reps))
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
