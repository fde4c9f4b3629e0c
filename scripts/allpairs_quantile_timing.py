"""Timing of the exact all-pairs quantiles (ops.lipschitz_allpairs_quantiles) on LIDVAE-decoded latent samples, like
bench.lipschitz_times: at each N, with CUDA events after a warm-up,
  - the all-pairs statistics kernel (ops.lipschitz_allpairs),
  - each count pass and each locate of the select,
  - the whole 0.05 / 0.95 quantile call,
  - the sampled estimator (utils.estimate_local_lipschitz, 5000 random pairs, its two decodes included),
  - for N <= 20000 the brute-force PyTorch alternative: cdist ratio matrix, gather of the upper triangle, sort.
Kernel times replay a CUDA graph of `--reps` launches (one Python-issued launch costs more host time than a kernel runs);
`*_call_ms` are what a Python caller sees.  Writes <out>/allpairs_quantile.json with the card name and power limit.

    python scripts/allpairs_quantile_timing.py --out results/allpairs_quantile
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402


def card():
    info = {"name": torch.cuda.get_device_name()}
    try:   # read-only query
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        lim, clk = r.stdout.strip().splitlines()[torch.cuda.current_device()].split(",")
        info.update(power_limit=lim.strip(), max_sm_clock=clk.strip())
    except Exception as e:  # noqa: BLE001
        info["power_limit"] = f"unknown ({e})"
    return info


def events(fn, n):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def graph_ms(fn, reps):
    """Per-launch time of `fn` from a CUDA graph of `reps` back-to-back calls (captured on a warmed side stream)."""
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fn()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        for _ in range(reps):
            fn()
    return events(g.replay, 5) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="results/allpairs_quantile")
    ap.add_argument("--sizes", type=int, nargs="+", default=[5000, 20000, 50000])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--q", type=float, default=0.05)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("allpairs_quantile_timing.py needs a CUDA device")
    from bench import MODEL_KW
    from vae_song_b200 import _C, model, ops, utils
    torch.manual_seed(0)
    m = model.LIDVAE(**MODEL_KW).cuda()
    rng = np.random.default_rng(7)
    for ic in (m.decoder[0], m.decoder[1]):
        utils.trained_like_icnn_(ic, rng)
    m.eval()
    q0, q1 = args.q, 1.0 - args.q
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = {"card": card(), "library": os.path.relpath(_C.LIB_PATH, root), "quantiles": [q0, q1], "reps": args.reps,
           "sizes": {}}
    for N in args.sizes:
        Z = torch.randn(N, 2, device="cuda", generator=torch.Generator(device="cuda").manual_seed(N))
        with torch.no_grad():
            Y = m.decode(Z).contiguous()
        n = N * (N - 1) // 2
        r = {"pairs": n}
        r["stats_kernel_ms"] = graph_ms(lambda: ops.lipschitz_allpairs(Z, Y, 1e-3), args.reps)
        r["stats_call_ms"] = events(lambda: ops.lipschitz_allpairs(Z, Y, 1e-3), 10)
        state, hist = ops.lipschitz_select_buffers(Z.device)
        out = torch.empty(6, dtype=torch.float64, device="cuda")
        nt = ops.lipschitz_num_tiles(N)
        for p in range(_C.LIPSCHITZ_SELECT_PASSES):     # each pass on a state left by the real previous passes
            for pp in range(p):
                ops.lipschitz_select_count(Z, Y, 1e-3, 0, nt, pp, state, hist)
                ops.lipschitz_select_locate(N, q0, q1, pp, hist, state, out)
            r[f"count_pass{p}_ms"] = graph_ms(lambda: ops.lipschitz_select_count(Z, Y, 1e-3, 0, nt, p, state, hist), args.reps)
            ops.lipschitz_select_count(Z, Y, 1e-3, 0, nt, p, state, hist)
            r[f"locate_pass{p}_ms"] = events(lambda: ops.lipschitz_select_locate(N, q0, q1, p, hist, state, out), 20)
        r["quantile_graph_ms"] = graph_ms(lambda: ops.lipschitz_allpairs_quantiles(Z, Y, (q0, q1)), max(1, args.reps // 4))
        r["quantile_call_ms"] = events(lambda: ops.lipschitz_allpairs_quantiles(Z, Y, (q0, q1)), 10)
        r["quantile_over_stats"] = r["quantile_graph_ms"] / r["stats_kernel_ms"]
        v = ops.lipschitz_allpairs_quantiles(Z, Y, (q0, q1)).tolist()
        r["values"] = v[:2]
        r["sampled_estimator_ms"] = events(lambda: utils.estimate_local_lipschitz(m.decode, Z, num_pairs=5000), 5)
        if N <= 20000:
            iu = torch.triu_indices(N, N, 1, device="cuda")
            ks = [ops.lipschitz_quantile_ranks(n, q) for q in (q0, q1)]

            def brute():
                R = torch.cdist(Y, Y).clamp(min=1e-3) / torch.cdist(Z, Z).clamp(min=1e-3)
                s = torch.sort(R[iu[0], iu[1]]).values.double()
                return [s[k] + w * (s[min(k + 1, n - 1)] - s[k]) for k, w in ks]
            r["bruteforce_torch_ms"] = events(brute, 3)
            r["bruteforce_values"] = [float(x) for x in brute()]
            del iu
            torch.cuda.empty_cache()
        res["sizes"][str(N)] = r
        print(N, json.dumps(r), flush=True)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "allpairs_quantile.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
