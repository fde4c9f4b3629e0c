"""Kernel timeline of bench.py's flagship train step (configs[1], graph replay), from torch.profiler with CUDA activities.

    python scripts/step_timeline.py [--batch 65536] [--precision f16x3] [--steps 5] [--out DIR]

Builds the step exactly as bench.py does (same model, weights, trainer and captured graph), replays it --steps times with
an L2 flush and a synchronise before each replay, and reports for the last replay:
  - every kernel with its stream, start and end (us from the step's first kernel),
  - the gap from step start to the first ICNN tensor-core kernel and from the last one to step end,
  - the idle time on the main stream (the stream of the first kernel) between the step's first and last kernel,
  - the card name and power limit.
Writes DIR/step_timeline.json and prints a summary.  Run it in a process of its own: tracing slows the host, so
end-to-end step times come from bench.py, not from here.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ICNN = re.compile(r"icnn_tc3_(fwd|bwd|dP0)\w*_kernel")     # the ICNN pair kernels (not prepare / finalize)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [s.strip() for s in q.split(",")[:2]]
        return {"name": name, "power_limit": power}
    except Exception as exc:       # noqa: BLE001 - reported, not fatal
        return {"name": "unknown", "power_limit": "unknown", "error": str(exc)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=65536)
    ap.add_argument("--precision", default="f16x3")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--out", default=".", help="directory for step_timeline.json")
    args = ap.parse_args()

    import numpy as np
    import torch
    from torch.profiler import ProfilerActivity, profile

    import bench
    from vae_song_b200 import model, train

    if not torch.cuda.is_available():
        raise SystemExit("step_timeline.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    torch.manual_seed(42)
    m = bench.trained_like_(model.LIDVAE(precision=args.precision, **bench.MODEL_KW)).to(dev).train()
    tr = train.DataParallelTrainer(m, lr=bench.LR)
    x = torch.from_numpy(bench.chessboard(args.batch, np.random.default_rng(100))).to(dev)
    tr.step(x)
    tr.capture(x)
    for _ in range(3):
        tr.step_graphed(x)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    torch.cuda.synchronize()

    with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
        for _ in range(args.steps):
            flush.fill_(1.0)
            torch.cuda.synchronize()
            tr.step_graphed(x)
            torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            trace = json.load(f)
    kern = sorted((e for e in trace["traceEvents"] if e.get("cat") == "kernel"), key=lambda e: e["ts"])
    # the kernels after the last flush fill belong to the last replay
    fills = [i for i, e in enumerate(kern) if "fill" in e["name"].lower() and e["dur"] > 20]
    step = kern[fills[-1] + 1:]
    if not step:
        raise SystemExit("no kernels recorded after the last flush")
    t0 = step[0]["ts"]
    t1 = max(e["ts"] + e["dur"] for e in step)
    main_stream = step[0]["args"].get("stream")
    rows = [{"name": e["name"][:120], "stream": e["args"].get("stream"), "start_us": round(e["ts"] - t0, 2),
             "end_us": round(e["ts"] + e["dur"] - t0, 2)} for e in step]
    icnn = [r for r in rows if ICNN.search(r["name"])]
    busy, cur_end = 0.0, None
    for r in rows:
        if r["stream"] != main_stream:
            continue
        s, e = r["start_us"], r["end_us"]
        if cur_end is None or s >= cur_end:
            busy += e - s
            cur_end = e
        elif e > cur_end:
            busy += e - cur_end
            cur_end = e
    main_span = max(r["end_us"] for r in rows if r["stream"] == main_stream)
    res = {
        "card": card(), "batch": args.batch, "precision": args.precision,
        "step_us": round(t1 - t0, 2), "kernels": len(rows),
        "streams": sorted({r["stream"] for r in rows}, key=lambda s: (s != main_stream, s)),
        "start_to_first_icnn_us": icnn[0]["start_us"] if icnn else None,
        "last_icnn_to_end_us": round((t1 - t0) - max(r["end_us"] for r in icnn), 2) if icnn else None,
        "main_stream_idle_us": round(main_span - busy, 2),
        "timeline": rows,
    }
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "step_timeline.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "timeline"}))
    for r in rows:
        print(f"  s{r['stream']:<4} {r['start_us']:9.2f} {r['end_us']:9.2f}  {r['name']}")


if __name__ == "__main__":
    main()
