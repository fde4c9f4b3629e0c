#!/usr/bin/env python
"""bench.py -- LID-VAE train samples/s (BASELINE.json metric) on N B200s of one node, plus the fused ICNN
decode+grad-psi kernel against its roofline and the CPU oracle port as baseline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch B] [--precision fp32]
                    [--dump-outputs DIR]
    N>1:  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N

Workload (config.workload): BASELINE.json configs[1] -- LIDVAE(dataset='pinwheel'), latent_dim 2, ICNN(2,512) +
ICNN(2,1024) Brenier decoder, synthetic chessboard 2-D points, per-GPU batch 65536 (weak scaling).  One step =
forward -> loss -> backward -> gradient all-reduce (N>1) -> Adam, i.e. lipschitz.py:36-43.
`value`  : inputs resident in HBM.           `e2e`: same step through the public module API with pinned HOST
inputs (H2D copy) and the loss read back (D2H) inside the timed region.

`--impl reference` runs the UNMODIFIED reference (oracle/_ref/, populated by oracle/fetch_ref.py from a reference checkout):
its own `model.LIDVAE` driven by its own loop `lipschitz.train_model` (lipschitz.py:23-44) in PyTorch on the host cores,
on the SAME config -- batch 65536 per step, encoder and Adam included, same weights, same synthetic data.  The numpy
oracle port is only the fallback when oracle/_ref/ is absent (the line then says kind "port").
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def chessboard(n, rng):
    """Synthetic 2-D chessboard points in [-4,4]^2 (own generator; shape/statistics of dataset.py:72-102)."""
    pts = np.empty((0, 2), dtype=np.float32)
    while pts.shape[0] < n:
        c = rng.uniform(-4, 4, (2 * n, 2)).astype(np.float32)
        keep = (np.floor(c[:, 0]) + np.floor(c[:, 1])) % 2 == 0
        pts = np.concatenate([pts, c[keep]], 0)
    return pts[:n]


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """SM clock / power / throttle reasons sampled every ~2 ms through NVML in a background thread (the timed region of
    a 3 ms step x K steps is far shorter than nvidia-smi's sampling period); falls back to `nvidia-smi -lms 100`."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.rows, self.proc, self.nvml, self._stop = [], None, None, False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                          str(index), "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _poll(self):
        n = self.nvml
        R = {"hw_slowdown": n.nvmlClocksThrottleReasonHwSlowdown, "hw_thermal_slowdown": n.nvmlClocksThrottleReasonHwThermalSlowdown,
             "sw_thermal_slowdown": n.nvmlClocksThrottleReasonSwThermalSlowdown, "sw_power_cap": n.nvmlClocksThrottleReasonSwPowerCap}
        while not self._stop:
            try:
                sm = float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM))
                pw = n.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                mask = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.rows.append((time.time(), [str(sm), str(self.max_sm), str(pw)] +
                                  ["Active" if (mask & R[k]) else "Not Active" for k in
                                   ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")]))
            except Exception:
                pass
            time.sleep(0.002)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def window(self, t0, t1):
        rows = [r for t, r in self.rows if t0 <= t <= t1]
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": len(rows), "source": "nvml" if self.nvml else "nvidia-smi"}
        try:
            sm = sorted(float(r[0]) for r in rows)
            out["sm_mhz"] = sm[len(sm) // 2]
            out["sm_max_mhz"] = float(rows[0][1])
            out["power_w_max"] = max(float(r[2]) for r in rows)
            for i, name in enumerate(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")):
                if any(r[3 + i].lower().startswith("active") for r in rows):
                    out["reasons"].append(name)
        except Exception:
            pass
        return out

    def stop(self):
        self._stop = True
        if self.proc:
            self.proc.terminate()


# ----------------------------------------------------------------------------------------- shared workload definition
WORKLOAD = "configs[1]: LIDVAE(pinwheel/chessboard 2-D, latent 2, encoder [2,2,2,2], ICNN(2,512)+ICNN(2,1024)) train step"
MODEL_KW = dict(dataset="pinwheel", inverse_lipschitz=0.2, beta=1.0)
LR = 1e-3


def make_config(B, world):
    """The `config` object of BOTH arms (the reference arm runs "your arm's config"): only what defines the workload."""
    return {"workload": WORKLOAD, "per_gpu_batch": B, "global_batch": B * world, "parallelism": f"dp{world}",
            "step": "forward -> loss -> backward -> Adam(lr 1e-3): lipschitz.py:36-43", "encoder": "included", "optimizer": "Adam lr 1e-3",
            "weights": "seed 42 init + O(1)-scale ICNN weights (numpy seed 7)", "inputs": "chessboard 2-D points, numpy seed 100+rank",
            "l2": "flushed between timed iterations (256 MB write) on the GPU; inputs larger than cache on the CPU"}


def trained_like_(m):
    """O(1)-scale random ICNN weights, identical for both arms (default exp(W)~1 init gives 1e20 losses whose squares
    overflow Adam's v).  Works on the reference's and on this package's LIDVAE (same attribute names)."""
    import torch
    wr = np.random.default_rng(7)
    with torch.no_grad():
        for ic in (m.decoder[0], m.decoder[1]):
            H = ic.A0.weight.shape[0]
            ic.W[0].param.copy_(torch.tensor(wr.normal(np.log(1.0 / H), 1.0, (H, H)), dtype=torch.float32))
            ic.W[1].param.copy_(torch.tensor(wr.normal(np.log(2.0 / H), 1.0, (1, H)), dtype=torch.float32))
            ic.A[0].bias.copy_(torch.tensor(wr.normal(-0.3, 1.0, (H,)), dtype=torch.float32))
    return m


# ----------------------------------------------------------------------------------------- reference arm (CPU / same GPU)
def ref_available():
    try:
        from oracle import fetch_ref
        return fetch_ref.available()
    except Exception:
        return False


class _TimedLoader:
    """Feeds `lipschitz.train_model` W + K batches and time-stamps every hand-over: the reference's own loop
    (lipschitz.py:36-43) runs unmodified and the time between two `__next__` calls is one of its steps.  On CUDA the stamps
    are events on the current stream (the loop launches everything there) and the L2 is flushed before each step."""

    def __init__(self, batches, device, flush=None):
        self.batches, self.device, self.flush = batches, device, flush
        self.marks = []

    def _mark(self):
        if self.device == "cpu":
            return time.perf_counter()
        import torch
        ev = torch.cuda.Event(enable_timing=True)
        ev.record()
        return ev

    def __iter__(self):
        for x in self.batches:
            end_prev = self._mark()
            if self.flush is not None:
                self.flush.fill_(1.0)
            self.marks.append((end_prev, self._mark()))
            yield x, None
        self.marks.append((self._mark(), None))

    def step_times_ms(self):
        out = []
        for i in range(len(self.marks) - 1):
            t0, t1 = self.marks[i][1], self.marks[i + 1][0]
            out.append((t1 - t0) * 1e3 if self.device == "cpu" else t0.elapsed_time(t1))
        return out


def time_reference(batches, device, warmup, flush=None):
    """UNMODIFIED reference: model.LIDVAE (model.py:637-886) trained by lipschitz.train_model (lipschitz.py:23-44), stock
    PyTorch (FP32, TF32 off = torch default) on `device`.  Returns per-step ms of the steps after `warmup`."""
    import torch
    from oracle import fetch_ref
    ns = fetch_ref.import_ref()
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    torch.manual_seed(42)
    m = trained_like_(ns.model.LIDVAE(**MODEL_KW))
    loader = _TimedLoader(batches, "cpu" if device == "cpu" else "cuda", flush)
    import contextlib, io
    with contextlib.redirect_stderr(io.StringIO()):          # tqdm progress bar of train_model
        ns.lipschitz.train_model(m, loader, epochs=1, lr=LR, device=device)
    if device != "cpu":
        torch.cuda.synchronize()
    ts = loader.step_times_ms()
    return ts[warmup:], fetch_ref.verify()


def oracle_step_factory(seed=0):
    """FALLBACK when oracle/_ref/ is absent: the oracle port of one LID-VAE decoder train step (decode fwd + double-backward
    + losses), fp32 numpy (multi-threaded BLAS).  The tiny [2,2,2,2] encoder and Adam are omitted (<1% of the flops)."""
    from oracle import icnn_oracle as io
    from oracle import loss_oracle as lo
    rng = np.random.default_rng(seed)
    p0 = io.random_params(rng, 2, 512, np.float32, "mixed")
    p1 = io.random_params(rng, 2, 1024, np.float32, "mixed")

    def step(x, eps):
        mu, lv = x * np.float32(0.5), np.abs(x) * np.float32(0.1)      # stand-in encoder outputs
        z = lo.reparam(mu, lv, eps)
        y, _, _, _ = io.lidvae_decode(z, p0, p1, 2, 0, 0.1)
        rec, kl = lo.recon_mse(x, y), lo.kl(mu, lv)
        vy = lo.recon_mse_grad(x, y).astype(np.float32)
        io.lidvae_decode_backward(z, vy, p0, p1, 2, 0, 0.1)
        return float(rec + kl)
    return step


def cpu_reference_times(B, steps, warmup):
    """(per-step ms list, kind, note) of the reference's CPU path on this box's host cores at per-step batch B."""
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    rng = np.random.default_rng(100)
    if ref_available():
        batches = [torch.from_numpy(chessboard(B, rng)) for _ in range(min(4, steps + warmup))]
        batches = [batches[i % len(batches)] for i in range(steps + warmup)]
        ts, unmodified = time_reference(batches, "cpu", warmup)
        return ts, "reference", ("unmodified reference (oracle/_ref: model.LIDVAE + lipschitz.train_model, PyTorch CPU FP32, "
                                 f"{torch.get_num_threads()} threads); files match the fetch-time SHA-256: {unmodified}")
    step = oracle_step_factory()
    x, eps = chessboard(B, rng), rng.normal(0, 1, (B, 2)).astype(np.float32)
    ts = []
    for i in range(steps + warmup):
        t0 = time.perf_counter(); step(x, eps); ts.append((time.perf_counter() - t0) * 1e3)
    return ts[warmup:], "port", "oracle/_ref absent: numpy oracle port of the decoder train step (no encoder, no Adam)"


def run_reference(args, rank):
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    B = args.batch
    ts, kind, note = cpu_reference_times(B, args.steps, max(args.warmup, 1))
    ms = float(np.mean(ts))
    val = B / (ms * 1e-3)
    line = {"impl": "reference", "metric": "LID-VAE train samples/s", "value": val, "unit": "samples/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": make_config(B, max(args.gpus, 1)),
            "cpu_baseline": {"value": val, "unit": "samples/s", "cores": cores, "kind": kind,
                             "sample": f"{B} samples per step x {args.steps} steps (rank 0 only: one CPU process); {note}"},
            "e2e": {"value": val, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def eager_icnn_potential(z, mode, A0w, A0b, A1w, A1b, A2w, A2b, W0, W1):
    """psi [B,1] of an ICNN written with ordinary differentiable torch ops -- module.py:142-148 verbatim semantics
    (PositiveLinear = exp / clamp(min=1e-2) of the raw weight, LeakyReLU(0.2), first layer squared).  NOT product code: the
    stock-PyTorch formulation that the fused kernels are timed against where oracle/_ref is not used."""
    import torch
    act = torch.nn.functional.leaky_relu
    lin = torch.nn.functional.linear
    pos = (lambda W: W.exp()) if mode == 0 else (lambda W: W.clamp(min=1e-2))
    x = act(lin(z, A0w, A0b), 0.2).pow(2)
    x = act(lin(x, pos(W0)) + lin(z, A1w, A1b), 0.2)
    return act(lin(x, pos(W1)) + lin(z, A2w, A2b), 0.2)


def eager_same_gpu(m, x, flush, steps=5):
    """The reference's own formulation of this train step (lipschitz.py:36-43 over model.py:818-886: stock nn.Modules for
    the encoder, ICNN.forward as torch ops, two autograd.grad(create_graph=True) calls, autograd double-backward,
    torch.optim.Adam) run by stock PyTorch eager in FP32 (TF32 off, the reference's default) on THIS GPU -- the number the
    fused path has to beat (SURVEY.md 8(d)).  Same weights, same batch."""
    import copy
    import torch
    import torch.nn.functional as F
    from vae_song_b200 import ops
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    ref = copy.deepcopy(m).train()
    opt = torch.optim.Adam(ref.parameters(), lr=1e-3)
    kappa = ref.il_factor

    def brenier(ic, zz):
        psi = eager_icnn_potential(zz, ic._mode(), *ic._flat_params()) + kappa * zz.pow(2).sum(1, keepdim=True)
        return torch.autograd.grad(psi, [zz], torch.ones_like(psi), create_graph=True)[0]

    def step():
        opt.zero_grad()
        ret = ref.encoder(x)                                    # stock Linear / BatchNorm1d / LeakyReLU modules
        mu, var = ret.split(ret.shape[1] // 2, 1)
        lv = F.softplus(var)
        z = mu + torch.randn_like(mu) * torch.exp(0.5 * lv)
        y = brenier(ref.decoder[1], F.linear(brenier(ref.decoder[0], z), ref.B))
        rec = ((x - y) ** 2).mean(0).sum()
        kl = (-0.5 * (1 + lv - mu ** 2 - lv.exp())).mean(0).sum()
        (rec + ref.beta * kl).backward()
        opt.step()
    for _ in range(2):
        step()
    torch.cuda.synchronize()
    ts = []
    for _ in range(steps):
        flush.fill_(1.0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); step(); e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ms = float(np.mean(ts))
    del ref, opt
    torch.cuda.empty_cache()
    return {"train_ms": ms, "samples_per_s": x.shape[0] / (ms * 1e-3), "batch": int(x.shape[0]),
            "what": "reference formulation (torch ops + autograd.grad(create_graph=True) + autograd double-backward + "
                    "torch.optim.Adam), stock PyTorch eager, FP32 with TF32 off, same weights and batch, this GPU"}


def lipschitz_times(m, dev):
    """north_star kernel (4): the tiled all-pairs estimator and the reference-semantics random-pair estimator
    (utils.py:532-567) on N = 5000 latent samples of this model (lipschitz.py:157-194 sizes), plus N = 50000.  The kernel
    alone is timed by replaying a CUDA graph of 20 launches (a single Python-issued launch costs more host time than the
    kernel runs); the `*_call_ms` figures are what a caller of ops.lipschitz_allpairs sees."""
    import torch
    from vae_song_b200 import ops, utils

    def t(fn, n=10):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record(); torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n
    out = {}
    for N in (5000, 50000):
        X = torch.randn(N, 2, device=dev)
        with torch.no_grad():
            Y = m.decode(X)
        call_ms = t(lambda: ops.lipschitz_allpairs(X, Y, 1e-3))
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            ops.lipschitz_allpairs(X, Y, 1e-3)
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize()
        g, reps = torch.cuda.CUDAGraph(), 20
        with torch.cuda.graph(g):
            for _ in range(reps):
                ops.lipschitz_allpairs(X, Y, 1e-3)
        k_ms = t(g.replay, 5) / reps
        pairs = N * (N - 1) // 2
        # per pair (d = Dx = 2): 4 sub + 4 fma/mul for the two squared distances, 2 max, 2 mul, 1 MUFU (rsqrt), max / min / add
        # = 17 FP32-pipe lane-ops + 1 MUFU op; bounds: 148 SM x 128 lanes x 1.965 GHz and 148 x 16 MUFU lanes x 1.965 GHz
        fp32_bound = 148 * 128 * 1.965e9 / 17.0
        mufu_bound = 148 * 16 * 1.965e9
        out[f"N{N}"] = {"pairs": pairs, "allpairs_kernel_ms": k_ms, "allpairs_call_ms": call_ms,
                        "pairs_per_s": pairs / (k_ms * 1e-3),
                        "roofline": {"bound": "fp32 issue (17 lane-ops per pair) / MUFU (1 per pair)", "achieved": pairs / (k_ms * 1e-3),
                                     "peak": min(fp32_bound, mufu_bound), "unit": "pairs/s",
                                     "frac": pairs / (k_ms * 1e-3) / min(fp32_bound, mufu_bound),
                                     "fp32_issue_bound": fp32_bound, "mufu_bound": mufu_bound}}
    X = torch.randn(5000, 2, device=dev)
    out["random_pairs_estimate_ms"] = t(lambda: utils.estimate_local_lipschitz(m.decode, X, num_pairs=5000), 5)
    out["note"] = ("all-pairs: 64x64 tiles of the upper triangle, 4x4 pairs per thread in registers, one MUFU per pair, ordered "
                   "per-CTA partials + last-block reduce in ONE launch; random pairs: 2 decodes of 5000 rows + ratio kernel + 2 "
                   "quantiles + one host sync")
    return out


def mnist_shaped_times(dev, flush, precision):
    """BASELINE configs[3] (parity-test config, reported for reference): the MNIST-shaped LIDVAE decoder ICNN(32,512) ->
    implicit eye(784,32) pad -> ICNN(784,1024) through the wide-input tcgen05 kernels, against the reference's own
    formulation (module.py:142-148 + autograd.grad(create_graph=True)) run by stock PyTorch (cuBLAS FP32) on this GPU."""
    import torch
    from vae_song_b200 import module, ops
    torch.backends.cuda.matmul.allow_tf32 = False
    rng = np.random.default_rng(0)
    ics = []
    for d, H in ((32, 512), (784, 1024)):
        ic = module.ICNN(d, H, precision=precision).to(dev)
        with torch.no_grad():
            ic.W[0].param.copy_(torch.tensor(rng.normal(np.log(1.0 / H), 1.0, (H, H)), dtype=torch.float32))
            ic.W[1].param.copy_(torch.tensor(rng.normal(np.log(2.0 / H), 1.0, (1, H)), dtype=torch.float32))
            ic.A[0].bias.copy_(torch.tensor(rng.normal(-0.3, 1.0, (H,)), dtype=torch.float32))
        ics.append(ic)
    out = {"precision": precision}
    for B in (256, 8192):
        z = torch.randn(B, 32, device=dev, requires_grad=True)
        vy = torch.randn(B, 784, device=dev)

        def fused(train):
            _, x1 = ics[0].brenier(z, 0.1)
            _, y = ics[1].brenier(x1, 0.1)
            if train:
                (y * vy).sum().backward()

        def eager(train):
            def br(ic, x):
                psi = eager_icnn_potential(x, ic._mode(), *ic._flat_params()) + 0.1 * x.pow(2).sum(1, keepdim=True)
                return torch.autograd.grad(psi, [x], torch.ones_like(psi), create_graph=True)[0]
            y = br(ics[1], torch.nn.functional.linear(br(ics[0], z), torch.eye(784, 32, device=dev)))
            if train:
                (y * vy).sum().backward()

        def t(fn, train):
            for _ in range(3):
                fn(train)
            ts = []
            for _ in range(8):
                for ic in ics:
                    ic.zero_grad(set_to_none=True)
                z.grad = None
                flush.fill_(1.0)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); fn(train); e1.record()
                torch.cuda.synchronize()
                ts.append(e0.elapsed_time(e1))
            return float(np.mean(ts))
        out[f"B{B}"] = {"decode_ms": t(fused, False), "train_ms": t(fused, True),
                        "pytorch_eager_fp32_decode_ms": t(eager, False), "pytorch_eager_fp32_train_ms": t(eager, True)}
    return out


DUMP_MAX_BYTES = 60 * 1024 * 1024          # array data of --dump-outputs; with the .npy headers it stays under 64 MB


def dump_step_outputs(out_dir, tr, losses, with_grads):
    """--dump-outputs: what a caller of the timed train step holds after its last step -- the (total, recon, KL) losses
    (mean over ranks), every parameter after the Adam update, the BatchNorm buffers and, on one GPU, the gradients that
    update used -- as out_dir/<name>.npy in float32 (float64 for integer buffers), so that two builds can be compared
    output for output.  (With several GPUs the flat gradient buffer of a rank holds its own or a partly reduced sum, not
    the gradient the update used, so it is left out.)

    Over the size budget, every array larger than one common element count C is replaced by a fixed sample of C of its
    flattened elements, the same positions for every array of the same size (numpy default_rng(0)); the kept positions
    are written beside it as <name>.index.npy (float64) and the original shape as <name>.shape.npy."""
    import torch
    arrays = {f"loss_{k}": v.reshape(1) for k, v in zip(("total", "recon", "kl"), losses)}
    for name, p in tr.model.named_parameters():
        arrays[f"param.{name}"] = p
        if with_grads and p.grad is not None:
            arrays[f"grad.{name}"] = p.grad
    for name, b in tr.model.named_buffers():
        arrays[f"buffer.{name}"] = b
    out = {}
    for name, t in arrays.items():
        a = t.detach().cpu().numpy().reshape(t.shape)
        out[name] = a.astype(np.float32 if a.dtype.kind == "f" and a.itemsize <= 4 else np.float64)

    def cost(c):       # bytes written when arrays above c elements keep c of them (+ 8-byte positions, + shape)
        return sum(a.nbytes if a.size <= c else c * (a.itemsize + 8) + 8 * a.ndim for a in out.values())
    cap = max(a.size for a in out.values())
    if cost(cap) > DUMP_MAX_BYTES:
        lo, hi = 0, cap
        while lo < hi:
            mid = (lo + hi + 1) // 2
            lo, hi = (mid, hi) if cost(mid) <= DUMP_MAX_BYTES else (lo, mid - 1)
        cap = lo
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        if a.size > cap:
            idx = np.sort(np.random.default_rng(0).choice(a.size, cap, replace=False))
            np.save(os.path.join(out_dir, f"{name}.index.npy"), idx.astype(np.float64))
            np.save(os.path.join(out_dir, f"{name}.shape.npy"), np.array(a.shape, dtype=np.float64))
            a = a.reshape(-1)[idx]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)
    print(f"[bench] wrote {len(out)} arrays ({cost(cap) / 2**20:.1f} MiB) to {out_dir}", file=sys.stderr, flush=True)


# ----------------------------------------------------------------------------------------- GPU arm
def run_ours(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist

    from vae_song_b200 import _C, model, ops, train
    from vae_song_b200 import utils as vutils

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    torch.manual_seed(42)
    B = args.batch
    m = trained_like_(model.LIDVAE(precision=args.precision, **MODEL_KW)).to(dev).train()
    tr = train.DataParallelTrainer(m, lr=LR, comm=args.comm)
    exchange = "none (1 GPU)" if world == 1 else (
        "peer-memory kernels over NVLink: BatchNorm statistics inside the encoder finalize kernels, two-shot gradient "
        "all-reduce fused with Adam (no NCCL call in the step)" if tr.peer is not None else
        "NCCL: all_gather/all_reduce per BatchNorm layer + one flat gradient all-reduce")
    rng = np.random.default_rng(100 + rank)
    n_pool = 4
    host_pool = [torch.from_numpy(chessboard(B, rng)).pin_memory() for _ in range(n_pool)]
    dev_pool = [h.to(dev) for h in host_pool]
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)   # > 126 MB L2
    loss_host = torch.empty(1, dtype=torch.float32).pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(step_fn, K, W):
        for i in range(W):
            step_fn(i)
        barrier()
        evs = []
        for i in range(K):
            flush.fill_(1.0)                      # evict L2 between timed iterations (not timed)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); step_fn(i); e1.record()
            evs.append((e0, e1))
        barrier()
        tot = sum(a.elapsed_time(b) for a, b in evs)
        t = torch.tensor([tot], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t) / K

    barrier()
    n_before = _C.launch_count()
    tr.step(dev_pool[0])                                   # one eager step: counts this library's launches per step
    torch.cuda.synchronize()
    launches_per_step = _C.launch_count() - n_before
    use_graph = not args.no_graph
    if use_graph:                                          # whole step (incl. the NCCL all-reduce) as one CUDA graph
        tr.capture(dev_pool[0])
    run_step = tr.step_graphed if use_graph else tr.step

    last_out = [None]

    def step_resident(i):
        last_out[0] = run_step(dev_pool[i % n_pool])

    def step_e2e(i):
        if use_graph:      # H2D of THIS step's batch was started by the previous call (next_x): it overlaps that step
            total, _, _ = tr.step_graphed(host_pool[i % n_pool], next_x=host_pool[(i + 1) % n_pool])
        else:
            total, _, _ = tr.step(host_pool[i % n_pool].to(dev, non_blocking=True))
        loss_host.copy_(total.reshape(1), non_blocking=True)
        torch.cuda.current_stream().synchronize()

    # the same loop as a training script would write it: the loss of step i is copied to pinned memory every step but READ
    # on the host one step later (after step i+1 has been enqueued), so the host never idles the GPU.  Same copies inside
    # the timed region; reported beside the blocking figure, which stays the headline `e2e.value`.
    loss_ring = torch.zeros(2, dtype=torch.float32).pin_memory()
    ring_ev = [torch.cuda.Event(), torch.cuda.Event()]
    seen = []

    def step_e2e_pipelined(i):
        if use_graph:
            total, _, _ = tr.step_graphed(host_pool[i % n_pool], next_x=host_pool[(i + 1) % n_pool])
        else:
            total, _, _ = tr.step(host_pool[i % n_pool].to(dev, non_blocking=True))
        loss_ring[i & 1:(i & 1) + 1].copy_(total.reshape(1), non_blocking=True)
        ring_ev[i & 1].record()
        if i > 0:
            ring_ev[(i - 1) & 1].synchronize()
            seen.append(float(loss_ring[(i - 1) & 1]))

    sampler = ClockSampler(local_rank) if rank == 0 else None
    t_start = time.time()
    ms = timed(step_resident, args.steps, args.warmup)
    t_end = time.time()
    if args.dump_outputs:
        losses = tr.global_losses(*last_out[0])              # collective: every rank joins the mean over ranks
        if rank == 0:                                        # parameters and buffers are identical on every replica
            dump_step_outputs(args.dump_outputs, tr, losses, with_grads=world == 1)
    launches = launches_per_step * args.steps
    clocks = sampler.window(t_start, t_end) if sampler else {}
    if world > 1:
        dist.barrier()
    if sampler is not None or world > 1:
        # the timed region can be shorter than nvidia-smi's sampling period: keep the same loop running ~1 s
        # (untimed, all ranks) so that the clock / throttle record is taken under this exact load
        need_more = torch.tensor([1.0 if (rank == 0 and clocks.get("samples", 0) < 3) else 0.0], device=dev)
        if world > 1:
            dist.all_reduce(need_more, op=dist.ReduceOp.MAX)
        if float(need_more) > 0:
            t0c = time.time()
            reps = max(int(1000.0 / max(ms, 0.05)), 1)
            for i in range(reps):
                step_resident(i)
            torch.cuda.synchronize()
            if sampler is not None:
                clocks = sampler.window(t0c + 0.1, time.time())
                clocks["note"] = "sampled during an untimed ~1 s continuation of the timed loop (timed region < sampling period)"
    ms_e2e = timed(step_e2e, args.steps, args.warmup)
    ms_e2e_pipe = timed(step_e2e_pipelined, args.steps, args.warmup)
    exchange_ok = True
    try:
        tr.check()                                         # a peer exchange that timed out would have produced garbage
    except Exception as exc:                               # noqa: BLE001 - report it in the line instead of losing the run
        exchange_ok = False
        print(f"[bench] rank {rank}: {exc}", file=sys.stderr, flush=True)
    value = world * B / (ms * 1e-3)
    e2e = world * B / (ms_e2e * 1e-3)

    # ---- the same train step in the other arithmetic modes (1 GPU only; same weights, graph replay) ----
    by_prec_train = {args.precision: {"ms_per_step": ms, "samples_per_s": value}}
    if world == 1:
        import copy
        for pname in ("fp32", "tf32x3", "f16x3", "tf32"):
            if pname == args.precision:
                continue
            m2 = copy.deepcopy(m)
            m2.precision = pname
            tr2 = train.DataParallelTrainer(m2, lr=1e-3)
            tr2.step(dev_pool[0])
            if use_graph:
                tr2.capture(dev_pool[0])
            stepf = tr2.step_graphed if use_graph else tr2.step
            ms2 = timed(lambda i: stepf(dev_pool[i % n_pool]), max(3, min(args.steps, 10)), 3)
            by_prec_train[pname] = {"ms_per_step": ms2, "samples_per_s": B / (ms2 * 1e-3)}
            tr2._graph = None
            del tr2, m2

    # ---- fused ICNN decode + grad-psi kernel vs roofline at batch 65536 (north_star), every precision ----
    roof, extra = None, {}
    if rank == 0:
        pk, pk_kind = peaks()
        Bk = 65536
        z = torch.randn(Bk, 2, device=dev)
        byp = {}
        for pname in ("fp32", "tf32x3", "f16x3", "tf32"):
            prec = _C.PRECISIONS[pname]
            res = {}
            for H in (512, 1024):
                ic = m.decoder[0] if H == 512 else m.decoder[1]
                params = [p.detach() for p in ic._flat_params()]
                ws = ops.icnn_prepare(params, 2, H, 0, prec, Bk, False)
                for _ in range(3):
                    ops.icnn_decode_fwd(z, ws, 2, H, 0, 0.1, prec)
                torch.cuda.synchronize()
                ts = []
                for _ in range(10):
                    flush.fill_(1.0)
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(); ops.icnn_decode_fwd(z, ws, 2, H, 0, 0.1, prec); e1.record()
                    torch.cuda.synchronize()
                    ts.append(e0.elapsed_time(e1))
                res[H] = float(np.mean(ts))
            both = Bk / ((res[512] + res[1024]) * 1e-3)
            byp[pname] = {"decode_ms_H512": res[512], "decode_ms_H1024": res[1024], "decode_samples_per_s": both,
                          "tflops_H1024": vutils.flops_decode(2, 1024) * Bk / (res[1024] * 1e-3) / 1e12,
                          "tflops_2icnn": both * (vutils.flops_decode(2, 512) + vutils.flops_decode(2, 1024)) / 1e12}
        try:      # dram__bytes_read.sum + dram__bytes_write.sum per launch, from the committed `ncu --set full` captures
            traffic_tab = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        except Exception:
            traffic_tab = {}
        # executed / algorithmic flops (hi/lo operand splits: 3 MMAs per MAC in GEMM1, 2 in GEMM2)
        mult_of = {"fp32": 1.0, "tf32": 1.0, "tf32x3": 2.5, "f16x3": 2.5}

        def tensor_peak(pn):      # kind::f16 MMAs (f16x3) run at the bf16 rate, kind::tf32 at half of it
            return 74.4 if pn == "fp32" else (pk["bf16_tflops"] if pn == "f16x3" else pk["bf16_tflops"] / 2)

        def kernel_roof(pn):
            peak = tensor_peak(pn)
            ach = byp[pn]["tflops_H1024"]
            return {"bound": "fp32 fma pipe" if pn == "fp32" else "tensor", "precision": pn,
                    "kernel": f"icnn_decode_fwd (psi + grad psi), d=2, H=1024, B=65536, {pn}",
                    "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                    "executed": ach * mult_of[pn], "frac_executed": ach * mult_of[pn] / peak,
                    "kernel_ms": byp[pn]["decode_ms_H1024"],
                    "traffic": traffic_tab.get(f"icnn_decode_fwd_{pn}_H1024_B65536"),
                    "traffic_source": "static: one `ncu --set full` capture of this kernel committed under profiles/ "
                                      "(profiles/traffic.json), not re-measured in this run",
                    "peak_kind": "FP32 FMA peak 148 SM x 128 x 2 x 1.965 GHz" if pn == "fp32" else
                                 (f"{pk_kind} cuBLAS bf16 burst (kind::f16 MMAs on fp16 hi/lo operands run at the bf16 rate)"
                                  if pn == "f16x3" else f"{pk_kind} cuBLAS bf16 burst / 2 (TF32 runs at half the bf16 rate)")}
        # `roofline` describes the dominant kernel IN THE ARITHMETIC THE TIMED STEP RAN IN (dtype of this line).  achieved /
        # frac count ALGORITHMIC flops (SURVEY.md 8(d): 4H^2+8dH+2H+4d per sample); 3xTF32 executes 2.5 tensor flops per
        # algorithmic flop, so an fp32-grade kernel that keeps the tensor pipe full sits at frac ~0.4 and frac_executed ~1.
        # f16x3 (fp16 hi/lo operands on kind::f16 MMAs, the default) executes the same 2.5 MMAs per MAC at twice the rate.
        # No mode is both >= 0.9 ALGORITHMIC of the tensor roofline and inside the FP32 bounds: `by_precision.tf32` is the
        # >= 0.9 mode (bounds psi 2e-4 / xhat 5e-3), f16x3 / tf32x3 are the fp32-grade modes (bounds in DESIGN.md section 4).
        rp = args.roofline_precision or args.precision
        roof = kernel_roof(rp)
        roof["algorithmic_flop_per_sample"] = vutils.flops_decode(2, 1024)
        roof["precision_equals_step_dtype"] = (rp == args.precision)
        roof["by_precision"] = {pn: kernel_roof(pn) for pn in ("tf32", "f16x3", "tf32x3", "fp32")}
        step_flop = vutils.flops_train(2, 512) + vutils.flops_train(2, 1024)
        step_tf = step_flop * B / (ms * 1e-3) / 1e12
        step_peak = tensor_peak(args.precision)
        roof["train_step"] = {"bound": roof["bound"], "precision": args.precision, "achieved": step_tf, "peak": step_peak,
                              "unit": "TFLOP/s", "frac": step_tf / step_peak, "algorithmic_flop_per_sample": step_flop,
                              "ms_per_step": ms, "note": "whole timed step (encoder, loss, Adam, exchange included in the time), "
                              "decoder flops 8H^2+22dH per ICNN only"}
        extra = {"decode_by_precision": byp, "train_step_by_precision": by_prec_train,
                 "pytorch_eager_same_gpu": eager_same_gpu(m, dev_pool[0], flush) if world == 1 else None,
                 "lipschitz_estimator": lipschitz_times(m, dev),
                 "mnist_shaped_decoder": mnist_shaped_times(dev, flush, args.precision) if world == 1 else None}
        # ---- the UNMODIFIED reference on THIS GPU (stock PyTorch eager CUDA, FP32, same config) and on the host cores ----
        ref_gpu, cpu = None, None
        if world == 1:
            if ref_available():
                nref = 6
                ts, unmodified = time_reference([dev_pool[i % n_pool] for i in range(nref + 2)], dev, 2, flush)
                rms = float(np.mean(ts))
                ref_gpu = {"value": B / (rms * 1e-3), "unit": "samples/s", "ms_per_step": rms, "steps": len(ts), "batch": B,
                           "speedup_of_this_arm": rms / ms, "unmodified": unmodified,
                           "what": "oracle/_ref model.LIDVAE + lipschitz.train_model, stock PyTorch eager on this GPU, FP32 "
                                   "(TF32 off), same weights / batch / data, L2 flushed between steps, inputs resident"}
            csteps = 8                                    # ~10 s of CPU work (1.2 s per 65536-sample step)
            ts, kind, note = cpu_reference_times(B, csteps, 1)
            cms = float(np.min(ts))
            cpu = {"value": B / (cms * 1e-3), "unit": "samples/s", "cores": os.cpu_count(), "kind": kind,
                   "sample": f"{csteps} steps of {B} samples after 1 warm-up, best step {cms / 1e3:.2f} s "
                             f"({sum(ts) / 1e3:.0f} s of CPU work); {note}"}
        line = {"metric": "LID-VAE train samples/s", "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32" if args.precision == "fp32" else args.precision, "data": "synthetic",
                "config": make_config(B, world),
                "run": {"precision": args.precision, "optimizer_impl": "fused Adam over the flat parameter buffer",
                        "exchange": exchange, "exchange_ok": exchange_ok, "cuda_graph": bool(use_graph),
                        "own_kernel_launches_per_step": int(launches_per_step)},
                "e2e": {"value": e2e, "unit": "samples/s", "ms_per_step": ms_e2e, "h2d_bytes_per_step": B * 2 * 4 * world,
                        "d2h_bytes_per_step": 4 * world,
                        "how": "every step: pinned host batch -> device (copy stream, started one step ahead like a prefetching "
                               "loader: step_graphed(x, next_x=...)), whole-step graph, loss -> pinned host, host blocks on the "
                               "stream before the next step",
                        "pipelined": {"value": world * B / (ms_e2e_pipe * 1e-3), "ms_per_step": ms_e2e_pipe,
                                      "how": "same copies every step; the host reads loss i after enqueueing step i+1",
                                      "losses_read": len(seen)}},
                "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "cpu_baseline": cpu,
                "reference_same_gpu": ref_gpu, "extra": extra}
    if sampler:
        sampler.stop()
    # ---- multi-GPU: parity of the exchange path and the sharded all-pairs estimator, reported in the same line ----
    if world > 1:
        par = exchange_parity(dev, rank, world)
        ap_sh = allpairs_sharded_times(m, dev, rank, world, tr.peer)
        if rank == 0:
            line["exchange_parity"] = par
            line["extra"]["allpairs_sharded"] = ap_sh
    if rank == 0:
        print(json.dumps(line), flush=True)
    sys.stdout.flush()
    # Normal interpreter exit (at-exit hooks run).  The graph is released first: tearing down NCCL communicators that a
    # live CUDA graph still references can block; a watchdog turns a stuck teardown into a plain exit after 60 s.
    tr._graph = None
    del tr
    import gc
    gc.collect()
    torch.cuda.synchronize()
    if world > 1:
        import atexit

        def _bail():
            try:
                atexit._run_exitfuncs()
            finally:
                os._exit(0)
        wd = threading.Timer(60.0, _bail)
        wd.daemon = True
        wd.start()
        dist.barrier()
        dist.destroy_process_group()
        wd.cancel()


def exchange_parity(dev, rank, world, k=4):
    """k Adam steps from a fixed seed on a small LID-VAE (ICNN 128/256, FP32 kernels, global batch 1024): the batch-sharded
    run with the peer-memory exchange (eager and graph-replayed) and with the NCCL exchange against ONE process training on
    the full batch.  Collective; rank 0 returns the record."""
    import torch
    import torch.distributed as dist
    from vae_song_b200 import model, train

    def make():
        torch.manual_seed(0)
        mm = model.LIDVAE(dataset="pinwheel", icnn_channels=[128, 256], hidden_channels=[16, 8], inverse_lipschitz=0.2,
                          beta=0.5, precision="fp32")
        rng = np.random.default_rng(3)
        with torch.no_grad():
            for ic in (mm.decoder[0], mm.decoder[1]):
                H = ic.hidden_channel
                ic.W[0].param.copy_(torch.tensor(rng.normal(np.log(1.0 / H), 1.0, (H, H)), dtype=torch.float32))
                ic.W[1].param.copy_(torch.tensor(rng.normal(np.log(2.0 / H), 1.0, (1, H)), dtype=torch.float32))
                ic.A[0].bias.copy_(torch.tensor(rng.normal(-0.3, 1.0, (H,)), dtype=torch.float32))
        return mm.to(dev).train()

    solo = dist.new_group(ranks=[0])
    Bg = 1024
    g = torch.Generator(device="cpu").manual_seed(5)
    X = [torch.randn(Bg, 2, generator=g) for _ in range(k)]
    E = [torch.randn(Bg, 2, generator=g) for _ in range(k)]
    lo, hi = train.shard_rows(Bg, rank, world)
    single_losses = single_flat = None
    if rank == 0:
        ref = train.DataParallelTrainer(make(), lr=1e-3, process_group=solo)
        ref.world, ref.rank = 1, 0
        single_losses = [float(ref.step(x.to(dev), e.to(dev))[0]) for x, e in zip(X, E)]
        single_flat = ref.fp.flat.clone()
    out = {"steps": k, "global_batch": Bg, "world": world}
    flats = {}
    for name, mode, graphed in (("nccl", "nccl", False), ("peer", "peer", False), ("peer_graph", "peer", True)):
        try:
            tr = train.DataParallelTrainer(make(), lr=1e-3, comm=mode)
        except Exception as exc:                                # noqa: BLE001  (peer mapping unavailable: reported, not fatal)
            out[name] = {"error": str(exc)[:200]}
            continue
        if graphed:
            tr.capture(X[0][lo:hi].to(dev), E[0][lo:hi].to(dev))
        losses = []
        for x, e in zip(X, E):
            stepf = tr.step_graphed if graphed else tr.step
            total = stepf(x[lo:hi].to(dev), e[lo:hi].to(dev))[0]
            losses.append(float(tr.global_losses(total)[0]))
        timed_out = False
        try:
            tr.check()
        except Exception:                                       # noqa: BLE001
            timed_out = True
        mine = tr.fp.flat[:tr.fp.numel].clone()
        ref0 = mine.clone()
        dist.broadcast(ref0, src=0)
        flag = torch.tensor([int(torch.equal(mine, ref0))], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        flats[name] = mine
        if rank == 0:
            n = min(mine.numel(), single_flat.numel())
            out[name] = {"replicas_bit_identical": bool(int(flag) == 1), "exchange_timed_out": timed_out,
                         "max_rel_param_diff_vs_single_process": float((mine[:n] - single_flat[:n]).abs().max() / single_flat.abs().max()),
                         "max_rel_loss_diff_vs_single_process": max(abs(p - q) / abs(q) for p, q in zip(losses, single_losses)),
                         "losses": losses}
        tr._graph = None
        del tr
    if rank == 0:
        out["single_process_losses"] = single_losses
        if "peer" in flats and "nccl" in flats:
            out["max_rel_diff_peer_vs_nccl_path"] = float((flats["peer"] - flats["nccl"]).abs().max() / flats["nccl"].abs().max())
        ok = [v for v in out.values() if isinstance(v, dict) and "replicas_bit_identical" in v]
        out["pass"] = bool(ok) and all(v["replicas_bit_identical"] and not v["exchange_timed_out"] and
                                       v["max_rel_param_diff_vs_single_process"] < 5e-4 and
                                       v["max_rel_loss_diff_vs_single_process"] < 2e-4 for v in ok)
    return out


def allpairs_sharded_times(m, dev, rank, world, peer):
    """north_star: "the Lipschitz estimator shards pair tiles" -- utils.estimate_lipschitz_allpairs over N ranks (decode rows
    and pair tiles sharded, statistics combined by ONE peer-memory all-gather) against rank 0 alone, with device timings."""
    import torch
    import torch.distributed as dist
    from vae_song_b200 import utils as vutils
    solo = dist.new_group(ranks=[0])
    res = {}
    mm = m.eval()
    for N in (5000, 50000):
        torch.manual_seed(9)
        X = torch.randn(N, 2, device=dev)
        dist.broadcast(X, src=0)

        def t(fn, n=5):
            for _ in range(2):
                fn()
            torch.cuda.synchronize(); dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(n):
                out = fn()
            e1.record(); torch.cuda.synchronize()
            ms = torch.tensor([e0.elapsed_time(e1) / n], device=dev)
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            return float(ms), out
        sh_ms, sh = t(lambda: vutils.estimate_lipschitz_allpairs(mm.decode, X, peer=peer))
        if rank == 0:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            for _ in range(2):
                one = vutils.estimate_lipschitz_allpairs(mm.decode, X, process_group=solo)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(5):
                one = vutils.estimate_lipschitz_allpairs(mm.decode, X, process_group=solo)
            e1.record(); torch.cuda.synchronize()
            one_ms = e0.elapsed_time(e1) / 5
            pairs = N * (N - 1) // 2
            res[f"N{N}"] = {"pairs": pairs, "sharded_ms": sh_ms, "single_rank_ms": one_ms, "speedup": one_ms / sh_ms,
                            "sharded_pairs_per_s": pairs / (sh_ms * 1e-3),
                            "equal": bool(sh["count"] == one["count"] == pairs and sh["max"] == one["max"] and sh["min"] == one["min"]
                                          and abs(sh["mean"] - one["mean"]) <= 1e-6 * abs(one["mean"])),
                            "includes": "decode of this rank's rows + all-gather of Y + pair tiles + combine + host read-back"}
        dist.barrier()
    m.train()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=65536, help="per-GPU batch")
    ap.add_argument("--precision", default=os.environ.get("B200VAE_PRECISION", "f16x3"), choices=["fp32", "tf32", "tf32x3", "f16x3"],
                    help="arithmetic of the H x H contractions in the train step (fp32 = SIMT parity path)")
    ap.add_argument("--comm", default="auto", choices=["auto", "peer", "nccl"],
                    help="multi-GPU exchange back-end (train.DataParallelTrainer): peer-memory kernels or NCCL")
    ap.add_argument("--no-graph", action="store_true", help="launch the step eagerly instead of replaying a CUDA graph")
    ap.add_argument("--roofline-precision", default=None, choices=["fp32", "tf32", "tf32x3", "f16x3"],
                    help="precision of the kernel described by `roofline` (default: the step's --precision)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write what the last one computed (losses averaged over ranks, updated "
                         "parameters, BatchNorm buffers and, on one GPU, gradients) as DIR/<name>.npy; inputs and weights "
                         "are seeded, so runs with the same arguments on two builds can be compared array by array")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to the GPU arm (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
