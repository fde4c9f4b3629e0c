"""Diagnostic: tcgen05 ICNN forward vs fp64 oracle and vs the SIMT path, with timings (run on the GPU box)."""
import sys, os, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import numpy as np, torch
from oracle import icnn_oracle as io
from vae_song_b200 import ops, _C

def params_t(p):
    return [torch.tensor(np.asarray(p[k], np.float32), device="cuda") for k in io.PARAM_KEYS]

def run(d, H, B, regime, prec, kappa=0.1, seed=0):
    rng = np.random.default_rng(seed)
    p = io.random_params(rng, d, H, np.float64, regime)
    z = rng.normal(0, 1, (B, d))
    P = params_t(p)
    zt = torch.tensor(z, dtype=torch.float32, device="cuda")
    ws = ops.icnn_prepare(P, d, H, 0, prec, B, False)
    psi, xhat, m1, m2 = ops.icnn_decode_fwd(zt, ws, d, H, 0, kappa, prec, True, True, True)
    torch.cuda.synchronize()
    p64 = {k: np.asarray(p[k], np.float32).astype(np.float64) for k in io.PARAM_KEYS}
    n = min(B, 2048)
    rpsi, rxhat, aux = io.icnn_brenier(zt[:n].double().cpu().numpy(), p64, 0, kappa)
    e1 = np.abs(psi[:n].cpu().numpy() - rpsi).max() / np.abs(rpsi).max()
    ex = np.abs(xhat[:n].cpu().numpy() - rxhat)
    e2 = ex.max() / np.abs(rxhat).max()
    e2med = np.median(ex) / np.abs(rxhat).max()
    Hp = (H + 127) // 128 * 128
    bits = ((m1[:n].cpu().numpy().astype(np.uint32)[:, :, None] >> np.arange(32, dtype=np.uint32)) & 1).reshape(n, -1)[:, :H]
    flips = int((bits != aux["mask1"]).sum())
    print(f"d={d} H={H} B={B} {regime} prec={prec}: psi relmax {e1:.2e}  xhat relmax {e2:.2e} (median {e2med:.1e})  mask flips {flips}/{bits.size}  mask2 mism {(m2[:n].cpu().numpy().astype(bool) != aux['mask2']).sum()}")
    return zt, ws

if __name__ == "__main__":
    names = {0: "fp32", 1: "tf32", 3: "tf32x3", 4: "f16x3"}
    fwd_only = "--fwd-only" in sys.argv
    precs = (4, 3, 1) if fwd_only else (0, 4, 3, 1)
    if "--precs" in sys.argv:
        precs = tuple(int(x) for x in sys.argv[sys.argv.index("--precs") + 1].split(","))
    for prec in precs:
        for (d, H, B, regime) in ((2, 256, 256, "mixed"), (2, 96, 77, "mixed"), (3, 512, 1000, "mixed"), (2, 1024, 4096, "mixed"), (2, 1024, 512, "default")):
            run(d, H, B, regime, prec)
    # timing at the headline size
    for prec in precs:
        for H in (512, 1024):
            zt, ws = run(2, H, 65536, "mixed", prec)
            for _ in range(3):
                ops.icnn_decode_fwd(zt, ws, 2, H, 0, 0.1, prec)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(10):
                ops.icnn_decode_fwd(zt, ws, 2, H, 0, 0.1, prec)
            e1.record(); torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / 10
            tf = io.flops_decode(2, H) * 65536 / ms / 1e9
            print(f"   TIMING {names[prec]} H={H}: {ms:.3f} ms  -> {tf:.1f} TFLOP/s algorithmic, {65536/ms/1e3:.2f} M samples/s")
            if fwd_only:
                continue
            # backward (rows + dP0 + finalize)
            rng = np.random.default_rng(5)
            p = io.random_params(rng, 2, H, np.float64, "mixed")
            P = params_t(p)
            wsb = ops.icnn_prepare(P, 2, H, 0, prec, 65536, True)
            vt = torch.randn(65536, 2, device="cuda")
            _, _, m1, m2 = ops.icnn_decode_fwd(zt, wsb, 2, H, 0, 0.1, prec, True, True, True)
            for _ in range(2):
                ops.icnn_decode_bwd(zt, vt, None, m1, m2, P, wsb, 2, H, 0, 0.1, prec)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(5):
                dzz, gg = ops.icnn_decode_bwd(zt, vt, None, m1, m2, P, wsb, 2, H, 0, 0.1, prec)
            e1.record(); torch.cuda.synchronize()
            msb = e0.elapsed_time(e1) / 5
            print(f"   TIMING {names[prec]} H={H} backward: {msb:.3f} ms ({io.flops_train(2,H)*65536/ (ms+msb)/1e9:.1f} TFLOP/s train-algorithmic fwd+bwd)")
            if prec != 0:
                ws0 = ops.icnn_prepare(P, 2, H, 0, 0, 65536, True)
                dz0, g0 = ops.icnn_decode_bwd(zt, vt, None, m1, m2, P, ws0, 2, H, 0, 0.1, 0)
                rel = lambda a, b: float((a - b).abs().max() / b.abs().max())
                print("      bwd vs fp32 kernels (same masks): dz %.2e" % rel(dzz, dz0), " ".join(f"{k}:{rel(a, b):.1e}" for k, a, b in zip(io.PARAM_KEYS, gg, g0) if float(b.abs().max()) > 0))
