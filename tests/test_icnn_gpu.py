"""Parity of the fused ICNN kernels (through ops -> ctypes -> C ABI) against the oracle and the
reference-generated goldens.  Tolerances: the north_star's rtol 1e-5 for psi / xhat and 1e-4 for
parameter gradients, applied as |a-b| <= rtol*|b| + rtol*max|b| (see helpers.close_report) with NO fraction of
elements waved through: rows in which the oracle itself finds a LeakyReLU pre-activation within the kernels' rounding
error of its kink (helpers.kink_rows, |h| < 4e-6 max|h|) are the only ones held to the loose bound instead."""
import os

import numpy as np
import pytest
import torch

from oracle import golden
from oracle import icnn_oracle as io
from oracle.make_golden import ICNN_CASES, case_inputs

from conftest import GOLDEN
from helpers import H_RTOL, KEYS, close_report, close_rows, f32_as_f64, kink_rows, params_f32_as_f64, params_to_torch

pytestmark = pytest.mark.gpu
SMALL_D = [c for c in ICNN_CASES if c[1] <= 4]


def run_ours(p, z, v, gpsi, mode, kappa, precision=0):
    from vae_song_b200 import ops
    dev = "cuda"
    params = [t.requires_grad_(True) for t in params_to_torch(p, dev)]
    zt = torch.tensor(z, dtype=torch.float32, device=dev, requires_grad=True)
    psi, xhat = ops.IcnnBrenierFn.apply(zt, kappa, mode, precision, *params)
    L = (xhat * torch.tensor(v, dtype=torch.float32, device=dev)).sum()
    if gpsi is not None:
        L = L + (psi * torch.tensor(gpsi, dtype=torch.float32, device=dev)).sum()
    L.backward()
    g = {k: t.grad.cpu().numpy() for k, t in zip(KEYS, params)}
    return psi.detach().cpu().numpy(), xhat.detach().cpu().numpy(), zt.grad.cpu().numpy(), g


@pytest.mark.parametrize("case", SMALL_D, ids=[c[0] for c in SMALL_D])
def test_fwd_bwd_vs_oracle(case):
    name, d, H, B, regime, mode, kappa, seed, with_gpsi = case
    p, z, v, gpsi = case_inputs(d, H, B, regime, seed)
    gp = gpsi if with_gpsi else None
    psi, xhat, dz, g = run_ours(p, z, v, gp, mode, kappa)
    p64, z64, v64 = params_f32_as_f64(p), f32_as_f64(z), f32_as_f64(v)
    gp64 = f32_as_f64(gpsi) if with_gpsi else None
    rpsi, rxhat, aux = io.icnn_brenier(z64, p64, mode, kappa, keep=True)
    rdz, rg = io.icnn_brenier_backward(z64, v64, p64, mode, kappa, gp64)
    close_report(psi, rpsi, 1e-5, "psi")
    close_rows(xhat, rxhat, 1e-5, "xhat", kink_rows(aux, H_RTOL[0]))
    close_rows(dz, rdz, 1e-4, "dz", kink_rows(aux, H_RTOL[0], with_h0=True))
    for k in KEYS:
        if np.abs(rg[k]).max() == 0:
            assert np.abs(g[k]).max() == 0, k          # A1b / A2b exact zeros (not None)
        else:
            close_report(g[k], rg[k], 1e-4, "grad " + k)


@pytest.mark.parametrize("case", SMALL_D, ids=[c[0] for c in SMALL_D])
def test_vs_reference_fp32_golden(case):
    """Against what the reference itself produced in fp32 on CPU (both sides carry fp32 noise)."""
    name, d, H, B, regime, mode, kappa, seed, with_gpsi = case
    G = golden.load(os.path.join(GOLDEN, "icnn_cases.npz"))
    p, z, v, gpsi = case_inputs(d, H, B, regime, seed)
    psi, xhat, dz, g = run_ours(p, z, v, gpsi if with_gpsi else None, mode, kappa)
    pre = f"{name}/f32/"
    _, _, aux = io.icnn_brenier(f32_as_f64(z), params_f32_as_f64(p), mode, kappa)
    close_report(psi, G[pre + "psi"], 2e-5, "psi")
    close_rows(xhat, G[pre + "xhat"], 2e-5, "xhat", kink_rows(aux, 2 * H_RTOL[0]))      # both sides carry fp32 noise
    close_report(g["A0w"], G[pre + "g_A0w"], 2e-4, "grad A0w")
    close_report(g["W1"], G[pre + "g_W1"], 2e-4, "grad W1")
    if pre + "g_W0" in G.files:
        close_report(g["W0"], G[pre + "g_W0"], 2e-4, "grad W0")
    else:
        close_report(g["W0"].reshape(-1)[::97], G[pre + "g_W0_sample"], 2e-4, "grad W0 sample")


@pytest.mark.parametrize("B", [1, 7, 128, 129, 1000])
def test_ragged_batches(B):
    """Empty tail rows of the last 128-sample tile must not leak into outputs or batch-summed grads."""
    rng = np.random.default_rng(5)
    p = io.random_params(rng, 2, 160, np.float64, "mixed")     # H not a multiple of 128 -> padded units
    z, v = rng.normal(0, 1, (B, 2)), rng.normal(0, 1, (B, 2))
    psi, xhat, dz, g = run_ours(p, z, v, None, 0, 0.2)
    p64 = params_f32_as_f64(p)
    rpsi, rxhat, aux = io.icnn_brenier(f32_as_f64(z), p64, 0, 0.2, keep=True)
    rdz, rg = io.icnn_brenier_backward(f32_as_f64(z), f32_as_f64(v), p64, 0, 0.2)
    close_report(psi, rpsi, 1e-5, "psi")
    close_rows(xhat, rxhat, 1e-5, "xhat", kink_rows(aux, H_RTOL[0]))
    close_rows(dz, rdz, 1e-4, "dz", kink_rows(aux, H_RTOL[0], with_h0=True))
    for k in ("A0w", "A0b", "A1w", "A2w", "W0", "W1"):
        close_report(g[k], rg[k], 1e-4, "grad " + k)


def test_full_size_properties():
    """B = 65536 (BASELINE decode size), H = 512 and 1024: size-independent checks.
    (a) tiling invariance: any row decoded alone == decoded inside the big batch, bit for bit;
    (b) sampled rows match the fp64 oracle; (c) gradient of a convex potential is monotone;
    (d) backward is additive over batch splits and linear in v."""
    from vae_song_b200 import ops
    rng = np.random.default_rng(9)
    B = 65536
    for H in (512, 1024):
        p = io.random_params(rng, 2, H, np.float64, "mixed")
        params = params_to_torch(p)
        z = torch.tensor(rng.normal(0, 1, (B, 2)), dtype=torch.float32, device="cuda")
        psi, xhat = ops.IcnnBrenierFn.apply(z, 0.1, 0, 0, *params)
        sel = torch.arange(0, B, 257, device="cuda")
        psi_s, xhat_s = ops.IcnnBrenierFn.apply(z[sel].contiguous(), 0.1, 0, 0, *params)
        assert torch.equal(psi[sel], psi_s) and torch.equal(xhat[sel], xhat_s)
        rpsi, rxhat, aux = io.icnn_brenier(z[sel].double().cpu().numpy(), params_f32_as_f64(p), 0, 0.1)
        close_report(psi_s.cpu().numpy(), rpsi, 1e-5, "psi")
        close_rows(xhat_s.cpu().numpy(), rxhat, 1e-5, "xhat", kink_rows(aux, H_RTOL[0]))
        perm = torch.randperm(B, device="cuda")
        mono = ((xhat - xhat[perm]) * (z - z[perm])).sum(1)
        assert (mono >= -1e-3 * mono.abs().max()).all()
        # (d) additivity / linearity of the double-backward
        v1 = torch.randn(B, 2, device="cuda"); v2 = torch.randn(B, 2, device="cuda")

        def bwd(zz, vv):
            ps = [t.clone().requires_grad_(True) for t in params]
            zt = zz.clone().requires_grad_(True)
            _, xh = ops.IcnnBrenierFn.apply(zt, 0.1, 0, 0, *ps)
            (xh * vv).sum().backward()
            return zt.grad, [t.grad for t in ps]
        dz_a, g_a = bwd(z, v1)
        dz_b, g_b = bwd(z, v2)
        dz_c, g_c = bwd(z, v1 + v2)
        close_report((dz_a + dz_b).cpu().numpy(), dz_c.cpu().numpy(), 1e-4, "dz linear")
        for k, a, b, c in zip(KEYS, g_a, g_b, g_c):
            if c.abs().max() > 0:
                close_report((a + b).cpu().numpy(), c.cpu().numpy(), 2e-4, "lin " + k)
        h = B // 2
        _, g_lo = bwd(z[:h].contiguous(), v1[:h].contiguous())
        _, g_hi = bwd(z[h:].contiguous(), v1[h:].contiguous())
        for k, a, b, c in zip(KEYS, g_lo, g_hi, g_a):
            if c.abs().max() > 0:
                close_report((a + b).cpu().numpy(), c.cpu().numpy(), 2e-4, "split " + k)


def test_reference_idiom_double_backward():
    """module.ICNN used exactly as model.py:820-828 uses it: autograd.grad(create_graph=True) then
    backward -- on OUR module, compared with the golden of the reference module."""
    from vae_song_b200 import module
    G = golden.load(os.path.join(GOLDEN, "icnn_cases.npz"))
    name, d, H, B, regime, mode, kappa, seed, _ = ICNN_CASES[0]
    p, z, v, _ = case_inputs(d, H, B, regime, seed)
    icnn = module.ICNN(d, H).cuda()
    with torch.no_grad():
        for t, k in zip(icnn._flat_params(), KEYS):
            t.copy_(torch.tensor(p[k], dtype=torch.float32))
    zt = torch.tensor(z, dtype=torch.float32, device="cuda", requires_grad=True)
    psi = icnn(zt) + kappa * zt.pow(2).sum(1, keepdim=True)
    xhat = torch.autograd.grad(psi, [zt], torch.ones_like(psi), create_graph=True)[0]
    (xhat * torch.tensor(v, dtype=torch.float32, device="cuda")).sum().backward()
    pre = f"{name}/f64/"
    _, _, aux = io.icnn_brenier(f32_as_f64(z), params_f32_as_f64(p), mode, kappa, keep=True)
    close_rows(xhat.detach().cpu().numpy(), G[pre + "xhat"], 1e-5, "xhat", kink_rows(aux, H_RTOL[0]))
    close_rows(zt.grad.cpu().numpy(), G[pre + "dz"], 1e-4, "dz", kink_rows(aux, H_RTOL[0], with_h0=True))
    close_report(icnn.W[0].param.grad.cpu().numpy(), G[pre + "g_W0"], 1e-4, "grad W0")
    close_report(icnn.A0.weight.grad.cpu().numpy(), G[pre + "g_A0w"], 1e-4, "grad A0w")


def test_errors_are_loud():
    from vae_song_b200 import _C, ops
    rng = np.random.default_rng(1)
    p = io.random_params(rng, 2, 32, np.float64, "mixed")
    with pytest.raises(_C.B200VaeError):
        ops.IcnnBrenierFn.apply(torch.zeros(4, 2), 0.0, 0, 0, *params_to_torch(p, "cpu"))      # CPU tensors
    with pytest.raises(_C.B200VaeError):
        ops.IcnnBrenierFn.apply(torch.zeros(4, 3, device="cuda"), 0.0, 0, 0, *params_to_torch(p))  # wrong d
