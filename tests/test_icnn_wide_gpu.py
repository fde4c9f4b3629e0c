"""Parity of the fused wide-input ICNN kernels (csrc/icnn_wide.cu, d > 4: the MNIST-shaped decoder of BASELINE
configs[3]) against the fp64 oracle and the reference-generated goldens.  FP32 bounds of the north_star: rtol 1e-5 for
psi / xhat, 1e-4 for gradients (|a-b| <= rtol*|b| + rtol*max|b|, helpers.close_report); no fraction of elements is
exempted -- only the rows the oracle flags as kink-adjacent (helpers.kink_rows) are held to the loose bound."""
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
WIDE_GOLDEN = [c for c in ICNN_CASES if c[1] > 4]
# (d, H, B, regime, mode, kappa, seed): ragged sizes (d, H not multiples of 4 / 16 / 128; B across several row tiles),
# both weight modes, and the two shapes of the MNIST-shaped decoder at reduced batch
SHAPES = [
    (5, 40, 37, "mixed", 0, 0.1, 201),
    (7, 130, 300, "mixed", 1, 0.0, 202),
    (32, 512, 129, "mixed", 0, 0.1, 203),
    (784, 256, 40, "mixed", 0, 0.05, 204),
    (36, 96, 1000, "clampy", 1, 0.2, 205),
]


def run_wide(p, z, v, mode, kappa):
    from vae_song_b200 import ops
    dev = "cuda"
    params = [t.requires_grad_(True) for t in params_to_torch(p, dev)]
    zt = torch.tensor(z, dtype=torch.float32, device=dev, requires_grad=True)
    psi, xhat = ops.IcnnBrenierWideFn.apply(zt, kappa, mode, 0, *params)
    (xhat * torch.tensor(v, dtype=torch.float32, device=dev)).sum().backward()
    g = {k: t.grad.cpu().numpy() for k, t in zip(KEYS, params)}
    return psi.detach().cpu().numpy(), xhat.detach().cpu().numpy(), zt.grad.cpu().numpy(), g


def check_against_oracle(p, z, v, mode, kappa, out):
    psi, xhat, dz, g = out
    p64, z64, v64 = params_f32_as_f64(p), f32_as_f64(z), f32_as_f64(v)
    rpsi, rxhat, aux = io.icnn_brenier(z64, p64, mode, kappa, keep=True)
    rdz, rg = io.icnn_brenier_backward(z64, v64, p64, mode, kappa, None)
    close_report(psi, rpsi, 1e-5, "psi")
    close_rows(xhat, rxhat, 1e-5, "xhat", kink_rows(aux, H_RTOL[0]))
    close_rows(dz, rdz, 1e-4, "dz", kink_rows(aux, H_RTOL[0], with_h0=True), loose=5e-2)
    for k in KEYS:
        if np.abs(rg[k]).max() == 0:
            assert np.abs(g[k]).max() == 0, k          # A1b / A2b exact zeros (not None)
        else:
            close_report(g[k], rg[k], 1e-4, "grad " + k)


@pytest.mark.parametrize("shape", SHAPES, ids=[f"d{s[0]}_h{s[1]}_b{s[2]}" for s in SHAPES])
def test_wide_fwd_bwd_vs_oracle(shape):
    d, H, B, regime, mode, kappa, seed = shape
    p, z, v, _ = case_inputs(d, H, B, regime, seed)
    check_against_oracle(p, z, v, mode, kappa, run_wide(p, z, v, mode, kappa))


@pytest.mark.parametrize("case", WIDE_GOLDEN, ids=[c[0] for c in WIDE_GOLDEN])
def test_wide_vs_reference_golden(case):
    """Against what the unmodified reference produced (fp64 golden; oracle/make_golden.py)."""
    name, d, H, B, regime, mode, kappa, seed, with_gpsi = case
    assert not with_gpsi
    G = golden.load(os.path.join(GOLDEN, "icnn_cases.npz"))
    p, z, v, _ = case_inputs(d, H, B, regime, seed)
    psi, xhat, dz, g = run_wide(p, z, v, mode, kappa)
    pre = f"{name}/f64/"
    _, _, aux = io.icnn_brenier(f32_as_f64(z), params_f32_as_f64(p), mode, kappa, keep=True)
    close_report(psi, G[pre + "psi"], 2e-5, "psi")
    close_rows(xhat, G[pre + "xhat"], 2e-5, "xhat", kink_rows(aux, H_RTOL[0]))
    close_rows(dz, G[pre + "dz"], 1e-4, "dz", kink_rows(aux, H_RTOL[0], with_h0=True), loose=5e-2)
    for k in KEYS:
        key = pre + "g_" + k
        if key in G.files and np.abs(G[key]).max() > 0:
            close_report(g[k], G[key], 1e-4, "grad " + k)


def test_wide_is_deterministic_and_psi_only_inference():
    from vae_song_b200 import module, ops
    d, H, B = 32, 128, 70
    p, z, v, _ = case_inputs(d, H, B, "mixed", 77)
    a = run_wide(p, z, v, 0, 0.1)
    b = run_wide(p, z, v, 0, 0.1)
    for x, y in zip(a[:3], b[:3]):
        assert np.array_equal(x, y)                      # ordered reductions: bit-reproducible
    for k in KEYS:
        assert np.array_equal(a[3][k], b[3][k]), k
    ic = module.ICNN(d, H).cuda()
    with torch.no_grad():
        for t, src in zip(ic._flat_params(), params_to_torch(p, "cuda")):
            t.copy_(src)
        zt = torch.tensor(z, dtype=torch.float32, device="cuda")
        psi_inf = ic(zt)                                 # no_grad: fused psi-only kernels
    assert psi_inf.shape == (B, 1)
    close_report(psi_inf[:, 0].cpu().numpy(), a[0], 1e-6, "psi-only == psi of the Brenier call")
    zt2 = torch.tensor(z, dtype=torch.float32, device="cuda", requires_grad=True)
    psi_ad = ic(zt2)                                     # autograd idiom of the reference stays available
    xh = torch.autograd.grad(psi_ad, [zt2], torch.ones_like(psi_ad), create_graph=True)[0] + 2 * 0.1 * zt2
    _, _, aux = io.icnn_brenier(f32_as_f64(z), params_f32_as_f64(p), 0, 0.1)
    close_rows(xh.detach().cpu().numpy(), a[1], 1e-5, "autograd Brenier == fused", kink_rows(aux, H_RTOL[0]))


def test_wide_rejects_cpu():
    from vae_song_b200 import _C, ops
    p, z, v, _ = case_inputs(8, 16, 4, "mixed", 5)
    params = params_to_torch(p, "cpu")
    with pytest.raises(_C.B200VaeError):
        ops.IcnnBrenierWideFn.apply(torch.tensor(z, dtype=torch.float32), 0.0, 0, 0, *params)


PSI_SHAPES = [(8, 16, 4, "mixed", 0, 0.0, 5), (32, 128, 70, "mixed", 0, 0.1, 301), (36, 96, 300, "clampy", 1, 0.2, 302),
              (784, 64, 40, "mixed", 0, 0.05, 303)]


@pytest.mark.parametrize("with_v", [False, True], ids=["gpsi", "gpsi+v"])
@pytest.mark.parametrize("shape", PSI_SHAPES, ids=[f"d{s[0]}_h{s[1]}_b{s[2]}" for s in PSI_SHAPES])
def test_wide_psi_gradient_vs_oracle(shape, with_v):
    """First-order backward of psi for wide inputs (b200vae_icnn_wide_bwd_psi; SURVEY Appendix A last line), alone and
    together with the dL/dxhat path, against oracle.icnn_brenier_backward(..., gpsi): A1b / A2b are NOT zero here."""
    from vae_song_b200 import ops
    d, H, B, regime, mode, kappa, seed = shape
    p, z, v, gpsi = case_inputs(d, H, B, regime, seed)
    params = [t.requires_grad_(True) for t in params_to_torch(p, "cuda")]
    zt = torch.tensor(z, dtype=torch.float32, device="cuda", requires_grad=True)
    psi, xhat = ops.IcnnBrenierWideFn.apply(zt, kappa, mode, 0, *params)
    L = (psi * torch.tensor(gpsi, dtype=torch.float32, device="cuda")).sum()
    if with_v:
        L = L + (xhat * torch.tensor(v, dtype=torch.float32, device="cuda")).sum()
    L.backward()
    p64, z64 = params_f32_as_f64(p), f32_as_f64(z)
    _, _, aux = io.icnn_brenier(z64, p64, mode, kappa, keep=True)
    v64 = f32_as_f64(v) if with_v else np.zeros_like(z64)
    rdz, rg = io.icnn_brenier_backward(z64, v64, p64, mode, kappa, f32_as_f64(gpsi))
    close_rows(zt.grad.cpu().numpy(), rdz, 1e-4, "dz", kink_rows(aux, H_RTOL[0], with_h0=True), loose=5e-2)
    for k, t in zip(KEYS, params):
        assert np.abs(rg[k]).max() > 0, k
        close_report(t.grad.cpu().numpy(), rg[k], 1e-4, "grad " + k)


def test_wide_module_forward_is_twice_differentiable_on_the_fused_kernels():
    """module.ICNN(d > 4).forward used like the reference uses it: (a) psi.backward() -- first-order gradients through the
    fused psi-gradient kernels (no torch.nn.functional.linear on this path); (b) autograd.grad(create_graph=True) followed by
    backward -- the Brenier map and its double-backward (model.py:820-828)."""
    from vae_song_b200 import module
    d, H, B = 32, 128, 70
    p, z, v, gpsi = case_inputs(d, H, B, "mixed", 311)
    ic = module.ICNN(d, H).cuda()
    with torch.no_grad():
        for t, src in zip(ic._flat_params(), params_to_torch(p, "cuda")):
            t.copy_(src)
    p64, z64 = params_f32_as_f64(p), f32_as_f64(z)
    zt = torch.tensor(z, dtype=torch.float32, device="cuda", requires_grad=True)
    psi = ic(zt)
    assert psi.shape == (B, 1)
    (psi[:, 0] * torch.tensor(gpsi, dtype=torch.float32, device="cuda")).sum().backward()
    rdz, rg = io.icnn_brenier_backward(z64, np.zeros_like(z64), p64, 0, 0.0, f32_as_f64(gpsi))
    _, _, aux = io.icnn_brenier(z64, p64, 0, 0.0, keep=True)
    close_rows(zt.grad.cpu().numpy(), rdz, 1e-4, "dz of <gpsi, psi>", kink_rows(aux, H_RTOL[0], with_h0=True), loose=5e-2)
    for k, t in zip(KEYS, ic._flat_params()):
        close_report(t.grad.cpu().numpy(), rg[k], 1e-4, "grad " + k)
    ic.zero_grad(set_to_none=True)
    zt2 = torch.tensor(z, dtype=torch.float32, device="cuda", requires_grad=True)
    psi2 = ic(zt2) + 0.1 * zt2.pow(2).sum(1, keepdim=True)
    xh = torch.autograd.grad(psi2, [zt2], torch.ones_like(psi2), create_graph=True)[0]
    (xh * torch.tensor(v, dtype=torch.float32, device="cuda")).sum().backward()
    rdz2, rg2 = io.icnn_brenier_backward(z64, f32_as_f64(v), p64, 0, 0.1, None)
    _, rx, _ = io.icnn_brenier(z64, p64, 0, 0.1)
    close_rows(xh.detach().cpu().numpy(), rx, 1e-5, "xhat via autograd.grad", kink_rows(aux, H_RTOL[0]))
    close_rows(zt2.grad.cpu().numpy(), rdz2, 1e-4, "dz (double backward)", kink_rows(aux, H_RTOL[0], with_h0=True), loose=5e-2)
    for k, t in zip(KEYS, ic._flat_params()):
        if np.abs(rg2[k]).max() == 0:
            assert t.grad is None or float(t.grad.abs().max()) == 0.0, k
        else:
            close_report(t.grad.cpu().numpy(), rg2[k], 1e-4, "grad2 " + k)


def test_wide_implicit_zero_pad_equals_explicit_pad():
    """model.py:824 x = x1 B^T with B = eye(Dx, D) is a zero-pad: feeding [B,nz] to an ICNN(d) must equal feeding the
    explicitly padded [B,d] input -- outputs, dz (first nz columns) and every parameter gradient."""
    from vae_song_b200 import ops
    d, nz, H, B = 784, 32, 128, 50
    p, z, v, _ = case_inputs(d, H, B, "mixed", 31)
    z[:, nz:] = 0.0
    full = run_wide(p, z, v, 0, 0.1)
    params = [t.requires_grad_(True) for t in params_to_torch(p, "cuda")]
    zt = torch.tensor(z[:, :nz].copy(), dtype=torch.float32, device="cuda", requires_grad=True)
    psi, xhat = ops.IcnnBrenierWideFn.apply(zt, 0.1, 0, 0, *params)
    (xhat * torch.tensor(v, dtype=torch.float32, device="cuda")).sum().backward()
    assert xhat.shape == (B, d) and zt.grad.shape == (B, nz)
    close_report(psi.detach().cpu().numpy(), full[0], 1e-6, "psi")
    close_report(xhat.detach().cpu().numpy(), full[1], 1e-6, "xhat")
    close_report(zt.grad.cpu().numpy(), full[2][:, :nz], 1e-6, "dz")
    for k, t in zip(KEYS, params):
        if np.abs(full[3][k]).max() == 0:
            assert float(t.grad.abs().max()) == 0.0
        else:
            close_report(t.grad.cpu().numpy(), full[3][k], 1e-6, "grad " + k)
    check_against_oracle(p, z, v, 0, 0.1, full)


# ---- tcgen05 forward + backward (csrc/icnn_wide_tc.cu) ------------------------------------------------------------------------
# precision -> (psi, xhat, gradients).  tf32x3: north_star's FP32 bounds (four TMEM accumulators per tile: K in thirds +
# the lo-order products, icnn_wide_tc.cu); tf32: the stated looser bound (operands rounded to 11 bits; the batch-summed
# gradients of the 784-wide layer accumulate that over K = H = 1024 and B = 256: 2e-2 of the largest entry).
TC_BOUNDS = {3: (1e-5, 1e-5, 1e-4), 1: (2e-4, 5e-3, 2e-2)}
# ragged shapes, both weight modes, and the two EXACT shapes of the MNIST-shaped decoder at its config batch:
# ICNN(32,512) and ICNN(784,1024) at B = 256 (BASELINE configs[3])
TC_SHAPES = [(32, 512, 129, "mixed", 0, 0.1, 203), (784, 256, 40, "mixed", 0, 0.05, 204), (36, 96, 1000, "clampy", 1, 0.2, 205),
             (8, 1024, 300, "mixed", 0, 0.0, 206), (32, 512, 256, "mixed", 0, 0.1, 207), (784, 1024, 256, "mixed", 0, 0.1, 208)]


@pytest.mark.parametrize("prec", [3, 1], ids=["tf32x3", "tf32"])
@pytest.mark.parametrize("shape", TC_SHAPES, ids=[f"d{s[0]}_h{s[1]}_b{s[2]}" for s in TC_SHAPES])
def test_wide_tc_forward_and_backward_vs_oracle(shape, prec):
    from vae_song_b200 import ops
    d, H, B, regime, mode, kappa, seed = shape
    p, z, v, _ = case_inputs(d, H, B, regime, seed)
    params = [t.requires_grad_(True) for t in params_to_torch(p, "cuda")]
    zt = torch.tensor(z, dtype=torch.float32, device="cuda", requires_grad=True)
    psi, xhat = ops.IcnnBrenierWideFn.apply(zt, kappa, mode, prec, *params)
    (xhat * torch.tensor(v, dtype=torch.float32, device="cuda")).sum().backward()
    p64, z64, v64 = params_f32_as_f64(p), f32_as_f64(z), f32_as_f64(v)
    rpsi, rxhat, aux = io.icnn_brenier(z64, p64, mode, kappa, keep=True)
    rdz, rg = io.icnn_brenier_backward(z64, v64, p64, mode, kappa, None)
    bp, bx, bg = TC_BOUNDS[prec]
    close_report(psi.detach().cpu().numpy(), rpsi, bp, "psi")
    kr = kink_rows(aux, H_RTOL[prec])
    print(f"prec {prec} {shape[:3]}: {int(kr.sum())}/{B} kink-adjacent rows")
    close_rows(xhat.detach().cpu().numpy(), rxhat, bx, "xhat", kr, loose=2e-2)
    close_rows(zt.grad.cpu().numpy(), rdz, bg, "dz", kink_rows(aux, H_RTOL[prec], with_h0=True), loose=0.2)
    for k, t in zip(KEYS, params):
        if np.abs(rg[k]).max() == 0:
            assert float(t.grad.abs().max()) == 0.0, k
        else:
            # batch-summed: a kink-adjacent unit that lands on the other side moves one sample's share of a row, i.e.
            # O(1 / B) of it -- the only elements allowed outside the bound, and only in proportion to the kink rows
            close_report(t.grad.cpu().numpy(), rg[k], bg, "grad " + k, bad_frac=min(0.05, 2.0 * kr.mean() + 1e-9))


def test_wide_tc_matches_fp32_kernels_with_implicit_pad():
    from vae_song_b200 import ops
    d, nz, H, B = 784, 32, 512, 200
    p, z, v, _ = case_inputs(d, H, B, "mixed", 41)
    z[:, nz:] = 0.0
    params = params_to_torch(p, "cuda")
    zt = torch.tensor(z[:, :nz].copy(), dtype=torch.float32, device="cuda")
    ref = ops.IcnnBrenierWideFn.apply(zt, 0.1, 0, 0, *params)
    _, _, aux = io.icnn_brenier(f32_as_f64(z), params_f32_as_f64(p), 0, 0.1)
    for prec in (3, 1):
        bp, bx, _ = TC_BOUNDS[prec]
        got = ops.IcnnBrenierWideFn.apply(zt, 0.1, 0, prec, *params)
        assert got[1].shape == (B, d)
        close_report(got[0].cpu().numpy(), ref[0].cpu().numpy(), 2 * bp, "psi vs fp32 kernels")
        close_rows(got[1].cpu().numpy(), ref[1].cpu().numpy(), 2 * bx, "xhat vs fp32 kernels", kink_rows(aux, H_RTOL[prec]), loose=2e-2)
