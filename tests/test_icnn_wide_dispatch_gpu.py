"""Which kernels a wide-input call runs (b200vae_icnn_wide_fwd / _bwd): the oracle bounds of test_icnn_wide_gpu.py would
also hold if a tensor-core precision silently ran the FP32 kernels, so these tests pin the choice by comparing bits with
the FP32 path.  tcgen05 runs at tf32 / tf32x3 when d, nz and H are multiples of 4 and, in the forward, b0 / b1 / A2 are
16-byte aligned; otherwise the FP32 kernels run and give their bits exactly."""
import numpy as np
import pytest
import torch

from oracle import icnn_oracle as io
from oracle.make_golden import case_inputs

from helpers import H_RTOL, KEYS, close_report, close_rows, f32_as_f64, kink_rows, params_f32_as_f64, params_to_torch
from test_icnn_wide_gpu import TC_BOUNDS

pytestmark = pytest.mark.gpu


def run(p, z, v, mode, kappa, prec, a0b_offset=False):
    """psi, xhat, dz and the parameter gradients of <v, xhat>; with a0b_offset, A0b is a view 4 bytes into its buffer."""
    from vae_song_b200 import ops
    params = params_to_torch(p, "cuda")
    if a0b_offset:
        buf = torch.zeros(params[1].numel() + 1, dtype=torch.float32, device="cuda")
        buf[1:].copy_(params[1])
        params[1] = buf[1:]
        assert params[1].data_ptr() % 16 == 4
    params = [t.requires_grad_(True) for t in params]
    zt = torch.tensor(z, dtype=torch.float32, device="cuda", requires_grad=True)
    psi, xhat = ops.IcnnBrenierWideFn.apply(zt, kappa, mode, prec, *params)
    (xhat * torch.tensor(v, dtype=torch.float32, device="cuda")).sum().backward()
    g = {k: t.grad.cpu().numpy() for k, t in zip(KEYS, params)}
    return psi.detach().cpu().numpy(), xhat.detach().cpu().numpy(), zt.grad.cpu().numpy(), g


def test_tensor_core_shape_runs_tcgen05():
    d, H, B, regime, mode, kappa, seed = 32, 512, 129, "mixed", 0, 0.1, 203
    p, z, v, _ = case_inputs(d, H, B, regime, seed)
    ref, got = run(p, z, v, mode, kappa, 0), run(p, z, v, mode, kappa, 1)
    assert not np.array_equal(got[0], ref[0]), "tf32 psi has the FP32 kernels' bits"
    assert not np.array_equal(got[3]["W0"], ref[3]["W0"]), "tf32 dW0 has the FP32 kernels' bits"


@pytest.mark.parametrize("prec", [1, 3, 4], ids=["tf32", "tf32x3", "f16x3"])
def test_input_width_not_multiple_of_4_runs_fp32(prec):
    d, H, B, regime, mode, kappa, seed = 7, 132, 300, "mixed", 1, 0.1, 202
    p, z, v, _ = case_inputs(d, H, B, regime, seed)
    ref, got = run(p, z, v, mode, kappa, 0), run(p, z, v, mode, kappa, prec)
    for name, a, b in zip(("psi", "xhat", "dz"), got[:3], ref[:3]):
        assert np.array_equal(a, b), name
    for k in KEYS:
        assert np.array_equal(got[3][k], ref[3][k]), k


def test_unaligned_bias_forward_runs_fp32():
    d, H, B, regime, mode, kappa, seed = 32, 512, 129, "mixed", 0, 0.1, 203
    p, z, v, _ = case_inputs(d, H, B, regime, seed)
    ref = run(p, z, v, mode, kappa, 0, a0b_offset=True)
    got = run(p, z, v, mode, kappa, 1, a0b_offset=True)
    assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1])
    # the backward does not read b0 / b1 / A2 with 16-byte loads: it stays on tcgen05, within the tf32 bounds
    assert not np.array_equal(got[3]["W0"], ref[3]["W0"])
    p64, z64, v64 = params_f32_as_f64(p), f32_as_f64(z), f32_as_f64(v)
    _, _, aux = io.icnn_brenier(z64, p64, mode, kappa, keep=True)
    rdz, rg = io.icnn_brenier_backward(z64, v64, p64, mode, kappa, None)
    _, _, bg = TC_BOUNDS[1]
    kr = kink_rows(aux, H_RTOL[1])
    close_rows(got[2], rdz, bg, "dz", kink_rows(aux, H_RTOL[1], with_h0=True), loose=0.2)
    for k in KEYS:
        if np.abs(rg[k]).max() == 0:
            assert np.abs(got[3][k]).max() == 0, k
        else:
            close_report(got[3][k], rg[k], bg, "grad " + k, bad_frac=min(0.05, 2.0 * kr.mean() + 1e-9))


def test_unknown_precision_is_refused():
    from vae_song_b200 import _C
    p, z, v, _ = case_inputs(32, 64, 16, "mixed", 5)
    for prec in (2, 99):
        with pytest.raises(_C.B200VaeError):
            run(p, z, v, 0, 0.1, prec)
