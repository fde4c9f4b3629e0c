"""Building blocks with the reference's module.py API.

PositiveLinear / ICNN keep the reference parameter names and init order (module.py:97-140) so a
reference ``state_dict`` loads unchanged and a shared seed gives identical initial weights; their
arithmetic runs in the fused CUDA kernels (ops.IcnnPotentialFn / ops.IcnnBrenierFn).
Residual blocks are stock cuDNN/cuBLAS layers (out of the hot-path scope, SURVEY.md section 2).
"""
from __future__ import annotations

import math

import torch
from torch import nn

from . import _C, ops


class PositiveLinear(nn.Module):
    """Bias-free linear map with positive weights: exp(param) (default) or clamp(param, min=1e-2).
    Reference: module.py:97-114."""

    def __init__(self, in_channel, out_channel, is_exp=True):
        super().__init__()
        self.param = nn.Parameter(torch.empty(out_channel, in_channel))
        nn.init.kaiming_uniform_(self.param, a=math.sqrt(5.0))
        self.is_exp = is_exp

    def positive_weight(self):
        return self.param.exp() if self.is_exp else self.param.clamp(min=1e-2)

    def forward(self, input):
        # Stand-alone use only (inside ICNN the reparam is fused into the kernels' prepare step).
        return nn.functional.linear(input, self.positive_weight())


class ICNN(nn.Module):
    """Input-convex network psi(z): R^d -> R, 2 hidden layers (module.py:117-148).

    forward(z) -> psi [B,1], twice differentiable in z (so the reference idiom
    ``autograd.grad(icnn(z), [z], ones, create_graph=True)`` keeps working);
    brenier(z, kappa) -> (psi [B], grad_z(psi + kappa|z|^2) [B,d]) in ONE fused kernel.
    ``precision`` selects the arithmetic of the H x H contractions: fp32 (parity), f16x3 / tf32x3 (fp32-grade, tensor
    cores: fp16 / tf32 hi-lo operand pairs, three MMAs per product; f16x3 runs at twice the MMA rate), tf32."""

    def __init__(self, in_channel, hidden_channel=128, num_layers=2, precision="fp32"):
        super().__init__()
        if num_layers != 2:
            raise ValueError("the fused ICNN kernels implement the reference's num_layers=2 network")
        self.activation = nn.LeakyReLU(0.2)
        W, A = [], []
        for _ in range(num_layers - 1):
            W.append(PositiveLinear(hidden_channel, hidden_channel))
            A.append(nn.Linear(in_channel, hidden_channel))
        W.append(PositiveLinear(hidden_channel, 1))
        A.append(nn.Linear(in_channel, 1))
        self.W = nn.Sequential(*W)
        self.A = nn.Sequential(*A)
        self.A0 = nn.Linear(in_channel, hidden_channel)
        self.in_channel, self.hidden_channel = in_channel, hidden_channel
        self.precision = precision

    # order = _C.PARAM_FIELDS
    def _flat_params(self):
        return (self.A0.weight, self.A0.bias, self.A[0].weight, self.A[0].bias, self.A[1].weight, self.A[1].bias,
                self.W[0].param, self.W[1].param)

    def _mode(self):
        e0, e1 = self.W[0].is_exp, self.W[1].is_exp
        if e0 != e1:
            raise ValueError("mixed is_exp settings across the ICNN's PositiveLinear layers are not supported")
        return _C.WEIGHT_EXP if e0 else _C.WEIGHT_CLAMP

    def _prec(self):
        try:
            return _C.PRECISIONS[self.precision]
        except KeyError:
            raise ValueError(f"unknown precision {self.precision!r}; choose from {list(_C.PRECISIONS)}")

    FUSED_MAX_D = 4      # widest input the fused kernels keep in registers; wider inputs take the GEMM-composed path

    def forward(self, input):
        if self.in_channel > self.FUSED_MAX_D:
            return ops.IcnnPotentialWideFn.apply(input, self._mode(), self._prec(), *self._flat_params())
        return ops.IcnnPotentialFn.apply(input, self._mode(), self._prec(), *self._flat_params())

    FP32_TILED_BELOW = 6144   # measured crossover (scripts/fp32_crossover.py): below it the tiled GEMM chain is the faster FP32 path

    def brenier(self, input, kappa=0.0):
        """(psi [B], xhat [B,d]).  For wide ICNNs `input` may be [B,nz] with nz < d: zero-padded to d inside the kernels.

        Kernel choice: d > 4 -> the wide-input kernels (tcgen05 or FP32 tile GEMMs).  d <= 4: the fused sample-stationary
        kernels (tcgen05 pair kernels for tf32 / tf32x3 / f16x3; FP32 SIMT for fp32) -- except FP32 at small batches, where one CTA
        per 128 samples would leave most of the 148 SMs idle (a batch-256 step ran on 2 SMs): those go through the FP32
        tile-GEMM chain of csrc/icnn_wide.cu, which tiles over the hidden width as well (same arithmetic, same bounds)."""
        prec = self._prec()
        wide = self.in_channel > self.FUSED_MAX_D or (
            prec == _C.PREC_FP32 and input.dim() == 2 and input.shape[0] < self.FP32_TILED_BELOW
            and input.shape[1] == self.in_channel)
        params = self._flat_params()
        if not wide and not (torch.is_grad_enabled() and (input.requires_grad or any(p.requires_grad for p in params))):
            # inference: no graph, and the prepared workspace is reused while the weights are unchanged
            if not hasattr(self, "_infer_cache"):
                self._infer_cache = {}
            return ops.icnn_brenier_inference(input, float(kappa), self._mode(), prec, params, self._infer_cache)
        fn = ops.IcnnBrenierWideFn if wide else ops.IcnnBrenierFn
        if not wide:
            ops.set_defer_hint(self.defer_param_grads_ok)
        return fn.apply(input, float(kappa), self._mode(), prec, *params)

    defer_param_grads_ok = True      # see ops.set_defer_hint; model.LIDVAE clears it on its second ICNN

    def _check_jacobian_limits(self, what):
        d, H = self.in_channel, self.hidden_channel
        if d > self.FUSED_MAX_D:
            raise _C.B200VaeError(f"{what}: input width d = {d} exceeds the fused kernels' limit d <= {self.FUSED_MAX_D}")
        if self._prec() != _C.PREC_FP32 and (d > 3 or H > 1024):
            raise _C.B200VaeError(f"{what}: precision {self.precision!r} needs d <= 3 and H <= 1024 "
                                  f"(got d = {d}, H = {H}); use precision='fp32'")
        if not hasattr(self, "_infer_cache"):
            self._infer_cache = {}

    def brenier_jacobian(self, input, kappa=0.0):
        """(psi [B], xhat [B,d], jac [B,d,d]): brenier() plus the exact Jacobian d xhat / d z = A0^T diag(2 s0^2 gx1) A0
        + 2 kappa I, from the same fused forward (symmetric, >= 2 kappa I).  Plain tensors without an autograd graph:
        the Jacobian is not differentiable.  Every batch size runs the fused kernels (also FP32 below FP32_TILED_BELOW).
        Limits: d <= 4 (FP32), d <= 3 and H <= 1024 (tensor-core precisions); B200VaeError otherwise."""
        self._check_jacobian_limits("brenier_jacobian")
        return ops.icnn_brenier_jacobian(input, float(kappa), self._mode(), self._prec(), self._flat_params(),
                                         self._infer_cache)

    def brenier_inverse(self, x, kappa=0.0, z0=None, max_iter=ops.INVERSE_MAX_ITER, tol=None):
        """(z [B,d], status [B] int32, err_bound [B], rounds): the left inverse z = T^{-1}(x) of brenier()'s map
        T = grad(psi + kappa|.|^2), by batched Newton steps on the fused Jacobian kernels (ops.icnn_brenier_inverse;
        status values _C.INV_*).  ||z - T^{-1}(x)|| <= err_bound = ||T(z) - x|| / (2 kappa) on every row (+inf at
        kappa = 0).  Plain tensors, not differentiable.  Same limits as brenier_jacobian."""
        self._check_jacobian_limits("brenier_inverse")
        return ops.icnn_brenier_inverse(x, float(kappa), self._mode(), self._prec(), self._flat_params(), self._infer_cache,
                                        z0=z0, max_iter=max_iter, tol=tol)


class PlainConvolution(nn.Module):
    """conv3x3-BN-LReLU twice, no skip connection (module.py:4-26; stock cuDNN layers, outside the hot path)."""

    def __init__(self, in_channel, out_channel, stride=1):
        super().__init__()
        self.activation = nn.LeakyReLU()
        self.conv1 = nn.Sequential(nn.Conv2d(in_channel, out_channel, 3, stride, 1), nn.BatchNorm2d(out_channel),
                                   self.activation)
        self.conv2 = nn.Sequential(nn.Conv2d(out_channel, out_channel, 3, 1, 1), nn.BatchNorm2d(out_channel),
                                   self.activation)

    def forward(self, input):
        return self.conv2(self.conv1(input))


class ResidualConvBlock(nn.Module):
    """conv3x3-BN-LReLU-conv3x3-BN (+ 1x1 projection when shape changes) -> LReLU.  module.py:29-58."""

    def __init__(self, in_channel, out_channel, stride=1):
        super().__init__()
        self.activation = nn.LeakyReLU()
        self.conv1 = nn.Sequential(nn.Conv2d(in_channel, out_channel, 3, stride, 1), nn.BatchNorm2d(out_channel),
                                   self.activation)
        self.conv2 = nn.Sequential(nn.Conv2d(out_channel, out_channel, 3, 1, 1), nn.BatchNorm2d(out_channel))
        if stride == 1 and in_channel == out_channel:
            self.identity = nn.Identity()
        else:
            self.identity = nn.Sequential(nn.Conv2d(in_channel, out_channel, 1, stride, 0), nn.BatchNorm2d(out_channel))

    def forward(self, input):
        return self.activation(self.conv2(self.conv1(input)) + self.identity(input))


class ResidualMLPBlock(nn.Module):
    """Linear-BN-LReLU-Linear-BN (+ linear projection when width changes) -> LReLU.  module.py:62-93."""

    def __init__(self, in_channel, out_channel, stride=1):
        super().__init__()
        self.activation = nn.LeakyReLU()
        self.mlp1 = nn.Sequential(nn.Linear(in_channel, out_channel), nn.BatchNorm1d(out_channel), self.activation)
        self.mlp2 = nn.Sequential(nn.Linear(out_channel, out_channel), nn.BatchNorm1d(out_channel))
        if stride == 1 and in_channel == out_channel:
            self.identity = nn.Identity()
        else:
            self.identity = nn.Sequential(nn.Linear(in_channel, out_channel), nn.BatchNorm1d(out_channel))

    def forward(self, input):
        return self.activation(self.mlp2(self.mlp1(input)) + self.identity(input))


class LinearModule_EP(nn.Module):
    """The reference's unconstrained ICNN-shaped MLP (module.py:151-187: plain Linear W layers, last W maps to in_channel;
    not used by any model of the reference).  Kept for API parity: same attribute names, init order and forward."""

    def __init__(self, in_channel, hidden_channel=128, num_layers=2):
        super().__init__()
        self.activation = nn.LeakyReLU(0.2)
        W, A = [], []
        for _ in range(num_layers - 1):
            W.append(nn.Linear(hidden_channel, hidden_channel))
            A.append(nn.Linear(in_channel, hidden_channel))
        W.append(nn.Linear(hidden_channel, in_channel))
        A.append(nn.Linear(in_channel, 1))
        self.W = nn.Sequential(*W)
        self.A = nn.Sequential(*A)
        self.A0 = nn.Linear(in_channel, hidden_channel)

    def forward(self, input):
        x = self.activation(self.A0(input)).pow(2)
        for w, a in zip(self.W, self.A):
            x = self.activation(w(x) + a(input))
        return x
