"""VAE families with the reference's model.py API (constructor kwargs, forward/loss tuples, attribute
and state_dict names), backed by the fused CUDA kernels for the hot path:

  * LIDVAE.decode          two fused ICNN Brenier maps (ops.IcnnBrenierFn)   <- model.py:818-830
  * reparameterisation     ops.ReparamFn                                     <- model.py:843, :423-424
  * KL / recon / latent    ops.VaeLossFn (one launch)                        <- model.py:540-553, 587-616, 868-886

Encoder / MLP-conv decoder stacks are stock torch.nn layers (cuBLAS/cuDNN; out of scope, SURVEY.md
section 2).  Quirks kept on purpose (SURVEY.md Appendix B): LIDVAE.encode returns softplus(raw) as
log_var; losses are batch-mean-of-feature-sums; the latent-recon term averages over dim 0 (= L);
LRVAE.loss returns attached parts.  Reference defects D1/D2/D4 are fixed as supersets: LIDVAE accepts
image datasets, forward() accepts and ignores L, decode() needs no autograd graph.
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F
from torch import nn

from . import _C, module, ops

# dataset -> (in_channel, latent_channel, default hidden_channels, input_dim)
_FLEX_PRESETS = {
    "celeba": (3, 128, [32, 64, 128, 256], 64),
    "mnist": (1, 28, [32, 64, 128], 28),
    "fashionmnist": (1, 28, [32, 64, 128], 28),
    "cifar10": (3, 128, [32, 64, 128, 256], 32),
    "omniglot": (1, 32, [32, 64, 128, 256], 28),
    "pinwheel": (2, 2, [2, 2, 2, 2], 1),
    "chessboard": (2, 2, [2, 2, 2, 2], 1),
}
_LID_PRESETS = {
    "celeba": (3, 64, [32, 64, 128, 256], 64),
    "mnist": (1, 32, [32, 64, 128], 28),
    "fashionmnist": (1, 32, [32, 64, 128], 28),
    "cifar10": (3, 128, [32, 64, 128, 256], 32),
    "omniglot": (1, 32, [32, 64, 128], 28),
    "pinwheel": (2, 2, [2, 2, 2, 2], 1),
    "chessboard": (2, 2, [2, 2, 2, 2], 1),
}
_TOY = ("pinwheel", "chessboard")


def _halving_plan(input_dim, n):
    """Spatial size after n stride-2 stages and the output_padding each transposed conv needs."""
    pads, dim = [], input_dim
    for _ in range(n):
        pads.append((dim + 1) % 2)
        dim = (dim - 1) // 2 + 1
    return dim, pads[::-1]


def _lin_bn_act(i, o):
    return nn.Sequential(nn.Linear(i, o), nn.BatchNorm1d(o), nn.LeakyReLU())


def _vae_losses(x, xhat, mu, lv, z_in, z_rec, logmse):
    """(recon, kl, latent) through the fused loss kernel; absent parts come back as 0-d zeros."""
    return ops.VaeLossFn.apply(x, xhat, mu, lv, z_in, z_rec, bool(logmse))


class VAE(nn.Module):
    """Base class: alpha warm-up schedules (model.py:37-63)."""

    def __init__(self):
        super().__init__()
        self.last_kl_loss = 0.0

    # model.py:606 stores `loss_reg.item()` every step (one host sync per step, only ever read by the kl_adaptive warm-up once
    # per epoch).  Here the device scalar is kept and converted when somebody reads it, so the train step stays free of
    # host synchronisation (and capturable into a CUDA graph).
    @property
    def last_kl_loss(self):
        v = self.__dict__.get("_last_kl", 0.0)
        return float(v) if torch.is_tensor(v) else v

    @last_kl_loss.setter
    def last_kl_loss(self, v):
        self.__dict__["_last_kl"] = v

    # wu_alpha (the warm-up factor of the latent-recon term, model.py:37-63) is a Python float in the reference.  It stays
    # one here, but once `graph_scalars(device)` was called it is MIRRORED into a device scalar that the losses multiply
    # with, so that a CUDA graph captured once follows the per-epoch warm-up instead of baking the value in.  Classes that
    # never set it (LIDVAE, like the reference) have no such attribute: hasattr(model, "wu_alpha") is False for them.
    @property
    def wu_alpha(self):
        try:
            return self.__dict__["_wu_alpha"]
        except KeyError:
            raise AttributeError("wu_alpha") from None

    @wu_alpha.setter
    def wu_alpha(self, v):
        self.__dict__["_wu_alpha"] = float(v)
        dev = self.__dict__.get("_wu_dev")
        if dev is not None:
            dev.fill_(float(v))

    def graph_scalars(self, device):
        """Keep the warm-up factor on `device` as well (see wu_alpha); call before capturing the step into a CUDA graph."""
        if "_wu_alpha" in self.__dict__:
            self.__dict__["_wu_dev"] = torch.full((), self.__dict__["_wu_alpha"], dtype=torch.float32, device=device)
        return self

    def _lr_weight(self):
        """alpha * wu_alpha as the losses use it: a float, or a device scalar after graph_scalars()."""
        dev = self.__dict__.get("_wu_dev")
        return self.alpha * (dev if dev is not None else self.wu_alpha)

    def encode(self, input):
        raise NotImplementedError

    def decode(self, input):
        raise NotImplementedError

    def forward(self, input, latent_rand_sampling=True):
        raise NotImplementedError

    def loss(self, *args):
        raise NotImplementedError

    def warmup(self, epoch, max_epoch=None, wu_strat="linear", up_amount=None, start_epoch=0, repeat_interval=10):
        if not hasattr(self, "wu_alpha"):
            return False
        if epoch >= start_epoch:
            if wu_strat == "linear":
                inc = 1.0 / (max_epoch - start_epoch + 1) if up_amount is None else up_amount
                self.wu_alpha = min(self.wu_alpha + inc, 1.0)
            elif wu_strat == "exponential":
                t = epoch - start_epoch
                x = t * math.log(2) / (max_epoch - start_epoch) if up_amount is None else up_amount * t
                self.wu_alpha = max(min(math.exp(x) - 1.0, 1.0), 0.0)
            elif wu_strat == "repeat_linear":
                self.wu_alpha = min(1.0 / ((epoch % repeat_interval) + 1), 1.0)
            elif wu_strat == "kl_adaptive":
                self.wu_alpha = 1 / (1 + math.exp(self.last_kl_loss - 5))
        return True


class FlexibleVAE(VAE):
    """Config-driven MLP / conv VAE (model.py:69-501).  The stacks are stock layers; reparam and the
    losses (in the subclasses) go through the fused kernels."""

    def __init__(self, in_channel=1, latent_channel=32, hidden_channels=None, icnn_channels=None, input_dim=28,
                 beta=1.0, alpha=0.0, is_log_mse=False, dataset=None, z_source="Ex", bal_alpha=True, pwise_reg=False,
                 variational=True, encoder_type="mlp", decoder_type="mlp", residual_connection=False, fixed_var=False):
        if dataset not in _FLEX_PRESETS:
            raise ValueError(f"Invalid dataset: {dataset}")
        in_channel, latent_channel, default_h, input_dim = _FLEX_PRESETS[dataset]
        hidden_channels = list(default_h) if hidden_channels is None else hidden_channels
        super().__init__()
        self.variational = variational
        self.latent_channel = latent_channel
        self.beta, self.alpha = beta, alpha
        self.z_source = z_source
        self.wu_alpha = 0.0
        self.is_log_mse = is_log_mse
        self.balanced_alpha = bal_alpha
        self.pwise_reg = pwise_reg
        self.fixed_var = fixed_var
        self.data_type = "1d" if dataset in _TOY else "2d"
        self.residual_connection = residual_connection
        fc_dim, tpad = _halving_plan(input_dim, len(hidden_channels))
        rev = list(reversed(hidden_channels))

        if self.data_type == "1d" and encoder_type == "mlp":
            block = module.ResidualMLPBlock if residual_connection else _lin_bn_act
            self.encoder = self._mlp_stack(hidden_channels, in_channel, 2 * latent_channel, block)
        elif encoder_type == "mlp":
            self.encoder = self.make_encoder_mlp_2d(hidden_channels, in_channel, latent_channel)
        elif encoder_type == "conv":
            self.encoder = self.make_encoder_conv_2d(hidden_channels, in_channel, latent_channel, fc_dim)
        else:
            raise SystemExit(f"Invalid encoder type: {self.data_type} {encoder_type}")

        if self.data_type == "1d" and decoder_type == "mlp":
            if residual_connection:
                self.decoder = self.make_decoder_residual_mlp_1d(in_channel, latent_channel, rev)
            else:
                self.decoder = self.make_decoder_mlp_1d(in_channel, latent_channel, rev)
        elif decoder_type == "mlp":
            self.decoder = self.make_decoder_mlp_2d(in_channel, latent_channel, input_dim)
        elif decoder_type == "conv":
            self.decoder = self.make_decoder_conv_2d(in_channel, latent_channel, rev, fc_dim, tpad)
        else:
            raise SystemExit(f"Invalid decoder type: {self.data_type} {decoder_type}")

    # ---- builders (module nesting mirrors the reference so state_dict keys match) ----
    @staticmethod
    def _mlp_stack(hidden, i, o, block):
        dims = [i] + list(hidden) + [o]
        return nn.Sequential(*[block(a, b) for a, b in zip(dims[:-1], dims[1:])])

    def make_encoder_mlp_2d(self, hidden_channels, in_channel, latent_channel):
        blocks, last = [], in_channel
        for ch in hidden_channels:
            blocks.append(nn.Sequential(nn.Flatten(), nn.Linear(last, ch), nn.BatchNorm1d(ch), nn.LeakyReLU()))
            last = ch
        two = 2 * latent_channel
        blocks.append(nn.Sequential(nn.Linear(last, two), nn.BatchNorm1d(two), nn.LeakyReLU(), nn.Linear(two, two)))
        return nn.Sequential(*blocks)

    def make_encoder_conv_2d(self, hidden_channels, in_channel, latent_channel, fc_dim):
        blocks, last = [], in_channel
        for ch in hidden_channels:
            blocks.append(nn.Sequential(module.ResidualConvBlock(last, ch, 2), module.ResidualConvBlock(ch, ch, 1)))
            last = ch
        two = 2 * latent_channel
        blocks.append(nn.Sequential(nn.Flatten(), nn.Linear(last * fc_dim ** 2, two), nn.BatchNorm1d(two),
                                    nn.LeakyReLU(), nn.Linear(two, two)))
        return nn.Sequential(*blocks)

    def make_decoder_mlp_1d(self, in_channel, latent_channel, hidden_channels=()):
        blocks, last = [], latent_channel
        for ch in hidden_channels:
            blocks.append(_lin_bn_act(last, ch))
            last = ch
        tail_in = hidden_channels[-1] if len(hidden_channels) else in_channel   # reference quirk when empty
        blocks.append(nn.Sequential(nn.Linear(tail_in, in_channel)))
        return nn.Sequential(*blocks)

    def make_decoder_residual_mlp_1d(self, in_channel, latent_channel, hidden_channels=()):
        blocks, last = [], latent_channel
        for ch in hidden_channels:
            blocks.append(nn.Sequential(module.ResidualMLPBlock(last, ch)))
            last = ch
        tail_in = hidden_channels[-1] if len(hidden_channels) else in_channel
        blocks.append(nn.Sequential(module.ResidualMLPBlock(tail_in, in_channel)))
        return nn.Sequential(*blocks)

    def make_decoder_mlp_2d(self, in_channel, latent_channel, input_dim):
        full = input_dim ** 2 * in_channel
        half = full // 2
        return nn.Sequential(
            nn.Sequential(nn.Linear(latent_channel, half), nn.BatchNorm1d(half), nn.LeakyReLU(),
                          nn.Linear(half, half), nn.BatchNorm1d(half), nn.LeakyReLU()),
            nn.Sequential(nn.Linear(half, full), nn.BatchNorm1d(full), nn.LeakyReLU(), nn.Linear(full, full)),
            nn.Unflatten(1, (in_channel, input_dim, input_dim)),
        )

    def make_decoder_conv_2d(self, in_channel, latent_channel, hidden_channels, fc_dim, transpose_padding):
        last = hidden_channels[0]
        flat = last * fc_dim ** 2
        blocks = [nn.Sequential(nn.Linear(latent_channel, flat), nn.BatchNorm1d(flat), nn.LeakyReLU(),
                                nn.Unflatten(1, (last, fc_dim, fc_dim)), module.ResidualConvBlock(last, last, 1))]
        for ch, pad in zip(hidden_channels[1:], transpose_padding[:-1]):
            blocks.append(nn.Sequential(nn.ConvTranspose2d(last, ch, 3, 2, 1, pad), nn.BatchNorm2d(ch), nn.LeakyReLU()))
            last = ch
        blocks.append(nn.Sequential(nn.ConvTranspose2d(last, last, 3, 2, 1, transpose_padding[-1]),
                                    nn.BatchNorm2d(last), nn.LeakyReLU(), nn.ConvTranspose2d(last, in_channel, 3, 1, 1)))
        return nn.Sequential(*blocks)

    # ---- hot path ----
    # 1-D MLP stacks (Linear -> BatchNorm1d -> LeakyReLU chains) CAN run through the fused layer kernels (set True).  Off by
    # default: this family trains through main.py's staged, eagerly launched backward, which is HOST bound -- there the
    # Python-side autograd.Function costs more than the launches it saves (scripts/c1_run.py: 19.5 vs 14.2 ms per step at
    # batch 1024); it pays off when the step is replayed as a CUDA graph or the batch is large.
    fused_mlp = False

    def _stack_plan(self, name):
        """Cached ops.MlpPlan of self.encoder / self.decoder, or None when the stack is not a plain MLP chain."""
        if self.data_type != "1d" or self.residual_connection:
            return None
        return ops.cached_mlp_plan(self, name)

    def _run_stack(self, name, input):
        plan = self._stack_plan(name) if (self.fused_mlp and input.is_cuda and input.dim() == 2) else None
        if plan is not None and plan.linears[0].weight.device == input.device:
            return ops.fused_mlp(plan, input, self.training)
        return getattr(self, name)(input)

    def encode(self, input):
        ret = self._run_stack("encoder", input)
        mu, log_var = ret.split(ret.shape[1] // 2, 1)
        return mu, log_var

    def decode(self, input):
        return self._run_stack("decoder", input)

    def forward(self, input, latent_rand_sampling=True, L=1, eps=None):
        """-> (recon, mu, log_var, z_stack.detach() [L,B,D], z_recon_stack [L,B,D])   (model.py:418-447).
        `eps` ([L,B,D]) may be injected for tests; otherwise drawn with the reference's randn call."""
        mu, log_var = self.encode(input)
        if latent_rand_sampling:
            if eps is None:
                eps = torch.randn(L, *mu.shape, device=mu.device)
            z_stack = ops.ReparamFn.apply(mu, log_var, eps)          # [L,B,D]
        else:
            z_stack = mu.unsqueeze(0)
        Ls, B = z_stack.shape[0], input.shape[0]
        z_flat = z_stack.reshape(-1, z_stack.shape[-1])
        recon_attached = self.decode(z_flat)                          # grads reach decoder and encoder
        recon_lr = self.decode(z_flat.detach())                       # latent-recon path: decoder only ...
        z_rec_flat, _ = self.encode(recon_lr)                         # ... and the second encoder pass
        recon = recon_attached.view(Ls, B, *recon_attached.shape[1:]).mean(dim=0)
        z_rec_stack = z_rec_flat.view(Ls, B, *z_rec_flat.shape[1:])
        return recon, mu, log_var, z_stack.detach(), z_rec_stack


class NaiveAE(FlexibleVAE):
    def __init__(self, **kwargs):
        kwargs["variational"] = False
        super().__init__(**kwargs)

    def loss(self, input, output, mu, log_var, z_input=None, z_recon=None):
        rec, _, _ = _vae_losses(input, output, None, None, None, None, self.is_log_mse)
        return rec, rec.detach(), 0.0, 0.0


class VanillaVAE(FlexibleVAE):
    def loss(self, input, output, mu, log_var, z_input=None, z_recon=None):
        rec, reg, lr = _vae_losses(input, output, mu, log_var, z_input, z_recon, self.is_log_mse)
        return rec + reg * self.beta, rec.detach(), reg.detach(), lr.detach()


class LRVAE(FlexibleVAE):
    def __init__(self, alpha=0.01, **kwargs):
        super().__init__(**kwargs)
        self.alpha = alpha

    def loss(self, input, output, mu, log_var, z_input, z_recon):
        """-> (total, recon, beta*reg, alpha*wu*lr), all ATTACHED (main.py:262-284 back-propagates them
        one by one).  model.py:587-616."""
        rec, reg, lr = _vae_losses(input, output, mu, log_var, z_input, z_recon, self.is_log_mse)
        if self.pwise_reg:   # rarely used point-wise prior term, plain torch (model.py:608-611)
            mu_zp = z_input.mean(dim=1, keepdim=True)
            logvar_zp = torch.log(((z_input - mu_zp) ** 2).mean(dim=1))
            reg = reg / 2.0 + (-0.5 * (1 + logvar_zp - mu_zp ** 2 - logvar_zp.exp())).mean(dim=1).sum() / 2.0
        self.last_kl_loss = reg.detach()      # device scalar; converted on access (no host sync in the step)
        w = self._lr_weight()
        return rec + reg * self.beta + lr * w, rec, reg * self.beta, lr * w


class LIDVAE(VAE):
    """Left-invertible-decoder VAE: encoder + Brenier-map decoder of two ICNNs (model.py:637-886)."""

    def __init__(self, in_channel=1, latent_channel=32, hidden_channels=None, icnn_channels=[512, 1024], input_dim=28,
                 inverse_lipschitz=0.0, beta=1.0, is_log_mse=False, dataset=None, precision="fp32"):
        if len(icnn_channels) != 2:
            raise ValueError("2-length array was expected for `icnn_channels`")
        if dataset not in _LID_PRESETS:
            raise ValueError(f"Invalid dataset: {dataset}")
        in_channel, latent_channel, default_h, input_dim = _LID_PRESETS[dataset]
        hidden_channels = list(default_h) if hidden_channels is None else hidden_channels
        nn.Module.__init__(self)           # like the reference, VAE.__init__ is skipped: no wu_alpha attribute
        self.latent_channel = latent_channel
        self.il_factor = inverse_lipschitz / 2.0
        self.beta = beta
        self.is_log_mse = is_log_mse
        self.precision = precision
        fc_dim, _ = _halving_plan(input_dim, len(hidden_channels))
        if dataset in _TOY:
            self.encoder = self.make_encoder_1d(hidden_channels, in_channel, latent_channel)
            self.decoder = self.make_decoder_1d(in_channel, latent_channel, icnn_channels, input_dim)
        else:   # reference raises UnboundLocalError here (defect D1); this is the intended branch
            self.encoder = self.make_encoder_2d(hidden_channels, in_channel, latent_channel, fc_dim)
            self.decoder = self.make_decoder_2d(in_channel, latent_channel, icnn_channels, input_dim)

    def make_encoder_1d(self, hidden_channels, in_channel, latent_channel):
        blocks, last = [], in_channel
        for ch in hidden_channels:
            blocks.append(_lin_bn_act(last, ch))
            last = ch
        two = 2 * latent_channel
        blocks.append(nn.Sequential(nn.Linear(last, two), nn.BatchNorm1d(two), nn.LeakyReLU(), nn.Linear(two, two)))
        return nn.Sequential(*blocks)

    def make_encoder_2d(self, hidden_channels, in_channel, latent_channel, fc_dim):
        return FlexibleVAE.make_encoder_conv_2d(self, hidden_channels, in_channel, latent_channel, fc_dim)

    def _make_decoder(self, data_dim, latent_channel, icnn_channels, tail):
        first = module.ICNN(latent_channel, icnn_channels[0], precision=self.precision)
        self.register_buffer("B", torch.eye(data_dim, latent_channel, requires_grad=False))
        second = module.ICNN(data_dim, icnn_channels[1], precision=self.precision)
        return nn.ModuleList([first, second, tail])

    def make_decoder_1d(self, in_channel, latent_channel, icnn_channels, input_dim):
        return self._make_decoder(input_dim * in_channel, latent_channel, icnn_channels, nn.Identity())

    def make_decoder_2d(self, in_channel, latent_channel, icnn_channels, input_dim):
        return self._make_decoder(input_dim ** 2 * in_channel, latent_channel, icnn_channels,
                                  nn.Unflatten(1, (in_channel, input_dim, input_dim)))

    fused_encoder = True    # 1-D MLP encoders run through the fused Linear+BN+LeakyReLU layer kernels when they match

    def _encoder_plan(self):
        return ops.cached_mlp_plan(self, "encoder")

    def encode(self, input):
        plan = self._encoder_plan() if (self.fused_encoder and input.is_cuda and input.dim() == 2) else None
        if plan is not None:
            return ops.fused_mlp(plan, input, self.training, softplus_head=True)
        ret = self.encoder(input)
        mu, var = ret.split(ret.shape[1] // 2, 1)
        return mu, F.softplus(var)

    def decode(self, input):
        """y = grad(psi_1 + k|.|^2)( B . grad(psi_0 + k|.|^2)(z) ): two fused kernels, no autograd graph
        needed (works under no_grad and on plain tensors, unlike the reference)."""
        for ic in (self.decoder[0], self.decoder[1]):
            ic.precision = self.precision
        self.decoder[1].defer_param_grads_ok = False     # its dz feeds the first ICNN's backward, not the encoder
        _, x = self.decoder[0].brenier(input, self.il_factor)
        Dx, D = self.B.shape
        # x = x1 B^T (model.py:824): with B = eye(Dx, D) this is a zero-pad, which the wide kernels take implicitly
        # (input [B,D] of an ICNN(Dx,.)); a user-modified B falls back to the literal product
        if not self._B_is_eye():
            x = F.linear(x, self.B)
        elif Dx != D and Dx <= module.ICNN.FUSED_MAX_D:
            x = F.pad(x, (0, Dx - D))
        _, y = self.decoder[1].brenier(x, self.il_factor)
        return self.decoder[2](y)

    def decode_jacobian(self, input):
        """(recon, J [B,Dx,D], svals [B,min(Dx,D)]): decode(input), the decoder's exact Jacobian J = J2(x) . B . J1(z) and
        its singular values (descending) -- two fused Brenier-map forwards that also return their Jacobians
        (module.ICNN.brenier_jacobian) and one chain kernel (ops.jacobian_chain); the model's `B` buffer is the middle
        factor, so a user-modified B is honoured like decode() honours it.  recon is what decode() computes with the same
        kernels.  sigma_min >= inverse_lipschitz^2 is the decoder's inverse-Lipschitz guarantee (each map is 2 kappa-strongly
        monotone, kappa = inverse_lipschitz / 2).  Plain tensors, no autograd graph (not differentiable).  Decoders whose
        second ICNN is wider than the fused kernels take (the image-shaped ones, Dx > 4) raise B200VaeError."""
        first, second = self.decoder[0], self.decoder[1]
        for ic in (first, second):
            ic.precision = self.precision
        Dx, D = self.B.shape
        if Dx > module.ICNN.FUSED_MAX_D or D > module.ICNN.FUSED_MAX_D:
            raise _C.B200VaeError(f"decode_jacobian: the decoder's ICNN inputs (D = {D}, Dx = {Dx}) exceed the fused "
                                  f"kernels' limit of {module.ICNN.FUSED_MAX_D}")
        with torch.no_grad():
            _, x, J1 = first.brenier_jacobian(input, self.il_factor)
            if not self._B_is_eye():                       # the same x as decode() computes
                x = F.linear(x, self.B)
            elif Dx != D:
                x = F.pad(x, (0, Dx - D))
            _, y, J2 = second.brenier_jacobian(x, self.il_factor)
            J, svals = ops.jacobian_chain(J2, self.B, J1)
            return self.decoder[2](y), J, svals

    def decode_inverse(self, recon, z0=None, max_iter=ops.INVERSE_MAX_ITER, tol=None):
        """(z [B,D], status [B] int32, err_bound [B]): the decoder's left inverse, z with decode(z) ~ recon, by batched
        Newton steps on both Brenier maps (module.ICNN.brenier_inverse): x = T1^{-1}(recon), x1 = B^+ x (a slice when
        B = eye(Dx, D); a user-modified B through its pseudo-inverse -- rank-deficient B raises), z = T0^{-1}(x1).
        err_bound = e0 + ||B^+||_2 e1 / (2 kappa) bounds ||z - z*|| (T0^{-1} is 1/(2 kappa)-Lipschitz; +inf at
        inverse_lipschitz = 0); status is the worse of the two stages' (_C.INV_*, larger = worse).  z0 [B,D] warm-starts
        stage 0 and B . T0(z0) stage 1.  Plain tensors, no autograd graph.  Decoders whose ICNN inputs are wider than 4
        (the image-shaped ones) raise B200VaeError."""
        first, second = self.decoder[0], self.decoder[1]
        for ic in (first, second):
            ic.precision = self.precision
        Dx, D = self.B.shape
        if Dx > module.ICNN.FUSED_MAX_D or D > module.ICNN.FUSED_MAX_D:
            raise _C.B200VaeError(f"decode_inverse: the decoder's ICNN inputs (D = {D}, Dx = {Dx}) exceed the fused "
                                  f"kernels' limit of {module.ICNN.FUSED_MAX_D}")
        eye = self._B_is_eye()
        with torch.no_grad():
            if eye:
                pinv_norm = 1.0
            else:
                s = torch.linalg.svdvals(self.B.double())
                if s[-1] <= s[0] * D * torch.finfo(torch.float32).eps:
                    raise _C.B200VaeError(f"decode_inverse: the decoder's B buffer is rank-deficient (singular values "
                                          f"{s.tolist()}); it has no left inverse")
                pinv = torch.linalg.pinv(self.B.double()).float()
                pinv_norm = float(1.0 / s[-1])
            x0 = None
            if z0 is not None:
                _, x0 = first.brenier(z0, self.il_factor)
                x0 = F.pad(x0, (0, Dx - D)) if eye else F.linear(x0, self.B)
            x, st1, e1, _ = second.brenier_inverse(recon.reshape(recon.shape[0], -1), self.il_factor, z0=x0,
                                                   max_iter=max_iter, tol=tol)
            x1 = x[:, :D].contiguous() if eye else F.linear(x, pinv)
            z, st0, e0, _ = first.brenier_inverse(x1, self.il_factor, z0=z0, max_iter=max_iter, tol=tol)
            bound = e0 + pinv_norm * e1 / (2.0 * self.il_factor) if self.il_factor > 0 else torch.full_like(e0, float("inf"))
            return z, torch.maximum(st0, st1), bound

    def _prepare_decoder_early(self, input):
        """Training steps on the fused d <= 4 kernels: start building both ICNNs' prepared operands (they depend on the
        weights only) on side streams before the encoder runs -- ops.icnn_prepare_early.  Anything this cannot predict
        (wide inputs, FP32 small-batch routing, inference) simply prepares at the point of use as before."""
        if not (input.is_cuda and input.dim() == 2 and torch.is_grad_enabled() and self.early_prepare):
            return
        for slot, ic in enumerate((self.decoder[0], self.decoder[1])):
            ic.precision = self.precision
            prec, params = ic._prec(), ic._flat_params()
            if ic.in_channel > module.ICNN.FUSED_MAX_D or prec == _C.PREC_FP32 or not any(p.requires_grad for p in params):
                continue
            ops.icnn_prepare_early(params, ic.in_channel, ic.hidden_channel, ic._mode(), prec, input.shape[0], True, slot)

    early_prepare = True          # False: prepare inside the decoder call (the bit-identical reference arm of the tests)

    def _B_is_eye(self):
        v = self.__dict__.get("_b_eye_cache")
        if v is None or v[0] != self.B._version or v[1] != self.B.data_ptr():
            ok = bool(torch.equal(self.B, torch.eye(*self.B.shape, device=self.B.device, dtype=self.B.dtype)))
            v = (self.B._version, self.B.data_ptr(), ok)
            self.__dict__["_b_eye_cache"] = v
        return v[2]

    def forward(self, input, latent_recon=False, latent_rand_sampling=True, L=None, eps=None):
        """-> (recon, mu, log_var, z, None | z_recon).  `L` is accepted and ignored (reference defect D2);
        `eps` may be injected for tests."""
        self._prepare_decoder_early(input)
        mu, log_var = self.encode(input)
        if latent_rand_sampling:
            if eps is None:
                eps = torch.randn_like(mu)
            z = ops.ReparamFn.apply(mu, log_var, eps)
        else:
            z = mu
        recon = self.decode(z)
        if not latent_recon:
            return recon, mu, log_var, z, None
        z_recon, _ = self.encode(recon)
        return recon, mu, log_var, z, z_recon

    def forward_vae(self, input, latent_rand_sampling=True):
        return self.forward(input, latent_recon=False, latent_rand_sampling=latent_rand_sampling)

    def forward_Ex(self, input, latent_rand_sampling=True):
        return self.forward(input, latent_recon=True, latent_rand_sampling=latent_rand_sampling)

    def loss(self, input, output, mu, log_var, z_input=None, z_recon=None):
        rec, reg, _ = _vae_losses(input, output, mu, log_var, None, None, self.is_log_mse)
        return rec + reg * self.beta, rec.detach(), reg.detach(), 0.0


# ------------------------------------------------------------------------------------------------ set models
def chamfer_distance(points_pred, points_gt):
    """Symmetric Chamfer distance (model.py:896-912) through the tiled nearest-neighbour kernel: the [B,Np,Ng]
    matrix of torch.cdist is never materialised.  points_* [B, N, 3] -> scalar."""
    m_pg, m_gp = ops.NearestSqDistFn.apply(points_pred, points_gt)
    return (m_pg.mean(dim=1) + m_gp.mean(dim=1)).mean()


def _lin_bn_relu(i, o):
    return nn.Sequential(nn.Linear(i, o), nn.BatchNorm1d(o), nn.ReLU())


class SetEncoder(nn.Module):
    """DeepSets encoder (model.py:915-948): per-point MLP, permutation-invariant pooling, two heads."""

    def __init__(self, point_dim=3, hidden_dims=[128, 256, 512], latent_dim=128, pool_type="max"):
        super().__init__()
        self.pool_type = pool_type
        dims = [point_dim] + list(hidden_dims)
        self.phi = nn.ModuleList([_lin_bn_relu(a, b) for a, b in zip(dims[:-1], dims[1:])])
        self.fc_mu = nn.Linear(dims[-1], latent_dim)
        self.fc_logvar = nn.Linear(dims[-1], latent_dim)

    def forward(self, points):
        B, N, D = points.shape
        x = points.reshape(B * N, D)
        for layer in self.phi:
            x = layer(x)
        x = x.view(B, N, -1)
        s = x.mean(dim=1) if self.pool_type == "mean" else (x.sum(dim=1) if self.pool_type == "sum" else x.max(dim=1)[0])
        return self.fc_mu(s), self.fc_logvar(s)


class SetEncoderAttn(nn.Module):
    """Transformer set encoder (model.py:951-971), stock nn.TransformerEncoder + max pooling."""

    def __init__(self, point_dim=3, latent_dim=128, d_model=256, num_heads=4, num_layers=2, ff_dim=512, dropout=0.0):
        super().__init__()
        self.input_proj = nn.Linear(point_dim, d_model)
        layer = nn.TransformerEncoderLayer(d_model=d_model, nhead=num_heads, dim_feedforward=ff_dim, dropout=dropout,
                                           batch_first=True)
        self.encoder = nn.TransformerEncoder(layer, num_layers=num_layers)
        self.pool = nn.AdaptiveMaxPool1d(1)
        self.fc_mu = nn.Linear(d_model, latent_dim)
        self.fc_logvar = nn.Linear(d_model, latent_dim)

    def forward(self, points):
        x = self.encoder(self.input_proj(points))
        s = self.pool(x.transpose(1, 2)).squeeze(-1)
        return self.fc_mu(s), self.fc_logvar(s)


class SetDecoderAttn(nn.Module):
    """Learned point queries cross-attending to one latent token (model.py:974-994)."""

    def __init__(self, latent_dim=128, num_points=2048, d_model=256, num_heads=4, num_layers=2, ff_dim=512, dropout=0.0):
        super().__init__()
        self.num_points = num_points
        self.query_embed = nn.Parameter(torch.randn(num_points, d_model) * 0.02)
        self.latent_to_token = nn.Linear(latent_dim, d_model)
        layer = nn.TransformerDecoderLayer(d_model=d_model, nhead=num_heads, dim_feedforward=ff_dim, dropout=dropout,
                                           batch_first=True)
        self.decoder = nn.TransformerDecoder(layer, num_layers=num_layers)
        self.output_proj = nn.Linear(d_model, 3)

    def forward(self, z):
        memory = self.latent_to_token(z).unsqueeze(1)
        queries = self.query_embed.unsqueeze(0).expand(z.shape[0], -1, -1)
        return self.output_proj(self.decoder(tgt=queries, memory=memory))


class SetDecoder(nn.Module):
    """MLP decoder over [z, per-point query] (model.py:996-1029)."""

    def __init__(self, latent_dim=128, num_points=2048, hidden_dims=[512, 256, 128], point_dim=3):
        super().__init__()
        self.num_points = num_points
        self.point_queries = nn.Parameter(torch.randn(num_points, 64) * 0.02)
        dims = [latent_dim + 64] + list(hidden_dims)
        self.mlp = nn.ModuleList([_lin_bn_relu(a, b) for a, b in zip(dims[:-1], dims[1:])] + [nn.Linear(dims[-1], point_dim)])

    def forward(self, z):
        B = z.shape[0]
        q = self.point_queries.unsqueeze(0).expand(B, -1, -1)
        x = torch.cat([z.unsqueeze(1).expand(-1, self.num_points, -1), q], dim=-1).reshape(B * self.num_points, -1)
        for layer in self.mlp[:-1]:
            x = layer(x)
        return self.mlp[-1](x).view(B, self.num_points, -1)


class SetVAE(VAE):
    """Set VAE on point clouds (model.py:1032-1083); Chamfer reconstruction + Gaussian KL through the fused kernels."""

    def __init__(self, latent_channel=128, num_points=2048, encoder_hidden=[128, 256, 512], decoder_hidden=[512, 256, 128],
                 beta=1.0, is_log_mse=False, dataset="shapenet", pool_type="max", use_attention=True, d_model=256,
                 num_heads=4, num_encoder_layers=2, num_decoder_layers=2, ff_dim=512, attn_dropout=0.0):
        super().__init__()
        self.latent_channel, self.beta, self.is_log_mse, self.num_points = latent_channel, beta, is_log_mse, num_points
        self.data_type = "set"
        if use_attention:
            self.encoder = SetEncoderAttn(3, latent_channel, d_model, num_heads, num_encoder_layers, ff_dim, attn_dropout)
            self.decoder = SetDecoderAttn(latent_channel, num_points, d_model, num_heads, num_decoder_layers, ff_dim, attn_dropout)
        else:
            self.encoder = SetEncoder(3, encoder_hidden, latent_channel, pool_type)
            self.decoder = SetDecoder(latent_channel, num_points, decoder_hidden, 3)

    def encode(self, input):
        return self.encoder(input)

    def decode(self, input):
        return self.decoder(input)

    def _sample(self, mu, log_var, latent_rand_sampling, eps):
        if not latent_rand_sampling:
            return mu
        return ops.ReparamFn.apply(mu, log_var, torch.randn_like(mu) if eps is None else eps)

    def forward(self, input, latent_rand_sampling=True, L=1, eps=None):
        mu, log_var = self.encode(input)
        z = self._sample(mu, log_var, latent_rand_sampling, eps)
        return self.decode(z), mu, log_var, z, None

    def loss(self, input, output, mu, log_var, z_input=None, z_recon=None):
        rec = chamfer_distance(output, input)
        _, reg, _ = _vae_losses(None, None, mu, log_var, None, None, False)
        return rec + self.beta * reg, rec.detach(), reg.detach(), torch.tensor(0.0, device=input.device)


class SetLRVAE(SetVAE):
    """Set LR-VAE (model.py:1086-1114): decodes z.detach() and re-encodes for the latent-reconstruction term."""

    def __init__(self, alpha=0.01, **kwargs):
        super().__init__(**kwargs)
        self.alpha = alpha
        self.wu_alpha = 0.0

    def forward(self, input, latent_rand_sampling=True, L=1, eps=None):
        mu, log_var = self.encode(input)
        z = self._sample(mu, log_var, latent_rand_sampling, eps)
        recon = self.decode(z.detach())
        z_recon, _ = self.encode(recon)
        return recon, mu, log_var, z, z_recon

    def loss(self, input, output, mu, log_var, z_input, z_recon):
        rec = chamfer_distance(output, input)
        # [B,D] latents: dim 0 of the latent-recon mean is the batch here (no L axis); the fused kernel's Lz = B
        _, reg, lr = _vae_losses(None, None, mu, log_var, z_input, z_recon, False)
        self.last_kl_loss = reg.detach()      # device scalar; converted on access (no host sync in the step)
        w = self._lr_weight()
        return rec + self.beta * reg + w * lr, rec.detach(), (self.beta * reg).detach(), (w * lr).detach()
