#!/usr/bin/env python
"""Generate tests/golden/*.npz by RUNNING THE UNMODIFIED REFERENCE.

    python oracle/make_golden.py            # needs a reference checkout (oracle/fetch_ref.find_reference); writes tests/golden/

The reference (pure Python/PyTorch) is imported from that checkout exactly as shipped; nothing
is copied.  utils.py imports matplotlib (absent here) at module scope, so empty stub modules are
registered first (SURVEY.md section 8(c)).  Inputs and ICNN parameters are drawn with numpy's
``default_rng`` through ``oracle.icnn_oracle.random_params`` so that tests can rebuild them
bit-identically on any box from (seed, shape) alone; only reference OUTPUTS are stored.
The fixtures never travel back into the product path: tests read them, nothing else does.
"""
from __future__ import annotations

import os
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
OUT = os.path.join(ROOT, "tests", "golden")

from oracle import golden  # noqa: E402
from oracle import icnn_oracle as io  # noqa: E402
from oracle.fetch_ref import REF_SRC as REF  # noqa: E402


def import_reference():
    if not (REF and os.path.isfile(os.path.join(REF, "module.py"))):
        raise FileNotFoundError("no reference checkout: set VAE_SONG_REFERENCE or place it beside the repository")
    for name in ("matplotlib", "matplotlib.pyplot"):
        if name not in sys.modules:
            m = types.ModuleType(name)
            sys.modules[name] = m
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    sys.path.insert(0, REF)
    import module as ref_module  # noqa
    import model as ref_model  # noqa
    import utils as ref_utils  # noqa
    return ref_module, ref_model, ref_utils


def load_icnn(icnn, p, tdtype):
    t = lambda a: torch.tensor(np.asarray(a, dtype=np.float64), dtype=tdtype)
    with torch.no_grad():
        icnn.A0.weight.copy_(t(p["A0w"])); icnn.A0.bias.copy_(t(p["A0b"]))
        icnn.A[0].weight.copy_(t(p["A1w"])); icnn.A[0].bias.copy_(t(p["A1b"]))
        icnn.A[1].weight.copy_(t(p["A2w"])); icnn.A[1].bias.copy_(t(p["A2b"]))
        icnn.W[0].param.copy_(t(p["W0"])); icnn.W[1].param.copy_(t(p["W1"]))


def icnn_grads(icnn):
    g = lambda q: q.grad.detach().numpy().copy()
    return dict(A0w=g(icnn.A0.weight), A0b=g(icnn.A0.bias), A1w=g(icnn.A[0].weight), A1b=g(icnn.A[0].bias),
                A2w=g(icnn.A[1].weight), A2b=g(icnn.A[1].bias), W0=g(icnn.W[0].param), W1=g(icnn.W[1].param))


# (name, d, H, B, regime, mode, kappa, seed, with_gpsi)
ICNN_CASES = [
    ("d2_h32_mixed_exp", 2, 32, 33, "mixed", 0, 0.15, 101, False),
    ("d2_h32_mixed_gpsi", 2, 32, 33, "mixed", 0, 0.0, 102, True),
    ("d3_h64_clampy_clamp", 3, 64, 40, "clampy", 1, 0.1, 103, False),
    ("d1_h32_mixed_exp", 1, 32, 17, "mixed", 0, 0.05, 104, False),
    ("d4_h96_default_exp", 4, 96, 21, "default", 0, 0.0, 105, False),
    ("d2_h512_mixed_exp", 2, 512, 96, "mixed", 0, 0.1, 106, False),
    ("d2_h1024_mixed_exp", 2, 1024, 96, "mixed", 0, 0.1, 107, False),
    ("d2_h512_default_exp", 2, 512, 64, "default", 0, 0.0, 108, False),
    ("d2_h1024_default_clamp", 2, 1024, 64, "default", 1, 0.25, 109, False),
    ("d32_h128_mixed_exp", 32, 128, 24, "mixed", 0, 0.1, 110, False),
    ("d784_h64_mixed_exp", 784, 64, 8, "mixed", 0, 0.05, 111, False),
]


def case_inputs(d, H, B, regime, seed):
    rng = np.random.default_rng(seed)
    p = io.random_params(rng, d, H, np.float64, regime)
    z = rng.normal(0, 1.0, (B, d))
    v = rng.normal(0, 1.0, (B, d))
    gpsi = rng.normal(0, 1.0, (B,))
    return p, z, v, gpsi


def gen_icnn(ref_module):
    out = {}
    for name, d, H, B, regime, mode, kappa, seed, with_gpsi in ICNN_CASES:
        p, z, v, gpsi = case_inputs(d, H, B, regime, seed)
        for tag, tdtype in (("f64", torch.float64), ("f32", torch.float32)):
            icnn = ref_module.ICNN(d, H).to(tdtype)
            for w in icnn.W:
                w.is_exp = (mode == 0)
            load_icnn(icnn, p, tdtype)
            zt = torch.tensor(z, dtype=tdtype, requires_grad=True)
            psi = icnn(zt) + kappa * zt.pow(2).sum(1, keepdim=True)        # model.py:820
            xhat = torch.autograd.grad(psi, [zt], torch.ones_like(psi), create_graph=True)[0]  # :822
            L = (xhat * torch.tensor(v, dtype=tdtype)).sum()
            if with_gpsi:
                L = L + (icnn(zt)[:, 0] * torch.tensor(gpsi, dtype=tdtype)).sum()
            L.backward()
            g = icnn_grads(icnn)
            pre = f"{name}/{tag}/"
            out[pre + "psi"] = (psi[:, 0] - kappa * zt.pow(2).sum(1)).detach().numpy()
            out[pre + "xhat"] = xhat.detach().numpy()
            out[pre + "dz"] = zt.grad.numpy().copy()
            for k, a in g.items():
                if k == "W0" and H >= 512:   # keep fixtures small: strided sample + sums
                    out[pre + "g_W0_sample"] = a.reshape(-1)[::97].copy()
                    out[pre + "g_W0_sum"] = np.array([a.sum(dtype=np.float64), np.abs(a).sum(dtype=np.float64)])
                else:
                    out[pre + "g_" + k] = a
    golden.save(os.path.join(OUT, "icnn_cases.npz"), out)
    print("icnn_cases.npz:", len(out), "arrays")


def sd_to_np(sd):
    return {k: v.detach().cpu().numpy().copy() for k, v in sd.items()}


def gen_lidvae(ref_model):
    """Model-level goldens: small LIDVAE (pinwheel shape) fwd / loss / every .grad, fp32 and fp64."""
    out = {}
    for name, kw in (
        ("pin_small", dict(dataset="pinwheel", icnn_channels=[64, 128], hidden_channels=[16, 8],
                           inverse_lipschitz=0.3, beta=0.7)),
        ("pin_logmse", dict(dataset="chessboard", icnn_channels=[32, 64], hidden_channels=[8, 8, 4],
                            inverse_lipschitz=0.0, beta=0.01, is_log_mse=True)),
    ):
        torch.manual_seed(7)
        m32 = ref_model.LIDVAE(**kw)
        # move away from the exp(W)~1 default so that outputs are O(1) and masks are mixed
        rng = np.random.default_rng(11)
        with torch.no_grad():
            for ic in (m32.decoder[0], m32.decoder[1]):
                H = ic.A0.weight.shape[0]
                ic.W[0].param.copy_(torch.tensor(rng.normal(np.log(1.0 / H), 1.0, ic.W[0].param.shape), dtype=torch.float32))
                ic.W[1].param.copy_(torch.tensor(rng.normal(np.log(2.0 / H), 1.0, ic.W[1].param.shape), dtype=torch.float32))
                ic.A[0].bias.copy_(torch.tensor(rng.normal(-0.3, 1.0, ic.A[0].bias.shape), dtype=torch.float32))
        sd = sd_to_np(m32.state_dict())
        x = rng.normal(0, 1.5, (48, 2)).astype(np.float32)
        eps = rng.normal(0, 1.0, (48, 2)).astype(np.float32)
        for k, a in sd.items():
            out[f"{name}/sd/{k}"] = a
        out[f"{name}/x"], out[f"{name}/eps"] = x, eps
        for tag, tdtype in (("f32", torch.float32), ("f64", torch.float64)):
            m = ref_model.LIDVAE(**kw).to(tdtype)
            m.load_state_dict({k: torch.tensor(a).to(tdtype) if a.dtype.kind == "f" else torch.tensor(a) for k, a in sd.items()})
            m.train()
            xt = torch.tensor(x, dtype=tdtype)
            # forward_vae (model.py:840-846) with eps injected instead of randn_like
            mu, lv = m.encode(xt)
            z = mu + torch.tensor(eps, dtype=tdtype) * torch.exp(lv * 0.5)
            recon = m.decode(z)
            total, lrec, lreg, _ = m.loss(xt, recon, mu, lv, z, None)
            total.backward()
            pre = f"{name}/{tag}/"
            out[pre + "mu"], out[pre + "lv"], out[pre + "z"] = (t.detach().numpy() for t in (mu, lv, z))
            out[pre + "recon"] = recon.detach().numpy()
            out[pre + "loss"] = np.array([float(total), float(lrec), float(lreg)])
            for k, q in m.named_parameters():
                out[pre + "grad/" + k] = q.grad.numpy().copy()
    golden.save(os.path.join(OUT, "lidvae_cases.npz"), out)
    print("lidvae_cases.npz:", len(out), "arrays")


def gen_mnist_shaped(ref_model):
    """MNIST-shaped ICNN decoder through the D1 work-around (SURVEY.md section 8(c)); reduced widths."""
    out = {}
    torch.manual_seed(3)
    m = ref_model.LIDVAE(dataset="pinwheel")
    del m.B
    m.latent_channel = 8
    m.il_factor = 0.1
    m.encoder = m.make_encoder_2d([4, 8], 1, 8, 7)
    m.decoder = m.make_decoder_2d(1, 8, [48, 64], 28)
    rng = np.random.default_rng(12)
    with torch.no_grad():
        for ic in (m.decoder[0], m.decoder[1]):
            H = ic.A0.weight.shape[0]
            ic.W[0].param.copy_(torch.tensor(rng.normal(np.log(1.0 / H), 1.0, ic.W[0].param.shape), dtype=torch.float32))
            ic.W[1].param.copy_(torch.tensor(rng.normal(np.log(2.0 / H), 1.0, ic.W[1].param.shape), dtype=torch.float32))
            ic.A[0].bias.copy_(torch.tensor(rng.normal(-0.3, 1.0, ic.A[0].bias.shape), dtype=torch.float32))
    m = m.double()
    z = rng.normal(0, 1.0, (6, 8))
    vy = rng.normal(0, 1.0, (6, 1, 28, 28))
    zt = torch.tensor(z, requires_grad=True)
    y = m.decode(zt)
    (y * torch.tensor(vy)).sum().backward()
    for i in (0, 1):
        ic = m.decoder[i]
        for k, a in dict(A0w=ic.A0.weight, A0b=ic.A0.bias, A1w=ic.A[0].weight, A1b=ic.A[0].bias, A2w=ic.A[1].weight,
                         A2b=ic.A[1].bias, W0=ic.W[0].param, W1=ic.W[1].param).items():
            out[f"p{i}/{k}"] = a.detach().numpy().copy()
            out[f"g{i}/{k}"] = a.grad.numpy().copy()
    out["z"], out["vy"], out["y"], out["dz"] = z, vy, y.detach().numpy(), zt.grad.numpy().copy()
    out["kappa"] = np.array(0.1)
    golden.save(os.path.join(OUT, "mnist_shaped.npz"), out)
    print("mnist_shaped.npz:", len(out), "arrays")


def gen_losses(ref_model, ref_utils):
    out = {}
    rng = np.random.default_rng(21)
    # LRVAE.loss model.py:587-616 on [L,B,D] stacks (1-D data), VanillaVAE.loss :540-553
    for name, L, B, D, Dx in (("l1", 1, 37, 2, 2), ("l4", 4, 19, 2, 2), ("l4_wide", 4, 16, 28, 50)):
        x = rng.normal(0, 1, (B, Dx)); xh = rng.normal(0, 1, (B, Dx))
        mu = rng.normal(0, 1, (B, D)); lv = rng.normal(-1, 1, (B, D))
        zin = rng.normal(0, 1, (L, B, D)); zrec = rng.normal(0, 1, (L, B, D))
        m = ref_model.LRVAE(alpha=0.3, beta=0.05, dataset="pinwheel", hidden_channels=[4])
        m.wu_alpha = 0.6
        T = lambda a, rg=False: torch.tensor(a, dtype=torch.float64, requires_grad=rg)
        xht, mut, lvt, zrt = T(xh, True), T(mu, True), T(lv, True), T(zrec, True)
        total, lrec, lreg, llr = m.loss(T(x), xht, mut, lvt, T(zin), zrt)
        total.backward()
        pre = f"lrvae_{name}/"
        for k, a in dict(x=x, xh=xh, mu=mu, lv=lv, zin=zin, zrec=zrec).items():
            out[pre + k] = a
        out[pre + "out"] = np.array([float(total), float(lrec), float(lreg), float(llr)])
        out[pre + "hyper"] = np.array([0.3, 0.05, 0.6])  # alpha, beta, wu_alpha
        out[pre + "g_xh"], out[pre + "g_mu"], out[pre + "g_lv"], out[pre + "g_zrec"] = (
            t.grad.numpy().copy() for t in (xht, mut, lvt, zrt))
    # LIDVAE.loss log-MSE branch model.py:872-882 on image-shaped data
    x = rng.uniform(0, 1, (9, 1, 6, 6)); xh = rng.uniform(0, 1, (9, 1, 6, 6))
    mu = rng.normal(0, 1, (9, 5)); lv = rng.uniform(0.1, 2, (9, 5))
    m = ref_model.LIDVAE(dataset="pinwheel", icnn_channels=[8, 8], is_log_mse=True, beta=0.4)
    T = lambda a, rg=False: torch.tensor(a, dtype=torch.float64, requires_grad=rg)
    xht, mut, lvt = T(xh, True), T(mu, True), T(lv, True)
    total, lrec, lreg, _ = m.loss(T(x), xht, mut, lvt)
    total.backward()
    for k, a in dict(x=x, xh=xh, mu=mu, lv=lv).items():
        out["lid_logmse/" + k] = a
    out["lid_logmse/out"] = np.array([float(total), float(lrec), float(lreg)])
    out["lid_logmse/g_xh"], out["lid_logmse/g_mu"], out["lid_logmse/g_lv"] = (t.grad.numpy().copy() for t in (xht, mut, lvt))
    # utils.kld utils.py:140-141
    out["kld/val"] = np.array(ref_utils.kld(T(mu), T(lv)))
    golden.save(os.path.join(OUT, "loss_cases.npz"), out)
    print("loss_cases.npz:", len(out), "arrays")


def gen_lipschitz(ref_model, ref_utils):
    """utils.estimate_local_lipschitz utils.py:532-567 driven exactly as lipschitz.py:184 does."""
    out = {}
    g = np.load(os.path.join(OUT, "lidvae_cases.npz"))
    kw = dict(dataset="pinwheel", icnn_channels=[64, 128], hidden_channels=[16, 8], inverse_lipschitz=0.3, beta=0.7)
    m = ref_model.LIDVAE(**kw).double()
    sd = {k[len("pin_small/sd/"):]: g[k] for k in g.files if k.startswith("pin_small/sd/")}
    m.load_state_dict({k: torch.tensor(a).double() if a.dtype.kind == "f" else torch.tensor(a) for k, a in sd.items()})
    m.eval()
    rng = np.random.default_rng(31)
    for name, N, P in (("n500_p2000", 500, 2000), ("n100_p100", 100, 100), ("n5_p64_dups", 5, 64)):
        Z = rng.normal(0, 1.0, (N, 2))
        if name.endswith("dups"):
            Z[3] = Z[1]      # coincident points -> both clamps -> ratio exactly 1.0 (SURVEY section 4)
        Zt = torch.tensor(Z)
        gen = torch.Generator(device="cpu").manual_seed(0)
        i1 = torch.randint(0, N, (P,), generator=gen)
        i2 = torch.randint(0, N, (P,), generator=gen)
        res = ref_utils.estimate_local_lipschitz(m.decode, Zt, num_pairs=P, use_grad=True)
        Y = m.decode(Zt.clone().requires_grad_(True)).detach().numpy()
        out[f"{name}/Z"], out[f"{name}/Y"] = Z, Y
        out[f"{name}/i1"], out[f"{name}/i2"] = i1.numpy(), i2.numpy()
        out[f"{name}/res"] = np.array(res)
    golden.save(os.path.join(OUT, "lipschitz_cases.npz"), out)
    print("lipschitz_cases.npz:", len(out), "arrays")


def _run_family(out, name, make, x, eps, patch_name, L=None):
    """Reference forward/loss/backward of a FlexibleVAE / Set model with the noise draw replaced by `eps`
    (unittest.mock on torch.randn / torch.randn_like for the duration of the call; the reference source is untouched)."""
    from unittest import mock
    torch.manual_seed(5)
    m32 = make()
    sd = sd_to_np(m32.state_dict())
    for k, a in sd.items():
        out[f"{name}/sd/{k}"] = a
    out[f"{name}/x"], out[f"{name}/eps"] = x, eps
    m = make().double()
    m.load_state_dict({k: torch.tensor(a).double() if a.dtype.kind == "f" else torch.tensor(a) for k, a in sd.items()})
    m.train()
    if hasattr(m, "wu_alpha"):
        m.wu_alpha = 0.6
    xt = torch.tensor(x, dtype=torch.float64)
    et = torch.tensor(eps, dtype=torch.float64)
    with mock.patch.object(torch, patch_name, side_effect=lambda *a, **k: et.clone()):
        res = m(xt, L=L) if L is not None else m(xt)
    recon, mu, lv, z_in, z_rec = res
    total, lrec, lreg, llr = m.loss(xt, recon, mu, lv, z_in, z_rec)
    total.backward()
    pre = f"{name}/f64/"
    out[pre + "recon"], out[pre + "mu"], out[pre + "lv"] = (t.detach().numpy() for t in (recon, mu, lv))
    out[pre + "z_in"] = z_in.detach().numpy()
    if z_rec is not None:
        out[pre + "z_rec"] = z_rec.detach().numpy()
    out[pre + "loss"] = np.array([float(total), float(lrec), float(lreg), float(llr)])
    for k, q in m.named_parameters():
        out[pre + "grad/" + k] = np.zeros(q.shape) if q.grad is None else q.grad.numpy().copy()


def gen_families(ref_model):
    """BASELINE configs[0] (pinwheel LR-VAE), configs[3] (conv LR-VAE / beta-VAE on MNIST-shaped data), configs[4]
    (set LR-VAE on point clouds) at reduced widths: forward tuple, loss 4-tuple, every parameter gradient."""
    out = {}
    rng = np.random.default_rng(41)
    _run_family(out, "c1_lrvae_pinwheel",
                lambda: ref_model.LRVAE(alpha=0.3, beta=0.01, dataset="pinwheel", hidden_channels=[16] * 3,
                                        encoder_type="mlp", decoder_type="mlp"),
                rng.normal(0, 1.5, (64, 2)).astype(np.float32), rng.normal(0, 1, (3, 64, 2)).astype(np.float32), "randn", L=3)
    _run_family(out, "c3_lrvae_conv",
                lambda: ref_model.LRVAE(alpha=0.1, beta=0.001, dataset="mnist", hidden_channels=[4, 8],
                                        encoder_type="conv", decoder_type="conv"),
                rng.uniform(0, 1, (6, 1, 28, 28)).astype(np.float32), rng.normal(0, 1, (2, 6, 28)).astype(np.float32), "randn", L=2)
    _run_family(out, "c3_vanilla_conv_logmse",
                lambda: ref_model.VanillaVAE(beta=0.5, dataset="mnist", hidden_channels=[4, 8], encoder_type="conv",
                                             decoder_type="conv", is_log_mse=True),
                rng.uniform(0, 1, (5, 1, 28, 28)).astype(np.float32), rng.normal(0, 1, (1, 5, 28)).astype(np.float32), "randn", L=1)
    kw = dict(latent_channel=8, num_points=48, d_model=16, num_heads=2, num_encoder_layers=1, num_decoder_layers=1, ff_dim=32)
    _run_family(out, "c4_setlrvae_attn", lambda: ref_model.SetLRVAE(alpha=0.1, beta=0.2, use_attention=True, **kw),
                rng.normal(0, 1, (4, 48, 3)).astype(np.float32), rng.normal(0, 1, (4, 8)).astype(np.float32), "randn_like")
    _run_family(out, "c4_setvae_deepsets",
                lambda: ref_model.SetVAE(beta=0.2, latent_channel=8, num_points=40, encoder_hidden=[16, 32],
                                         decoder_hidden=[32, 16], use_attention=False),
                rng.normal(0, 1, (5, 40, 3)).astype(np.float32), rng.normal(0, 1, (5, 8)).astype(np.float32), "randn_like")
    # chamfer_distance model.py:896-912 on ragged set sizes, values and gradients
    a = rng.normal(0, 1, (3, 70, 3)); b = rng.normal(0, 1, (3, 300, 3))
    at, bt = torch.tensor(a, requires_grad=True), torch.tensor(b, requires_grad=True)
    cd = ref_model.chamfer_distance(at, bt)
    cd.backward()
    out["chamfer/a"], out["chamfer/b"], out["chamfer/cd"] = a, b, np.array(float(cd))
    out["chamfer/ga"], out["chamfer/gb"] = at.grad.numpy().copy(), bt.grad.numpy().copy()
    golden.save(os.path.join(OUT, "family_cases.npz"), out)
    print("family_cases.npz:", len(out), "arrays")


def gen_train_trajectory(ref_model):
    """Training TRAJECTORY of the unmodified reference loop: lipschitz.train_model (lipschitz.py:23-44: Adam, forward,
    loss, backward, step) on a small LIDVAE for 2 epochs x 6 batches in fp32 on CPU.  The only intervention is the
    ENVIRONMENT: torch.randn_like is wrapped so that the eps draws of model.py:843 come from a recorded list (the CPU and
    CUDA generators produce different streams), and the loader is a plain list of batches.  Stored: per-step total /
    recon / KL losses (captured by wrapping model.loss), the initial state_dict, the final parameters and BatchNorm buffers."""
    import lipschitz as ref_lipschitz        # the reference's own training loop
    rng = np.random.default_rng(21)
    kw = dict(dataset="pinwheel", icnn_channels=[32, 64], hidden_channels=[16, 8], inverse_lipschitz=0.2, beta=0.3)
    torch.manual_seed(3)
    m = ref_model.LIDVAE(**kw)
    with torch.no_grad():
        for ic in (m.decoder[0], m.decoder[1]):
            H = ic.A0.weight.shape[0]
            ic.W[0].param.copy_(torch.tensor(rng.normal(np.log(1.0 / H), 1.0, ic.W[0].param.shape), dtype=torch.float32))
            ic.W[1].param.copy_(torch.tensor(rng.normal(np.log(2.0 / H), 1.0, ic.W[1].param.shape), dtype=torch.float32))
            ic.A[0].bias.copy_(torch.tensor(rng.normal(-0.3, 1.0, ic.A[0].bias.shape), dtype=torch.float32))
    out = {f"sd0/{k}": a for k, a in sd_to_np(m.state_dict()).items()}
    nb, B, epochs = 6, 64, 2
    X = rng.normal(0, 1.5, (nb, B, 2)).astype(np.float32)
    eps = rng.normal(0, 1.0, (epochs * nb, B, 2)).astype(np.float32)
    out["X"], out["eps"] = X, eps
    loader = [(torch.tensor(X[i]), torch.zeros(B, dtype=torch.int64)) for i in range(nb)]
    draws = iter(eps)
    real_randn_like = torch.randn_like
    torch.randn_like = lambda t, *a, **k: torch.tensor(next(draws), dtype=t.dtype)
    losses = []
    real_loss = m.loss

    def recording_loss(*a, **k):
        r = real_loss(*a, **k)
        losses.append([float(r[0]), float(r[1]), float(r[2])])
        return r
    m.loss = recording_loss
    try:
        ref_lipschitz.train_model(m, loader, epochs, 1e-3, "cpu")
    finally:
        torch.randn_like = real_randn_like
        del m.loss
    out["losses"] = np.array(losses, dtype=np.float64)
    for k, a in sd_to_np(m.state_dict()).items():
        out[f"sd1/{k}"] = a
    out["cfg"] = np.array([nb, B, epochs])
    golden.save(os.path.join(OUT, "train_trajectory.npz"), out)
    print("train_trajectory.npz:", len(out), "arrays; first / last loss", losses[0][0], losses[-1][0])


WARMUP_CASES = [   # (name, kwargs of VAE.warmup besides epoch/max_epoch)
    ("linear", dict(wu_strat="linear")),
    ("linear_up", dict(wu_strat="linear", up_amount=0.07, start_epoch=3)),
    ("exponential", dict(wu_strat="exponential", start_epoch=2)),
    ("exponential_up", dict(wu_strat="exponential", up_amount=0.05)),
    ("repeat_linear", dict(wu_strat="repeat_linear", repeat_interval=4, start_epoch=1)),
    ("kl_adaptive", dict(wu_strat="kl_adaptive")),
]


def gen_host_logic(ref_model, ref_utils):
    """Host-side schedules of the reference: VAE.warmup (model.py:37-63) per strategy over 24 epochs, and
    utils.apply_grad_clip (utils.py) on fixed gradients."""
    out = {}
    kl_seq = np.linspace(9.0, 1.0, 24)
    for name, kw in WARMUP_CASES:
        m = ref_model.LRVAE(beta=0.01, alpha=0.1, dataset="pinwheel", hidden_channels=[4], encoder_type="mlp", decoder_type="mlp")
        seq = []
        for epoch in range(24):
            m.last_kl_loss = float(kl_seq[epoch])
            m.warmup(epoch=epoch, max_epoch=20, **kw)
            seq.append(m.wu_alpha)
        out["warmup/" + name] = np.asarray(seq, np.float64)
    out["warmup/kl_seq"] = kl_seq
    rng = np.random.default_rng(11)
    g = [rng.normal(0, 1, (3, 4)).astype(np.float32), rng.normal(0, 2, (5,)).astype(np.float32)]
    for tag, cfg in (("norm", {"enabled": True, "clip_type": "norm", "max_norm": 0.7, "norm_type": 2.0}),
                     ("value", {"enabled": True, "clip_type": "value", "clip_value": 0.5}),
                     ("off", {"enabled": False, "clip_type": "norm", "max_norm": 0.1})):
        lin = torch.nn.Linear(4, 3)
        lin.weight.grad = torch.tensor(g[0]); lin.bias.grad = torch.tensor(g[1][:3])
        ref_utils.apply_grad_clip(lin, cfg)
        out[f"clip/{tag}/w"] = lin.weight.grad.numpy().copy(); out[f"clip/{tag}/b"] = lin.bias.grad.numpy().copy()
    out["clip/g_w"], out["clip/g_b"] = g[0], g[1][:3]
    golden.save(os.path.join(OUT, "host_cases.npz"), out)
    print("host_cases.npz:", len(out), "arrays")


BASELINE_ICNN_KW = dict(dataset="pinwheel", inverse_lipschitz=0.2, beta=1.0)      # icnn_channels = the reference default [512, 1024]


def baseline_icnn_weights(model_obj, seed=17):
    """The big H x H matrices (and the rows that make the LeakyReLU masks mixed) are drawn with numpy so that the test can
    rebuild them from the seed; works on the reference's LIDVAE and on vae_song_b200's (same attribute names)."""
    rng = np.random.default_rng(seed)
    with torch.no_grad():
        for ic in (model_obj.decoder[0], model_obj.decoder[1]):
            H = ic.A0.weight.shape[0]
            ic.W[0].param.copy_(torch.tensor(rng.normal(np.log(1.0 / H), 1.0, (H, H))).to(ic.W[0].param.dtype))
            ic.W[1].param.copy_(torch.tensor(rng.normal(np.log(2.0 / H), 1.0, (1, H))).to(ic.W[1].param.dtype))
            ic.A[0].bias.copy_(torch.tensor(rng.normal(-0.3, 1.0, (H,))).to(ic.A[0].bias.dtype))


def gen_lidvae_baseline(ref_model):
    """Model-level golden at the BASELINE widths: LIDVAE(pinwheel) with the reference's DEFAULT icnn_channels=[512,1024]
    (model.py:644) and default encoder, fp64, batch 96: forward tuple, loss parts, dz-side tensors, every small gradient in
    full and the two H x H gradients as strided samples + sums (the fixture stays ~100 KB).  The H x H weights are not
    stored: the test redraws them from the numpy seed."""
    out = {}
    torch.manual_seed(13)
    m = ref_model.LIDVAE(**BASELINE_ICNN_KW).double()
    baseline_icnn_weights(m)
    for k, a in sd_to_np(m.state_dict()).items():
        if not k.endswith("W.0.param"):
            out["sd/" + k] = a
    rng = np.random.default_rng(19)
    x = rng.normal(0, 1.5, (96, 2)).astype(np.float32)
    eps = rng.normal(0, 1.0, (96, 2)).astype(np.float32)
    out["x"], out["eps"] = x, eps
    m.train()
    xt = torch.tensor(x, dtype=torch.float64)
    mu, lv = m.encode(xt)
    z = mu + torch.tensor(eps, dtype=torch.float64) * torch.exp(lv * 0.5)
    recon = m.decode(z)
    total, lrec, lreg, _ = m.loss(xt, recon, mu, lv, z, None)
    total.backward()
    out["mu"], out["lv"], out["z"], out["recon"] = (t.detach().numpy() for t in (mu, lv, z, recon))
    out["loss"] = np.array([float(total), float(lrec), float(lreg)])
    for k, q in m.named_parameters():
        g = q.grad.numpy()
        if k.endswith("W.0.param"):
            out["grad_sample/" + k] = g.reshape(-1)[::97].copy()
            out["grad_sum/" + k] = np.array([g.sum(dtype=np.float64), np.abs(g).sum(dtype=np.float64), np.abs(g).max()])
        else:
            out["grad/" + k] = g.copy()
    golden.save(os.path.join(OUT, "lidvae_baseline_icnn.npz"), out)
    print("lidvae_baseline_icnn.npz:", len(out), "arrays")


def main():
    os.makedirs(OUT, exist_ok=True)
    ref_module, ref_model, ref_utils = import_reference()
    torch.set_num_threads(8)
    if len(sys.argv) > 1 and sys.argv[1] == "host":        # only the (cheap) host-logic fixtures
        return gen_host_logic(ref_model, ref_utils)
    if len(sys.argv) > 1 and sys.argv[1] == "baseline":    # only the BASELINE-width model golden
        return gen_lidvae_baseline(ref_model)
    gen_icnn(ref_module)
    gen_lidvae(ref_model)
    gen_lidvae_baseline(ref_model)
    gen_mnist_shaped(ref_model)
    gen_losses(ref_model, ref_utils)
    gen_lipschitz(ref_model, ref_utils)
    gen_families(ref_model)
    gen_train_trajectory(ref_model)
    gen_host_logic(ref_model, ref_utils)


if __name__ == "__main__":
    main()
