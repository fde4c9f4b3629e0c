"""Drop-in parity of the nn.Module surface on the GPU: load the reference's state_dict, compare
forward / loss / every .grad with what the reference produced (tests/golden/lidvae_cases.npz)."""
import os
import types

import numpy as np
import pytest
import torch

from oracle import loss_oracle as lo

from oracle import golden
from oracle import icnn_oracle as io

from conftest import GOLDEN
from helpers import H_RTOL, close_report, close_rows, kink_rows

pytestmark = pytest.mark.gpu


def bn_shadowed(name, model):
    """Bias of a Linear that feeds a BatchNorm directly (block index 0 -> BN at index 1): its gradient is
    mathematically zero, both implementations return pure rounding noise (and Adam turns that noise into
    +-lr steps that no output depends on), so these entries are excluded from elementwise comparisons."""
    if not name.endswith(".0.bias"):
        return False
    return name[:-len("0.bias")] + "1.running_mean" in model.state_dict()

CASES = {
    "pin_small": dict(dataset="pinwheel", icnn_channels=[64, 128], hidden_channels=[16, 8], inverse_lipschitz=0.3, beta=0.7),
    "pin_logmse": dict(dataset="chessboard", icnn_channels=[32, 64], hidden_channels=[8, 8, 4], inverse_lipschitz=0.0,
                       beta=0.01, is_log_mse=True),
}


def _load(name):
    from vae_song_b200 import model
    G = np.load(os.path.join(GOLDEN, "lidvae_cases.npz"))
    m = model.LIDVAE(**CASES[name])
    sd = {k[len(name) + 4:]: torch.tensor(G[k]) for k in G.files if k.startswith(name + "/sd/")}
    missing, unexpected = m.load_state_dict(sd, strict=True)
    assert not missing and not unexpected
    return m.cuda().train(), G


def _icnn_p64(ic):
    f = lambda t: t.detach().double().cpu().numpy()
    return dict(A0w=f(ic.A0.weight), A0b=f(ic.A0.bias), A1w=f(ic.A[0].weight), A1b=f(ic.A[0].bias), A2w=f(ic.A[1].weight),
                A2b=f(ic.A[1].bias), W0=f(ic.W[0].param), W1=f(ic.W[1].param))


def _decoder_kink_rows(m, z, h_rtol):
    """Rows of a LIDVAE decode in which EITHER ICNN has a LeakyReLU pre-activation within h_rtol * max|h| of its kink
    (oracle evaluation in fp64 of the model's own weights): the only rows allowed the loose bound (helpers.kink_rows)."""
    z64 = z.detach().double().cpu().numpy()
    _, x1, a0 = io.icnn_brenier(z64, _icnn_p64(m.decoder[0]), 0, m.il_factor)
    _, _, a1 = io.icnn_brenier(io.pad_eye(x1, m.decoder[1].in_channel), _icnn_p64(m.decoder[1]), 0, m.il_factor)
    return kink_rows(a0, h_rtol) | kink_rows(a1, h_rtol)


@pytest.mark.parametrize("precision,rtol_y,rtol_g", [("fp32", 2e-5, 2e-4), ("tf32x3", 2e-5, 2e-4), ("f16x3", 2e-5, 2e-4),
                                                     ("tf32", 1e-2, 1e-2)])
def test_lidvae_baseline_widths_vs_reference_golden(precision, rtol_y, rtol_g):
    """The BASELINE model itself -- LIDVAE(pinwheel) with the reference's default icnn_channels=[512,1024] (model.py:644)
    and default encoder -- against what the unmodified reference produced in fp64 (oracle/make_golden.py
    gen_lidvae_baseline): forward tuple, loss parts and every parameter gradient, on the FP32 kernels, on the fp32-grade
    tensor-core path at the same bounds, and on 1xTF32 at its stated looser bound."""
    from oracle.make_golden import BASELINE_ICNN_KW, baseline_icnn_weights
    from vae_song_b200 import model
    G = np.load(os.path.join(GOLDEN, "lidvae_baseline_icnn.npz"))
    m = model.LIDVAE(precision=precision, **BASELINE_ICNN_KW)
    sd = {k[3:]: torch.tensor(G[k]).float() if G[k].dtype.kind == "f" else torch.tensor(G[k]) for k in G.files if k.startswith("sd/")}
    missing, unexpected = m.load_state_dict(sd, strict=False)
    assert not unexpected and sorted(missing) == ["decoder.0.W.0.param", "decoder.1.W.0.param"]
    baseline_icnn_weights(m)                                  # the H x H matrices are redrawn from the numpy seed
    m = m.cuda().train()
    x, eps = torch.tensor(G["x"], device="cuda"), torch.tensor(G["eps"], device="cuda")
    recon, mu, lv, z, _ = m(x, eps=eps)
    total, lrec, lreg, _ = m.loss(x, recon, mu, lv, z, None)
    total.backward()
    close_report(mu.detach().cpu().numpy(), G["mu"], 2e-5, "mu")
    close_report(z.detach().cpu().numpy(), G["z"], 2e-5, "z")
    prec_id = {"fp32": 0, "tf32x3": 3, "f16x3": 4, "tf32": 1}[precision]
    kr = _decoder_kink_rows(m, z, 2 * H_RTOL[prec_id])
    close_rows(recon.detach().cpu().numpy(), G["recon"], rtol_y, "recon", kr, loose=5e-2)
    np.testing.assert_allclose([float(total), float(lrec), float(lreg)], G["loss"], rtol=10 * rtol_y)
    gscale = max(np.abs(G[k]).max() for k in G.files if k.startswith("grad/"))
    for k, q in m.named_parameters():
        if bn_shadowed(k, m):
            assert float(q.grad.abs().max()) <= 1e-4 * gscale, k
        elif k.endswith("W.0.param"):
            g = q.grad.cpu().numpy()
            close_report(g.reshape(-1)[::97], G["grad_sample/" + k], rtol_g, "grad sample " + k, floor=G["grad_sum/" + k][2])
            np.testing.assert_allclose([g.sum(dtype=np.float64), np.abs(g).sum(dtype=np.float64)], G["grad_sum/" + k][:2],
                                       rtol=10 * rtol_g)
        elif np.abs(G["grad/" + k]).max() == 0:
            assert float(q.grad.abs().max()) == 0.0, k
        else:
            close_report(q.grad.cpu().numpy(), G["grad/" + k], 10 * rtol_g if k.startswith("encoder") else rtol_g, "grad " + k,
                         floor=1e-4 * gscale)


@pytest.mark.parametrize("name", list(CASES))
def test_lidvae_forward_loss_grads(name):
    m, G = _load(name)
    x = torch.tensor(G[f"{name}/x"], device="cuda")
    eps = torch.tensor(G[f"{name}/eps"], device="cuda")
    recon, mu, lv, z, none = m(x, eps=eps)
    assert none is None
    total, lrec, lreg, zero = m.loss(x, recon, mu, lv, z, None)
    assert zero == 0.0 and not lrec.requires_grad and not lreg.requires_grad
    total.backward()
    for tag, rt in (("f64", 1.0), ("f32", 2.0)):
        pre = f"{name}/{tag}/"
        close_report(mu.detach().cpu().numpy(), G[pre + "mu"], 2e-5 * rt, "mu")
        close_report(z.detach().cpu().numpy(), G[pre + "z"], 2e-5 * rt, "z")
        close_rows(recon.detach().cpu().numpy(), G[pre + "recon"], 1e-4 * rt, "recon", _decoder_kink_rows(m, z, H_RTOL[0] * rt))
        np.testing.assert_allclose([float(total), float(lrec), float(lreg)], G[pre + "loss"], rtol=1e-4 * rt)
        worst = 0.0
        # Linear biases feeding a BatchNorm have mathematically zero gradients (pure rounding noise in both
        # implementations): compare those against the model-wide gradient scale instead of their own.
        gscale = max(np.abs(G[pre + "grad/" + k]).max() for k, _ in m.named_parameters())
        for k, q in m.named_parameters():
            ref = G[pre + "grad/" + k]
            if bn_shadowed(k, m):
                assert float(q.grad.abs().max()) <= 1e-4 * gscale, k
                continue
            if np.abs(ref).max() == 0:
                assert q.grad is None or float(q.grad.abs().max()) == 0.0, k
            else:
                worst = max(worst, close_report(q.grad.cpu().numpy(), ref, 1e-3 * rt, "grad " + k, floor=1e-4 * gscale))
        assert worst < 2e-3


def test_decode_without_autograd_graph():
    """Reference defect D4: decode() fails under no_grad; ours must work and agree."""
    m, G = _load("pin_small")
    z = torch.randn(64, 2, device="cuda")
    with torch.no_grad():
        y0 = m.decode(z)
    y1 = m.decode(z.clone().requires_grad_(True))
    assert torch.equal(y0, y1.detach())


def test_forward_accepts_L_and_latent_recon():
    m, _ = _load("pin_small")
    x = torch.randn(32, 2, device="cuda")
    out = m(x, L=4)                        # reference defect D2: main.py passes L
    assert len(out) == 5 and out[4] is None
    out = m(x, latent_recon=True)
    assert out[4].shape == (32, 2)


def test_train_loop_matches_torch_composition():
    """Three optimiser steps of lipschitz.train_model semantics: fused kernels vs the same model whose
    decode/loss are recomposed from plain torch ops + autograd (the reference formulation) on the GPU."""
    from vae_song_b200 import model
    import copy
    torch.manual_seed(0)
    m, _ = _load("pin_small")
    ref = copy.deepcopy(m)

    def ref_icnn(ic, z):
        act = torch.nn.functional.leaky_relu
        x = act(ic.A0(z), 0.2).pow(2)
        for w, a in zip(ic.W, ic.A):
            x = act(torch.nn.functional.linear(x, w.param.exp()) + a(z), 0.2)
        return x

    def ref_decode(mm, z):
        x = ref_icnn(mm.decoder[0], z) + mm.il_factor * z.pow(2).sum(1, keepdim=True)
        x = torch.autograd.grad(x, [z], torch.ones_like(x), create_graph=True)[0]
        y = ref_icnn(mm.decoder[1], x) + mm.il_factor * x.pow(2).sum(1, keepdim=True)
        return torch.autograd.grad(y, [x], torch.ones_like(y), create_graph=True)[0]

    o1 = torch.optim.Adam(m.parameters(), lr=1e-3)
    o2 = torch.optim.Adam(ref.parameters(), lr=1e-3)
    g = torch.Generator(device="cuda").manual_seed(1)
    for step in range(3):
        x = torch.randn(256, 2, device="cuda", generator=g)
        eps = torch.randn(256, 2, device="cuda", generator=g)
        o1.zero_grad(); o2.zero_grad()
        recon, mu, lv, z, _ = m(x, eps=eps)
        l1 = m.loss(x, recon, mu, lv, z, None)[0]
        l1.backward(); o1.step()
        mu2, lv2 = ref.encode(x)
        z2 = mu2 + eps * torch.exp(lv2 * 0.5)
        r2 = ref_decode(ref, z2)
        l2 = ((x - r2) ** 2).mean(0).sum() + ref.beta * (-0.5 * (1 + lv2 - mu2 ** 2 - lv2.exp())).mean(0).sum()
        l2.backward(); o2.step()
        assert abs(float(l1) - float(l2)) <= 2e-4 * abs(float(l2)), (step, float(l1), float(l2))
    for (k, a), (_, b) in zip(m.named_parameters(), ref.named_parameters()):
        if not bn_shadowed(k, m):
            close_report(a.detach().cpu().numpy(), b.detach().cpu().numpy(), 1e-3, "param " + k)


def test_flexible_family_losses_and_staged_backward():
    """LRVAE (config C1 shape): forward tuple shapes, attached loss parts, main.py's staged backward."""
    from vae_song_b200 import model
    torch.manual_seed(0)
    m = model.LRVAE(alpha=1e-2, beta=0.01, dataset="pinwheel", hidden_channels=[16] * 3).cuda().train()
    m.wu_alpha = 0.5
    x = torch.randn(64, 2, device="cuda")
    eps = torch.randn(4, 64, 2, device="cuda")
    recon, mu, lv, z_in, z_rec = m(x, L=4, eps=eps)
    assert z_in.shape == (4, 64, 2) and z_rec.shape == (4, 64, 2) and not z_in.requires_grad
    total, lrec, lreg, llr = m.loss(x, recon, mu, lv, z_in, z_rec)
    f = lambda t: t.detach().double().cpu().numpy()
    rec_o, reg_o, lr_o = lo.recon_mse(f(x), f(recon)), lo.kl(f(mu), f(lv)), lo.latent_recon(f(z_in), f(z_rec))
    np.testing.assert_allclose([float(lrec), float(lreg), float(llr)], [rec_o, 0.01 * reg_o, 1e-2 * 0.5 * lr_o], rtol=2e-5)
    # staged backward exactly as main.py:262-284
    m.zero_grad()
    llr.backward(retain_graph=True)
    for q in m.encoder.parameters():
        if q.grad is not None:
            q.grad *= 1e-4
    lreg.backward(retain_graph=True)
    lrec.backward()
    staged = [q.grad.clone() for q in m.parameters()]
    names = [k for k, _ in m.named_parameters()]
    gscale = max(float(g.abs().max()) for g in staged)
    # same thing composed from plain torch ops on the same graph inputs
    m.zero_grad()
    recon, mu, lv, z_in, z_rec = m(x, L=4, eps=eps)
    l_lr = ((z_in - z_rec) ** 2).mean(0).sum() * 1e-2 * 0.5
    l_reg = (-0.5 * (1 + lv - mu ** 2 - lv.exp())).mean(0).sum() * 0.01
    l_rec = ((x - recon) ** 2).mean(0).sum()
    l_lr.backward(retain_graph=True)
    for q in m.encoder.parameters():
        if q.grad is not None:
            q.grad *= 1e-4
    l_reg.backward(retain_graph=True)
    l_rec.backward()
    for k, a, q in zip(names, staged, m.parameters()):
        if bn_shadowed(k, m):
            assert float(a.abs().max()) <= 1e-4 * gscale
        else:
            close_report(a.cpu().numpy(), q.grad.cpu().numpy(), 1e-4, "staged grad " + k, floor=1e-6 * gscale)


def test_graphed_step_equals_eager_step():
    """DataParallelTrainer.capture(): replaying the whole-step CUDA graph == launching the step eagerly
    (same eps), and capturing does not advance the optimiser."""
    from vae_song_b200 import train
    import copy
    m, _ = _load("pin_small")
    m2 = copy.deepcopy(m)
    a = train.DataParallelTrainer(m, lr=1e-3)
    b = train.DataParallelTrainer(m2, lr=1e-3)
    g = torch.Generator(device="cuda").manual_seed(3)
    xs = [torch.randn(256, 2, device="cuda", generator=g) for _ in range(4)]
    es = [torch.randn(256, 2, device="cuda", generator=g) for _ in range(4)]
    a.capture(xs[0], es[0])
    assert torch.equal(a.fp.flat, b.fp.flat) and int(a.t_dev) == 0
    for x, e in zip(xs, es):
        la = a.step_graphed(x, e)[0].clone()
        lb = b.step(x, e)[0]
        assert abs(float(la) - float(lb)) <= 1e-5 * abs(float(lb))
    close_report(a.fp.flat.cpu().numpy(), b.fp.flat.cpu().numpy(), 1e-5, "params after 4 steps", floor=1e-3)
    assert int(a.t_dev) == 4 == int(b.t_dev)


def test_wide_input_icnn_mnist_shaped():
    """MNIST-shaped ICNN decoder (reference defect D1 recipe, SURVEY 8(c)): ICNN(8,48) -> eye(784,8) pad ->
    ICNN(784,64); forward and every gradient against the reference-generated golden (fp64) and the oracle."""
    from vae_song_b200 import module
    G = golden.load(os.path.join(GOLDEN, "mnist_shaped.npz"))
    keys = ("A0w", "A0b", "A1w", "A1b", "A2w", "A2b", "W0", "W1")
    ics = []
    for i, (d, H) in enumerate(((8, 48), (784, 64))):
        ic = module.ICNN(d, H).cuda()
        with torch.no_grad():
            for t, k in zip(ic._flat_params(), keys):
                t.copy_(torch.tensor(G[f"p{i}/{k}"], dtype=torch.float32))
        ics.append(ic)
    kappa = float(G["kappa"])
    z = torch.tensor(G["z"], dtype=torch.float32, device="cuda", requires_grad=True)
    _, x1 = ics[0].brenier(z, kappa)
    x = torch.nn.functional.pad(x1, (0, 784 - 8))
    _, y = ics[1].brenier(x, kappa)
    (y * torch.tensor(G["vy"].reshape(6, -1), dtype=torch.float32, device="cuda")).sum().backward()
    none = np.zeros(6, dtype=bool)                     # 6 rows, trained-like weights: no unit sits within rounding of a kink
    close_rows(y.detach().cpu().numpy(), G["y"].reshape(6, -1), 2e-5, "y", none)
    close_rows(z.grad.cpu().numpy(), G["dz"], 1e-4, "dz", none)
    for i, ic in enumerate(ics):
        for t, k in zip(ic._flat_params(), keys):
            ref = G[f"g{i}/{k}"]
            if np.abs(ref).max() == 0:
                assert float(t.grad.abs().max()) == 0.0
            else:
                close_report(t.grad.cpu().numpy(), ref, 1e-4, f"grad{i} {k}")
    # psi via forward() stays twice differentiable for wide inputs (reference idiom)
    zz = torch.tensor(G["z"], dtype=torch.float32, device="cuda", requires_grad=True)
    psi = ics[0](zz) + kappa * zz.pow(2).sum(1, keepdim=True)
    xh = torch.autograd.grad(psi, [zz], torch.ones_like(psi), create_graph=True)[0]
    close_rows(xh.detach().cpu().numpy(), x1.detach().cpu().numpy(), 1e-5, "autograd Brenier == fused", none)


def test_lidvae_mnist_constructs_and_trains_one_step():
    """LIDVAE(dataset='mnist') (UnboundLocalError in the reference): decode + loss + backward run end to end."""
    from vae_song_b200 import model
    torch.manual_seed(0)
    m = model.LIDVAE(dataset="mnist", icnn_channels=[64, 128], hidden_channels=[4, 8], inverse_lipschitz=0.2).cuda().train()
    x = torch.rand(16, 1, 28, 28, device="cuda")
    recon, mu, lv, z, _ = m(x, L=4)
    assert recon.shape == x.shape and mu.shape == (16, 32)
    total, lrec, lreg, _ = m.loss(x, recon, mu, lv, z, None)
    total.backward()
    assert all(p.grad is not None and torch.isfinite(p.grad).all() for p in m.parameters())


def test_inference_workspace_cache_follows_the_weights():
    """decode under no_grad keeps the prepared ICNN workspace (exp(W) in every kernel layout) while the weights are unchanged;
    every way this package changes weights must invalidate it: torch optimisers / copy_ (version counters), the fused Adam
    kernel (raw pointers) and a CUDA-graph replay of the whole step (no Python runs)."""
    from vae_song_b200 import _C, model, train
    torch.manual_seed(0)
    m = model.LIDVAE(dataset="pinwheel", icnn_channels=[32, 64], hidden_channels=[8, 4], inverse_lipschitz=0.2,
                     precision="tf32x3").cuda()
    z = torch.randn(64, 2, device="cuda")
    x = torch.randn(256, 2, device="cuda")

    def both():
        with torch.no_grad():
            a = m.decode(z)
        b = m.decode(z.clone().requires_grad_(True)).detach()      # autograd path: prepares afresh every call
        return a, b
    a, b = both()
    assert torch.equal(a, b)
    n0 = _C.launch_count()
    with torch.no_grad():
        m.decode(z)
    assert _C.launch_count() - n0 == 2                              # two decode kernels, no prepare launches
    with torch.no_grad():
        m.decoder[1].A0.weight.mul_(1.5)                            # in-place edit: version counter
    a2, b2 = both()
    assert torch.equal(a2, b2) and not torch.equal(a2, a)
    tr = train.DataParallelTrainer(m, lr=1e-2)
    tr.step(x)                                                      # fused Adam through raw pointers
    a3, b3 = both()
    assert torch.equal(a3, b3) and not torch.equal(a3, a2)
    tr.capture(x)
    tr.step_graphed(x)                                              # graph replay
    a4, b4 = both()
    assert torch.equal(a4, b4) and not torch.equal(a4, a3)


@pytest.mark.parametrize("precision", ["fp32", "f16x3"])
def test_unmodified_reference_driver_runs_on_this_package(precision):
    """Drop-in proof with the reference's OWN driver file (on the FP32 parity kernels and on the 3xFP16 tensor-core kernels): oracle/_ref/lipschitz.py (byte-identical copy of the reference,
    oracle/fetch_ref.py) is imported with `module`, `model`, `utils` bound to vae_song_b200's modules instead of the
    reference's -- exactly what a user does by replacing three imports (INTEGRATION.md A).  Its train_model
    (lipschitz.py:23-44) then trains OUR LIDVAE on the GPU kernels and must follow the reference's recorded trajectory
    (golden: the reference's model under the same loop), and its per-cell evaluation (lipschitz.py:48-105) must return what
    this package's batched driver returns."""
    from oracle import fetch_ref
    if not fetch_ref.available():
        pytest.skip("oracle/_ref not populated (no reference checkout for oracle/fetch_ref.py)")
    from vae_song_b200 import lipschitz as our_lip, model, module, utils
    ns = fetch_ref.import_ref(swap={"module": module, "model": model, "utils": utils})
    assert fetch_ref.verify()                                           # the driver file is the unmodified reference
    assert ns.lipschitz.LIDVAE is model.LIDVAE and ns.lipschitz.estimate_local_lipschitz is utils.estimate_local_lipschitz
    G = np.load(os.path.join(GOLDEN, "train_trajectory.npz"))
    nb, B, epochs = (int(v) for v in G["cfg"])
    m = model.LIDVAE(dataset="pinwheel", icnn_channels=[32, 64], hidden_channels=[16, 8], inverse_lipschitz=0.2, beta=0.3,
                     precision=precision)
    m.load_state_dict({k[4:]: torch.tensor(G[k]) for k in G.files if k.startswith("sd0/")})
    loader = [(torch.tensor(G["X"][i]), torch.zeros(B, dtype=torch.int64)) for i in range(nb)]
    draws = iter(G["eps"])
    real_randn_like, losses, real_loss = torch.randn_like, [], m.loss

    def recording_loss(*a, **k):
        r = real_loss(*a, **k)
        losses.append([float(r[0].detach()), float(r[1]), float(r[2])])
        return r
    m.loss = recording_loss
    torch.randn_like = lambda t, *a, **k: torch.tensor(next(draws), dtype=t.dtype, device=t.device)
    import contextlib, io
    try:
        with contextlib.redirect_stderr(io.StringIO()):                 # the reference's tqdm bar
            ns.lipschitz.train_model(m, loader, epochs, 1e-3, "cuda")
    finally:
        torch.randn_like = real_randn_like
        del m.loss
    np.testing.assert_allclose(np.array(losses), G["losses"], rtol=2e-4, err_msg="per-step (total, recon, KL) losses")
    # the reference's X-cell sweep (one estimator call per cell) == this package's batched sweep, same seeds
    rng = np.random.default_rng(3)
    ds = types.SimpleNamespace(X=torch.tensor(rng.uniform(-2, 2, (600, 2)), dtype=torch.float32), y=None)
    K = 3
    cell = np.clip(((ds.X.numpy() + 2) / 4 * K).astype(int), 0, K - 1)
    ds.y = torch.tensor(cell[:, 1] * K + cell[:, 0])
    m.eval()
    torch.manual_seed(11)
    want = ns.lipschitz._get_kl_and_lipschitz_for_x_cells(m, ds, K, "cuda", nsamples_z=4, num_pairs_lips=200)
    torch.manual_seed(11)
    got = our_lip._get_kl_and_lipschitz_for_x_cells(m, ds, K, "cuda", nsamples_z=4, num_pairs_lips=200)
    for a, b, name in zip(got, want, ("kl", "lips", "inv_lips", "bi_lips")):
        np.testing.assert_allclose(a, b, rtol=1e-4, err_msg=name)


@pytest.mark.parametrize("hidden", [[2, 2, 2, 2], [128, 64, 64, 32, 16, 8, 4, 2], [16]])
@pytest.mark.parametrize("training", [True, False])
def test_fused_encoder_matches_stock_modules(hidden, training):
    """Fused Linear+BN+LeakyReLU layers (csrc/mlp.cu) vs the very same nn.Modules run by PyTorch: outputs, every
    gradient, and the BatchNorm running statistics."""
    from vae_song_b200 import model
    import copy
    torch.manual_seed(0)
    m = model.LIDVAE(dataset="pinwheel", icnn_channels=[32, 32], hidden_channels=hidden).cuda()
    with torch.no_grad():
        for mod in m.encoder.modules():
            if isinstance(mod, torch.nn.BatchNorm1d):
                mod.weight.uniform_(0.5, 1.5); mod.bias.uniform_(-0.5, 0.5)
                mod.running_mean.uniform_(-0.2, 0.2); mod.running_var.uniform_(0.5, 1.5)
    ref = copy.deepcopy(m)
    ref.fused_encoder = False
    m.train(training); ref.train(training)
    assert m._encoder_plan() is not None
    x = torch.randn(777, 2, device="cuda", requires_grad=True)
    x2 = x.detach().clone().requires_grad_(True)
    g = torch.randn(777, 4, device="cuda")
    mu, lv = m.encode(x)
    (torch.cat([mu, lv], 1) * g).sum().backward()
    mu2, lv2 = ref.encode(x2)
    (torch.cat([mu2, lv2], 1) * g).sum().backward()
    close_report(mu.detach().cpu().numpy(), mu2.detach().cpu().numpy(), 2e-5, "mu")
    close_report(lv.detach().cpu().numpy(), lv2.detach().cpu().numpy(), 2e-5, "lv")
    gscale = max(float(q.grad.abs().max()) for q in ref.encoder.parameters())
    close_report(x.grad.cpu().numpy(), x2.grad.cpu().numpy(), 2e-4, "dx", floor=1e-4 * gscale)
    for (k, a), (_, b) in zip(m.encoder.named_parameters(), ref.encoder.named_parameters()):
        if bn_shadowed("encoder." + k, m):
            assert float(a.grad.abs().max()) <= 1e-4 * gscale
        else:
            close_report(a.grad.cpu().numpy(), b.grad.cpu().numpy(), 2e-4, "grad " + k, floor=1e-5 * gscale)
    for (k, a), (_, b) in zip(m.encoder.named_buffers(), ref.encoder.named_buffers()):
        close_report(a.float().cpu().numpy(), b.float().cpu().numpy(), 1e-5, "buffer " + k)


def test_train_model_follows_the_reference_trajectory():
    """a10 (lipschitz.py:23-44): 12 Adam steps of the UNMODIFIED reference's train_model on a small LIDVAE (fp32, CPU; golden
    from oracle/make_golden.py::gen_train_trajectory) against train.train_model on the GPU kernels -- same initial
    state_dict, same batches, same eps draws (torch.randn_like wrapped on both sides): per-step losses and the final
    parameters / BatchNorm buffers must agree."""
    from vae_song_b200 import model, train
    G = np.load(os.path.join(GOLDEN, "train_trajectory.npz"))
    nb, B, epochs = (int(v) for v in G["cfg"])
    m = model.LIDVAE(dataset="pinwheel", icnn_channels=[32, 64], hidden_channels=[16, 8], inverse_lipschitz=0.2, beta=0.3)
    sd0 = {k[4:]: torch.tensor(G[k]) for k in G.files if k.startswith("sd0/")}
    m.load_state_dict(sd0)
    loader = [(torch.tensor(G["X"][i]), torch.zeros(B, dtype=torch.int64)) for i in range(nb)]
    draws = iter(G["eps"])
    real_randn_like, losses, real_loss = torch.randn_like, [], m.loss

    def recording_loss(*a, **k):
        r = real_loss(*a, **k)
        losses.append([float(r[0].detach()), float(r[1]), float(r[2])])
        return r
    m.loss = recording_loss
    torch.randn_like = lambda t, *a, **k: torch.tensor(next(draws), dtype=t.dtype, device=t.device)
    try:
        train.train_model(m, loader, epochs, 1e-3, "cuda")
    finally:
        torch.randn_like = real_randn_like
        del m.loss
    np.testing.assert_allclose(np.array(losses), G["losses"], rtol=2e-4, err_msg="per-step (total, recon, KL) losses")
    assert G["losses"][-1, 0] < G["losses"][0, 0]
    sd1 = m.state_dict()
    import re
    for k in G.files:
        if not k.startswith("sd1/"):
            continue
        if re.fullmatch(r"sd1/encoder\.\d+\.(0\.bias|1\.running_mean)", k):
            # a Linear bias feeding BatchNorm: its gradient is mathematically 0.  The reference's autograd leaves ~1e-9
            # rounding noise there, which Adam normalises into +-lr steps in random directions; the fused encoder returns
            # exact zeros.  The parameter has no effect on any output (BatchNorm subtracts it; only that layer's
            # running_mean carries it along), so neither is compared.
            continue
        ours, ref = sd1[k[4:]].detach().cpu().numpy(), G[k]
        if ref.dtype.kind != "f":
            assert np.array_equal(ours, ref), k
        else:      # 12 Adam steps amplify fp32 rounding differences of tiny gradients (update = lr * g/|g|): absolute floor
            np.testing.assert_allclose(ours, ref, rtol=2e-3, atol=2e-4, err_msg=k)


@pytest.mark.parametrize("training", [True, False])
def test_flexible_vae_fused_mlp_stacks_match_stock_modules(training):
    """FlexibleVAE-family 1-D MLP stacks (BASELINE configs[0]: pinwheel LR-VAE, encoder ENDING in BatchNorm + LeakyReLU,
    decoder ending in a bare Linear) through the fused layer kernels vs the very same nn.Modules run by PyTorch: the
    whole forward (two decodes, two encodes, L = 2), the loss parts, every gradient and the BatchNorm buffers."""
    from vae_song_b200 import model
    import copy
    torch.manual_seed(0)
    m = model.LRVAE(alpha=0.3, beta=0.2, dataset="pinwheel", hidden_channels=[16, 16, 16], encoder_type="mlp", decoder_type="mlp").cuda()
    m.wu_alpha = 1.0
    with torch.no_grad():
        for mod in m.modules():
            if isinstance(mod, torch.nn.BatchNorm1d):
                mod.weight.uniform_(0.5, 1.5); mod.bias.uniform_(-0.5, 0.5)
                mod.running_mean.uniform_(-0.2, 0.2); mod.running_var.uniform_(0.5, 1.5)
    ref = copy.deepcopy(m)
    m.fused_mlp, ref.fused_mlp = True, False
    m.train(training); ref.train(training)
    pe, pd = m._stack_plan("encoder"), m._stack_plan("decoder")
    assert pe is not None and pe.identity_tail and pd is not None and not pd.identity_tail
    assert sum(p.numel() for p in m.parameters()) == sum(p.numel() for p in ref.parameters())     # the identity layer is not a parameter
    x = torch.randn(300, 2, device="cuda")
    eps = torch.randn(2, 300, m.latent_channel, device="cuda")
    outs = []
    for mm in (m, ref):
        res = mm(x, L=2, eps=eps)
        parts = mm.loss(x, *res)
        parts[0].backward()
        outs.append((res, parts))
    for a, b, name in zip(outs[0][0], outs[1][0], ("recon", "mu", "log_var", "z", "z_recon")):
        close_report(a.detach().cpu().numpy(), b.detach().cpu().numpy(), 5e-5, name)
    for a, b, name in zip(outs[0][1], outs[1][1], ("total", "recon", "reg", "lr")):
        assert abs(float(a) - float(b)) <= 1e-4 * max(1.0, abs(float(b))), name
    gscale = max(float(q.grad.abs().max()) for q in ref.parameters())
    for (k, a), (_, b) in zip(m.named_parameters(), ref.named_parameters()):
        if bn_shadowed(k, m):
            assert float(a.grad.abs().max()) <= 1e-4 * gscale, k
        else:
            close_report(a.grad.cpu().numpy(), b.grad.cpu().numpy(), 5e-4, "grad " + k, floor=1e-4 * gscale)
    for (k, a), (_, b) in zip(m.named_buffers(), ref.named_buffers()):
        close_report(a.float().cpu().numpy(), b.float().cpu().numpy(), 2e-5, "buffer " + k)


def test_early_prepare_on_side_streams_changes_nothing():
    """LIDVAE.forward starts preparing both ICNNs' operands on side streams before the encoder runs
    (ops.icnn_prepare_early); results and gradients are bit-identical to preparing at the point of use, eagerly and when
    the whole step is replayed as a CUDA graph, and no parked workspace is left behind."""
    import copy
    from vae_song_b200 import model, ops, train
    torch.manual_seed(3)
    m0 = model.LIDVAE(dataset="pinwheel", icnn_channels=[64, 128], hidden_channels=[8, 4], inverse_lipschitz=0.2,
                      precision="f16x3").cuda().train()
    x, eps = torch.randn(300, 2, device="cuda"), torch.randn(300, 2, device="cuda")
    outs = []
    for early in (True, False):
        m = copy.deepcopy(m0)
        m.early_prepare = early
        recon, mu, lv, z, _ = m(x, eps=eps)
        total, _, _, _ = m.loss(x, recon, mu, lv, z, None)
        total.backward()
        torch.cuda.synchronize()
        assert not ops._EARLY
        outs.append((recon.detach().clone(), float(total), [p.grad.clone() for p in m.parameters()]))
    assert torch.equal(outs[0][0], outs[1][0]) and outs[0][1] == outs[1][1]
    for a, b in zip(outs[0][2], outs[1][2]):
        assert torch.equal(a, b)
    # graph replay of the whole step with the forked prepare branches == the eager step without them (same eps)
    ma, mb = copy.deepcopy(m0), copy.deepcopy(m0)
    mb.early_prepare = False
    ta, tb = train.DataParallelTrainer(ma, lr=1e-3), train.DataParallelTrainer(mb, lr=1e-3)
    g = torch.Generator(device="cuda").manual_seed(3)
    xs = [torch.randn(300, 2, device="cuda", generator=g) for _ in range(4)]
    es = [torch.randn(300, 2, device="cuda", generator=g) for _ in range(4)]
    ta.capture(xs[0], es[0])
    for xb, eb in zip(xs, es):
        la = ta.step_graphed(xb, eb)[0].clone()
        lb = tb.step(xb, eb)[0]
        assert float(la) == float(lb)
    torch.cuda.synchronize()
    assert torch.equal(ta.fp.flat, tb.fp.flat) and not ops._EARLY


def test_step_graphed_prefetch_of_the_next_host_batch():
    """step_graphed(x, next_x=...) starts the next batch's host-to-device copy on a copy stream while this step runs; the
    following call recognises the tensor and takes the staged copy.  Same trajectory as feeding device tensors."""
    import copy
    from vae_song_b200 import train
    m, _ = _load("pin_small")
    m2 = copy.deepcopy(m)
    a, b = train.DataParallelTrainer(m, lr=1e-3), train.DataParallelTrainer(m2, lr=1e-3)
    g = torch.Generator(device="cuda").manual_seed(5)
    xs = [torch.randn(256, 2, device="cuda", generator=g) for _ in range(6)]
    es = [torch.randn(256, 2, device="cuda", generator=g) for _ in range(6)]
    hs = [x.cpu().pin_memory() for x in xs]
    a.capture(xs[0], es[0]); b.capture(xs[0], es[0])
    for i in range(6):
        nxt = hs[i + 1] if i + 1 < 6 and i != 2 else None          # one step without a prefetch in the middle
        la = a.step_graphed(hs[i], es[i], next_x=nxt)[0].clone()
        lb = b.step_graphed(xs[i], es[i])[0].clone()
        assert float(la) == float(lb), i
    torch.cuda.synchronize()
    assert torch.equal(a.fp.flat, b.fp.flat)


def test_deferred_parameter_gradients_change_nothing():
    """DataParallelTrainer.step launches the parameter half of every tensor-core ICNN backward (b200vae_icnn_decode_bwd_params)
    on a side stream beside the encoder's backward and joins before it gathers the gradients: bit-identical training,
    eagerly and as a replayed graph; a model that uses one ICNN twice in a step falls back to in-order execution."""
    import copy
    from vae_song_b200 import model, ops, train
    torch.manual_seed(4)
    m0 = model.LIDVAE(dataset="pinwheel", icnn_channels=[64, 128], hidden_channels=[8, 4], inverse_lipschitz=0.2,
                      precision="f16x3").cuda().train()
    g = torch.Generator(device="cuda").manual_seed(9)
    xs = [torch.randn(300, 2, device="cuda", generator=g) for _ in range(5)]
    es = [torch.randn(300, 2, device="cuda", generator=g) for _ in range(5)]
    ma, mb, mc = copy.deepcopy(m0), copy.deepcopy(m0), copy.deepcopy(m0)
    ta, tb, tc_ = (train.DataParallelTrainer(m, lr=1e-3) for m in (ma, mb, mc))
    tb.defer_param_grads = False
    assert ta.defer_param_grads
    tc_.capture(xs[0], es[0])
    for x, e in zip(xs, es):
        la, lb, lc = ta.step(x, e)[0], tb.step(x, e)[0], tc_.step_graphed(x, e)[0].clone()
        assert float(la) == float(lb) == float(lc)
    torch.cuda.synchronize()
    assert torch.equal(ta.fp.flat, tb.fp.flat) and torch.equal(ta.fp.flat, tc_.fp.flat)
    assert not ops._DEFER["keep"] and not ops._DEFER["seen"] and not ops._DEFER["on"]
    # the same ICNN twice inside one deferred backward: second call joins first, gradients add up correctly
    ic = m0.decoder[0]
    z1 = torch.randn(64, 2, device="cuda", requires_grad=True)
    z2 = torch.randn(64, 2, device="cuda", requires_grad=True)

    def twice():
        for p in ic.parameters():
            p.grad = None
        (ic.brenier(z1, 0.1)[1].sum() + 2.0 * ic.brenier(z2, 0.1)[1].sum()).backward()
        return [p.grad.clone() for p in ic.parameters()]
    want = twice()
    with ops.deferred_param_grads():
        got = twice()
    torch.cuda.synchronize()
    for a, b in zip(got, want):
        assert torch.equal(a, b)
