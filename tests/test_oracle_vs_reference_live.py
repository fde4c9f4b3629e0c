"""Randomised comparison of the CPU oracle with the UNMODIFIED reference, run live where a checkout of
claviclecrusher/vae-song is found (oracle/fetch_ref.find_reference); skipped elsewhere (the repository does not ship the
reference -- there the committed fixtures of tests/golden/, made from it by oracle/make_golden.py, are the pin).  Shapes, weight regimes,
reparam modes, kappa and the psi-gradient path are drawn per seed, beyond the 11 fixed golden cases."""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import fetch_ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = fetch_ref.REF_SRC
pytestmark = pytest.mark.skipif(not (REF and os.path.isfile(os.path.join(REF, "module.py"))),
                                reason="no checkout of the reference (VAE_SONG_REFERENCE, ../reference, ../vae-song)")


@pytest.fixture(scope="module")
def ref():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import make_golden as mg
    return mg, mg.import_reference()


@pytest.mark.parametrize("seed", range(12))
def test_icnn_oracle_matches_live_reference(seed, ref):
    from oracle import icnn_oracle as io
    mg, (ref_module, _, _) = ref
    rng = np.random.default_rng(1000 + seed)
    d = int(rng.choice([1, 2, 3, 5, 17]))
    H = int(rng.choice([8, 24, 33, 64, 130]))
    B = int(rng.integers(1, 40))
    regime = str(rng.choice(["default", "mixed", "clampy"]))
    mode = int(rng.integers(0, 2))
    kappa = float(rng.choice([0.0, 0.07, 0.5]))
    with_gpsi = bool(rng.integers(0, 2))
    p = io.random_params(rng, d, H, np.float64, regime)
    z, v, gpsi = rng.normal(0, 1, (B, d)), rng.normal(0, 1, (B, d)), rng.normal(0, 1, (B,))

    icnn = ref_module.ICNN(d, H).to(torch.float64)
    for w in icnn.W:
        w.is_exp = (mode == 0)
    mg.load_icnn(icnn, p, torch.float64)
    zt = torch.tensor(z, dtype=torch.float64, requires_grad=True)
    psi = icnn(zt) + kappa * zt.pow(2).sum(1, keepdim=True)                                   # model.py:820
    xhat = torch.autograd.grad(psi, [zt], torch.ones_like(psi), create_graph=True)[0]         # model.py:822
    L = (xhat * torch.tensor(v)).sum()
    if with_gpsi:
        L = L + (icnn(zt)[:, 0] * torch.tensor(gpsi)).sum()
    L.backward()
    g_ref = mg.icnn_grads(icnn)

    o_psi, o_xhat, _ = io.icnn_brenier(z, p, mode, kappa)
    o_dz, o_g = io.icnn_brenier_backward(z, v, p, mode, kappa, gpsi=gpsi if with_gpsi else None)
    tol = dict(rtol=1e-10, atol=1e-12)
    np.testing.assert_allclose(o_psi, (psi[:, 0] - kappa * zt.pow(2).sum(1)).detach().numpy(), **tol)
    np.testing.assert_allclose(o_xhat, xhat.detach().numpy(), **tol)
    np.testing.assert_allclose(o_dz, zt.grad.numpy(), rtol=1e-9, atol=1e-11)
    for k in io.PARAM_KEYS:
        scale = max(float(np.abs(g_ref[k]).max()), 1e-30)
        np.testing.assert_allclose(o_g[k].reshape(g_ref[k].shape), g_ref[k], rtol=1e-9, atol=1e-11 * scale + 1e-14)


@pytest.mark.parametrize("seed", range(4))
def test_lidvae_decode_chain_matches_live_reference(seed, ref):
    """LIDVAE.decode (model.py:818-830) of the unmodified reference, 2-D toy presets, random weights and inverse-Lipschitz."""
    from oracle import icnn_oracle as io
    mg, (_, ref_model, _) = ref
    rng = np.random.default_rng(2000 + seed)
    il = float(rng.choice([0.0, 0.2, 1.0]))
    m = ref_model.LIDVAE(dataset="pinwheel", icnn_channels=[24, 40], inverse_lipschitz=il).to(torch.float64)
    p0 = io.random_params(rng, 2, 24, np.float64, "mixed")
    p1 = io.random_params(rng, 2, 40, np.float64, "mixed")
    mg.load_icnn(m.decoder[0], p0, torch.float64)
    mg.load_icnn(m.decoder[1], p1, torch.float64)
    z = rng.normal(0, 1, (19, 2))
    y_ref = m.decode(torch.tensor(z, requires_grad=True)).detach().numpy()
    y, _, _, _ = io.lidvae_decode(z, p0, p1, 2, 0, il / 2.0)
    np.testing.assert_allclose(y, y_ref, rtol=1e-10, atol=1e-12)


@pytest.mark.parametrize("seed", range(8))
def test_lipschitz_estimator_oracle_matches_live_reference(seed, ref):
    """utils.estimate_local_lipschitz (utils.py:532-567) of the unmodified reference on CPU, random maps / sizes / quantiles,
    against the oracle fed with the same pair indices (same generator, same call order)."""
    from oracle import loss_oracle as lo
    _, (_, _, ref_utils) = ref
    rng = np.random.default_rng(3000 + seed)
    N = int(rng.integers(2, 300)); P = int(rng.choice([50, 2000, 5000])); d = int(rng.choice([2, 3, 16]))
    q = float(rng.choice([0.05, 0.1, 0.25])); eps = float(rng.choice([1e-3, 1e-2]))
    W = torch.tensor(rng.normal(0, 1, (d, 12)))
    func = lambda x: torch.tanh(x @ W).reshape(-1, 3, 2, 2) * 3.0                 # image-shaped output: rows are flattened
    X = torch.tensor(rng.normal(0, 1, (N, d)))
    if seed % 3 == 0:
        X[N // 2:] = X[:N - N // 2].clone()                                       # coincident points: both clamps active
    got = ref_utils.estimate_local_lipschitz(func, X, num_pairs=P, quantile=q, eps=eps,
                                             generator=torch.Generator().manual_seed(5 + seed))
    g = torch.Generator().manual_seed(5 + seed)
    i1 = torch.randint(0, N, (P,), generator=g).numpy()
    i2 = torch.randint(0, N, (P,), generator=g).numpy()
    r = lo.lipschitz_ratios(X.numpy(), func(X).numpy(), i1, i2, eps)
    np.testing.assert_allclose(lo.lipschitz_from_ratios(r, q, eps), got, rtol=1e-10)
