"""Pin the numpy oracle against outputs of the unmodified reference (tests/golden/, made by
oracle/make_golden.py).  CPU only.  fp64 fixtures: <=1e-11 relative-to-max; fp32 fixtures are
checked against the fp64 oracle at the fp32 noise floor."""
import os

import numpy as np
import pytest

from oracle import golden
from oracle import icnn_oracle as io
from oracle import loss_oracle as lo
from oracle.make_golden import ICNN_CASES, case_inputs

from conftest import GOLDEN


def relmax(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / (np.abs(b).max() + 1e-300))


@pytest.fixture(scope="module")
def icnn_golden():
    return golden.load(os.path.join(GOLDEN, "icnn_cases.npz"))


@pytest.mark.parametrize("case", ICNN_CASES, ids=[c[0] for c in ICNN_CASES])
def test_icnn_oracle_vs_reference_fp64(case, icnn_golden):
    name, d, H, B, regime, mode, kappa, seed, with_gpsi = case
    p, z, v, gpsi = case_inputs(d, H, B, regime, seed)
    psi, xhat, _ = io.icnn_brenier(z, p, mode, kappa)
    dz, g = io.icnn_brenier_backward(z, v, p, mode, kappa, gpsi if with_gpsi else None)
    G = icnn_golden
    pre = f"{name}/f64/"
    assert relmax(psi, G[pre + "psi"]) < 1e-12
    assert relmax(xhat, G[pre + "xhat"]) < 1e-12
    assert relmax(dz, G[pre + "dz"]) < 1e-11
    for k in io.PARAM_KEYS:
        if pre + "g_" + k in G.files:
            ref = G[pre + "g_" + k]
            if np.abs(ref).max() == 0:
                assert np.abs(g[k]).max() == 0, k      # A1b / A2b: exact zeros on the <v,xhat> path
            else:
                assert relmax(g[k], ref) < 1e-11, k
        else:
            assert relmax(g[k].reshape(-1)[::97], G[pre + "g_W0_sample"]) < 1e-11
            s = G[pre + "g_W0_sum"]
            assert abs(g[k].sum() - s[0]) <= 1e-9 * s[1]


@pytest.mark.parametrize("case", ICNN_CASES[:6], ids=[c[0] for c in ICNN_CASES[:6]])
def test_icnn_oracle_fp32_noise_floor(case, icnn_golden):
    """The reference run in fp32 differs from fp64 by fp32 rounding only (away from kinks)."""
    name, d, H, B, regime, mode, kappa, seed, with_gpsi = case
    p, z, v, gpsi = case_inputs(d, H, B, regime, seed)
    psi, xhat, _ = io.icnn_brenier(z, p, mode, kappa)
    pre = f"{name}/f32/"
    assert relmax(psi, icnn_golden[pre + "psi"]) < 5e-5
    assert relmax(xhat, icnn_golden[pre + "xhat"]) < 5e-4   # kink flips allowed for a few units


def test_mnist_shaped_decode_chain():
    G = golden.load(os.path.join(GOLDEN, "mnist_shaped.npz"))
    p0 = {k: G[f"p0/{k}"] for k in io.PARAM_KEYS}
    p1 = {k: G[f"p1/{k}"] for k in io.PARAM_KEYS}
    z, vy, kappa = G["z"], G["vy"].reshape(6, -1), float(G["kappa"])
    y, _, _, _ = io.lidvae_decode(z, p0, p1, 784, 0, kappa)
    assert relmax(y, G["y"].reshape(6, -1)) < 1e-12
    dz, g0, g1 = io.lidvae_decode_backward(z, vy, p0, p1, 784, 0, kappa)
    assert relmax(dz, G["dz"]) < 1e-11
    for k in io.PARAM_KEYS:
        for gi, g in ((0, g0), (1, g1)):
            ref = G[f"g{gi}/{k}"]
            if np.abs(ref).max() == 0:
                assert np.abs(g[k]).max() == 0
            else:
                assert relmax(g[k], ref) < 1e-11, (gi, k)


def test_losses_vs_reference():
    G = np.load(os.path.join(GOLDEN, "loss_cases.npz"))
    for name in ("l1", "l4", "l4_wide"):
        pre = f"lrvae_{name}/"
        x, xh, mu, lv, zin, zrec = (G[pre + k] for k in ("x", "xh", "mu", "lv", "zin", "zrec"))
        alpha, beta, wu = G[pre + "hyper"]
        rec, reg, lr = lo.recon_mse(x, xh), lo.kl(mu, lv), lo.latent_recon(zin, zrec)
        total = rec + beta * reg + alpha * wu * lr
        np.testing.assert_allclose([total, rec, beta * reg, alpha * wu * lr], G[pre + "out"], rtol=1e-12)
        np.testing.assert_allclose(lo.recon_mse_grad(x, xh), G[pre + "g_xh"], rtol=1e-12, atol=1e-15)
        gmu, glv = lo.kl_grad(mu, lv, beta)
        np.testing.assert_allclose(gmu, G[pre + "g_mu"], rtol=1e-12, atol=1e-15)
        np.testing.assert_allclose(glv, G[pre + "g_lv"], rtol=1e-12, atol=1e-15)
        np.testing.assert_allclose(lo.latent_recon_grad(zin, zrec, alpha * wu), G[pre + "g_zrec"], rtol=1e-12, atol=1e-15)
    pre = "lid_logmse/"
    x, xh, mu, lv = (G[pre + k] for k in ("x", "xh", "mu", "lv"))
    rec, reg = lo.recon_logmse(x, xh), lo.kl(mu, lv)
    np.testing.assert_allclose([rec + 0.4 * reg, rec, reg], G[pre + "out"], rtol=1e-12)
    np.testing.assert_allclose(lo.recon_logmse_grad(x, xh), G[pre + "g_xh"], rtol=1e-11, atol=1e-15)
    np.testing.assert_allclose(lo.kl(mu, lv), G["kld/val"], rtol=1e-12)


def test_lipschitz_vs_reference():
    G = np.load(os.path.join(GOLDEN, "lipschitz_cases.npz"))
    for name in ("n500_p2000", "n100_p100", "n5_p64_dups"):
        Z, Y, i1, i2, res = (G[f"{name}/{k}"] for k in ("Z", "Y", "i1", "i2", "res"))
        r = lo.lipschitz_ratios(Z, Y, i1, i2)
        got = lo.lipschitz_from_ratios(r)
        np.testing.assert_allclose(got, res, rtol=1e-10)
    # coincident pairs hit both clamps -> ratio exactly 1.0 (reference quirk, SURVEY.md section 4)
    Z, Y, i1, i2 = (G[f"n5_p64_dups/{k}"] for k in ("Z", "Y", "i1", "i2"))
    r = lo.lipschitz_ratios(Z, Y, i1, i2)
    assert (r[i1 == i2] == 1.0).all() and (i1 == i2).any()
