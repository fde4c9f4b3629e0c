"""The Brenier map's exact Jacobian without a GPU: the fp64 oracle (oracle.jacobian_oracle: icnn_jacobian and the
decoder chain) against central finite differences and its structure (symmetric, >= 2 kappa I), against the unmodified reference's
autograd Jacobian where a checkout is found, and the C ABI's validation of the new entry points (it refuses before any CUDA
call, so it runs here)."""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import fetch_ref
from oracle import icnn_oracle as io
from oracle import jacobian_oracle as jo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _fd_rows(f, z, h):
    """Central differences of f: [B,d] -> [B,m] per row -> [B,m,d]."""
    B, d = z.shape
    cols = []
    for j in range(d):
        e = np.zeros_like(z)
        e[:, j] = h
        cols.append((f(z + e) - f(z - e)) / (2 * h))
    return np.stack(cols, -1)


def _stable_rows(z, p, mode, h):
    """Rows whose masks (h0, h1, h2 signs) do not change anywhere within +-h along each axis: there the map is affine."""
    _, _, a = io.icnn_brenier(z, p, mode, keep=True)
    ok = np.ones(z.shape[0], dtype=bool)
    for j in range(z.shape[1]):
        for sgn in (-1, 1):
            e = np.zeros_like(z)
            e[:, j] = sgn * h
            _, _, b = io.icnn_brenier(z + e, p, mode, keep=True)
            ok &= ((a["h0"] > 0) == (b["h0"] > 0)).all(1) & (a["mask1"] == b["mask1"]).all(1) & (a["mask2"] == b["mask2"])
    return ok


@pytest.mark.parametrize("d,H,regime,mode,kappa", [(1, 16, "mixed", 0, 0.0), (2, 32, "mixed", 0, 0.15),
                                                   (3, 24, "default", 0, 0.15), (4, 40, "clampy", 1, 0.0),
                                                   (3, 64, "mixed", 1, 0.5)])
def test_icnn_jacobian_matches_finite_differences(d, H, regime, mode, kappa):
    rng = np.random.default_rng(d * 100 + H)
    p = io.random_params(rng, d, H, np.float64, regime)
    z = rng.normal(0, 1, (64, d))
    h = 1e-6
    ok = _stable_rows(z, p, mode, h)
    assert ok.sum() >= 16
    J = jo.icnn_jacobian(z, p, mode, kappa)
    Jfd = _fd_rows(lambda zz: io.icnn_brenier(zz, p, mode, kappa)[1], z, h)
    scale = np.abs(J).max()
    assert np.abs(J[ok] - Jfd[ok]).max() <= 1e-7 * scale
    np.testing.assert_allclose(J, np.swapaxes(J, 1, 2), rtol=0, atol=1e-14 * scale)
    ev = np.linalg.eigvalsh(J)
    assert (ev >= 2 * kappa - 1e-12 * scale).all()


@pytest.mark.parametrize("D,Dx,eye", [(2, 2, True), (2, 3, True), (3, 2, False), (1, 4, False)])
def test_decoder_jacobian_chain_matches_finite_differences(D, Dx, eye):
    rng = np.random.default_rng(7 * D + Dx)
    p0 = io.random_params(rng, D, 32, np.float64, "mixed")
    p1 = io.random_params(rng, Dx, 48, np.float64, "mixed")
    M = np.eye(Dx, D) if eye else rng.normal(0, 1, (Dx, D))
    kappa = 0.1
    z = rng.normal(0, 1, (48, D))

    def dec(zz):
        x1 = io.icnn_brenier(zz, p0, 0, kappa)[1]
        return io.icnn_brenier(x1 @ M.T, p1, 0, kappa)[1]

    h = 1e-6
    x = io.icnn_brenier(z, p0, 0, kappa)[1] @ M.T
    ok = _stable_rows(z, p0, 0, 4 * h) & _stable_rows(x, p1, 0, 50 * h * max(1.0, np.abs(M).max()))
    assert ok.sum() >= 8
    J, J1, J2 = jo.lidvae_decode_jacobian(z, p0, p1, Dx, 0, kappa, M=M)
    assert J.shape == (48, Dx, D)
    Jfd = _fd_rows(dec, z, h)
    assert np.abs(J[ok] - Jfd[ok]).max() <= 1e-6 * np.abs(J).max()
    if eye:      # the default M matches lidvae_decode's zero pad
        np.testing.assert_allclose(io.lidvae_decode(z, p0, p1, Dx, 0, kappa)[0], dec(z), rtol=0, atol=0)
        Jd, _, _ = jo.lidvae_decode_jacobian(z, p0, p1, Dx, 0, kappa)
        np.testing.assert_array_equal(Jd, J)
        # inverse-Lipschitz guarantee of the composed maps: sigma_min(J) >= (2 kappa)^2 when Dx >= D
        if Dx >= D:
            assert np.linalg.svd(J, compute_uv=False)[:, -1].min() >= (2 * kappa) ** 2 * (1 - 1e-12)


REF = fetch_ref.REF_SRC


@pytest.mark.skipif(not (REF and os.path.isfile(os.path.join(REF, "module.py"))),
                    reason="no checkout of the reference (VAE_SONG_REFERENCE, ../reference, ../vae-song)")
@pytest.mark.parametrize("seed", range(4))
def test_oracle_jacobian_matches_reference_autograd(seed):
    """torch.autograd.functional.jacobian of the reference's own Brenier map (model.py:820-822) in fp64."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import make_golden as mg
    ref_module, _, _ = mg.import_reference()
    rng = np.random.default_rng(500 + seed)
    d, H = int(rng.choice([1, 2, 3, 4])), int(rng.choice([16, 33, 64]))
    mode, kappa = int(rng.integers(0, 2)), float(rng.choice([0.0, 0.15]))
    p = io.random_params(rng, d, H, np.float64, "mixed")
    icnn = ref_module.ICNN(d, H).to(torch.float64)
    for w in icnn.W:
        w.is_exp = (mode == 0)
    mg.load_icnn(icnn, p, torch.float64)
    z = rng.normal(0, 1, (12, d))

    def brenier(zr):
        zr = zr.unsqueeze(0)
        psi = icnn(zr) + kappa * zr.pow(2).sum(1, keepdim=True)
        return torch.autograd.grad(psi, [zr], torch.ones_like(psi), create_graph=True)[0][0]

    Jref = np.stack([torch.autograd.functional.jacobian(brenier, torch.tensor(zi)).numpy() for zi in z])
    np.testing.assert_allclose(jo.icnn_jacobian(z, p, mode, kappa), Jref, rtol=1e-9, atol=1e-11 * np.abs(Jref).max())


# ---- C ABI validation (no GPU needed: every refusal happens before a CUDA call) -----------------------------------
def _lib():
    from vae_song_b200 import _C
    try:
        return _C, _C.load()
    except _C.B200VaeError as e:
        pytest.skip(str(e))


@pytest.mark.parametrize("d,H,prec", [(5, 256, 0), (4, 256, 3), (4, 256, 4), (4, 256, 1), (2, 1280, 4), (2, 1280, 3),
                                      (2, 1280, 1), (2, 256, 2)])
def test_decode_jac_refuses_unsupported_shapes(d, H, prec):
    _C, lib = _lib()
    assert lib.b200vae_icnn_jac_scratch_bytes(256, d, H, prec) == 0
    rc = lib.b200vae_icnn_decode_jac(None, 256, d, H, 0.0, None, None, None, None, None, prec, None, 0, None, 0, None)
    assert rc == -2     # B200VAE_EUNSUP


def test_decode_jac_scratch_sizes_and_chain_validation():
    _C, lib = _lib()
    # tensor cores: Bp * NP * 2 float4 slots, two per slot at d = 3; FP32 needs none
    assert lib.b200vae_icnn_jac_scratch_bytes(65536, 3, 1024, 4) == 65536 * 4 * 2 * 2 * 16
    assert lib.b200vae_icnn_jac_scratch_bytes(65536, 2, 512, 3) == 65536 * 2 * 2 * 16
    assert lib.b200vae_icnn_jac_scratch_bytes(1, 1, 100, 1) == 256 * 1 * 2 * 16
    assert lib.b200vae_icnn_jac_scratch_bytes(1000, 4, 4096, 0) == 0
    assert lib.b200vae_icnn_decode_jac(None, 0, 2, 256, 0.0, None, None, None, None, None, 0, None, 0, None, 0, None) == -1
    assert lib.b200vae_icnn_decode_jac(None, 8, 2, 256, 0.0, None, None, None, None, None, 0, None, 0, None, 0, None) == -3
    assert lib.b200vae_jacobian_chain(None, None, None, 8, 5, 2, None, None, None) == -2
    assert lib.b200vae_jacobian_chain(None, None, None, 8, 2, 5, None, None, None) == -2
    assert lib.b200vae_jacobian_chain(None, None, None, 0, 2, 2, None, None, None) == -1
    assert lib.b200vae_jacobian_chain(None, None, None, 8, 2, 2, None, None, None) == -3


def test_icnn_brenier_jacobian_names_the_limit():
    from vae_song_b200 import _C, module
    with pytest.raises(_C.B200VaeError, match="d <= 4"):
        module.ICNN(5, 16).brenier_jacobian(torch.zeros(2, 5))
    with pytest.raises(_C.B200VaeError, match="d <= 3 and H <= 1024"):
        module.ICNN(4, 16, precision="f16x3").brenier_jacobian(torch.zeros(2, 4))
    with pytest.raises(_C.B200VaeError, match="d <= 3 and H <= 1024"):
        module.ICNN(2, 1280, precision="tf32x3").brenier_jacobian(torch.zeros(2, 2))


def test_lipschitz_parser_accepts_jacobian():
    from vae_song_b200 import lipschitz
    args = lipschitz.build_parser().parse_args(["--lipschitz_pairs", "jacobian", "--model", "lidvae"])
    assert args.lipschitz_pairs == "jacobian"
    with pytest.raises(ValueError, match="lidvae"):
        lipschitz.main(["--lipschitz_pairs", "jacobian", "--model", "lrvae"])
    with pytest.raises(ValueError, match="jacobian"):
        lipschitz._get_data_based_lipschitz(None, None, "cpu", pairs="hessian")
