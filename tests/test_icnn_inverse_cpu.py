"""The Brenier map's left inverse without a GPU: the fp64 Newton solver of oracle.inverse_oracle (the step kernel's state
machine) on round trips and off-image targets, and the C ABI's validation of the new entry points (it refuses before any
CUDA call, so it runs here)."""
import numpy as np
import pytest

from oracle import icnn_oracle as io
from oracle import inverse_oracle as ivo
from oracle import jacobian_oracle as jo

from helpers import kink_rows


def _round_trip(d, regime, kappa, B=64, H=32):
    rng = np.random.default_rng(100 * d + 10 * (regime == "clampy") + int(kappa * 10))
    mode = io.MODE_CLAMP if regime == "clampy" else io.MODE_EXP
    p = io.random_params(rng, d, H, np.float64, regime)
    zt = rng.normal(0, 1, (B, d))
    x = io.icnn_brenier(zt, p, mode, kappa)[1]
    z, st, err, rounds = ivo.brenier_inverse(x, p, mode, kappa)
    _, _, aux = io.icnn_brenier(zt, p, mode, kappa, keep=True)
    kink = kink_rows(aux, 1e-6, with_h0=True)
    rel = np.linalg.norm(z - zt, axis=1) / np.maximum(np.linalg.norm(zt, axis=1), 1e-300)
    return p, mode, x, zt, z, st, err, kink, rel


@pytest.mark.parametrize("kappa", [0.0, 0.1])
@pytest.mark.parametrize("regime", ["mixed", "clampy"])
@pytest.mark.parametrize("d", [1, 2, 3, 4])
def test_oracle_round_trip_recovers_z(d, regime, kappa):
    p, mode, x, zt, z, st, err, kink, rel = _round_trip(d, regime, kappa)
    ok = ~kink
    assert ok.sum() >= 32
    # a CONVERGED row is always right; a row that is not must say so
    conv = ok & (st == ivo.CONVERGED)
    assert (rel[conv] <= 1e-10).all(), rel[conv].max()
    assert np.isin(st[ok & ~conv], [ivo.STALLED]).all(), np.bincount(st, minlength=6)
    if regime == "mixed":      # trained-like weights: every kink-free row converges
        assert conv.sum() == ok.sum(), np.bincount(st[ok], minlength=6)
    else:
        assert conv.sum() >= 0.8 * ok.sum(), np.bincount(st[ok], minlength=6)
    if kappa > 0:              # the certificate holds on every row, stalled and kink rows included
        dist = np.linalg.norm(z - zt, axis=1)
        xz = io.icnn_brenier(z, p, mode, kappa)[1]
        np.testing.assert_allclose(err, np.linalg.norm(xz - x, axis=1) / (2 * kappa), rtol=1e-12, atol=1e-300)
        assert (dist <= err * (1 + 1e-9) + 1e-12).all()
    else:
        assert np.isinf(err).all()


@pytest.mark.parametrize("d", [2, 3])
def test_oracle_off_image_targets(d):
    """Random targets, many of which fall into the jump of the gradient at the h2 kink (there the minimiser lies on the
    kink surface): every row carries its certificate and ends below its start in f = psi + kappa|.|^2 - <x, .>; a
    CONVERGED row is a minimiser against small moves.  Rows stalled on the kink surface are not (DESIGN.md section 7)."""
    rng = np.random.default_rng(40 + d)
    kappa, mode = 0.1, io.MODE_EXP
    p = io.random_params(rng, d, 24, np.float64, "mixed")
    zs = rng.normal(0, 1, (48, d))
    x = io.icnn_brenier(zs, p, mode, kappa)[1] + rng.normal(0, 0.5, (48, d))
    z, st, err, _ = ivo.brenier_inverse(x, p, mode, kappa)
    psi, xz, _ = io.icnn_brenier(z, p, mode, kappa)
    np.testing.assert_allclose(err, np.linalg.norm(xz - x, axis=1) / (2 * kappa), rtol=1e-12, atol=1e-300)
    assert np.isin(st, [ivo.CONVERGED, ivo.STALLED]).all(), np.bincount(st, minlength=6)
    conv = st == ivo.CONVERGED
    assert conv.sum() >= 12

    def f(zz):
        return io.icnn_brenier(zz, p, mode, kappa)[0] + kappa * (zz * zz).sum(1) - (x * zz).sum(1)

    f0 = f(z)
    scale = np.abs(f0).max() + 1.0
    assert (f0 <= f(np.zeros_like(z)) + 1e-12 * scale).all()
    for _ in range(16):
        delta = rng.normal(0, 1, z.shape)
        delta *= 1e-4 / np.linalg.norm(delta, axis=1, keepdims=True)
        assert (f0[conv] <= f(z + delta)[conv] + 1e-12 * scale).all()


@pytest.mark.parametrize("regime,mode", [("mixed", io.MODE_EXP), ("clampy", io.MODE_CLAMP)])
def test_oracle_stop_at_any_round_keeps_an_evaluated_z(regime, mode):
    """A solve stopped after ANY round (a fixed round budget, a CUDA-graph capture) returns a z whose xhat has been
    evaluated: err == ||xhat(z) - x|| / (2 kappa), also when the last round proposed a kink crossing, and the certificate
    ||z - z*|| <= err holds for round-trip targets."""
    rng = np.random.default_rng(7 + mode)
    kappa, d = 0.1, 2
    p = io.random_params(rng, d, 24, np.float64, regime)
    zt = rng.normal(0, 1, (48, d))
    x = io.icnn_brenier(zt, p, mode, kappa)[1]
    x_off = x + rng.normal(0, 0.5, x.shape)
    pending = 0
    for target, known in ((x, True), (x_off, False)):
        rows, trial, _, _, _ = ivo.init(target, None, 1e-13, 1e-13, rnd=ivo._f64)
        for k in range(60):
            xh = io.icnn_brenier(trial, p, mode, kappa)[1]
            J = jo.icnn_jacobian(trial, p, mode, kappa)
            stop = ivo.newton_step(rows, target, xh, J, kappa, final=True, rnd=ivo._f64)
            pending += int((rows[ivo.F_CROSSED] == 2).sum())
            z, err = stop[2], stop[4]
            assert (stop[3] != ivo.ACTIVE).all()
            np.testing.assert_allclose(err, np.linalg.norm(io.icnn_brenier(z, p, mode, kappa)[1] - target, axis=1)
                                       / (2 * kappa), rtol=1e-12, atol=1e-300)
            if known:
                assert (np.linalg.norm(z - zt, axis=1) <= err * (1 + 1e-9) + 1e-12).all(), k
            rows, trial, _, _, _, active = ivo.newton_step(rows, target, xh, J, kappa, rnd=ivo._f64)
            if active == 0:
                break
    assert pending > 0          # some stops fell on a round that had proposed a kink crossing


def test_oracle_step_statuses():
    """Init refuses non-finite rows; a singular Jacobian stops the row; finished rows keep z and their trial point."""
    x = np.array([[1.0, 2.0], [np.nan, 0.0], [0.5, 0.5]])
    rows, trial, z, st, err = ivo.init(x, None, 1e-5, 1e-5)
    assert list(st) == [ivo.ACTIVE, ivo.NONFINITE, ivo.ACTIVE] and np.isinf(err).all()
    xhat = np.array([[0.0, 0.0], [0.0, 0.0], [0.5, 0.5]])
    jac = np.stack([np.eye(2) * 2.0, np.eye(2), np.zeros((2, 2))])
    rows2, trial2, z2, st2, err2, active = ivo.newton_step(rows, x, xhat, jac, 0.1)
    assert list(st2) == [ivo.ACTIVE, ivo.NONFINITE, ivo.CONVERGED] and active == 1
    np.testing.assert_array_equal(trial2[0], [0.5, 1.0])        # z + p, p = -J^{-1} r
    np.testing.assert_array_equal(trial2[2], z2[2])
    assert err2[2] == 0.0
    jac[0] = 0.0
    rows3, _, _, st3, _, _ = ivo.newton_step(rows, x, xhat, jac, 0.0)
    assert st3[0] == ivo.SINGULAR


# ---- C ABI validation (no GPU needed: every refusal happens before a CUDA call) -----------------------------------
def _lib():
    from vae_song_b200 import _C
    try:
        return _C, _C.load()
    except _C.B200VaeError as e:
        pytest.skip(str(e))


def test_inverse_abi_validation():
    _C, lib = _lib()
    assert lib.b200vae_brenier_inverse_state_bytes(1000, 2) == ivo.state_bytes(1000)
    assert lib.b200vae_brenier_inverse_state_bytes(1000, 4) == ivo.state_bytes(1000)
    for B, d in [(0, 2), (-3, 2), (8, 0), (8, 5)]:
        assert lib.b200vae_brenier_inverse_state_bytes(B, d) == 0
    init, step = lib.b200vae_brenier_inverse_init, lib.b200vae_brenier_newton_step
    assert init(None, None, 8, 5, 1e-5, 1e-5, None, 0, None, None, None, None, None) == -2        # EUNSUP
    assert init(None, None, 0, 2, 1e-5, 1e-5, None, 0, None, None, None, None, None) == -1        # ESHAPE
    assert init(None, None, -1, 2, 1e-5, 1e-5, None, 0, None, None, None, None, None) == -1
    assert init(None, None, 8, 2, 1e-5, 1e-5, None, 0, None, None, None, None, None) == -3        # EALIGN
    assert step(None, None, None, 8, 5, 0.1, 0, 0, None, 0, None, None, None, None, None) == -2
    assert step(None, None, None, 0, 2, 0.1, 0, 0, None, 0, None, None, None, None, None) == -1
    assert step(None, None, None, 8, 2, 0.1, -1, 0, None, 0, None, None, None, None, None) == -1
    assert step(None, None, None, 8, 2, 0.1, 0, 0, None, 0, None, None, None, None, None) == -3


def test_brenier_inverse_names_the_limit():
    import torch
    from vae_song_b200 import _C, module
    with pytest.raises(_C.B200VaeError, match="d <= 4"):
        module.ICNN(5, 16).brenier_inverse(torch.zeros(2, 5))
    with pytest.raises(_C.B200VaeError, match="d <= 3 and H <= 1024"):
        module.ICNN(4, 16, precision="f16x3").brenier_inverse(torch.zeros(2, 4))
