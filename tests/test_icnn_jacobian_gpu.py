"""The Brenier map's exact Jacobian on the GPU (b200vae_icnn_decode_jac, b200vae_jacobian_chain) and what is built on it.

Bounds, vs the fp64 oracle (oracle.jacobian_oracle) evaluated with the KERNEL'S masks, |a-b| <= rtol*|b| + rtol*max|b|:
xhat's bounds -- 1e-5 for fp32 / tf32x3 / f16x3, 5e-3 for tf32.  J also jumps where a FIRST-layer pre-activation crosses
its kink (it carries s0^2), which the returned masks do not show: only the rows helpers.kink_rows(..., with_h0=True) flags
are held to the loose bound."""
import numpy as np
import pytest
import torch

from oracle import icnn_oracle as io
from oracle import jacobian_oracle as jo

from helpers import (H_RTOL, check_decode_with_masks, close_rows, f32_as_f64, kink_rows, params_f32_as_f64, params_to_torch,
                     unpack_mask1)

pytestmark = pytest.mark.gpu

PRECS = [0, 1, 3, 4]
X_RTOL = {0: 1e-5, 1: 5e-3, 3: 1e-5, 4: 1e-5}
# (B, weight mode, kappa): every value of each axis appears for every (precision, d, H)
COMBOS = [(1, 0, 0.0), (7, 1, 0.15), (256, 0, 0.15), (65536, 1, 0.0)]


def _setup(d, H, B, mode, seed, regime="mixed", zscale=1.0):
    rng = np.random.default_rng(seed)
    p = io.random_params(rng, d, H, np.float64, "clampy" if mode == 1 else regime)
    z = rng.normal(0, zscale, (B, d)).astype(np.float32)
    return p, params_to_torch(p), z, torch.tensor(z, device="cuda")


def _check_jac(jac, m1, m2, z, p, rows, mode, kappa, prec, name):
    p64 = params_f32_as_f64(p)
    z64 = f32_as_f64(z[rows])
    H = p["A0w"].shape[0]
    km = (unpack_mask1(m1, H)[rows], m2.cpu().numpy().astype(bool)[rows])
    ref = jo.icnn_jacobian(z64, p64, mode, kappa, masks=km)
    _, _, aux = io.icnn_brenier(z64, p64, mode, kappa, keep=True)
    kink = kink_rows(aux, H_RTOL[prec], with_h0=True)
    return close_rows(jac.cpu().numpy()[rows], ref, X_RTOL[prec], name, kink, loose=5e-2)


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("d", [1, 2, 3, 4])
@pytest.mark.parametrize("H", [512, 1024, 300])
def test_jacobian_matches_oracle_and_decode_bitwise(prec, d, H):
    from vae_song_b200 import ops
    if d == 4 and prec != 0:
        pytest.skip("tensor-core precisions take d <= 3")
    for i, (B, mode, kappa) in enumerate(COMBOS):
        p, P, z, zt = _setup(d, H, B, mode, 1000 * d + H + i)
        ws = ops.icnn_prepare(P, d, H, mode, prec, B, False)
        psi, xhat, jac, m1, m2 = ops.icnn_decode_jac(zt, ws, d, H, kappa, prec, save_masks=True)
        fpsi, fxhat, fm1, fm2 = ops.icnn_decode_fwd(zt, ws, d, H, mode, kappa, prec, True, True, True)
        # the Jacobian variant runs the decode's arithmetic unchanged
        assert torch.equal(psi, fpsi) and torch.equal(xhat, fxhat) and torch.equal(m1, fm1) and torch.equal(m2, fm2)
        assert jac.shape == (B, d, d) and torch.isfinite(jac).all()
        assert torch.equal(jac, jac.transpose(1, 2))
        rows = np.arange(B) if B <= 256 else np.random.default_rng(i).choice(B, 512, replace=False)
        _check_jac(jac, m1, m2, z, p, rows, mode, kappa, prec, f"jac prec {prec} d {d} H {H} B {B}")


@pytest.mark.parametrize("zscale,wspread", [(1e-3, 2.0), (1.0, 2.0), (300.0, 2.0), (1e-2, 2.0)],
                         ids=["tiny_z", "unit_z", "huge_z", "small_z"])
def test_f16x3_jacobian_is_scale_robust(zscale, wspread):
    """The |z| and weight range of test_icnn_tc_gpu.py::test_f16x3_is_scale_robust: FP16 operands scaled per row / tensor."""
    from vae_song_b200 import ops
    d, H, B, mode, prec, kappa = 2, 512, 600, 0, 4, 0.15
    rng = np.random.default_rng(int(zscale * 1e3) + 17)
    p = io.random_params(rng, d, H, np.float64, "mixed")
    p["W0"] = p["W0"] + rng.normal(0, wspread, p["W0"].shape)
    P = params_to_torch(p)
    z = rng.normal(0, zscale, (B, d)).astype(np.float32)
    zt = torch.tensor(z, device="cuda")
    ws = ops.icnn_prepare(P, d, H, mode, prec, B, False)
    psi, xhat, jac, m1, m2 = ops.icnn_decode_jac(zt, ws, d, H, kappa, prec, save_masks=True)
    check_decode_with_masks(psi, xhat, m1, m2, f32_as_f64(z), params_f32_as_f64(p), mode, kappa, 1e-5, 1e-5, H_RTOL[prec],
                            f"scale {zscale}")
    _check_jac(jac, m1, m2, z, p, np.arange(B), mode, kappa, prec, f"jac scale {zscale}")


@pytest.mark.parametrize("prec", PRECS)
def test_jacobian_columns_match_autograd_through_the_backward_kernels(prec):
    from vae_song_b200 import module
    d, H, B = 3, 512, 1000
    torch.manual_seed(3)
    ic = module.ICNN(d, H, precision=["fp32", "tf32", None, "tf32x3", "f16x3"][prec]).cuda()
    with torch.no_grad():
        for w in ic.W:
            w.param.sub_(np.log(H) / 2)
    z = torch.randn(B, d, device="cuda")
    _, _, jac = ic.brenier_jacobian(z, 0.15)
    zg = z.clone().requires_grad_(True)
    _, xhat = ic.brenier(zg, 0.15)
    for i in range(d):
        e = torch.zeros_like(xhat)
        e[:, i] = 1.0
        (g,) = torch.autograd.grad(xhat, zg, e, retain_graph=True)
        ref = g.double().cpu().numpy()              # row i of J (J^T e_i; J is symmetric)
        err = np.abs(jac[:, i, :].double().cpu().numpy() - ref).max() / np.abs(ref).max()
        assert err <= (5e-3 if prec == 1 else 1e-4), (i, err)


@pytest.mark.parametrize("prec", [1, 3, 4])
def test_workspace_guards(prec):
    """A Jacobian call never writes the saved GEMM2 accumulators nor the saved-state bookkeeping."""
    from vae_song_b200 import ops
    d, H, B, mode = 2, 1024, 4096, 0
    p, P, z, zt = _setup(d, H, B, mode, 77)
    v = torch.randn(B, d, device="cuda")
    z2 = torch.randn(B, d, device="cuda")

    def train_pair(interpose):
        ws = ops.icnn_prepare(P, d, H, mode, prec, B, True)
        _, _, m1, m2 = ops.icnn_decode_fwd(zt, ws, d, H, mode, 0.1, prec, True, True, True)
        if interpose:
            ops.icnn_decode_jac(z2, ws, d, H, 0.1, prec)
        return ops.icnn_decode_bwd(zt, v, None, m1, m2, P, ws, d, H, mode, 0.1, prec, allow_defer=False)

    dz_a, g_a = train_pair(False)
    dz_b, g_b = train_pair(True)
    assert torch.equal(dz_a, dz_b) and all(torch.equal(a, b) for a, b in zip(g_a, g_b))

    ws = ops.icnn_prepare(P, d, H, mode, prec, B, True)
    j1 = ops.icnn_decode_jac(zt, ws, d, H, 0.1, prec, save_masks=True)
    j2 = ops.icnn_decode_jac(zt, ws, d, H, 0.1, prec, save_masks=True)
    assert all(torch.equal(a, b) for a, b in zip(j1, j2))
    after = ops.icnn_decode_fwd(z2, ws, d, H, mode, 0.1, prec, True, True, True)
    fresh = ops.icnn_decode_fwd(z2, ops.icnn_prepare(P, d, H, mode, prec, B, True), d, H, mode, 0.1, prec, True, True, True)
    assert all(torch.equal(a, b) for a, b in zip(after, fresh))


def _toy_lidvae(precision, il=0.2, H=(512, 1024)):
    from vae_song_b200 import model
    torch.manual_seed(11)
    m = model.LIDVAE(dataset="pinwheel", icnn_channels=list(H), hidden_channels=[16, 2], inverse_lipschitz=il,
                     precision=precision).cuda().eval()
    with torch.no_grad():
        for ic in (m.decoder[0], m.decoder[1]):
            for w in ic.W:
                w.param.sub_(np.log(ic.hidden_channel) / 2)
    return m


def _icnn_np(ic):
    return {k: t.detach().double().cpu().numpy() for k, t in zip(io.PARAM_KEYS, ic._flat_params())}


@pytest.mark.parametrize("precision", ["fp32", "tf32", "tf32x3", "f16x3"])
@pytest.mark.parametrize("B", [300, 8192])
def test_decode_jacobian_lidvae(precision, B):
    from vae_song_b200 import module
    m = _toy_lidvae(precision)
    z = torch.randn(B, 2, device="cuda", generator=torch.Generator("cuda").manual_seed(B))
    recon, J, s = m.decode_jacobian(z)
    with torch.no_grad():
        ref_recon = m.decode(z)
    if precision != "fp32" or B >= module.ICNN.FP32_TILED_BELOW:
        assert torch.equal(recon, ref_recon)
    else:    # fp32 decode takes the tiled chain below FP32_TILED_BELOW
        r = ref_recon.double().cpu().numpy()
        assert np.abs(recon.double().cpu().numpy() - r).max() <= 1e-5 * np.abs(r).max()
    prec = {"fp32": 0, "tf32": 1, "tf32x3": 3, "f16x3": 4}[precision]
    z64 = z.double().cpu().numpy()
    p0, p1 = _icnn_np(m.decoder[0]), _icnn_np(m.decoder[1])
    kappa = m.il_factor
    Jref, _, _ = jo.lidvae_decode_jacobian(z64, p0, p1, 2, 0, kappa)
    _, _, a0 = io.icnn_brenier(z64, p0, 0, kappa, keep=True)
    x64 = io.icnn_brenier(z64, p0, 0, kappa)[1]
    _, _, a1 = io.icnn_brenier(x64, p1, 0, kappa, keep=True)
    kink = kink_rows(a0, H_RTOL[prec], with_h0=True) | kink_rows(a1, H_RTOL[prec], with_h0=True)
    close_rows(J.cpu().numpy(), Jref, 2e-2 if prec == 1 else 1e-4, f"decoder J {precision}", kink, loose=1e-1)
    Jk = J.double().cpu().numpy()
    sv = np.linalg.svd(Jk, compute_uv=False)
    sk = s.double().cpu().numpy()
    assert (np.abs(sk - sv) <= 1e-6 * sv[:, :1]).all()
    assert (sk[:, :-1] >= sk[:, 1:]).all()
    il = 2 * kappa
    assert sk[:, -1].min() >= il * il * (1 - 1e-5)


def test_decode_jacobian_honours_a_modified_B_and_refuses_wide_decoders():
    from vae_song_b200 import _C, model
    m = _toy_lidvae("fp32", H=(64, 128))
    with torch.no_grad():
        m.B.copy_(torch.tensor([[1.0, 0.5], [-0.25, 2.0]]))
    z = torch.randn(700, 2, device="cuda")
    recon, J, _ = m.decode_jacobian(z)
    with torch.no_grad():
        ref = m.decode(z)
    assert np.abs((recon - ref).double().cpu().numpy()).max() <= 1e-5 * ref.abs().max().item()
    z64 = z.double().cpu().numpy()
    Jref, _, _ = jo.lidvae_decode_jacobian(z64, _icnn_np(m.decoder[0]), _icnn_np(m.decoder[1]), 2, 0, m.il_factor,
                                           M=m.B.double().cpu().numpy())
    err = np.abs(J.double().cpu().numpy() - Jref).max(axis=(1, 2)) / np.abs(Jref).max()
    assert np.median(err) <= 1e-5
    wide = model.LIDVAE(dataset="mnist", icnn_channels=[64, 128], hidden_channels=[4, 8]).cuda()
    with pytest.raises(_C.B200VaeError, match="exceed"):
        wide.decode_jacobian(torch.randn(4, wide.latent_channel, device="cuda"))


def test_jacobian_chain_general_shapes():
    from vae_song_b200 import ops
    g = torch.Generator("cuda").manual_seed(5)
    for Dx, D in [(1, 1), (4, 2), (2, 4), (3, 3), (4, 4)]:
        J2 = torch.randn(257, Dx, Dx, device="cuda", generator=g)
        M = torch.randn(Dx, D, device="cuda", generator=g)
        J1 = torch.randn(257, D, D, device="cuda", generator=g)
        J, s = ops.jacobian_chain(J2, M, J1)
        ref = J2.double() @ M.double() @ J1.double()
        assert (J.double() - ref).abs().max() <= 1e-6 * ref.abs().max()
        sv = np.linalg.svd(J.double().cpu().numpy(), compute_uv=False)
        assert np.abs(s.double().cpu().numpy() - sv).max() <= 1e-6 * sv.max()


def test_estimators_equal_numpy_on_the_same_singular_values():
    from vae_song_b200 import lipschitz, utils
    m = _toy_lidvae("f16x3")
    z = torch.randn(5000, 2, device="cuda", generator=torch.Generator("cuda").manual_seed(1))
    r = utils.estimate_local_lipschitz_jacobian(m, z)
    s = m.decode_jacobian(z)[2].cpu().numpy()
    A = max(float(np.quantile(s[:, -1].astype(np.float64), 0.05)), 1e-3)
    Bq = float(np.quantile(s[:, 0].astype(np.float64), 0.95))
    np.testing.assert_allclose(r, (1 / A, Bq, max(1 / A, Bq)), rtol=1e-6)
    assert utils.estimate_local_lipschitz_jacobian(m, z[:0]) == (0.0, 0.0, 0.0)

    ds = lipschitz.GaussianMixture2D(4, 800, seed=3)
    torch.manual_seed(9)
    m.eval()
    with torch.no_grad():
        zz, _, _ = lipschitz._data_based_samples(m, ds, "cuda", 5000)
        want = utils.estimate_local_lipschitz_jacobian(m, zz)
    torch.manual_seed(9)
    got = lipschitz._get_data_based_lipschitz(m, ds, "cuda", pairs="jacobian")
    assert got == want


@pytest.mark.parametrize("precision", ["fp32", "f16x3"])
def test_decode_jacobian_replays_in_a_cuda_graph(precision):
    m = _toy_lidvae(precision)
    B = 8192
    zs = torch.randn(B, 2, device="cuda")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            m.decode_jacobian(zs)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):          # the warm-up's stream: the prepared workspace is reused, not rebuilt
        out = m.decode_jacobian(zs)
    znew = torch.randn(B, 2, device="cuda")
    zs.copy_(znew)
    g.replay()
    torch.cuda.synchronize()
    ref = m.decode_jacobian(znew)
    for a, b in zip(out, ref):
        assert torch.equal(a, b)
