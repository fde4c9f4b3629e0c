"""The Brenier map's left inverse on the GPU (b200vae_brenier_inverse_init / b200vae_brenier_newton_step on
b200vae_icnn_decode_jac) and LIDVAE.decode_inverse.

The step kernel is checked one launch at a time against oracle.inverse_oracle.newton_step on the same state; round trips
x = T(z_true) against the certificate ||z - z*|| <= err_bound, widened by what the kernel's xhat may be off (the Jacobian
suite's bound: X_RTOL (|xhat| + max|xhat|) per element) over 2 kappa."""
import numpy as np
import pytest
import torch

from oracle import icnn_oracle as io
from oracle import inverse_oracle as ivo
from oracle import jacobian_oracle as jo

from helpers import H_RTOL, kink_rows, params_to_torch

pytestmark = pytest.mark.gpu

PRECS = [0, 1, 3, 4]
X_RTOL = {0: 1e-5, 1: 5e-3, 3: 1e-5, 4: 1e-5}
COMBOS = [(1, 0, 0.1), (7, 1, 0.15), (256, 0, 0.0), (5000, 1, 0.1), (65536, 0, 0.15)]


def _rows_view(state, B):
    return state[ivo.HEADER_BYTES:].view(torch.float64).view(ivo.N_FIELDS, B)


@pytest.mark.parametrize("d,H,prec,off_image", [(3, 300, 0, False), (2, 512, 4, True), (1, 1024, 1, True)])
def test_step_kernel_matches_oracle(d, H, prec, off_image):
    """Launch by launch against oracle.inverse_oracle.newton_step, through kink crossings, until the last round
    (final_round); then every row's bound belongs to the z returned with it: err == ||xhat(z) - x|| / (2 kappa)."""
    from vae_song_b200 import _C, ops
    lib = _C.load()
    B, mode, kappa, rounds = 2000, 0, 0.1, 40
    rng = np.random.default_rng(3 + d)
    p = io.random_params(rng, d, H, np.float64, "mixed")
    P = params_to_torch(p)
    zt = rng.normal(0, 1, (B, d))
    x64 = io.icnn_brenier(zt, p, mode, kappa)[1]
    if off_image:
        x64 = x64 + rng.normal(0, 0.5, x64.shape)
    x = torch.tensor(x64, dtype=torch.float32, device="cuda")
    ws = ops.icnn_prepare(P, d, H, mode, prec, B, False)
    nst = lib.b200vae_brenier_inverse_state_bytes(B, d)
    state = torch.empty(nst, dtype=torch.uint8, device="cuda")
    trial, z = torch.empty(B, d, device="cuda"), torch.empty(B, d, device="cuda")
    status, err = torch.empty(B, dtype=torch.int32, device="cuda"), torch.empty(B, device="cuda")
    s = ops._stream()
    _C.check(lib.b200vae_brenier_inverse_init(ops._ptr(x), None, B, d, 1e-5, 1e-5, ops._ptr(state), nst, ops._ptr(trial),
                                              ops._ptr(z), ops._ptr(status), ops._ptr(err), s), "init")
    rows0, trial0, _, _, _ = ivo.init(x.double().cpu().numpy(), None, np.float32(1e-5), np.float32(1e-5))
    np.testing.assert_allclose(_rows_view(state, B).cpu().numpy(), rows0, rtol=1e-7)
    halvings, crossed = set(), set()
    for k in range(rounds):
        final = k == rounds - 1
        _, xhat, jac, _, _ = ops.icnn_decode_jac(trial, ws, d, H, kappa, prec)
        before = _rows_view(state, B).cpu().numpy().copy()
        act = before[ivo.F_STATUS] == ivo.ACTIVE
        if not act.any():
            break
        ref = ivo.newton_step(before, x.cpu().numpy(), xhat.cpu().numpy(), jac.cpu().numpy(), kappa, final=final)
        _C.check(lib.b200vae_brenier_newton_step(ops._ptr(x), ops._ptr(xhat), ops._ptr(jac), B, d, kappa, k, int(final),
                                                 ops._ptr(state), nst, ops._ptr(trial), ops._ptr(z), ops._ptr(status),
                                                 ops._ptr(err), s), "step")
        got = _rows_view(state, B).cpu().numpy()
        # the same decisions
        for f in (ivo.F_STATUS, ivo.F_NSTEP, ivo.F_NHALF, ivo.F_CROSSED, ivo.F_T, ivo.F_LO, ivo.F_HI):
            np.testing.assert_array_equal(got[f], ref[0][f], err_msg=f"field {f} round {k}")
        np.testing.assert_allclose(got[ivo.F_Z:ivo.F_Z + d], ref[0][ivo.F_Z:ivo.F_Z + d], rtol=2 ** -23, atol=1e-30)
        np.testing.assert_allclose(got[ivo.F_P:ivo.F_P + d], ref[0][ivo.F_P:ivo.F_P + d], rtol=1e-9,
                                   atol=1e-9 * np.abs(ref[0][ivo.F_P:ivo.F_P + d]).max())
        np.testing.assert_allclose(trial.cpu().numpy()[act], ref[1][act], rtol=2 ** -23, atol=1e-30)
        np.testing.assert_array_equal(status.cpu().numpy()[act], ref[3][act])
        assert int(state[:8].view(torch.int32)[k & 1]) == ref[5]
        halvings.update(np.unique(got[ivo.F_NHALF]).tolist())
        crossed.update(np.unique(got[ivo.F_CROSSED]).tolist())
    st = status.cpu().numpy()
    assert (st != ivo.ACTIVE).all()
    assert max(halvings) >= 1                   # the line search was exercised
    if off_image and d > 1:                     # ... and the kink crossings, the stalls and the last-round cut
        assert {1.0, 2.0} <= crossed and (st == ivo.STALLED).any() and (st == ivo.MAXITER).any(), (crossed, st)
    _, xz, _, _, _ = ops.icnn_decode_jac(z, ws, d, H, kappa, prec)
    want = (xz.double() - x.double()).norm(dim=1) / (2 * kappa)
    np.testing.assert_allclose(err.double().cpu().numpy(), want.cpu().numpy(), rtol=1e-6, atol=0)


def _round_trip_case(prec, d, H, B, mode, kappa, seed):
    from vae_song_b200 import ops
    rng = np.random.default_rng(seed)
    p = io.random_params(rng, d, H, np.float64, "clampy" if mode == 1 else "mixed")
    p = {k: v.astype(np.float32).astype(np.float64) for k, v in p.items()}
    P = params_to_torch(p)
    z_true = rng.normal(0, 1, (B, d)).astype(np.float32).astype(np.float64)
    x64 = io.icnn_brenier(z_true, p, mode, kappa)[1]
    x = torch.tensor(x64, dtype=torch.float32, device="cuda")
    z, st, err, rounds = ops.icnn_brenier_inverse(x, kappa, mode, prec, P, {})
    rows = np.arange(B) if B <= 5000 else np.random.default_rng(seed).choice(B, 4096, replace=False)
    z, st, err = z.double().cpu().numpy()[rows], st.cpu().numpy()[rows], err.double().cpu().numpy()[rows]
    zt, xs = z_true[rows], x64[rows]
    _, _, aux = io.icnn_brenier(zt, p, mode, kappa, keep=True)
    kink = kink_rows(aux, H_RTOL[prec], with_h0=True)
    return p, zt, xs, z, st, err, kink, rounds


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("d", [1, 2, 3, 4])
@pytest.mark.parametrize("H", [300, 512, 1024])
def test_round_trip(prec, d, H):
    if d == 4 and prec != 0:
        pytest.skip("tensor-core precisions take d <= 3")
    for i, (B, mode, kappa) in enumerate(COMBOS):
        p, zt, xs, z, st, err, kink, rounds = _round_trip_case(prec, d, H, B, mode, kappa, 700 * d + H + i)
        name = f"prec {prec} d {d} H {H} B {B} mode {mode} kappa {kappa}"
        ok = ~kink
        hist = np.bincount(st, minlength=6)
        assert (st != ivo.ACTIVE).all() and not np.isin(st, [ivo.SINGULAR, ivo.NONFINITE]).any(), (name, hist)
        conv = st[ok] == ivo.CONVERGED
        # a few kink-free rows stall on a kink surface on the way (DESIGN.md section 7): at most 1 % with trained-like
        # ("mixed") weights, 10 % with clamp-mode weights; a stalled row is still held to the certificate below
        if ok.any():
            assert conv.mean() >= (0.99 if mode == 0 else 0.9), (name, hist, np.bincount(st[ok], minlength=6))
        dist = np.linalg.norm(z - zt, axis=1)
        xn = np.linalg.norm(xs, axis=1)
        acc = X_RTOL[prec] * (xn + np.sqrt(d) * np.abs(xs).max())
        if kappa > 0:       # the certificate, on every row
            assert (dist <= err + acc / (2 * kappa) + 1e-6 * np.linalg.norm(zt, axis=1)).all(), (name, (dist - err).max())
        else:               # the local bound from sigma_min(J(z_true)) on converged kink-free rows
            smin = np.linalg.eigvalsh(jo.icnn_jacobian(zt, p, 0 if mode == 0 else 1, 0.0))[:, 0]
            c = ok & (st == ivo.CONVERGED)
            tol = X_RTOL[prec] * (xn + 1.0)
            assert (dist[c] <= 2 * (tol[c] + acc[c]) / smin[c] + 1e-6 * np.linalg.norm(zt[c], axis=1)).all(), name


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


@pytest.mark.parametrize("precision", ["fp32", "tf32", "tf32x3", "f16x3"])
@pytest.mark.parametrize("il", [0.0, 0.2])
def test_decode_inverse_round_trip(precision, il):
    from vae_song_b200 import _C
    m = _toy_lidvae(precision, il)
    z = torch.randn(8192, 2, device="cuda", generator=torch.Generator("cuda").manual_seed(5))
    with torch.no_grad():
        y = m.decode(z)
        y_before = m.decode(z)
    zi, st, bound = m.decode_inverse(y)
    with torch.no_grad():
        assert torch.equal(m.decode(z), y_before)             # decode is not disturbed
    assert zi.shape == z.shape and not zi.requires_grad
    stn = st.cpu().numpy()
    assert (stn == _C.INV_CONVERGED).mean() >= 0.99, np.bincount(stn, minlength=6)
    dist = (zi - z).norm(dim=1)
    c = st == _C.INV_CONVERGED
    rel = {"tf32": 2e-2}.get(precision, 1e-3)
    assert (dist[c] <= rel * (1 + z.norm(dim=1)[c])).float().mean() >= 0.99
    if il > 0:
        acc = 1e-2 if precision == "tf32" else 1e-4
        assert (dist <= bound + acc * (1 + z.norm(dim=1))).all()
    else:
        assert torch.isinf(bound).all()


def test_decode_inverse_modified_B_warm_start_and_refusals():
    from vae_song_b200 import _C, model
    m = _toy_lidvae("fp32", 0.2, H=(64, 128))
    with torch.no_grad():
        m.B.copy_(torch.tensor([[1.0, 0.5], [-0.25, 2.0]]))
    z = torch.randn(3000, 2, device="cuda")
    with torch.no_grad():
        y = m.decode(z)
    zi, st, bound = m.decode_inverse(y)
    c = st == _C.INV_CONVERGED
    assert c.float().mean() >= 0.99
    assert ((zi - z).norm(dim=1)[c] <= 1e-3 * (1 + z.norm(dim=1)[c])).all()
    zw, stw, _ = m.decode_inverse(y, z0=z + 1e-3)
    assert (stw == _C.INV_CONVERGED).float().mean() >= 0.99
    with torch.no_grad():
        m.B.copy_(torch.tensor([[1.0, 2.0], [0.5, 1.0]]))
    with pytest.raises(_C.B200VaeError, match="rank-deficient"):
        m.decode_inverse(y)
    wide = model.LIDVAE(dataset="mnist", icnn_channels=[64, 128], hidden_channels=[4, 8]).cuda()
    with pytest.raises(_C.B200VaeError, match="exceed"):
        wide.decode_inverse(torch.randn(4, 1, 28, 28, device="cuda"))


def test_inverse_is_reproducible_and_replays_in_a_cuda_graph():
    from vae_song_b200 import module
    torch.manual_seed(2)
    ic = module.ICNN(2, 512, precision="f16x3").cuda()
    with torch.no_grad():
        for w in ic.W:
            w.param.sub_(np.log(512) / 2)
        x = ic.brenier(torch.randn(4096, 2, device="cuda"), 0.1)[1]
    a = ic.brenier_inverse(x, 0.1, max_iter=24)
    b = ic.brenier_inverse(x, 0.1, max_iter=24)
    assert a[3] == b[3] and all(torch.equal(u, v) for u, v in zip(a[:3], b[:3]))
    xs = x.clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            ic.brenier_inverse(xs, 0.1, max_iter=24)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        out = ic.brenier_inverse(xs, 0.1, max_iter=24)
    assert out[3] == 24
    xnew = x.flip(0).contiguous()
    xs.copy_(xnew)
    g.replay()
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        ref = ic.brenier_inverse(xnew, 0.1, max_iter=24)
    torch.cuda.current_stream().wait_stream(s)
    # eager stops early once every row is done; finished rows do not change, so the results agree
    for u, v in zip(out[:3], ref[:3]):
        assert torch.equal(u, v)
