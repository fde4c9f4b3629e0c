"""Exact all-pairs quantiles (ops.lipschitz_allpairs_quantiles, b200vae_lipschitz_select_*) against the fp64 oracle, the
stats kernel's min / max, tie blocks, one-device sharding, graph capture, more than 2^31 pairs and the public wrappers."""
import json

import numpy as np
import pytest
import torch

from oracle import loss_oracle as lo

pytestmark = pytest.mark.gpu
T = lambda a: torch.tensor(np.asarray(a, dtype=np.float32), device="cuda")


def _data(N, dx, dy, seed=None):
    rng = np.random.default_rng(N if seed is None else seed)
    X, Y = rng.normal(0, 1, (N, dx)).astype(np.float32), rng.normal(0, 2, (N, dy)).astype(np.float32)
    if N > 10:
        X[5] = X[3]; Y[5] = Y[3]                       # coincident pair -> ratio 1.0 via both clamps
    return X, Y


def _quant(X, Y, q0, q1=None):
    from vae_song_b200 import ops
    qs = (q0,) if q1 is None else (q0, q1)
    return ops.lipschitz_allpairs_quantiles(X, Y, qs, 1e-3).cpu().numpy()


@pytest.mark.parametrize("N,dx,dy", [(2, 2, 2), (3, 2, 2), (63, 2, 2), (200, 2, 2), (5000, 2, 2), (333, 3, 17)])
def test_quantiles_vs_oracle(N, dx, dy):
    X, Y = _data(N, dx, dy)
    r = lo.lipschitz_allpairs(X, Y)["ratios"]
    for q in (0.05, 0.5):
        out = _quant(T(X), T(Y), q, 1.0 - q)
        np.testing.assert_allclose(out[:2], [lo.torch_quantile_linear(r, q), lo.torch_quantile_linear(r, 1.0 - q)], rtol=2e-5)
        single = _quant(T(X), T(Y), q)
        assert single[0] == out[0]
    v = _quant(T(X), T(Y), 0.05, 0.95)
    inv = 1.0 / max(v[0], 1e-3)
    np.testing.assert_allclose([inv, v[1], max(inv, v[1])], lo.lipschitz_from_ratios(r, 0.05, 1e-3), rtol=2e-5)


@pytest.mark.parametrize("N,dx,dy", [(2, 2, 2), (200, 2, 2), (5000, 2, 2), (4097, 1, 3), (333, 3, 17)])
def test_extreme_quantiles_bit_equal_stats_min_max(N, dx, dy):
    from vae_song_b200 import ops
    X, Y = _data(N, dx, dy)
    mx, mn, _, _ = ops.lipschitz_allpairs(T(X), T(Y), 1e-3)[0].tolist()
    out = _quant(T(X), T(Y), 0.0, 1.0)
    assert out[0] == mn and out[1] == mx and out[2] == mn and out[5] == mx


def test_all_keys_tied():
    from vae_song_b200 import ops
    X, Y = np.tile([[0.3, -1.2]], (300, 1)), np.tile([[2.0, 0.5]], (300, 1))
    mx, mn, _, _ = ops.lipschitz_allpairs(T(X), T(Y), 1e-3)[0].tolist()
    assert mx == mn
    for q in (0.0, 0.05, 0.37, 0.5, 1.0):
        out = _quant(T(X), T(Y), q, 1.0 - q)
        assert (out == mn).all(), out


def test_tie_blocks_at_and_beside_boundaries():
    M, R = 40, 50
    rng = np.random.default_rng(7)
    X = np.repeat(rng.normal(0, 1, (M, 2)), R, 0).astype(np.float32)
    Y = np.repeat(rng.normal(0, 2, (M, 2)), R, 0).astype(np.float32)
    r = np.sort(lo.lipschitz_allpairs(X, Y)["ratios"])
    n = r.shape[0]
    edges = np.flatnonzero(np.diff(r) > 0) + 1                       # first rank of each tie block
    assert len(edges) > 100
    qs = []
    for b in edges[:: max(1, len(edges) // 12)]:
        qs += [b / (n - 1), (b - 0.5) / (n - 1), (b + 0.5) / (n - 1), (b - 1) / (n - 1)]
    for q in qs:
        q = min(max(q, 0.0), 1.0)
        np.testing.assert_allclose(_quant(T(X), T(Y), q)[0], lo.torch_quantile_linear(r, q), rtol=2e-5, err_msg=str(q))


@pytest.mark.parametrize("N,dx,dy", [(5000, 2, 2), (333, 3, 17)])
def test_sharded_count_equals_unsharded(N, dx, dy):
    from vae_song_b200 import _C, ops
    X, Y = _data(N, dx, dy)
    Xt, Yt = T(X), T(Y)
    ref = _quant(Xt, Yt, 0.05, 0.95)
    lib = _C.load()
    state = torch.empty(lib.b200vae_lipschitz_select_state_bytes(), dtype=torch.uint8, device="cuda")
    part = torch.empty(lib.b200vae_lipschitz_select_hist_bytes() // 8, dtype=torch.int64, device="cuda")
    total = torch.empty_like(part)
    out = torch.empty(6, dtype=torch.float64, device="cuda")
    nt = ops.lipschitz_num_tiles(N)
    for p in range(_C.LIPSCHITZ_SELECT_PASSES):
        total.zero_()
        for lo_, hi_ in ((0, nt // 3), (nt // 3, nt // 2), (nt // 2, nt)):
            ops.lipschitz_select_count(Xt, Yt, 1e-3, lo_, hi_, p, state, part)
            total += part
        ops.lipschitz_select_locate(N, 0.05, 0.95, p, total, state, out)
    assert (out.cpu().numpy() == ref).all()


def test_reproducible_and_graph_capturable():
    from vae_song_b200 import ops
    X, Y = _data(20000, 2, 2)
    X2, Y2 = _data(20000, 2, 2, seed=99)
    a, b = _quant(T(X), T(Y), 0.05, 0.95), _quant(T(X), T(Y), 0.05, 0.95)
    assert (a == b).all()
    Xd, Yd = T(X), T(Y)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ops.lipschitz_allpairs_quantiles(Xd, Yd, (0.05, 0.95))           # warm-up: buffers for this stream
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        out = ops.lipschitz_allpairs_quantiles(Xd, Yd, (0.05, 0.95))
    Xd.copy_(T(X2)); Yd.copy_(T(Y2))
    g.replay()
    torch.cuda.synchronize()
    eager = _quant(T(X2), T(Y2), 0.05, 0.95)
    assert (out.cpu().numpy() == eager).all()
    assert not (eager == a).all()


def test_more_than_2_31_pairs():
    from vae_song_b200 import ops
    N = 70000
    n = N * (N - 1) // 2
    assert n > 2 ** 31
    X, Y = _data(N, 2, 2)
    Xt, Yt = T(X), T(Y)
    mx, mn, _, cnt = ops.lipschitz_allpairs(Xt, Yt, 1e-3)[0].tolist()
    assert cnt == n
    ext = _quant(Xt, Yt, 0.0, 1.0)
    assert ext[0] == mn and ext[1] == mx
    vals = {q: _quant(Xt, Yt, q)[0] for q in (0.05, 0.5, 0.95)}
    d = 2e-5
    thr = torch.tensor([[v * (1 - d), v * (1 + d)] for v in vals.values()], dtype=torch.float64, device="cuda")
    below = torch.zeros(len(vals), dtype=torch.int64, device="cuda")    # #{r < v(1-d)}
    upto = torch.zeros(len(vals), dtype=torch.int64, device="cuda")     # #{r <= v(1+d)}
    Xd, Yd = Xt.double(), Yt.double()
    cols = torch.arange(N, device="cuda")
    for a in range(0, N, 2048):
        b = min(a + 2048, N)
        sx = ((Xd[a:b, None, :] - Xd[None, :, :]) ** 2).sum(-1).sqrt().clamp(min=1e-3)
        sy = ((Yd[a:b, None, :] - Yd[None, :, :]) ** 2).sum(-1).sqrt().clamp(min=1e-3)
        rr = (sy / sx)[cols[None, :] > torch.arange(a, b, device="cuda")[:, None]]
        for t in range(len(vals)):
            below[t] += (rr < thr[t, 0]).sum()
            upto[t] += (rr <= thr[t, 1]).sum()
        del sx, sy, rr
    below, upto = below.tolist(), upto.tolist()
    for t, q in enumerate(vals):
        k, _ = ops.lipschitz_quantile_ranks(n, q)
        assert below[t] <= k and upto[t] >= k + 1, (q, k, below[t], upto[t])


def _lidvae():
    from vae_song_b200 import model
    torch.manual_seed(0)
    m = model.LIDVAE(inverse_lipschitz=0.2, beta=0.5, dataset="pinwheel", icnn_channels=[64, 128], hidden_channels=[16, 8, 2])
    rng = np.random.default_rng(3)
    with torch.no_grad():
        for ic in (m.decoder[0], m.decoder[1]):
            H = ic.hidden_channel
            ic.W[0].param.copy_(torch.tensor(rng.normal(np.log(1.0 / H), 1.0, (H, H)), dtype=torch.float32))
            ic.W[1].param.copy_(torch.tensor(rng.normal(np.log(2.0 / H), 1.0, (1, H)), dtype=torch.float32))
    return m.cuda().eval()


def test_estimate_lipschitz_allpairs_quantile():
    from vae_song_b200 import utils
    m = _lidvae()
    Z = torch.randn(700, 2, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))
    with torch.no_grad():
        Yd = m.decode(Z)
    r = lo.lipschitz_allpairs(Z.double().cpu().numpy(), Yd.double().cpu().numpy())["ratios"]
    got = utils.estimate_lipschitz_allpairs(m.decode, Z, quantile=0.05)
    np.testing.assert_allclose([got["inverse_lipschitz"], got["lipschitz"], got["bi_lipschitz"]],
                               lo.lipschitz_from_ratios(r, 0.05, 1e-3), rtol=2e-5)
    np.testing.assert_allclose(got["quantiles"], [lo.torch_quantile_linear(r, 0.05), lo.torch_quantile_linear(r, 0.95)],
                               rtol=2e-5)
    plain = utils.estimate_lipschitz_allpairs(m.decode, Z)
    assert set(plain) == {"max", "min", "mean", "count"}
    assert all(plain[k] == got[k] for k in plain)
    one = utils.estimate_lipschitz_allpairs(m.decode, Z[:1], quantile=0.05)
    assert (one["inverse_lipschitz"], one["lipschitz"], one["bi_lipschitz"]) == (0.0, 0.0, 0.0)


def test_data_based_all_pairs_and_cli(tmp_path):
    from vae_song_b200 import lipschitz as L
    m = _lidvae()
    ds = L.GaussianMixture2D(4, 3000, center_range=4, stds=0.3, seed=2)
    torch.manual_seed(7)
    got = L._get_data_based_lipschitz(m, ds, "cuda", num_samples=1000, pairs="all")
    torch.manual_seed(7)
    with torch.no_grad():
        z, _, _ = L._data_based_samples(m, ds, "cuda", 1000)
        Yd = m.decode(z)
    r = lo.lipschitz_allpairs(z.double().cpu().numpy(), Yd.double().cpu().numpy())["ratios"]
    np.testing.assert_allclose(got, lo.lipschitz_from_ratios(r, 0.05, 1e-3), rtol=2e-5)
    with pytest.raises(ValueError):
        L._get_data_based_lipschitz(m, ds, "cuda", num_samples=100, pairs="some")
    argv = ["--model", "lidvae", "--IL", "0.2", "--beta", "0.001", "--K", "4", "--K_z", "3", "--std", "0.3", "--epochs", "1",
            "--hidden_channels", "8", "4", "2", "--train_total_samples", "512", "--batch_size", "128", "--device", "cuda",
            "--seed", "3"]
    runs = {}
    for mode in ("sampled", "all"):
        out = tmp_path / mode
        extra = [] if mode == "sampled" else ["--lipschitz_pairs", "all"]
        runs[mode] = L.main(argv + ["--output_dir", str(out)] + extra)
        summ = json.load(open(out / "summary.json"))
        assert summ["data_lipschitz_pairs"] == mode and summ["args"]["lipschitz_pairs"] == mode
        assert summ["data_bi_lips"] == max(summ["data_inv_lips"], summ["data_lips"])
    a, b = runs["sampled"], runs["all"]
    for k in a:                                   # the per-cell grids keep sampled pairs: only the data triple moves
        if k in ("data_inv_lips", "data_lips", "data_bi_lips"):
            continue
        np.testing.assert_allclose(a[k], b[k], rtol=1e-6, err_msg=k)
    assert (a["data_inv_lips"], a["data_lips"]) != (b["data_inv_lips"], b["data_lips"])
