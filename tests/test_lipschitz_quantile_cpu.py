"""Host side of the exact all-pairs quantiles (include/b200vae.h, b200vae_lipschitz_select_*): exported symbols, argument
validation before any launch (no device needed) and the fp64 rank rule against the oracle's torch.quantile convention."""
import ctypes as C
import math
import os

import numpy as np
import pytest

from oracle import loss_oracle as lo

NEW = ("b200vae_lipschitz_select_state_bytes", "b200vae_lipschitz_select_hist_bytes", "b200vae_lipschitz_quantile_ranks",
       "b200vae_lipschitz_select_count", "b200vae_lipschitz_select_locate")
ESHAPE, EALIGN = -1, -3


@pytest.fixture(scope="module")
def lib():
    from vae_song_b200 import _C
    if not os.path.exists(_C.LIB_PATH):
        _C.build()
    return _C.load()


def test_select_symbols_exported(lib):
    from vae_song_b200 import _C
    for s in NEW:
        assert s in _C.EXPORTS and hasattr(lib, s), s
    assert lib.b200vae_lipschitz_select_state_bytes() >= 104
    assert lib.b200vae_lipschitz_select_hist_bytes() == 4 * 1024 * 8
    assert _C.LIPSCHITZ_SELECT_PASSES == 3


def test_select_argument_validation_without_device(lib):
    P = lambda a: C.c_void_p(a)                                   # fake device addresses: validation never touches them
    X, Y, st, h, out = P(1 << 20), P(2 << 20), P(3 << 20), P(4 << 20), P(5 << 20)
    nt = lib.b200vae_lipschitz_num_tiles(100)
    cnt = lambda X=X, Y=Y, N=100, dx=2, dy=2, eps=1e-3, tb=0, te=nt, p=0, st=st, h=h: lib.b200vae_lipschitz_select_count(
        X, Y, N, dx, dy, eps, tb, te, p, st, h, None)
    assert cnt(X=None) == EALIGN and cnt(Y=None) == EALIGN and cnt(st=None) == EALIGN and cnt(h=None) == EALIGN
    assert cnt(st=P((3 << 20) + 8)) == EALIGN and cnt(h=P((4 << 20) + 4)) == EALIGN
    assert cnt(te=nt + 1) == ESHAPE and cnt(tb=-1) == ESHAPE and cnt(tb=5, te=4) == ESHAPE
    assert cnt(p=-1) == ESHAPE and cnt(p=3) == ESHAPE
    assert cnt(N=1, te=1) == ESHAPE and cnt(dx=0) == ESHAPE and cnt(eps=0.0) == ESHAPE
    loc = lambda N=100, q0=0.05, q1=0.95, p=0, h=h, st=st, out=out: lib.b200vae_lipschitz_select_locate(
        N, q0, q1, p, h, st, out, None)
    assert loc(h=None) == EALIGN and loc(st=None) == EALIGN and loc(out=None) == EALIGN and loc(out=P((5 << 20) + 4)) == EALIGN
    assert loc(q0=-0.01) == ESHAPE and loc(q1=1.5) == ESHAPE and loc(q0=math.nan) == ESHAPE
    assert loc(p=3) == ESHAPE and loc(p=-1) == ESHAPE and loc(N=1) == ESHAPE
    k, w = C.c_longlong(), C.c_double()
    assert lib.b200vae_lipschitz_quantile_ranks(0, 0.5, C.byref(k), C.byref(w)) == ESHAPE
    assert lib.b200vae_lipschitz_quantile_ranks(10, 1.0001, C.byref(k), C.byref(w)) == ESHAPE
    assert lib.b200vae_lipschitz_quantile_ranks(10, 0.5, None, C.byref(w)) == EALIGN


@pytest.mark.parametrize("n", [1, 2, 3, 1000, 2 ** 24 + 1, 2 ** 31 + 5])
@pytest.mark.parametrize("q", [0.0, 0.05, 0.5, 0.95, 1.0])
def test_quantile_ranks_follow_torch_linear_rule(lib, n, q):
    from vae_song_b200 import ops
    k, w = ops.lipschitz_quantile_ranks(n, q)
    kh = min(k + 1, n - 1)
    assert 0 <= k <= n - 1 and 0.0 <= w < 1.0
    if n <= 2 ** 24 + 1:
        # on the sorted values 0..n-1 the oracle's quantile IS the interpolated rank: k + w (kh - k)
        assert lo.torch_quantile_linear(np.arange(n, dtype=np.float64), q) == k + w * (kh - k)
    else:   # the oracle's arithmetic, without materialising 2^31 values
        pos = q * (n - 1)
        assert (k, w) == (int(np.floor(pos)), pos - int(np.floor(pos)))
