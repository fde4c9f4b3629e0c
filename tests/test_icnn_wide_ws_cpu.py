"""Size rule of b200vae_icnn_wide_workspace_bytes and the wide entries' precision check, on the host alone (validation
runs before any launch, so no device is needed)."""
import ctypes as C
import os

import pytest

FP32, TF32, TF32X3, F16X3 = 0, 1, 3, 4
EUNSUP = -2
# (B, d, H): the MNIST-shaped decoder's two ICNNs at the config batch and at a large batch, a narrow-input shape the FP32
# small-batch routing sends here, and ragged sizes
SHAPES = [(256, 32, 512), (256, 784, 1024), (8192, 784, 1024), (4096, 2, 512), (37, 5, 40), (1000, 36, 96)]


@pytest.fixture(scope="module")
def lib():
    from vae_song_b200 import _C
    if not os.path.exists(_C.LIB_PATH):
        _C.build()
    return _C.load()


def test_refused_calls_get_no_workspace(lib):
    ws = lib.b200vae_icnn_wide_workspace_bytes
    for bwd in (0, 1):
        for prec in (FP32, TF32, TF32X3, F16X3):
            for B, d, H in ((0, 32, 512), (256, 0, 512), (256, 32, 0), (-1, 32, 512), (256, -3, 512), (256, 32, -8)):
                assert ws(B, d, H, prec, bwd) == 0, (B, d, H, prec, bwd)
        for prec in (2, -1, 5, 99):                   # 2 is reserved
            assert ws(256, 32, 512, prec, bwd) == 0, (prec, bwd)


@pytest.mark.parametrize("shape", SHAPES, ids=[f"b{s[0]}_d{s[1]}_h{s[2]}" for s in SHAPES])
def test_size_rule(lib, shape):
    ws = lambda prec, bwd: lib.b200vae_icnn_wide_workspace_bytes(*shape, prec, bwd)
    for bwd in (0, 1):
        assert ws(F16X3, bwd) == ws(TF32X3, bwd)    # f16x3 runs as tf32x3
        for prec in (FP32, TF32, TF32X3):
            assert ws(prec, bwd) > 0 and ws(prec, bwd) % 256 == 0
            # a tensor-core precision may run the FP32 kernels (nz % 4 != 0, unaligned biases): it never gets less
            assert ws(prec, bwd) >= ws(FP32, bwd)
    for prec in (FP32, TF32, TF32X3, F16X3):
        assert ws(prec, 1) >= ws(prec, 0)


def test_entries_refuse_unknown_precision_before_any_launch(lib):
    from vae_song_b200 import _C
    fake = lambda a: C.c_void_p(a << 20)             # never dereferenced: the precision check comes first
    p = _C.IcnnParams(*[fake(i + 1).value for i in range(8)])
    g = _C.IcnnGrads()
    B, d, nz, H = 256, 32, 32, 512
    for prec in (2, -1, 99):
        assert lib.b200vae_icnn_wide_fwd(fake(10), B, d, nz, H, C.byref(p), 0, 0.1, fake(11), fake(12), fake(13), fake(14),
                                         fake(15), fake(16), prec, fake(17), 1 << 30, None) == EUNSUP
        assert lib.b200vae_icnn_wide_bwd(fake(10), fake(11), fake(12), fake(13), fake(14), B, d, nz, H, C.byref(p), 0, 0.1,
                                         C.byref(g), fake(15), fake(16), fake(17), fake(18), fake(19), prec, fake(20),
                                         1 << 30, None) == EUNSUP
