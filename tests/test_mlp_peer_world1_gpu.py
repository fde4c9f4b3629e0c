"""Cross-rank (peer) BatchNorm layer entries with a one-rank PeerComm against the single-GPU entries on the same inputs:
batch statistics, running statistics, local and global (S1, S2) sums, dyhat.  With one rank the rank merge is exact, so
the two routes differ only in how they merge the per-CTA partials: above 64 partials both merge lane-strided in the same
order (equal bits), below that the single-GPU route merges per thread in CTA order (reordered FP32 sums)."""
import pytest
import torch

pytestmark = pytest.mark.gpu

# (width, batch): a narrow layer and a tile layer whose finalize is fused into the layer kernel, and a tile layer with
# 513 CTAs x 128 columns > 65536 partial loads, which runs the stand-alone finalize kernels
CASES = [(4, 4097), (128, 4096), (128, 65664)]


@pytest.fixture(scope="module")
def comm(tmp_path_factory):
    import torch.distributed as dist
    from vae_song_b200 import peer
    path = tmp_path_factory.mktemp("pg") / "init"
    dist.init_process_group("gloo", init_method=f"file://{path}", rank=0, world_size=1)
    c = peer.PeerComm()
    yield c
    c.close()
    dist.destroy_process_group()


def _tol(nparts, what):
    return dict(rtol=0, atol=0, msg=what) if nparts > 64 else dict(rtol=1e-6, atol=1e-7, msg=what)


@pytest.mark.parametrize("w,B", CASES, ids=[f"w{w}-B{B}" for w, B in CASES])
def test_peer_world1_matches_single_gpu(comm, w, B):
    from vae_song_b200 import _C
    from vae_song_b200.ops import _ptr, _stream
    lib = _C.load()
    gen = torch.Generator(device="cuda").manual_seed(w * 7 + B)
    dev = dict(dtype=torch.float32, device="cuda")
    x = torch.randn(B, w, generator=gen, **dev) * 2 + 0.5
    W = torch.randn(w, w, generator=gen, **dev) / w ** 0.5
    bias = torch.randn(w, generator=gen, **dev)
    gamma = torch.rand(w, generator=gen, **dev) + 0.5
    beta = torch.rand(w, generator=gen, **dev) - 0.5
    da = torch.randn(B, w, generator=gen, **dev)
    rm0 = torch.rand(w, generator=gen, **dev) - 0.5
    rv0 = torch.rand(w, generator=gen, **dev) + 0.5
    slope, eps, mom = 0.01, 1e-5, 0.1
    nbytes = lib.b200vae_mlp_scratch_bytes(B)

    def fwd(peer):
        y, st = torch.empty(B, w, **dev), torch.empty(4, w, **dev)
        rm, rv = rm0.clone(), rv0.clone()
        scratch = torch.zeros(nbytes, dtype=torch.uint8, device="cuda")
        args = (_ptr(x), None, None, None, slope, _ptr(W), _ptr(bias), B, w, w, _ptr(y), _ptr(st), eps, _ptr(rm), _ptr(rv),
                mom, _ptr(scratch))
        if peer:
            _C.check(lib.b200vae_mlp_layer_fwd_peer(*args, comm.ref, comm.new_slot(), _stream()), "mlp_layer_fwd_peer")
        else:
            _C.check(lib.b200vae_mlp_layer_fwd(*args, _stream()), "mlp_layer_fwd")
        return y, st, rm, rv

    y, st, rm, rv = fwd(False)
    y_p, st_p, rm_p, rv_p = fwd(True)
    ncta = min(-(-B // 256), 592) if w <= 8 else -(-B // 128)
    torch.testing.assert_close(y_p, y, rtol=0, atol=0)
    torch.testing.assert_close(st_p, st, **_tol(ncta, "stats"))
    torch.testing.assert_close(rm_p, rm, **_tol(ncta, "running_mean"))
    torch.testing.assert_close(rv_p, rv, **_tol(ncta, "running_var"))

    def bwd_reduce(peer):
        dyhat, sums = torch.empty(B, w, **dev), torch.empty(2, w, **dev)
        scratch = torch.zeros(nbytes, dtype=torch.uint8, device="cuda")
        args = (_ptr(da), _ptr(y), _ptr(st), _ptr(gamma), _ptr(beta), slope, B, w, _ptr(dyhat))
        if peer:
            glob = torch.empty(2, w, **dev)
            _C.check(lib.b200vae_mlp_layer_bwd_reduce_peer(*args, _ptr(sums), _ptr(glob), _ptr(scratch), comm.ref,
                                                           comm.new_slot(), _stream()), "mlp_layer_bwd_reduce_peer")
            return dyhat, sums, glob
        _C.check(lib.b200vae_mlp_layer_bwd_reduce(*args, _ptr(sums), _ptr(scratch), _stream()), "mlp_layer_bwd_reduce")
        return dyhat, sums

    dyhat, sums = bwd_reduce(False)
    dyhat_p, loc_p, glob_p = bwd_reduce(True)
    nblk = min(max(-(-B * w // 1024), 1), 296)
    torch.testing.assert_close(dyhat_p, dyhat, rtol=0, atol=0)
    torch.testing.assert_close(loc_p, sums, **_tol(nblk, "local sums"))
    torch.testing.assert_close(glob_p, loc_p, rtol=0, atol=0)     # one rank: the global sums are the local ones
