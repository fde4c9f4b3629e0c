"""The one-launch narrow encoder stack (b200vae_mlp_stack_fwd / _bwd) against the per-layer fused kernels and against
stock nn.Modules + F.softplus: outputs, BatchNorm running statistics and num_batches_tracked, every gradient, graph
replay."""
import copy

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

# 160000 rows: the per-layer kernels' grid hits its 592-CTA cap; with an 8-wide layer the stack's co-resident grid is
# smaller there, so its statistics come from a different partition of the rows (same values up to reordered FP32 sums)
BATCHES = [1, 255, 256, 4097, 65536, 160000]


def _encoder(hidden, seed=0):
    from vae_song_b200 import model
    torch.manual_seed(seed)
    m = model.LIDVAE(dataset="pinwheel", icnn_channels=[32, 32], hidden_channels=hidden).cuda()
    with torch.no_grad():
        for mod in m.encoder.modules():
            if isinstance(mod, torch.nn.BatchNorm1d):
                mod.weight.uniform_(0.5, 1.5); mod.bias.uniform_(-0.5, 0.5)
                mod.running_mean.uniform_(-0.2, 0.2); mod.running_var.uniform_(0.5, 1.5)
    return m


def _per_layer(m, x, training):
    """The per-layer path (FusedMlpFn) with the softplus head in autograd."""
    from vae_song_b200 import ops
    plan = m._encoder_plan()
    out = ops.FusedMlpFn.apply(x, plan, training, *plan.params())
    mu, var = out.split(out.shape[1] // 2, 1)
    return mu, F.softplus(var)


def _run(enc, x, gmu, glv):
    xx = x.detach().clone().requires_grad_(True)
    mu, lv = enc(xx)
    (mu * gmu).sum().add((lv * glv).sum()).backward()
    return mu.detach(), lv.detach(), xx.grad


@pytest.mark.parametrize("B", BATCHES)
@pytest.mark.parametrize("training", [True, False], ids=["train", "eval"])
@pytest.mark.parametrize("hidden", [[2, 2, 2, 2], [8, 4, 2]], ids=["2-2-2-2", "8-4-2"])
def test_stack_matches_per_layer_kernels(B, training, hidden):
    from vae_song_b200 import ops
    a = _encoder(hidden).train(training)
    b = copy.deepcopy(a)
    plan = a._encoder_plan()
    assert ops._stack_ok(plan, training)
    gen = torch.Generator(device="cuda").manual_seed(B)
    x = torch.randn(B, 2, device="cuda", generator=gen)
    gmu = torch.randn(B, 2, device="cuda", generator=gen)
    glv = torch.randn(B, 2, device="cuda", generator=gen)
    from vae_song_b200 import _C
    n0 = _C.launch_count()
    mu, lv, dx = _run(a.encode, x, gmu, glv)
    assert _C.launch_count() - n0 == 2                       # one forward, one backward
    mu2, lv2, dx2 = _run(lambda t: _per_layer(b, t, training), x, gmu, glv)
    # same grid as the per-layer kernels: always for widths <= 4 (4 CTAs/SM co-resident), up to 148 SMs x 2 CTAs with an
    # 8-wide layer
    exact = not training or max(hidden) <= 4 or B <= 296 * 256
    tol = dict(rtol=0, atol=0) if exact else dict(rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(mu, mu2, **tol)
    torch.testing.assert_close(lv, lv2, **tol)
    for (k, p), q in zip(a.encoder.named_buffers(), b.encoder.buffers()):
        torch.testing.assert_close(p, q, **tol, msg=k)
    gscale = max(float(p.grad.abs().max()) for p in b.encoder.parameters())
    for (k, p), q in zip(a.encoder.named_parameters(), b.encoder.parameters()):
        # gradients: the backward sums (S1, S2) group the rows differently -> reordered FP32 sums only
        torch.testing.assert_close(p.grad, q.grad, rtol=1e-4, atol=1e-5 * gscale, msg=k)
    torch.testing.assert_close(dx, dx2, rtol=1e-4, atol=1e-5 * max(float(dx2.abs().max()), 1e-30))
    # biases that feed a BatchNorm: exactly zero
    for blk in a.encoder:
        assert float(blk[0].bias.grad.abs().max()) == 0.0


@pytest.mark.parametrize("training", [True, False], ids=["train", "eval"])
def test_stack_matches_stock_modules(training):
    """(mu, softplus(var)) and its backward, folded into the stack kernels, against nn.Sequential + F.softplus."""
    a = _encoder([2, 2, 2, 2], seed=3).train(training)
    ref = copy.deepcopy(a)
    ref.fused_encoder = False
    B = 4097
    gen = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randn(B, 2, device="cuda", generator=gen) * 3
    gmu, glv = torch.randn(B, 2, device="cuda", generator=gen), torch.randn(B, 2, device="cuda", generator=gen)
    mu, lv, dx = _run(a.encode, x, gmu, glv)
    mu2, lv2, dx2 = _run(ref.encode, x, gmu, glv)
    assert mu.is_contiguous() and lv.is_contiguous()
    torch.testing.assert_close(mu, mu2, rtol=2e-5, atol=2e-5)
    torch.testing.assert_close(lv, lv2, rtol=2e-5, atol=2e-5)
    gscale = max(float(p.grad.abs().max()) for p in ref.encoder.parameters())
    for (k, p), q in zip(a.encoder.named_parameters(), ref.encoder.parameters()):
        if k.endswith(".0.bias"):
            continue                                         # BN-fed bias: 0 here, rounding noise in the reference
        torch.testing.assert_close(p.grad, q.grad, rtol=2e-4, atol=1e-4 * gscale, msg=k)
    torch.testing.assert_close(dx, dx2, rtol=2e-4, atol=1e-4 * float(dx2.abs().max()))
    for (k, p), q in zip(a.encoder.named_buffers(), ref.encoder.buffers()):
        torch.testing.assert_close(p.float(), q.float(), rtol=1e-5, atol=1e-6, msg=k)


def test_stack_only_mu_used():
    """An unused output gets no gradient tensor from autograd: the kernel reads it as zero."""
    a = _encoder([2, 2, 2, 2]).train()
    b = copy.deepcopy(a)
    x = torch.randn(3000, 2, device="cuda")
    mu, _ = a.encode(x)
    mu.pow(2).sum().backward()
    mu2, _ = _per_layer(b, x, True)
    mu2.pow(2).sum().backward()
    for p, q in zip(a.encoder.parameters(), b.encoder.parameters()):
        torch.testing.assert_close(p.grad, q.grad, rtol=1e-4, atol=1e-6)


def test_stack_graph_replay_equals_eager():
    """Captured into a CUDA graph: every replay equals an eager call on the same inputs and state, bit for bit
    (the barrier counter and exit ticket are left zero by every launch)."""
    a = _encoder([2, 2, 2, 2]).train()
    b = copy.deepcopy(a)
    B = 65536
    x = torch.randn(B, 2, device="cuda")
    gmu, glv = torch.randn(B, 2, device="cuda"), torch.randn(B, 2, device="cuda")
    xs = x.clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):                                   # warm-up on the capture stream (scratch allocated there)
            a.zero_grad(set_to_none=True)
            mu, lv = a.encode(xs)
            ((mu * gmu).sum() + (lv * glv).sum()).backward()
    torch.cuda.current_stream().wait_stream(s)
    b.load_state_dict(a.state_dict())
    g = torch.cuda.CUDAGraph()
    a.zero_grad(set_to_none=False)
    with torch.cuda.graph(g):
        mu, lv = a.encode(xs)
        ((mu * gmu).sum() + (lv * glv).sum()).backward()
    for it in range(3):
        for p in a.encoder.parameters():
            p.grad.zero_()
        g.replay()
        torch.cuda.synchronize()
        b.zero_grad(set_to_none=True)
        mu2, lv2 = b.encode(x)
        ((mu2 * gmu).sum() + (lv2 * glv).sum()).backward()
        assert torch.equal(mu, mu2) and torch.equal(lv, lv2), it
        for p, q in zip(a.encoder.parameters(), b.encoder.parameters()):
            assert torch.equal(p.grad, q.grad), it
        for p, q in zip(a.encoder.buffers(), b.encoder.buffers()):
            assert torch.equal(p, q), it
