"""torch.autograd.Function wrappers over the C-ABI kernels (vae_song_b200/_C.py).

PyTorch is plumbing here: it owns device memory and the stream; every Function hands raw pointers to
libb200vae.so.  No CPU path -- tensors must be CUDA fp32.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _C
from ._C import PARAM_FIELDS


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _req(t: torch.Tensor, name: str):
    if not t.is_cuda:
        raise _C.B200VaeError(f"{name}: expected a CUDA tensor; vae_song_b200 has no CPU fallback")
    if t.dtype != torch.float32:
        raise _C.B200VaeError(f"{name}: expected float32, got {t.dtype}")
    return t.contiguous()


def _params_struct(params):
    s = _C.IcnnParams()
    for k, t in zip(PARAM_FIELDS, params):
        setattr(s, k, t.data_ptr())
    return s


# ------------------------------------------------------------------------------------------ ICNN
def icnn_prepare(params, d, H, mode, precision, B, for_backward):
    """params: 8 tensors in PARAM_FIELDS order -> workspace tensor (uint8) holding the positive weights."""
    lib = _C.load()
    params = [_req(p.detach(), k) for p, k in zip(params, PARAM_FIELDS)]
    nbytes = lib.b200vae_icnn_workspace_bytes(B, d, H, precision, 1 if for_backward else 0)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=params[0].device)
    ps = _params_struct(params)
    _C.check(lib.b200vae_icnn_prepare(C.byref(ps), d, H, mode, precision, _ptr(ws), nbytes, _stream()), "icnn_prepare")
    return ws


# ---- prepare ahead of use --------------------------------------------------------------------------------------------
# The prepared operands depend on the weights only, so a training step can build them while its encoder still runs: the
# chain of small prepare launches (~30 us per ICNN) leaves the critical path.  `icnn_prepare_early` forks a side stream from
# the current one (this also works inside a CUDA-graph capture: the side stream joins the capture and becomes a parallel
# branch of the graph), runs the prepare there and parks the workspace; IcnnBrenierFn.forward picks it up -- after making
# the current stream wait for the side stream -- if and only if it was built for exactly its configuration.
_EARLY = {}
_SIDE_STREAMS = {}


def _early_key(params, d, H, mode, precision, B, for_backward):
    return (tuple(p.data_ptr() for p in params), d, H, mode, precision, B, bool(for_backward),
            torch.cuda.current_stream().cuda_stream)


def icnn_prepare_early(params, d, H, mode, precision, B, for_backward, slot=0):
    lib = _C.load()
    params = [_req(p.detach(), k) for p, k in zip(params, PARAM_FIELDS)]
    dev = params[0].device
    main = torch.cuda.current_stream(dev)
    side = _SIDE_STREAMS.get((dev, slot))
    if side is None:
        side = _SIDE_STREAMS[(dev, slot)] = torch.cuda.Stream(dev)
    key = _early_key(params, d, H, mode, precision, B, for_backward)
    nbytes = lib.b200vae_icnn_workspace_bytes(B, d, H, precision, 1 if for_backward else 0)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)        # owned by the consuming stream's allocator pool
    ps = _params_struct(params)
    side.wait_stream(main)                                         # the weights this step reads are final on `main`
    with torch.cuda.stream(side):
        _C.check(lib.b200vae_icnn_prepare(C.byref(ps), d, H, mode, precision, _ptr(ws), nbytes, _stream()), "icnn_prepare")
    _EARLY[key] = (ws, side)


def _take_early(params, d, H, mode, precision, B, for_backward):
    if not _EARLY:
        return None
    ent = _EARLY.pop(_early_key(params, d, H, mode, precision, B, for_backward), None)
    if ent is None:
        return None
    ws, side = ent
    torch.cuda.current_stream(ws.device).wait_stream(side)
    return ws


def icnn_decode_fwd(z, ws, d, H, mode, kappa, precision, want_psi=True, want_xhat=True, save_masks=False):
    lib = _C.load()
    B = z.shape[0]
    Hp = (H + 127) // 128 * 128
    psi = torch.empty(B, dtype=torch.float32, device=z.device) if want_psi else None
    xhat = torch.empty(B, d, dtype=torch.float32, device=z.device) if want_xhat else None
    mask1 = torch.empty(B, Hp // 32, dtype=torch.int32, device=z.device) if save_masks else None
    mask2 = torch.empty(B, dtype=torch.uint8, device=z.device) if save_masks else None
    _C.check(lib.b200vae_icnn_decode_fwd(_ptr(z), B, d, H, mode, float(kappa), _ptr(psi), _ptr(xhat), _ptr(mask1),
                                         _ptr(mask2), precision, _ptr(ws), ws.numel(), _stream()), "icnn_decode_fwd")
    return psi, xhat, mask1, mask2


# ---- parameter gradients off the critical path ------------------------------------------------------------------------
# The backward of an ICNN has two halves: the rows part (dz, needed by whatever produced z -- the encoder) and the parameter
# gradients (the batch-reduced H x H weight gradient + finalize kernels, ~40 % of the time, needed only by the optimiser).
# Inside `deferred_param_grads()` the second half of every tensor-core backward is launched on a side stream, so that it
# overlaps the encoder's backward (a dozen small latency-bound kernels that leave the GPU mostly idle); leaving the context
# makes the current stream wait for it.  Only code that reads the gradients AFTER the context may use it -- the trainers of
# this package do (train.DataParallelTrainer.step); plain autograd users never see a gradient from another stream.
_DEFER = {"on": False, "stream": None, "keep": [], "seen": set(), "hint": True}


def set_defer_hint(ok):
    """Called by a module right before it applies IcnnBrenierFn: may THIS call's parameter gradients be deferred?  Deferring
    pays where the consumer of dz is light (the encoder); where dz feeds another ICNN's backward -- a kernel that wants the
    whole GPU -- the deferred kernels would only delay it (LIDVAE: second ICNN no, first ICNN yes)."""
    _DEFER["hint"] = bool(ok)


def _join_deferred(device=None):
    """Make the current stream wait for the deferred parameter-gradient work, hand the gradients to their parameters and
    release the tensors the side stream was reading."""
    if _DEFER["keep"]:
        torch.cuda.current_stream(device).wait_stream(_DEFER["stream"])
        for _, _, _, _, _, params, grads in _DEFER["keep"]:
            for p, g in zip(params, grads):
                if p.requires_grad:
                    p.grad = g if p.grad is None else p.grad + g
        _DEFER["keep"].clear()
    _DEFER["seen"].clear()


class deferred_param_grads:
    def __enter__(self):
        _DEFER["on"] = True
        return self

    def __exit__(self, *exc):
        _DEFER["on"] = False
        _join_deferred()
        return False


def icnn_decode_bwd(z, v, gpsi, mask1, mask2, params, ws, d, H, mode, kappa, precision, need_dz=True,
                    need_params=True, allow_defer=True):
    lib = _C.load()
    B = z.shape[0]
    dz = torch.empty_like(z) if need_dz else None
    grads = [torch.empty_like(p) for p in params] if need_params else None
    gs = _C.IcnnGrads()
    if grads is not None:
        for k, t in zip(PARAM_FIELDS, grads):
            setattr(gs, k, t.data_ptr())
    ps = _params_struct(params)
    defer = _DEFER["on"] and allow_defer and grads is not None and gpsi is None and v is not None and precision != _C.PREC_FP32
    if _DEFER["on"] and grads is not None and params[6].data_ptr() in _DEFER["seen"]:
        # the same ICNN a second time in one backward: autograd will ADD the two gradients on this stream right away, so the
        # first one must be complete -- join, then run this call in one piece
        _join_deferred(z.device)
    elif defer:
        # rows part here (grads = NULL), parameter part on the side stream, ordered after it
        _C.check(lib.b200vae_icnn_decode_bwd(_ptr(z), _ptr(v), None, _ptr(mask1), _ptr(mask2), B, d, H, C.byref(ps), mode,
                                             float(kappa), None, _ptr(dz), precision, _ptr(ws), ws.numel(), _stream()),
                 "icnn_decode_bwd")
        main = torch.cuda.current_stream(z.device)
        if _DEFER["stream"] is None or _DEFER["stream"].device != z.device:
            _DEFER["stream"] = torch.cuda.Stream(z.device)
        side = _DEFER["stream"]
        side.wait_stream(main)
        with torch.cuda.stream(side):
            _C.check(lib.b200vae_icnn_decode_bwd_params(_ptr(z), _ptr(v), _ptr(mask1), _ptr(mask2), B, d, H, C.byref(ps), mode,
                                                        C.byref(gs), precision, _ptr(ws), ws.numel(), _stream()),
                     "icnn_decode_bwd_params")
        # What the side stream reads must not be recycled by the allocator before the join (autograd frees the saved tensors
        # as soon as this node has run).  The gradients do NOT travel through autograd (None is returned for them): it would
        # accumulate -- or, if anybody else holds a reference, clone -- them on THIS stream at once, before the side stream
        # has written them; the join assigns them to `.grad` instead (`params` are the leaf tensors themselves).
        _DEFER["keep"].append((z, v, mask1, mask2, ws, params, grads))
        _DEFER["seen"].add(params[6].data_ptr())
        return dz, None
    _C.check(lib.b200vae_icnn_decode_bwd(_ptr(z), _ptr(v), _ptr(gpsi), _ptr(mask1), _ptr(mask2), B, d, H, C.byref(ps),
                                         mode, float(kappa), C.byref(gs) if grads is not None else None, _ptr(dz),
                                         precision, _ptr(ws), ws.numel(), _stream()), "icnn_decode_bwd")
    return dz, grads


_weights_epoch = [0]


def bump_weights_epoch():
    """Called by everything in this package that changes parameters behind autograd's back (the fused Adam kernels write
    through raw pointers, a CUDA-graph replay of a train step runs no Python at all): invalidates every cached
    inference workspace.  Call it yourself after replaying your OWN graph that contains b200vae_adam_* launches."""
    _weights_epoch[0] += 1


def _param_state(params):
    """Identity + in-place version of every parameter tensor (torch optimisers, copy_, load_state_dict, the re-homing of
    train.FlatParams all change one of them) + this package's own weights epoch."""
    return (_weights_epoch[0],) + tuple((p.data_ptr(), p._version, tuple(p.shape)) for p in params)


def _cached_ws(z, mode, precision, params, cache, name="z"):
    """(z, H, d, prepared inference workspace) -- the workspace kept in `cache` and rebuilt only when its key changes."""
    z = _req(z.detach(), name)
    params = [_req(p.detach(), k) for p, k in zip(params, PARAM_FIELDS)]
    H, d = params[0].shape
    if z.dim() != 2 or z.shape[1] != d:
        raise _C.B200VaeError(f"{name} must be [B,{d}], got {tuple(z.shape)}")
    key = (z.shape[0], mode, precision, z.device, torch.cuda.current_stream().cuda_stream, _param_state(params))
    if cache.get("key") != key:
        cache["ws"] = icnn_prepare(params, d, H, mode, precision, z.shape[0], False)
        cache["key"] = key
    return z, H, d, cache["ws"]


def icnn_brenier_inference(z, kappa, mode, precision, params, cache):
    """(psi, xhat) without an autograd graph -- evaluation loops (utils.estimate_local_lipschitz*, lipschitz.py's per-cell
    sweeps, decode under no_grad).  The prepared workspace (positive weights in every kernel layout: 4 launches) is kept in
    `cache` (a dict owned by the module) and reused while the parameters are unchanged (their `_version` counters and data
    pointers), the batch size and the precision are the same; module.py:110 re-materialises exp(W) on every call instead."""
    z, H, d, ws = _cached_ws(z, mode, precision, params, cache)
    psi, xhat, _, _ = icnn_decode_fwd(z, ws, d, H, mode, kappa, precision, True, True, False)
    return psi, xhat


# ---- exact Jacobians (b200vae_icnn_decode_jac, b200vae_jacobian_chain) ------------------------------------------------
# With the LeakyReLU masks fixed the Brenier map is affine in z, so its Jacobian A0^T diag(2 s0^2 gx1) A0 + 2 kappa I comes out
# of the same fused forward.  These functions return plain tensors: the Jacobian is NOT differentiable (no autograd graph;
# a Jacobian penalty in training would need its own backward).
def icnn_decode_jac(z, ws, d, H, kappa, precision, save_masks=False):
    """(psi [B], xhat [B,d], jac [B,d,d], mask1 | None, mask2 | None) on a prepared workspace `ws`."""
    lib = _C.load()
    B, dev = z.shape[0], z.device
    Hp = (H + 127) // 128 * 128
    psi = torch.empty(B, dtype=torch.float32, device=dev)
    xhat = torch.empty(B, d, dtype=torch.float32, device=dev)
    jac = torch.empty(B, d, d, dtype=torch.float32, device=dev)
    mask1 = torch.empty(B, Hp // 32, dtype=torch.int32, device=dev) if save_masks else None
    mask2 = torch.empty(B, dtype=torch.uint8, device=dev) if save_masks else None
    nscr = lib.b200vae_icnn_jac_scratch_bytes(B, d, H, precision)
    scr = torch.empty(nscr, dtype=torch.uint8, device=dev) if nscr else None
    _C.check(lib.b200vae_icnn_decode_jac(_ptr(z), B, d, H, float(kappa), _ptr(psi), _ptr(xhat), _ptr(jac), _ptr(mask1),
                                         _ptr(mask2), precision, _ptr(ws), ws.numel(), _ptr(scr), nscr, _stream()),
             "icnn_decode_jac")
    return psi, xhat, jac, mask1, mask2


def icnn_brenier_jacobian(z, kappa, mode, precision, params, cache):
    """(psi [B], xhat [B,d], jac [B,d,d] = d xhat / d z) without an autograd graph; the prepared workspace is shared with
    icnn_brenier_inference through `cache` (same key).  jac is not differentiable."""
    z, H, d, ws = _cached_ws(z, mode, precision, params, cache)
    psi, xhat, jac, _, _ = icnn_decode_jac(z, ws, d, H, kappa, precision)
    return psi, xhat, jac


# ---- left inverse (b200vae_brenier_inverse_init, b200vae_brenier_newton_step) -----------------------------------------
# z = T^{-1}(x) for T = grad(psi + kappa|.|^2): Newton steps on f(z) = psi(z) + kappa|z|^2 - <x, z>, whose gradient and
# Hessian come from the Jacobian forward.  One round = one b200vae_icnn_decode_jac at every row's trial point + one step
# kernel (csrc/inverse.cu).  Plain tensors, not differentiable.
INVERSE_TOL = {_C.PREC_FP32: 1e-5, _C.PREC_TF32: 5e-3, _C.PREC_TF32X3: 1e-5, _C.PREC_F16X3: 1e-5}   # declared xhat accuracy
INVERSE_MAX_ITER = 100
INVERSE_CHECK_EVERY = 4


def icnn_brenier_inverse(x, kappa, mode, precision, params, cache, z0=None, max_iter=INVERSE_MAX_ITER, tol=None):
    """(z [B,d], status [B] int32 (_C.INV_*), err_bound [B], rounds): z ~ T^{-1}(x) with ||z - T^{-1}(x)|| <= err_bound
    (= ||xhat(z) - x|| / (2 kappa), +inf at kappa = 0).  A row converges when ||xhat(z) - x|| <= tol (||x|| + 1); tol
    defaults to the precision's declared xhat accuracy.  z0 [B,d] warm-starts (default 0).  The prepared workspace is the
    one of icnn_brenier_inference / icnn_brenier_jacobian (same `cache`, same key).  Eager: stops once every row has
    finished, reading the device's count of active rows (4 bytes) every INVERSE_CHECK_EVERY rounds; while a CUDA graph is
    being captured: exactly max_iter rounds.  Rows still active after the last round are MAXITER."""
    lib = _C.load()
    x, H, d, ws = _cached_ws(x, mode, precision, params, cache, "x")
    B, dev = x.shape[0], x.device
    if max_iter < 1:
        raise _C.B200VaeError(f"max_iter must be >= 1, got {max_iter}")
    if z0 is not None:
        z0 = _req(z0.detach(), "z0")
        if z0.shape != x.shape:
            raise _C.B200VaeError(f"z0 must be {tuple(x.shape)}, got {tuple(z0.shape)}")
    tol = INVERSE_TOL[precision] if tol is None else float(tol)
    nst = lib.b200vae_brenier_inverse_state_bytes(B, d)
    state = torch.empty(nst, dtype=torch.uint8, device=dev)
    trial = torch.empty(B, d, dtype=torch.float32, device=dev)
    z = torch.empty(B, d, dtype=torch.float32, device=dev)
    status = torch.empty(B, dtype=torch.int32, device=dev)
    err = torch.empty(B, dtype=torch.float32, device=dev)
    psi = torch.empty(B, dtype=torch.float32, device=dev)
    xhat = torch.empty(B, d, dtype=torch.float32, device=dev)
    jac = torch.empty(B, d, d, dtype=torch.float32, device=dev)
    nscr = lib.b200vae_icnn_jac_scratch_bytes(B, d, H, precision)
    scr = torch.empty(nscr, dtype=torch.uint8, device=dev) if nscr else None
    active = state[:8].view(torch.int32)
    st = _stream()
    _C.check(lib.b200vae_brenier_inverse_init(_ptr(x), _ptr(z0), B, d, tol, tol, _ptr(state), nst, _ptr(trial), _ptr(z),
                                              _ptr(status), _ptr(err), st), "brenier_inverse_init")
    capturing = torch.cuda.is_current_stream_capturing()
    rounds = max_iter
    for k in range(max_iter):
        _C.check(lib.b200vae_icnn_decode_jac(_ptr(trial), B, d, H, float(kappa), _ptr(psi), _ptr(xhat), _ptr(jac), None,
                                             None, precision, _ptr(ws), ws.numel(), _ptr(scr), nscr, st), "icnn_decode_jac")
        _C.check(lib.b200vae_brenier_newton_step(_ptr(x), _ptr(xhat), _ptr(jac), B, d, float(kappa), k,
                                                 1 if k == max_iter - 1 else 0, _ptr(state), nst, _ptr(trial), _ptr(z),
                                                 _ptr(status), _ptr(err), st), "brenier_newton_step")
        if not capturing and (k + 1) % INVERSE_CHECK_EVERY == 0 and k + 1 < max_iter and int(active[k & 1]) == 0:
            rounds = k + 1
            break
    return z, status, err, rounds


def jacobian_chain(J2, M, J1, want_J=True, want_svals=True):
    """J = J2 . M . J1 [B,Dx,D] and its singular values [B,min(Dx,D)] (descending), one kernel, fp64 inside; either output
    may be skipped (None returned).  J2 [B,Dx,Dx], M [Dx,D], J1 [B,D,D]; Dx, D <= 4.  Not differentiable."""
    lib = _C.load()
    J2, M, J1 = (_req(t.detach(), n) for t, n in ((J2, "J2"), (M, "M"), (J1, "J1")))
    B, Dx, D = J2.shape[0], M.shape[0], M.shape[1]
    if J2.shape != (B, Dx, Dx) or J1.shape != (B, D, D):
        raise _C.B200VaeError(f"jacobian_chain: shapes J2 {tuple(J2.shape)}, M {tuple(M.shape)}, J1 {tuple(J1.shape)} "
                              "do not chain")
    J = torch.empty(B, Dx, D, dtype=torch.float32, device=J1.device) if want_J else None
    s = torch.empty(B, min(Dx, D), dtype=torch.float32, device=J1.device) if want_svals else None
    if B == 0:
        return J, s
    _C.check(lib.b200vae_jacobian_chain(_ptr(J2), _ptr(M), _ptr(J1), B, Dx, D, _ptr(J), _ptr(s), _stream()),
             "jacobian_chain")
    return J, s


class IcnnBrenierFn(torch.autograd.Function):
    """(psi [B], xhat [B,d]) = fused ICNN potential + Brenier map.  Replaces module.py:142-148 followed
    by model.py:820-822.  backward = the double-backward PyTorch would run through autograd.grad."""

    @staticmethod
    def forward(ctx, z, kappa, mode, precision, *params):
        z = _req(z, "z")
        params = [_req(p, k) for p, k in zip(params, PARAM_FIELDS)]
        H, d = params[0].shape
        if z.dim() != 2 or z.shape[1] != d:
            raise _C.B200VaeError(f"z must be [B,{d}], got {tuple(z.shape)}")
        needs_bwd = any(ctx.needs_input_grad)
        ws = _take_early(params, d, H, mode, precision, z.shape[0], needs_bwd)
        if ws is None:
            ws = icnn_prepare(params, d, H, mode, precision, z.shape[0], needs_bwd)
        psi, xhat, m1, m2 = icnn_decode_fwd(z, ws, d, H, mode, kappa, precision, True, True, needs_bwd)
        if needs_bwd:
            ctx.save_for_backward(z, m1, m2, ws, *params)
            ctx.cfg = (d, H, mode, float(kappa), precision)
            ctx.defer_ok, _DEFER["hint"] = _DEFER["hint"], True
        ctx.set_materialize_grads(False)
        return psi, xhat

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gpsi, gxhat):
        z, m1, m2, ws, *params = ctx.saved_tensors
        d, H, mode, kappa, precision = ctx.cfg
        if gpsi is None and gxhat is None:
            return (None,) * (4 + len(params))
        v = None if gxhat is None else _req(gxhat, "grad_xhat")
        gp = None if gpsi is None else _req(gpsi, "grad_psi")
        need_params = any(ctx.needs_input_grad[4:])
        dz, grads = icnn_decode_bwd(z, v, gp, m1, m2, params, ws, d, H, mode, kappa, precision,
                                    need_dz=ctx.needs_input_grad[0], need_params=need_params, allow_defer=ctx.defer_ok)
        if grads is None:
            grads = [None] * len(params)
        return (dz, None, None, None, *grads)


class _FirstOrderOnly(torch.autograd.Function):
    """Identity on `t` that ties it to `anchor`'s graph and fails loudly if anyone differentiates THROUGH it: the parameter
    gradients of psi are produced by kernels without a graph, so a create_graph=True caller who went on to differentiate
    them would otherwise silently get zeros."""

    @staticmethod
    def forward(ctx, t, anchor, what):
        ctx.what = what
        return t.view_as(t)

    @staticmethod
    def backward(ctx, g):
        raise _C.B200VaeError(f"second-order derivatives through {ctx.what} are not implemented (the fused kernels "
                              "differentiate psi twice in z -- the Brenier-map path -- not its parameter gradients)")


def _guard_param_grads(pgrads, anchor):
    if not (torch.is_grad_enabled() and anchor.requires_grad):
        return pgrads
    return [None if g is None else _FirstOrderOnly.apply(g, anchor, "the parameter gradients of psi") for g in pgrads]


class IcnnPotentialFn(torch.autograd.Function):
    """psi = ICNN(z) [B,1] exactly as module.ICNN.forward returns it, and -- like the reference -- it stays
    differentiable TWICE in z: backward computes grad_z = gpsi * xhat through IcnnBrenierFn (itself a
    Function with a backward), so `torch.autograd.grad(psi, [z], ones, create_graph=True)` followed by
    `.backward()` (model.py:822, lipschitz.py:41) works on this module unchanged."""

    @staticmethod
    def forward(ctx, z, mode, precision, *params):
        z = _req(z, "z")
        params = [_req(p, k) for p, k in zip(params, PARAM_FIELDS)]
        H, d = params[0].shape
        ws = icnn_prepare(params, d, H, mode, precision, z.shape[0], False)
        psi, _, _, _ = icnn_decode_fwd(z, ws, d, H, mode, 0.0, precision, True, False, False)
        ctx.save_for_backward(z, *params)
        ctx.cfg = (mode, precision)
        return psi.unsqueeze(1)

    @staticmethod
    def backward(ctx, gpsi):
        z, *params = ctx.saved_tensors
        mode, precision = ctx.cfg
        need_z = ctx.needs_input_grad[0]
        need_p = any(ctx.needs_input_grad[3:])
        g = gpsi[:, 0]
        dz, pgrads = None, [None] * len(params)
        if need_z:
            # differentiable in (z, params, gpsi) when create_graph=True: the Brenier map is a Function too
            _, xhat = IcnnBrenierFn.apply(z, 0.0, mode, precision, *params)
            dz = g.unsqueeze(1) * xhat
        if need_p:
            with torch.no_grad():
                H, d = params[0].shape
                zz = z.detach()
                ws = icnn_prepare(params, d, H, mode, precision, zz.shape[0], True)
                _, _, m1, m2 = icnn_decode_fwd(zz, ws, d, H, mode, 0.0, precision, False, False, True)
                _, grads = icnn_decode_bwd(zz, None, _req(g.detach(), "grad_psi"), m1, m2, [p.detach() for p in params],
                                           ws, d, H, mode, 0.0, precision, need_dz=False, need_params=True)
            pgrads = _guard_param_grads([gr if need else None for gr, need in zip(grads, ctx.needs_input_grad[3:])], gpsi)
        return (dz, None, None, *pgrads)


# ------------------------------------------------------------------------------------------ wide-input ICNN
def _grads_struct(tensors):
    g = _C.IcnnGrads()
    for k, t in zip(PARAM_FIELDS, tensors):
        setattr(g, k, None if t is None else t.data_ptr())
    return g


def icnn_wide_fwd(z, params, mode, kappa, want_xhat=True, precision=0):
    """Fused forward of a wide-input ICNN (b200vae_icnn_wide_fwd; an unknown precision id raises B200VaeError).  Returns (psi [B], xhat [B,d] | None, saved) with
    saved = (h0 [B,H], mask1 [B,H] uint8, s2 [B]) -- what the backward needs besides z."""
    lib = _C.load()
    B, nz = z.shape
    H, d = params[0].shape
    dev = z.device
    ws = torch.empty(lib.b200vae_icnn_wide_workspace_bytes(B, d, H, precision, 0), dtype=torch.uint8, device=dev)
    psi = torch.empty(B, dtype=torch.float32, device=dev)
    h0 = torch.empty(B, H, dtype=torch.float32, device=dev)
    mask1 = torch.empty(B, H, dtype=torch.uint8, device=dev)
    s2 = torch.empty(B, dtype=torch.float32, device=dev)
    xhat = torch.empty(B, d, dtype=torch.float32, device=dev) if want_xhat else None
    g0 = torch.empty(B, H, dtype=torch.float32, device=dev) if want_xhat else None
    ps = _params_struct(params)
    _C.check(lib.b200vae_icnn_wide_fwd(_ptr(z), B, d, nz, H, C.byref(ps), mode, float(kappa), _ptr(psi), _ptr(xhat), _ptr(h0),
                                       _ptr(mask1), _ptr(s2), _ptr(g0), precision, _ptr(ws), ws.numel(), _stream()),
             "icnn_wide_fwd")
    return psi, xhat, (h0, mask1, s2)


class IcnnBrenierWideFn(torch.autograd.Function):
    """Same contract as IcnnBrenierFn for input widths the register-resident kernels do not cover (d > 4, e.g. the
    MNIST-shaped ICNN(32,512) / ICNN(784,1024) of BASELINE configs[3]).  Here the thin products A.z are dense
    [B,d]x[d,H] contractions as well; the path is a chain of fused FP32 tile-GEMM kernels with generated operands and
    elementwise epilogues (csrc/icnn_wide.cu): the ANALYTIC forward-then-reverse sweep and double-backward of SURVEY
    Appendix A, no autograd graph, h0 + a byte mask saved instead of ~20 activations.  `precision`: fp32 = those kernels;
    tf32 / tf32x3 (f16x3 runs as tf32x3) = the forward and every GEMM of the dL/dxhat backward, batch reductions included,
    on tcgen05 (csrc/icnn_wide_tc.cu) when d, nz and H are multiples of 4 -- else, and for a forward whose b0 / b1 / A2
    are not 16-byte aligned, the FP32 kernels; the psi-gradient term always runs on the FP32 kernels.  z may be NARROWER than the ICNN input ([B,nz], nz <= d): it is then
    taken as zero-padded to d columns -- the eye(Dx,D) pad of model.py:824 fused away -- and dz is [B,nz]."""

    @staticmethod
    def forward(ctx, z, kappa, mode, precision, *params):
        z = _req(z, "z")
        params = [_req(p, k) for p, k in zip(params, PARAM_FIELDS)]
        H, d = params[0].shape
        if z.dim() != 2 or not (1 <= z.shape[1] <= d):
            raise _C.B200VaeError(f"z must be [B,nz] with nz <= {d}, got {tuple(z.shape)}")
        psi, xhat, saved = icnn_wide_fwd(z, params, mode, kappa, True, precision)
        if any(ctx.needs_input_grad):
            ctx.save_for_backward(z, *saved, *params)
            ctx.cfg = (float(kappa), mode, precision)
        ctx.set_materialize_grads(False)
        return psi, xhat

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gpsi, v):
        z, h0, mask1, s2, *params = ctx.saved_tensors
        kappa, mode, precision = ctx.cfg
        if gpsi is None and v is None:
            return (None,) * 12
        need = ctx.needs_input_grad
        dz, grads = None, [None] * len(params)
        if v is not None:                          # double-backward of the Brenier map (dL/dxhat)
            dz, grads = icnn_wide_bwd(z, _req(v, "grad_xhat"), h0, mask1, s2, params, mode, kappa, precision, need[0], need[4:])
        if gpsi is not None:                       # first-order backward of psi (Appendix A, last line), FP32 tile kernels
            dz2, g2 = icnn_wide_bwd_psi(z, _req(gpsi, "grad_psi"), h0, mask1, s2, params, mode, need[0], need[4:])
            dz = dz2 if dz is None else (dz + dz2 if dz2 is not None else dz)
            grads = [b if a is None else (a + b if b is not None else a) for a, b in zip(grads, g2)]
        return (dz, None, None, None, *grads)


def icnn_wide_bwd(z, v, h0, mask1, s2, params, mode, kappa, precision, need_dz=True, need_params=None):
    """dL/dz and parameter gradients of L = <v, xhat> for the wide-input ICNN (b200vae_icnn_wide_bwd)."""
    lib = _C.load()
    B, nz = z.shape
    H, d = params[0].shape
    dev = z.device
    need_params = [True] * len(params) if need_params is None else list(need_params)
    ws = torch.empty(lib.b200vae_icnn_wide_workspace_bytes(B, d, H, precision, 1), dtype=torch.uint8, device=dev)
    scratch = torch.empty(4, B, H, dtype=torch.float32, device=dev)          # u0, q1, g0, t0
    grads = [torch.empty_like(p) if n else None for p, n in zip(params, need_params)]
    dz = torch.empty_like(z) if need_dz else None
    ps, gs = _params_struct(params), _grads_struct(grads)
    _C.check(lib.b200vae_icnn_wide_bwd(_ptr(z), _ptr(v), _ptr(h0), _ptr(mask1), _ptr(s2), B, d, nz, H, C.byref(ps), mode,
                                       float(kappa), C.byref(gs), _ptr(dz), _ptr(scratch[0]), _ptr(scratch[1]),
                                       _ptr(scratch[2]), _ptr(scratch[3]), precision, _ptr(ws), ws.numel(), _stream()),
             "icnn_wide_bwd")
    return dz, grads


def icnn_wide_bwd_psi(z, gpsi, h0, mask1, s2, params, mode, need_dz=True, need_params=None):
    """dL/dz and parameter gradients of L = <gpsi, psi> for the wide-input ICNN (b200vae_icnn_wide_bwd_psi)."""
    lib = _C.load()
    B, nz = z.shape
    H, d = params[0].shape
    dev = z.device
    need_params = [True] * len(params) if need_params is None else list(need_params)
    ws = torch.empty(lib.b200vae_icnn_wide_workspace_bytes(B, d, H, _C.PREC_FP32, 1), dtype=torch.uint8, device=dev)
    scratch = torch.empty(2, B, H, dtype=torch.float32, device=dev)          # x1, gpsi*g0
    s2g = torch.empty(B, dtype=torch.float32, device=dev)
    grads = [torch.empty_like(p) if n else None for p, n in zip(params, need_params)]
    dz = torch.empty_like(z) if need_dz else None
    ps, gs = _params_struct(params), _grads_struct(grads)
    _C.check(lib.b200vae_icnn_wide_bwd_psi(_ptr(z), _ptr(gpsi), _ptr(h0), _ptr(mask1), _ptr(s2), B, d, nz, H, C.byref(ps), mode,
                                           C.byref(gs), _ptr(dz), _ptr(scratch[0]), _ptr(scratch[1]), _ptr(s2g), _ptr(ws),
                                           ws.numel(), _stream()), "icnn_wide_bwd_psi")
    return dz, grads


class IcnnPotentialWideFn(torch.autograd.Function):
    """psi = ICNN(z) [B,1] for wide inputs (d > 4), exactly as module.ICNN.forward returns it and -- like the reference and
    like IcnnPotentialFn for d <= 4 -- differentiable TWICE in z: backward computes grad_z = gpsi * xhat through
    IcnnBrenierWideFn (a Function with its own analytic backward), and the parameter gradients of <gpsi, psi> with the
    fused first-order backward.  Replaces module.py:142-148 for ICNN(32,.) / ICNN(784,.)."""

    @staticmethod
    def forward(ctx, z, mode, precision, *params):
        z = _req(z, "z")
        params = [_req(p, k) for p, k in zip(params, PARAM_FIELDS)]
        psi, _, saved = icnn_wide_fwd(z, params, mode, 0.0, False, precision)
        ctx.save_for_backward(z, *saved, *params)
        ctx.cfg = (mode, precision)
        return psi.unsqueeze(1)

    @staticmethod
    def backward(ctx, gpsi):
        z, h0, mask1, s2, *params = ctx.saved_tensors
        mode, precision = ctx.cfg
        need_z, need_p = ctx.needs_input_grad[0], ctx.needs_input_grad[3:]
        g = gpsi[:, 0]
        dz, pgrads = None, [None] * len(params)
        if need_z:
            # differentiable in (z, params, gpsi) when create_graph=True: the Brenier map is a Function too
            _, xhat = IcnnBrenierWideFn.apply(z, 0.0, mode, precision, *params)
            dz = g.unsqueeze(1) * xhat
        if any(need_p):
            with torch.no_grad():
                _, pgrads = icnn_wide_bwd_psi(z.detach(), _req(g.detach(), "grad_psi"), h0, mask1, s2,
                                              [p.detach() for p in params], mode, False, need_p)
            pgrads = _guard_param_grads(pgrads, gpsi)
        return (dz, None, None, *pgrads)


# ------------------------------------------------------------------------------------------ losses
_loss_scratch = {}


def _loss_out(device):
    """Zero-initialised reduction scratch (+ results) per (device, stream); the kernel leaves it zeroed."""
    key = (device, torch.cuda.current_stream().cuda_stream)
    buf = _loss_scratch.get(key)
    if buf is None:
        buf = torch.zeros(_C.LOSS_OUT_FLOATS, dtype=torch.float32, device=device)
        _loss_scratch[key] = buf
    return buf


class ReparamFn(torch.autograd.Function):
    """z[l] = mu + eps[l] * exp(0.5*lv).  eps [B,D] or [L,B,D] (model.py:843 / :423-424)."""

    @staticmethod
    def forward(ctx, mu, lv, eps):
        mu, lv, eps = _req(mu, "mu"), _req(lv, "log_var"), _req(eps, "eps")
        B, D = mu.shape
        L = 1 if eps.dim() == 2 else eps.shape[0]
        z = torch.empty_like(eps)
        out = _loss_out(mu.device)
        _C.check(_C.load().b200vae_loss_fwd(_ptr(mu), _ptr(lv), _ptr(eps), _ptr(z), L, B, D, None, None, 0, 0, None,
                                            None, None, 0, 0, 0, _ptr(out), _stream()), "reparam_fwd")
        ctx.save_for_backward(mu, lv, eps)
        return z

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gz):
        mu, lv, eps = ctx.saved_tensors
        B, D = mu.shape
        L = 1 if eps.dim() == 2 else eps.shape[0]
        gz = _req(gz, "grad_z")
        d_mu, d_lv = torch.empty_like(mu), torch.empty_like(lv)
        _C.check(_C.load().b200vae_loss_bwd(_ptr(mu), _ptr(lv), _ptr(eps), _ptr(gz), L, B, D, None, None, 0, 0, None,
                                            None, None, 0, 0, 0, None, None, None, _ptr(d_mu), _ptr(d_lv), None, None,
                                            _stream()), "reparam_bwd")
        return d_mu, d_lv, None


class VaeLossFn(torch.autograd.Function):
    """(recon, kl, latent) scalars in one launch.  x/xhat [B,...]; mu/lv [B,D]; z_in/z_rec [L,B,D] or None."""

    @staticmethod
    def forward(ctx, x, xhat, mu, lv, z_in, z_rec, logmse):
        dev = (xhat if xhat is not None else mu).device
        x_ = None if x is None else _req(x, "x")
        xh = None if xhat is None else _req(xhat, "xhat")
        mu_ = None if mu is None else _req(mu, "mu")
        lv_ = None if lv is None else _req(lv, "log_var")
        zi = None if z_in is None else _req(z_in, "z_in")
        zr = None if z_rec is None else _req(z_rec, "z_rec")
        B = (xh if xh is not None else mu_).shape[0]
        Dx = 0 if xh is None else xh.numel() // B
        D = 0 if mu_ is None else mu_.shape[1]
        Lz = Bz = Dz = 0
        if zi is not None:
            if zi.shape != zr.shape:
                raise _C.B200VaeError("z_in / z_rec shape mismatch")
            Lz = zi.shape[0]
            Bz = zi.shape[1] if zi.dim() > 1 else 1
            Dz = zi.numel() // (Lz * Bz)
        mse_rows = torch.empty(B, dtype=torch.float32, device=dev) if (logmse and xh is not None) else None
        out = _loss_out(dev)
        _C.check(_C.load().b200vae_loss_fwd(_ptr(mu_), _ptr(lv_), None, None, 0, B, D, _ptr(x_), _ptr(xh), Dx,
                                            1 if logmse else 0, _ptr(mse_rows), _ptr(zi), _ptr(zr), Lz, Bz, Dz,
                                            _ptr(out), _stream()), "loss_fwd")
        res = out[:3].clone()
        ctx.save_for_backward(x_, xh, mu_, lv_, zi, zr, mse_rows)
        ctx.dims = (B, D, Dx, Lz, Bz, Dz, bool(logmse))
        ctx.set_materialize_grads(False)
        return res[0], res[1], res[2]

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g_rec, g_kl, g_lat):
        x_, xh, mu_, lv_, zi, zr, mse_rows = ctx.saved_tensors
        B, D, Dx, Lz, Bz, Dz, logmse = ctx.dims
        need_xh = ctx.needs_input_grad[1] and xh is not None and g_rec is not None
        need_ml = (ctx.needs_input_grad[2] or ctx.needs_input_grad[3]) and mu_ is not None and g_kl is not None
        need_zr = ctx.needs_input_grad[5] and zr is not None and g_lat is not None
        d_xh = torch.empty_like(xh) if need_xh else None
        d_mu = torch.empty_like(mu_) if need_ml else None
        d_lv = torch.empty_like(lv_) if need_ml else None
        d_zr = torch.empty_like(zr) if need_zr else None
        if need_xh or need_ml or need_zr:
            f = lambda g: None if g is None else _req(g.reshape(1), "grad")
            gr, gk, gl = f(g_rec), f(g_kl), f(g_lat)
            _C.check(_C.load().b200vae_loss_bwd(_ptr(mu_), _ptr(lv_), None, None, 0, B, D, _ptr(x_), _ptr(xh), Dx,
                                                1 if logmse else 0, _ptr(mse_rows), _ptr(zi), _ptr(zr), Lz, Bz, Dz,
                                                _ptr(gr), _ptr(gk), _ptr(gl), _ptr(d_mu), _ptr(d_lv), _ptr(d_xh),
                                                _ptr(d_zr), _stream()), "loss_bwd")
        d_zi = None
        if ctx.needs_input_grad[4] and d_zr is not None:
            d_zi = -d_zr
        d_x = None
        if ctx.needs_input_grad[0] and d_xh is not None:
            d_x = -d_xh
        return d_x, d_xh, d_mu, d_lv, d_zi, d_zr, None


# ------------------------------------------------------------------------------------------ fused MLP encoder
def _flat_params(Ws, bs, gs, bes):
    """The parameter order of FusedMlpFn / FusedMlpStackFn: (W, b) of every Linear, then (gamma, beta) of every BN."""
    out = []
    for W, b in zip(Ws, bs):
        out += [W, b]
    for g, be in zip(gs, bes):
        out += [g, be]
    return out


class MlpPlan:
    """Structure of a [Linear -> BatchNorm1d -> LeakyReLU] x n (+ trailing Linear) stack, extracted from stock
    nn.Modules (which keep owning the parameters / buffers, so state_dict keys do not change).  `source` holds the
    identities of the leaf modules it was read from; `identity_tail`: the trailing Linear is an appended identity."""

    def __init__(self, linears, bns, slope, source=(), identity_tail=False):
        self.linears, self.bns, self.slope = linears, bns, slope       # len(bns) == len(linears) - 1
        self.source, self.identity_tail = source, identity_tail

    def params(self):
        return _flat_params([l.weight for l in self.linears], [l.bias for l in self.linears],
                            [b.weight for b in self.bns], [b.bias for b in self.bns])


def _leaf_modules(mod):
    nn = torch.nn
    if isinstance(mod, nn.Sequential):
        out = []
        for c in mod:
            out += _leaf_modules(c)
        return out
    return [mod]


def mlp_plan_from_modules(seq):
    """MlpPlan for ANY nesting of Sequentials whose leaves read (Linear, BatchNorm1d, LeakyReLU)+ [Linear] -- the 1-D MLP
    stacks of FlexibleVAE (model.py:186-208, 360-374: the encoder ENDS in BN + LeakyReLU, the decoder in a bare Linear) as
    well as LIDVAE's encoder (model.py:711-734).  A stack without the trailing Linear gets a frozen identity layer appended (not registered
    anywhere: act(BN(y)) . I + 0 is exact), so that the last BatchNorm + activation is applied by the same layer kernels.
    Returns None when the modules do not match; `plan.source` holds the leaf identities for staleness checks."""
    nn = torch.nn
    leaves = _leaf_modules(seq)
    mods = [m for m in leaves if not isinstance(m, nn.Flatten)]
    lin, bns, slopes, i = [], [], [], 0
    while i + 2 < len(mods) + 0 and isinstance(mods[i], nn.Linear) and isinstance(mods[i + 1], nn.BatchNorm1d) \
            and isinstance(mods[i + 2], nn.LeakyReLU):
        lin.append(mods[i]); bns.append(mods[i + 1]); slopes.append(mods[i + 2].negative_slope)
        i += 3
    rest = mods[i:]
    if not lin or len(rest) > 1 or (rest and not isinstance(rest[0], nn.Linear)):
        return None
    identity = not rest
    if identity:
        w = lin[-1].out_features
        tail = nn.Linear(w, w).to(lin[-1].weight.device)
        with torch.no_grad():
            tail.weight.copy_(torch.eye(w)); tail.bias.zero_()
        tail.weight.requires_grad_(False); tail.bias.requires_grad_(False)
        lin.append(tail)
    else:
        lin.append(rest[0])
    ok_w = all(1 <= l.out_features <= 128 and (l.out_features & (l.out_features - 1)) == 0 for l in lin)
    ok_w = ok_w and 1 <= lin[0].in_features <= 128
    ok_bn = all(b.affine and b.track_running_stats and b.momentum is not None for b in bns)
    if not (ok_w and ok_bn and len(set(slopes)) == 1 and all(l.bias is not None for l in lin)):
        return None
    return MlpPlan(lin, bns, float(slopes[0]), tuple(id(m) for m in leaves), identity)


def mlp_plan_is_current(plan, seq):
    return plan is not None and plan.source == tuple(id(m) for m in _leaf_modules(seq)) \
        and plan.linears[0].weight.device == plan.linears[-1].weight.device


def cached_mlp_plan(module, name):
    """MlpPlan of module.<name>, cached on the module and rebuilt when its leaf modules are no longer the ones the plan
    was read from (a SyncBatchNorm conversion, a replaced layer).  None when the stack does not match."""
    seq = getattr(module, name)
    cache = module.__dict__.setdefault("_mlp_plans", {})
    plan = cache.get(name, False)
    if plan is False or (plan is not None and not mlp_plan_is_current(plan, seq)):
        plan = cache[name] = mlp_plan_from_modules(seq)
    return plan


def _bn_group(bn):
    """Process group for cross-rank statistics (train.SyncBatchNorm1d carries one), or None for local BN."""
    import torch.distributed as dist
    if type(bn).__name__ == "SyncBatchNorm1d" and dist.is_available() and dist.is_initialized() and dist.get_world_size(bn.group) > 1:
        return bn.group if bn.group is not None else dist.group.WORLD
    return None


def _unpack_params(nl, params):
    """(Ws, bs, gammas, betas) from the flat order of _flat_params"""
    Ws = [_req(params[2 * i], "W") for i in range(nl)]
    bs = [_req(params[2 * i + 1], "b") for i in range(nl)]
    gs = [_req(params[2 * nl + 2 * i], "gamma") for i in range(nl - 1)]
    bes = [_req(params[2 * nl + 2 * i + 1], "beta") for i in range(nl - 1)]
    return Ws, bs, gs, bes


def _eval_stats(st, bn, B):
    """stats [4][w] of an eval-mode BatchNorm: its running statistics are constants"""
    st[0].copy_(bn.running_mean); st[1].copy_(bn.running_var)
    st[2].copy_(torch.rsqrt(bn.running_var + bn.eps)); st[3].fill_(float(B))


_mlp_scratch_cache = {}


def _mlp_scratch(nbytes, device):
    """Per (device, stream, size) scratch of the fused layer kernels.  Its tail holds the last-block ticket, which must be
    zero before the first call and is left zero by every call, so the buffer is zero-initialised ONCE and reused (the
    partials in it never outlive one C call; calls on one stream are ordered)."""
    key = (device, torch.cuda.current_stream().cuda_stream, int(nbytes))
    buf = _mlp_scratch_cache.get(key)
    if buf is None:
        buf = _mlp_scratch_cache[key] = torch.zeros(int(nbytes), dtype=torch.uint8, device=device)
    return buf


class FusedMlpFn(torch.autograd.Function):
    """out = Linear_n( act(BN_{n-1}( ... act(BN_0(Linear_0(x))) ... )) ) through the fused layer kernels (csrc/mlp.cu)."""

    @staticmethod
    def forward(ctx, x, plan, training, *params):
        lib = _C.load()
        x = _req(x, "x")
        B = x.shape[0]
        nl = len(plan.linears)
        Ws, bs, gs, bes = _unpack_params(nl, params)
        scratch = _mlp_scratch(lib.b200vae_mlp_scratch_bytes(B), x.device)
        ys, stats, counts = [], [], []
        ticks = []                # num_batches_tracked counters, advanced by one multi-tensor launch at the end
        prev = (x, None, None, None)
        for i in range(nl):
            wo, wi = Ws[i].shape
            has_bn = i < nl - 1
            y = torch.empty(B, wo, dtype=torch.float32, device=x.device)
            st = None
            rm = rv = None
            mom = 0.0
            grp = peer = None
            if has_bn:
                bn = plan.bns[i]
                grp = _bn_group(bn) if training else None
                peer = getattr(bn, "peer", None) if grp is not None else None
                st = torch.empty(4, wo, dtype=torch.float32, device=x.device)
                if training and (grp is None or peer is not None):
                    rm, rv, mom = bn.running_mean, bn.running_var, float(bn.momentum)
                    ticks.append(bn.num_batches_tracked)
            if peer is not None:          # cross-rank statistics exchanged by the finalize kernel itself (peer memory)
                _C.check(lib.b200vae_mlp_layer_fwd_peer(_ptr(prev[0]), _ptr(prev[1]), _ptr(prev[2]), _ptr(prev[3]), plan.slope,
                                                        _ptr(Ws[i]), _ptr(bs[i]), B, wi, wo, _ptr(y), _ptr(st),
                                                        float(bn.eps), _ptr(rm), _ptr(rv), mom, _ptr(scratch), peer.ref,
                                                        bn.peer_slots[0], _stream()), "mlp_layer_fwd_peer")
            else:
                _C.check(lib.b200vae_mlp_layer_fwd(_ptr(prev[0]), _ptr(prev[1]), _ptr(prev[2]), _ptr(prev[3]), plan.slope,
                                                   _ptr(Ws[i]), _ptr(bs[i]), B, wi, wo, _ptr(y),
                                                   _ptr(st) if (has_bn and training) else None,
                                                   float(plan.bns[i].eps) if has_bn else 0.0, _ptr(rm), _ptr(rv), mom,
                                                   _ptr(scratch), _stream()), "mlp_layer_fwd")
            n_glob = float(B)
            if has_bn:
                bn = plan.bns[i]
                if not training:
                    _eval_stats(st, bn, B)
                elif peer is not None:
                    n_glob = None
                elif grp is not None:     # cross-rank: one all_gather of (mean, var, count), Chan combine, no host sync
                    import torch.distributed as dist
                    world = dist.get_world_size(grp)
                    pack = torch.cat([st[0], st[1], st[3, :1]])
                    outs = [torch.empty_like(pack) for _ in range(world)]
                    dist.all_gather(outs, pack, group=grp)
                    allp = torch.stack(outs)
                    means, vars_, cnt = allp[:, :wo], allp[:, wo:2 * wo], allp[:, 2 * wo:]
                    N = cnt.sum()
                    mean = (means * cnt).sum(0) / N
                    var = ((vars_ + (means - mean) ** 2) * cnt).sum(0) / N
                    st[0].copy_(mean); st[1].copy_(var); st[2].copy_(torch.rsqrt(var + bn.eps)); st[3].copy_(N.expand(wo))
                    bn.running_mean.mul_(1 - bn.momentum).add_(mean, alpha=bn.momentum)
                    bn.running_var.mul_(1 - bn.momentum).add_(var * (N / (N - 1)), alpha=bn.momentum)
                    bn.num_batches_tracked.add_(1)
                    n_glob = None         # read from st[3] in backward (device value)
            ys.append(y); stats.append(st); counts.append(n_glob)
            prev = (y, st, gs[i] if has_bn else None, bes[i] if has_bn else None)
        if ticks:
            torch._foreach_add_(ticks, 1)
        ctx.plan, ctx.training, ctx.nl = plan, training, nl
        ctx.save_for_backward(x, *ys, *[s for s in stats if s is not None], *Ws, *gs, *bes)
        ctx.scratch = scratch
        return ys[-1]

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dout):
        lib = _C.load()
        plan, training, nl = ctx.plan, ctx.training, ctx.nl
        sv = ctx.saved_tensors
        x = sv[0]; ys = sv[1:1 + nl]; sts = list(sv[1 + nl:nl + nl]) + [None]
        Ws = sv[2 * nl:3 * nl]; gs = sv[3 * nl:4 * nl - 1]; bes = sv[4 * nl - 1:5 * nl - 2]
        B = x.shape[0]
        scratch = ctx.scratch
        dWs, dbs, dgs, dbes = [None] * nl, [None] * nl, [None] * (nl - 1), [None] * (nl - 1)
        da = _req(dout, "grad_out")
        # biases that feed a BatchNorm get exactly-zero gradients: ONE zero fill per backward, sliced per layer
        zero_db = torch.zeros(sum(W.shape[0] for W in Ws[:nl - 1]), dtype=torch.float32, device=x.device) if nl > 1 else None
        zoff = [0]
        for W in Ws[:nl - 1]:
            zoff.append(zoff[-1] + W.shape[0])
        for i in range(nl - 1, -1, -1):
            wo, wi = Ws[i].shape
            has_bn = i < nl - 1
            st = sts[i]
            dyhat = torch.empty(B, wo, dtype=torch.float32, device=x.device)
            sums = torch.empty(2, wo, dtype=torch.float32, device=x.device)
            grp = _bn_group(plan.bns[i]) if (has_bn and training) else None
            peer = getattr(plan.bns[i], "peer", None) if grp is not None else None
            inv_n = 1.0 / B
            if peer is not None:          # local sums (dbeta, dgamma) + rank-ordered global sums in one kernel
                loc = torch.empty(2, wo, dtype=torch.float32, device=x.device)
                _C.check(lib.b200vae_mlp_layer_bwd_reduce_peer(_ptr(da), _ptr(ys[i]), _ptr(st), _ptr(gs[i]), _ptr(bes[i]),
                                                               plan.slope, B, wo, _ptr(dyhat), _ptr(loc), _ptr(sums),
                                                               _ptr(scratch), peer.ref, plan.bns[i].peer_slots[1],
                                                               _stream()), "mlp_layer_bwd_reduce_peer")
                dbes[i], dgs[i] = loc[0], loc[1]
                dbs[i] = zero_db[zoff[i]:zoff[i + 1]]
                inv_n = 1.0 / (B * peer.world)                            # equal shards (train.shard_rows)
            else:
                _C.check(lib.b200vae_mlp_layer_bwd_reduce(_ptr(da), _ptr(ys[i]), _ptr(st), _ptr(gs[i]) if has_bn else None,
                                                          _ptr(bes[i]) if has_bn else None, plan.slope, B, wo, _ptr(dyhat),
                                                          _ptr(sums), _ptr(scratch), _stream()), "mlp_layer_bwd_reduce")
            if peer is not None:
                pass
            elif has_bn:
                # local sums = parameter gradients; copied only where `sums` is modified below (eval mode, NCCL all-reduce)
                if (not training) or grp is not None:
                    dbes[i], dgs[i] = sums[0].clone(), sums[1].clone()
                else:
                    dbes[i], dgs[i] = sums[0], sums[1]
                dbs[i] = zero_db[zoff[i]:zoff[i + 1]]                     # bias feeding a BatchNorm: exactly 0
                if not training:
                    sums.zero_()                                          # eval-mode BN is affine: dy = gamma*invstd*dyhat
                else:
                    if grp is not None:
                        import torch.distributed as dist
                        dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=grp)
                        inv_n = 1.0 / (B * dist.get_world_size(grp))      # equal shards (train.shard_rows)
            else:
                dbs[i] = sums[0].clone()
            prev_y = x if i == 0 else ys[i - 1]
            prev_st = None if i == 0 else sts[i - 1]
            need_da = i > 0 or ctx.needs_input_grad[0]
            da_prev = torch.empty(B, wi, dtype=torch.float32, device=x.device) if need_da else None
            dW = torch.empty_like(Ws[i])
            _C.check(lib.b200vae_mlp_layer_bwd(_ptr(dyhat), _ptr(ys[i]), _ptr(st), _ptr(gs[i]) if has_bn else None,
                                               _ptr(bes[i]) if has_bn else None, _ptr(sums), inv_n, plan.slope, _ptr(Ws[i]),
                                               _ptr(prev_y), _ptr(prev_st), _ptr(gs[i - 1]) if i > 0 else None,
                                               _ptr(bes[i - 1]) if i > 0 else None, B, wo, wi, _ptr(da_prev), _ptr(dW),
                                               _ptr(scratch), _stream()), "mlp_layer_bwd")
            dWs[i] = dW
            da = da_prev
        return (da if ctx.needs_input_grad[0] else None, None, None, *_flat_params(dWs, dbs, dgs, dbes))


STACK_MAX_WIDTH, STACK_MAX_LAYERS = 8, 16


def _stack_ok(plan, training):
    """Every layer narrow and no cross-rank BatchNorm: the whole stack runs as one launch per direction."""
    lin = plan.linears
    if len(lin) > STACK_MAX_LAYERS or any(l.in_features > STACK_MAX_WIDTH or l.out_features > STACK_MAX_WIDTH for l in lin):
        return False
    return not (training and any(_bn_group(b) is not None for b in plan.bns))


def _stack_layers(plan, ys, stats, Ws, bs, gs, bes, training):
    nl = len(Ws)
    arr = (_C.MlpLayer * nl)()
    for i in range(nl):
        L = arr[i]
        wo, wi = Ws[i].shape
        L.W, L.bias, L.y, L.wi, L.wo = _ptr(Ws[i]), _ptr(bs[i]), _ptr(ys[i]), wi, wo
        if i < nl - 1:
            bn = plan.bns[i]
            L.gamma, L.beta, L.stats, L.eps, L.momentum = _ptr(gs[i]), _ptr(bes[i]), _ptr(stats[i]), float(bn.eps), float(bn.momentum)
            if training:
                L.running_mean, L.running_var = _ptr(bn.running_mean), _ptr(bn.running_var)
                L.num_batches_tracked = _ptr(bn.num_batches_tracked)
    return arr


class FusedMlpStackFn(torch.autograd.Function):
    """FusedMlpFn for a stack whose layers are all at most 8 wide: one cooperative launch per direction
    (b200vae_mlp_stack_fwd / _bwd).  head > 0: returns (mu, softplus(var)) -- the two halves of the last layer's output,
    the second through F.softplus -- instead of the output itself."""

    @staticmethod
    def forward(ctx, x, plan, training, head, *params):
        lib = _C.load()
        x = _req(x, "x")
        B, dev = x.shape[0], x.device
        nl = len(plan.linears)
        Ws, bs, gs, bes = _unpack_params(nl, params)
        scratch = _mlp_scratch(lib.b200vae_mlp_scratch_bytes(B), dev)
        ys = [torch.empty(B, W.shape[0], dtype=torch.float32, device=dev) for W in Ws]
        stats = [torch.empty(4, W.shape[0], dtype=torch.float32, device=dev) for W in Ws[:nl - 1]]
        if not training:
            for st, bn in zip(stats, plan.bns):
                _eval_stats(st, bn, B)
        layers = _stack_layers(plan, ys, stats, Ws, bs, gs, bes, training)
        mu = lv = None
        if head:
            mu = torch.empty(B, head, dtype=torch.float32, device=dev)
            lv = torch.empty(B, head, dtype=torch.float32, device=dev)
        _C.check(lib.b200vae_mlp_stack_fwd(layers, nl, _ptr(x), B, plan.slope, int(training), head, _ptr(mu), _ptr(lv),
                                           _ptr(scratch), _stream()), "mlp_stack_fwd")
        ctx.plan, ctx.training, ctx.nl, ctx.head = plan, training, nl, head
        ctx.save_for_backward(x, *ys, *stats, *Ws, *bs, *gs, *bes)
        ctx.scratch = scratch
        ctx.set_materialize_grads(False)
        return (mu, lv) if head else ys[-1]

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, *grads):
        lib = _C.load()
        plan, training, nl, head = ctx.plan, ctx.training, ctx.nl, ctx.head
        sv = ctx.saved_tensors
        x = sv[0]; ys = sv[1:1 + nl]; stats = sv[1 + nl:2 * nl]; Ws = sv[2 * nl:3 * nl]; bs = sv[3 * nl:4 * nl]
        gs = sv[4 * nl:5 * nl - 1]; bes = sv[5 * nl - 1:6 * nl - 2]
        B = x.shape[0]
        g0 = _req(grads[0], "grad_out") if grads[0] is not None else None
        g1 = _req(grads[1], "grad_out") if head and grads[1] is not None else None
        if not head and g0 is None:
            g0 = torch.zeros_like(ys[-1])
        # every parameter gradient in one buffer, written completely by the kernel (zeros included)
        sizes = []
        for i in range(nl):
            wo, wi = Ws[i].shape
            sizes += [wo * wi, wo] + ([wo, wo] if i < nl - 1 else [])
        flat = torch.empty(sum(sizes), dtype=torch.float32, device=x.device)
        parts = list(flat.split(sizes))
        garr = (_C.MlpGrad * nl)()
        dWs, dbs, dgs, dbes = [], [], [], []
        for i in range(nl):
            wo, wi = Ws[i].shape
            dW, db = parts.pop(0).view(wo, wi), parts.pop(0)
            garr[i].dW, garr[i].db = _ptr(dW), _ptr(db)
            dWs.append(dW); dbs.append(db)
            if i < nl - 1:
                dg, dbe = parts.pop(0), parts.pop(0)
                garr[i].dgamma, garr[i].dbeta = _ptr(dg), _ptr(dbe)
                dgs.append(dg); dbes.append(dbe)
        dx = torch.empty_like(x) if ctx.needs_input_grad[0] else None
        layers = _stack_layers(plan, ys, stats, Ws, bs, gs, bes, False)
        _C.check(lib.b200vae_mlp_stack_bwd(layers, garr, nl, _ptr(x), B, plan.slope, int(training), head, _ptr(g0),
                                           _ptr(g1), _ptr(dx), _ptr(ctx.scratch), _stream()), "mlp_stack_bwd")
        return (dx, None, None, None, *_flat_params(dWs, dbs, dgs, dbes))


def fused_mlp(plan, x, training, softplus_head=False):
    """Output of the stack; softplus_head: (mu, softplus(var)) of its two halves (LIDVAE.encode)."""
    params = plan.params()
    if _stack_ok(plan, training):
        head = plan.linears[-1].out_features // 2 if softplus_head else 0
        return FusedMlpStackFn.apply(x, plan, training, head, *params)
    out = FusedMlpFn.apply(x, plan, training, *params)
    if not softplus_head:
        return out
    mu, var = out.split(out.shape[1] // 2, 1)
    return mu, torch.nn.functional.softplus(var)


# ------------------------------------------------------------------------------------------ chamfer
class NearestSqDistFn(torch.autograd.Function):
    """(min_j |a_i - b_j|^2 [B,Na],  min_i |b_j - a_i|^2 [B,Nb]) for point sets a [B,Na,dim], b [B,Nb,dim] without the
    [B,Na,Nb] distance matrix of torch.cdist (model.py:905-912)."""

    @staticmethod
    def forward(ctx, a, b):
        lib = _C.load()
        a, b = _req(a, "points_pred"), _req(b, "points_gt")
        B, Na, dim = a.shape
        Nb = b.shape[1]
        ma = torch.empty(B, Na, dtype=torch.float32, device=a.device)
        mb = torch.empty(B, Nb, dtype=torch.float32, device=a.device)
        ia = torch.empty(B, Na, dtype=torch.int32, device=a.device)
        ib = torch.empty(B, Nb, dtype=torch.int32, device=a.device)
        _C.check(lib.b200vae_nn_sqdist_fwd(_ptr(a), _ptr(b), B, Na, Nb, dim, _ptr(ma), _ptr(ia), _stream()), "nn_sqdist_fwd")
        _C.check(lib.b200vae_nn_sqdist_fwd(_ptr(b), _ptr(a), B, Nb, Na, dim, _ptr(mb), _ptr(ib), _stream()), "nn_sqdist_fwd")
        ctx.save_for_backward(a, b, ia, ib)
        ctx.set_materialize_grads(False)
        return ma, mb

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, ga, gb):
        lib = _C.load()
        a, b, ia, ib = ctx.saved_tensors
        B, Na, dim = a.shape
        Nb = b.shape[1]
        ga = None if ga is None else _req(ga, "grad")
        gb = None if gb is None else _req(gb, "grad")
        da = db = None
        if ctx.needs_input_grad[0] and (ga is not None or gb is not None):
            da = torch.empty_like(a)
            _C.check(lib.b200vae_nn_sqdist_bwd(_ptr(a), _ptr(b), _ptr(ia), _ptr(ib), _ptr(ga), _ptr(gb), B, Na, Nb, dim,
                                               _ptr(da), _stream()), "nn_sqdist_bwd")
        if ctx.needs_input_grad[1] and (ga is not None or gb is not None):
            db = torch.empty_like(b)
            _C.check(lib.b200vae_nn_sqdist_bwd(_ptr(b), _ptr(a), _ptr(ib), _ptr(ia), _ptr(gb), _ptr(ga), B, Nb, Na, dim,
                                               _ptr(db), _stream()), "nn_sqdist_bwd")
        return da, db


# ------------------------------------------------------------------------------------------ Lipschitz
def lipschitz_pair_ratios(X, Y, i1, i2, eps=1e-3):
    """ratio[p] = clamp(|Y[i1]-Y[i2]|,eps)/clamp(|X[i1]-X[i2]|,eps)  (utils.py:548-562)."""
    X = _req(X.detach().reshape(X.shape[0], -1), "X")
    Y = _req(Y.detach().reshape(Y.shape[0], -1), "Y")
    i1 = i1.to(torch.int64).contiguous()
    i2 = i2.to(torch.int64).contiguous()
    P = i1.numel()
    ratio = torch.empty(P, dtype=torch.float32, device=X.device)
    _C.check(_C.load().b200vae_lipschitz_pairs(_ptr(X), _ptr(Y), _ptr(i1), _ptr(i2), P, X.shape[0], X.shape[1],
                                               Y.shape[1], float(eps), _ptr(ratio), _stream()), "lipschitz_pairs")
    return ratio


_ap_scratch = {}


def _allpairs_scratch(device):
    """Zero-initialised partials + ticket per (device, stream); the kernel leaves it ready for the next call."""
    key = (device, torch.cuda.current_stream().cuda_stream)
    buf = _ap_scratch.get(key)
    if buf is None:
        buf = torch.zeros(_C.load().b200vae_lipschitz_scratch_bytes(), dtype=torch.uint8, device=device)
        _ap_scratch[key] = buf
    return buf


def lipschitz_allpairs(X, Y, eps=1e-3, tile_begin=0, tile_end=None, nbins=0, hist_lo=-20.0, hist_hi=20.0):
    """All unordered pairs i<j in tiles [tile_begin, tile_end): returns (stats fp64 [max,min,sum,count], hist)."""
    lib = _C.load()
    X = _req(X.detach().reshape(X.shape[0], -1), "X")
    Y = _req(Y.detach().reshape(Y.shape[0], -1), "Y")
    N = X.shape[0]
    nt = lib.b200vae_lipschitz_num_tiles(N)
    if tile_end is None:
        tile_end = nt
    stats = torch.empty(4, dtype=torch.float64, device=X.device)
    hist = torch.empty(nbins, dtype=torch.int32, device=X.device) if nbins > 0 else None
    _C.check(lib.b200vae_lipschitz_allpairs(_ptr(X), _ptr(Y), N, X.shape[1], Y.shape[1], float(eps), int(tile_begin),
                                            int(tile_end), _ptr(stats), _ptr(hist), nbins, float(hist_lo),
                                            float(hist_hi), _ptr(_allpairs_scratch(X.device)), _stream()),
             "lipschitz_allpairs")
    return stats, hist


def lipschitz_num_tiles(N):
    return int(_C.load().b200vae_lipschitz_num_tiles(N))


# exact all-pairs quantiles: a 3-pass radix select over the keys of lipschitz_allpairs (include/b200vae.h)
_select_buffers = {}


def lipschitz_select_buffers(device):
    """(state uint8, hist int64) per (device, stream), allocated on first use; the passes need no initialisation.  Make one
    call on a stream before capturing it into a CUDA graph, so that the capture allocates nothing."""
    key = (device, torch.cuda.current_stream().cuda_stream)
    bufs = _select_buffers.get(key)
    if bufs is None:
        if torch.cuda.is_current_stream_capturing():
            raise _C.B200VaeError("lipschitz_allpairs_quantiles: make one call on this stream before capturing it")
        lib = _C.load()
        bufs = _select_buffers[key] = (
            torch.empty(lib.b200vae_lipschitz_select_state_bytes(), dtype=torch.uint8, device=device),
            torch.empty(lib.b200vae_lipschitz_select_hist_bytes() // 8, dtype=torch.int64, device=device))
    return bufs


def lipschitz_select_count(X, Y, eps, tile_begin, tile_end, pass_, state, hist):
    """One count pass over the pairs of tiles [tile_begin, tile_end): OVERWRITES `hist` (int64) with this shard's bins."""
    X = _req(X.detach().reshape(X.shape[0], -1), "X")
    Y = _req(Y.detach().reshape(Y.shape[0], -1), "Y")
    _C.check(_C.load().b200vae_lipschitz_select_count(_ptr(X), _ptr(Y), X.shape[0], X.shape[1], Y.shape[1], float(eps),
                                                      int(tile_begin), int(tile_end), int(pass_), _ptr(state), _ptr(hist),
                                                      _stream()), "lipschitz_select_count")


def lipschitz_select_locate(N, q0, q1, pass_, hist, state, out):
    """Narrow the targets with `hist` (summed over every shard); after the last pass out (fp64 [6]) holds
    (v(q0), v(q1), key[k0], key[k0+1], key[k1], key[k1+1])."""
    _C.check(_C.load().b200vae_lipschitz_select_locate(int(N), float(q0), float(q1), int(pass_), _ptr(hist), _ptr(state),
                                                       _ptr(out), _stream()), "lipschitz_select_locate")


def lipschitz_quantile_ranks(n, q):
    """(k, w) of torch.quantile's linear rule for n values, in fp64 (the library owns the rule)."""
    k, w = C.c_longlong(), C.c_double()
    _C.check(_C.load().b200vae_lipschitz_quantile_ranks(int(n), float(q), C.byref(k), C.byref(w)), "lipschitz_quantile_ranks")
    return k.value, w.value


def lipschitz_allpairs_quantiles(X, Y, qs, eps=1e-3, tile_begin=0, tile_end=None, reduce_hist=None):
    """Exact quantiles (torch.quantile's linear rule, ranks in fp64) of the keys of `lipschitz_allpairs` over every pair
    i<j: one or two quantiles `qs`.  Returns a new fp64 device tensor [6] = (v(qs[0]), v(qs[-1]), the two order statistics
    behind each).  With shards, every rank passes its tile range and `reduce_hist(hist)` sums the int64 histogram over the
    ranks in place between count and locate.  No host synchronisation: capturable into a CUDA graph (call once first)."""
    qs = [float(q) for q in qs]
    if not 1 <= len(qs) <= 2:
        raise ValueError("lipschitz_allpairs_quantiles: one or two quantiles")
    N = X.shape[0]
    if tile_end is None:
        tile_end = lipschitz_num_tiles(N)
    state, hist = lipschitz_select_buffers(X.device)
    out = torch.empty(6, dtype=torch.float64, device=X.device)
    for p in range(_C.LIPSCHITZ_SELECT_PASSES):
        lipschitz_select_count(X, Y, eps, tile_begin, tile_end, p, state, hist)
        if reduce_hist is not None:
            reduce_hist(hist)
        lipschitz_select_locate(N, qs[0], qs[-1], p, hist, state, out)
    return out


# ------------------------------------------------------------------------------------------ Adam
def adam_step_(param, grad, m, v, step, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, grad_scale=1.0):
    """In-place fused Adam over flat fp32 buffers (torch.optim.Adam semantics; lipschitz.py:25,43)."""
    _C.check(_C.load().b200vae_adam_step(_ptr(param), _ptr(grad), _ptr(m), _ptr(v), param.numel(), float(lr),
                                         float(betas[0]), float(betas[1]), float(eps), float(weight_decay), int(step),
                                         float(grad_scale), _stream()), "adam_step")
    bump_weights_epoch()


def adam_step_dev_(param, grad, m, v, step_dev, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, grad_scale=1.0):
    """Graph-capturable fused Adam: `step_dev` is an int64 device scalar, incremented by the call."""
    _C.check(_C.load().b200vae_adam_step_dev(_ptr(param), _ptr(grad), _ptr(m), _ptr(v), param.numel(), float(lr),
                                             float(betas[0]), float(betas[1]), float(eps), float(weight_decay),
                                             _ptr(step_dev), float(grad_scale), _stream()), "adam_step_dev")
    bump_weights_epoch()


def adam_step_sched_(param, grad, m, v, step_dev, lr0, betas, eps, weight_decay, grad_scale, sched_kind, sched_T):
    """adam_step_dev_ with the learning rate computed on the device from the step counter (0 constant, 1 cosine annealing
    to 0 over sched_T steps: main.py:200-203)."""
    _C.check(_C.load().b200vae_adam_step_sched(_ptr(param), _ptr(grad), _ptr(m), _ptr(v), param.numel(), float(lr0),
                                               float(betas[0]), float(betas[1]), float(eps), float(weight_decay),
                                               _ptr(step_dev), float(grad_scale), int(sched_kind), int(sched_T), _stream()),
             "adam_step_sched")
    bump_weights_epoch()


def peer_allreduce_adam_(comm, slot, grad_buf, param_buf, m, v, n, step_dev, lr=1e-3, betas=(0.9, 0.999), eps=1e-8,
                         weight_decay=0.0, grad_scale=1.0):
    """Gradient all-reduce fused with Adam over peer memory (include/b200vae.h b200vae_peer_allreduce_adam).
    grad_buf / param_buf: peer.PeerBuffer holding the flat gradient / parameter buffers of every rank."""
    lib = _C.load()
    _C.check(lib.b200vae_peer_allreduce_adam(comm.ref, slot, grad_buf.ptr_array(), param_buf.ptr_array(), _ptr(_req(m, "m")),
                                             _ptr(_req(v, "v")), n, lr, betas[0], betas[1], eps, weight_decay,
                                             _ptr(step_dev), grad_scale, _stream()), "peer_allreduce_adam")
    bump_weights_epoch()
