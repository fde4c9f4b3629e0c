"""ctypes binding of libb200vae.so (include/b200vae.h).  No torch types cross this boundary: raw
device pointers, sizes and the current CUDA stream handle only.

There is NO CPU fallback: if the shared library is missing ``load()`` raises, and every compute entry
returns an error code that is turned into ``B200VaeError`` here.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B200VAE_LIB", os.path.join(_HERE, "libb200vae.so"))   # override: A/B builds of the library
CSRC = os.path.join(_HERE, "csrc")

WEIGHT_EXP, WEIGHT_CLAMP = 0, 1
PREC_FP32, PREC_TF32, PREC_TF32X3, PREC_F16X3 = 0, 1, 3, 4          # 2 is reserved (include/b200vae.h)
PRECISIONS = {"fp32": PREC_FP32, "tf32": PREC_TF32, "tf32x3": PREC_TF32X3, "f16x3": PREC_F16X3}
LOSS_OUT_FLOATS = 2048

_ERR = {-1: "bad shape", -2: "unsupported configuration", -3: "null or misaligned pointer",
        -4: "CUDA error", -5: "workspace too small"}

EXPORTS = [
    "b200vae_icnn_workspace_bytes", "b200vae_icnn_prepare", "b200vae_icnn_decode_fwd", "b200vae_icnn_decode_bwd",
    "b200vae_icnn_decode_bwd_params",
    "b200vae_loss_fwd", "b200vae_loss_bwd", "b200vae_lipschitz_pairs", "b200vae_lipschitz_allpairs",
    "b200vae_lipschitz_num_tiles", "b200vae_lipschitz_scratch_bytes", "b200vae_adam_step", "b200vae_adam_step_dev", "b200vae_adam_step_sched", "b200vae_mlp_scratch_bytes", "b200vae_mlp_layer_fwd",
    "b200vae_mlp_layer_bwd_reduce", "b200vae_mlp_layer_bwd", "b200vae_nn_sqdist_fwd", "b200vae_nn_sqdist_bwd", "b200vae_last_cuda_error", "b200vae_version",
    "b200vae_launch_count",
    "b200vae_peer_exchange_bytes", "b200vae_peer_num_slots", "b200vae_peer_max_payload", "b200vae_peer_alloc", "b200vae_peer_open",
    "b200vae_peer_close", "b200vae_peer_free", "b200vae_peer_timed_out", "b200vae_peer_allgather", "b200vae_mlp_layer_fwd_peer",
    "b200vae_mlp_layer_bwd_reduce_peer", "b200vae_peer_allreduce_adam",
    "b200vae_icnn_wide_workspace_bytes", "b200vae_icnn_wide_fwd", "b200vae_icnn_wide_bwd", "b200vae_icnn_wide_bwd_psi",
    "b200vae_mi_logqz", "b200vae_nll_iw_lse", "b200vae_nll_iw_scratch_bytes", "b200vae_mlp_stack_fwd",
    "b200vae_mlp_stack_bwd", "b200vae_lipschitz_select_state_bytes", "b200vae_lipschitz_select_hist_bytes",
    "b200vae_lipschitz_quantile_ranks", "b200vae_lipschitz_select_count", "b200vae_lipschitz_select_locate",
    "b200vae_icnn_jac_scratch_bytes", "b200vae_icnn_decode_jac", "b200vae_jacobian_chain",
    "b200vae_brenier_inverse_state_bytes", "b200vae_brenier_inverse_init", "b200vae_brenier_newton_step",
]
LIPSCHITZ_SELECT_PASSES = 3
# per-row status of the Newton left inverse (B200VAE_INV_*); a larger value is a worse outcome
INV_ACTIVE, INV_CONVERGED, INV_MAXITER, INV_STALLED, INV_SINGULAR, INV_NONFINITE = range(6)
PEER_MAX_WORLD, PEER_HANDLE_BYTES = 16, 64


class B200VaeError(RuntimeError):
    pass


class IcnnParams(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("A0w", "A0b", "A1w", "A1b", "A2w", "A2b", "W0", "W1")]


class IcnnGrads(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("A0w", "A0b", "A1w", "A1b", "A2w", "A2b", "W0", "W1")]


class PeerStruct(C.Structure):
    """b200vae_peer_t"""
    _fields_ = [("world", C.c_int), ("rank", C.c_int), ("buf", C.c_void_p * 16)]


class MlpLayer(C.Structure):
    """b200vae_mlp_layer_t"""
    _fields_ = [(k, C.c_void_p) for k in ("W", "bias", "gamma", "beta", "y", "stats", "running_mean", "running_var",
                                          "num_batches_tracked")] + \
        [("eps", C.c_float), ("momentum", C.c_float), ("wi", C.c_int), ("wo", C.c_int)]


class MlpGrad(C.Structure):
    """b200vae_mlp_grad_t"""
    _fields_ = [(k, C.c_void_p) for k in ("dW", "db", "dgamma", "dbeta")]


PARAM_FIELDS = ("A0w", "A0b", "A1w", "A1b", "A2w", "A2b", "W0", "W1")

_lib = None


def build(verbose: bool = False) -> str:
    """Compile the CUDA sources in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    r = subprocess.run(["make", "-C", CSRC, "-j8"], capture_output=True, text=True)
    if r.returncode != 0:
        raise B200VaeError("building libb200vae.so failed:\n" + r.stdout[-4000:] + r.stderr[-4000:])
    if verbose:
        print(r.stdout[-2000:])
    return LIB_PATH


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise B200VaeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(make -C vae_song_b200/csrc).  There is no CPU fallback for this path.")
    lib = C.CDLL(LIB_PATH)
    vp, i, f, ll, sz = C.c_void_p, C.c_int, C.c_float, C.c_longlong, C.c_size_t
    lib.b200vae_icnn_workspace_bytes.restype = sz
    lib.b200vae_icnn_workspace_bytes.argtypes = [i, i, i, i, i]
    lib.b200vae_icnn_prepare.restype = i
    lib.b200vae_icnn_prepare.argtypes = [C.POINTER(IcnnParams), i, i, i, i, vp, sz, vp]
    lib.b200vae_icnn_decode_fwd.restype = i
    lib.b200vae_icnn_decode_fwd.argtypes = [vp, i, i, i, i, f, vp, vp, vp, vp, i, vp, sz, vp]
    lib.b200vae_icnn_decode_bwd.restype = i
    lib.b200vae_icnn_decode_bwd.argtypes = [vp, vp, vp, vp, vp, i, i, i, C.POINTER(IcnnParams), i, f,
                                            C.POINTER(IcnnGrads), vp, i, vp, sz, vp]
    lib.b200vae_icnn_decode_bwd_params.restype = i
    lib.b200vae_icnn_decode_bwd_params.argtypes = [vp, vp, vp, vp, i, i, i, C.POINTER(IcnnParams), i, C.POINTER(IcnnGrads), i,
                                                   vp, sz, vp]
    lib.b200vae_icnn_jac_scratch_bytes.restype = sz
    lib.b200vae_icnn_jac_scratch_bytes.argtypes = [i, i, i, i]
    lib.b200vae_icnn_decode_jac.restype = i
    lib.b200vae_icnn_decode_jac.argtypes = [vp, i, i, i, f, vp, vp, vp, vp, vp, i, vp, sz, vp, sz, vp]
    lib.b200vae_jacobian_chain.restype = i
    lib.b200vae_jacobian_chain.argtypes = [vp, vp, vp, i, i, i, vp, vp, vp]
    lib.b200vae_brenier_inverse_state_bytes.restype = sz
    lib.b200vae_brenier_inverse_state_bytes.argtypes = [i, i]
    lib.b200vae_brenier_inverse_init.restype = i
    lib.b200vae_brenier_inverse_init.argtypes = [vp, vp, i, i, f, f, vp, sz, vp, vp, vp, vp, vp]
    lib.b200vae_brenier_newton_step.restype = i
    lib.b200vae_brenier_newton_step.argtypes = [vp, vp, vp, i, i, f, i, i, vp, sz, vp, vp, vp, vp, vp]
    lib.b200vae_loss_fwd.restype = i
    lib.b200vae_loss_fwd.argtypes = [vp, vp, vp, vp, i, i, i, vp, vp, i, i, vp, vp, vp, i, i, i, vp, vp]
    lib.b200vae_loss_bwd.restype = i
    lib.b200vae_loss_bwd.argtypes = [vp, vp, vp, vp, i, i, i, vp, vp, i, i, vp, vp, vp, i, i, i, vp, vp, vp,
                                     vp, vp, vp, vp, vp]
    lib.b200vae_lipschitz_pairs.restype = i
    lib.b200vae_lipschitz_pairs.argtypes = [vp, vp, vp, vp, i, i, i, i, f, vp, vp]
    lib.b200vae_lipschitz_allpairs.restype = i
    lib.b200vae_lipschitz_allpairs.argtypes = [vp, vp, i, i, i, f, ll, ll, vp, vp, i, f, f, vp, vp]
    lib.b200vae_lipschitz_scratch_bytes.restype = sz
    lib.b200vae_lipschitz_scratch_bytes.argtypes = []
    lib.b200vae_lipschitz_num_tiles.restype = ll
    lib.b200vae_lipschitz_num_tiles.argtypes = [i]
    d = C.c_double
    lib.b200vae_lipschitz_select_state_bytes.restype = sz
    lib.b200vae_lipschitz_select_state_bytes.argtypes = []
    lib.b200vae_lipschitz_select_hist_bytes.restype = sz
    lib.b200vae_lipschitz_select_hist_bytes.argtypes = []
    lib.b200vae_lipschitz_quantile_ranks.restype = i
    lib.b200vae_lipschitz_quantile_ranks.argtypes = [ll, d, C.POINTER(ll), C.POINTER(d)]
    lib.b200vae_lipschitz_select_count.restype = i
    lib.b200vae_lipschitz_select_count.argtypes = [vp, vp, i, i, i, f, ll, ll, i, vp, vp, vp]
    lib.b200vae_lipschitz_select_locate.restype = i
    lib.b200vae_lipschitz_select_locate.argtypes = [i, d, d, i, vp, vp, vp, vp]
    lib.b200vae_adam_step.restype = i
    lib.b200vae_adam_step.argtypes = [vp, vp, vp, vp, ll, f, f, f, f, f, ll, f, vp]
    lib.b200vae_adam_step_dev.restype = i
    lib.b200vae_adam_step_dev.argtypes = [vp, vp, vp, vp, ll, f, f, f, f, f, vp, f, vp]
    lib.b200vae_adam_step_sched.restype = i
    lib.b200vae_adam_step_sched.argtypes = [vp, vp, vp, vp, ll, f, f, f, f, f, vp, f, i, ll, vp]
    lib.b200vae_mlp_scratch_bytes.restype = sz
    lib.b200vae_mlp_scratch_bytes.argtypes = [i]
    lib.b200vae_mlp_layer_fwd.restype = i
    lib.b200vae_mlp_layer_fwd.argtypes = [vp, vp, vp, vp, f, vp, vp, i, i, i, vp, vp, f, vp, vp, f, vp, vp]
    lib.b200vae_mlp_layer_bwd_reduce.restype = i
    lib.b200vae_mlp_layer_bwd_reduce.argtypes = [vp, vp, vp, vp, vp, f, i, i, vp, vp, vp, vp]
    lib.b200vae_mlp_layer_bwd.restype = i
    lib.b200vae_mlp_layer_bwd.argtypes = [vp, vp, vp, vp, vp, vp, f, f, vp, vp, vp, vp, vp, i, i, i, vp, vp, vp, vp]
    lib.b200vae_mlp_stack_fwd.restype = i
    lib.b200vae_mlp_stack_fwd.argtypes = [C.POINTER(MlpLayer), i, vp, i, f, i, i, vp, vp, vp, vp]
    lib.b200vae_mlp_stack_bwd.restype = i
    lib.b200vae_mlp_stack_bwd.argtypes = [C.POINTER(MlpLayer), C.POINTER(MlpGrad), i, vp, i, f, i, i, vp, vp, vp, vp, vp]
    lib.b200vae_nn_sqdist_fwd.restype = i
    lib.b200vae_nn_sqdist_fwd.argtypes = [vp, vp, i, i, i, i, vp, vp, vp]
    lib.b200vae_nn_sqdist_bwd.restype = i
    lib.b200vae_nn_sqdist_bwd.argtypes = [vp, vp, vp, vp, vp, vp, i, i, i, i, vp, vp]
    lib.b200vae_icnn_wide_workspace_bytes.restype = sz
    lib.b200vae_icnn_wide_workspace_bytes.argtypes = [i, i, i, i, i]
    lib.b200vae_icnn_wide_fwd.restype = i
    lib.b200vae_icnn_wide_fwd.argtypes = [vp, i, i, i, i, C.POINTER(IcnnParams), i, f, vp, vp, vp, vp, vp, vp, i, vp, sz, vp]
    lib.b200vae_icnn_wide_bwd.restype = i
    lib.b200vae_icnn_wide_bwd.argtypes = [vp, vp, vp, vp, vp, i, i, i, i, C.POINTER(IcnnParams), i, f, C.POINTER(IcnnGrads), vp,
                                          vp, vp, vp, vp, i, vp, sz, vp]
    lib.b200vae_icnn_wide_bwd_psi.restype = i
    lib.b200vae_icnn_wide_bwd_psi.argtypes = [vp, vp, vp, vp, vp, i, i, i, i, C.POINTER(IcnnParams), i, C.POINTER(IcnnGrads), vp,
                                              vp, vp, vp, vp, sz, vp]
    lib.b200vae_mi_logqz.restype = i
    lib.b200vae_mi_logqz.argtypes = [vp, vp, vp, i, i, vp, vp]
    lib.b200vae_nll_iw_lse.restype = i
    lib.b200vae_nll_iw_lse.argtypes = [vp, vp, vp, i, i, i, vp, vp, vp]
    lib.b200vae_nll_iw_scratch_bytes.restype = sz
    lib.b200vae_nll_iw_scratch_bytes.argtypes = []
    pp = C.POINTER(PeerStruct)
    lib.b200vae_peer_exchange_bytes.restype = sz
    lib.b200vae_peer_exchange_bytes.argtypes = []
    lib.b200vae_peer_num_slots.restype = i
    lib.b200vae_peer_max_payload.restype = i
    lib.b200vae_peer_alloc.restype = i
    lib.b200vae_peer_alloc.argtypes = [sz, C.POINTER(vp), C.c_char_p]
    lib.b200vae_peer_open.restype = i
    lib.b200vae_peer_open.argtypes = [C.c_char_p, C.POINTER(vp)]
    lib.b200vae_peer_close.restype = i
    lib.b200vae_peer_close.argtypes = [vp]
    lib.b200vae_peer_free.restype = i
    lib.b200vae_peer_free.argtypes = [vp]
    lib.b200vae_peer_timed_out.restype = i
    lib.b200vae_peer_timed_out.argtypes = [pp, C.POINTER(i)]
    lib.b200vae_peer_allgather.restype = i
    lib.b200vae_peer_allgather.argtypes = [pp, i, vp, i, vp, vp]
    lib.b200vae_mlp_layer_fwd_peer.restype = i
    lib.b200vae_mlp_layer_fwd_peer.argtypes = [vp, vp, vp, vp, f, vp, vp, i, i, i, vp, vp, f, vp, vp, f, vp, pp, i, vp]
    lib.b200vae_mlp_layer_bwd_reduce_peer.restype = i
    lib.b200vae_mlp_layer_bwd_reduce_peer.argtypes = [vp, vp, vp, vp, vp, f, i, i, vp, vp, vp, vp, pp, i, vp]
    lib.b200vae_peer_allreduce_adam.restype = i
    lib.b200vae_peer_allreduce_adam.argtypes = [pp, i, C.POINTER(vp), C.POINTER(vp), vp, vp, ll, f, f, f, f, f, vp, f, vp]
    lib.b200vae_last_cuda_error.restype = i
    lib.b200vae_version.restype = C.c_char_p
    lib.b200vae_launch_count.restype = ll
    _lib = lib
    return lib


def check(rc: int, what: str):
    if rc != 0:
        extra = ""
        if rc == -4:
            extra = f" (cudaError {load().b200vae_last_cuda_error()})"
        raise B200VaeError(f"{what}: {_ERR.get(rc, rc)}{extra}")


def launch_count() -> int:
    return int(load().b200vae_launch_count())


def version() -> str:
    return load().b200vae_version().decode()
