"""ctypes binding of ``csrc/libl2o_b200.so`` (C-ABI declared in ``include/l2o_b200.h``).

There is deliberately NO fallback: if the shared library is missing or a call fails, this module
raises.  The product path never routes through ``oracle/`` or plain PyTorch math.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.environ.get("L2O_LIB") or os.path.join(CSRC, "libl2o_b200.so")  # L2O_LIB: A/B-test an alternative build
INCLUDE = os.path.join(_ROOT, "include")

L2O_OK, L2O_E_INVALID, L2O_E_UNSUPPORTED, L2O_E_CUDA, L2O_E_NOMEM = 0, -1, -2, -3, -4
PRE_IDENTITY, PRE_LOGSIGN, PRE_FC = 0, 1, 2
OPT_NONE, OPT_RASTRIGIN_SEP, OPT_QUADRATIC_DIAG, OPT_QUADRATIC_BATCH = 0, 1, 2, 3
ENGINE_AUTO, ENGINE_FFMA, ENGINE_TC = 0, 1, 2
RULE_SGD, RULE_ADAM = 0, 1

# every symbol include/l2o_b200.h declares (tests check the .so exports all of them)
EXPORTS = [
    "l2o_net_create", "l2o_net_destroy", "l2o_net_set_engine", "l2o_theta_count", "l2o_state_floats", "l2o_workspace_bytes",
    "l2o_step", "l2o_unroll_fwd", "l2o_unroll_bwd", "l2o_adam_step", "l2o_log_and_sign", "l2o_lasso_grad",
    "l2o_dense_create", "l2o_dense_destroy", "l2o_dense_theta_count", "l2o_dense_state_floats", "l2o_dense_step",
    "l2o_dense_unroll_bwd",
    "l2o_launch_count", "l2o_status_string", "l2o_last_cuda_error", "l2o_version",
    "l2o_hrnn_create", "l2o_hrnn_destroy", "l2o_hrnn_theta_count", "l2o_hrnn_state_floats", "l2o_hrnn_coords",
    "l2o_hrnn_workspace_bytes", "l2o_hrnn_init_state", "l2o_hrnn_prepare", "l2o_hrnn_step",
    "l2o_hrnn_set_global_sizes", "l2o_hrnn_reduce_layout", "l2o_hrnn_prepare_local", "l2o_hrnn_prepare_finish",
    "l2o_hrnn_step_local", "l2o_hrnn_step_finish", "l2o_hrnn_coord_bwd", "l2o_hrnn_workspace_layout",
    "l2o_rule_state_floats", "l2o_rule_step", "l2o_rule_unroll_fwd",
]


class NetDesc(C.Structure):
    _fields_ = [("n_layers", C.c_int32), ("hidden", C.c_int32 * 2), ("preprocess", C.c_int32),
                ("n_in", C.c_int32), ("fc_dim", C.c_int32), ("logsign_k", C.c_float), ("scale", C.c_float),
                ("tanh_output", C.c_int32)]


_fp = C.c_void_p


class StepArgs(C.Structure):
    _fields_ = [("n", C.c_int64), ("theta", _fp), ("in0", _fp), ("in1", _fp), ("m", _fp), ("v", _fp),
                ("beta1", C.c_float), ("beta2", C.c_float), ("p", C.c_float), ("state_in", _fp),
                ("state_out", _fp), ("x", _fp), ("delta", _fp), ("feat_out", _fp), ("step_ptr", _fp), ("t_offset", C.c_int32),
                ("reuse_weights", C.c_int32)]


class UnrollArgs(C.Structure):
    _fields_ = [("n", C.c_int64), ("T", C.c_int32), ("theta", _fp), ("in_seq", _fp), ("opt_kind", C.c_int32),
                ("opt_a", _fp), ("opt_b", _fp), ("opt_alpha", C.c_float), ("opt_fscale", C.c_float), ("x", _fp),
                ("state", _fp), ("ckpt", _fp), ("m", _fp), ("v", _fp), ("beta1", C.c_float), ("beta2", C.c_float),
                ("step0", C.c_int32), ("g_rec", _fp), ("feat_rec", _fp), ("fx", _fp), ("delta_seq", _fp),
                ("labels", _fp), ("imit_loss", _fp), ("n_total", C.c_int64), ("opt_group", C.c_int32)]


class BwdArgs(C.Structure):
    _fields_ = [("n", C.c_int64), ("T", C.c_int32), ("theta", _fp), ("in_seq", _fp), ("ckpt", _fp), ("g_rec", _fp),
                ("labels", _fp), ("n_total", C.c_int64), ("dtheta", _fp), ("delta_seq", _fp), ("scratch", _fp)]


class LassoArgs(C.Structure):
    _fields_ = [("batch", C.c_int32), ("m", C.c_int32), ("n", C.c_int32), ("A", _fp), ("y", _fp), ("x", _fp),
                ("scale", _fp), ("l1", C.c_float), ("g", _fp), ("f", _fp)]


class DenseDesc(C.Structure):
    _fields_ = [("n_layers", C.c_int32), ("hidden", C.c_int32 * 2), ("n_in", C.c_int32), ("preprocess", C.c_int32),
                ("logsign_k", C.c_float), ("n_out", C.c_int32), ("scale", C.c_float), ("tanh_output", C.c_int32)]


class DenseStepArgs(C.Structure):
    _fields_ = [("rows", C.c_int64), ("theta", _fp), ("in_", _fp), ("state_in", _fp), ("state_out", _fp), ("x", _fp),
                ("delta", _fp)]


class DenseBwdArgs(C.Structure):
    _fields_ = [("rows", C.c_int64), ("T", C.c_int32), ("theta", _fp), ("in_seq", _fp), ("ckpt", _fp), ("g_rec", _fp),
                ("labels", _fp), ("n_total", C.c_int64), ("dtheta", _fp)]


class HrnnArgs(C.Structure):
    _fields_ = [("theta", _fp), ("x", _fp), ("g", _fp), ("state", _fp), ("layer", _fp), ("global_", _fp),
                ("workspace", _fp), ("update", _fp)]


class HrnnBwdArgs(C.Structure):
    _fields_ = [("theta", _fp), ("state_old", _fp), ("g", _fp), ("bias0", _fp), ("zero_flag", _fp), ("mean_log_lr", _fp),
                ("d_state_new", _fp), ("d_upd", _fp), ("d_sums", _fp), ("d_state_old", _fp), ("d_theta", _fp),
                ("d_bias0", _fp), ("d_mean_log_lr", _fp)]


class RuleDesc(C.Structure):
    _fields_ = [("kind", C.c_int32), ("learning_rate", C.c_double), ("beta1", C.c_double), ("beta2", C.c_double),
                ("epsilon", C.c_double)]


class RuleStepArgs(C.Structure):
    _fields_ = [("n", C.c_int64), ("g", _fp), ("state_in", _fp), ("state_out", _fp), ("x", _fp), ("delta", _fp)]


class RuleUnrollArgs(C.Structure):
    _fields_ = [("n", C.c_int64), ("T", C.c_int32), ("opt_kind", C.c_int32), ("opt_a", _fp), ("opt_b", _fp),
                ("opt_alpha", C.c_float), ("opt_fscale", C.c_float), ("x", _fp), ("state", _fp), ("fx", _fp)]


class L2OError(RuntimeError):
    pass


NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-O3", "-lineinfo",
              "-I" + INCLUDE, "-I" + CSRC, "-Xcompiler", "-fPIC"]
OBJ_DIR = os.path.join(_ROOT, "build", "obj")


def translation_units():
    return [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith(".cu")]


def sources():
    return [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith((".cu", ".cuh", ".h"))] + \
           [os.path.join(INCLUDE, "l2o_b200.h")]


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every CUDA translation unit in-tree for sm_100a (nvcc cross-compiles without a GPU) and link
    ``libl2o_b200.so``.  Objects are rebuilt only when a source/header is newer."""
    from concurrent.futures import ThreadPoolExecutor
    os.makedirs(OBJ_DIR, exist_ok=True)
    newest_hdr = max(os.path.getmtime(p) for p in sources() if not p.endswith(".cu"))
    jobs = []
    for tu in translation_units():
        obj = os.path.join(OBJ_DIR, os.path.basename(tu)[:-3] + ".o")
        stale = force or not os.path.exists(obj) or os.path.getmtime(obj) < max(os.path.getmtime(tu), newest_hdr)
        jobs.append((tu, obj, stale))

    def compile_one(job):
        tu, obj, stale = job
        if not stale:
            return None
        cmd = ["nvcc"] + NVCC_FLAGS + ["-c", "-o", obj, tu]
        if verbose:
            print(" ".join(cmd), file=sys.stderr)
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise L2OError("nvcc failed for %s:\n%s%s" % (tu, r.stdout, r.stderr))
        return obj

    with ThreadPoolExecutor(max_workers=max(1, min(len(jobs), os.cpu_count() or 1))) as ex:
        rebuilt = [o for o in ex.map(compile_one, jobs) if o]
    objs = [j[1] for j in jobs]
    if rebuilt or not os.path.exists(LIB_PATH) or os.path.getmtime(LIB_PATH) < max(os.path.getmtime(o) for o in objs):
        cmd = ["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", LIB_PATH] + objs
        if verbose:
            print(" ".join(cmd), file=sys.stderr)
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise L2OError("link failed:\n" + r.stdout + r.stderr)
    return LIB_PATH


_lib = None


def lib():
    """Load the shared library (fails loudly if it was never built)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise L2OError(f"{LIB_PATH} not found - run `python -c 'import __graft_entry__ as g; g.build()'` "
                       "(there is no CPU/PyTorch fallback)")
    L = C.CDLL(LIB_PATH)
    L.l2o_net_create.argtypes = [C.POINTER(C.c_void_p), C.POINTER(NetDesc)]
    L.l2o_net_create.restype = C.c_int
    L.l2o_net_destroy.argtypes = [C.c_void_p]
    L.l2o_net_destroy.restype = None
    L.l2o_net_set_engine.argtypes = [C.c_void_p, C.c_int32]
    L.l2o_net_set_engine.restype = C.c_int
    L.l2o_theta_count.argtypes = [C.c_void_p]
    L.l2o_theta_count.restype = C.c_int64
    L.l2o_state_floats.argtypes = [C.c_void_p]
    L.l2o_state_floats.restype = C.c_int64
    L.l2o_workspace_bytes.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]
    L.l2o_workspace_bytes.restype = C.c_int
    L.l2o_step.argtypes = [C.c_void_p, C.POINTER(StepArgs), C.c_void_p]
    L.l2o_step.restype = C.c_int
    L.l2o_unroll_fwd.argtypes = [C.c_void_p, C.POINTER(UnrollArgs), C.c_void_p]
    L.l2o_unroll_fwd.restype = C.c_int
    L.l2o_unroll_bwd.argtypes = [C.c_void_p, C.POINTER(BwdArgs), C.c_void_p]
    L.l2o_unroll_bwd.restype = C.c_int
    L.l2o_adam_step.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_float,
                                C.c_float, C.c_float, C.c_float, C.c_void_p]
    L.l2o_adam_step.restype = C.c_int
    L.l2o_log_and_sign.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_float, C.c_void_p]
    L.l2o_log_and_sign.restype = C.c_int
    L.l2o_lasso_grad.argtypes = [C.POINTER(LassoArgs), C.c_void_p]
    L.l2o_lasso_grad.restype = C.c_int
    L.l2o_dense_create.argtypes = [C.POINTER(C.c_void_p), C.POINTER(DenseDesc)]
    L.l2o_dense_create.restype = C.c_int
    L.l2o_dense_destroy.argtypes = [C.c_void_p]
    L.l2o_dense_destroy.restype = None
    for name in ("l2o_dense_theta_count", "l2o_dense_state_floats"):
        getattr(L, name).argtypes = [C.c_void_p]
        getattr(L, name).restype = C.c_int64
    L.l2o_dense_step.argtypes = [C.c_void_p, C.POINTER(DenseStepArgs), C.c_void_p]
    L.l2o_dense_step.restype = C.c_int
    L.l2o_dense_unroll_bwd.argtypes = [C.c_void_p, C.POINTER(DenseBwdArgs), C.c_void_p]
    L.l2o_dense_unroll_bwd.restype = C.c_int
    L.l2o_launch_count.argtypes = []
    L.l2o_launch_count.restype = C.c_int64
    L.l2o_hrnn_create.argtypes = [C.POINTER(C.c_void_p), C.POINTER(C.c_int64), C.c_int32]
    L.l2o_hrnn_create.restype = C.c_int
    L.l2o_hrnn_destroy.argtypes = [C.c_void_p]
    L.l2o_hrnn_destroy.restype = None
    L.l2o_hrnn_theta_count.argtypes = []
    L.l2o_hrnn_theta_count.restype = C.c_int64
    L.l2o_hrnn_state_floats.argtypes = []
    L.l2o_hrnn_state_floats.restype = C.c_int64
    for name in ("l2o_hrnn_coords", "l2o_hrnn_workspace_bytes"):
        getattr(L, name).argtypes = [C.c_void_p]
        getattr(L, name).restype = C.c_int64
    L.l2o_hrnn_set_global_sizes.argtypes = [C.c_void_p, C.POINTER(C.c_int64)]
    L.l2o_hrnn_set_global_sizes.restype = C.c_int
    L.l2o_hrnn_reduce_layout.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    L.l2o_hrnn_reduce_layout.restype = C.c_int
    L.l2o_hrnn_coord_bwd.argtypes = [C.c_void_p, C.POINTER(HrnnBwdArgs), C.c_void_p]
    L.l2o_hrnn_coord_bwd.restype = C.c_int
    L.l2o_hrnn_workspace_layout.argtypes = [C.c_void_p, C.POINTER(C.c_int64)]
    L.l2o_hrnn_workspace_layout.restype = C.c_int
    for name in ("l2o_hrnn_init_state", "l2o_hrnn_prepare", "l2o_hrnn_step", "l2o_hrnn_prepare_local",
                 "l2o_hrnn_prepare_finish", "l2o_hrnn_step_local", "l2o_hrnn_step_finish"):
        getattr(L, name).argtypes = [C.c_void_p, C.POINTER(HrnnArgs), C.c_void_p]
        getattr(L, name).restype = C.c_int
    L.l2o_rule_state_floats.argtypes = [C.POINTER(RuleDesc), C.c_int64, C.POINTER(C.c_int64)]
    L.l2o_rule_state_floats.restype = C.c_int
    L.l2o_rule_step.argtypes = [C.POINTER(RuleDesc), C.POINTER(RuleStepArgs), C.c_void_p]
    L.l2o_rule_step.restype = C.c_int
    L.l2o_rule_unroll_fwd.argtypes = [C.POINTER(RuleDesc), C.POINTER(RuleUnrollArgs), C.c_void_p]
    L.l2o_rule_unroll_fwd.restype = C.c_int
    for name in ("l2o_status_string", "l2o_last_cuda_error", "l2o_version"):
        getattr(L, name).restype = C.c_char_p
    L.l2o_status_string.argtypes = [C.c_int]
    _lib = L
    return L


def check(rc: int, what: str):
    if rc != L2O_OK:
        L = lib()
        msg = L.l2o_status_string(rc).decode()
        if rc == L2O_E_CUDA:
            msg += ": " + L.l2o_last_cuda_error().decode()
        raise L2OError(f"{what} failed: {msg} ({rc})")
