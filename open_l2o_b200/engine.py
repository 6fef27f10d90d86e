"""Thin torch-tensor front end of the C-ABI (``include/l2o_b200.h``).  PyTorch is used only as the
owner of device memory and streams; all arithmetic happens in the CUDA library."""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import torch

from . import _lib
from ._lib import (BwdArgs, NetDesc, StepArgs, UnrollArgs, L2OError, PRE_FC, PRE_IDENTITY, PRE_LOGSIGN,
                   OPT_NONE, OPT_QUADRATIC_DIAG, OPT_RASTRIGIN_SEP, OPT_QUADRATIC_BATCH, ENGINE_AUTO, ENGINE_FFMA, ENGINE_TC,
                   RULE_ADAM, RULE_SGD)

_PRE = {"identity": PRE_IDENTITY, "LogAndSign": PRE_LOGSIGN, "fc": PRE_FC}
OPT_KINDS = {"rastrigin_sep": OPT_RASTRIGIN_SEP, "quadratic_diag": OPT_QUADRATIC_DIAG,
             "quadratic_batch": OPT_QUADRATIC_BATCH}


def _ptr(t: Optional[torch.Tensor], dtype=torch.float32, name="tensor"):
    if t is None:
        return None
    if not t.is_cuda:
        raise L2OError(f"{name}: expected a CUDA tensor (this engine has no CPU path)")
    if t.dtype != dtype:
        raise L2OError(f"{name}: expected dtype {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise L2OError(f"{name}: expected a contiguous tensor")
    return t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


class NetHandle:
    """One optimizer net: shape + run-time scalars (DM/networks.py:157-205)."""

    def __init__(self, layers: Sequence[int] = (20, 20), preprocess_name: str = "identity",
                 preprocess_options: Optional[dict] = None, scale: float = 1.0, tanh_output: bool = False,
                 n_in: int = 1):
        layers = tuple(int(h) for h in layers)
        if len(layers) > 2:
            raise L2OError("at most two LSTM layers are supported")
        if preprocess_name not in _PRE:
            raise L2OError(f"unsupported preprocess_name {preprocess_name!r}")
        opts = dict(preprocess_options or {})
        d = NetDesc()
        d.n_layers = len(layers)
        d.hidden[0] = layers[0] if len(layers) > 0 else 0
        d.hidden[1] = layers[1] if len(layers) > 1 else 0
        d.preprocess = _PRE[preprocess_name]
        d.n_in = n_in
        d.fc_dim = int(opts.get("dim", 0))
        d.logsign_k = float(opts.get("k", 0.0))
        d.scale = float(scale)
        d.tanh_output = 1 if tanh_output else 0
        self.desc = d
        self.layers = layers
        self.n_in = n_in
        self._h = C.c_void_p()
        L = _lib.lib()
        _lib.check(L.l2o_net_create(C.byref(self._h), C.byref(d)),
                   f"l2o_net_create(layers={layers}, preprocess={preprocess_name}, n_in={n_in})")
        self.n_theta = int(L.l2o_theta_count(self._h))
        self.state_floats = int(L.l2o_state_floats(self._h))

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                _lib.lib().l2o_net_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def state_size(self, n: int) -> int:
        """Floats of one state arena for n coordinates."""
        return self.state_floats * n

    def workspace_bytes(self, n: int, T: int):
        """(forward, backward) caller-owned buffer bytes for n coordinates and a T-step unroll."""
        f, b = C.c_size_t(), C.c_size_t()
        _lib.check(_lib.lib().l2o_workspace_bytes(self._h, n, T, C.byref(f), C.byref(b)), "l2o_workspace_bytes")
        return int(f.value), int(b.value)

    def set_engine(self, engine: int):
        _lib.check(_lib.lib().l2o_net_set_engine(self._h, engine), "l2o_net_set_engine")

    # ---- state arena helpers -------------------------------------------------------------
    def new_state(self, n: int, device) -> torch.Tensor:
        return torch.zeros(max(self.state_floats * n, 1), dtype=torch.float32, device=device)

    def state_views(self, arena: torch.Tensor, n: int):
        """Arena -> tuple over layers of (hidden, cell) views [n, H] (the reference's state structure)."""
        out, off = [], 0
        for h in self.layers:
            hh = arena[off:off + n * h].view(n, h)
            cc = arena[off + n * h:off + 2 * n * h].view(n, h)
            out.append((hh, cc))
            off += 2 * n * h
        return tuple(out)

    # ---- kernels -------------------------------------------------------------------------
    def step(self, theta, in0, state_in, state_out, *, in1=None, m=None, v=None, beta1=0.95, beta2=0.95, p=1.0,
             x=None, delta=None, feat_out=None, step_ptr=None, t_offset=0, reuse_weights=False):
        a = StepArgs()
        a.reuse_weights = 1 if reuse_weights else 0
        a.n = in0.numel()
        a.theta = _ptr(theta, name="theta")
        a.in0, a.in1 = _ptr(in0, name="in0"), _ptr(in1, name="in1")
        a.m, a.v = _ptr(m, name="m"), _ptr(v, name="v")
        a.beta1, a.beta2, a.p = beta1, beta2, p
        a.state_in, a.state_out = _ptr(state_in, name="state_in"), _ptr(state_out, name="state_out")
        a.x, a.delta, a.feat_out = _ptr(x, name="x"), _ptr(delta, name="delta"), _ptr(feat_out, name="feat_out")
        a.step_ptr, a.t_offset = _ptr(step_ptr, torch.int32, "step_ptr"), t_offset
        if theta.numel() != self.n_theta:
            raise L2OError(f"theta has {theta.numel()} elements, net needs {self.n_theta}")
        _lib.check(_lib.lib().l2o_step(self._h, C.byref(a), _stream()), "l2o_step")

    def unroll_fwd(self, theta, n, T, state, *, in_seq=None, opt_kind=OPT_NONE, opt_a=None, opt_b=None,
                   opt_alpha=10.0, opt_fscale=1.0, x=None, ckpt=None, m=None, v=None, beta1=0.95, beta2=0.95,
                   step0=1, g_rec=None, feat_rec=None, fx=None, delta_seq=None, labels=None, imit_loss=None,
                   n_total=0, opt_group=0):
        a = UnrollArgs()
        a.n, a.T = n, T
        a.theta = _ptr(theta, name="theta")
        a.in_seq = _ptr(in_seq, name="in_seq")
        a.opt_kind = opt_kind
        a.opt_a, a.opt_b = _ptr(opt_a, name="opt_a"), _ptr(opt_b, name="opt_b")
        a.opt_alpha, a.opt_fscale = opt_alpha, opt_fscale
        a.x, a.state, a.ckpt = _ptr(x, name="x"), _ptr(state, name="state"), _ptr(ckpt, name="ckpt")
        a.m, a.v = _ptr(m, name="m"), _ptr(v, name="v")
        a.beta1, a.beta2, a.step0 = beta1, beta2, step0
        a.g_rec, a.feat_rec = _ptr(g_rec, name="g_rec"), _ptr(feat_rec, name="feat_rec")
        a.fx = _ptr(fx, torch.float64, "fx")
        a.delta_seq, a.labels = _ptr(delta_seq, name="delta_seq"), _ptr(labels, name="labels")
        a.imit_loss = _ptr(imit_loss, torch.float64, "imit_loss")
        a.n_total = n_total
        a.opt_group = opt_group
        _lib.check(_lib.lib().l2o_unroll_fwd(self._h, C.byref(a), _stream()), "l2o_unroll_fwd")

    def unroll_bwd(self, theta, n, T, in_seq, ckpt, dtheta, *, g_rec=None, labels=None, n_total=0, delta_seq=None,
                   scratch=None):
        """BPTT over the T checkpoint slots.  ``scratch`` ([T, n, 20] floats) lets fc(20) nets (RNNProp) run on the
        tensor-core engine; ``delta_seq`` (the deltas the forward pass recorded) is what a tanh-output net's
        tensor-core BPTT differentiates the output layer with."""
        a = BwdArgs()
        a.n, a.T = n, T
        a.theta = _ptr(theta, name="theta")
        a.in_seq, a.ckpt = _ptr(in_seq, name="in_seq"), _ptr(ckpt, name="ckpt")
        a.g_rec, a.labels = _ptr(g_rec, name="g_rec"), _ptr(labels, name="labels")
        a.n_total = n_total
        a.dtheta = _ptr(dtheta, torch.float64, "dtheta")
        a.delta_seq = _ptr(delta_seq, name="delta_seq")
        if scratch is not None and scratch.numel() < T * n * 20:
            raise L2OError(f"scratch has {scratch.numel()} floats, the fc-net BPTT needs T*n*20 = {T * n * 20}")
        a.scratch = _ptr(scratch, name="scratch")
        _lib.check(_lib.lib().l2o_unroll_bwd(self._h, C.byref(a), _stream()), "l2o_unroll_bwd")


class DenseNetHandle:
    """Row-wise dense LSTM net with run-time shapes (StandardDeepLSTM with output_size > 1 = the reference's
    KernelDeepLSTM, DM/networks.py:154-236,303-351).  A variable of n = K * R elements in [kw, kh, cin, cout] order is
    R rows of K inputs (element (k, r) at k * R + r); state per ROW.  Same method surface as NetHandle where the
    meta-optimizer needs it (step / unroll_bwd / new_state / state_size)."""

    n_in = 1   # one gradient input per element (the RNNProp branches of the executor key on n_in == 2)

    def __init__(self, layers: Sequence[int], k_in: int, k_out: int, preprocess_name: str = "identity",
                 preprocess_options: Optional[dict] = None, scale: float = 1.0, tanh_output: bool = False):
        layers = tuple(int(h) for h in layers)
        if len(layers) > 2:
            raise L2OError("at most two LSTM layers are supported")
        if preprocess_name not in ("identity", "LogAndSign"):
            raise L2OError(f"unsupported preprocess_name {preprocess_name!r} for a dense net")
        d = _lib.DenseDesc()
        d.n_layers = len(layers)
        d.hidden[0] = layers[0] if len(layers) > 0 else 0
        d.hidden[1] = layers[1] if len(layers) > 1 else 0
        d.n_in, d.n_out = int(k_in), int(k_out)
        d.preprocess = _PRE[preprocess_name]
        d.logsign_k = float((preprocess_options or {}).get("k", 0.0))
        d.scale, d.tanh_output = float(scale), 1 if tanh_output else 0
        self.layers, self.k_in, self.k_out = layers, int(k_in), int(k_out)
        self._h = C.c_void_p()
        L = _lib.lib()
        _lib.check(L.l2o_dense_create(C.byref(self._h), C.byref(d)),
                   f"l2o_dense_create(layers={layers}, k_in={k_in}, k_out={k_out}, preprocess={preprocess_name})")
        self.n_theta = int(L.l2o_dense_theta_count(self._h))
        self.state_floats = int(L.l2o_dense_state_floats(self._h))   # per ROW

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                _lib.lib().l2o_dense_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def rows(self, n: int) -> int:
        if n % self.k_in:
            raise L2OError(f"{n} elements are not a whole number of rows of {self.k_in}")
        return n // self.k_in

    def state_size(self, n: int) -> int:
        return self.state_floats * self.rows(n)

    def new_state(self, n: int, device) -> torch.Tensor:
        return torch.zeros(max(self.state_size(n), 1), dtype=torch.float32, device=device)

    def state_views(self, arena: torch.Tensor, n: int):
        out, off, r = [], 0, self.rows(n)
        for h in self.layers:
            out.append((arena[off:off + r * h].view(r, h), arena[off + r * h:off + 2 * r * h].view(r, h)))
            off += 2 * r * h
        return tuple(out)

    def set_engine(self, engine: int):
        if engine == ENGINE_TC:
            raise L2OError("dense nets run on the CUDA-core engine only")

    def step(self, theta, in0, state_in, state_out, *, x=None, delta=None, reuse_weights=False, **unused):
        a = _lib.DenseStepArgs()
        a.rows = self.rows(in0.numel())
        a.theta, a.in_ = _ptr(theta, name="theta"), _ptr(in0, name="in0")
        a.state_in, a.state_out = _ptr(state_in, name="state_in"), _ptr(state_out, name="state_out")
        a.x, a.delta = _ptr(x, name="x"), _ptr(delta, name="delta")
        if theta.numel() != self.n_theta:
            raise L2OError(f"theta has {theta.numel()} elements, net needs {self.n_theta}")
        _lib.check(_lib.lib().l2o_dense_step(self._h, C.byref(a), _stream()), "l2o_dense_step")

    def unroll_bwd(self, theta, n, T, in_seq, ckpt, dtheta, *, g_rec=None, labels=None, n_total=0, delta_seq=None):
        a = _lib.DenseBwdArgs()
        a.rows, a.T = self.rows(n), T
        a.theta = _ptr(theta, name="theta")
        a.in_seq, a.ckpt = _ptr(in_seq, name="in_seq"), _ptr(ckpt, name="ckpt")
        a.g_rec, a.labels = _ptr(g_rec, name="g_rec"), _ptr(labels, name="labels")
        a.n_total = n_total
        a.dtheta = _ptr(dtheta, torch.float64, "dtheta")
        _lib.check(_lib.lib().l2o_dense_unroll_bwd(self._h, C.byref(a), _stream()), "l2o_dense_unroll_bwd")


class RuleHandle:
    """A hand-written update rule (networks.Sgd / networks.Adam, DM/networks.py:354-420) on the ``l2o_rule_*``
    kernels: state size, a fresh state, one step, a fused unroll.  No theta, no BPTT."""

    n_in = 1

    def __init__(self, kind: int, learning_rate: float, beta1: float = 0.9, beta2: float = 0.999,
                 epsilon: float = 1e-8):
        d = _lib.RuleDesc()
        d.kind, d.learning_rate, d.beta1, d.beta2, d.epsilon = kind, learning_rate, beta1, beta2, epsilon
        self.desc = d
        self.state_size(0)   # validates the descriptor (negative rate, beta outside [0, 1), unknown kind)

    def state_size(self, n: int) -> int:
        """Floats of one state arena for n coordinates (Sgd 0, Adam 4 + 2n)."""
        out = C.c_int64()
        _lib.check(_lib.lib().l2o_rule_state_floats(C.byref(self.desc), n, C.byref(out)), "l2o_rule_state_floats")
        return int(out.value)

    def new_state(self, n: int, device) -> torch.Tensor:
        return torch.zeros(max(self.state_size(n), 1), dtype=torch.float32, device=device)

    def step(self, g, state_in, state_out, *, x=None, delta=None):
        a = _lib.RuleStepArgs()
        a.n = g.numel()
        a.g = _ptr(g, name="g")
        a.state_in, a.state_out = _ptr(state_in, name="state_in"), _ptr(state_out, name="state_out")
        a.x, a.delta = _ptr(x, name="x"), _ptr(delta, name="delta")
        _lib.check(_lib.lib().l2o_rule_step(C.byref(self.desc), C.byref(a), _stream()), "l2o_rule_step")

    def unroll_fwd(self, n, T, state, *, opt_kind, opt_a, opt_b, opt_alpha=10.0, opt_fscale=1.0, x, fx=None):
        a = _lib.RuleUnrollArgs()
        a.n, a.T, a.opt_kind = n, T, opt_kind
        a.opt_a, a.opt_b = _ptr(opt_a, name="opt_a"), _ptr(opt_b, name="opt_b")
        a.opt_alpha, a.opt_fscale = opt_alpha, opt_fscale
        a.x, a.state, a.fx = _ptr(x, name="x"), _ptr(state, name="state"), _ptr(fx, torch.float64, "fx")
        _lib.check(_lib.lib().l2o_rule_unroll_fwd(C.byref(self.desc), C.byref(a), _stream()), "l2o_rule_unroll_fwd")


def adam_step(theta, dtheta, m, v, k: int, lr=0.01, beta1=0.9, beta2=0.999, eps=1e-8):
    """tf.train.AdamOptimizer update of theta in place (DM/meta.py:411-413)."""
    _lib.check(_lib.lib().l2o_adam_step(_ptr(theta, name="theta"), _ptr(dtheta, torch.float64, "dtheta"),
                                        _ptr(m, name="m"), _ptr(v, name="v"), theta.numel(), k, lr, beta1, beta2,
                                        eps, _stream()), "l2o_adam_step")


def log_and_sign(g: torch.Tensor, k: float) -> torch.Tensor:
    """preprocess.LogAndSign on a flat tensor; returns [2, n] (log row, sign row)."""
    out = torch.empty(2, g.numel(), dtype=torch.float32, device=g.device)
    _lib.check(_lib.lib().l2o_log_and_sign(_ptr(g, name="g"), _ptr(out), g.numel(), k, _stream()), "l2o_log_and_sign")
    return out


def lasso_grad(A, y, x, l1, g, f=None, scale=None):
    """f and df/dx of problems.lasso / lasso_fixed in one launch (DM/problems.py:103-175): A [B,m,n], y [B,m(,1)],
    x [B*n] flat; writes g [B*n] and accumulates the scalar loss into the fp64 tensor ``f`` (if given)."""
    a = _lib.LassoArgs()
    a.batch, a.m, a.n = int(A.shape[0]), int(A.shape[1]), int(A.shape[2])
    if x.numel() != a.batch * a.n or g.numel() != a.batch * a.n or y.numel() != a.batch * a.m:
        raise L2OError("lasso_grad: shape mismatch")
    a.A, a.y, a.x = _ptr(A, name="A"), _ptr(y, name="y"), _ptr(x, name="x")
    a.scale = _ptr(scale, name="scale")
    a.l1 = float(l1)
    a.g = _ptr(g, name="g")
    a.f = _ptr(f, torch.float64, "f")
    _lib.check(_lib.lib().l2o_lasso_grad(C.byref(a), _stream()), "l2o_lasso_grad")


_graph_replayed = 0  # kernels of this library launched through CUDA-graph replays (not visible to the C-side counter)


def note_graph_replay(kernels_in_graph: int):
    global _graph_replayed
    _graph_replayed += int(kernels_in_graph)


def launch_count() -> int:
    """Kernels of this library launched so far: direct C-ABI launches + kernels replayed inside captured graphs."""
    return int(_lib.lib().l2o_launch_count()) + _graph_replayed
