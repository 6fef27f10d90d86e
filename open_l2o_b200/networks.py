"""Optimizer networks behind the reference's ``networks`` surface (DM/networks.py).

``factory`` / ``save`` / ``Network.__call__(inputs, prev_state) -> (delta, next_state)`` /
``initial_state_for_inputs`` keep the reference's names, argument meaning and error behaviour;
the arithmetic runs in the CUDA library (one fused kernel per call instead of ~40 TF ops).
"""
from __future__ import annotations

import collections
import math
import pickle
import sys
from typing import Optional

import numpy as np
import torch

from . import engine as _engine
from ._lib import L2OError

try:  # the reference pickles with dill (DM/networks.py:25); the wire format is plain pickle-compatible
    import dill as _pickle
except Exception:  # pragma: no cover
    _pickle = pickle


def factory(net, net_options=(), net_path=None):
    """Network factory (DM/networks.py:34-44)."""
    net_class = getattr(sys.modules[__name__], net)
    net_options = dict(net_options)
    if net_path:
        with open(net_path, "rb") as f:
            net_options["initializer"] = _pickle.load(f)
    return net_class(**net_options)


def save(network, sess=None, filename=None):
    """Save the variables of a network: ``{module_name: {variable_name: ndarray}}`` (DM/networks.py:47-62)."""
    to_save = collections.defaultdict(dict)
    for (mod, var, shp), arr in zip(network.variable_shapes(), network.get_variables()):
        to_save[mod][var] = arr
    if filename:
        with open(filename, "wb") as f:
            _pickle.dump(dict(to_save), f)
    return dict(to_save)


class State(tuple):
    """Tuple over layers of (hidden, cell) views [N, H] that remembers its backing arena."""
    arena: Optional[torch.Tensor] = None


def _trunc_normal(shape, std, gen):
    t = torch.empty(shape, dtype=torch.float64)
    torch.nn.init.trunc_normal_(t, mean=0.0, std=std, a=-2 * std, b=2 * std, generator=gen)
    return t.float()


def _convert_initializer(init, shape, gen):
    """DM/networks.py:75-95: string -> tf.<name>_initializer, ndarray -> constant, else callable."""
    if isinstance(init, str):
        if init == "zeros":
            return torch.zeros(shape)
        if init == "ones":
            return torch.ones(shape)
        raise ValueError("unsupported initializer string {!r}".format(init))
    if isinstance(init, (np.ndarray, torch.Tensor)):
        return torch.as_tensor(np.asarray(init), dtype=torch.float32).reshape(shape).clone()
    if callable(init):
        return torch.as_tensor(init(shape, gen), dtype=torch.float32).reshape(shape)
    raise ValueError("unsupported initializer {!r}".format(type(init)))


def _lookup_initializer(initializers, layer_name, field):
    """DM/networks.py:98-151 (_get_initializers / _get_layer_initializers)."""
    if initializers is None:
        return None
    if isinstance(initializers, dict) and layer_name in initializers:
        initializers = initializers[layer_name]
    if isinstance(initializers, dict):
        return initializers.get(field)
    return initializers


class Network(object):
    """Base class for meta-optimizer networks (DM/networks.py:65-72)."""

    def initial_state_for_inputs(self, inputs, **kwargs):
        raise NotImplementedError


class StandardDeepLSTM(Network):
    """LSTM layers with a Linear layer on top (DM/networks.py:154-236).  Only the coordinate-wise uses
    (output_size == 1) are on the accelerated path."""

    _n_in = 1

    def __init__(self, output_size, layers, preprocess_name="identity", preprocess_options=None, scale=1.0,
                 initializer=None, name="deep_lstm", tanh_output=False, seed=0, device=None):
        if output_size != 1:
            raise NotImplementedError("only coordinate-wise nets (output_size=1) are accelerated")
        self.name = name
        self._layers = tuple(int(h) for h in layers)
        self._preprocess_name = preprocess_name
        self._preprocess_options = dict(preprocess_options or {})
        self._scale = scale
        self.tanh_output = tanh_output
        self._handle = _engine.NetHandle(layers=self._layers, preprocess_name=preprocess_name,
                                         preprocess_options=self._preprocess_options, scale=scale,
                                         tanh_output=tanh_output, n_in=self._n_in)
        self.device = torch.device(device) if device is not None else (
            torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else torch.device("cpu"))
        gen = torch.Generator().manual_seed(seed)
        parts = []
        for mod, var, shp in self.variable_shapes():
            init = _lookup_initializer(initializer, mod, var)
            if init is not None:
                t = _convert_initializer(init, shp, gen)
            elif mod.startswith("lstm"):
                fan_in = [s for m, v, s in self.variable_shapes() if m == mod and v == "w_gates"][0][0]
                t = _trunc_normal(shp, 1.0 / math.sqrt(fan_in), gen)      # Sonnet 1.x LSTM default
            elif var == "w":
                t = _trunc_normal(shp, 1.0 / math.sqrt(shp[0]), gen)      # Sonnet Linear default
            else:
                t = torch.zeros(shp)
            parts.append(t.reshape(-1))
        self.theta = torch.cat(parts).to(self.device).contiguous()
        assert self.theta.numel() == self._handle.n_theta

    # ---- variables ---------------------------------------------------------------------------
    @property
    def feat(self):
        if self._preprocess_name == "fc":
            return int(self._preprocess_options["dim"])
        if self._preprocess_name == "LogAndSign":
            return 2 * self._n_in
        return self._n_in

    def variable_shapes(self):
        """(module, variable, shape) in Sonnet creation order == flat theta order."""
        out = []
        if self._preprocess_name == "fc":
            out += [("input_projection", "w", (self._n_in, self.feat)), ("input_projection", "b", (self.feat,))]
        k = self.feat
        for i, h in enumerate(self._layers, start=1):
            out += [("lstm_{}".format(i), "w_gates", (k + h, 4 * h)), ("lstm_{}".format(i), "b_gates", (4 * h,))]
            k = h
        out += [("linear", "w", (k, 1)), ("linear", "b", (1,))]
        return out

    def get_variables(self):
        th = self.theta.detach().cpu().numpy()
        out, off = [], 0
        for _, _, shp in self.variable_shapes():
            n = int(np.prod(shp))
            out.append(th[off:off + n].reshape(shp).copy())
            off += n
        return out

    def set_variables(self, data):
        """``data``: {module: {var: ndarray}} (the .l2l format)."""
        parts = [torch.as_tensor(np.asarray(data[m][v]), dtype=torch.float32).reshape(-1)
                 for m, v, _ in self.variable_shapes()]
        self.theta.copy_(torch.cat(parts).to(self.theta.device))

    @property
    def handle(self):
        return self._handle

    # ---- operator surface --------------------------------------------------------------------
    def _reshape_inputs(self, inputs):
        return inputs.reshape(-1)

    def _state_arena(self, prev_state, n):
        arena = getattr(prev_state, "arena", None)
        if arena is not None:
            return arena
        parts = []
        for h, c in prev_state:
            parts += [h.reshape(-1), c.reshape(-1)]
        return torch.cat(parts).contiguous() if parts else torch.zeros(1, device=self.theta.device)

    def _wrap_state(self, arena, n):
        st = State(self._handle.state_views(arena, n))
        st.arena = arena
        return st

    def __call__(self, inputs, prev_state):
        """delta, next_state = net(gradients, prev_state) (DM/networks.py:207-232, 254-271)."""
        flat = self._reshape_inputs(inputs).contiguous()
        n = flat.numel()
        arena_in = self._state_arena(prev_state, n)
        arena_out = torch.empty_like(arena_in)
        delta = torch.empty(n, dtype=torch.float32, device=flat.device)
        self._handle.step(self.theta, flat, arena_in, arena_out, delta=delta)
        return delta.reshape(inputs.shape), self._wrap_state(arena_out, n)

    def initial_state_for_inputs(self, inputs, **kwargs):
        """Zero (hidden, cell) per layer, batch = number of coordinates (DM/networks.py:234-236, 273-276)."""
        n = int(np.prod(inputs.shape)) if len(inputs.shape) else 1
        return self._wrap_state(self._handle.new_state(n, self.theta.device), n)


class CoordinateWiseDeepLSTM(StandardDeepLSTM):
    """Coordinate-wise ``DeepLSTM`` (DM/networks.py:239-276)."""

    def __init__(self, name="cw_deep_lstm", **kwargs):
        super(CoordinateWiseDeepLSTM, self).__init__(1, name=name, **kwargs)


class RNNprop(StandardDeepLSTM):
    """DM/networks.py:279-300: net(m, g, prev_state), inputs stacked in the order (m~, g~)."""

    _n_in = 2

    def __init__(self, name="RNNprop", **kwargs):
        super(RNNprop, self).__init__(1, name=name, **kwargs)

    def __call__(self, m, g, prev_state):
        mf, gf = m.reshape(-1).contiguous(), g.reshape(-1).contiguous()
        n = gf.numel()
        arena_in = self._state_arena(prev_state, n)
        arena_out = torch.empty_like(arena_in)
        delta = torch.empty(n, dtype=torch.float32, device=gf.device)
        self._handle.step(self.theta, mf, arena_in, arena_out, in1=gf, delta=delta)
        return delta.reshape(g.shape), self._wrap_state(arena_out, n)


class KernelDeepLSTM(Network):
    """``DeepLSTM`` for convolutional filters (DM/networks.py:303-351): the input is a filter bank
    [kernel_w, kernel_h, n_input_channels, n_output_channels]; every (input, output) channel pair is one ROW whose
    kernel_w*kernel_h entries are the LSTM's inputs, and the output Linear produces the row's kernel_w*kernel_h updates.
    Runs on the run-time-shaped dense engine (``l2o_dense_*``)."""

    per_variable = True   # one run per optimizee variable (rows differ per filter bank)

    def __init__(self, kernel_shape, layers, preprocess_name="identity", preprocess_options=None, scale=1.0,
                 initializer=None, name="kernel_deep_lstm", tanh_output=False, seed=0, device=None):
        self.name = name
        self._kernel_shape = list(kernel_shape)
        self._k = int(np.prod(kernel_shape))
        self._layers = tuple(int(h) for h in layers)
        self._preprocess_name = preprocess_name
        self._preprocess_options = dict(preprocess_options or {})
        self._handle = _engine.DenseNetHandle(self._layers, self._k, self._k, preprocess_name=preprocess_name,
                                              preprocess_options=self._preprocess_options, scale=scale,
                                              tanh_output=tanh_output)
        self.device = torch.device(device) if device is not None else (
            torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else torch.device("cpu"))
        gen = torch.Generator().manual_seed(seed)
        parts = []
        for mod, var, shp in self.variable_shapes():
            init = _lookup_initializer(initializer, mod, var)
            if init is not None:
                t = _convert_initializer(init, shp, gen)
            elif mod.startswith("lstm"):     # Sonnet 1.x LSTM default: TruncatedNormal(1/sqrt(fan_in)) for w and b
                fan_in = [s_ for m, v, s_ in self.variable_shapes() if m == mod and v == "w_gates"][0][0]
                t = _trunc_normal(shp, 1.0 / math.sqrt(fan_in), gen)
            elif var == "w":                 # Sonnet Linear default
                t = _trunc_normal(shp, 1.0 / math.sqrt(shp[0]), gen)
            else:
                t = torch.zeros(shp)
            parts.append(t.reshape(-1))
        self.theta = torch.cat(parts).to(self.device).contiguous()
        assert self.theta.numel() == self._handle.n_theta

    @property
    def handle(self):
        return self._handle

    @property
    def feat(self):
        return 2 * self._k if self._preprocess_name == "LogAndSign" else self._k

    def variable_shapes(self):
        out, k = [], self.feat
        for i, h in enumerate(self._layers, start=1):
            out += [("lstm_{}".format(i), "w_gates", (k + h, 4 * h)), ("lstm_{}".format(i), "b_gates", (4 * h,))]
            k = h
        out += [("linear", "w", (k, self._k)), ("linear", "b", (self._k,))]
        return out

    get_variables = StandardDeepLSTM.get_variables
    set_variables = StandardDeepLSTM.set_variables

    def _check(self, inputs):
        if inputs.dim() != 4 or list(inputs.shape[:2]) != self._kernel_shape:
            raise ValueError("KernelDeepLSTM expects a [kw, kh, cin, cout] tensor with kernel shape {}; got {}".format(
                self._kernel_shape, list(inputs.shape)))

    def initial_state_for_inputs(self, inputs, **kwargs):
        """Batch size = n_input_channels * n_output_channels (DM/networks.py:347-351)."""
        self._check(inputs)
        n = inputs.numel()
        arena = self._handle.new_state(n, self.theta.device)
        st = State(self._handle.state_views(arena, n))
        st.arena = arena
        return st

    def __call__(self, inputs, prev_state):
        """update, next_state = net(filter_gradient, prev_state) (DM/networks.py:329-346)."""
        self._check(inputs)
        flat = inputs.contiguous().reshape(-1)     # element (k, r) at k * R + r: the transposes are index arithmetic
        n = flat.numel()
        arena_in = getattr(prev_state, "arena", None)
        if arena_in is None:
            arena_in = torch.cat([t.reshape(-1) for hc in prev_state for t in hc]).contiguous()
        arena_out = torch.empty_like(arena_in)
        delta = torch.empty(n, dtype=torch.float32, device=flat.device)
        self._handle.step(self.theta, flat, arena_in, arena_out, delta=delta)
        st = State(self._handle.state_views(arena_out, n))
        st.arena = arena_out
        return delta.reshape(inputs.shape), st


class _Rule(Network):
    """A hand-written update rule: no trainable variables, no theta; the step runs in ``l2o_rule_step``."""

    def variable_shapes(self):
        return []

    def get_variables(self):
        return []

    def set_variables(self, data):
        pass

    @property
    def handle(self):
        return self._handle

    def _step(self, g, arena_in=None):
        flat = g.reshape(-1).contiguous()
        arena_out = torch.empty_like(arena_in) if arena_in is not None else None
        delta = torch.empty_like(flat)
        self._handle.step(flat, arena_in, arena_out, delta=delta)
        return delta.reshape(g.shape), arena_out


class Sgd(_Rule):
    """Identity network which acts like SGD: update = -learning_rate * g (DM/networks.py:354-371)."""

    def __init__(self, learning_rate=0.001, name="sgd"):
        self.name = name
        self._learning_rate = learning_rate
        self._handle = _engine.RuleHandle(_engine.RULE_SGD, learning_rate)

    def __call__(self, inputs, prev_state):
        return self._step(inputs)[0], []

    def initial_state_for_inputs(self, inputs, **kwargs):
        return []


class Adam(_Rule):
    """Adam as an optimizer net (DM/networks.py:374-420).  State (t, m, v): a 0-d step counter and [N, 1] moments,
    views of one arena [t, pad, pad, pad | m | v] (include/l2o_b200.h)."""

    def __init__(self, learning_rate=1e-3, beta1=0.9, beta2=0.999, epsilon=1e-8, name="adam"):
        self.name = name
        self._learning_rate, self._beta1, self._beta2, self._epsilon = learning_rate, beta1, beta2, epsilon
        self._handle = _engine.RuleHandle(_engine.RULE_ADAM, learning_rate, beta1, beta2, epsilon)

    @staticmethod
    def state_views(arena, n):
        return arena[0], arena[4:4 + n].view(n, 1), arena[4 + n:4 + 2 * n].view(n, 1)

    def _wrap_state(self, arena, n):
        st = State(self.state_views(arena, n))
        st.arena = arena
        return st

    def __call__(self, g, prev_state):
        n = g.numel()
        arena = getattr(prev_state, "arena", None)
        if arena is None:
            t, m, v = prev_state
            arena = torch.cat([t.reshape(1).float(), torch.zeros(3, device=g.device), m.reshape(-1).float(),
                               v.reshape(-1).float()]).contiguous()
        update, arena_out = self._step(g, arena)
        return update, self._wrap_state(arena_out, n)

    def initial_state_for_inputs(self, inputs, **kwargs):
        n = int(np.prod(inputs.shape)) if len(inputs.shape) else 1
        return self._wrap_state(self._handle.new_state(n, inputs.device), n)
