"""Learning-to-learn (meta) optimizer behind the reference's ``MetaOptimizer`` surface (DM/meta.py).

The reference builds a TF graph and crosses the device boundary once per unroll with
``sess.run([cost, update, step])``.  Here ``meta_loss`` / ``meta_minimize`` return lightweight op
handles and ``Session.run`` executes one fused unroll (forward T steps [+ BPTT + Adam] + carry-over)
with the same fetch semantics:

  * all fetches of one ``run`` are evaluated from the same pre-update theta / x / state
    (TF evaluates ``update`` and ``step`` in the same step as ``cost``);
  * ``update`` commits x <- x_T, state <- s_T (truncated-BPTT carry-over, DM/meta.py:385-389);
  * ``step`` applies TF-Adam to the optimizer nets' variables (DM/meta.py:411-413);
  * ``reset`` re-runs the initializers of state + x + constants (DM/meta.py:378-383).

Two regimes (DESIGN.md): *fused* (separable optimizee evaluated in-kernel, one launch for all T steps) and
*external-gradient* (torch autograd between single-step launches, state checkpointed in HBM).
"""
from __future__ import annotations

import collections
import os

import numpy as np
import torch

from . import engine as _engine
from . import networks
from .variables import variable_getter

_PRODUCER_KINDS = ("lasso_batch", "mlp_xent")
MetaLoss = collections.namedtuple("MetaLoss", "loss, update, reset, fx, x")
MetaStep = collections.namedtuple("MetaStep", "step, update, reset, fx, x")


class Op(object):
    """Handle returned in MetaLoss / MetaStep; evaluated by Session.run."""

    def __init__(self, kind, program):
        self.kind, self.program = kind, program

    def __repr__(self):
        return "<l2o op {}>".format(self.kind)


class Placeholder(object):
    def __init__(self, name):
        self.name = name


class Session(object):
    """Minimal stand-in for tf.Session: ``run(fetches, feed_dict)``."""

    def run(self, fetches, feed_dict=None):
        flat = []

        def walk(f):
            if isinstance(f, (list, tuple)):
                for g in f:
                    walk(g)
            elif isinstance(f, Op):
                flat.append(f)
            elif f is not None:
                raise TypeError("cannot fetch {!r}".format(f))
        walk(fetches)
        results = {}
        for prog in {id(op.program): op.program for op in flat}.values():
            kinds = set(op.kind for op in flat if op.program is prog)
            results[id(prog)] = prog.execute(kinds, feed_dict or {})

        def build(f):
            if isinstance(f, list):
                return [build(g) for g in f]
            if isinstance(f, tuple):
                return tuple(build(g) for g in f)
            if f is None:
                return None
            return results[id(f.program)].get(f.kind)
        return build(fetches)

    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


# ------------------------------------------------------------------------------------------------
def _get_variables(func, gen, device):
    """Call ``func`` once, capturing the tensors it creates (DM/meta.py:102-128).
    Returns (variables, constants): lists of dicts {name, shape, init}."""
    variables, constants = [], []

    def getter(name, shape, dtype, initializer, trainable):
        if initializer is None:
            raise ValueError("variable {!r} needs an initializer".format(name))
        rec = dict(name=name, shape=shape, init=initializer)
        (variables if trainable else constants).append(rec)
        return initializer(shape, gen).to(device=device, dtype=torch.float32)

    with variable_getter(getter), torch.no_grad():
        func()
    return variables, constants


def _make_nets(variables, config, net_assignments):
    """DM/meta.py:162-216, same errors."""
    name_to_index = dict((v["name"], i) for i, v in enumerate(variables))
    if net_assignments is None:
        if len(config) != 1:
            raise ValueError("Default net_assignments can only be used if there is a single net config.")
        key = next(iter(config))
        nets = {key: networks.factory(**config[key])}
        keys, subsets = [key], [list(range(len(variables)))]
    else:
        nets, keys, subsets = {}, [], []
        for key, names in net_assignments:
            if key in nets:
                raise ValueError("Repeated netid in net_assigments.")
            nets[key] = networks.factory(**config[key])
            subsets.append([name_to_index[name] for name in names])
            keys.append(key)
    return nets, keys, subsets


def _is_rule(net):
    """Sgd / Adam: a hand-written rule, nothing to train and nothing to differentiate through."""
    return isinstance(net, networks._Rule)


class _Run(object):
    """A maximal contiguous slice of the flat coordinate arena served by one net."""

    def __init__(self, key, net, off, n):
        self.key, self.net, self.off, self.n = key, net, off, n


class _Program(object):
    """One meta_loss graph: variables, nets, state, workspaces and the unroll executor."""

    def __init__(self, optimizer, make_loss, len_unroll, net_assignments, second_derivatives, learning_rate=None):
        if second_derivatives:
            raise NotImplementedError("second_derivatives=True needs optimizee Hessian-vector products "
                                      "(out of scope, SURVEY.md Appendix B)")
        if not torch.cuda.is_available():
            raise _engine.L2OError("MetaOptimizer needs a CUDA device (no CPU path)")
        self.opt = optimizer
        self.make_loss = make_loss
        self.T = int(len_unroll)
        self.device = torch.device("cuda", torch.cuda.current_device())
        self.gen = torch.Generator().manual_seed(optimizer.seed)
        self.learning_rate = learning_rate
        self.variables, self.constants = _get_variables(make_loss, torch.Generator().manual_seed(optimizer.seed),
                                                        self.device)
        print("Optimizee variables")
        print([v["name"] for v in self.variables])
        print("Problem variables")
        print([c["name"] for c in self.constants])
        self.nets, self.net_keys, self.subsets = _make_nets(self.variables, optimizer._config, net_assignments)
        optimizer._nets = self.nets
        if any(_is_rule(net) for net in self.nets.values()):
            if optimizer.rnnprop:
                raise NotImplementedError("Sgd / Adam nets in an RNNProp program: every net there is called as "
                                          "net(m, g, state), which a hand-written rule does not take")
            if optimizer.distributed:
                raise NotImplementedError("Sgd / Adam nets in a sharded (_distributed=True) program")
        # the nets with trainable variables: only they get a meta-gradient accumulator and meta-Adam slots
        self.learned = {k: net for k, net in self.nets.items() if not _is_rule(net)}

        # flat arena: variables ordered so that each net's subset is contiguous where possible
        order = []
        for subset in self.subsets:
            for j in subset:
                if j not in order:
                    order.append(j)
        for j in range(len(self.variables)):
            if j not in order:
                order.append(j)
        self.var_off, off = {}, 0
        for j in order:
            self.var_off[j] = off
            off += int(np.prod(self.variables[j]["shape"])) if self.variables[j]["shape"] else 1
        self.N = off
        self.runs = []
        for key, subset in zip(self.net_keys, self.subsets):
            cur = None
            for j in subset:
                n = int(np.prod(self.variables[j]["shape"])) if self.variables[j]["shape"] else 1
                o = self.var_off[j]
                if cur is not None and cur.off + cur.n == o and not getattr(self.nets[key], "per_variable", False):
                    cur.n += n
                else:
                    cur = _Run(key, self.nets[key], o, n)
                    self.runs.append(cur)
        self.X = torch.zeros(self.N, device=self.device)
        self.const_vals = {}
        self.fused = getattr(make_loss, "fused", None) if os.environ.get("L2O_DISABLE_FUSED") != "1" else None
        one_net = len(self.runs) == 1 and self.runs[0].n == self.N
        if self.fused is not None and not (one_net and (len(self.variables) == 1 or self.fused.kind == "mlp_xent")):
            self.fused = None
        if self.fused is not None and self.fused.kind == "quadratic_batch" and _is_rule(self.runs[0].net):
            self.fused = None   # the rule unroll has no dense-group optimizee: step at a time instead
        # "producer" optimizees (SURVEY.md 8(f) row 4): f and df/dx come from ONE library kernel per step instead of
        # torch autograd (~15 launches); the unroll stays step-at-a-time (the gradient couples coordinates) and is
        # captured into one CUDA graph like every external-gradient unroll
        self.producer = None
        if self.fused is not None and self.fused.kind in _PRODUCER_KINDS:
            self.producer, self.fused = self.fused, None
        self.adam = {k: dict(m=torch.zeros_like(net.theta), v=torch.zeros_like(net.theta), k=0)
                     for k, net in self.learned.items()}
        self.dtheta = {k: torch.zeros(net.theta.numel(), dtype=torch.float64, device=self.device)
                       for k, net in self.learned.items()}
        self.step_placeholder = Placeholder("step")
        # per-variable scale placeholders (random-scaling trick, DM/meta_dm_train.py:336-338,384-385): fx = f(x * scale)
        self.scale_placeholders = [Placeholder(v["name"] + "_scale") for v in self.variables]
        self.scale_flat = torch.ones(self.N, device=self.device)
        self.step_dev = torch.ones(1, dtype=torch.int32, device=self.device)  # step0 of the current unroll (RNNProp)
        self.scale_active = False
        self.mt_tasks = []
        self.unroll_idx = 0
        self._graphs, self._eager_calls, self._graph_failed, self._graph_kernels = {}, {}, False, {}
        self._alloc_workspaces()
        self.reset()

    # ---- memory ---------------------------------------------------------------------------------
    def _alloc_workspaces(self):
        T = self.T
        for r in self.runs:
            r.state = r.net.handle.new_state(r.n, self.device)
            r.rule = _is_rule(r.net)
            if r.rule:
                # no checkpoints, no recorded gradients, no BPTT scratch: the state ping-pongs between two arenas
                r.pp = (r.net.handle.new_state(r.n, self.device), r.net.handle.new_state(r.n, self.device))
                r.x_work = torch.zeros(r.n, device=self.device)
                continue
            r.ckpt = torch.zeros((T + 1) * max(r.net.handle.state_size(r.n), 1), device=self.device)
            r.g_rec = torch.zeros(T + 1, r.n, device=self.device)
            r.x_work = torch.zeros(r.n, device=self.device)
            if r.net.handle.n_in == 2:
                r.m = torch.zeros(r.n, device=self.device)
                r.v = torch.zeros(r.n, device=self.device)
                r.m_work, r.v_work = torch.zeros_like(r.m), torch.zeros_like(r.v)
                r.feat_rec = torch.zeros(T, 2, r.n, device=self.device)
            # what the tensor-core BPTT of a tanh-output / fc(20) net (RNNProp) needs on top: the recorded deltas
            # (tanh' of the output layer) and the hand-over buffer between its layer-2 and layer-1 pass
            r.delta_rec = r.bwd_scratch = None
            h = r.net.handle
            if getattr(r.net, "tanh_output", False) and isinstance(h, _engine.NetHandle):
                r.delta_rec = torch.zeros(T, r.n, device=self.device)
            if h.n_in == 2 and isinstance(h, _engine.NetHandle) and tuple(h.layers) == (20, 20):
                r.bwd_scratch = torch.zeros(T, r.n, 20, device=self.device)
        self.fx_buf = torch.zeros(T + 1, dtype=torch.float64, device=self.device)

    def reset_x(self):
        """Re-run the initializers of x + constants only (``reset_x`` of DM/data_generator.py:50,80).  The tensors are
        refilled IN PLACE: captured CUDA graphs and views handed out earlier keep pointing at live, current data."""
        for v, j in zip(self.variables, range(len(self.variables))):
            n = int(np.prod(v["shape"])) if v["shape"] else 1
            o = self.var_off[j]
            self.X[o:o + n].copy_(v["init"](v["shape"], self.gen).reshape(-1).to(self.device))
        for c in self.constants:
            new = c["init"](c["shape"], self.gen).to(torch.float32).contiguous()
            cur = self.const_vals.get(c["name"])
            if cur is None or cur.shape != new.shape:
                self.const_vals[c["name"]] = new.to(self.device)
            else:
                cur.copy_(new)

    def reset(self):
        """variables_initializer(state + x + constants) (DM/meta.py:378-383)."""
        self.reset_x()
        for r in self.runs:
            r.state.zero_()
            if r.net.handle.n_in == 2:
                r.m.zero_()
                r.v.zero_()
        self.unroll_idx = 0

    # ---- optimizee evaluation --------------------------------------------------------------------
    def _var_views(self, Xflat):
        """The optimizee variables as views of the flat arena (creation order)."""
        out = []
        for j, v in enumerate(self.variables):
            n = int(np.prod(v["shape"])) if v["shape"] else 1
            o = self.var_off[j]
            out.append(Xflat[o:o + n].view(v["shape"]))
        return out

    def _loss_from_vars(self, var_list):
        """_make_with_custom_variables (DM/meta.py:131-155): trainables popped in creation order."""
        queue = collections.deque(range(len(self.variables)))

        def getter(name, shape, dtype, initializer, trainable):
            if trainable:
                return var_list[queue.popleft()]
            return self.const_vals[name]

        if self.scale_active:   # x (.) scale of the enhanced recipe (DM/meta_dm_train.py:336-338,384-385)
            var_list = [v * sc for v, sc in zip(var_list, self._var_views(self.scale_flat))]
        with variable_getter(getter):
            return self.make_loss()

    def _loss_at(self, Xflat):
        return self._loss_from_vars(self._var_views(Xflat))

    def _apply_scale_feed(self, feed):
        fed = [p for p in self.scale_placeholders if p in feed]
        if not fed:
            if self.scale_active:
                self.scale_flat.fill_(1.0)
                self.scale_active = False
            return
        self.scale_flat.fill_(1.0)
        for j, p in enumerate(self.scale_placeholders):
            if p in feed:
                n = int(np.prod(self.variables[j]["shape"])) if self.variables[j]["shape"] else 1
                o = self.var_off[j]
                self.scale_flat[o:o + n].copy_(torch.as_tensor(np.asarray(feed[p], dtype=np.float32)).reshape(-1))
        self.scale_active = True

    def assign_x(self, values):
        """assign_func of DM/train_dm.py:101-113: overwrite the optimizee variables (list in creation order)."""
        for j, val in enumerate(values):
            n = int(np.prod(self.variables[j]["shape"])) if self.variables[j]["shape"] else 1
            o = self.var_off[j]
            self.X[o:o + n].copy_(torch.as_tensor(np.asarray(val, dtype=np.float32)).reshape(-1))

    def x_values(self):
        return [self.X[self.var_off[j]:self.var_off[j] + (int(np.prod(v["shape"])) if v["shape"] else 1)]
                .reshape(v["shape"]).cpu().numpy() for j, v in enumerate(self.variables)]

    def _produce(self, Xflat):
        """f(x) and df/dx from the fused producer kernel (one launch)."""
        p = self.producer
        g = torch.empty_like(Xflat)
        fx = torch.zeros((), dtype=torch.float64, device=self.device)
        if p.kind == "lasso_batch":
            _engine.lasso_grad(self.const_vals[p.a], self.const_vals[p.b], Xflat, p.alpha, g, f=fx,
                               scale=self.scale_flat if self.scale_active else None)
        elif p.kind == "mlp_xent":
            from .problems import mlp_value_and_grad
            with torch.no_grad():
                xs = Xflat * self.scale_flat if self.scale_active else Xflat    # f(x (.) scale), DM/meta_dm_train.py:384
                fx = mlp_value_and_grad(self._var_views(xs), self.const_vals[p.a], self.const_vals[p.b],
                                        p.extra["activation"], self._var_views(g)).double()
                if self.scale_active:
                    g.mul_(self.scale_flat)
        else:
            raise ValueError(p.kind)
        return fx, g

    def _value_and_grad(self, Xflat):
        """f(x) and df/dx as a flat [N] tensor.  Each variable is its own autograd leaf (a view of the arena), so the
        backward pass produces one gradient per variable and never materialises zero-filled [N] tensors."""
        if self.producer is not None:
            return self._produce(Xflat)
        leaves = [v.detach().requires_grad_(True) for v in self._var_views(Xflat)]
        with torch.enable_grad():
            fx = self._loss_from_vars(leaves)
            grads = torch.autograd.grad(fx, leaves, allow_unused=True)
        g = torch.empty_like(Xflat)
        for gv, gj in zip(self._var_views(g), grads):
            if gj is None:
                gv.zero_()
            else:
                gv.copy_(gj)
        return fx.detach(), g

    # ---- the unroll --------------------------------------------------------------------------------
    def _step0(self, feed):
        if self.step_placeholder in feed:
            return int(feed[self.step_placeholder])
        return self.unroll_idx * self.T + 1

    def _forward_fused(self, train, step0):
        r, T, f = self.runs[0], self.T, self.fused
        h = r.net.handle
        r.x_work.copy_(self.X)
        if r.rule:
            r.pp[0].copy_(r.state)
            self.fx_buf.zero_()
            h.unroll_fwd(r.n, T, r.pp[0], opt_kind=_engine.OPT_KINDS[f.kind],
                         opt_a=self.const_vals[f.a].reshape(-1), opt_b=self.const_vals[f.b].reshape(-1),
                         opt_alpha=f.alpha, opt_fscale=f.fscale, x=r.x_work, fx=self.fx_buf)
            r.state_final = r.pp[0]
            return self.fx_buf
        state = r.ckpt[:max(h.state_size(r.n), 1)]
        work_state = r.state.clone()
        self.fx_buf.zero_()
        kw = {}
        if h.n_in == 2:
            r.m_work.copy_(r.m)
            r.v_work.copy_(r.v)
            kw = dict(m=r.m_work, v=r.v_work, beta1=self.opt.beta1, beta2=self.opt.beta2, step0=step0,
                      feat_rec=r.feat_rec)
        if train and r.delta_rec is not None:
            kw["delta_seq"] = r.delta_rec
        h.unroll_fwd(r.net.theta, r.n, T, work_state, opt_kind=_engine.OPT_KINDS[f.kind],
                     opt_a=self.const_vals[f.a].reshape(-1), opt_b=self.const_vals[f.b].reshape(-1),
                     opt_alpha=f.alpha, opt_fscale=f.fscale, x=r.x_work, ckpt=r.ckpt if train else None,
                     g_rec=r.g_rec, fx=self.fx_buf, opt_group=getattr(f, "group", 0), **kw)
        del state
        r.state_final = work_state
        return self.fx_buf

    def _forward_external(self, train, step0):
        T = self.T
        Xw = self.X.clone()
        fxs = []
        for r in self.runs:
            if r.rule:
                r.pp[0].copy_(r.state)
                continue
            r.ckpt[:max(r.net.handle.state_size(r.n), 1)].copy_(r.state)
            if r.net.handle.n_in == 2:
                r.m_work.copy_(r.m)
                r.v_work.copy_(r.v)
        for t in range(T):
            fx, g = self._value_and_grad(Xw)
            fxs.append(fx)
            for r in self.runs:
                h = r.net.handle
                if r.rule:
                    h.step(g[r.off:r.off + r.n], r.pp[t % 2], r.pp[(t + 1) % 2], x=Xw[r.off:r.off + r.n])
                    continue
                slot = max(h.state_size(r.n), 1)
                r.g_rec[t].copy_(g[r.off:r.off + r.n])
                kw = {}
                if h.n_in == 2:
                    kw = dict(m=r.m_work, v=r.v_work, beta1=self.opt.beta1, beta2=self.opt.beta2,
                              step_ptr=self.step_dev, t_offset=t, feat_out=r.feat_rec[t])
                if train and r.delta_rec is not None:
                    kw["delta"] = r.delta_rec[t]
                # theta is constant inside an unroll: the weight image built at t = 0 serves every later step (runs that
                # share a net share its handle, so only the first run of step 0 rebuilds)
                h.step(r.net.theta, r.g_rec[t], r.ckpt[t * slot:(t + 1) * slot], r.ckpt[(t + 1) * slot:(t + 2) * slot],
                       x=Xw[r.off:r.off + r.n], reuse_weights=(t > 0), **kw)
        if train:
            fx, g = self._value_and_grad(Xw)
            for r in self.runs:
                if not r.rule:
                    r.g_rec[T].copy_(g[r.off:r.off + r.n])
        else:
            if self.producer is not None:
                fx = self._produce(Xw)[0]
            else:
                with torch.no_grad():
                    fx = self._loss_at(Xw)
        fxs.append(fx)
        for r in self.runs:
            if r.rule:
                r.state_final = r.pp[T % 2]
            else:
                slot = max(r.net.handle.state_size(r.n), 1)
                r.state_final = r.ckpt[T * slot:(T + 1) * slot]
            r.x_work = Xw[r.off:r.off + r.n]
        self._Xw = Xw
        return torch.stack([f.reshape(()).double() for f in fxs])

    # ---- CUDA-graph path of the external-gradient regime ------------------------------------------------
    def _graph_body(self, train, step0):
        """Everything of one unroll that is launch-bound and shape-static: T x (autograd + step kernel) [+ BPTT]."""
        fx = self._forward_external(train, step0)
        if train:
            for d in self.dtheta.values():
                d.zero_()
            for r in self.runs:
                if r.rule:
                    continue
                h = r.net.handle
                in_seq = r.feat_rec if h.n_in == 2 else r.g_rec
                h.unroll_bwd(r.net.theta, r.n, self.T, in_seq, r.ckpt, self.dtheta[r.key], g_rec=r.g_rec,
                             **self._bwd_extra(r))
        return fx

    @staticmethod
    def _bwd_extra(r):
        kw = {}
        if r.delta_rec is not None:
            kw["delta_seq"] = r.delta_rec
        if r.bwd_scratch is not None:
            kw["scratch"] = r.bwd_scratch
        return kw

    def _graph_eligible(self):
        # RNNProp's bias-correction exponent p = step0 + t is read from a device scalar (self.step_dev), so the graph
        # stays valid from unroll to unroll
        return os.environ.get("L2O_CUDA_GRAPH", "1") != "0" and self.fused is None and not self.scale_active

    def _run_external(self, train, step0):
        """Eager on the first two calls (warm-up: lazy allocations, autograd caches), then capture once per mode and
        replay: the per-step launches (~15 tiny kernels) collapse into one graph launch."""
        self.step_dev.fill_(int(step0))
        key = bool(train)
        if not self._graph_eligible() or self._graph_failed:
            return self._graph_body(train, step0)
        self._eager_calls[key] = self._eager_calls.get(key, 0) + 1
        if self._eager_calls[key] <= 2:
            return self._graph_body(train, step0)
        if key not in self._graphs:
            try:
                # garbage from earlier programs (their CUDAGraph objects free device memory when collected) must not be
                # finalised in the middle of this capture: a cudaFree during capture invalidates it
                import gc
                gc.collect()
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                n0 = _engine.launch_count()
                with torch.cuda.graph(g):
                    fx = self._graph_body(train, step0)
                self._graph_kernels[key] = _engine.launch_count() - n0   # library kernels recorded in this graph
                self._graphs[key] = (g, fx, self._Xw, [r.state_final for r in self.runs], [r.x_work for r in self.runs])
            except Exception as e:  # capture not possible for this optimizee: keep running the same kernels eagerly
                import warnings
                warnings.warn("CUDA-graph capture of the unroll failed (%r); staying eager" % (e,))
                self._graph_failed = True
                torch.cuda.synchronize()
                return self._graph_body(train, step0)
        g, fx, xw, finals, xworks = self._graphs[key]
        g.replay()
        _engine.note_graph_replay(self._graph_kernels[key])
        self._Xw = xw
        for r, f, xk in zip(self.runs, finals, xworks):
            r.state_final, r.x_work = f, xk
        return fx

    def execute(self, kinds, feed):
        if kinds == {"reset"}:
            self.reset()
            return {}
        if "reset" in kinds:
            raise ValueError("fetch `reset` on its own (the reference runs it separately, DM/util.py:37)")
        mt_kinds = set(k for k in kinds if ":" in k)
        if mt_kinds:
            out = {}
            for ti in sorted(set(int(k.split(":")[1]) for k in mt_kinds)):
                out.update(self.mt_tasks[ti].execute(set(k.split(":")[0] for k in mt_kinds if int(k.split(":")[1]) == ti), feed))
            kinds = kinds - mt_kinds
            if not kinds:
                return out
            out.update(self.execute(kinds, feed))
            return out
        train = "step" in kinds
        commit = "update" in kinds
        step0 = self._step0(feed)
        T = self.T
        out = {}
        self._apply_scale_feed(feed)
        if self.fused is not None and not self.scale_active:
            fx = self._forward_fused(train, step0)
            if train:
                for d in self.dtheta.values():
                    d.zero_()
                for r in self.runs:
                    if r.rule:
                        continue
                    h = r.net.handle
                    in_seq = r.feat_rec if h.n_in == 2 else r.g_rec
                    h.unroll_bwd(r.net.theta, r.n, T, in_seq, r.ckpt, self.dtheta[r.key], g_rec=r.g_rec,
                                 **self._bwd_extra(r))
        else:
            fx = self._run_external(train, step0)
        if train:
            if self.opt.distributed:
                from .dist import allreduce_meta_grad
                fx = allreduce_meta_grad(self.dtheta, fx)
        elif self.opt.distributed:
            import torch.distributed as dist
            fx = fx.clone()
            dist.all_reduce(fx)
        if "loss" in kinds:
            out["loss"] = float(fx.sum().item())
        if "fx" in kinds:
            out["fx"] = float(fx[T].item())
        used_fused = self.fused is not None and not self.scale_active
        if "x" in kinds:
            xf = self.runs[0].x_work if used_fused else self._Xw
            out["x"] = [xf[self.var_off[j]:self.var_off[j] + (int(np.prod(v["shape"])) if v["shape"] else 1)]
                        .reshape(v["shape"]).cpu().numpy() for j, v in enumerate(self.variables)]
        self.last_fx = fx
        if train:
            for k, net in self.learned.items():
                ad = self.adam[k]
                ad["k"] += 1
                _engine.adam_step(net.theta, self.dtheta[k], ad["m"], ad["v"], ad["k"], lr=self.learning_rate)
            out["step"] = None
        if commit:
            if used_fused:
                self.X.copy_(self.runs[0].x_work)
            else:
                self.X.copy_(self._Xw)
            for r in self.runs:
                r.state.copy_(r.state_final)
                if r.net.handle.n_in == 2:
                    r.m.copy_(r.m_work)
                    r.v.copy_(r.v_work)
            self.unroll_idx += 1
            out["update"] = None
        return out



class _MtTask(object):
    """One imitation-learning ("mt") task (DM/meta_dm_train.py:421-499): the optimizer nets run over PRE-RECORDED
    gradient sequences [T, N] with their own LSTM state; loss = sum_t 0.5 ||label_t - delta_t||^2 / N_total; its own
    Adam slots on the shared theta (DM/meta_dm_train.py:549-553).  This is the fully fused regime: one forward-unroll
    launch + one BPTT launch per subset, no optimizee in the loop."""

    def __init__(self, prog, index):
        self.prog, self.index = prog, index
        T = prog.T
        if len(prog.learned) != len(prog.nets):
            raise NotImplementedError("imitation tasks with an Sgd / Adam net (nothing to imitate with)")
        self.subsets = []
        for key, subset in zip(prog.net_keys, prog.subsets):
            runs = [r for r in prog.runs if r.key == key]
            if len(runs) != 1:
                raise NotImplementedError("imitation tasks need each net's variables contiguous in the arena")
            r = runs[0]
            h = r.net.handle
            if getattr(r.net, "per_variable", False):
                raise NotImplementedError("imitation tasks are implemented for the coordinate-wise nets")
            sb = dict(run=r, n=r.n, state=h.new_state(r.n, prog.device),
                      ckpt=torch.zeros((T + 1) * max(h.state_size(r.n), 1), device=prog.device),
                      dseq=torch.zeros(T * r.n, device=prog.device),
                      inp=Placeholder("mt{}_input_subset{}".format(index, len(self.subsets))),
                      lab=Placeholder("mt{}_label_subset{}".format(index, len(self.subsets))))
            if h.n_in == 2:   # RNNProp: the task carries its own Adam moments (DM/meta_rnnprop_train.py:469-486)
                sb.update(m=torch.zeros(r.n, device=prog.device), v=torch.zeros(r.n, device=prog.device),
                          feat=torch.zeros(T, 2, r.n, device=prog.device),
                          scratch=r.bwd_scratch)   # hand-over buffer of the two-pass tensor-core BPTT (shared with the run)
            self.subsets.append(sb)
        self.n_total = sum(sb["n"] for sb in self.subsets)
        self.adam = {k: dict(m=torch.zeros_like(net.theta), v=torch.zeros_like(net.theta), k=0)
                     for k, net in prog.nets.items()}
        self.il = torch.zeros(1, dtype=torch.float64, device=prog.device)

    def _dev(self, arr, T, n):
        t = torch.as_tensor(np.asarray(arr, dtype=np.float32)) if not torch.is_tensor(arr) else arr.float()
        return t.reshape(T, n).to(self.prog.device).contiguous()

    def execute(self, kinds, feed):
        prog, T = self.prog, self.prog.T
        if kinds == {"reset_mt"}:
            for sb in self.subsets:
                sb["state"].zero_()
                if "m" in sb:
                    sb["m"].zero_()
                    sb["v"].zero_()
            return {}
        train, commit = "step_mt" in kinds, "update_mt" in kinds
        self.il.zero_()
        if train:
            for d in prog.dtheta.values():
                d.zero_()
        finals = []
        step0 = prog._step0(feed)
        for sb in self.subsets:
            r, n = sb["run"], sb["n"]
            h = r.net.handle
            inp, lab = self._dev(feed[sb["inp"]], T, n), self._dev(feed[sb["lab"]], T, n)
            work = sb["state"].clone()
            if h.n_in == 2:
                # RNNProp imitation unroll (DM/meta_rnnprop_train.py:505-534): raw gradients in, Adam features formed
                # in-kernel from the task's own (m, v) with p = float(step + t), recorded for the backward sweep
                mw, vw = sb["m"].clone(), sb["v"].clone()
                h.unroll_fwd(r.net.theta, n, T, work, in_seq=inp, ckpt=sb["ckpt"] if train else None, labels=lab,
                             imit_loss=self.il, n_total=self.n_total, m=mw, v=vw, beta1=prog.opt.beta1,
                             beta2=prog.opt.beta2, step0=step0, feat_rec=sb["feat"],
                             delta_seq=sb["dseq"] if train else None)
                if train:
                    h.unroll_bwd(r.net.theta, n, T, sb["feat"], sb["ckpt"], prog.dtheta[r.key], labels=lab,
                                 n_total=self.n_total, delta_seq=sb["dseq"], scratch=sb["scratch"])
                finals.append((work, mw, vw))
                continue
            h.unroll_fwd(r.net.theta, n, T, work, in_seq=inp, ckpt=sb["ckpt"] if train else None, labels=lab,
                         imit_loss=self.il, n_total=self.n_total, delta_seq=sb["dseq"] if train else None)
            if train:  # the recorded deltas let the tensor-core BPTT run in imitation mode too
                h.unroll_bwd(r.net.theta, n, T, inp, sb["ckpt"], prog.dtheta[r.key], labels=lab, n_total=self.n_total,
                             delta_seq=sb["dseq"])
            finals.append((work, None, None))
        out = {}
        if "loss_mt" in kinds:
            out["loss_mt:%d" % self.index] = float(self.il.item())
        if train:
            for k, net in prog.nets.items():
                ad = self.adam[k]
                ad["k"] += 1
                _engine.adam_step(net.theta, prog.dtheta[k], ad["m"], ad["v"], ad["k"], lr=prog.learning_rate)
            out["step_mt:%d" % self.index] = None
        if commit:
            for sb, (w, mw, vw) in zip(self.subsets, finals):
                sb["state"].copy_(w)
                if mw is not None:
                    sb["m"].copy_(mw)
                    sb["v"].copy_(vw)
            out["update_mt:%d" % self.index] = None
        return out

class MetaOptimizer(object):
    """Learning to learn (meta) optimizer (DM/meta.py:219-414)."""

    beta1 = 0.95
    beta2 = 0.95
    rnnprop = False   # RNNProp programs call every net as net(m, g, state)

    def __init__(self, **kwargs):
        """``MetaOptimizer(**net_config)`` exactly as the reference (DM/meta.py:228): every keyword is a net id.  The
        two engine-side knobs ride on underscore-prefixed names that cannot collide with a net id the reference's
        drivers use: ``_seed`` (generator seed of the optimizee initializers, default 0) and ``_distributed``
        (coordinates sharded over torch.distributed ranks, one all-reduce of [dtheta | fx] per meta-step)."""
        self._nets = None
        self.seed = int(kwargs.pop("_seed", 0))
        self.distributed = bool(kwargs.pop("_distributed", False))
        if not kwargs:
            # default coordinatewise network (DM/meta.py:244-255)
            self._config = {
                "coordinatewise": {
                    "net": "CoordinateWiseDeepLSTM",
                    "net_options": {
                        "layers": (20, 20),
                        "preprocess_name": "LogAndSign",
                        "preprocess_options": {"k": 5},
                        "scale": 0.01,
                    }}}
        else:
            self._config = kwargs

    def save(self, sess=None, path=None, index=None):
        """Save meta-optimizer (DM/meta.py:255-267; ``index`` as in DM/meta_dm_train.py:257-272)."""
        result = {}
        for k, net in self._nets.items():
            if path is None:
                filename, key = None, k
            elif index is not None:
                filename = os.path.join(path, "{}.l2l-{}".format(k, index))
                key = filename
            else:
                filename = os.path.join(path, "{}.l2l".format(k))
                key = filename
            result[key] = networks.save(net, sess, filename=filename)
        return result

    def restore(self, sess, path, index):
        """DM/meta_dm_train.py:290-302: load ``<net id>.l2l-<index>`` into the live nets (Adam slots are untouched,
        exactly as the reference's assign ops leave them)."""
        for k, net in self._nets.items():
            with open(os.path.join(path, "{}.l2l-{}".format(k, index)), "rb") as f:
                data = networks._pickle.load(f)
            for m, v, shp in net.variable_shapes():
                if m not in data or v not in data[m] or tuple(np.shape(data[m][v])) != tuple(shp):
                    raise ValueError("{}.l2l-{}: variable {}/{} missing or of the wrong shape".format(k, index, m, v))
            net.set_variables(data)

    def meta_loss(self, make_loss, len_unroll, net_assignments=None, second_derivatives=False):
        """Returns ops computing the meta-loss (DM/meta.py:269-396)."""
        prog = _Program(self, make_loss, len_unroll, net_assignments, second_derivatives)
        self.program = prog
        self.step_placeholder = prog.step_placeholder
        return MetaLoss(Op("loss", prog), Op("update", prog), Op("reset", prog), Op("fx", prog), Op("x", prog))

    def meta_minimize(self, make_loss, len_unroll, learning_rate=0.01, **kwargs):
        """Returns ops minimizing the meta-loss with Adam (DM/meta.py:398-414)."""
        info = self.meta_loss(make_loss, len_unroll, **kwargs)
        self.program.learning_rate = learning_rate
        self._check_trainable()
        return MetaStep(Op("step", self.program), *info[1:])

    def _check_trainable(self):
        """tf.train.AdamOptimizer.minimize raises when no net has a variable (Sgd / Adam only): the optimizee and
        state variables are trainable=False (DM/meta.py:60-77,115-120)."""
        if not self.program.learned:
            raise ValueError("No variables to optimize: every net of this meta-optimizer is a hand-written rule")


class RNNpropMetaOptimizer(MetaOptimizer):
    """DM/meta_rnnprop_train.py / meta_rnnprop_eval.py: per-coordinate Adam moments feed the net."""

    rnnprop = True

    def __init__(self, beta1=0.95, beta2=0.95, **kwargs):
        super(RNNpropMetaOptimizer, self).__init__(**kwargs)
        self.beta1, self.beta2 = beta1, beta2
