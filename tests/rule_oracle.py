"""CPU oracle of the hand-written update rules networks.Sgd / networks.Adam (DM/networks.py:354-420) and of an unroll
in which several nets (learned coordinate-wise LSTMs and rules) share one optimizee (DM/meta.py:338-376).

Test infrastructure, not product code: an fp32 (optionally fp64) restatement on torch-CPU tensors, built on the
coordinate-wise net of ``oracle/l2o_oracle.py``.  The product package never imports it."""
from __future__ import annotations

from dataclasses import dataclass
from typing import Callable, Optional

import torch

from oracle.l2o_oracle import net_apply


@dataclass
class RuleSpec:
    """Constructor arguments of networks.Sgd (kind "sgd") / networks.Adam (kind "adam")."""
    kind: str
    learning_rate: float = 1e-3
    beta1: float = 0.9
    beta2: float = 0.999
    epsilon: float = 1e-8


def rule_initial_state(rule: RuleSpec, n: int, dtype=torch.float32):
    """Sgd: () ; Adam: (t 0-d, m [n], v [n]) zeros (DM/networks.py:370-371,415-420)."""
    if rule.kind == "sgd":
        return ()
    return torch.zeros((), dtype=dtype), torch.zeros(n, dtype=dtype), torch.zeros(n, dtype=dtype)


def rule_apply(rule: RuleSpec, g, state):
    """update, next_state = net(g, state) (DM/networks.py:367-368,374-379,393-413) in g's dtype with TF's operation
    order: each Python-float hyper-parameter enters as one scalar of that dtype, (1 - b) is formed in Python first,
    every product / sum / quotient is rounded on its own."""
    dt = g.dtype

    def c(v):
        return torch.tensor(v, dtype=dt)
    if rule.kind == "sgd":
        return c(-rule.learning_rate) * g, ()
    t, m, v = state
    t = t + 1
    m = c(rule.beta1) * m + c(1 - rule.beta1) * g
    v = c(rule.beta2) * v + c(1 - rule.beta2) * (g * g)
    m_hat = m / (1 - torch.pow(c(rule.beta1), t))
    v_hat = v / (1 - torch.pow(c(rule.beta2), t))
    return (c(-rule.learning_rate) * m_hat) / (torch.sqrt(v_hat) + c(rule.epsilon)), (t, m, v)


@dataclass
class MixedResult:
    fx: torch.Tensor          # [T+1]
    loss: torch.Tensor
    x_final: torch.Tensor     # flat
    states: list              # one per assignment


def mixed_unroll(assignments, x0, states0, f: Callable, T: int, grad_of: Optional[Callable] = None) -> MixedResult:
    """DM/meta.py:338-376 with several nets over one flat x.  ``assignments``: [(net, sl)] where ``net`` is a
    ``(NetSpec, theta)`` pair (coordinate-wise LSTM, not RNNProp) or a ``RuleSpec`` and ``sl`` the slice of x it
    updates; ``states0``: one state per assignment.  The gradient every net sees is stop-gradient'ed
    (DM/meta.py:328-329), so a rule's coordinates depend on theta only through the recorded gradients."""
    x, states, fxs = x0, list(states0), []
    for t in range(T):
        if grad_of is not None:
            fx, g = grad_of(x)
        else:
            xg = x.detach().requires_grad_(True)
            with torch.enable_grad():
                (g,) = torch.autograd.grad(f(xg), xg)
            fx = f(x)
        fxs.append(fx)
        g = g.detach().reshape(-1)
        x_next = x.clone()
        for i, (net, sl) in enumerate(assignments):
            if isinstance(net, RuleSpec):
                delta, states[i] = rule_apply(net, g[sl], states[i])
            else:
                spec, theta = net
                if spec.rnnprop:
                    raise ValueError("mixed_unroll: RNNProp nets take (m, g) inputs")
                delta, states[i] = net_apply(spec, theta, g[sl].unsqueeze(-1), states[i])
            x_next[sl] = x[sl] + delta
        x = x_next
    fxs.append(grad_of(x)[0] if grad_of is not None else f(x))
    fx = torch.stack([v.reshape(()) for v in fxs])
    return MixedResult(fx, fx.sum(), x, states)


def mixed_meta_grad(assignments, x0, states0, f, T, grad_of=None):
    """dL/dtheta of every learned net of ``mixed_unroll`` by autograd (None for a rule)."""
    leaves, asg = [], []
    for net, sl in assignments:
        if isinstance(net, RuleSpec):
            asg.append((net, sl))
            leaves.append(None)
        else:
            th = net[1].detach().clone().requires_grad_(True)
            asg.append(((net[0], th), sl))
            leaves.append(th)
    res = mixed_unroll(asg, x0, states0, f, T, grad_of=grad_of)
    live = [th for th in leaves if th is not None]
    grads = iter(torch.autograd.grad(res.loss, live)) if live else iter(())
    return [next(grads) if th is not None else None for th in leaves], res
