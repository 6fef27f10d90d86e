"""Evaluation-time MetaOptimizer of L2O-RNNProp (DM/meta_rnnprop_eval.py): the same unroll as the training module
without imitation tasks.  Return arities follow the reference:

    info, scale, x, step = opt.meta_loss(...)            DM/meta_rnnprop_eval.py:306-466
    step_info, scale, x, seq_step = opt.meta_minimize(...)   DM/meta_rnnprop_eval.py:468-485
"""
from __future__ import annotations

from . import meta as _meta
from .meta import MetaLoss, MetaStep, Op, Session  # noqa: F401
from .meta_dm_train import VariableRef


class MetaOptimizer(_meta.MetaOptimizer):
    rnnprop = True

    def __init__(self, beta1, beta2, **kwargs):
        """DM/meta_rnnprop_eval.py:230-256."""
        super(MetaOptimizer, self).__init__(**kwargs)
        self.beta1, self.beta2 = beta1, beta2

    def _extras(self):
        prog = self.program
        return (list(prog.scale_placeholders), [VariableRef(prog, j) for j in range(len(prog.variables))],
                prog.step_placeholder)

    def meta_loss(self, make_loss, len_unroll, net_assignments=None, second_derivatives=False):
        info = super(MetaOptimizer, self).meta_loss(make_loss, len_unroll, net_assignments, second_derivatives)
        return (info,) + self._extras()

    def meta_minimize(self, make_loss, len_unroll, learning_rate=0.01, **kwargs):
        info = _meta.MetaOptimizer.meta_loss(self, make_loss, len_unroll, **kwargs)
        self.program.learning_rate = learning_rate
        return (MetaStep(Op("step", self.program), *info[1:]),) + self._extras()

    def restorer(self):
        """DM/meta_rnnprop_eval.py:276-289: nothing to build in an eager engine (``restore`` assigns directly)."""
        return None
