"""Training-time MetaOptimizer of the enhanced L2O-RNNProp recipe (DM/meta_rnnprop_train.py): per-coordinate Adam
moments feed the net (:371-395), ``num_mt`` imitation tasks carry their own (state, m, v) (:441-555), and the bias-
correction exponent ``p = float(step + t)`` comes from the ``step`` placeholder fed per unroll (DM/util.py:59-60).
Return arities follow the reference:

    info, scale, x, constants, subsets, step, loss_mt, update_mt, reset_mt, mt_labels, mt_inputs = opt.meta_loss(...)
    step_info, scale, x, constants, subsets, seq_step, loss_mt, steps_mt, update_mt, reset_mt, mt_labels, mt_inputs
        = opt.meta_minimize(...)
"""
from __future__ import annotations

from . import meta as _meta
from . import meta_dm_train as _dm
from .meta import MetaLoss, MetaStep, Op, Session  # noqa: F401  (re-exported like the reference module's names)


class MetaOptimizer(_dm.MetaOptimizer):
    rnnprop = True

    def __init__(self, num_mt, beta1, beta2, **kwargs):
        """DM/meta_rnnprop_train.py:230-257."""
        super(MetaOptimizer, self).__init__(num_mt, **kwargs)
        self.beta1, self.beta2 = beta1, beta2

    def meta_loss(self, make_loss, len_unroll, net_assignments=None, second_derivatives=False):
        """DM/meta_rnnprop_train.py:306-593."""
        info = _meta.MetaOptimizer.meta_loss(self, make_loss, len_unroll, net_assignments, second_derivatives)
        scale, x, constants, subsets, loss_mt, _, update_mt, reset_mt, mt_labels, mt_inputs = self._extras(self.program)
        return (info, scale, x, constants, subsets, self.program.step_placeholder, loss_mt, update_mt, reset_mt,
                mt_labels, mt_inputs)

    def meta_minimize(self, make_loss, len_unroll, learning_rate=0.01, **kwargs):
        """DM/meta_rnnprop_train.py:595-624."""
        info = _meta.MetaOptimizer.meta_loss(self, make_loss, len_unroll, **kwargs)
        self.program.learning_rate = learning_rate
        scale, x, constants, subsets, loss_mt, steps_mt, update_mt, reset_mt, mt_labels, mt_inputs = \
            self._extras(self.program)
        return (MetaStep(Op("step", self.program), *info[1:]), scale, x, constants, subsets,
                self.program.step_placeholder, loss_mt, steps_mt, update_mt, reset_mt, mt_labels, mt_inputs)
