"""Training-time MetaOptimizer of the enhanced L2O-DM recipe (DM/meta_dm_train.py): adds the per-variable ``scale``
placeholders of the random-scaling trick and ``num_mt`` imitation-learning tasks to the plain optimizer of
``open_l2o_b200.meta``.  Return arities follow the reference:

    info, scale, x, constants, subsets, loss_mt, update_mt, reset_mt, mt_labels, mt_inputs = opt.meta_loss(...)
    step_info, scale, x, constants, subsets, loss_mt, steps_mt, update_mt, reset_mt, mt_labels, mt_inputs
        = opt.meta_minimize(...)
"""
from __future__ import annotations

from . import meta as _meta
from .meta import MetaLoss, MetaStep, Op, Session  # noqa: F401  (re-exported like the reference module's names)


class VariableRef(object):
    """Stand-in for the tf.Variable handles ``var_x`` the reference returns (DM/train_dm.py:84-90,103-113)."""

    def __init__(self, prog, index):
        self._prog, self._index = prog, index
        self.name = prog.variables[index]["name"] + ":0"
        self.shape = tuple(prog.variables[index]["shape"])

    def value(self):
        return self._prog.x_values()[self._index]


class MetaOptimizer(_meta.MetaOptimizer):
    def __init__(self, num_mt, **kwargs):
        super(MetaOptimizer, self).__init__(**kwargs)
        self.num_mt = num_mt

    def _extras(self, prog):
        prog.mt_tasks = [_meta._MtTask(prog, i) for i in range(self.num_mt)]
        scale = list(prog.scale_placeholders)
        x = [VariableRef(prog, j) for j in range(len(prog.variables))]
        constants = [c["name"] for c in prog.constants]
        subsets = [list(sb) for sb in prog.subsets]
        loss_mt = [Op("loss_mt:%d" % i, prog) for i in range(self.num_mt)]
        steps_mt = [Op("step_mt:%d" % i, prog) for i in range(self.num_mt)]
        update_mt = [Op("update_mt:%d" % i, prog) for i in range(self.num_mt)]
        reset_mt = [Op("reset_mt:%d" % i, prog) for i in range(self.num_mt)]
        mt_labels = [[sb["lab"] for sb in t.subsets] for t in prog.mt_tasks]
        mt_inputs = [[sb["inp"] for sb in t.subsets] for t in prog.mt_tasks]
        return scale, x, constants, subsets, loss_mt, steps_mt, update_mt, reset_mt, mt_labels, mt_inputs

    def meta_loss(self, make_loss, len_unroll, net_assignments=None, second_derivatives=False):
        """DM/meta_dm_train.py:304-527."""
        info = super(MetaOptimizer, self).meta_loss(make_loss, len_unroll, net_assignments, second_derivatives)
        scale, x, constants, subsets, loss_mt, _, update_mt, reset_mt, mt_labels, mt_inputs = self._extras(self.program)
        return info, scale, x, constants, subsets, loss_mt, update_mt, reset_mt, mt_labels, mt_inputs

    def meta_minimize(self, make_loss, len_unroll, learning_rate=0.01, **kwargs):
        """DM/meta_dm_train.py:529-558."""
        info = _meta.MetaOptimizer.meta_loss(self, make_loss, len_unroll, **kwargs)
        self.program.learning_rate = learning_rate
        self._check_trainable()
        extras = self._extras(self.program)
        return (MetaStep(Op("step", self.program), *info[1:]),) + extras

    def restorer(self):
        """DM/meta_dm_train.py:274-288 builds one placeholder + assign op per net variable; an eager engine assigns
        directly, so this only records (per net) the ``{module: {variable: shape}}`` map ``restore`` will check the
        ``.l2l-<index>`` files against."""
        self.restore_pl = {k: {m: {} for m, _, _ in net.variable_shapes()} for k, net in self._nets.items()}
        for k, net in self._nets.items():
            for m, v, shp in net.variable_shapes():
                self.restore_pl[k][m][v] = tuple(shp)
        return self.restore_pl

    def assign_func(self, values):
        self.program.assign_x(values)
