"""Epoch runners and the problem -> net-config registry (DM/util.py)."""
from __future__ import annotations

from timeit import default_timer as timer

import numpy as np

from . import problems


def run_epoch(sess, cost_op, ops, reset, num_unrolls,
              scale=None, rd_scale=False, rd_scale_bound=3.0, assign_func=None, var_x=None,
              step=None, unroll_len=None,
              task_i=-1, data=None, label_pl=None, input_pl=None):
    """Runs one optimization epoch (DM/util.py:31-75), including the random-scaling branch (:40-54) and the
    imitation-task branch (:62-74)."""
    start = timer()
    sess.run(reset)
    cost = None
    if task_i == -1:
        if rd_scale:
            assert scale is not None and var_x is not None and assign_func is not None
            r_scale = [np.exp(np.random.uniform(-rd_scale_bound, rd_scale_bound, size=k.shape)).astype(np.float32)
                       for k in var_x]
            assign_func([v.value() / r for v, r in zip(var_x, r_scale)])
            feed_dict = {p: v for p, v in zip(scale, r_scale)}
        else:
            feed_dict = {}
        for i in range(num_unrolls):
            if step is not None:
                feed_dict[step] = i * unroll_len + 1
            cost = sess.run([cost_op] + list(ops), feed_dict=feed_dict)[0]
    else:
        assert data is not None and input_pl is not None and label_pl is not None
        feed_dict = {}
        for ri in range(num_unrolls):
            for pl, dat in zip(label_pl, data["labels"][ri]):
                feed_dict[pl] = dat
            for pl, dat in zip(input_pl, data["inputs"][ri]):
                feed_dict[pl] = dat
            if step is not None:
                feed_dict[step] = ri * unroll_len + 1
            cost = sess.run([cost_op] + list(ops), feed_dict=feed_dict)[0]
    return timer() - start, cost


def run_eval_epoch(sess, cost_op, ops, num_unrolls, step=None, unroll_len=None):
    """DM/util.py:78-89."""
    start = timer()
    total_cost = []
    feed_dict = {}
    for i in range(num_unrolls):
        if step is not None:
            feed_dict[step] = i * unroll_len + 1
        cost = sess.run([cost_op] + list(ops), feed_dict=feed_dict)[0]
        total_cost.append(cost)
    return timer() - start, total_cost


def print_stats(header, total_error, total_time, n):
    """DM/util.py:92-96."""
    print(header)
    print("Log Mean Final Error: {:.2f}".format(np.log10(total_error / n)))
    print("Mean epoch time: {:.2f} s".format(total_time / n))


def get_default_net_config(path):
    """DM/util.py:99-109."""
    return {
        "net": "CoordinateWiseDeepLSTM",
        "net_options": {
            "layers": (20, 20),
            "preprocess_name": "LogAndSign",
            "preprocess_options": {"k": 5},
            "scale": 0.01,
        },
        "net_path": path
    }


def _cw20(path):
    return {"cw": {"net": "CoordinateWiseDeepLSTM", "net_options": {"layers": (20, 20)}, "net_path": path}}


def get_config(problem_name, path=None, mode=None, num_hidden_layer=None, net_name=None):
    """Returns problem configuration (DM/util.py:112-265) for the synthetic problems that exist offline."""
    net_assignments = None
    if problem_name == "simple":
        problem = problems.simple()
        net_config = {"cw": {"net": "CoordinateWiseDeepLSTM", "net_options": {"layers": (), "initializer": "zeros"},
                             "net_path": path}}
    elif problem_name == "simple-multi":
        problem = problems.simple_multi_optimizer()
        net_config = {
            "cw": {"net": "CoordinateWiseDeepLSTM", "net_options": {"layers": (), "initializer": "zeros"},
                   "net_path": path},
            "adam": {"net": "Adam", "net_options": {"learning_rate": 0.01}},
        }
        net_assignments = [("cw", ["x_0"]), ("adam", ["x_1"])]
    elif problem_name == "quadratic":
        problem = problems.quadratic(batch_size=128, num_dims=10)
        net_config = _cw20(path)
    elif problem_name == "rastrigin":
        problem = problems.rastrigin(batch_size=128, num_dims=2)
        net_config = _cw20(path)
    elif problem_name == "lasso":
        problem = problems.lasso(batch_size=128, num_dims=2)
        net_config = _cw20(path)
    elif problem_name == "rastrigin_separable":   # BASELINE config #5
        problem = problems.rastrigin_separable(num_dims=1000000)
        net_config = _cw20(path)
    elif problem_name == "mlp":                   # BASELINE config #3 / target line (synthetic data)
        problem = problems.mlp(layers=(100,) if num_hidden_layer is None else (100,) * num_hidden_layer)
        net_config = {"cw": get_default_net_config(path)}
    else:
        raise ValueError("{} is not a valid problem".format(problem_name))

    if net_name == "RNNprop":  # DM/util.py:251-263
        net_config = {"rp": {
            "net": "RNNprop",
            "net_options": {"layers": (20, 20), "preprocess_name": "fc", "preprocess_options": {"dim": 20},
                            "scale": 0.01, "tanh_output": True},
            "net_path": path}}
    return problem, net_config, net_assignments
