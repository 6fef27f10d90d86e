"""GPU tests of the hand-written update rules networks.Sgd / networks.Adam (DM/networks.py:354-420): the reference's
SgdTest / AdamTest (SW/networks_test.py:119-190), step and fused-unroll parity against the oracle, mixed programs of a
learned net and a rule (SW/meta_test.py:92-101, DM/util.py:122-135), CUDA-graph replay and the error surface."""
import os
import tempfile
import types

import numpy as np
import pytest
import torch

from oracle import l2o_oracle as orc
from tests import rule_oracle as ro
from tests.helpers import REL_TOL, assert_theta_close, rel_err

pytestmark = pytest.mark.gpu

DEV = "cuda"


def _detach(s):
    return tuple(_detach(v) for v in s) if isinstance(s, (tuple, list)) else s.detach()


def train(sess, minimize_ops, num_epochs, num_unrolls):
    """L2L training (SW/meta_test.py:33-43)."""
    step, update, reset, loss_last, x_last = minimize_ops
    for _ in range(num_epochs):
        sess.run(reset)
        for _ in range(num_unrolls):
            cost, final_x, _, _ = sess.run([loss_last, x_last, update, step])
    return cost, final_x


# ---- SgdTest / AdamTest ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["Sgd", "Adam"])
def test_shape_and_non_trainable(name):
    from open_l2o_b200 import networks
    shape = [10, 5]
    gradients = torch.randn(shape, device=DEV)
    net = getattr(networks, name)()
    state = net.initial_state_for_inputs(gradients)
    update, _ = net(gradients, state)
    assert list(update.shape) == shape
    assert net.variable_shapes() == [] and net.get_variables() == [] and networks.save(net) == {}


def test_sgd_results_exact():
    from open_l2o_b200 import networks
    for shape in ([10], [1], [1001, 3]):
        learning_rate = 0.01
        gradients = torch.randn(shape, device=DEV)
        net = networks.Sgd(learning_rate=learning_rate)
        update, state = net(gradients, net.initial_state_for_inputs(gradients))
        assert state == [] and torch.equal(update, -learning_rate * gradients)


def test_adam_zero_learning_rate():
    from open_l2o_b200 import networks
    gradients = torch.randn(10, device=DEV)
    net = networks.Adam(learning_rate=0)
    state = net.initial_state_for_inputs(gradients)
    for _ in range(2):
        update, state = net(gradients, state)
        assert torch.equal(update, torch.zeros(10, device=DEV))


def test_adam_state_surface_and_chaining():
    """(t, m, v): a 0-d counter and [N, 1] moments, views of one arena; a plain tuple is accepted as well."""
    from open_l2o_b200 import networks
    net = networks.Adam(learning_rate=0.02, beta1=0.8, beta2=0.99)
    rule = ro.RuleSpec("adam", 0.02, 0.8, 0.99)
    g = torch.randn(7, 9)
    st = net.initial_state_for_inputs(g.to(DEV))
    t, m, v = st
    assert t.shape == () and tuple(m.shape) == (63, 1) and tuple(v.shape) == (63, 1) and st.arena is not None
    st_ref = ro.rule_initial_state(rule, 63)
    for k in range(3):
        upd, st = net(g.to(DEV) * (k + 1), st)
        upd_ref, st_ref = ro.rule_apply(rule, g.reshape(-1) * (k + 1), st_ref)
        assert tuple(upd.shape) == (7, 9) and rel_err(upd, upd_ref) <= REL_TOL
    assert float(st[0]) == 3.0 and rel_err(st[1], st_ref[1]) <= REL_TOL and rel_err(st[2], st_ref[2]) <= REL_TOL
    plain = tuple(s.clone() for s in st)
    upd_a, _ = net(g.to(DEV), st)
    upd_b, _ = net(g.to(DEV), plain)
    assert torch.equal(upd_a, upd_b)


# ---- step kernel parity -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 1000, 1_000_003])
@pytest.mark.parametrize("kind", ["sgd", "adam"])
@pytest.mark.parametrize("mode", ["delta", "x", "x+delta"])
def test_rule_step_matches_oracle(n, kind, mode):
    from open_l2o_b200.engine import RULE_ADAM, RULE_SGD, RuleHandle
    rule = ro.RuleSpec(kind, learning_rate=0.003, beta1=0.9, beta2=0.999, epsilon=1e-8)
    h = RuleHandle(RULE_ADAM if kind == "adam" else RULE_SGD, 0.003, 0.9, 0.999, 1e-8)
    gen = torch.Generator().manual_seed(n)
    arenas = [h.new_state(n, DEV), h.new_state(n, DEV)]
    st_ref = ro.rule_initial_state(rule, n)
    x_ref = torch.randn(n, generator=gen)
    x = x_ref.to(DEV) if "x" in mode else None
    for k in range(4):
        g = torch.randn(n, generator=gen) * 10.0 ** torch.randint(-4, 2, (n,), generator=gen).float()
        delta = torch.full((n,), float("nan"), device=DEV) if "delta" in mode else None
        h.step(g.to(DEV), arenas[k % 2], arenas[(k + 1) % 2], x=x, delta=delta)
        d_ref, st_ref = ro.rule_apply(rule, g, st_ref)
        x_ref = x_ref + d_ref
        if delta is not None:
            if kind == "sgd":
                assert torch.equal(delta.cpu(), d_ref), k
            else:
                assert rel_err(delta, d_ref) <= REL_TOL, k
        if x is not None:
            assert rel_err(x, x_ref) <= REL_TOL, k
        if kind == "adam":
            a = arenas[(k + 1) % 2].cpu()
            assert float(a[0]) == k + 1 and torch.equal(a[1:4], torch.zeros(3))
            assert rel_err(a[4:4 + n], st_ref[1]) <= REL_TOL and rel_err(a[4 + n:], st_ref[2]) <= REL_TOL, k


def test_rule_step_unaligned_views():
    """Views at odd offsets take the scalar path; the result is the same as the aligned (vectorised) one."""
    from open_l2o_b200.engine import RULE_ADAM, RuleHandle
    h = RuleHandle(RULE_ADAM, 0.01)
    n = 4096
    g = torch.randn(n + 1, device=DEV)
    outs = []
    for off in (0, 1):
        gv = g[off:off + n] if off else g[1:].clone()
        s_in, s_out = h.new_state(n, DEV), h.new_state(n, DEV)
        buf = torch.zeros(n + 1, device=DEV)
        x = buf[1:] if off else torch.zeros(n, device=DEV)
        h.step(gv, s_in, s_out, x=x)
        outs.append((x.clone(), s_out.clone()))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])


# ---- fused unroll parity --------------------------------------------------------------------------------------------
def _rule_cfg(kind, problem, n):
    if kind == "adam":
        return {"net": "Adam", "net_options": {"learning_rate": 0.01}}, ro.RuleSpec("adam", 0.01)
    lr = (5e-4 if problem == "rastrigin_sep" else 0.01) * n   # the optimizees are normalised by 1/n
    return {"net": "Sgd", "net_options": {"learning_rate": lr}}, ro.RuleSpec("sgd", lr)


def _fused_problem(problem, n):
    from open_l2o_b200 import problems
    return problems.rastrigin_separable(num_dims=n) if problem == "rastrigin_sep" else problems.quadratic_diag(n)


@pytest.mark.parametrize("kind", ["sgd", "adam"])
@pytest.mark.parametrize("problem", ["rastrigin_sep", "quadratic_diag"])
def test_fused_rule_unroll_matches_oracle(kind, problem):
    """T = 100 rule steps in one launch; a second unroll carried over through `update` continues the oracle's."""
    from open_l2o_b200 import meta
    n, T = 100_000, 100
    cfg, rule = _rule_cfg(kind, problem, n)
    opt = meta.MetaOptimizer(r=cfg)
    loss, update, reset, fx, x = opt.meta_loss(_fused_problem(problem, n), T)
    prog = opt.program
    assert prog.fused is not None and not hasattr(prog.runs[0], "ckpt")
    sess = meta.Session()
    sess.run(reset)
    f = prog.fused
    fp = orc.FusedProblem(problem, prog.const_vals[f.a].cpu().reshape(-1), prog.const_vals[f.b].cpu().reshape(-1),
                          alpha=f.alpha, fscale=f.fscale)
    x_ref, st_ref = prog.X.cpu().clone(), ro.rule_initial_state(rule, n)
    # Adam's first moment on Rastrigin: the gradient 2 pi alpha c sin(2 pi x) + (x - b) changes sign from step to step, so
    # max |m| is far below max |g| while m sums the last-bit differences of sincosf against the CPU's sin / cos.  Measured
    # on the B200: 3.7e-5 after the first unroll, 2.5e-5 after the second (x 4e-7, v 3.6e-7, fx 9e-8).
    m_tol = 1e-4 if problem == "rastrigin_sep" else REL_TOL
    for it in range(2):
        cost, final = sess.run([loss, fx, update])[:2]
        fxs = []
        for t in range(T):
            fv, g = fp.f_and_g(x_ref)
            fxs.append(fv)
            d, st_ref = ro.rule_apply(rule, g, st_ref)
            x_ref = x_ref + d
        fxs.append(fp.f_and_g(x_ref)[0])
        fx_ref = torch.stack(fxs).double()
        assert rel_err(prog.last_fx, fx_ref) <= REL_TOL, it
        assert abs(final - float(fx_ref[-1])) <= REL_TOL * abs(float(fx_ref[-1])), it
        assert rel_err(prog.X, x_ref) <= REL_TOL, it
        if kind == "adam":
            s = prog.runs[0].state.cpu()
            assert float(s[0]) == (it + 1) * T
            assert rel_err(s[4:4 + n], st_ref[1]) <= m_tol and rel_err(s[4 + n:], st_ref[2]) <= REL_TOL, it


@pytest.mark.parametrize("kind", ["sgd", "adam"])
def test_fused_rule_unroll_equals_step_at_a_time(kind, monkeypatch):
    """The one-launch unroll and T external-regime steps (graph-captured on the third call) agree."""
    from open_l2o_b200 import meta
    n, T = 20_000, 30
    cfg, _ = _rule_cfg(kind, "rastrigin_sep", n)
    out = []
    for disable in ("0", "1"):
        monkeypatch.setenv("L2O_DISABLE_FUSED", disable)
        opt = meta.MetaOptimizer(r=cfg)
        ms = opt.meta_loss(_fused_problem("rastrigin_sep", n), T)
        assert (opt.program.fused is None) == (disable == "1")
        sess = meta.Session()
        sess.run(ms.reset)
        fxs = []
        for _ in range(3):
            sess.run([ms.loss, ms.update])
            fxs.append(opt.program.last_fx.clone())
        out.append((torch.cat(fxs), opt.program.X.clone(), opt.program.runs[0].state.clone()))
    (f1, x1, s1), (f2, x2, s2) = out
    assert rel_err(f1, f2) <= REL_TOL and rel_err(x1, x2) <= REL_TOL and rel_err(s1, s2) <= REL_TOL


# ---- mixed programs ---------------------------------------------------------------------------------------------------
def test_multi_optimizer_different_optimizers():
    """The "Different optimizers" case of SW/meta_test.py:92-101."""
    from open_l2o_b200 import meta, problems
    problem = problems.simple_multi_optimizer(num_dims=2)
    optimizer = meta.MetaOptimizer(net1={"net": "CoordinateWiseDeepLSTM", "net_options": {"layers": (1,)}},
                                   net2={"net": "Adam"})
    minimize_ops = optimizer.meta_minimize(problem, 3, net_assignments=[("net1", ["x_0"]), ("net2", ["x_1"])])
    cost, x = train(meta.Session(), minimize_ops, 1, 2)
    assert np.isfinite(cost)


def test_simple_multi_config_runs_epochs():
    """util.get_config("simple-multi") (DM/util.py:122-135) through util.run_epoch: Adam(0.01) moves x_1 by ~0.01 per
    step while the zero-initialised net leaves x_0 where it is in the first unroll."""
    from open_l2o_b200 import meta, util
    problem, net_config, net_assignments = util.get_config("simple-multi")
    optimizer = meta.MetaOptimizer(**net_config)
    ms = optimizer.meta_minimize(problem, 5, learning_rate=0.01, net_assignments=net_assignments)
    sess = meta.Session()
    _, cost = util.run_epoch(sess, ms.fx, [ms.update, ms.step], ms.reset, 1)
    rule = ro.RuleSpec("adam", 0.01)
    x1, st = torch.ones(1), ro.rule_initial_state(rule, 1)
    for _ in range(5):
        d, st = ro.rule_apply(rule, 2.0 * x1, st)
        x1 = x1 + d
    assert abs(cost - (1.0 + float(x1) ** 2)) <= 1e-6
    for _ in range(2):
        _, cost = util.run_epoch(sess, ms.fx, [ms.update, ms.step], ms.reset, 3)
        assert np.isfinite(cost) and cost < 2.0


def _coupled(n):
    """A two-variable optimizee whose gradients couple the variables: f = mean((w a + b - y)^2) + 0.1 mean(b^2)."""
    from open_l2o_b200.variables import get_variable, random_normal_initializer, random_uniform_initializer

    def build():
        a = get_variable("a", shape=[n], initializer=random_normal_initializer(stddev=1.0))
        b = get_variable("b", shape=[n], initializer=random_normal_initializer(stddev=1.0))
        w = get_variable("w", shape=[n], initializer=random_uniform_initializer(0.5, 1.5), trainable=False)
        y = get_variable("y", shape=[n], initializer=random_uniform_initializer(), trainable=False)
        return torch.mean((w * a + b - y) ** 2) + 0.1 * torch.mean(b ** 2)
    return build


def test_mixed_lstm_adam_training_matches_oracle():
    """LSTM-20x2 on `a`, Adam on `b` of a coupled optimizee: fx[0..T], x and theta after TF-Adam over three meta-steps
    against autograd through the oracle's mixed unroll.  The Adam coordinates reach dtheta only through the gradients
    the LSTM is fed."""
    from open_l2o_b200 import meta
    n, T, lr = 40, 5, 0.001
    optimizer = meta.MetaOptimizer(lstm={"net": "CoordinateWiseDeepLSTM",
                                         "net_options": {"layers": (20, 20), "scale": 0.1}},
                                   adam={"net": "Adam", "net_options": {"learning_rate": 0.05}})
    ms = optimizer.meta_minimize(_coupled(n), T, learning_rate=lr, net_assignments=[("lstm", ["a"]), ("adam", ["b"])])
    prog = optimizer.program
    assert set(prog.dtheta) == {"lstm"} and set(prog.adam) == {"lstm"}
    rr = [r for r in prog.runs if r.key == "adam"][0]
    assert not hasattr(rr, "ckpt") and not hasattr(rr, "g_rec")
    sess = meta.Session()
    sess.run(ms.reset)
    w, y = prog.const_vals["w"].cpu(), prog.const_vals["y"].cpu()
    oa, ob = prog.var_off[0], prog.var_off[1]

    def f(x):
        a, b = x[oa:oa + n], x[ob:ob + n]
        return torch.mean((w * a + b - y) ** 2) + 0.1 * torch.mean(b ** 2)
    spec, rule = orc.NetSpec(layers=(20, 20), scale=0.1), ro.RuleSpec("adam", 0.05)
    lstm = prog.nets["lstm"]
    tr = types.SimpleNamespace(theta=lstm.theta.cpu().clone(), last_grad=None)
    m, v = torch.zeros_like(tr.theta), torch.zeros_like(tr.theta)
    x_ref = prog.X.cpu().clone()
    states = [orc.initial_state(spec, n), ro.rule_initial_state(rule, n)]
    for it in range(3):
        cost, xs, _, _ = sess.run([ms.fx, ms.x, ms.update, ms.step])
        (g, none), res = ro.mixed_meta_grad([((spec, tr.theta), slice(oa, oa + n)), (rule, slice(ob, ob + n))],
                                             x_ref, states, f, T)
        tr.last_grad = g
        tr.theta, m, v = orc.tf_adam_step(tr.theta, g, m, v, it + 1, lr=lr)
        x_ref = res.x_final.detach()
        states = [_detach(s) for s in res.states]
        assert rel_err(prog.last_fx, res.fx.detach()) <= 1e-5, it
        assert abs(cost - float(res.fx[-1])) <= 1e-5 * abs(float(res.fx[-1])) + 1e-9, it
        assert rel_err(np.concatenate([xs[0], xs[1]]), torch.cat([x_ref[oa:oa + n], x_ref[ob:ob + n]])) <= REL_TOL
        assert_theta_close(lstm.theta, tr, it)


def test_graph_replay_after_reset_matches_eager_with_adam(monkeypatch):
    """External-gradient regime with an Adam run: the counter t lives on the device, so the captured unroll stays right
    across replays and after `reset` (3 unrolls, reset, 2 unrolls: the same costs and x with and without graphs)."""
    from open_l2o_b200 import meta, problems

    def run():
        optimizer = meta.MetaOptimizer(adam={"net": "Adam", "net_options": {"learning_rate": 0.003}})
        ms = optimizer.meta_loss(problems.quadratic(batch_size=128, num_dims=10), 20)
        sess, out = meta.Session(), []
        for n_unrolls in (4, 3):
            sess.run(ms.reset)
            for _ in range(n_unrolls):
                cost, xs, _ = sess.run([ms.fx, ms.x, ms.update])
                out.append((cost, xs[0].copy(), float(optimizer.program.runs[0].state[0])))
        return out, optimizer.program

    monkeypatch.setenv("L2O_CUDA_GRAPH", "1")
    graphed, prog = run()
    assert False in prog._graphs
    monkeypatch.setenv("L2O_CUDA_GRAPH", "0")
    eager, prog2 = run()
    assert not prog2._graphs
    assert [t for _, _, t in graphed] == [20.0, 40.0, 60.0, 80.0, 20.0, 40.0, 60.0]
    for (c1, x1, t1), (c2, x2, t2) in zip(graphed, eager):
        assert t1 == t2 and abs(c1 - c2) <= 1e-6 * abs(c2) and rel_err(x1, x2) <= 1e-6


# ---- errors and save ------------------------------------------------------------------------------------------------
def test_meta_minimize_needs_a_trainable_net():
    from open_l2o_b200 import meta, problems
    cfg = {"adam": {"net": "Adam", "net_options": {"learning_rate": 0.1}}}
    with pytest.raises(ValueError):
        meta.MetaOptimizer(**cfg).meta_minimize(problems.simple(), 3)
    ms = meta.MetaOptimizer(**cfg).meta_loss(problems.simple(), 3)
    sess = meta.Session()
    sess.run(ms.reset)
    loss, final = sess.run([ms.loss, ms.fx])
    assert final < 1.0 and np.isfinite(loss)


def test_rule_net_unsupported_programs():
    from open_l2o_b200 import meta, meta_dm_train, problems
    cfg = {"cw": {"net": "CoordinateWiseDeepLSTM", "net_options": {"layers": (1,)}}, "adam": {"net": "Adam"}}
    asg = [("cw", ["x_0"]), ("adam", ["x_1"])]
    with pytest.raises(NotImplementedError):
        meta_dm_train.MetaOptimizer(1, **cfg).meta_minimize(problems.simple_multi_optimizer(), 3, net_assignments=asg)
    with pytest.raises(NotImplementedError):
        meta.RNNpropMetaOptimizer(adam={"net": "Adam"}).meta_loss(problems.simple(), 3)
    # without imitation tasks the training-time optimizer takes the mixed config
    out = meta_dm_train.MetaOptimizer(0, **cfg).meta_minimize(problems.simple_multi_optimizer(), 3, net_assignments=asg)
    assert out[0].step is not None


def test_save_writes_empty_dict_for_rule_net():
    from open_l2o_b200 import meta, networks, problems
    cfg = {"cw": {"net": "CoordinateWiseDeepLSTM", "net_options": {"layers": (2, 3)}}, "adam": {"net": "Adam"}}
    optimizer = meta.MetaOptimizer(**cfg)
    ms = optimizer.meta_minimize(problems.simple_multi_optimizer(), 3, net_assignments=[("cw", ["x_0"]),
                                                                                         ("adam", ["x_1"])])
    train(meta.Session(), ms, 1, 1)
    tmp_dir = tempfile.mkdtemp()
    result = optimizer.save(path=tmp_dir)
    adam_path, cw_path = os.path.join(tmp_dir, "adam.l2l"), os.path.join(tmp_dir, "cw.l2l")
    assert result[adam_path] == {}
    assert set(result[cw_path]) == {"lstm_1", "lstm_2", "linear"}
    with open(adam_path, "rb") as fh:
        assert networks._pickle.load(fh) == {}
    with open(cw_path, "rb") as fh:
        assert np.allclose(networks._pickle.load(fh)["linear"]["w"], result[cw_path]["linear"]["w"])
    for p in (adam_path, cw_path):
        os.remove(p)
    os.rmdir(tmp_dir)
