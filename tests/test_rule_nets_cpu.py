"""CPU-only tests of the hand-written update rules (networks.Sgd / networks.Adam, DM/networks.py:354-420): the oracle
against what the reference states or implies, argument validation of the l2o_rule_* entry points before any CUDA
call, and the simple-multi config (DM/util.py:122-135)."""
import ctypes
import os

import pytest
import torch

from oracle import l2o_oracle as orc
from tests import rule_oracle as ro
from open_l2o_b200 import _lib


def test_oracle_sgd_is_minus_lr_times_g():
    g = torch.randn(257, generator=torch.Generator().manual_seed(0))
    upd, state = ro.rule_apply(ro.RuleSpec("sgd", learning_rate=0.01), g, ro.rule_initial_state(
        ro.RuleSpec("sgd"), g.numel()))
    assert torch.equal(upd, -0.01 * g) and state == ()


def test_oracle_adam_zero_learning_rate_gives_zeros():
    rule = ro.RuleSpec("adam", learning_rate=0)
    g = torch.randn(10, generator=torch.Generator().manual_seed(1))
    state = ro.rule_initial_state(rule, 10)
    for _ in range(3):
        upd, state = ro.rule_apply(rule, g, state)
        assert torch.equal(upd, torch.zeros(10))
    assert float(state[0]) == 3.0


def test_oracle_adam_constant_gradient():
    """Under a constant gradient both debiased moments are exact: step k is -lr*g/(|g|+eps) up to fp32 rounding.  The
    largest part of that rounding is TF's: fp32(0.999) + fp32(1 - 0.999) = 1 + 1.3e-8, and v' = b2 v + (1-b2) g^2
    debiased by 1 - fp32(b2)^t then overshoots g^2 by up to 1.3e-5 (6.5e-6 after the square root); measured 1.03e-5
    in all, hence 2e-5."""
    rule = ro.RuleSpec("adam", learning_rate=0.003)
    g = torch.randn(1000, generator=torch.Generator().manual_seed(2)) * torch.logspace(-3, 2, 1000)
    state = ro.rule_initial_state(rule, g.numel())
    want = -0.003 * g.double() / (g.double().abs() + 1e-8)
    for k in range(1, 31):
        upd, state = ro.rule_apply(rule, g, state)
        assert float(state[0]) == k
        assert float((upd.double() - want).abs().max() / want.abs().max()) < 2e-5, k


def test_oracle_mixed_unroll_single_assignment_is_unroll():
    spec = orc.NetSpec(layers=(20, 20), scale=0.1)
    theta = orc.init_theta(spec, seed=3)
    gen = torch.Generator().manual_seed(4)
    n, T = 50, 6
    a, b, x0 = torch.randn(n, generator=gen), torch.randn(n, generator=gen), torch.randn(n, generator=gen)
    prob = orc.FusedProblem("rastrigin_sep", a, b, alpha=10.0, fscale=1.0 / n)
    ref = orc.unroll(spec, theta, x0, orc.initial_state(spec, n), None, T, grad_of=prob.f_and_g)
    res = ro.mixed_unroll([((spec, theta), slice(0, n))], x0, [orc.initial_state(spec, n)], None, T,
                           grad_of=prob.f_and_g)
    assert torch.equal(res.fx, ref.fx) and torch.equal(res.x_final, ref.x_final)
    g_ref, _ = orc.meta_grad(spec, theta, x0, orc.initial_state(spec, n), None, T, grad_of=prob.f_and_g)
    (g,), _ = ro.mixed_meta_grad([((spec, theta), slice(0, n))], x0, [orc.initial_state(spec, n)], None, T,
                                  grad_of=prob.f_and_g)
    assert torch.equal(g, g_ref)


def test_oracle_mixed_rule_coordinates_only_feed_gradients():
    """With a rule on the other half of a separable optimizee the learned net's meta-gradient is the one it has alone."""
    spec = orc.NetSpec(layers=(1,))
    theta = orc.init_theta(spec, seed=5)
    x0 = torch.randn(8, generator=torch.Generator().manual_seed(6))

    def f(x):
        return torch.sum(x * x)
    rule = ro.RuleSpec("adam", learning_rate=0.1)
    (g_mixed, none), _ = ro.mixed_meta_grad([((spec, theta), slice(0, 4)), (rule, slice(4, 8))], x0,
                                             [orc.initial_state(spec, 4), ro.rule_initial_state(rule, 4)], f, 4)
    (g_alone,), _ = ro.mixed_meta_grad([((spec, theta), slice(0, 4))], x0[:4], [orc.initial_state(spec, 4)], f, 4)
    assert none is None and torch.allclose(g_mixed, g_alone, rtol=1e-6, atol=0)


# ---- the C-ABI: validation happens before any CUDA call --------------------------------------------------------------
needs_lib = pytest.mark.skipif(not os.path.exists(_lib.LIB_PATH), reason="library not built")


def _desc(kind=_lib.RULE_ADAM, lr=1e-3, b1=0.9, b2=0.999, eps=1e-8):
    d = _lib.RuleDesc()
    d.kind, d.learning_rate, d.beta1, d.beta2, d.epsilon = kind, lr, b1, b2, eps
    return d


@needs_lib
def test_rule_state_floats():
    L = _lib.lib()
    out = ctypes.c_int64(-7)
    assert L.l2o_rule_state_floats(ctypes.byref(_desc(_lib.RULE_SGD)), 1000, ctypes.byref(out)) == _lib.L2O_OK
    assert out.value == 0
    for n in (0, 1, 1_000_003):
        assert L.l2o_rule_state_floats(ctypes.byref(_desc()), n, ctypes.byref(out)) == _lib.L2O_OK
        assert out.value == 4 + 2 * n
    assert L.l2o_rule_state_floats(ctypes.byref(_desc()), -1, ctypes.byref(out)) == _lib.L2O_E_INVALID
    assert L.l2o_rule_state_floats(ctypes.byref(_desc()), 5, None) == _lib.L2O_E_INVALID
    assert L.l2o_rule_state_floats(None, 5, ctypes.byref(out)) == _lib.L2O_E_INVALID


@needs_lib
@pytest.mark.parametrize("desc", [
    dict(kind=2), dict(kind=-1), dict(lr=-1e-3), dict(b1=1.0), dict(b1=-0.1), dict(b2=1.0), dict(b2=float("nan")),
])
def test_rule_bad_descriptor(desc):
    L = _lib.lib()
    d = _desc(**desc)
    out = ctypes.c_int64()
    assert L.l2o_rule_state_floats(ctypes.byref(d), 4, ctypes.byref(out)) == _lib.L2O_E_INVALID
    buf = (ctypes.c_float * 64)()
    a = _lib.RuleStepArgs(n=4, g=ctypes.addressof(buf), state_in=ctypes.addressof(buf) + 64,
                          state_out=ctypes.addressof(buf) + 128)
    assert L.l2o_rule_step(ctypes.byref(d), ctypes.byref(a), None) == _lib.L2O_E_INVALID
    with pytest.raises(_lib.L2OError):
        from open_l2o_b200.engine import RuleHandle
        RuleHandle(d.kind, d.learning_rate, d.beta1, d.beta2, d.epsilon)


@needs_lib
def test_rule_step_validation():
    L = _lib.lib()
    buf = (ctypes.c_float * 256)()
    p = ctypes.addressof(buf)
    n = 8                                  # Adam arena: 4 + 2n = 20 floats = 80 bytes
    adam, sgd = _desc(), _desc(_lib.RULE_SGD)

    def step(d, **kw):
        a = _lib.RuleStepArgs(**kw)
        return L.l2o_rule_step(ctypes.byref(d), ctypes.byref(a), None)
    assert step(adam, n=n, g=None, state_in=p, state_out=p + 512) == _lib.L2O_E_INVALID            # no gradient
    assert step(adam, n=-1, g=p, state_in=p + 128, state_out=p + 512) == _lib.L2O_E_INVALID        # n < 0
    assert step(adam, n=n, g=p, state_in=None, state_out=p + 512) == _lib.L2O_E_INVALID            # no state
    assert step(adam, n=n, g=p, state_in=p + 128, state_out=None) == _lib.L2O_E_INVALID
    assert step(adam, n=n, g=p, state_in=p + 128, state_out=p + 128) == _lib.L2O_E_INVALID         # aliasing
    assert step(adam, n=n, g=p, state_in=p + 128, state_out=p + 128 + 76) == _lib.L2O_E_INVALID    # overlap
    assert step(adam, n=n, g=p, state_in=p + 128 + 76, state_out=p + 128) == _lib.L2O_E_INVALID
    assert step(adam, n=0, g=p, state_in=None, state_out=p) == _lib.L2O_E_INVALID
    assert step(sgd, n=0, g=p) == _lib.L2O_OK                                                       # nothing to do
    assert step(sgd, n=n, g=None) == _lib.L2O_E_INVALID
    assert step(_desc(kind=7), n=n, g=p) == _lib.L2O_E_INVALID
    assert L.l2o_rule_step(ctypes.byref(adam), None, None) == _lib.L2O_E_INVALID


@needs_lib
def test_rule_unroll_validation():
    L = _lib.lib()
    buf = (ctypes.c_float * 64)()
    p = ctypes.addressof(buf)
    fx = (ctypes.c_double * 8)()

    def unroll(d=None, **kw):
        base = dict(n=4, T=3, opt_kind=_lib.OPT_RASTRIGIN_SEP, opt_a=p, opt_b=p + 16, opt_alpha=10.0, opt_fscale=1.0,
                    x=p + 32, state=p + 64, fx=ctypes.addressof(fx))
        base.update(kw)
        a = _lib.RuleUnrollArgs(**base)
        return L.l2o_rule_unroll_fwd(ctypes.byref(d or _desc()), ctypes.byref(a), None)
    for kind in (_lib.OPT_QUADRATIC_BATCH, _lib.OPT_NONE):
        assert unroll(opt_kind=kind) == _lib.L2O_E_UNSUPPORTED
        assert unroll(_desc(_lib.RULE_SGD), opt_kind=kind) == _lib.L2O_E_UNSUPPORTED
    assert unroll(opt_kind=9) == _lib.L2O_E_INVALID
    assert unroll(opt_kind=-1) == _lib.L2O_E_INVALID
    assert unroll(n=-1) == _lib.L2O_E_INVALID
    assert unroll(T=-1) == _lib.L2O_E_INVALID
    assert unroll(x=None) == _lib.L2O_E_INVALID
    assert unroll(opt_a=None) == _lib.L2O_E_INVALID
    assert unroll(opt_b=None) == _lib.L2O_E_INVALID
    assert unroll(state=None) == _lib.L2O_E_INVALID                 # Adam needs its state
    assert unroll(_desc(b2=1.5)) == _lib.L2O_E_INVALID
    assert unroll(n=0) == _lib.L2O_OK                              # nothing to do
    assert L.l2o_rule_unroll_fwd(ctypes.byref(_desc()), None, None) == _lib.L2O_E_INVALID


def test_rule_structs_follow_the_header_field_order():
    from tests.test_lib_abi import _struct_fields
    for cname, cls in [("l2o_rule_desc", _lib.RuleDesc), ("l2o_rule_step_args", _lib.RuleStepArgs),
                       ("l2o_rule_unroll_args", _lib.RuleUnrollArgs)]:
        assert [f[0] for f in cls._fields_] == _struct_fields(cname), cname


def test_get_config_simple_multi():
    """DM/util.py:122-135."""
    from open_l2o_b200 import util
    problem, net_config, net_assignments = util.get_config("simple-multi", path="/some/where")
    assert net_config == {
        "cw": {"net": "CoordinateWiseDeepLSTM", "net_options": {"layers": (), "initializer": "zeros"},
               "net_path": "/some/where"},
        "adam": {"net": "Adam", "net_options": {"learning_rate": 0.01}},
    }
    assert net_assignments == [("cw", ["x_0"]), ("adam", ["x_1"])]
    assert callable(problem)


@needs_lib
def test_rule_nets_have_no_variables_and_factory_options():
    from open_l2o_b200 import networks
    for net in (networks.factory("Sgd"), networks.factory("Adam", {"learning_rate": 0.01})):
        assert net.variable_shapes() == [] and net.get_variables() == [] and networks.save(net) == {}
    assert networks.Sgd().name == "sgd" and networks.Adam().name == "adam"
    with pytest.raises(TypeError):
        networks.factory("Adam", {"learning_rte": 0.01})
    with pytest.raises(TypeError):
        networks.factory("Sgd", {"beta1": 0.9})
