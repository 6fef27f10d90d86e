"""Measures the hand-written update rules (networks.Sgd / networks.Adam) on the GPU and prints one JSON line:

  * step kernel: one Adam step (l2o_rule_step) over 32 M coordinates, 28 B per coordinate moved (g, x in/out, m and v
    in and out), so the working set is far past the 126 MB L2.  CUDA events over many launches after warm-up; achieved
    bytes/s against the project's measured HBM peak.
  * fused unroll: the Adam net on problems.rastrigin_separable(1_000_000), T = 100, through MetaOptimizer.meta_loss
    (inference: one launch for the T steps), beside the LSTM-20x2 inference unroll of the same problem.
  * consistency: the fused Adam unroll and T external-regime steps (torch autograd gradient + step kernel) give the same
    fx (REL_TOL) and x_T (X_REL_TOL) on the same seeded inputs; asserted after the line is printed.

The card's name, power limit and max SM clock are part of the line.  Nothing is written to the tree."""
import contextlib
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

REL_TOL = 1e-5
# x_T of the two regimes: torch autograd forms the Rastrigin gradient in another operation order than the in-kernel
# formula (last-bit differences of g), and the curvature 1 + 4 pi^2 alpha c cos(2 pi x) (up to ~400 |c|) amplifies them
# along 100 Adam steps; the worst of 1 M coordinates was measured at 2.3e-5 (B200), fx at 1.2e-7.
X_REL_TOL = 1e-4
HBM_PEAK_GBS = 6561.0   # measured HBM peak of the project's B200 (BASELINE.md section 2)
BYTES_PER_COORD = 28    # Adam step: g 4 + x 8 + m 8 + v 8


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else "unknown"
    except Exception as e:  # the numbers stay meaningful only with the card line: say why it is missing
        return "nvidia-smi unavailable: %r" % (e,)


def event_ms(fn, iters, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(iters):
        fn()
    end.record()
    end.synchronize()
    return start.elapsed_time(end) / iters


def step_kernel(n=32 << 20, iters=200, warmup=20):
    from open_l2o_b200.engine import RULE_ADAM, RuleHandle
    h = RuleHandle(RULE_ADAM, 1e-3)
    gen = torch.Generator(device="cuda").manual_seed(0)
    g = torch.randn(n, device="cuda", generator=gen)
    x = torch.randn(n, device="cuda", generator=gen)
    arenas = [h.new_state(n, "cuda"), h.new_state(n, "cuda")]
    k = [0]

    def one():
        h.step(g, arenas[k[0] % 2], arenas[(k[0] + 1) % 2], x=x)
        k[0] += 1
    ms = event_ms(one, iters, warmup)
    gbs = BYTES_PER_COORD * n / (ms * 1e-3) / 1e9
    return dict(n=n, us_per_step=round(ms * 1e3, 2), achieved_GB_s=round(gbs, 1),
                frac_of_measured_hbm_peak=round(gbs / HBM_PEAK_GBS, 3))


def unroll(net_config, n, T, iters, warmup):
    from open_l2o_b200 import meta, problems
    opt = meta.MetaOptimizer(net=net_config)
    ms_ops = opt.meta_loss(problems.rastrigin_separable(num_dims=n), T)
    assert opt.program.fused is not None
    sess = meta.Session()
    sess.run(ms_ops.reset)
    ms = event_ms(lambda: sess.run(ms_ops.loss), iters, warmup)
    out = dict(n=n, T=T, ms_per_unroll=round(ms, 3), coord_updates_per_s=float("%.4g" % (n * T / (ms * 1e-3))))
    del opt, ms_ops, sess
    torch.cuda.empty_cache()
    return out


def consistency(n, T):
    """One fused Adam unroll vs T external-regime steps, same seed (same x_0 and constants)."""
    from open_l2o_b200 import meta, problems
    cfg = {"net": "Adam", "net_options": {"learning_rate": 1e-3}}
    res = []
    for disable in ("0", "1"):
        os.environ["L2O_DISABLE_FUSED"] = disable
        opt = meta.MetaOptimizer(net=cfg)
        ms_ops = opt.meta_loss(problems.rastrigin_separable(num_dims=n), T)
        assert (opt.program.fused is None) == (disable == "1")
        sess = meta.Session()
        sess.run(ms_ops.reset)
        sess.run([ms_ops.loss, ms_ops.update])
        res.append((opt.program.last_fx.double().cpu(), opt.program.X.double().cpu()))
        del opt, ms_ops, sess
    os.environ.pop("L2O_DISABLE_FUSED")

    def rel(a, b):
        return float((a - b).abs().max() / b.abs().max())
    return dict(n=n, T=T, fx_rel_err=rel(res[0][0], res[1][0]), x_rel_err=rel(res[0][1], res[1][1]), fx_tol=REL_TOL,
                x_tol=X_REL_TOL)


def main():
    if not torch.cuda.is_available():
        raise SystemExit("rule_bench.py measures on a CUDA device; none is visible")
    n, T = 1_000_000, 100
    with contextlib.redirect_stdout(sys.stderr):   # program construction prints variable lists; stdout = one JSON line
        line = dict(card=card(), step_kernel=step_kernel(),
                    adam_fused_unroll=unroll({"net": "Adam", "net_options": {"learning_rate": 1e-3}}, n, T, 20, 3),
                    lstm20x2_inference_unroll=unroll({"net": "CoordinateWiseDeepLSTM",
                                                      "net_options": {"layers": (20, 20)}}, n, T, 10, 2),
                    consistency=consistency(n, T))
    print(json.dumps(line), flush=True)
    c = line["consistency"]
    assert c["fx_rel_err"] <= REL_TOL and c["x_rel_err"] <= X_REL_TOL, c


if __name__ == "__main__":
    main()
