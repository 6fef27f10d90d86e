#!/usr/bin/env python
"""bench.py - coordinate-updates/sec of the learned-optimizer inner loop (BASELINE.json metric).

A "step" is one full ``meta_minimize`` unroll of the hot path: T-step forward unroll (fused, state
on-chip) + BPTT + d-theta reduction [+ one NCCL all-reduce at N>1] + TF-Adam, through the public
``MetaOptimizer`` / ``Session.run([fx, update, step])`` surface.  Workload (default): BASELINE config #5,
L2O-DM (LSTM-20x2, identity preprocess) on separable Rastrigin, 1M coordinates PER GPU (weak scaling),
unroll T=100.  Synthetic data, random-init weights (seeded).

  python bench.py --gpus 1 --steps 5 --warmup 3
  python bench.py --gpus 1 --steps 5 --warmup 3 --dump-outputs DIR   # + the last timed step's outputs as DIR/*.npy
  torchrun --nproc-per-node N ... bench.py --gpus N ...
  python bench.py --impl reference ...     # the CPU oracle (port of the reference's algorithm) on host cores
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

FLOP_PER_UPDATE_INFER = {"dm_identity": 9800.0, "dm_logsign": 9960.0, "rnnprop": 12920.0}  # SURVEY.md 8(d)
C_SF_BYTES = 320  # LSTM-20x2 checkpoint row per coordinate-update
METRIC = "coordinate-updates/sec (N_params x unroll_steps)"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="rastrigin",
                    choices=["rastrigin", "lasso", "mlp", "rnnprop_mlp", "quadratic", "hrnn_convnet"])
    ap.add_argument("--coords", type=int, default=0, help="coordinates per GPU (0 = workload default)")
    ap.add_argument("--unroll", type=int, default=0, help="T (0 = workload default)")
    ap.add_argument("--engine", default="auto", choices=["auto", "ffma", "tc"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-also", action="store_true", help="skip the short runs of the other BASELINE configs (N=1 default run)")
    ap.add_argument("--cpu-sample-coords", type=int, default=0,
                    help="coordinates of the CPU-oracle sample (0 = best of the workload's default sample sizes)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --coords per GPU (default 1M each); strong: --coords in TOTAL (default 1M) sharded over the ranks")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed meta-step computed as DIR/<name>.npy "
                         "(rank 0's view; under 64 MB in all) so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and (args.impl != "ours" or args.workload == "hrnn_convnet"):
        ap.error("--dump-outputs covers the MetaOptimizer workloads of --impl ours")
    return args


# ------------------------------------------------------------------------------------------------
WORKLOADS = {
    # name: (description, default coords/GPU, default T, net kind)
    "rastrigin": ("L2O-DM, separable Rastrigin d=1e6 per GPU, LSTM-20x2 identity, unroll=100 (BASELINE config #5)",
                  1000000, 100, "dm_identity"),
    "lasso": ("L2O-DM, Lasso m=250 n=500 batch=128 synthetic, unroll=100 (BASELINE config #2)", 64000, 100,
              "dm_identity"),
    "mlp": ("L2O-DM LogAndSign, 1M-coordinate MLP 784-1263-10 synthetic batch 128, unroll=20 (target line)",
            1004105, 20, "dm_logsign"),
    "rnnprop_mlp": ("L2O-RNNProp, MLP 784-100-10 synthetic batch 128, unroll=20 (BASELINE config #3)", 79510, 20,
                    "rnnprop"),
    "quadratic": ("L2O-DM, quadratic 128x10, unroll=20 (BASELINE config #1; the reference's CPU-runnable case)", 1280,
                  20, "dm_identity"),
}
# Net output scale per workload.  The reference's synthetic-problem configs are {"layers": (20, 20)} => scale 1.0
# (DM/util.py:136-143,231-246); with RANDOM-INIT weights (no trained .l2l exists offline) scale 1.0 drives x to
# overflow within an unroll of 100, so the synthetic workloads run the same net at scale 0.1 (SURVEY.md 8(d): "final
# Linear x0.1 so trajectories stay finite").  The arithmetic per coordinate-update does not depend on it.
NET_SCALE = {"rastrigin": 0.1, "lasso": 0.1, "quadratic": 0.1, "mlp": 0.01, "rnnprop_mlp": 0.01}
# step-at-a-time regime, SURVEY.md 8(d): state 640 + g 4 + x 8 (+ m, v 8 for RNNProp) per coordinate-update forward;
# the BPTT sweep reads the checkpoint row (320) + the recorded gradient and net input (8) again
STEP_BYTES = {"dm_identity": 652.0, "dm_logsign": 652.0, "rnnprop": 668.0}
BWD_BYTES = {"dm_identity": 328.0, "dm_logsign": 328.0, "rnnprop": 336.0}


def make_problem(name, coords, rank, shard=None):
    from open_l2o_b200 import problems
    if name == "rastrigin":
        return problems.rastrigin_separable(num_dims=coords, shard=shard), {"cw": {
            "net": "CoordinateWiseDeepLSTM", "net_options": {"layers": (20, 20), "scale": 0.1}}}, "dm"
    if name == "quadratic":
        return problems.quadratic(batch_size=128, num_dims=10), {"cw": {"net": "CoordinateWiseDeepLSTM", "net_options": {
            "layers": (20, 20), "scale": 0.1}}}, "dm"
    if name == "lasso":
        g = torch.Generator().manual_seed(2 + rank)
        A = torch.randn(128, 250, 500, generator=g) / (250 ** 0.5)
        b = torch.randn(128, 250, 1, generator=g)
        return problems.lasso_fixed(A, b), {"cw": {"net": "CoordinateWiseDeepLSTM", "net_options": {
            "layers": (20, 20), "scale": 0.1}}}, "dm"
    if name == "mlp":
        from open_l2o_b200 import util
        return problems.mlp(layers=(1263,)), {"cw": util.get_default_net_config(None)}, "dm"
    if name == "rnnprop_mlp":
        return problems.mlp(layers=(100,)), {"rp": {"net": "RNNprop", "net_options": {
            "layers": (20, 20), "preprocess_name": "fc", "preprocess_options": {"dim": 20}, "scale": 0.01,
            "tanh_output": True}}}, "rnnprop"
    raise ValueError(name)


DUMP_BYTES = 60 << 20   # array data of --dump-outputs; with the .npy headers the files stay under 64 MB


def last_step_outputs(prog):
    """What the last ``Session.run([fx, update, step])`` hands its caller: the objective over the unroll (``fx[T]`` is
    the fetched fx), the optimizee's coordinates after the committed update and each net's weights after TF-Adam."""
    out = {"fx": prog.last_fx.double(), "x": prog.X.float()}
    for key, net in prog.nets.items():
        out["theta_" + key] = net.theta.detach().float()
    return {name: t.detach().cpu().numpy().reshape(-1) for name, t in out.items()}


def dump_outputs(outdir, arrays):
    """Write each array as ``outdir/<name>.npy``, DUMP_BYTES in all.  The smaller arrays are kept whole; one that does
    not fit its share is cut to a seeded sample of its elements, the same indices in every run of the same size."""
    os.makedirs(outdir, exist_ok=True)
    import numpy as np
    names = sorted(arrays, key=lambda k: arrays[k].nbytes)
    left = DUMP_BYTES
    for i, name in enumerate(names):
        a = arrays[name]
        cap = left // (len(names) - i) // a.itemsize
        if a.size > cap:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, cap, replace=False))]
        np.save(os.path.join(outdir, name + ".npy"), a)
        left -= a.nbytes


class ClockSampler(threading.Thread):
    """nvidia-smi clock / throttle-reason sampler (B200_PROFILING.md): one streaming `nvidia-smi -lms` process; only
    samples whose arrival time falls inside [t_begin, t_end] of the timed region are summarised."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.proc = index, [], None
        self.t_begin, self.t_end = None, None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "50"], stdout=subprocess.PIPE, text=True)
            for line in self.proc.stdout:
                parts = [p.strip() for p in line.strip().split(",")]
                if len(parts) >= 6:
                    self.samples.append((time.perf_counter(), parts))
        except Exception:
            pass

    def stop(self):
        if self.proc is not None:
            try:
                self.proc.terminate()
            except Exception:
                pass

    def summary(self):
        inside = [p for (ts, p) in self.samples if self.t_begin is not None and self.t_begin <= ts <= self.t_end]
        use = inside if inside else [p for (_, p) in self.samples]
        if not use:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(int(float(s[0])) for s in use)
        reasons = set()
        for s in use:
            for name, val in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], s[2:6]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": int(float(use[0][1])), "reasons": sorted(reasons),
                "samples": len(sm), "samples_in_timed_region": len(inside)}


def _peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def external_roofline(prog, netkind, T, t_unroll):
    """HBM roofline of the step-at-a-time (external-gradient) regime, SURVEY.md 8(d): one `l2o_step` launch moves
    652 B (668 B RNNProp) per coordinate; the BPTT sweep re-reads 328 B.  The step kernel and the BPTT kernel are timed
    ALONE here with CUDA events on this workload's own buffers (inside the captured graph they cannot be bracketed)."""
    from open_l2o_b200 import engine as eng
    peaks = _peaks()
    peak = float(peaks.get("hbm_gbs", 6500.0))
    r = prog.runs[0]
    h = r.net.handle
    n = r.n
    slot = max(h.state_size(n), 1)
    xw = prog.X.clone()
    kw = {}
    if h.n_in == 2:
        kw = dict(m=r.m_work, v=r.v_work, beta1=prog.opt.beta1, beta2=prog.opt.beta2, step_ptr=prog.step_dev,
                  t_offset=0, feat_out=r.feat_rec[0])
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn, reps):
        fn()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / 1e3 / reps
    # walk the checkpoint slots so consecutive launches touch different state rows (no L2 reuse between launches)
    idx = [0]

    def step_once():
        t = idx[0] % T
        idx[0] += 1
        h.step(r.net.theta, r.g_rec[t], r.ckpt[t * slot:(t + 1) * slot], r.ckpt[(t + 1) * slot:(t + 2) * slot],
               x=xw[r.off:r.off + n], **kw)
    t_step = timed(step_once, 2 * T)
    dth = torch.zeros_like(prog.dtheta[r.key])
    in_seq = r.feat_rec if h.n_in == 2 else r.g_rec
    t_bwd = timed(lambda: h.unroll_bwd(r.net.theta, n, T, in_seq, r.ckpt, dth, g_rec=r.g_rec, **prog._bwd_extra(r)), 3)
    sb, bb = STEP_BYTES[netkind], BWD_BYTES[netkind]
    ach = sb * n / t_step / 1e9
    step_traffic = None   # measured DRAM bytes of one l2o_step launch (ncu --set full capture of the DM step kernel)
    if netkind != "rnnprop":
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            step_traffic = tj["step_dram_bytes_per_coord_update"] * n
        except Exception:
            pass
    ws = (T + 1) * slot * 4
    return {"bound": "hbm", "kernel": "l2o_step (one coordinate-wise LSTM step, state in HBM)", "achieved": ach,
            "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": step_traffic,
            "algorithmic_bytes_per_coord_update": sb, "step_us": 1e6 * t_step, "coord_updates_per_s_step_kernel": n / t_step,
            "bptt": {"kernel": "l2o_unroll_bwd over the T checkpoint slots", "ms": 1e3 * t_bwd,
                     "algorithmic_bytes_per_coord_update": bb, "achieved": bb * n * T / t_bwd / 1e9,
                     "frac": bb * n * T / t_bwd / 1e9 / peak, "coord_updates_per_s": n * T / t_bwd},
            "train_unroll": {"algorithmic_bytes_per_coord_update": sb + bb,
                             "achieved": (sb + bb) * n * T / t_unroll / 1e9,
                             "frac": (sb + bb) * n * T / t_unroll / 1e9 / peak,
                             "note": "whole unroll incl. the optimizee's own forward/backward (torch autograd) and Adam"},
            "working_set_bytes": ws, "l2_resident": bool(ws < 126e6),
            "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6.5 TB/s (B200_PROFILING.md)"}


def quick_measure(workload, steps, warmup, with_cpu=True):
    """Short device-resident train-mode measurement of another BASELINE config through the same public surface
    (MetaOptimizer.meta_minimize + Session.run([fx, update, step])); reported under "also" at N=1 with its own
    roofline and CPU baseline."""
    from open_l2o_b200 import engine as eng, meta
    desc, coords, T, netkind = WORKLOADS[workload]
    problem, net_config, flavour = make_problem(workload, coords, 0)
    cls = meta.RNNpropMetaOptimizer if flavour == "rnnprop" else meta.MetaOptimizer
    optimizer = cls(_seed=0, **net_config)
    _stdout = sys.stdout
    sys.stdout = open(os.devnull, "w")
    try:
        ms = optimizer.meta_minimize(problem, T, learning_rate=0.001)
    finally:
        sys.stdout = _stdout
    prog = optimizer.program
    sess = meta.Session()
    sess.run(ms.reset)
    fetch = [ms.fx, ms.update, ms.step]
    for _ in range(warmup):
        sess.run(fetch)
    torch.cuda.synchronize()
    l0 = eng.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        cost = sess.run(fetch)[0]
    e1.record()
    torch.cuda.synchronize()
    t = e0.elapsed_time(e1) / 1e3
    launches = int(eng.launch_count() - l0)
    out = {"workload": desc, "coords": prog.N, "unroll": T, "mode": "train (fwd+BPTT+Adam)",
           "regime": "fused" if prog.fused is not None else (
               "external-gradient (%s between step kernels, one captured CUDA graph per unroll)" % (
                   "gradient producer '%s'" % prog.producer.kind if prog.producer is not None else "torch autograd")),
           "value": prog.N * T * steps / t, "unit": "coordinate-updates/s",
           "ms_per_step": 1e3 * t / steps, "steps": steps, "warmup": warmup,
           "gpu_launches": launches, "last_fx": cost, "net_scale": NET_SCALE[workload]}
    out["roofline"] = external_roofline(prog, netkind, T, t / steps)
    if with_cpu:
        try:
            out["cpu_baseline"] = cpu_baseline_for(workload, T, pick_cpu_threads(), timed=1)
            out["vs_cpu_baseline"] = out["value"] / out["cpu_baseline"]["value"]
        except Exception as ex:
            out["cpu_baseline"] = {"error": repr(ex)[:200]}
    prog._graphs.clear()
    del sess, ms, prog, optimizer, problem
    import gc
    gc.collect()
    torch.cuda.empty_cache()
    return out


def quick_measure_hrnn(steps, warmup, T=20, batch=128):
    """BASELINE config #4: L2O-Scale HierarchicalRNN [10,20,20] optimizing a ConvNet on CIFAR-shaped synthetic data
    (354,218 coordinates, unroll 20; inference path = the update step; SURVEY.md 8(f) row 1).  Also times the
    step's three kernels alone on a large synthetic state for the HBM roofline of the per-coordinate kernel."""
    from open_l2o_b200 import engine as eng, hierarchical_rnn as hr
    from open_l2o_b200.scale_problems import ConvNet
    dev = torch.device("cuda", torch.cuda.current_device())
    prob = ConvNet((3, 32, 32), 10, [(3, 3, 32), (5, 5, 32)])
    params = prob.init_tensors(seed=1, device=dev)
    gen = torch.Generator().manual_seed(2)
    data = torch.rand(batch, 32, 32, 3, generator=gen).to(dev)
    labels = torch.nn.functional.one_hot(torch.randint(10, (batch,), generator=gen), 10).float().to(dev)
    opt = hr.HierarchicalRNN(random_seed=0, **hr.metarun_flags())

    def objective(*ps):
        return prob.objective(list(ps), data, labels)

    def unroll():   # the public call: T optimizer steps, objective values read back at the end
        return opt.minimize(objective, params, T)[-1]
    for _ in range(warmup):
        unroll()
    torch.cuda.synchronize()
    l0 = eng.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss = unroll()
    e1.record()
    torch.cuda.synchronize()
    t = e0.elapsed_time(e1) / 1e3
    n = opt.N
    launches = int(eng.launch_count() - l0)
    # the optimizer step alone (3 launches), same state
    e0.record()
    for _ in range(steps * T):
        opt.step_flat()
    e1.record()
    torch.cuda.synchronize()
    t_step = e0.elapsed_time(e1) / 1e3 / (steps * T)
    out = {"workload": "L2O-Scale HierarchicalRNN [10,20,20], ConvNet 3x32x32 [(3,3,32),(5,5,32)] synthetic batch %d, "
                       "unroll=%d (BASELINE config #4)" % (batch, T),
           "coords": n, "unroll": T, "mode": "infer (the optimizer step); meta-training measured under \"meta_train\"",
           "regime": "external-gradient (torch autograd ConvNet forward/backward between l2o_hrnn_step calls; one "
                     "iteration captured as a CUDA graph by HierarchicalRNN.minimize)",
           "value": n * T * steps / t, "unit": "coordinate-updates/s", "ms_per_step": 1e3 * t / steps, "steps": steps,
           "warmup": warmup, "gpu_launches": launches, "last_fx": float(loss),
           "optimizer_step_us": 1e6 * t_step}
    # meta-training of the optimizer itself on the same optimizee (hrnn_train.MetaTrainer.train_step: T-step unroll,
    # BPTT through it, clipped RMSProp; SC/optimizer/trainable_optimizer.py:200-470)
    try:
        from open_l2o_b200 import hrnn_train as ht
        tr = ht.MetaTrainer(prob.param_shapes, device=str(dev), random_seed=0)
        p0 = [p.detach() for p in params]
        obj_list = lambda ps: prob.objective(ps, data, labels)
        tr.train_step(obj_list, p0, T)
        torch.cuda.synchronize()
        reps = 3
        e0.record()
        for _ in range(reps):
            meta = tr.train_step(obj_list, p0, T)[0]
        e1.record()
        torch.cuda.synchronize()
        t_mt = e0.elapsed_time(e1) / 1e3 / reps
        out["meta_train"] = {"ms_per_meta_step": 1e3 * t_mt, "coordinate_updates_per_s": n * T / t_mt,
                             "meta_objective": float(meta),
                             "what": "one unroll of T steps forward (tcgen05 step kernel) + BPTT (l2o_hrnn_coord_bwd, per-tensor "
                                     "pieces by torch autograd) + RMSProp on the 8,349 optimizer weights; eager, no CUDA graph"}
        del tr
    except Exception as ex:   # reported, never fatal for the headline line
        out["meta_train"] = {"error": repr(ex)[:200]}
    del opt, params
    # HBM roofline of the step on a state that does not fit L2: 16 tensors x 2M coordinates
    sizes = [2_000_000] * 16
    big = [torch.zeros(sz, device=dev).requires_grad_(True) for sz in sizes]
    opt2 = hr.HierarchicalRNN(random_seed=0, **hr.metarun_flags())
    g = [torch.randn(sz, device=dev) * 0.1 for sz in sizes]
    opt2.apply_gradients(zip(g, big))
    for _ in range(3):
        opt2.step_flat()
    torch.cuda.synchronize()
    reps = 10
    e0.record()
    for _ in range(reps):
        opt2.step_flat()
    e1.record()
    torch.cuda.synchronize()
    t_big = e0.elapsed_time(e1) / 1e3 / reps
    nbig = opt2.N
    bytes_per = 192.0   # coord kernel 88 B read + 88 B written, apply kernel 16 B (DESIGN.md 3.4)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6500.0))
    ach = bytes_per * nbig / t_big / 1e9
    out["roofline"] = {"bound": "hbm", "kernel": "l2o::hrnn::tcg::coord_tc_kernel + tensor_kernel + apply_kernel (one l2o_hrnn_step)",
                       "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": 174.41 * nbig,   # dram bytes of coord_tc_kernel per launch (ncu --set full, profiles/r02j_hrnn_coord_tc.raw.csv)
                       "coords": nbig, "ms": 1e3 * t_big, "coord_updates_per_s": nbig / t_big,
                       "algorithmic_bytes_per_coord_update": bytes_per,
                       "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6.5 TB/s"}
    del opt2, big, g
    torch.cuda.empty_cache()
    return out


def pick_cpu_threads():
    """All host cores the op-for-op CPU path can actually use: intra-op threading of [N,80]-sized tensors stops
    scaling (and then regresses) beyond a few dozen threads, so cap at 32 and report the number used."""
    return max(1, min(os.cpu_count() or 1, 32))


CPU_SAMPLES = {"rastrigin": (8192, 32768), "mlp": (15910,), "lasso": (2000,), "rnnprop_mlp": (15910,), "quadratic": (1280,)}


def cpu_oracle_unroll(workload, T, coords, threads, mode="train"):
    """One unroll of the oracle (CPU restatement of the reference's algorithm, torch-CPU ops on all usable host
    cores) on a bounded SAMPLE of `workload`: same net, same optimizee family, same T, `coords` coordinates instead of
    the GPU arm's.  Returns (callable timing one unroll, coordinates of the sample, description)."""
    from oracle import l2o_oracle as orc   # bench.py's cpu_baseline / --impl reference leg only
    torch.set_num_threads(threads)
    gen = torch.Generator().manual_seed(1)
    grad_of, f = None, None
    if workload == "rastrigin":
        spec = orc.NetSpec(layers=(20, 20), scale=NET_SCALE[workload])
        a, b, x0 = (torch.randn(coords, generator=gen) for _ in range(3))
        grad_of = orc.FusedProblem("rastrigin_sep", a, b, 10.0, 1.0 / coords).f_and_g
        what = "separable Rastrigin d=%d" % coords
    elif workload == "quadratic":
        spec = orc.NetSpec(layers=(20, 20), scale=NET_SCALE[workload])
        B = max(1, coords // 10)
        w, y = torch.rand(B, 10, 10, generator=gen), torch.rand(B, 10, generator=gen)
        x0 = torch.randn(B, 10, generator=gen) * 0.01
        f = lambda x: orc.quadratic_f(x, w, y)   # noqa: E731
        what = "quadratic batch %d x 10" % B
    elif workload == "lasso":
        spec = orc.NetSpec(layers=(20, 20), scale=NET_SCALE[workload])
        B = max(1, coords // 500)
        A = torch.randn(B, 250, 500, generator=gen) / (250 ** 0.5)
        bb = torch.randn(B, 250, 1, generator=gen)
        x0 = torch.randn(B, 500, generator=gen) * 0.01
        f = lambda x: orc.lasso_f(x, A, bb)      # noqa: E731
        what = "Lasso m=250 n=500 batch %d (of the GPU arm's 128)" % B
    elif workload in ("mlp", "rnnprop_mlp"):
        if workload == "mlp":
            spec = orc.NetSpec(layers=(20, 20), preprocess_name="LogAndSign", preprocess_options={"k": 5}, scale=0.01)
        else:
            spec = orc.NetSpec(layers=(20, 20), preprocess_name="fc", preprocess_options={"dim": 20}, scale=0.01,
                               tanh_output=True, rnnprop=True)
        hid = max(1, round((coords - 10) / 795.0))       # 784 h + h + 10 h + 10
        data = torch.rand(128, 784, generator=gen)
        labels = torch.randint(0, 10, (128,), generator=gen)
        shapes = [(784, hid), (hid,), (hid, 10), (10,)]
        n = sum(a * (b[0] if b else 1) for a, *b in shapes)
        x0 = torch.randn(n, generator=gen) * 0.01

        def f(xf):
            off, ts = 0, []
            for sh in shapes:
                k = 1
                for d in sh:
                    k *= d
                ts.append(xf[off:off + k].view(sh))
                off += k
            h = torch.sigmoid(data @ ts[0] + ts[1])
            return torch.nn.functional.cross_entropy(h @ ts[2] + ts[3], labels)
        what = "sigmoid MLP 784-%d-10, synthetic batch 128 (the GPU arm's optimizee at reduced width)" % hid
    else:
        raise ValueError(workload)
    theta = orc.init_theta(spec, seed=0, out_gain=1.0)
    tr = orc.MetaTrainerOracle(spec, theta, f, lr=0.001, grad_of=grad_of)
    tr.reset(x0)
    n = x0.numel()

    def one(T_=T):
        t0 = time.perf_counter()
        tr.run_unroll(T_, train=(mode == "train"))
        return time.perf_counter() - t0
    return one, n, what


def cpu_baseline_for(workload, T, threads, sample_coords=0, timed=2):
    """cpu_baseline object of one workload: best rate over the workload's sample sizes (torch's intra-op threading of
    [N,80]-shaped tensors depends on N, so the sample size that suits the host is chosen by measurement)."""
    best = None
    sizes = (sample_coords,) if sample_coords else CPU_SAMPLES[workload]
    for n_s in sizes:
        one, n, what = cpu_oracle_unroll(workload, T, n_s, threads)
        one(min(T, 5))                       # warm-up (allocator, thread pool) on a short unroll
        ts = [one() for _ in range(timed)]
        rate = n * T * len(ts) / sum(ts)
        if best is None or rate > best["value"]:
            best = {"value": rate, "unit": "coordinate-updates/s", "cores": threads, "kind": "port",
                    "sample": "%d coordinates x T=%d train unroll (fwd + autograd BPTT + TF-Adam) of %s; torch-CPU oracle, "
                              "%d timed unroll(s) after a short warm-up%s" % (
                                  n, T, what, len(ts), "" if len(sizes) == 1 else "; best of samples %s" % (list(sizes),)),
                    "sample_coords": n}
    return best


def run_reference(args):
    """--impl reference: the reference's algorithm on the host cores (TF-1.14/Sonnet cannot be installed here,
    DESIGN.md; the oracle port stands in, kind="port").  The line's `config` is what this arm actually ran: a bounded
    SAMPLE of the workload (`cpu_sample: true`, `coords_per_gpu` = the sample's coordinates)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    desc, dcoords, dT, _ = WORKLOADS[args.workload]
    T = args.unroll or dT
    threads = pick_cpu_threads()
    sizes = (args.cpu_sample_coords,) if args.cpu_sample_coords else CPU_SAMPLES[args.workload]
    best = None
    for n_s in sizes:                        # probe: one short + one full unroll per candidate sample size
        one, n, what = cpu_oracle_unroll(args.workload, T, n_s, threads)
        one(min(T, 5))
        rate = n * T / one()
        if best is None or rate > best[0]:
            best = (rate, one, n, what)
    _, one, n, what = best
    for _ in range(args.warmup):
        one()
    times = [one() for _ in range(args.steps)]
    tot = sum(times)
    value = n * T * args.steps / tot
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "coordinate-updates/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot / args.steps, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": desc, "coords_per_gpu": n, "cpu_sample": True,
                   "gpu_arm_coords": args.coords or dcoords, "unroll": T, "mode": "train (fwd+BPTT+Adam)",
                   "net_scale": NET_SCALE[args.workload], "sample_sizes_probed": list(sizes)},
        "cpu_baseline": {"value": value, "unit": "coordinate-updates/s", "cores": threads, "kind": "port",
                         "sample": "%d coordinates x T=%d train unroll per step of %s (torch-CPU oracle, autograd BPTT); "
                                   "a bounded sample of the GPU arm's workload, not its full size" % (n, T, what)},
        "e2e": {"value": value, "unit": "coordinate-updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)
    if args.workload == "hrnn_convnet":   # side workload: its own line (N=1 only)
        torch.cuda.set_device(0)
        print(json.dumps(quick_measure_hrnn(steps=args.steps, warmup=args.warmup)))
        return

    import torch.distributed as dist
    from open_l2o_b200 import engine as eng, meta

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    distributed = world > 1
    if distributed:
        # NCCL prints its version banner on stdout when the communicator is created; keep stdout = the one JSON line
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.all_reduce(torch.zeros(1, device=dev))
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    desc, dcoords, dT, netkind = WORKLOADS[args.workload]
    coords = args.coords or dcoords
    T = args.unroll or dT
    strong = args.scaling == "strong"
    if strong:
        # BASELINE config #5 as written: ONE 1M-coordinate problem, coordinates sharded over the ranks (SURVEY.md 8(e))
        if args.workload != "rastrigin":
            raise SystemExit("--scaling strong is defined for the coordinate-sharded rastrigin workload")
        from open_l2o_b200.dist import shard_range
        total_coords = coords
        problem, net_config, flavour = make_problem(args.workload, total_coords, rank,
                                                    shard=shard_range(total_coords, rank, world))
        seed = 0           # every rank draws the same global tensors and keeps its slice
    else:
        problem, net_config, flavour = make_problem(args.workload, coords, rank)
        seed = rank
    cls = meta.RNNpropMetaOptimizer if flavour == "rnnprop" else meta.MetaOptimizer
    optimizer = cls(_seed=seed, _distributed=distributed, **net_config)
    _stdout = sys.stdout
    sys.stdout = open(os.devnull, "w")      # the reference prints variable lists at graph build; keep stdout = 1 JSON line
    try:
        ms = optimizer.meta_minimize(problem, T, learning_rate=0.001)
    finally:
        sys.stdout = _stdout
    prog = optimizer.program
    coords = prog.N
    if args.engine != "auto":
        for net in prog.nets.values():
            net.handle.set_engine({"ffma": eng.ENGINE_FFMA, "tc": eng.ENGINE_TC}[args.engine])
    sess = meta.Session()
    sess.run(ms.reset)
    fetch = [ms.fx, ms.update, ms.step]

    def barrier():
        if distributed:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput ("value") -----------------------------------------------------
    sampler = ClockSampler(local)
    sampler.start()
    for _ in range(args.warmup):
        sess.run(fetch)
    barrier()
    sampler.t_begin = time.perf_counter()
    l0 = eng.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        cost = sess.run(fetch)[0]
    e1.record()
    barrier()
    sampler.t_end = time.perf_counter()
    launches = eng.launch_count() - l0
    t_dev = e0.elapsed_time(e1) / 1e3
    sampler.stop()
    if args.dump_outputs and rank == 0:     # before the kernel timings and the e2e steps below overwrite them
        dump_outputs(args.dump_outputs, last_step_outputs(prog))
    tt = torch.tensor([t_dev], dtype=torch.float64, device=dev)
    if distributed:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    t_dev = float(tt.item())
    job_coords = total_coords if strong else coords * world      # coordinates the WHOLE job updates per step
    value = job_coords * T * args.steps / t_dev

    # ---- N>1 consistency: after the all-reduced meta-steps every rank must hold the identical theta ----------------
    theta_check = None
    if distributed:
        th = next(iter(prog.nets.values())).theta
        ck = torch.stack([th.double().sum(), th.double().abs().sum()])
        allck = [torch.zeros_like(ck) for _ in range(world)]
        dist.all_gather(allck, ck)
        theta_check = {"rank0_sum": float(allck[0][0]), "identical_on_all_ranks": bool(all(torch.equal(allck[0], c) for c in allck))}
        if not theta_check["identical_on_all_ranks"]:
            raise SystemExit("theta diverged across ranks: %r" % ([c.tolist() for c in allck],))

    # ---- per-kernel timing of the dominant kernel (BPTT) for the roofline ---------------------------
    kb0, kb1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kf0, kf1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    r = prog.runs[0]
    h = r.net.handle
    roof = None
    if prog.fused is not None and args.workload == "rastrigin":
        fw, bw = [], []
        for _ in range(max(2, min(args.steps, 3))):
            prog.fx_buf.zero_()
            xw = prog.X.clone()
            st = r.state.clone()
            kf0.record()
            h.unroll_fwd(r.net.theta, r.n, T, st, opt_kind=eng.OPT_KINDS[prog.fused.kind],
                         opt_a=prog.const_vals[prog.fused.a], opt_b=prog.const_vals[prog.fused.b],
                         opt_alpha=prog.fused.alpha, opt_fscale=prog.fused.fscale, x=xw, ckpt=r.ckpt, g_rec=r.g_rec,
                         fx=prog.fx_buf)
            kf1.record()
            dth = torch.zeros_like(prog.dtheta[r.key])
            kb0.record()
            h.unroll_bwd(r.net.theta, r.n, T, r.g_rec, r.ckpt, dth, g_rec=r.g_rec)
            kb1.record()
            torch.cuda.synchronize()
            fw.append(kf0.elapsed_time(kf1) / 1e3)
            bw.append(kb0.elapsed_time(kb1) / 1e3)
        t_f, t_b = sum(fw) / len(fw), sum(bw) / len(bw)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("bf16_tflops", 1700.0))   # burst figure: the kernels are timed alone (launch, sync)
        fl = FLOP_PER_UPDATE_INFER[netkind]
        ach_b = 2.0 * fl * r.n * T / t_b / 1e12          # backward = two more GEMMs of the forward's shape
        ach_f = fl * r.n * T / t_f / 1e12
        traffic, traffic_src = None, None
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            traffic = tj["unroll_bwd_dram_bytes_per_coord_update"] * r.n * T
            traffic_src = tj.get("source")
        except Exception:
            pass
        alg_bytes = (C_SF_BYTES + 8) * r.n * T      # checkpoint row + g_rec + in_seq per coordinate-update (read)
        roof = {"bound": "tensor", "kernel": "tcb2::unroll_bwd2_kernel (layer-pipelined tcgen05 BPTT)", "achieved": ach_b, "peak": peak,
                "unit": "TFLOP/s", "frac": ach_b / peak, "traffic": traffic, "traffic_source": traffic_src,
                "algorithmic_bytes": alg_bytes,
                "peak_source": "MEASURED_PEAKS.json bf16_tflops (burst: kernel timed alone)" if peaks else "fallback 1.7 PF (B200_PROFILING.md)",
                "fwd_kernel": {"name": "tc::unroll_fwd_kernel (tcgen05)", "achieved": ach_f, "frac": ach_f / peak,
                               "ms": 1e3 * t_f, "coord_updates_per_s": r.n * T / t_f},
                "bwd_ms": 1e3 * t_b, "bwd_coord_updates_per_s": r.n * T / t_b,
                "alg_flop_per_coord_update": {"fwd": fl, "bwd": 2 * fl},
                "algorithmic_bytes_8d_fused": 8.0 * r.n * T,
                "traffic_over_8d_fused": (traffic / (8.0 * r.n * T)) if traffic else None,
                "traffic_note": "SURVEY.md 8(d) puts the fused regime at 4-8 B per coordinate-update (inference: g in, "
                                "x out).  TRAINING by recompute must also write (forward) and read (BPTT) the "
                                "checkpoint row: 320 B + g 4 B + net input 4 B = 328 B per coordinate-update per "
                                "direction = `algorithmic_bytes`; the measured DRAM traffic is ~41x the 8 B figure and "
                                "1.01x the checkpoint figure",
                "notes": "fp32 parity => 3xTF32 for the gate recompute and dX (tf32 = 1/2 the bf16 rate: a 100%-busy tensor "
                         "pipe reads 1/6 of this peak) and bf16 hi/lo for dW^T; ncu r02e: tensor pipe 28%, issue slots "
                         "36%, XU 28%, warps active 31% in the BPTT kernel (profiles/r02_ncu_summary.json); the kernel is "
                         "bound by instruction issue inside the two overlapping layer phases (130 warp-instructions per "
                         "coordinate-update, 30% of them operand splitting) and by the serial MMA round trips of each chain; "
                         "the activation pipe (320 MUFU ops per coordinate-update forward, 400 backward) caps the path "
                         "near 1.4e10 upd/s/GPU"}

    if roof is None:      # external-gradient workloads: HBM roofline of the step kernel (+ BPTT) on this workload
        roof = external_roofline(prog, netkind, T, t_dev / args.steps)

    # ---- infer mode (evaluate_dm.py: forward unroll only, no checkpoints) -----------------------------
    infer = None
    if prog.fused is not None and args.workload == "rastrigin":
        ts = []
        for _ in range(max(2, min(args.steps, 3))):
            xw = prog.X.clone()
            st = r.state.clone()
            kf0.record()
            h.unroll_fwd(r.net.theta, r.n, T, st, opt_kind=eng.OPT_KINDS[prog.fused.kind],
                         opt_a=prog.const_vals[prog.fused.a], opt_b=prog.const_vals[prog.fused.b],
                         opt_alpha=prog.fused.alpha, opt_fscale=prog.fused.fscale, x=xw, fx=prog.fx_buf)
            kf1.record()
            torch.cuda.synchronize()
            ts.append(kf0.elapsed_time(kf1) / 1e3)
        t_i = sum(ts) / len(ts)
        ti = torch.tensor([t_i], dtype=torch.float64, device=dev)
        if distributed:
            dist.all_reduce(ti, op=dist.ReduceOp.MAX)
        infer = {"value": job_coords * T / float(ti.item()), "unit": "coordinate-updates/s", "ms_per_unroll": 1e3 * t_i,
                 "mode": "infer (forward unroll only, state on-chip, no checkpoint writes; l2o_unroll_fwd)"}

    # ---- end-to-end through the public API with HOST buffers ------------------------------------
    # every step: the optimizee's parameters AND problem constants come from pinned host memory (H2D inside the timed
    # region, written in place so captured graphs stay valid), one meta-step through Session.run, the loss is read
    # back by float(fx) and the updated parameters are copied to the host
    hx = prog.X.cpu().pin_memory()
    hconst = {k: v.cpu().pin_memory() for k, v in prog.const_vals.items()}
    hout = torch.empty(coords, dtype=torch.float32).pin_memory()
    fetch2 = [ms.fx, ms.update, ms.step]
    barrier()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record()
    for _ in range(args.steps):
        prog.X.copy_(hx, non_blocking=True)
        for k, hv in hconst.items():
            prog.const_vals[k].copy_(hv, non_blocking=True)
        cost = sess.run(fetch2)[0]                 # float(fx) = device->host read of the loss
        hout.copy_(prog.X, non_blocking=True)      # updated parameters back to the host
    g1.record()
    barrier()
    t_e = torch.tensor([g0.elapsed_time(g1) / 1e3], dtype=torch.float64, device=dev)
    if distributed:
        dist.all_reduce(t_e, op=dist.ReduceOp.MAX)
    e2e = {"value": job_coords * T * args.steps / float(t_e.item()), "unit": "coordinate-updates/s",
           "h2d_bytes_per_step": 4 * (hx.numel() + sum(v.numel() for v in hconst.values())),
           "d2h_bytes_per_step": 4 * coords + 8, "bytes_are": "per rank"}

    # ---- CPU baseline (oracle port on the host cores; rank 0, N=1 only) ----------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline_for(args.workload, T, pick_cpu_threads(), args.cpu_sample_coords)

    also = None
    if rank == 0 and world == 1 and args.workload == "rastrigin" and not args.no_also:
        also = []
        for w in ("mlp", "lasso", "rnnprop_mlp", "quadratic"):
            try:
                also.append(quick_measure(w, steps=max(args.steps, 5), warmup=max(args.warmup, 3)))
            except Exception as ex:  # the headline line must survive a failure of a side measurement
                also.append({"workload": WORKLOADS[w][0], "error": repr(ex)[:200]})
        try:
            also.append(quick_measure_hrnn(steps=max(args.steps, 5), warmup=max(args.warmup, 3)))
        except Exception as ex:
            also.append({"workload": "L2O-Scale HierarchicalRNN (BASELINE config #4)", "error": repr(ex)[:200]})

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "coordinate-updates/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * t_dev / args.steps, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": desc if not strong else desc.replace("d=1e6 per GPU", "d=%d in total" % total_coords),
                       "coords_per_gpu": coords, "coords_total": job_coords, "unroll": T,
                       "mode": "train (fwd+BPTT+Adam)",
                       "regime": "fused" if prog.fused is not None else (
                           "external-gradient (producer %s)" % prog.producer.kind if prog.producer is not None
                           else "external-gradient (torch autograd)"),
                       "engine": args.engine, "parallelism": "dp%d (coordinates sharded)" % world,
                       "net_scale": NET_SCALE[args.workload], "theta_check": theta_check,
                       "l2_policy": "working set (checkpoints %.1f GB/GPU) >> 126 MB L2" % (r.ckpt.numel() * 4 / 1e9),
                       "last_fx": cost},
            "clocks": sampler.summary(), "e2e": e2e, "gpu_launches": int(launches), "roofline": roof,
            "cpu_baseline": cpu, "infer": infer, "also": also,
        }
        print(json.dumps(line))
    if distributed:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
