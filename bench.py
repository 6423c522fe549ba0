#!/usr/bin/env python
"""bench.py — benchmark of the hot path (contract in the task statement / DESIGN.md section 7).

Headline workload (BASELINE.json configs[2], the config the metric is quoted on, ``--config 3``, the default):
lid-driven-cavity Navier-Stokes Re=100 (nu=0.01, rho=1), MLP (x,y)->256x6->(u,v,p) tanh, 2^20 collocation points per
GPU per step, fp32, synthetic points U[0,1]^2, labels 0, MSELoss("mean"), Xavier-uniform weights.
``--config 1|2|4|5`` run the other BASELINE configurations at their named shapes (SURVEY.md section 8(d)).

A "step" = one pass of the hot path over one batch: forward jets + residual + MSE + adjoint -> flat weight gradient
(+ one NCCL all-reduce of that buffer when N>1) + fused Adam.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 1..5] [--dump-outputs DIR]

``--dump-outputs DIR`` writes what the last timed step handed back to its caller, as ``DIR/<name>.npy`` in the
workload's dtype: ``loss_<residual>`` (the per-residual losses it returned) and ``params`` / ``adam_exp_avg`` /
``adam_exp_avg_sq`` (the weights and Adam moments it updated in place; the gradient itself is consumed by Adam and
cleared).  Inputs and initial weights are seeded, so two builds run with the same arguments can be compared file by file.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time
from typing import Optional

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

UNIT = "points/s"
NU, RHO = 0.01, 1.0
# dram__bytes_read.sum + dram__bytes_write.sum of the hidden-layer kernels of cfg3 from the committed `ncu --set full`
# captures of this round (profiles/r02_summary.md; one 65,536-point chunk, all five hidden->hidden layers): bytes PER POINT.
# Equal to the plane sets the design streams (no re-reads): fwd 1 read + 10 written sets, dx 6 read + 5 written, dW 10 read.
NCU_DRAM_BYTES_PER_POINT_CFG3 = {"fwd_gemm": (364.1e6 + 3294.9e6) / 65536, "dx_gemm": (2060.0e6 + 1635.9e6) / 65536,
                                 "dw_gemm": 5 * (671.5e6 + 4.3e6) / 65536}  # profiles/r02c_ncu_*_details.txt (final build)

# name, metric label, points per GPU, dtype
CONFIGS = {
    1: dict(metric="collocation-points/sec PDE residual loss+grad (Laplace2D)", n=10201, dtype="f32",
            workload="BASELINE configs[0]: Laplace2D, MLP (x,y)->20x4->u tanh, 10,201 evenly spaced interior points "
                     "(101 x 101 grid, the reference's evenly=True set), MSELoss(sum), Adam"),
    2: dict(metric="collocation-points/sec PDE residual loss+grad (Allen-Cahn)", n=1 << 18, dtype="f32",
            workload="BASELINE configs[1]: Allen-Cahn eps=0.01, MLP (t,x)->128x4->u tanh, periodic in x (period 2), "
                     "2^18 collocation points per GPU per step, MSELoss(mean), Adam"),
    3: dict(metric="collocation-points/sec PDE residual loss+grad (LDC N-S)", n=1 << 20, dtype="f32",
            workload="BASELINE configs[2]: LDC Navier-Stokes Re=100 (nu=0.01, rho=1), MLP (x,y)->256x6->(u,v,p) tanh, "
                     "2^20 collocation points per GPU per step, 3 residuals, MSELoss(mean), Adam"),
    4: dict(metric="collocation-points/sec PDE residual loss+grad (Biharmonic2D, fp64)", n=1 << 18, dtype="f64",
            workload="BASELINE configs[3]: Biharmonic2D (4th-order jets, C=17), MLP (x,y)->128x5->u tanh, fp64, "
                     "2^18 collocation points per GPU per step, MSELoss(mean), Adam"),
    5: dict(metric="(u,y) pairs/sec DeepONet loss+grad (antiderivative)", n=1 << 20, dtype="f32",
            workload="BASELINE configs[4]: DeepONet, branch MLP 100->128x3->128, trunk MLP 1->128x3->128 (+ trunk act), "
                     "2^20 (u,y) pairs per GPU per step, MSELoss(mean), Adam"),
}

_T0 = time.perf_counter()


def log(msg: str):
    """Progress to stderr (never to stdout: stdout carries the JSON line; never into the source tree, which may be
    read-only)."""
    print(f"[bench +{time.perf_counter() - _T0:7.1f}s] {msg}", file=sys.stderr, flush=True)


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir: str, arrays) -> None:
    """Write ``{name: tensor}`` as ``out_dir/<name>.npy`` (float32 / float64, as computed) for output-by-output
    comparison of two builds."""
    import numpy as np

    host = {k: v.detach().cpu().numpy() for k, v in arrays.items()}
    for k, a in host.items():
        if a.dtype not in (np.float32, np.float64):
            raise TypeError(f"--dump-outputs: {k} is {a.dtype}, expected float32 or float64")
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_LIMIT_BYTES:
        raise ValueError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for k, a in host.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), a)


def flops_per_point(C: int, widths_list) -> float:
    """SURVEY.md section 8(d): F_total = 3*C*F_v, F_v = 2*sum(in*out) (summed over the sub-networks)."""
    fv = sum(2.0 * sum(a * b for a, b in zip(w[:-1], w[1:])) for w in widths_list)
    return 3.0 * C * fv


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu_index = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.gpu_index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.strip().split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = sorted(int(float(r[1])) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit())
        mx = [int(float(r[2])) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 9 for n, v in zip(names, r[5:9]) if v.lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"bf16_tflops_sustained": p.get("bf16_tflops_sustained"), "bf16_tflops": p.get("bf16_tflops"),
                "hbm_gbs": p.get("hbm_gbs"), "source": "MEASURED_PEAKS.json"}
    return {"bf16_tflops_sustained": 1400.0, "bf16_tflops": 1590.0, "hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md)"}


def measure_tf32_peak(dev):
    """Dense tf32 tensor-core throughput measured in THIS run (the peaks file has no tf32 figure): cuBLAS fp32 GEMM
    with TF32 allowed, 8192^3, best of 8 after 2 warm-ups, CUDA events.  Library call used as a yardstick only."""
    import torch

    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        n = 8192
        a = torch.randn(n, n, device=dev)
        b = torch.randn(n, n, device=dev)
        c = torch.empty(n, n, device=dev)
        best = float("inf")
        for i in range(10):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch.matmul(a, b, out=c)
            e1.record()
            torch.cuda.synchronize(dev)
            if i >= 2:
                best = min(best, e0.elapsed_time(e1))
        return 2.0 * n ** 3 / (best * 1e-3) / 1e12
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old


# --------------------------------------------------------------------------------------------------
# workloads
# --------------------------------------------------------------------------------------------------
def oracle_problem(cfg: int):
    """(OracleMLP or DeepONet oracle, exprs, input sampler) of the reference-algorithm restatement for config `cfg`."""
    import sympy as sp
    import torch

    from oracle import ppsci_oracle as O

    if cfg == 1:
        return O.OracleMLP(("x", "y"), ("u",), [20] * 4, "tanh"), O.laplace_expr(2), "sum", {"x": (0, 1), "y": (0, 1)}
    if cfg == 2:
        om = O.OracleMLP(("t", "x"), ("u",), [128] * 4, "tanh", {"x": (2.0, False)})
        return om, O.allen_cahn_callable(0.01), "mean", {"t": (0, 1), "x": (-1, 1)}
    if cfg == 3:
        return (O.OracleMLP(("x", "y"), ("u", "v", "p"), [256] * 6, "tanh"), O.navier_stokes_expr(NU, RHO, 2, False), "mean",
                {"x": (0, 1), "y": (0, 1)})
    if cfg == 4:
        xs, ys = sp.symbols("x y")
        q = 2.0 * sp.sin(sp.pi * xs / 2) * sp.sin(sp.pi * ys / 3)
        return O.OracleMLP(("x", "y"), ("u",), [128] * 5, "tanh"), O.biharmonic_expr(2, q, 1.5), "mean", {"x": (0, 2), "y": (0, 3)}
    raise ValueError(cfg)


def cpu_reference_leg(cfg: int, n_sample: int, iters: int, warmup: int, budget_s: Optional[float] = 25.0):
    """Time the reference's algorithm (oracle = torch CPU restatement: Paddle is not installable, DESIGN.md
    section 6) on the host cores for the same workload at a bounded number of points.  ``budget_s=None`` runs exactly
    ``iters`` timed iterations."""
    import torch

    from oracle import ppsci_oracle as O

    cores = min(os.cpu_count() or 1, 64)  # all host threads torch's intra-op pool can use productively
    torch.set_num_threads(cores)
    dt = torch.float64 if CONFIGS[cfg]["dtype"] == "f64" else torch.float32
    g = torch.Generator().manual_seed(42)
    if cfg == 5:
        don = O.OracleDeepONet(100, 128, [128] * 3, [128] * 3, "tanh", "tanh", True)
        pb = O.xavier_uniform_params(don.bw, 1, dt)
        pt = O.xavier_uniform_params(don.tw, 2, dt)
        u = torch.randn(n_sample, 100, generator=g, dtype=dt)
        y = torch.rand(n_sample, 1, generator=g, dtype=dt)
        lab = torch.randn(n_sample, 1, generator=g, dtype=dt)

        def once():
            a, b, c = pb.clone().requires_grad_(True), pt.clone().requires_grad_(True), torch.zeros(1, dtype=dt, requires_grad=True)
            loss = ((don(a, b, c, u, y) - lab) ** 2).mean()
            loss.backward()
    else:
        om, exprs, red, ranges = oracle_problem(cfg)
        params = O.xavier_uniform_params(om.widths, 1, dt)
        names = list(exprs.keys())
        x = {k: (torch.rand(n_sample, 1, generator=g, dtype=dt) * (hi - lo) + lo) for k, (lo, hi) in ranges.items()}
        labels = {k: torch.zeros(n_sample, 1, dtype=dt) for k in names}

        def once():
            O.train_forward_backward(om, params, exprs, x, labels, None, red, None)
    for _ in range(warmup):
        once()
    times = []
    t_begin = time.perf_counter()
    for _ in range(iters):
        t0 = time.perf_counter()
        once()
        times.append(time.perf_counter() - t0)
        if budget_s is not None and time.perf_counter() - t_begin > budget_s and len(times) >= 2:
            break
    iters = len(times)
    sec = sum(times) / len(times)
    return {"value": n_sample / sec, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{iters} timed iterations (after {warmup} warm-up) of forward residuals + MSE + backward to the "
                      f"weights on {n_sample} of the {CONFIGS[cfg]['n']} points per step, torch CPU autograd restatement of "
                      f"the reference (Paddle not installable), {cores} threads",
            "ms_per_sample_step": sec * 1e3}


CPU_SAMPLE = {1: 10201, 2: 1 << 15, 3: 1 << 14, 4: 2048, 5: 1 << 16}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = args.config
    n_sample = CPU_SAMPLE[cfg]
    cb = cpu_reference_leg(cfg, n_sample, args.steps, max(1, min(args.warmup, 2)), budget_s=None)
    line = {
        "impl": "reference", "metric": CONFIGS[cfg]["metric"], "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": cb["ms_per_sample_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": CONFIGS[cfg]["dtype"], "data": "synthetic",
        "config": {"workload": CONFIGS[cfg]["workload"] + f"; each step a bounded sample of {n_sample} points (CPU)",
                   "points_per_step": n_sample},
        "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def build_workload(cfg: int, dev, rank: int):
    """Model, constraint-like object, pinned host inputs / labels of config `cfg` through the public API."""
    import numpy as np
    import sympy as sp
    import torch

    import ppsci

    n = CONFIGS[cfg]["n"]
    dt = torch.float64 if CONFIGS[cfg]["dtype"] == "f64" else torch.float32
    ppsci.utils.misc.set_random_seed(42)
    g = torch.Generator().manual_seed(1234 + rank)
    red = "mean"
    labels_host = None
    if cfg == 1:
        model = ppsci.arch.MLP(("x", "y"), ("u",), 4, 20, "tanh")
        equation = ppsci.equation.Laplace(2)
        from oracle import ppsci_oracle as O  # grid construction only (the reference's evenly=True point set)

        pts = O.hypercube_uniform_points((0.0, 0.0), (1.0, 1.0), n, boundary=True)
        host = {"x": torch.as_tensor(pts[:, 0:1], dtype=dt), "y": torch.as_tensor(pts[:, 1:2], dtype=dt)}
        red = "sum"
    elif cfg == 2:
        model = ppsci.arch.MLP(("t", "x"), ("u",), 4, 128, "tanh", periods={"x": (2.0, False)})
        equation = ppsci.equation.AllenCahn(0.01)
        host = {"t": torch.rand(n, 1, generator=g), "x": torch.rand(n, 1, generator=g) * 2 - 1}
    elif cfg == 3:
        model = ppsci.arch.MLP(("x", "y"), ("u", "v", "p"), 6, 256, "tanh")
        equation = ppsci.equation.NavierStokes(NU, RHO, 2, False)
        host = {"x": torch.rand(n, 1, generator=g), "y": torch.rand(n, 1, generator=g)}
    elif cfg == 4:
        model = ppsci.arch.MLP(("x", "y"), ("u",), 5, 128, "tanh", dtype=torch.float64)
        xs, ys = sp.symbols("x y")
        equation = ppsci.equation.Biharmonic(2, 2.0 * sp.sin(sp.pi * xs / 2) * sp.sin(sp.pi * ys / 3), 1.5)
        host = {"x": torch.rand(n, 1, generator=g, dtype=dt) * 2, "y": torch.rand(n, 1, generator=g, dtype=dt) * 3}
    else:
        model = ppsci.arch.DeepONet("u", "y", "G", 100, 128, 3, 3, 128, 128, branch_activation="tanh", trunk_activation="tanh")
        equation = None
        host = {"u": torch.randn(n, 100, generator=g), "y": torch.rand(n, 1, generator=g)}
        labels_host = {"G": torch.randn(n, 1, generator=g)}
    model = model.to(dev)

    class _Cst:  # a constraint as ExpressionSolver sees it: expressions + loss + names
        name = "EQ"
        loss = ppsci.loss.MSELoss(red)

    cst = _Cst()
    if equation is not None:
        cst.output_expr = dict(equation.equations)
        cst.output_keys = tuple(equation.equations.keys())
    else:
        cst.output_expr = {"G": lambda out: out["G"]}
        cst.output_keys = ("G",)
    host = {k: v.to(dt).pin_memory() for k, v in host.items()}
    if labels_host is None:
        labels_host = {k: torch.zeros(n, 1, dtype=dt) for k in cst.output_keys}
    return model, cst, host, labels_host, dt


# --------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the engine has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    import ppsci

    cfg = args.config
    N = CONFIGS[cfg]["n"]
    model, cst, host, labels_host, dt = build_workload(cfg, dev, rank)
    if world > 1:  # same initial weights on every rank (DataParallel broadcast semantics)
        dist.broadcast(model.flat.data, 0)
    constraint = {"EQ": cst}
    helper = ppsci.utils.ExpressionSolver()
    opt = ppsci.optimizer.Adam(1e-3)(model)
    labels = {k: v.to(dev) for k, v in labels_host.items()}
    model.flat.grad = torch.zeros_like(model.flat.data)
    is_don = cfg == 5
    if is_don:
        plan, C = None, 1
        widths_list = [model._branch.widths, model._trunk.widths]
    else:
        cc = helper.compiled_for(model, cst, None)
        plan = cc.plan(dt)
        C = plan.channels
        widths_list = [model.net_spec().widths]
    fpp = flops_per_point(C, widths_list)
    params_init = model.engine_params().detach().clone() if plan is not None else None  # parity is checked on these too
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def make_step(lab, comm=True):
        def step(inp):
            losses_all, _ = helper.train_forward((cst.output_expr,), (inp,), model, constraint, (lab,), (None,))
            if world > 1:
                if comm:
                    dist.all_reduce(model.flat.grad)
                opt.grad_scale = 1.0 / world
            opt.step()
            opt.clear_grad()
            return losses_all
        return step

    step = make_step(labels)

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, inp, steps):
        """K steps bracketed by barrier + synchronize, CUDA events per step, L2 flushed (untimed) between steps;
        returns max-over-ranks ms per step."""
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        sync_all()
        out = None
        for a, b in evs:
            flush.fill_(1)
            a.record()
            out = fn(inp)
            b.record()
        sync_all()
        ms_total = torch.tensor([sum(a.elapsed_time(b) for a, b in evs)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms_total, op=dist.ReduceOp.MAX)
        return float(ms_total) / steps, out

    log(f"setup done: config {cfg}, C={C}, tcgen05={plan.uses_tcgen05 if plan else 'n/a'}")
    # ---------------- device-resident timing ("value") ----------------
    dev_in = {k: v.to(dev) for k, v in host.items()}
    for _ in range(args.warmup):
        step(dev_in)
    sync_all()
    log("warm-up done")
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    don_launches0 = sum(p.two_phase_launches for p in model._get_plans()) if plan is None else 0
    t_wall0 = time.perf_counter()
    ms_per_step, losses = timed(step, dev_in, args.steps)
    t_wall = time.perf_counter() - t_wall0
    if plan is not None:
        launches_per_step = plan.last_launches + 1  # + fused Adam
    else:  # DeepONet: every two-phase call of both sub-network plans over the timed steps, + head kernels + fused Adam
        tp = sum(p.two_phase_launches for p in model._get_plans()) - don_launches0
        n_slices = (N + min(p.chunk_points for p in model._get_plans()) - 1) // min(p.chunk_points for p in model._get_plans())
        launches_per_step = tp // args.steps + n_slices + 1
    value = world * N / (ms_per_step * 1e-3)
    log(f"timed region done: {ms_per_step:.2f} ms/step")
    if args.dump_outputs and rank == 0:  # before the passes below train the weights further
        dump_outputs(args.dump_outputs, {**{f"loss_{k}": v for k, v in losses.items()}, "params": model.flat.data,
                                         "adam_exp_avg": opt.exp_avg, "adam_exp_avg_sq": opt.exp_avg_sq})
        log(f"outputs of the last timed step written to {args.dump_outputs}")

    # ---------------- end to end through the public API with host buffers ("e2e") ----------------
    def host_step():
        inp = {k: v.to(dev, non_blocking=True) for k, v in host.items()}
        l_all = step(inp)
        return torch.stack([l_all[k] for k in cst.output_keys]).cpu()  # D2H read of the step's result

    for _ in range(2):
        host_step()
    sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    d2h = 0
    e0.record()
    for _ in range(args.steps):
        hl = host_step()
        d2h = hl.numel() * hl.element_size()
    e1.record()
    sync_all()
    ms_e2e = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms_e2e, op=dist.ReduceOp.MAX)
    e2e_value = world * N / (float(ms_e2e) / args.steps * 1e-3)
    clocks = sampler.stop() if rank == 0 else None
    log(f"e2e done: {float(ms_e2e) / args.steps:.2f} ms/step")

    # ---------------- parity of THIS run's residuals against the fp64 oracle on a fixed subset (untimed) ----------------
    def parity_check(tag, params, scale=None):
        """Residuals of the engine against the fp64 oracle on 4,096 strided points of the benchmark batch with weights
        ``params``.  ``scale``: per-residual norms to normalise with instead of the oracle residual's own norm — training
        drives the residual itself towards zero (that is its purpose), so on trained weights the plain relative error
        grows although the absolute error does not; the error is then stated relative to the residual norm at the
        initial weights (and the plain ratio is reported beside it)."""
        if plan is None or rank != 0:
            return None
        from oracle import ppsci_oracle as O

        sub = torch.arange(0, N, max(1, N // 4096))[:4096]
        om, exprs, red, _ = oracle_problem(cfg)
        _, res_e = plan.forward({k: v[sub.to(dev)].contiguous() for k, v in dev_in.items()}, params)
        lo_, ro, _ = O.train_forward_backward(om, params.detach().cpu().double(), exprs,
                                              {k: v[sub].double() for k, v in host.items()},
                                              {k: torch.zeros(len(sub), 1, dtype=torch.float64) for k in cst.output_keys},
                                              None, red, None, want_grad=False)
        diff = {k: float((res_e[k].cpu().double() - ro[k]).norm()) for k in cst.output_keys}
        norms = {k: float(ro[k].norm()) for k in cst.output_keys}
        plain = {k: diff[k] / max(norms[k], 1e-300) for k in cst.output_keys}
        errs = plain if scale is None else {k: diff[k] / max(scale[k], norms[k], 1e-300) for k in cst.output_keys}
        tol = 1e-5 if dt == torch.float32 else 1e-11
        rec = {"residual_rel_l2": max(errs.values()), "per_residual": errs, "points": int(len(sub)), "tol": tol,
               "ok": max(errs.values()) <= tol, "weights": tag,
               "abs_rms_error": {k: diff[k] / len(sub) ** 0.5 for k in cst.output_keys},
               "oracle_residual_rms": {k: norms[k] / len(sub) ** 0.5 for k in cst.output_keys},
               "against": "fp64 oracle (torch restatement of the reference), 4,096 strided points of the benchmark batch, "
                          "outside the timed region"}
        if scale is not None:
            rec["plain_rel_l2"] = plain
            rec["normalised_by"] = "max(residual norm at these weights, residual norm at the initial weights)"
        log(f"parity check ({tag}): {rec['residual_rel_l2']:.3e}")
        return rec, norms

    parity, parity_trained, init_norms = None, None, None
    if plan is not None and rank == 0:
        parity, init_norms = parity_check("initial weights of this run (Xavier uniform, seed fixed): the weights of step 1", params_init)
        parity_trained, _ = parity_check("after the timed region and the end-to-end pass", model.engine_params(), init_norms)

    # ---------------- the same step replayed as ONE CUDA graph (Solver(to_static=True)), single process ----------------
    graph_rec = None
    if world == 1 and not is_don and args.graph != "off":
        import types

        from paddlescience_b200.solver.graph_step import GraphedTrainStep

        gs = GraphedTrainStep(types.SimpleNamespace(model=model, constraint=constraint, forward_helper=helper,
                                                    loss_aggregator=ppsci.loss.mtl.Sum(), optimizer=opt, world_size=1,
                                                    update_freq=1, global_step=0))

        def gstep(inp):
            return gs((inp,), (labels,), (None,))[0]

        for _ in range(GraphedTrainStep.WARMUP + 3):  # eager iterations, the capture, replays
            gstep(dev_in)
        ms_g, _ = timed(gstep, dev_in, args.steps)
        gs.always_copy = True  # the end-to-end figure pays the H2D copy of every input on every step
        for _ in range(2):
            gstep(host).cpu()
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            gstep(host).cpu()  # pinned host inputs -> the graph's static buffers, D2H read of the total loss
        e1.record()
        sync_all()
        graph_rec = {"ms_per_step": ms_g, "value": N / (ms_g * 1e-3), "unit": UNIT,
                     "e2e_value": N / (e0.elapsed_time(e1) / args.steps * 1e-3), "replays": gs.replays,
                     "note": "the identical step (same kernels, same inputs) captured once and replayed with one graph launch; "
                             "lr / Adam bias corrections read from device memory (ppsci_b200_adam_step_dev)"}
        log(f"cuda-graph pass done: {ms_g:.3f} ms/step")

    # ---------------- strong scaling: the SAME global batch (N points) split over the ranks ----------------
    strong = None
    if world > 1:
        ns = N // world
        s_in = {k: v[:ns].contiguous() for k, v in dev_in.items()}
        s_step = make_step({k: v[:ns].contiguous() for k, v in labels.items()})
        for _ in range(3):
            s_step(s_in)
        ms_s, _ = timed(s_step, s_in, args.steps)
        # where the strong-scaling step goes: the same step without the all-reduce (weights then differ per rank: done
        # last, on a throw-away copy of the step), and the all-reduce of the flat gradient alone
        nocomm_step = make_step({k: v[:ns].contiguous() for k, v in labels.items()}, comm=False)
        ms_nc, _ = timed(nocomm_step, s_in, args.steps)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        for _ in range(3):
            dist.all_reduce(model.flat.grad)
        sync_all()
        ev[0].record()
        for _ in range(20):
            dist.all_reduce(model.flat.grad)
        ev[1].record()
        sync_all()
        ar_ms = torch.tensor([ev[0].elapsed_time(ev[1]) / 20], device=dev, dtype=torch.float64)
        dist.all_reduce(ar_ms, op=dist.ReduceOp.MAX)
        dist.broadcast(model.flat.data, 0)  # the no-comm steps let the ranks drift apart: re-synchronise the weights
        model.flat.grad.zero_()
        strong = {"global_points": ns * world, "points_per_gpu": ns, "ms_per_step": ms_s, "value": ns * world / (ms_s * 1e-3),
                  "unit": UNIT, "ms_per_step_without_allreduce": ms_nc, "allreduce_ms_back_to_back": float(ar_ms),
                  "allreduce_bytes": int(model.flat.grad.numel() * model.flat.grad.element_size()),
                  "note": "strong scaling: the N=1 global batch split over the ranks, same step, same timing rules; "
                          "ms_per_step_without_allreduce = the identical step with the NCCL all-reduce left out, "
                          "allreduce_ms_back_to_back = 20 all-reduces of the flat gradient timed alone (max over ranks)"}
        log(f"strong-scaling pass done: {ms_s:.2f} ms/step")

    # ---------------- per-kernel-class shares (separate, untimed pass) ----------------
    prof = None
    don_prof = None
    if plan is not None:
        plan.set_profile(True)
        prof_acc = None
        for _ in range(2):
            step(dev_in)
            torch.cuda.synchronize(dev)
            p = plan.get_profile()
            prof_acc = p if prof_acc is None else {k: {"ms": prof_acc[k]["ms"] + v["ms"], "launches": v["launches"]} for k, v in p.items()}
        plan.set_profile(False)
        prof = {k: {"ms": v["ms"] / 2, "launches": v["launches"]} for k, v in prof_acc.items()}
    else:  # DeepONet: the LAST native call of each sub-network's plan in the step (its adjoint over the last slice)
        plans = model._get_plans()
        for p_ in plans:
            p_.set_profile(True)
        step(dev_in)
        torch.cuda.synchronize(dev)
        don_prof = {name: {k: round(v["ms"], 3) for k, v in p_.get_profile().items()} for name, p_ in zip(("branch", "trunk"), plans)}
        for p_ in plans:
            p_.set_profile(False)

    parity_end = None
    if plan is not None and rank == 0 and (graph_rec or strong):
        parity_end, _ = parity_check("after every sub-record of this run (CUDA-graph replays / strong-scaling pass included)",
                                     model.engine_params(), init_norms)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = measured_peaks()
    roofline = None
    if prof is not None:
        # Dominant kernel class = the hidden-layer class (forward / dx / dW) with the largest device time.
        # SURVEY.md section 8(d): the bound is the TENSOR pipe; algorithmic FLOPs of a class = C * 2 * sum_{hidden->hidden}
        # in*out per point (elementwise work excluded).  `achieved` = algorithmic fp32 TFLOP/s of that class, `peak` = the
        # dense tf32 throughput measured in this run (cuBLAS, the MMA kind the kernels use; 3xTF32 issues 3 MMA FLOPs per
        # algorithmic FLOP, so the ceiling of `frac` is 1/3).
        w = widths_list[0]
        hh_flops_pt = C * 2.0 * sum(a * b for a, b in zip(w[1:-2], w[2:-1]))
        classes = {"fwd_gemm": hh_flops_pt, "dx_gemm": hh_flops_pt, "dw_gemm": hh_flops_pt}
        dom = max(classes, key=lambda k: prof[k]["ms"])
        dom_ms, dom_launches = prof[dom]["ms"], max(1, prof[dom]["launches"])
        on_tc = bool(plan.uses_tcgen05)
        tf32_peak = measure_tf32_peak(dev) if on_tc else None
        ach = classes[dom] * N / (dom_ms * 1e-3) / 1e12 if dom_ms > 0 else None
        # plane-set traffic of the class in this design (HBM figure beside the tensor figure)
        n_hh = max(1, len(w) - 3)
        H = w[1]
        esz = 8 if dt == torch.float64 else 4
        n_chunks = math.ceil(N / max(1, plan.chunk_points))
        fused = on_tc and 0 < prof["fwd_gemm"]["launches"] <= n_chunks  # one launch per point chunk instead of one per layer
        sets = {"fwd_gemm": (2 * n_hh + 1) if fused else 3 * n_hh, "dx_gemm": (2 * n_hh + 1) if fused else 3 * n_hh, "dw_gemm": 2 * n_hh}
        design_bytes = sets[dom] * C * N * H * esz
        if on_tc:
            roofline = {"bound": "tensor", "kernel": dom, "achieved": ach, "peak": tf32_peak, "unit": "TFLOP/s",
                        "frac": (ach / tf32_peak) if ach and tf32_peak else None,
                        "issued_mma_frac": (3 * ach / tf32_peak) if ach and tf32_peak else None}
        else:
            hbm = design_bytes / (dom_ms * 1e-3) / 1e9 if dom_ms > 0 else None
            roofline = {"bound": "hbm", "kernel": dom, "achieved": hbm, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                        "frac": hbm / peaks["hbm_gbs"] if hbm else None}
        roofline.update({
            "traffic": (NCU_DRAM_BYTES_PER_POINT_CFG3[dom] * N / dom_launches) if cfg == 3 else None,
            "class_ms_per_step": round(dom_ms, 3), "launches_per_step": dom_launches,
            "alg_flops_per_step": classes[dom] * N,
            "hbm_gbs_design_traffic": design_bytes / (dom_ms * 1e-3) / 1e9 if dom_ms > 0 else None,
            "hbm_peak_gbs": peaks["hbm_gbs"],
            "whole_step_tflops": fpp * N / (ms_per_step * 1e-3) / 1e12,
            "class_ms": {k: round(v["ms"], 3) for k, v in prof.items()},
            "backend": "tcgen05 (3xTF32, kind::tf32)" if on_tc else ("simt-fp64" if dt == torch.float64 else "simt-fp32"),
            "note": f"{dom}: algorithmic fp32 FLOPs of the hidden->hidden layers (C={C} jet channels) / device time of the class "
                    "measured with CUDA events around every launch on the launch stream (untimed profile pass); peak = dense tf32 "
                    "GEMM throughput measured in this run (cuBLAS 8192^3, best of 8)" +
                    (f"; bf16 sustained peak from {peaks['source']}: {peaks['bf16_tflops_sustained']}" if on_tc else "") +
                    "; `traffic` = dram bytes per launch of this class from the committed ncu capture (profiles/r02_summary.md), "
                    "scaled to the points per launch, not re-measured here; hbm_gbs_design_traffic = plane sets this design "
                    "streams for the class / its time",
        })
    if roofline is None:  # DeepONet (C = 1, no input derivatives): SURVEY section 8(d) gives 408 algorithmic bytes per pair
        alg_bytes = 408.0 * N
        hbm = alg_bytes / (ms_per_step * 1e-3) / 1e9
        roofline = {"bound": "hbm", "kernel": "whole step (branch + trunk MLPs, head, adjoints, Adam)", "achieved": hbm,
                    "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": hbm / peaks["hbm_gbs"], "traffic": None,
                    "whole_step_tflops": fpp * N / (ms_per_step * 1e-3) / 1e12,
                    "last_adjoint_call_class_ms": don_prof,
                    "note": "algorithmic bytes = 408 B per (u, y) pair (the 100-float sensor row + y + label) over the whole "
                            "step time; the step is compute / stash bound, not input bound"}
    log("profile pass done; timing the CPU baseline")
    cb = cpu_reference_leg(cfg, CPU_SAMPLE[cfg], 8, 1)
    log("cpu baseline done")
    h2d = sum(v.numel() * v.element_size() for v in host.values())
    line = {
        "metric": CONFIGS[cfg]["metric"], "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": CONFIGS[cfg]["dtype"], "data": "synthetic",
        "config": {"workload": CONFIGS[cfg]["workload"],
                   "points_per_gpu": N, "global_points": world * N, "parallelism": f"dp{world}", "jet_channels": C,
                   "flops_per_point": fpp, "l2": "256 MiB buffer written between timed iterations (L2 flush, untimed)",
                   "step": "fwd jets + residual + MSE + adjoint -> flat grad (+ NCCL all-reduce if N>1) + fused Adam"},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": world * h2d, "d2h_bytes_per_step": world * d2h,
                "api": "ppsci.utils.ExpressionSolver.train_forward + ppsci.optimizer.Adam.step, pinned host inputs"},
        "gpu_launches": int(world * launches_per_step * args.steps),
        "roofline": roofline,
        "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "parity": parity,
        "parity_trained": parity_trained,
        "parity_end": parity_end,
        "loss": {k: float(v) for k, v in losses.items()},
        "wall_s_timed_region": t_wall,
    }
    if strong is not None:
        line["strong_scaling"] = strong
    if graph_rec is not None:
        line["cuda_graph"] = graph_rec
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=3, choices=[1, 2, 3, 4, 5])
    ap.add_argument("--graph", default="on", choices=["on", "off"],
                    help="also time the step replayed as a CUDA graph (sub-record `cuda_graph`; the headline stays the eager step)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the losses, weights and Adam moments of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
