"""Shared parity cases: engine (CUDA library on a B200, or the CPU emulation build of the same
kernel sources) versus the torch oracle (oracle/ppsci_oracle.py), same seeded inputs."""
from __future__ import annotations

import math
from typing import Dict, Optional

import sympy as sp
import torch

from oracle import ppsci_oracle as O
from paddlescience_b200.engine.compiler import NetSpec, compile_residuals
from paddlescience_b200.engine.plan import ResidualPlan


def make_net(in_keys, out_keys, hidden, act, periods=None, gated=False) -> NetSpec:
    feat_src, feat_kind, feat_omega = [], [], []
    for i, k in enumerate(in_keys):
        if periods and k in periods:
            w = 2 * math.pi / periods[k][0]
            feat_src += [i, i]
            feat_kind += [1, 2]
            feat_omega += [w, w]
        else:
            feat_src.append(i)
            feat_kind.append(0)
            feat_omega.append(0.0)
    return NetSpec(tuple(in_keys), tuple(out_keys), feat_src, feat_kind, feat_omega,
                   [len(feat_src)] + list(hidden) + [len(out_keys)], act, gated=gated)


def _ac_exprs():
    t, x = sp.symbols("t x")
    u = sp.Function("u")(t, x)
    return {"allen_cahn": u.diff(t) - 0.01**2 * u.diff(x, 2) + 5 * u**3 - 5 * u}


def _biharm_exprs():
    xs, ys = sp.symbols("x y")
    q = 2.0 * sp.sin(sp.pi * xs / 2) * sp.sin(sp.pi * ys / 3)
    return O.biharmonic_expr(2, q, 1.5)


def _value_exprs():
    x, y = sp.symbols("x y")
    return {"u": sp.Function("u")(x, y), "v": sp.Function("v")(x, y)}


def _mixed_exprs():
    x, y = sp.symbols("x y")
    u = sp.Function("u")(x, y)
    v = sp.Function("v")(x, y)
    return {"mixed": u.diff(x).diff(y) * v + sp.sin(x) * v.diff(y, 2).diff(x) - u * y,
            "third": u.diff(x, 3) + v.diff(y) * u.diff(y)}


def _first_order_exprs():
    # piecewise-linear activations: every second input derivative of the network vanishes identically and the autograd
    # oracle (like Paddle) cannot differentiate the resulting constant again — first derivatives only
    x, y = sp.symbols("x y")
    u = sp.Function("u")(x, y)
    v = sp.Function("v")(x, y)
    return {"div": u.diff(x) + v.diff(y) - u * y, "adv": u * v.diff(x) + sp.sin(x) * u.diff(y)}


CASES = {
    # name: dict(in_keys, out_keys, hidden, act, exprs, dtype, periods, reduction, weights, labels_rand, oracle_exprs, ranges, chunk,
    #            param_scale)
    "ns_f32": dict(in_keys=("x", "y"), out_keys=("u", "v", "p"), hidden=[20, 20], act="tanh",
                   exprs=lambda: O.navier_stokes_expr(0.01, 1.0, 2, False), dtype=torch.float32),
    "laplace_f32_sum_w": dict(in_keys=("x", "y"), out_keys=("u",), hidden=[20] * 4, act="tanh",
                              exprs=lambda: O.laplace_expr(2), dtype=torch.float32, reduction="sum",
                              labels_rand=True, weights=True),
    "ns_f64_wide": dict(in_keys=("x", "y"), out_keys=("u", "v", "p"), hidden=[150, 140], act="tanh",
                        exprs=lambda: O.navier_stokes_expr(0.1, 1.0, 2, False), dtype=torch.float64),
    "ns_f32_wide": dict(in_keys=("x", "y"), out_keys=("u", "v", "p"), hidden=[150, 140], act="tanh",
                        exprs=lambda: O.navier_stokes_expr(0.1, 1.0, 2, False), dtype=torch.float32),
    "ns_f64_chunks": dict(in_keys=("x", "y"), out_keys=("u", "v", "p"), hidden=[16, 16], act="tanh",
                          exprs=lambda: O.navier_stokes_expr(0.1, 1.0, 2, False), dtype=torch.float64,
                          chunk_div=3, weights=True),
    "allen_cahn_period_f64": dict(in_keys=("t", "x"), out_keys=("u",), hidden=[16, 16, 16], act="tanh",
                                  exprs=_ac_exprs, dtype=torch.float64, periods={"x": (2.0, False)},
                                  oracle_exprs=lambda: O.allen_cahn_callable(0.01), ranges={"x": (-1, 1)}),
    "allen_cahn_period_f32": dict(in_keys=("t", "x"), out_keys=("u",), hidden=[32, 32], act="tanh",
                                  exprs=_ac_exprs, dtype=torch.float32, periods={"x": (2.0, False)},
                                  oracle_exprs=lambda: O.allen_cahn_callable(0.01), ranges={"x": (-1, 1)}),
    "biharmonic_f64": dict(in_keys=("x", "y"), out_keys=("u",), hidden=[16, 16, 16], act="tanh",
                           exprs=_biharm_exprs, dtype=torch.float64, ranges={"x": (0, 2), "y": (0, 3)}),
    "ns3d_time_sin_f64": dict(in_keys=("t", "x", "y", "z"), out_keys=("u", "v", "w", "p"), hidden=[12, 12],
                              act="sin", exprs=lambda: O.navier_stokes_expr(0.1, 1.0, 3, True), dtype=torch.float64),
    "laplace3d_silu_f64": dict(in_keys=("x", "y", "z"), out_keys=("u",), hidden=[12, 12], act="silu",
                               exprs=lambda: O.laplace_expr(3), dtype=torch.float64),
    "mixed_third_gelu_f64": dict(in_keys=("x", "y"), out_keys=("u", "v"), hidden=[12, 12], act="gelu",
                                 exprs=_mixed_exprs, dtype=torch.float64),
    "poisson_sigmoid_f64": dict(in_keys=("x", "y"), out_keys=("p",), hidden=[12, 12], act="sigmoid",
                                exprs=lambda: O.poisson_expr(2), dtype=torch.float64),
    # the reference's piecewise activations (activation.py:139-145: nn.ELU(), nn.SELU(), nn.LeakyReLU() with paddle's defaults)
    "ns_elu_f64": dict(in_keys=("x", "y"), out_keys=("u", "v", "p"), hidden=[12, 12], act="elu",
                       exprs=lambda: O.navier_stokes_expr(0.1, 1.0, 2, False), dtype=torch.float64),
    "laplace_selu_f32": dict(in_keys=("x", "y"), out_keys=("u",), hidden=[16, 16], act="selu",
                             exprs=lambda: O.laplace_expr(2), dtype=torch.float32),
    "laplace_siren_f64": dict(in_keys=("x", "y"), out_keys=("u",), hidden=[12, 12], act="siren",
                              exprs=lambda: O.laplace_expr(2), dtype=torch.float64, siren_init=True),
    # ModifiedMLP (mlp.py:318-506): embed_u / embed_v + y <- y u + (1 - y) v after every hidden layer (kernels_gate.cuh)
    "modified_ns_f64": dict(in_keys=("x", "y"), out_keys=("u", "v", "p"), hidden=[12, 12, 12], act="tanh", modified=True,
                            exprs=lambda: O.navier_stokes_expr(0.1, 1.0, 2, False), dtype=torch.float64),
    "modified_laplace_f32": dict(in_keys=("x", "y"), out_keys=("u",), hidden=[20, 20], act="tanh", modified=True,
                                 exprs=lambda: O.laplace_expr(2), dtype=torch.float32),
    "modified_biharmonic_silu_f64": dict(in_keys=("x", "y"), out_keys=("u",), hidden=[10, 10], act="silu", modified=True,
                                         exprs=_biharm_exprs, dtype=torch.float64),
    "modified_ac_period_f64": dict(in_keys=("t", "x"), out_keys=("u",), hidden=[12, 12], act="tanh", modified=True,
                                   periods={"x": (2.0, False)}, exprs=_ac_exprs, dtype=torch.float64,
                                   ranges={"x": (-1, 1)}),
    "first_order_leaky_relu_f64": dict(in_keys=("x", "y"), out_keys=("u", "v"), hidden=[12, 12], act="leaky_relu",
                                       exprs=_first_order_exprs, dtype=torch.float64),
}

# Cases added after the round's last GPU minutes were spent (never run on hardware): kept out of CASES so that the early
# test_gpu_parity.py cannot stop a ``pytest -x`` run on them; the emulated CPU test runs them beside CASES and
# tests/test_zzz_trainable_activations.py runs them on the GPU at the very end of the suite.
LATE_CASES = {
    # activations with a trainable parameter (activation.py:28-58): Stan's beta per unit, Swish's beta per layer — the dx
    # epilogue also reduces dLoss/dbeta
    "ns_stan_f64": dict(in_keys=("x", "y"), out_keys=("u", "v", "p"), hidden=[12, 12, 12], act="stan", trainable_act=True,
                        exprs=lambda: O.navier_stokes_expr(0.1, 1.0, 2, False), dtype=torch.float64),
    "biharmonic_swish_b_f64": dict(in_keys=("x", "y"), out_keys=("u",), hidden=[10, 10], act="swish", trainable_act=True,
                                   exprs=_biharm_exprs, dtype=torch.float64),
    "laplace_stan_f32": dict(in_keys=("x", "y"), out_keys=("u",), hidden=[20, 20], act="stan", trainable_act=True,
                             exprs=lambda: O.laplace_expr(2), dtype=torch.float32),
}

# shapes served by the tcgen05 kernels (hidden widths multiple of 32/128); CPU emulation skips them
TC_CASES = {
    "ns_f32_tc_256": dict(in_keys=("x", "y"), out_keys=("u", "v", "p"), hidden=[256, 256, 256], act="tanh",
                          exprs=lambda: O.navier_stokes_expr(0.01, 1.0, 2, False), dtype=torch.float32),
    "ns_f32_tc_128_sin": dict(in_keys=("x", "y"), out_keys=("u", "v", "p"), hidden=[128, 128, 128], act="sin",
                              exprs=lambda: O.navier_stokes_expr(0.01, 1.0, 2, False), dtype=torch.float32),
    "ac_f32_tc_128": dict(in_keys=("t", "x"), out_keys=("u",), hidden=[128] * 4, act="tanh", exprs=_ac_exprs,
                          dtype=torch.float32, periods={"x": (2.0, False)},
                          oracle_exprs=lambda: O.allen_cahn_callable(0.01), ranges={"x": (-1, 1)}),
    # several workspace chunks per call on the tensor-core path (chunk = ceil(n / 3))
    "ns_f32_tc_256_chunks": dict(in_keys=("x", "y"), out_keys=("u", "v", "p"), hidden=[256, 256, 256], act="tanh",
                                 exprs=lambda: O.navier_stokes_expr(0.01, 1.0, 2, False), dtype=torch.float32,
                                 chunk_div=3, weights=True),
    # widths that give odd K-chunk counts (3, 5), odd 32-column block counts and a 16-row weight half per CTA
    "ns_f32_tc_mixed": dict(in_keys=("x", "y"), out_keys=("u", "v", "p"), hidden=[96, 160, 64, 32], act="tanh",
                            exprs=lambda: O.navier_stokes_expr(0.01, 1.0, 2, False), dtype=torch.float32),
    # C = 7 (three second-order directions): pair kernels with two producer groups of 5 warps + 4 idle producer warps
    "ns3d_f32_tc_256": dict(in_keys=("x", "y", "z"), out_keys=("u", "v", "w", "p"), hidden=[256, 256, 256], act="tanh",
                            exprs=lambda: O.navier_stokes_expr(0.05, 1.0, 3, False), dtype=torch.float32),
    # C = 1 (no derivatives: a boundary / supervised constraint): 128 points per tile, three producer passes
    "value_f32_tc_256": dict(in_keys=("x", "y"), out_keys=("u", "v"), hidden=[256, 256, 256], act="tanh",
                             exprs=lambda: _value_exprs(), dtype=torch.float32, labels_rand=True),
    "biharmonic_f32_tc_128": dict(in_keys=("x", "y"), out_keys=("u",), hidden=[128, 128, 128], act="tanh",
                                  exprs=_biharm_exprs, dtype=torch.float32, ranges={"x": (0, 2), "y": (0, 3)}),
}

# The five BASELINE.json configs at their named shapes (VERDICT r1 NS-2).  Network widths / depths, jet channels,
# reductions and point counts follow SURVEY.md section 8(d); "n" is the point count of the GPU test.
NAMED_CASES = {
    # cfg1: examples/laplace/laplace2d.py:48-59 — 101 x 101 evenly spaced interior grid, MSELoss("sum")
    "cfg1_laplace_4x20": dict(in_keys=("x", "y"), out_keys=("u",), hidden=[20] * 4, act="tanh",
                              exprs=lambda: O.laplace_expr(2), dtype=torch.float32, reduction="sum",
                              grid=((0.0, 0.0), (1.0, 1.0)), n=10201),
    "cfg1_laplace_5x20": dict(in_keys=("x", "y"), out_keys=("u",), hidden=[20] * 5, act="tanh",
                              exprs=lambda: O.laplace_expr(2), dtype=torch.float32, reduction="sum",
                              grid=((0.0, 0.0), (1.0, 1.0)), n=10201),
    # cfg2: Allen-Cahn, 4 x 128, periodic in x, 2^18 points
    "cfg2_allen_cahn_4x128": dict(in_keys=("t", "x"), out_keys=("u",), hidden=[128] * 4, act="tanh", exprs=_ac_exprs,
                                  dtype=torch.float32, periods={"x": (2.0, False)},
                                  oracle_exprs=lambda: O.allen_cahn_callable(0.01), ranges={"x": (-1, 1)}, n=1 << 18),
    # cfg3: LDC Navier-Stokes Re=100, 6 x 256 — the headline shape
    "cfg3_ldc_6x256": dict(in_keys=("x", "y"), out_keys=("u", "v", "p"), hidden=[256] * 6, act="tanh",
                           exprs=lambda: O.navier_stokes_expr(0.01, 1.0, 2, False), dtype=torch.float32, n=1 << 16),
    # cfg4: Biharmonic2D, 5 x 128, fp64, C = 17 (x, y, x+y, x-y to order 4)
    "cfg4_biharmonic_5x128_f64": dict(in_keys=("x", "y"), out_keys=("u",), hidden=[128] * 5, act="tanh",
                                      exprs=_biharm_exprs, dtype=torch.float64, ranges={"x": (0, 2), "y": (0, 3)},
                                      n=1 << 15),
}

TOL = {  # (loss rel, residual rel-L2, grad rel-L2)
    torch.float32: (2e-6, 5e-6, 1e-5),
    torch.float64: (1e-12, 1e-11, 1e-11),
}


def oracle_in_blocks(om, params, exprs, inputs, labels, wts, reduction, lw, block: int = 8192):
    """O.train_forward_backward over blocks of points (the fp64 double-backward graph of 6 x 256 holds ~0.6 MB per
    point): per-point residuals concatenate, "sum" losses and their gradients add, "mean" = sum / n."""
    n = next(iter(inputs.values())).shape[0]
    if n <= block:
        return O.train_forward_backward(om, params, exprs, inputs, labels, wts, reduction, lw)
    losses, res, grad = {}, {}, None
    for s in range(0, n, block):
        sl = slice(s, min(n, s + block))
        l_, r_, g_ = O.train_forward_backward(om, params, exprs, {k: v[sl] for k, v in inputs.items()},
                                              {k: v[sl] for k, v in labels.items()},
                                              {k: v[sl] for k, v in wts.items()} if wts else None, "sum", lw)
        for k, v in l_.items():
            losses[k] = losses.get(k, 0.0) + v
        for k, v in r_.items():
            res.setdefault(k, []).append(v)
        grad = g_ if grad is None else grad + g_
    scale = 1.0 / n if reduction == "mean" else 1.0
    return ({k: v * scale for k, v in losses.items()}, {k: torch.cat(v) for k, v in res.items()}, grad * scale)


def run_case(name, n: int, library=None, device="cpu", backend: int = 0, seed: int = 0,
             oracle_subset: int = 0) -> Dict[str, float]:
    """``name``: key of CASES / TC_CASES / NAMED_CASES, or a case dict.  ``oracle_subset`` > 0: the engine runs all
    ``n`` points, the oracle only ``oracle_subset`` evenly strided points; residuals are compared on that subset and
    the engine's loss against the mean / sum of its own residuals (loss / grad errors are then not oracle errors)."""
    c = name if isinstance(name, dict) else (CASES.get(name) or LATE_CASES.get(name) or TC_CASES.get(name) or NAMED_CASES[name])
    torch.manual_seed(seed)
    dtype = c["dtype"]
    exprs = c["exprs"]()
    periods = c.get("periods")
    net = make_net(c["in_keys"], c["out_keys"], c["hidden"], {"swish": "swish_b"}.get(c["act"], c["act"]) if c.get("trainable_act") else c["act"],
                   periods, gated=bool(c.get("modified")))
    cr = compile_residuals(net, exprs)
    nres = len(cr.names)
    reduction = c.get("reduction", "mean")
    chunk = (n + c["chunk_div"] - 1) // c["chunk_div"] if c.get("chunk_div") else 0
    plan = ResidualPlan(cr, dtype, [reduction] * nres, [1.0 + 0.5 * k for k in range(nres)], chunk_points=chunk,
                        backend=backend, library=library)
    inputs = {}
    if c.get("grid"):  # the reference's evenly=True interior set (geometry_nd.py:83-110): itertools.product order
        pts = O.hypercube_uniform_points(*c["grid"], n, boundary=True)
        n = pts.shape[0]
        for i, k in enumerate(c["in_keys"]):
            inputs[k] = torch.as_tensor(pts[:, i:i + 1], dtype=torch.float64).to(dtype)
    else:
        for k in c["in_keys"]:
            lo, hi = (c.get("ranges") or {}).get(k, (0, 1))
            inputs[k] = (torch.rand(n, 1, dtype=torch.float64) * (hi - lo) + lo).to(dtype)
    om = O.OracleMLP(c["in_keys"], c["out_keys"], c["hidden"], c["act"], periods, modified=bool(c.get("modified")),
                     trainable_act=bool(c.get("trainable_act")))
    params = O.xavier_uniform_params(om.widths, 1, torch.float64)
    if c.get("modified"):  # [Wu | bu | Wv | bv] behind the layers
        params = torch.cat([params, O.xavier_uniform_params([om.widths[0], om.widths[1]], 2, torch.float64),
                            O.xavier_uniform_params([om.widths[0], om.widths[1]], 3, torch.float64)])
    params = (params + 0.1 * torch.randn_like(params))
    if c.get("param_scale"):  # weights and biases away from the init scale (a trained or a shrunk network)
        params = params * float(c["param_scale"])
    if c.get("trainable_act"):  # Stan.beta per unit / Swish.beta per layer, behind the layers (1 at start in the reference)
        params = torch.cat([params, 1.0 + 0.2 * torch.randn(sum(om.beta_len), dtype=torch.float64)])
    if c.get("siren_init"):  # weights on the scale Siren's initialisers use (sqrt(6 / in) / w0, activation.py:103-136)
        params = params / 30.0
    params = params.to(dtype)
    labels = {k: (torch.randn(n, 1, dtype=torch.float64).to(dtype) if c.get("labels_rand") else torch.zeros(n, 1, dtype=dtype))
              for k in cr.names}
    wts = {k: torch.rand(n, 1, dtype=torch.float64).to(dtype) for k in cr.names} if c.get("weights") else None
    lw = {k: 1.0 + 0.5 * i for i, k in enumerate(cr.names)}
    oracle_exprs = c["oracle_exprs"]() if c.get("oracle_exprs") else exprs
    sub = None
    if oracle_subset and oracle_subset < n:
        sub = torch.arange(0, n, n // oracle_subset)[:oracle_subset]
    pick = (lambda v: v[sub]) if sub is not None else (lambda v: v)
    lo_, ro, go = oracle_in_blocks(
        om, params.double(), oracle_exprs, {k: pick(v).double() for k, v in inputs.items()},
        {k: pick(v).double() for k, v in labels.items()}, {k: pick(v).double() for k, v in wts.items()} if wts else None,
        reduction, lw)
    dev = torch.device(device)
    d_in = {k: v.to(dev) for k, v in inputs.items()}
    d_par = params.to(dev)
    d_grads = torch.zeros_like(d_par)
    d_lab = {k: v.to(dev) for k, v in labels.items()}
    d_w = {k: v.to(dev) for k, v in wts.items()} if wts else None
    d_res = {k: torch.empty(n, 1, dtype=dtype, device=dev) for k in cr.names}
    loss = plan.loss_fwd_bwd(d_in, d_par, d_grads, labels=d_lab, weights=d_w, residual_out=d_res)
    loss = loss.cpu()
    if sub is not None:
        # loss: against the engine's own residuals reduced in fp64 (self-consistency at full size)
        def own(i, k):
            r = d_res[k].cpu().double()
            e2 = (r - labels[k].double()) ** 2
            if wts:
                e2 = e2 * wts[k].double()
            return float(lw[k] * (e2.mean() if reduction == "mean" else e2.sum()))
        lerr = max(abs(float(loss[i]) - own(i, k)) / max(1e-30, abs(own(i, k))) for i, k in enumerate(cr.names))
        rerr = max(float((d_res[k].cpu().double()[sub] - ro[k]).norm() / ro[k].norm().clamp_min(1e-30)) for k in cr.names)
        gerr = float("nan")
    else:
        lerr = max(abs(float(loss[i]) - float(lo_[k])) / max(1e-30, abs(float(lo_[k]))) for i, k in enumerate(cr.names))
        rerr = max(float((d_res[k].cpu().double() - ro[k]).norm() / ro[k].norm().clamp_min(1e-30)) for k in cr.names)
        gerr = float((d_grads.cpu().double() - go).norm() / go.norm())
    # forward-only entry point must agree with the fused call
    _, res2 = plan.forward(d_in, d_par, want_jets=False)
    ferr = max(float((res2[k] - d_res[k]).abs().max()) for k in cr.names)
    return dict(loss=lerr, res=rerr, grad=gerr, fwd_vs_fused=ferr, channels=cr.channels, launches=plan.last_launches,
                tc=plan.uses_tcgen05)
