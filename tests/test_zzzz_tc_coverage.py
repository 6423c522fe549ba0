"""Tensor-core coverage beyond tanh at the init scale.

On a B200 the default backend sends every fp32, non-gated plan whose activation is not stan / swish and which has one
tensor-core-eligible layer (K a multiple of 32 up to 1024, N a multiple of 32 up to 256) to the tcgen05 kernels; any
activation other than tanh runs there with the runtime jet layout.  These tests follow that selection:

* every activation of ``binding.ACT_IDS`` (without the trainable stan / swish) on the tensor cores against the fp64
  oracle, second-order residuals for the smooth ones, first-order ones for the piecewise-linear family, plus one third-
  and one fourth-order residual;
* ``MLP(fourier=...)``: the embedding layer's ``sin`` is not the network's activation, so these plans must run on the
  CUDA-core kernels (the tensor-core kernels apply one activation to every hidden layer) and match the oracle; a forced
  ``backend=2`` must be refused, never return a result;
* weights and inputs away from the init scale (parameters x0.05 / x3, inputs in [-20, 20]).

Every tensor-core case asserts ``r["tc"]`` so that a change of kernel selection is noticed.  The emulated cases run the
same kernel sources compiled for the CPU (tests/emul); the GPU cases run the default backend on a B200.  The GPU cases
sit in the last test file so that a ``pytest -x`` run reaches every older test first."""
import pytest
import torch

import ppsci
from oracle import ppsci_oracle as O
from paddlescience_b200.engine import binding as B
from paddlescience_b200.engine.compiler import compile_residuals
from paddlescience_b200.engine.plan import ResidualPlan
from tests.cases import NAMED_CASES, TOL, _biharm_exprs, _first_order_exprs, _mixed_exprs, run_case

TOL_TC = dict(loss=1e-5, res=1e-5, grad=5e-5)
TOL_SIMT32 = dict(zip(("loss", "res", "grad"), TOL[torch.float32]))

# stan / swish_b carry a trainable parameter (CUDA-core kernels only); "swish" is an alias of silu's id
TC_ACTS = sorted(set(B.ACT_IDS) - {"stan", "swish", "swish_b"})
# every second input derivative of these networks vanishes identically (or is a jump): first-order residuals only
PIECEWISE = ("identity", "relu", "leaky_relu", "elu", "selu")


def _act_case(act, hidden, exprs=None, out_keys=("u", "v"), **kw):
    if exprs is None and act in PIECEWISE:
        exprs = _first_order_exprs
    elif exprs is None:
        exprs, out_keys = (lambda: O.navier_stokes_expr(0.01, 1.0, 2, False)), ("u", "v", "p")
    c = dict(in_keys=("x", "y"), out_keys=out_keys, hidden=list(hidden), act=act, exprs=exprs, dtype=torch.float32,
             siren_init=act == "siren")
    c.update(kw)
    return c


def _check(r, tol=TOL_TC):
    assert r["loss"] <= tol["loss"], r
    assert r["res"] <= tol["res"], r
    assert r["grad"] <= tol["grad"], r


@pytest.fixture(scope="module")
def emul_lib():
    from tests.emul.build_emul import build

    return B.Library(build())


# ---- activation matrix ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("act", TC_ACTS)
def test_emulated_tc_activation_matches_oracle(emul_lib, act):
    r = run_case(_act_case(act, [32, 32, 32]), 60, library=emul_lib, device="cpu", backend=2)
    assert r["tc"]
    _check(r)
    assert r["fwd_vs_fused"] == 0.0, r


@pytest.mark.parametrize("act,exprs,ranges", [("gelu", _mixed_exprs, None),
                                              ("sin", _biharm_exprs, {"x": (0, 2), "y": (0, 3)})],
                         ids=["third_order_gelu", "fourth_order_sin"])
def test_emulated_tc_higher_order_runtime_layout(emul_lib, act, exprs, ranges):
    """Orders 3 and 4 through the runtime-layout (TC_LAY_DYN) tensor-core kernels."""
    c = _act_case(act, [32, 32, 32], exprs=exprs, out_keys=("u",) if exprs is _biharm_exprs else ("u", "v"), ranges=ranges)
    r = run_case(c, 60, library=emul_lib, device="cpu", backend=2)
    assert r["tc"]
    _check(r)


# ---- Fourier-feature MLPs ---------------------------------------------------------------------------------------
def _fourier_model(dim, hidden, periods=None, seed=5):
    ppsci.utils.misc.set_random_seed(seed)
    m = ppsci.arch.MLP(("x", "y"), ("u",), 3, hidden, "tanh", periods=periods, fourier={"dim": dim, "scale": 1.5},
                       dtype=torch.float32)
    with torch.no_grad():
        m.flat.data[: m._n_lin] += 0.1 * torch.randn(m._n_lin, dtype=torch.float32)  # biases off zero
    return m


def _fourier_oracle(m, dim, hidden, periods, inp):
    raw = m.flat.data.detach().cpu().double().clone().requires_grad_(True)
    om = O.OracleMLP(("x", "y"), ("u",), [hidden] * 3, "tanh", periods, fourier={"dim": dim, "scale": 1.5})
    assert om.n_params == raw.numel()
    x = {k: inp[k].detach().cpu().double().clone().requires_grad_(True) for k in ("x", "y")}
    out = om(raw, x)
    data = dict(x)
    data.update(out)
    loss = (O.eval_expr(O.laplace_expr(2)["laplace"], data) ** 2).mean()
    loss.backward()
    return float(loss.detach()), raw.grad, out["u"].detach()


def _fourier_errors(m, dim, hidden, periods, n, dev):
    """(loss, gradient, forward value) relative errors of ``train_forward`` / ``model(...)`` against the oracle."""
    eq = ppsci.equation.Laplace(2)
    rect = ppsci.geometry.Rectangle((0, 0), (1, 1))
    cst = ppsci.constraint.InteriorConstraint(eq.equations, {"laplace": 0}, rect,
                                              {"dataset": "IterableNamedArrayDataset", "iters_per_epoch": 1, "batch_size": n},
                                              ppsci.loss.MSELoss("mean"), name="EQ")
    ds = cst.data_loader.loader
    inp = {k: v.to(dev, torch.float32) for k, v in ds.input.items()}
    lab = {k: v.to(dev, torch.float32) for k, v in ds.label.items()}
    losses_all, _ = ppsci.utils.ExpressionSolver().train_forward((cst.output_expr,), [inp], m, {"EQ": cst}, [lab], [None])
    cols = {k: inp[k] for k in ("x", "y")}
    if dev == "cpu":  # MLP.forward refuses host tensors; the emulated kernels take its value plan directly
        got_u = m._plan_values().forward(cols, m.engine_params(), want_jets=True, want_residuals=False)[0][0][:, :1]
    else:
        got_u = m(cols)["u"]
    got_u = got_u.detach().cpu().double()
    loss, grad, u = _fourier_oracle(m, dim, hidden, periods, inp)
    lerr = abs(float(losses_all["laplace"]) - loss) / abs(loss)
    gerr = float((m.flat.grad.detach().cpu().double() - grad).norm() / grad.norm())
    verr = float((got_u - u).norm() / u.norm())
    return lerr, gerr, verr


def _fourier_plan(m, backend=0):
    return ResidualPlan(compile_residuals(m.net_spec(), O.laplace_expr(2)), torch.float32, ["mean"], [1.0], backend=backend)


# (fourier dim, hidden width, periods): dim == width would reach the fused kernels, dim 64 -> 32 the layer-at-a-time ones
FOURIER_SHAPES = [(32, 32, None), (64, 32, None), (32, 32, {"x": (2.0, False)})]


@pytest.mark.parametrize("dim,hidden,periods", FOURIER_SHAPES, ids=["fused_shape", "layerwise_shape", "periods"])
def test_emulated_fourier_mlp_matches_oracle_and_refuses_tc(monkeypatch, emul_lib, dim, hidden, periods):
    monkeypatch.setattr(B, "_default", emul_lib)
    m = _fourier_model(dim, hidden, periods)
    assert m.net_spec().act_first == "sin"
    assert not _fourier_plan(m).uses_tcgen05
    lerr, gerr, verr = _fourier_errors(m, dim, hidden, periods, 60, "cpu")
    assert lerr <= TOL_SIMT32["loss"] and gerr <= TOL_SIMT32["grad"] and verr <= TOL_SIMT32["res"], (lerr, gerr, verr)
    # a forced tensor-core plan applies tanh to the embedding layer: it must be refused, not computed
    monkeypatch.setenv("PPSCI_B200_BACKEND", "2")
    m.flat.grad = None
    try:
        lerr, gerr, verr = _fourier_errors(m, dim, hidden, periods, 60, "cpu")
    except B.EngineError as e:
        assert "backend=2 (tcgen05) requested but the plan is not eligible" in str(e)
    else:
        pytest.fail(f"backend=2 returned a result for a Fourier MLP: loss error {lerr:.3g}, gradient error {gerr:.3g}, "
                    f"value error {verr:.3g}")


# ---- parameters and inputs away from the init scale -------------------------------------------------------------
def _ns_range_case(hidden, scale, lim):
    return dict(in_keys=("x", "y"), out_keys=("u", "v", "p"), hidden=list(hidden), act="tanh",
                exprs=lambda: O.navier_stokes_expr(0.01, 1.0, 2, False), dtype=torch.float32, param_scale=scale,
                ranges={"x": (-lim, lim), "y": (-lim, lim)} if lim else None)


@pytest.mark.parametrize("lim", [0, 20], ids=["unit_inputs", "inputs_pm20"])
@pytest.mark.parametrize("scale", [0.05, 1.0, 3.0])
def test_emulated_tc_parameter_and_input_range(emul_lib, scale, lim):
    """3 x 128 tanh N-S: the layer-fused tf32 forward and the fused dx chain."""
    r = run_case(_ns_range_case([128] * 3, scale, lim), 45, library=emul_lib, device="cpu", backend=2)
    assert r["tc"]
    _check(r)


# 256-wide layers away from the init scale leave the 1e-5 bar (DESIGN.md section 4.1, "Away from the init scale"):
# at x0.05 the network is nearly linear, every point carries the same first-derivative jet and the same rounding, so the
# error is a common offset of the continuity residual that no averaging over points removes; at x3 it is the zero-mean
# part.  Bounds: the measured errors (emulated kernels, 60 points, seed 0) with a 1.25x margin.
TOL_FP16_EMUL = {0.05: dict(loss=6.1e-5, res=3.1e-5, grad=TOL_TC["grad"]),
                 3.0: dict(loss=1.7e-5, res=2.8e-5, grad=TOL_TC["grad"])}


@pytest.mark.parametrize("scale", sorted(TOL_FP16_EMUL))
def test_emulated_fused_fp16_forward_away_from_init_scale(emul_lib, scale):
    """4 x 256 tanh N-S: the fp16-operand fused forward (default for 256-wide layers) with its per-row operand scales."""
    r = run_case(_ns_range_case([256] * 4, scale, 0), 60, library=emul_lib, device="cpu", backend=2)
    assert r["tc"]
    _check(r, TOL_FP16_EMUL[scale])


# ---- GPU: default backend -----------------------------------------------------------------------------------------
# cos at 3 x 128: loss error 1.64e-5 measured on a B200 (1000 W power limit), a round-toward-zero residue common to all
# points (DESIGN.md section 4.1); residual 9.3e-6 and gradient 1.5e-6 stay within TOL_TC.  Bound = measurement x 1.25
TOL_ACT_B200 = {("cos", "3x128"): dict(TOL_TC, loss=2.1e-5)}


@pytest.mark.gpu
@pytest.mark.parametrize("hidden", [[128] * 3, [96, 160, 64, 32]], ids=["3x128", "mixed"])
@pytest.mark.parametrize("act", TC_ACTS)
def test_gpu_tc_activation_matches_oracle(act, hidden):
    r = run_case(_act_case(act, hidden), 3000, device="cuda:0")
    assert r["tc"], "fp32 MLPs with tensor-core-eligible layers must run on the tcgen05 kernels"
    _check(r, TOL_ACT_B200.get((act, "3x128" if hidden == [128] * 3 else "mixed"), TOL_TC))


@pytest.mark.gpu
@pytest.mark.parametrize("act", TC_ACTS)
def test_gpu_tc_activation_ragged_point_count(act):
    """A partial last tile and an odd tile count (one CTA of the last pair has no tile)."""
    r = run_case(_act_case(act, [128] * 3), 3013, device="cuda:0")
    assert r["tc"]
    _check(r)


@pytest.mark.gpu
@pytest.mark.parametrize("periods", [None, {"x": (2.0, False)}], ids=["plain", "periods"])
def test_gpu_fourier_mlp_matches_oracle(periods):
    """Fourier dim 128, 3 x 128 hidden: every layer after the embedding is tensor-core eligible, yet the plan runs on
    the CUDA-core kernels and training (loss, gradient) and ``model(...)`` agree with the oracle."""
    m = _fourier_model(128, 128, periods).to("cuda")
    lerr, gerr, verr = _fourier_errors(m, 128, 128, periods, 3000, "cuda")
    assert lerr <= TOL_SIMT32["loss"] and gerr <= TOL_SIMT32["grad"] and verr <= TOL_SIMT32["res"], (lerr, gerr, verr)
    assert not _fourier_plan(m).uses_tcgen05


# Every (shape, scale, mask) stays within TOL_TC on a B200 except cfg3 with its parameters x3, where even the CUDA-core
# fp32 kernels reach residual 1.3e-5 / gradient 2.3e-5 (DESIGN.md section 4.1).  Bounds there: the worse of the two input
# ranges measured on a B200 (1000 W power limit, 3,000 points, seed 0) x 1.25.
TOL_RANGE_B200 = {("cfg3_ldc_6x256", 3.0, 255): dict(loss=1.3e-5, res=7.4e-5, grad=1.18e-4),
                  ("cfg3_ldc_6x256", 3.0, 63): dict(loss=TOL_TC["loss"], res=2.9e-5, grad=TOL_TC["grad"])}


def _named_range_case(name, scale, lim):
    c = dict(NAMED_CASES[name], param_scale=scale)
    c.pop("n")
    if lim:
        c["ranges"] = {k: (-lim, lim) for k in c["in_keys"]}
    return c


@pytest.mark.gpu
@pytest.mark.parametrize("mask", [255, 63])
@pytest.mark.parametrize("lim", [0, 20], ids=["unit_inputs", "inputs_pm20"])
@pytest.mark.parametrize("scale", [0.05, 1.0, 3.0])
@pytest.mark.parametrize("name", ["cfg2_allen_cahn_4x128", "cfg3_ldc_6x256"])
def test_gpu_tc_named_shape_parameter_and_input_range(monkeypatch, name, scale, lim, mask):
    monkeypatch.setenv("PPSCI_B200_TC_MASK", str(mask))
    r = run_case(_named_range_case(name, scale, lim), 3000, device="cuda:0")
    assert r["tc"]
    _check(r, TOL_RANGE_B200.get((name, scale, mask), TOL_TC))
