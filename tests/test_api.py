"""Host-side API surface (no GPU): constructors, naming, datasets, schedulers, C-ABI loading and
the loud failures that replace a CPU fallback."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import sympy as sp
import torch

import ppsci
from paddlescience_b200.engine import binding as B

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_symbol_declared_in_header():
    lib = B.Library()  # built by __graft_entry__.build()
    header = open(os.path.join(ROOT, "include", "ppsci_b200.h")).read()
    declared = set(re.findall(r"\b(ppsci_b200_[a-z0-9_]+)\s*\(", header))
    assert declared == set(B.EXPORTED_SYMBOLS), declared ^ set(B.EXPORTED_SYMBOLS)
    for sym in declared:
        assert hasattr(lib.lib, sym), sym
    assert "sm_100a" in lib.version()


def test_plan_spec_struct_matches_header_size():
    # the C struct must be the ctypes struct byte for byte: compile a tiny C program and compare
    import subprocess
    import tempfile

    src = '#include <stdio.h>\n#include "ppsci_b200.h"\nint main(){printf("%zu", sizeof(ppsci_plan_spec));return 0;}\n'
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "s.c"), "w").write(src)
        subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), os.path.join(d, "s.c"), "-o", os.path.join(d, "s")], check=True)
        size = int(subprocess.run([os.path.join(d, "s")], capture_output=True, text=True).stdout)
    assert size == C.sizeof(B.PlanSpec)


def test_no_cpu_fallback_anywhere():
    model = ppsci.arch.MLP(("x", "y"), ("u",), 2, 8)
    with pytest.raises(RuntimeError, match="no .*CPU fallback"):
        model({"x": torch.rand(4, 1), "y": torch.rand(4, 1)})
    # plan creation itself needs a B200 as well: checked in a process that sees no CUDA device, so that the machine
    # running the suite having one does not matter
    import subprocess, sys
    code = ("import sys; sys.path.insert(0, %r)\n"
            "import torch, ppsci\n"
            "from paddlescience_b200.engine import binding as B\n"
            "from paddlescience_b200.engine.compiler import compile_residuals\n"
            "from paddlescience_b200.engine.plan import ResidualPlan\n"
            "cr = compile_residuals(ppsci.arch.MLP(('x', 'y'), ('u',), 2, 8).net_spec(), ppsci.equation.Laplace(2).equations)\n"
            "try:\n"
            "    ResidualPlan(cr, torch.float32, ['mean'], [1.0])\n"
            "except B.EngineError as e:\n"
            "    print('EngineError:', e)\n") % ROOT
    p = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True,
                       env={**os.environ, "CUDA_VISIBLE_DEVICES": ""})
    assert re.match(r"EngineError: .*(no CUDA device|sm_100a)", p.stdout), p.stdout + p.stderr
    # the package never imports the oracle or the emulation library
    code = ("import sys; sys.path.insert(0, %r); import ppsci, paddlescience_b200; "
            "bad=[m for m in sys.modules if m.startswith('oracle') or 'emul' in m]; print(bad)") % ROOT
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True).stdout.strip()
    assert out == "[]", out


def test_mlp_constructor_and_state_dict_layout():
    ppsci.utils.misc.set_random_seed(7)
    m = ppsci.arch.MLP(("t", "x"), ("u",), 3, 16, periods={"x": (2.0, False)})
    spec = m.net_spec()
    assert spec.widths == [3, 16, 16, 16, 1]  # (t, cos(pi x), sin(pi x))
    assert spec.feat_kind == [0, 1, 2] and spec.feat_src == [0, 1, 1]
    assert spec.feat_omega[1] == pytest.approx(np.pi)
    sd = m.state_dict()
    assert list(sd) == ["linears.0.weight", "linears.0.bias", "linears.1.weight", "linears.1.bias",
                        "linears.2.weight", "linears.2.bias", "last_fc.weight", "last_fc.bias"]
    assert tuple(sd["linears.0.weight"].shape) == (3, 16)  # [in, out] like paddle nn.Linear
    assert float(sd["linears.1.bias"].abs().max()) == 0.0
    lim = np.sqrt(6.0 / (16 + 16))
    assert float(sd["linears.1.weight"].abs().max()) <= lim
    m2 = ppsci.arch.MLP(("t", "x"), ("u",), 3, 16, periods={"x": (2.0, False)})
    m2.load_state_dict(sd)
    assert torch.equal(m2.flat.data, m.flat.data)
    assert m.num_params == sum(v.numel() for v in sd.values())
    with pytest.raises(ValueError):
        ppsci.arch.MLP(("x",), ("u",), None, 16)
    with pytest.raises(ValueError):
        ppsci.arch.MLP(("x",), ("u",), 2, 16, activation="nope")
    with pytest.raises(NotImplementedError):
        ppsci.arch.MLP(("x",), ("u",), 2, 16, skip_connection=True, weight_norm=True)


def test_equations_and_detach_strings_match_reference_docstring():
    eq = ppsci.equation.NavierStokes(1.0, 1.0, 2, False, detach_keys=("u", "v__y"))
    # ppsci/equation/pde/base.py:99-107 documents exactly this rewrite
    assert str(eq.equations["continuity"]) == "detach(Derivative(v(x, y), y)) + Derivative(u(x, y), x)"
    assert "detach(u(x, y))*Derivative(u(x, y), x)" in str(eq.equations["momentum_x"])
    assert "detach(Derivative(v(x, y), y))*v(x, y)" in str(eq.equations["momentum_y"])
    lap = ppsci.equation.Laplace(3)
    assert len(lap.equations["laplace"].atoms(sp.Derivative)) == 3
    bi = ppsci.equation.Biharmonic(2, -1.0, 1.0)
    orders = sorted(sum(c for _, c in d.variable_count) for d in bi.equations["biharmonic"].atoms(sp.Derivative))
    assert orders == [4, 4, 4]
    pde = ppsci.equation.PDE()
    pde.add_equation("linear_pde", 2 * sp.Symbol("x") + 2 * sp.Symbol("y"))
    assert "linear_pde: 2*x + 2*y" in str(pde)


def test_allen_cahn_callable_traces_to_the_documented_residual():
    from paddlescience_b200.utils.symbolic import trace_to_sympy

    ac = ppsci.equation.AllenCahn(0.01)
    e = trace_to_sympy(ac.equations["allen_cahn"], ("t", "x"), ("u",))
    t, x = sp.symbols("t x")
    u = sp.Function("u")(t, x)
    assert sp.simplify(e - (u.diff(t) - 0.01 ** 2 * u.diff(x, 2) + 5 * u ** 3 - 5 * u)) == 0
    with pytest.raises(TypeError, match="symbolic proxy"):
        ppsci.autodiff.jacobian(torch.rand(3, 1), torch.rand(3, 1))


def test_interior_constraint_builds_reference_batch_layout():
    ppsci.utils.misc.set_random_seed(42)
    rect = ppsci.geometry.Rectangle((0.0, 0.0), (1.0, 1.0))
    eq = ppsci.equation.Laplace(2)
    cst = ppsci.constraint.InteriorConstraint(
        eq.equations, {"laplace": 0.0}, rect,
        {"dataset": "IterableNamedArrayDataset", "iters_per_epoch": 1, "batch_size": 10201},
        ppsci.loss.MSELoss("sum"), evenly=True, name="EQ")
    inp, lab, wt = next(cst.data_iter)
    assert set(inp) == {"x", "y", "sdf"} and inp["x"].shape == (10201, 1) and inp["x"].dtype == torch.float32
    assert lab["laplace"].shape == (10201, 1) and float(lab["laplace"].abs().max()) == 0.0
    assert wt is None
    inp2, _, _ = next(cst.data_iter)  # the iterable dataset yields the whole set every iteration
    assert inp2["x"].data_ptr() == inp["x"].data_ptr()
    # sympy labels / callable weights
    x, y = sp.symbols("x y")
    cst2 = ppsci.constraint.InteriorConstraint(
        eq.equations, {"laplace": sp.sin(x) * y}, rect,
        {"dataset": "NamedArrayDataset", "iters_per_epoch": 2, "batch_size": 8,
         "sampler": {"name": "BatchSampler", "shuffle": False, "drop_last": True}},
        ppsci.loss.MSELoss("mean"), weight_dict={"laplace": lambda d: d["x"] * 2.0}, name="EQ2")
    inp, lab, wt = next(cst2.data_iter)
    assert inp["x"].shape == (8, 1)
    np.testing.assert_allclose(lab["laplace"].numpy(), np.sin(inp["x"].numpy()) * inp["y"].numpy(), rtol=1e-6)
    np.testing.assert_allclose(wt["laplace"].numpy(), 2 * inp["x"].numpy(), rtol=1e-6)


def test_boundary_constraint_criteria():
    ppsci.utils.misc.set_random_seed(1)
    rect = ppsci.geometry.Rectangle((-0.05, -0.05), (0.05, 0.05))
    bc = ppsci.constraint.BoundaryConstraint(
        {"u": lambda out: out["u"]}, {"u": 1.0}, rect,
        {"dataset": "IterableNamedArrayDataset", "iters_per_epoch": 1, "batch_size": 64},
        ppsci.loss.MSELoss("sum"), criteria=lambda x, y: np.isclose(y, 0.05), name="BC_top")
    inp, lab, _ = next(bc.data_iter)
    assert np.allclose(inp["y"].numpy(), 0.05) and inp["x"].shape == (64, 1)
    assert set(inp) == {"x", "y", "normal_x", "normal_y"}
    assert float(lab["u"].min()) == 1.0


def test_lr_schedules():
    sch = ppsci.optimizer.lr_scheduler.ExponentialDecay(10, 100, 1e-3, 0.9, 50)()
    lrs = []
    for _ in range(101):
        lrs.append(sch())
        sch.step()
    assert lrs[0] == pytest.approx(1e-3) and lrs[50] == pytest.approx(9e-4) and lrs[100] == pytest.approx(8.1e-4)
    cos = ppsci.optimizer.lr_scheduler.Cosine(2, 10, 1.0, eta_min=0.1, warmup_epoch=1)()
    vals = []
    for _ in range(20):
        vals.append(cos())
        cos.step()
    assert vals[0] == 0.0 and vals[10] == pytest.approx(1.0) and vals[19] < 0.2 and min(vals[10:]) >= 0.1
    assert not sch.by_epoch


def test_solver_compiles_constraints_on_cpu_and_refuses_to_train():
    model = ppsci.arch.MLP(("x", "y"), ("u", "v", "p"), 2, 16)
    eq = ppsci.equation.NavierStokes(0.01, 1.0, 2, False)
    rect = ppsci.geometry.Rectangle((0, 0), (1, 1))
    cst = ppsci.constraint.InteriorConstraint(
        eq.equations, {"continuity": 0, "momentum_x": 0, "momentum_y": 0}, rect,
        {"dataset": "IterableNamedArrayDataset", "iters_per_epoch": 1, "batch_size": 64},
        ppsci.loss.MSELoss("mean", {"continuity": 2.0}), name="EQ")
    solver = ppsci.solver.Solver(model, {"EQ": cst}, None, ppsci.optimizer.Adam(1e-3)(model), epochs=1, iters_per_epoch=1,
                                 device="cpu")
    cc = solver.forward_helper.compiled_for(model, cst)
    assert cc.names == ["continuity", "momentum_x", "momentum_y"] and cc.compiled.channels == 5
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        solver.train()
