"""Wiring of the example scripts on the GPU-less build box: every ``ppsci`` call of
``examples/allen_cahn/allen_cahn_piratenet.py`` (PirateNet with fourier + random_weight + periods, CausalMSELoss on a
ContinuousNamedArrayDataset, supervised initial condition, ExponentialDecay, mtl.GradNorm) runs two training iterations
in its small configuration through the CPU emulation of the kernel sources (test infrastructure; the product path is
the CUDA library).  The optimizer step is the same fused Adam kernel, called without the CUDA-device guard."""
import importlib.util
import os

import numpy as np
import pytest
import torch

import ppsci
from paddlescience_b200.engine import binding as B
from paddlescience_b200.optimizer import optimizer as opt_mod

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _load(path):
    spec = importlib.util.spec_from_file_location("example_" + os.path.basename(path)[:-3], os.path.join(ROOT, path))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_cartesian_product_known_answer():
    out = ppsci.utils.misc.cartesian_product(np.array([1, 2]), np.array([10, 20]), np.array([100, 200]))  # misc.py:487-500
    assert out.tolist() == [[1, 10, 100], [1, 10, 200], [1, 20, 100], [1, 20, 200], [2, 10, 100], [2, 10, 200],
                            [2, 20, 100], [2, 20, 200]]


@pytest.mark.parametrize("arch", ["piratenet", "modifiedmlp"])
def test_allen_cahn_piratenet_example_trains_two_iterations(monkeypatch, arch):
    from tests.emul.build_emul import build

    lib = B.Library(build())
    monkeypatch.setattr(B, "_default", lib)
    # the emulated library reads host memory: the Solver must keep the model and data on the host even where a GPU is
    # visible (it moves them to CUDA whenever one is)
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)

    def cpu_step(self):  # FlatAdam.step without the device guard, on the emulated library
        p = self.model.flat
        self._ensure_state()
        self.t += 1
        rc = lib.lib.ppsci_b200_adam_step(B.F64 if p.dtype == torch.float64 else B.F32, p.data.data_ptr(), p.grad.data_ptr(),
                                          self.exp_avg.data_ptr(), self.exp_avg_sq.data_ptr(), p.numel(), self.get_lr(),
                                          self.beta1, self.beta2, self.epsilon, self.weight_decay, self.t, self.grad_scale, None)
        assert rc == 0

    monkeypatch.setattr(opt_mod.FlatAdam, "step", cpu_step)
    ex = _load("examples/allen_cahn/allen_cahn_piratenet.py")
    cfg = ex.merged(ex.CFG, ex.SMALL)
    solver, model, equation, constraint, eval_data = ex.build(cfg, arch=arch)
    assert isinstance(model, ppsci.arch.PirateNet if arch == "piratenet" else ppsci.arch.ModifiedMLP)
    assert model.random_weight and model.fourier
    assert type(constraint["PDE"].loss).__name__ == "CausalMSELoss" and type(solver.loss_aggregator).__name__ == "GradNorm"
    p0 = model.flat.data.clone()
    from paddlescience_b200.solver import train as train_mod

    train_mod.train_epoch_func(solver, 1, solver.log_freq)  # Solver.train's epoch body (Solver.train itself insists on CUDA)
    assert solver.global_step == 2
    assert torch.isfinite(model.flat.data).all() and float((model.flat.data - p0).abs().max()) > 0
    if arch == "piratenet":
        assert float(model.alphas.abs().max()) > 0  # the residual weights take gradient from the first step on
