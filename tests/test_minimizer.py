"""minimize_bfgs (reference minimizers.py:8-51) over any object with ``compute(pos, box, forces)``."""
import types

import numpy as np
import pytest
import torch

from torchmd_b200.minimizers import minimize_bfgs


class Springs:
    """E = sum k |x - x0|^2 ; forces written in place like Forces.compute."""

    def __init__(self, x0, k=2.0):
        self.x0, self.k, self.calls = x0, k, 0

    def compute(self, pos, box, forces):
        self.calls += 1
        d = pos - self.x0
        forces.copy_(-2.0 * self.k * d)
        return [float((self.k * d * d).sum())]


def test_minimiser_finds_the_minimum_and_replaces_positions(capsys):
    torch.manual_seed(0)
    x0 = torch.randn(1, 20, 3)
    system = types.SimpleNamespace(pos=x0 + 0.5 * torch.randn(1, 20, 3), box=torch.zeros(1, 3, 3), forces=torch.zeros(1, 20, 3))
    f = Springs(x0)
    start = system.pos
    minimize_bfgs(system, f, fmax=1e-4, steps=200)
    assert system.pos is not start and system.pos.shape == (1, 20, 3) and system.pos.dtype == torch.float32
    assert (system.pos - x0).abs().max() < 1e-3 and f.calls >= 3
    out = capsys.readouterr().out.splitlines()
    assert out[0].split() == ["Iter", "Epot", "fmax"] and out[1].split()[0] == "0"
    minimize_bfgs(system, f, steps=0)  # no-op
    with pytest.raises(RuntimeError):
        minimize_bfgs(types.SimpleNamespace(pos=torch.zeros(2, 4, 3), box=None, forces=None), f)


class DiffSprings(Springs):
    """The same potential through the toNumpy=False convention (a list of differentiable energies per replica)."""

    def compute(self, pos, box, forces, toNumpy=True):
        if toNumpy:
            return super().compute(pos, box, forces)
        self.calls += 1
        return [(self.k * (p - x) ** 2).sum() for p, x in zip(pos, self.x0)]


def _system(x0, seed=1, spread=0.5):
    g = torch.Generator().manual_seed(seed)
    n = x0.shape[1]
    return types.SimpleNamespace(pos=x0 + spread * torch.randn(x0.shape, generator=g), box=torch.zeros(1, 3, 3), forces=torch.zeros(1, n, 3),
                                 nreplicas=1, natoms=n)


def test_conjugate_gradient_and_torch_lbfgs(capsys):
    from torchmd_b200.minimizers import minimize_cg, minimize_pytorch_bfgs

    x0 = torch.randn(1, 12, 3, generator=torch.Generator().manual_seed(0))
    f, s = Springs(x0), _system(x0)
    start = s.pos.clone()
    assert minimize_cg(s, f, steps=5, threshold=0.1) < 4  # a quadratic bowl: the line search ends within its 0.01 A tolerance of the minimum
    assert torch.equal(s.pos, start)  # like the reference: the coordinates stay in a local
    minimize_cg(s, f, steps=5, threshold=0.1, update_system=True)
    assert (s.pos - x0).abs().max() < 3e-2
    assert minimize_cg(_system(x0), f, steps=3, threshold=None) == 2

    f, s = DiffSprings(x0), _system(x0)
    energies = minimize_pytorch_bfgs(s, f, steps=3, max_iter=10)
    assert (s.pos - x0).abs().max() < 1e-3 and energies.shape[-1] == f.calls
    assert capsys.readouterr().out.splitlines()[0].split() == ["Iter", "Epot", "fmax"]
    assert minimize_pytorch_bfgs(s, f, steps=0) is None


def test_conjugate_gradient_follows_the_references_evaluations():
    """Same sequence of trial points as the reference's torchmd/minimizers.py evaluated (stored in
    tests/golden/minimizer_cg_trace.npz by make_golden_known_answers.py) on an anharmonic potential, where the bracket
    has to shrink and shift."""
    from conftest import load_golden
    from torchmd_b200 import minimizers as mine

    class Quartic:
        def __init__(self):
            self.trace = []

        def compute(self, pos, box, forces):
            p = pos.detach()
            self.trace.append(p.clone())
            forces.copy_(-(4 * p**3 - 6 * p + 0.5))
            return [float((p**4 - 3 * p**2 + 0.5 * p).sum())]

    g = load_golden("minimizer_cg_trace")
    f, s = Quartic(), _system(torch.zeros(1, 6, 3))
    s.pos = torch.tensor(g["start"])
    ret = mine.minimize_cg(s, f, steps=4)
    ref_trace = torch.tensor(g["trace"])[:, None]
    assert ret == int(g["returned"]) and len(f.trace) == len(ref_trace) > 20
    assert all(torch.equal(a, b) for a, b in zip(ref_trace, f.trace))
