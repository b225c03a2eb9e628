"""Known answers of the UNMODIFIED REFERENCE's integrator (torchmd/integrator.py) and conjugate-gradient minimiser
(torchmd/minimizers.py), on the scenarios of the reference's tests/test_integrator.py and on an anharmonic bowl.

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden_known_answers.py

Build container only (needs the reference checkout at /root/reference).  Writes

  integrator_known_answers.npz -- per case <c>: the inputs (c/masses, c/vel, c/pos, c/forces, c/batch, c/timestep,
      c/pot, c/precompute, c/niters) and what the reference returned after each step(niter) call k
      (c/ekin_k, c/temp_k, c/pot_k, c/pos_k, c/vel_k, c/natoms); kinetic_energy cases ke<i>/masses, ke<i>/vel, ke<i>/batch
      and ke<i>/out; init/dt and init/gamma of Integrator(timestep=0.001, gamma=1, T=300).
  minimizer_cg_trace.npz -- start positions, every point minimize_cg(steps=4) evaluated, and its return value.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True
sys.path.insert(0, "/root/reference")

from torchmd import minimizers as ref_min  # noqa: E402  (reference)
from torchmd.integrator import Integrator, kinetic_energy  # noqa: E402
from torchmd.systems import System  # noqa: E402

f32 = np.float32

# kinetic_energy(masses (N,1), vel (R,N,3), batch) cases; batch None = per replica
KE_CASES = [
    ([1.0, 2.0, 3.0], [[[1.0, 2.0, 3.0], [0.5, 1.0, 1.5], [2.0, 1.0, 0.5]]], None),
    ([1.0, 2.0], [[[1.0, 0.0, 0.0], [0.0, 1.0, 0.0]], [[2.0, 0.0, 0.0], [0.0, 2.0, 0.0]]], None),
    ([1.0, 2.0], np.zeros((1, 2, 3)), None),
    ([1.0, 2.0, 1.5], [[[1.0, 0.0, 0.0], [0.0, 1.0, 0.0], [2.0, 0.0, 0.0]], [[0.5, 0.0, 0.0], [0.0, 1.5, 0.0], [1.0, 0.0, 0.0]]], [0, 0, 1]),
    ([1.0, 2.0], [[[1.0, 0.0, 0.0], [0.0, 1.0, 0.0]]], [0, 2]),
    ([1.0, 2.0, 3.0], [[[1.0, 0.0, 0.0], [0.0, 2.0, 0.0], [0.0, 0.0, 3.0]]], [0, 1, 2]),
]

# velocity Verlet without thermostat under constant forces: (masses, pos, vel, forces, batch, timestep ps, pot,
# forces evaluated before the first step, step(niter) calls)
MD_CASES = {
    "mock": ([1.0, 2.0], np.zeros((1, 2, 3)), [[[1.0, 0.0, 0.0], [0.0, 1.0, 0.0]]], [[[0.1, 0.2, 0.3], [0.4, 0.5, 0.6]]],
             None, 0.001, 1.5, False, [1, 3]),
    "batches": ([1.0, 2.0, 1.5], np.zeros((1, 3, 3)), [[[1.0, 0.0, 0.0], [0.0, 2.0, 0.0], [0.0, 0.0, 3.0]]],
                [[[10.0, 0.0, 0.0], [0.0, 20.0, 0.0], [0.0, 0.0, 30.0]]], [0, 0, 1], 0.001, 2.5, False, [1]),
    "two_atoms": ([1.0, 2.0], [[[0.0, 0.0, 0.0], [1.0, 1.0, 1.0]]], [[[0.1, 0.2, 0.3], [0.1, 0.2, 0.3]]],
                  [[[1.0, 2.0, 3.0], [-0.5, 1.5, -2.5]]], None, 0.002, 0.0, True, [1]),
    "two_replicas": ([1.0, 2.0], [[[0.0, 0.0, 0.0], [1.0, 1.0, 1.0]]] * 2, [[[0.1, 0.2, 0.3], [0.1, 0.2, 0.3]]] * 2,
                     [[[1.0, 2.0, 3.0], [-0.5, 1.5, -2.5]], [[0.5, 1.0, 1.5], [-1.0, 2.0, -3.0]]], None, 0.002, 0.0, True, [1]),
}


class ConstantForces:
    def __init__(self, forces, pot):
        self.f, self.pot = forces, pot

    def compute(self, pos, box, forces):
        forces.copy_(self.f)
        return self.pot


class Quartic:
    def __init__(self):
        self.trace = []

    def compute(self, pos, box, forces):
        p = pos.detach()
        self.trace.append(p.clone())
        forces.copy_(-(4 * p**3 - 6 * p + 0.5))
        return [float((p**4 - 3 * p**2 + 0.5 * p).sum())]


def integrator_cases():
    out = {}
    for i, (m, v, b) in enumerate(KE_CASES):
        masses = torch.tensor(m, dtype=torch.float32)[:, None]
        vel = torch.tensor(np.asarray(v, f32))
        batch = None if b is None else torch.tensor(b, dtype=torch.long)
        out[f"ke{i}/masses"], out[f"ke{i}/vel"] = masses.numpy(), vel.numpy()
        if batch is not None:
            out[f"ke{i}/batch"] = batch.numpy()
        out[f"ke{i}/out"] = kinetic_energy(masses, vel, batch=batch).numpy()
    for c, (m, p, v, f, b, ts, pot, pre, niters) in MD_CASES.items():
        pos, vel, frc = (torch.tensor(np.asarray(x, f32)) for x in (p, v, f))
        system = System(pos.shape[1], pos.shape[0], torch.float32, "cpu")
        system.pos.copy_(pos)
        system.vel.copy_(vel)
        system.set_masses(torch.tensor(m, dtype=torch.float32))
        forces = ConstantForces(frc, pot)
        if pre:
            forces.compute(system.pos, system.box, system.forces)
        batch = None if b is None else torch.tensor(b, dtype=torch.long)
        integ = Integrator(system, forces, ts, "cpu", batch=batch)
        rec = {"masses": np.asarray(m, f32), "pos": pos.numpy(), "vel": vel.numpy(), "forces": frc.numpy(),
               "timestep": np.float64(ts), "pot": np.float64(pot), "precompute": np.bool_(pre), "niters": np.asarray(niters),
               "natoms": np.asarray(integ.natoms)}
        if batch is not None:
            rec["batch"] = batch.numpy()
        for k, n in enumerate(niters):
            ekin, epot, temp = integ.step(niter=n)
            rec.update({f"ekin_{k}": np.asarray(ekin), f"temp_{k}": np.asarray(temp), f"pot_{k}": np.float64(epot),
                        f"pos_{k}": system.pos.numpy().copy(), f"vel_{k}": system.vel.numpy().copy()})
        out.update({f"{c}/{k}": val for k, val in rec.items()})
    system = System(2, 1, torch.float32, "cpu")
    system.set_masses(torch.tensor([1.0, 2.0]))
    integ = Integrator(system, ConstantForces(torch.zeros(1, 2, 3), 0.0), 0.001, "cpu", gamma=1.0, T=300.0)
    out["init/dt"], out["init/gamma"] = np.float64(integ.dt), np.float64(integ.gamma)
    return out


def minimizer_trace():
    g = torch.Generator().manual_seed(3)
    x0 = torch.zeros(1, 6, 3)
    start = x0 + 1.5 * torch.randn(x0.shape, generator=g)
    import types

    s = types.SimpleNamespace(pos=start.clone(), box=torch.zeros(1, 3, 3), forces=torch.zeros(1, 6, 3), nreplicas=1, natoms=6)
    f = Quartic()
    ret = ref_min.minimize_cg(s, f, steps=4)
    return {"start": start.numpy(), "trace": torch.cat(f.trace).numpy(), "returned": np.asarray(ret)}


def main():
    for name, data in (("integrator_known_answers", integrator_cases()), ("minimizer_cg_trace", minimizer_trace())):
        path = os.path.join(HERE, name + ".npz")
        np.savez_compressed(path, **data)
        print(f"wrote {name}.npz {os.path.getsize(path) / 1024:.1f} KiB")


if __name__ == "__main__":
    main()
