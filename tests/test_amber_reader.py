"""The AMBER prmtop / NAMD coordinate readers (SURVEY.md section 8f-2) against the reference's STORED
known answers for its tests/data/prod_alanine_dipeptide_amber, through the CPU oracle.  The input files
are the reference's, copied into tests/golden/data/ (copy_reference_data.py); the GPU parity tests use
the parsed parameters committed in tests/golden/ala2_*.npz."""
import os

import numpy as np
import torch

from conftest import GOLDEN, load_golden
from oracle import refmd

ALA = os.path.join(GOLDEN, "data", "prod_alanine_dipeptide_amber")
TERMS = ["bonds", "angles", "dihedrals", "impropers", "1-4", "electrostatics", "lj"]


def energies(box, **cfg):
    from torchmd_b200 import amber

    sysm = amber.AmberSystem(os.path.join(ALA, "structure.prmtop"))
    xyz = amber.read_bincoor(os.path.join(ALA, "input.coor"))
    par = amber.amber_parameters(sysm, precision=torch.float64)
    of = refmd.OracleForces(par, TERMS, **cfg)
    pos = torch.tensor(xyz, dtype=torch.float64)[None]
    b = torch.zeros(1, 3, 3, dtype=torch.float64)
    for k in range(3):
        b[0, k, k] = float(box[k])
    return of.compute(pos, b, torch.zeros_like(pos))[0]


def test_topology_counts():
    from torchmd_b200 import amber

    s = amber.AmberSystem(os.path.join(ALA, "structure.prmtop"))
    assert s.natoms == 688 and s.ifbox == 1
    assert len(s.bonds) == 687 and len(s.angles) == 36 and len(s.impropers) == 4
    assert abs(float(s.charge.sum())) < 1e-3
    assert amber.read_bincoor(os.path.join(ALA, "input.coor")).shape == (688, 3)
    np.testing.assert_allclose(amber.read_xsc(os.path.join(ALA, "input.xsc")), [19.83881, 19.6193, 19.6342], rtol=1e-6)


def test_stored_energy_of_test_replicas():
    """tests/test_torchmd.py:517 -- cutoff 9, switch 7.5, reaction field, no box: -1722.3569.
    (The stored digits were produced with an older CODATA set in scipy.constants: 2e-4 drift.)"""
    e = energies(np.zeros(3), cutoff=9, switch_dist=7.5, rfa=True)
    assert abs(sum(e.values()) + 1722.3569) < 5e-4


def test_stored_energy_of_test_vmap():
    """tests/test_torchmd.py:605 -- no cutoff, no reaction field: -1768.8915."""
    e = energies(np.zeros(3), cutoff=None, switch_dist=7.5, rfa=False)
    assert abs(sum(e.values()) + 1768.8915) < 5e-4


def test_stored_energy_vector_of_the_tutorial():
    """examples/tutorial.ipynb:105 -- fp32 GPU run with the .xsc box, per term."""
    from torchmd_b200 import amber

    e = energies(amber.read_xsc(os.path.join(ALA, "input.xsc")), cutoff=9, switch_dist=7.5, rfa=True)
    want = dict(electrostatics=-2568.498, lj=359.251, bonds=3.9577, angles=2.8446, dihedrals=10.5799, impropers=1.2417)
    for k, v in want.items():
        assert abs(e[k] - v) < 2e-3, (k, e[k], v)
    assert e["1-4"] == 0.0  # 1-4 energies are booked under lj / electrostatics (forces.py:185-236)
    assert abs(sum(e.values()) + 2190.623) < 2e-3


def test_committed_parameters_match_a_fresh_parse():
    from torchmd_b200 import amber

    g = load_golden("ala2_xsc_rf")
    par = amber.amber_parameters(amber.AmberSystem(os.path.join(ALA, "structure.prmtop")), TERMS)
    assert np.array_equal(par.mapped_atom_types.numpy(), g["par_types"])
    np.testing.assert_allclose(par.charges.numpy(), g["par_charges"], rtol=1e-6)
    for name in ("bond", "angle", "dihedral", "improper", "nonbonded_14"):
        t = getattr(par, name + "_params")
        assert np.array_equal(t["idx"].numpy(), g[f"par_{name}_idx"])
        assert np.array_equal(t["map"].numpy(), g[f"par_{name}_map"])
        np.testing.assert_allclose(t["params"].numpy(), g[f"par_{name}_params"], rtol=1e-6)
