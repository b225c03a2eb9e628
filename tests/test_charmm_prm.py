"""CHARMM .prm reader (torchmd_b200/charmm.py CharmmPrmForceField) and the parameter tables built from it, against the
UNMODIFIED reference's Parameters on the reference's own small CHARMM fixtures.  The goldens (tests/golden/charmm_*.npz,
make_golden_charmm.py) hold the reference's tables and its Forces.compute results; the reader tests parse the reference's
input files, copied into tests/golden/data/ (copy_reference_data.py: the large parameters.prm files keep only the entries
of each fixture's own atom types)."""
import glob
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, golden_cfg, golden_system_tensors, load_golden, params_from_golden
from oracle import refmd

DATA = os.path.join(GOLDEN, "data")
CASES = ["1water", "2ions", "3ions", "1dihedral", "singledihedral", "4dihedrals", "benzamidine", "2watersperiodic", "sodiumperiodic", "waterbox"]


def files(name):
    folder = os.path.join(DATA, name)
    return tuple(glob.glob(os.path.join(folder, e))[0] for e in ("*.psf", "*.pdb", "*.prm"))


@pytest.mark.parametrize("name", CASES)
def test_tables_from_the_prm_reader_equal_the_reference_parameters(name):
    """yaml_parameters(mol, CharmmPrmForceField) -- the package's own table builder -- reproduces what the reference's
    Parameters class made of the same force-field object (stored in the golden file), array by array."""
    from torchmd_b200 import charmm
    from torchmd_b200.ff_yaml import yaml_parameters

    g = load_golden("charmm_" + name)
    psf, pdb, prm = files(name)
    mol = charmm.load_molecule(psf, pdb)
    par = yaml_parameters(mol, charmm.CharmmPrmForceField(prm, mol), terms=[str(t) for t in g["terms"]], precision=torch.float64)
    ref = params_from_golden(g, precision=torch.float64)
    assert np.array_equal(par.mapped_atom_types.numpy(), ref.mapped_atom_types.numpy())
    for attr in ("charges", "masses"):
        assert torch.equal(getattr(par, attr), getattr(ref, attr)), attr
    assert torch.equal(par.nonbonded_params["params"], ref.nonbonded_params["params"])  # sigma, epsilon per type
    for attr in ("bond_params", "angle_params", "dihedral_params", "improper_params", "nonbonded_14_params"):
        a, b = getattr(par, attr), getattr(ref, attr)
        assert (a is None) == (b is None), attr
        if a is not None:
            for key in ("idx", "map", "params"):
                assert torch.equal(a[key], b[key]), (attr, key)


def test_tip3p_in_the_prm_file_is_the_tip3p_of_the_reference_yaml():
    """The one cross-check the reference's own files offer: its CHARMM water parameters and its YAML water force field
    (tests/water) describe the same model."""
    from torchmd_b200 import charmm
    from torchmd_b200.ff_yaml import YamlForceField

    ff = charmm.CharmmPrmForceField(files("1water")[2])
    y = YamlForceField(os.path.join(DATA, "water", "water_forcefield.yaml"))
    assert ff.get_bond("OT", "HT") == tuple(y.get_bond("OT", "HT")) == ff.get_bond("HT", "OT")
    ka, ta = ff.get_angle("HT", "OT", "HT")
    ky, ty = y.get_angle("HT", "OT", "HT")
    assert ka == ky and abs(ta - ty) < 1e-12
    for t in ("OT", "HT"):
        (s1, e1), (s2, e2) = ff.get_LJ(t), y.get_LJ(t)
        # (the YAML keeps CHARMM's negative sign; every use is sqrt(eps_i * eps_j), which does not see it)
        assert abs(s1 - s2) < 1e-12 and abs(e1 - abs(e2)) < 1e-12, (t, s1, s2, e1, e2)


@pytest.mark.parametrize("name", CASES)
@pytest.mark.parametrize("tag,dtype", [("f32", torch.float32), ("f64", torch.float64)])
def test_oracle_on_the_charmm_fixtures(name, tag, dtype):
    g = load_golden("charmm_" + name)
    par = params_from_golden(g, precision=dtype)
    of = refmd.OracleForces(par, [str(t) for t in g["terms"]], **golden_cfg(g))
    pos, box = golden_system_tensors(g, dtype)
    F = torch.zeros_like(pos)
    E = of.compute(pos, box, F)
    assert np.array_equal(F.numpy(), g[f"forces_{tag}"])
    for r in range(len(E)):
        for c, k in enumerate(g["energy_keys"]):
            assert E[r][str(k)] == g[f"energies_{tag}"][r, c]
