"""Copy the reference's input fixtures that the reader tests parse into tests/golden/data/.

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/copy_reference_data.py

Build container only (needs the reference checkout at /root/reference).  Copies, per directory of the reference's
tests/: the AMBER alanine-dipeptide topology and coordinates (data/prod_alanine_dipeptide_amber), the tests/water PSF,
PDB and YAML force field (water), and the PSF / PDB / PRM of each CHARMM fixture (data/<case>).  Files are copied
byte for byte except the 778 kB CHARMM parameter files (parameters.prm), which keep only the lines a fixture's own
atom types can look up: section headers, keyword lines, and MASS / BONDS / ANGLES / DIHEDRALS / IMPROPER / NONBONDED
entries whose type names are all among the fixture's types.  The reader does exact type look-ups (no wildcards), so
the shrunk file gives the same tables; the script asserts that for every type tuple of the fixture.
"""
import glob
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
REF = "/root/reference/tests"
sys.dont_write_bytecode = True
sys.path.insert(0, REPO)

from torchmd_b200 import charmm  # noqa: E402

CHARMM_CASES = ["1water", "2ions", "3ions", "1dihedral", "singledihedral", "4dihedrals", "benzamidine", "2watersperiodic", "sodiumperiodic", "waterbox"]
WIDTH = {"BONDS": 2, "ANGLES": 3, "DIHEDRALS": 4, "IMPROPER": 4, "NONBONDED": 1}


def shrink_prm(src, dst, types):
    keep, section, carry = [], None, False
    alias = {"THETAS": "ANGLES", "PHI": "DIHEDRALS", "IMPROPERS": "IMPROPER", "IMPHI": "IMPROPER", "NBONDED": "NONBONDED"}
    for raw in open(src):
        line = raw.split("!")[0].strip()
        if not line or line.startswith("*"):
            continue
        w = line.split()
        head = w[0].upper()
        if carry or line.endswith("-"):  # a continued line (the NONBONDED header) is kept whole
            keep.append(raw)
        elif head in charmm.CharmmPrmForceField.SECTIONS:
            section = alias.get(head, head)
            keep.append(raw)
        elif head == "MASS":
            if len(w) >= 4 and w[2].upper() in types:
                keep.append(raw)
        elif section in WIDTH and all(t.upper() in types for t in w[: WIDTH[section]]):
            keep.append(raw)
        carry = line.endswith("-")
    with open(dst, "w") as fh:
        fh.writelines(keep)


def main():
    out = os.path.join(HERE, "data")
    shutil.rmtree(out, ignore_errors=True)
    d = os.path.join(out, "prod_alanine_dipeptide_amber")
    os.makedirs(d)
    for f in ("structure.prmtop", "input.coor", "input.xsc"):
        shutil.copyfile(os.path.join(REF, "data", "prod_alanine_dipeptide_amber", f), os.path.join(d, f))
    d = os.path.join(out, "water")
    os.makedirs(d)
    for f in ("structure.psf", "structure.pdb", "water_forcefield.yaml"):
        shutil.copyfile(os.path.join(REF, "water", f), os.path.join(d, f))
    for case in CHARMM_CASES:
        src, d = os.path.join(REF, "data", case), os.path.join(out, case)
        os.makedirs(d)
        (psf,), (pdb,), (prm,) = (glob.glob(os.path.join(src, "*." + ext)) for ext in ("psf", "pdb", "prm"))
        for f in (psf, pdb):
            shutil.copyfile(f, os.path.join(d, os.path.basename(f)))
        mol = charmm.load_molecule(psf, pdb)
        target = os.path.join(d, os.path.basename(prm))
        if os.path.getsize(prm) < 100_000:
            shutil.copyfile(prm, target)
            continue
        types = {str(t).upper() for t in mol.atomtype}
        shrink_prm(prm, target, types)
        full, small = charmm.CharmmPrmForceField(prm, mol), charmm.CharmmPrmForceField(target, mol)
        for attr in ("bonds", "angles", "dihedrals", "impropers", "lj", "masses"):
            a, b = getattr(full, attr), getattr(small, attr)
            want = {k: v for k, v in a.items() if all(t in types for t in (k if isinstance(k, tuple) else (k,)))}
            assert want == b, (case, attr)
        print(f"{case}: parameters.prm {os.path.getsize(prm)} -> {os.path.getsize(target)} bytes, types {sorted(types)}")
    total = sum(os.path.getsize(os.path.join(r, f)) for r, _, fs in os.walk(out) for f in fs)
    print(f"tests/golden/data: {total / 1024:.0f} KiB")


if __name__ == "__main__":
    main()
