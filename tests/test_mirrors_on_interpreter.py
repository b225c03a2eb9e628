"""The `-m gpu` tests themselves, run on the CPU: the Python mirrors (Forces, Integrator, Wrapper, the autograd
path) drive the C ABI of the host SIMT-interpreter build of the library (tests/simt) with CPU tensors.

The product refuses that build (torchmd_b200/_lib.py) and refuses CPU tensors; here, and only here, the loaded
handle, the "is on the device" predicate and torch's stream query are patched so that the *same test functions*
that run on the B200 execute every line of the host classes and of the C entry points without a GPU.  It checks
plumbing and logic (argument marshalling, return formats, rebuild protocol, error paths) -- what the B200 run adds
is the device arithmetic and speed.  The slow cases stay with the GPU suite.
"""
import os

import numpy as np
import pytest
import torch

import test_simt_kernels as T


class _Stream:
    cuda_stream = None  # the interpreter runs every launch on the spot


def _install(monkeypatch, tag):
    from torchmd_b200 import _lib

    handle = T.load(T.build_simt(tag, T.VARIANTS[tag]))
    monkeypatch.setattr(_lib, "_lib", handle)
    monkeypatch.setattr(_lib, "on_device", lambda t: True)
    monkeypatch.setattr(torch.cuda, "current_stream", lambda *a, **k: _Stream())
    monkeypatch.setattr(torch.cuda, "current_device", lambda: 0)
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a, **k: None)
    import test_autograd_path, test_gpu_forces, test_gpu_integrator, test_wrapper

    for mod in (test_autograd_path, test_gpu_forces, test_gpu_integrator, test_wrapper):
        monkeypatch.setattr(mod, "DEV", "cpu")
    return handle


@pytest.fixture
def hostsim(monkeypatch):
    return _install(monkeypatch, "")


@pytest.fixture
def hostsim_r2(monkeypatch):
    """The build with every opt-in path compiled in as the default (packed fixed-point pair kernel, culled two-atom
    list build, overlapped bonded kernel, fused integrate+prepare and bonded fold)."""
    return _install(monkeypatch, "_r2")


FORCE_CASES = ["water291_rf_switch", "water291_plain", "argon100_nocut", "chain_amber_vacuum", "chain_amber_periodic",
               "chain_charmm_periodic", "ala2_xsc_rf", "benzamidine_amber_nocut", "ligand_amber_nocut"]
FORCE_CASES += ["charmm_" + n for n in ("1water", "2ions", "3ions", "1dihedral", "singledihedral", "4dihedrals", "benzamidine", "2watersperiodic", "sodiumperiodic", "waterbox")]


@pytest.mark.parametrize("name", FORCE_CASES)
def test_forces_compute_against_the_goldens(hostsim, name):
    import test_gpu_forces as G

    G.test_golden_forces_energies(name)
    if name != "water291_plain":
        G.test_golden_neighbour_pairs_bit_exact(name)


def test_forces_api_formats_errors_replicas_and_skin(hostsim):
    import test_gpu_forces as G

    G.test_api_errors_and_formats()
    G.test_forces_deterministic_and_replicas_identical()
    G.test_results_do_not_depend_on_skin(0.3)
    G.test_molecules_several_boxes_away_meet_the_plain_yardstick()  # (gated on the GPU until its first B200 run)


def test_box_upload_and_overflow_checks_on_every_path(hostsim):
    import test_gpu_forces as G

    G.test_a_fresh_box_tensor_per_call_is_always_taken()
    G.test_dense_cluster_in_a_large_box_without_the_numpy_outputs()


def test_repulsion_terms(hostsim):
    import test_gpu_zz_more_terms as M

    M.test_repulsion_terms("argon100_lj_rep_mix")


def test_integrator_step(hostsim):
    import test_gpu_integrator as I

    I.test_initialization_attributes()
    I.test_velocity_verlet_constant_force_known_answer(2)
    I.test_batch_kinetic_energy()
    I.test_nve_trajectory_matches_reference()
    I.test_langevin_with_injected_noise_matches_reference()
    I.test_stepwise_and_fused_paths_agree()


@pytest.mark.parametrize("name", ["water", "mixed", "nobonds", "zerobox"])
def test_wrapper_wrap(hostsim, name):
    import test_wrapper as W

    getattr(W.test_gpu_wrap_matches_reference_golden, "__wrapped__", W.test_gpu_wrap_matches_reference_golden)(name)


def test_wrapper_wrap_random_topologies(hostsim):
    import test_wrapper as W

    W.test_gpu_wrap_random_topologies()


def test_autograd_path(hostsim):
    import test_autograd_path as A

    A.test_gpu_autograd_mode_returns_the_reference_autograd_forces()
    A.test_gpu_energy_backward_and_vmap()


def test_minimizers_over_the_kernels(hostsim, capsys):
    """minimize_pytorch_bfgs (the autograd path: Epot.sum().backward() through the kernel pass) and minimize_cg
    (plain compute calls) on the water fixture: both lower the potential energy and leave finite coordinates."""
    from conftest import golden_cfg, load_golden, params_from_golden
    from torchmd_b200 import Forces, System
    from torchmd_b200.minimizers import minimize_cg, minimize_pytorch_bfgs

    g = load_golden("water291_rf_switch")
    terms = [str(x) for x in g["terms"]]
    n = len(g["coords"])

    def fresh():
        system = System(n, 1, torch.float32, "cpu")
        system.pos[:] = torch.tensor(np.asarray(g["coords"], np.float32))[None]
        system.box[0] = torch.diag(torch.tensor(np.asarray(g["box"], np.float32).reshape(-1)[:3]))
        forces = Forces(params_from_golden(g, device="cpu"), terms=terms, **golden_cfg(g))
        e0 = forces.compute(system.pos, system.box, system.forces)[0]
        return system, forces, e0

    system, forces, e0 = fresh()
    minimize_pytorch_bfgs(system, forces, steps=2, max_iter=4)
    e1 = forces.compute(system.pos, system.box, system.forces)[0]
    assert e1 < e0 - 1.0 and bool(torch.isfinite(system.pos).all()), (e0, e1)
    assert capsys.readouterr().out.splitlines()[0].split() == ["Iter", "Epot", "fmax"]

    system, forces, e0 = fresh()
    minimize_cg(system, forces, steps=3, update_system=True)
    e2 = forces.compute(system.pos, system.box, system.forces)[0]
    assert e2 < e0 - 1.0 and bool(torch.isfinite(system.pos).all()), (e0, e2)


def test_smoke_entry_point(hostsim, capsys):
    """__graft_entry__.smoke(), the function the driver runs on the B200 before the bench."""
    import __graft_entry__ as g

    g.smoke(dev="cpu")
    assert "neighbour pairs bit-exact" in capsys.readouterr().out


# ---- the gated tests (TMD_B200_VALIDATE=1 on a B200) of the opt-in kernels, as written, on the interpreter ----
@pytest.mark.parametrize("mode", [1, 2])
def test_gated_fixed_point_tests_run_as_written(hostsim, monkeypatch, mode):
    import test_gpu_zzz_fixedpoint as X

    monkeypatch.setattr(X, "DEV", "cpu")
    X.test_fixed_point_kernel_matches_golden("chain_amber_periodic", mode)
    X.test_fixed_point_kernel_matches_golden("water999_eq", mode)
    if mode == 2:
        X.test_packed_kernel_without_a_box("chain_amber_vacuum")
        X.test_fixed_point_kernel_is_accurate_for_drifted_molecules()
    # (test_fixed_point_trajectory_tracks_float_kernel and the 3000-atom box stay with the B200: hundreds of steps)


def test_gated_peer_to_peer_test_runs_as_written(hostsim, monkeypatch):
    """DecomposedIntegrator(exchange="p2p") with one rank: IPC set-up, double-buffered positions, push kernel, flag
    wait -- bitwise equal to Integrator.step (smaller system than on the B200, gloo instead of NCCL)."""
    import torch.distributed as dist

    import test_gpu_zzz_p2p as P

    monkeypatch.setattr(P, "DEV", "cpu")
    monkeypatch.setattr(P, "SIZE", dict(waters=64, cutoff=5.0, switch=4.0, skin=0.3, steps=(1, 2, 7), backend="gloo"))
    monkeypatch.setenv("MASTER_PORT", str(T_free_port()))
    try:
        P.test_p2p_world1_matches_integrator_bitwise(False)
        _fake_torch_graphs(monkeypatch, hostsim)
        launched = _graph_counters(hostsim)[0]
        P.test_p2p_world1_matches_integrator_bitwise(True)  # one captured step per (energy outputs, buffer parity)
        assert _graph_counters(hostsim)[0] - launched >= sum(P.SIZE["steps"]) + 3  # the steps really were replays
    finally:
        if dist.is_initialized():
            dist.destroy_process_group()


def _graph_counters(handle):
    import ctypes as C

    out = (C.c_longlong * 3)()
    handle.simt_graph_counters(out)
    return list(out)


def _fake_torch_graphs(monkeypatch, handle):
    """torch.cuda.CUDAGraph / torch.cuda.graph on the interpreter's record-and-replay capture (tests/simt/stub): what
    the library enqueues inside the `with` block is recorded on the null stream and `replay()` runs it again.  (A
    collective issued inside the block runs at capture time only -- fine for one rank, where it is the identity.)"""
    import ctypes as C

    handle.simt_capture_end.restype = C.c_void_p
    handle.simt_capture_begin.argtypes = handle.simt_capture_end.argtypes = handle.simt_graph_replay.argtypes = [C.c_void_p]

    class Graph:
        g = None

        def replay(self):
            assert handle.simt_graph_replay(self.g) == 0

    class Capture:
        def __init__(self, graph, **kw):
            assert kw.get("capture_error_mode", "global") in ("global", "relaxed", "thread_local")
            self.graph = graph

        def __enter__(self):
            assert handle.simt_capture_begin(None) == 0

        def __exit__(self, *exc):
            self.graph.g = handle.simt_capture_end(None)
            return False

    monkeypatch.setattr(torch.cuda, "CUDAGraph", Graph)
    monkeypatch.setattr(torch.cuda, "graph", Capture)


def T_free_port():
    import socket

    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_multi_rank_check_script_runs_with_one_rank(hostsim, monkeypatch, capsys):
    """scripts/p2p_check.py (the round-2 multi-GPU check of the peer-to-peer exchange against the all-gather path)
    executed with a single rank: its own logic is sound before box time is spent on it."""
    import importlib.util
    import os

    import torch.distributed as dist

    spec = importlib.util.spec_from_file_location("p2p_check", os.path.join(T.ROOT, "scripts", "p2p_check.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    for k, v in dict(RANK="0", WORLD_SIZE="1", LOCAL_RANK="0", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(T_free_port())).items():
        monkeypatch.setenv(k, v)
    try:
        with pytest.raises(SystemExit) as done:
            mod.main(dev="cpu", waters=64, cutoff=5.0, switch=4.0, skin=0.3, steps=(1, 2, 7), graphs=(False,))
    finally:
        if dist.is_initialized():
            dist.destroy_process_group()
    assert done.value.code == 0 and "P2P_CHECK PASS" in capsys.readouterr().out


def _bench_on_the_interpreter(monkeypatch):
    """bench.py's single-GPU arm on the host interpreter build: host events and buffers, no clock sampler, 64 waters."""
    import bench

    class _Event:
        def __init__(self, enable_timing=False):
            self.t = 0.0

        def record(self, *a):
            import time

            self.t = time.perf_counter()

        def elapsed_time(self, other):
            return (other.t - self.t) * 1e3

    real_empty = torch.empty

    def empty(*a, **k):
        k.pop("pin_memory", None)
        return real_empty(*a, **k)

    class _NoSampler:
        def __init__(self, *a):
            pass

        def stop(self):
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}

    monkeypatch.setattr(torch.cuda, "Event", _Event)
    monkeypatch.setattr(torch, "empty", empty)
    monkeypatch.setattr(bench, "ClockSampler", _NoSampler)
    monkeypatch.setattr(bench, "N_WATERS", 64)
    monkeypatch.setattr(bench, "CFG", dict(bench.CFG, cutoff=5.0, switch_dist=4.0))
    monkeypatch.delenv("WORLD_SIZE", raising=False)
    monkeypatch.setattr(bench, "DEVICE_OVERRIDE", "cpu")
    return bench


def test_bench_single_gpu_arm_dry_run(hostsim, monkeypatch, capsys):
    """bench.py's own single-GPU body on a 64-water box: every library call, the profiling hooks, the host-buffer
    entry and the JSON line's keys -- a bench that dies on a typo at round end has no number at all."""
    import argparse
    import json

    bench = _bench_on_the_interpreter(monkeypatch)
    args = argparse.Namespace(gpus=1, steps=6, warmup=3, equil=100, e2e_steps=3, no_cpu_baseline=True, impl="ours", workload="water100k",
                              dump_outputs=None)
    bench.gpu_arm(args)
    line = json.loads([l for l in capsys.readouterr().out.splitlines() if l.startswith("{")][-1])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline", "cpu_baseline"):
        assert key in line, key
    assert line["gpu_launches"] > 0 and line["value"] > 0 and line["e2e"]["value"] > 0
    assert line["roofline"]["pairs_in_cutoff"] > 0 and line["roofline"]["launches_sampled"] > 0
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(line["roofline"])
    # the reference's own small test systems as workloads (BASELINE configs 2 and 3), two replicas included
    for wl in ("water291", "ala2"):
        args = argparse.Namespace(gpus=1, steps=4, warmup=3, equil=0, e2e_steps=2, no_cpu_baseline=True, impl="ours", workload=wl,
                                  dump_outputs=None)
        bench.gpu_arm(args)
        line = json.loads([l for l in capsys.readouterr().out.splitlines() if l.startswith("{")][-1])
        assert line["value"] > 0 and line["metric"] == bench.METRICS[wl] and line["state"]["replicas"] == (2 if wl == "water291" else 1)


def test_bench_dump_outputs_are_reproducible(hostsim, monkeypatch, capsys, tmp_path):
    """--dump-outputs: the same arguments write the same outputs twice, and --steps sets the number of timed steps."""
    import argparse
    import json

    bench = _bench_on_the_interpreter(monkeypatch)
    dumps = []
    for run, steps in enumerate((4, 4, 5)):
        out = tmp_path / str(run)
        args = argparse.Namespace(gpus=1, steps=steps, warmup=3, equil=0, e2e_steps=2, no_cpu_baseline=True, impl="ours", workload="water100k",
                                  dump_outputs=str(out))
        bench.gpu_arm(args)
        assert json.loads([l for l in capsys.readouterr().out.splitlines() if l.startswith("{")][-1])["steps"] == steps
        dumps.append({p.stem: np.load(p) for p in sorted(out.glob("*.npy"))})
    assert set(dumps[0]) == {"positions", "velocities", "forces", "kinetic_energy", "potential_energy", "temperature"}
    assert dumps[0]["positions"].shape == (1, 192, 3) and dumps[0]["positions"].dtype == np.float32
    assert dumps[0]["potential_energy"].shape == (1,) and dumps[0]["potential_energy"].dtype == np.float64
    assert all(np.array_equal(dumps[0][k], dumps[1][k]) for k in dumps[0])
    assert not np.array_equal(dumps[0]["positions"], dumps[2]["positions"])  # one more timed step, a different state


def test_bench_reference_arm_reports_what_it_measured(monkeypatch, capsys):
    """--impl reference: `value` is the steps/s measured at the size that ran, `config.natoms` says that size, the O(N^2)
    extrapolation to 99,999 atoms sits in its own labelled field."""
    import argparse
    import json

    import bench

    monkeypatch.setattr(bench, "_probe_threads", lambda: (2, 2))
    args = argparse.Namespace(gpus=1, steps=1, warmup=0, impl="reference", workload="water100k")
    bench.reference_arm(args)
    line = json.loads([l for l in capsys.readouterr().out.splitlines() if l.startswith("{")][-1])
    n = line["cpu_baseline"]["measured_natoms"]
    assert line["config"]["natoms"] == n < 99999 and line["impl"] == "reference"
    assert abs(line["value"] - 1e3 / line["cpu_baseline"]["ms_per_step_measured"]) < 1e-6 * line["value"]
    assert line["cpu_baseline"]["extrapolated_99999_atoms_steps_per_s"] < line["value"]
    args = argparse.Namespace(gpus=1, steps=1, warmup=0, impl="reference", workload="ala2")
    bench.reference_arm(args)
    line = json.loads([l for l in capsys.readouterr().out.splitlines() if l.startswith("{")][-1])
    assert line["config"]["natoms"] == 688 and "extrapolated_99999_atoms_steps_per_s" not in line["cpu_baseline"]


def test_round2_default_configuration_passes_the_gpu_tests(hostsim_r2, capsys):
    """The same GPU test functions with every opt-in path switched on by default: what `pytest -m gpu`, smoke() and the
    integrator will see once round 2 flips the defaults."""
    import __graft_entry__ as g
    import test_gpu_forces as G
    import test_gpu_integrator as I

    for name in ("water291_rf_switch", "chain_amber_periodic", "chain_charmm_periodic", "ala2_xsc_rf", "argon100_nocut"):
        G.test_golden_forces_energies(name)
        G.test_golden_neighbour_pairs_bit_exact(name)
    from conftest import load_golden

    f, *_ = G.run_gpu(load_golden("chain_amber_periodic"))
    assert hostsim_r2.tmd_pair_kernel(f._ctx) == 2  # the packed fixed-point kernel is what ran
    G.test_api_errors_and_formats()
    I.test_nve_trajectory_matches_reference()
    I.test_langevin_with_injected_noise_matches_reference()
    I.test_stepwise_and_fused_paths_agree()
    g.smoke(dev="cpu")


def test_ab_bench_script_dry_run(hostsim, monkeypatch, capsys):
    """scripts/ab_bench.py (round-2 tuning sweeps in one process) on a 64-water box."""
    import importlib.util
    import os
    import time

    import bench

    class _Event:
        def __init__(self, enable_timing=False):
            self.t = 0.0

        def record(self, *a):
            self.t = time.perf_counter()

        def elapsed_time(self, other):
            return (other.t - self.t) * 1e3

    spec = importlib.util.spec_from_file_location("ab_bench", os.path.join(T.ROOT, "scripts", "ab_bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    monkeypatch.setattr(torch.cuda, "Event", _Event)
    monkeypatch.setattr(mod, "DEVICE", "cpu")
    monkeypatch.setattr(bench, "N_WATERS", 64)
    monkeypatch.setattr(bench, "CFG", dict(bench.CFG, cutoff=5.0, switch_dist=4.0))
    mod.main(["default|TMD_B200_FX=0,TMD_B200_OVERLAP=0,TMD_B200_FUSEPREP=0,SKIN=0.3", "packed+overlap+fused|TMD_B200_FX=2,TMD_B200_OVERLAP=1,TMD_B200_FUSEPREP=1,SKIN=0.3", "--steps", "6", "--equil", "10", "--warmup", "2"])
    out = capsys.readouterr().out
    rows = [l for l in out.splitlines() if l.startswith(("default", "packed"))]
    assert len(rows) == 2 and "failed" not in out, out
    # same start, same seeds: the variants end at the same temperature, the fused one with fewer launches per step
    t = [float(r.split()[5]) for r in rows]
    launches = [float(r.split()[4]) for r in rows]
    assert abs(t[0] - t[1]) < 1e-3 * t[0] and launches[1] < launches[0], rows


def test_the_references_own_integrator_tests_pass_against_this_package(hostsim):
    """The scenarios of the reference's tests/test_integrator.py against what the unmodified reference computed on them
    (tests/golden/integrator_known_answers.npz, make_golden_known_answers.py), at that file's tolerance: kinetic energy
    with and without batches, constructor attributes, velocity-Verlet arithmetic with one and two replicas -- run through
    Integrator.step and the integrator kernels of the (host-interpreted) library."""
    from conftest import load_golden
    from torchmd_b200.integrator import Integrator, kinetic_energy, kinetic_to_temp
    from torchmd_b200.systems import System

    g = load_golden("integrator_known_answers")
    for i in range(6):
        batch = torch.tensor(g[f"ke{i}/batch"]) if f"ke{i}/batch" in g else None
        out = kinetic_energy(torch.tensor(g[f"ke{i}/masses"]), torch.tensor(g[f"ke{i}/vel"]), batch=batch)
        assert out.shape == g[f"ke{i}/out"].shape
        np.testing.assert_allclose(out.numpy(), g[f"ke{i}/out"], rtol=1e-6)

    class ConstantForces:
        def __init__(self, forces, pot):
            self.f, self.pot = forces, pot

        def compute(self, pos, box, forces):
            forces.copy_(self.f)
            return self.pot

    system = System(2, 1, torch.float32, "cpu")
    system.set_masses(torch.tensor([1.0, 2.0]))
    forces = ConstantForces(torch.zeros(1, 2, 3), 0.0)
    plain = Integrator(system, forces, 0.001, "cpu")
    assert plain.systems is system and plain.forces is forces and plain.device == "cpu"
    assert plain.T is None and plain.gamma is None
    assert plain.dt == pytest.approx(float(g["init/dt"]), rel=1e-12)
    thermo = Integrator(system, forces, 0.001, "cpu", gamma=1.0, T=300.0)
    assert thermo.T == 300.0 and thermo.gamma == pytest.approx(float(g["init/gamma"]), rel=1e-12)

    for c in ("mock", "batches", "two_atoms", "two_replicas"):
        pos = torch.tensor(g[c + "/pos"])
        system = System(pos.shape[1], pos.shape[0], torch.float32, "cpu")
        system.pos.copy_(pos)
        system.vel.copy_(torch.tensor(g[c + "/vel"]))
        system.set_masses(torch.tensor(g[c + "/masses"]))
        forces = ConstantForces(torch.tensor(g[c + "/forces"]), float(g[c + "/pot"]))
        if g[c + "/precompute"]:
            forces.compute(system.pos, system.box, system.forces)
        batch = torch.tensor(g[c + "/batch"]) if c + "/batch" in g else None
        integ = Integrator(system, forces, float(g[c + "/timestep"]), "cpu", batch=batch)
        assert integ.batch is batch and np.array_equal(integ.natoms, g[c + "/natoms"])
        for k, n in enumerate(g[c + "/niters"]):
            ekin, pot, temp = integ.step(niter=int(n))
            assert isinstance(ekin, np.ndarray) and isinstance(temp, np.ndarray) and isinstance(pot, (int, float))
            assert ekin.shape == temp.shape == g[f"{c}/ekin_{k}"].shape
            assert pot == float(g[f"{c}/pot_{k}"])
            np.testing.assert_allclose(system.pos.numpy(), g[f"{c}/pos_{k}"], rtol=1e-6, err_msg=c)
            np.testing.assert_allclose(system.vel.numpy(), g[f"{c}/vel_{k}"], rtol=1e-6, err_msg=c)
            np.testing.assert_allclose(ekin, g[f"{c}/ekin_{k}"], rtol=1e-6, err_msg=c)
            np.testing.assert_allclose(temp, g[f"{c}/temp_{k}"], rtol=1e-6, err_msg=c)
            np.testing.assert_allclose(ekin, kinetic_energy(system.masses, system.vel, batch=batch).numpy().flatten(), rtol=1e-6)
            np.testing.assert_allclose(temp, kinetic_to_temp(ekin, integ.natoms), rtol=1e-6)


def test_decomposed_integrator_replays_captured_steps(hostsim, monkeypatch):
    """DecomposedIntegrator with its default exchange and use_graph=True (one rank): the step it captures -- half-kick,
    exchange, force call with the gated rebuild, second half-kick -- replays to the trajectory of Integrator.step."""
    import torch.distributed as dist

    import test_gpu_zzz_p2p as P
    from torchmd_b200 import Integrator
    from torchmd_b200.domain import DecomposedIntegrator

    monkeypatch.setattr(P, "DEV", "cpu")
    monkeypatch.setattr(P, "SIZE", dict(waters=64, cutoff=5.0, switch=4.0, skin=0.3, steps=(1, 2, 7), backend="gloo"))
    monkeypatch.setenv("MASTER_ADDR", "127.0.0.1")
    monkeypatch.setenv("MASTER_PORT", str(T_free_port()))
    _fake_torch_graphs(monkeypatch, hostsim)
    dist.init_process_group("gloo", rank=0, world_size=1)
    try:
        sa, fa = P._setup()
        torch.manual_seed(9)
        ia = Integrator(sa, fa, 1.0, "cpu", gamma=0.1, T=300.0)
        sb, fb = P._setup()
        torch.manual_seed(9)
        ib = DecomposedIntegrator(sb, fb, 1.0, "cpu", gamma=0.1, T=300.0, use_graph=True)
        assert ib.exchange == "allgather"
        launched = _graph_counters(hostsim)[0]
        for niter in (1, 2, 7):
            ea, eb = ia.step(niter=niter), ib.step(niter=niter)
            assert torch.equal(sa.pos, sb.pos) and torch.equal(sa.vel, sb.vel)
            np.testing.assert_allclose(ea[1], eb[1], rtol=1e-9, atol=1e-6)
        assert ib.use_graph and len(ib._graphs) == 2 and _graph_counters(hostsim)[0] - launched == 10
        assert fb.stats()["rebuilds"] >= 2
    finally:
        dist.destroy_process_group()


def _fuzz_module():
    import importlib.util

    spec = importlib.util.spec_from_file_location("fuzz_interpreter", os.path.join(T.ROOT, "scripts", "fuzz_interpreter.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.mark.parametrize("build", ["default", "round2"])
def test_differential_fuzz_sample(request, build):
    """A seeded sample of scripts/fuzz_interpreter.py (random non-cubic boxes, atoms a box away, replicas, exclusions,
    switching / reaction field / no cutoff) on the default build and on the build with every opt-in path on."""
    request.getfixturevalue("hostsim" if build == "default" else "hostsim_r2")
    fuzz = _fuzz_module()
    bad = []
    for seed in range(2000, 2016):
        ok, desc = fuzz.one_case(seed)
        if not ok:
            bad.append(desc)
    assert not bad, "\n".join(bad)


def test_differential_fuzz_far_images_strict(request, monkeypatch):
    """Atoms up to seven boxes away (image counts for which fl(L * count) is inexact): the float pair kernel's force
    VALUES use the unrounded image shift (physics.cuh straddle_value), so they meet the plain 1e-4 yardstick -- without
    the allowance for the reference's own fp32 deviation -- where the kernel without it fails 1 case in 6."""
    request.getfixturevalue("hostsim")
    monkeypatch.setenv("FAR", "7")
    monkeypatch.setenv("STRICT", "1")
    fuzz = _fuzz_module()
    bad = []
    for seed in list(range(1045, 1060)):  # 1049, 1052, 1058 fail with the rounded shift
        ok, desc = fuzz.one_case(seed)
        if not ok:
            bad.append(desc)
    assert not bad, "\n".join(bad)


@pytest.mark.parametrize("build", ["default", "round2"])
def test_differential_fuzz_bonded_terms(request, monkeypatch, build):
    """The fuzzer with random angles, multi-term dihedrals (cosine series or the all-periods-zero harmonic form), impropers
    and scaled 1-4 pairs over random atom tuples, periodic and not, several replicas."""
    request.getfixturevalue("hostsim" if build == "default" else "hostsim_r2")
    monkeypatch.setenv("BONDED", "1")
    fuzz = _fuzz_module()
    bad = []
    for seed in range(3000, 3012):
        ok, desc = fuzz.one_case(seed)
        if not ok:
            bad.append(desc)
    assert not bad, "\n".join(bad)


@pytest.mark.parametrize("env", [{"REPBOX": "1", "BONDED": "1"}, {"NOCUT": "1", "REPBOX": "1", "FAR": "3"}], ids=["replica-boxes", "periodic-no-cutoff"])
def test_differential_fuzz_box_variants(request, monkeypatch, env):
    """Every replica in its own box (own cell grid per replica), and periodic boxes without a cutoff (every pair at its
    minimum image: the guarded minimum-image variant of the pair kernel over the all-pairs list)."""
    request.getfixturevalue("hostsim")
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    fuzz = _fuzz_module()
    bad = []
    for seed in range(4000, 4010):
        ok, desc = fuzz.one_case(seed)
        if not ok:
            bad.append(desc)
    assert not bad, "\n".join(bad)


@pytest.mark.parametrize("n,periodic,cutoff,coords,npairs", [
    (1, True, 9.0, [[1.0, 2.0, 3.0]], 0),  # a single atom: empty list, zero force (the force buffer is overwritten)
    (1, False, None, [[1.0, 2.0, 3.0]], 0),
    (2, True, 9.0, [[1.0, 2.0, 3.0], [20.0, 2.0, 3.0]], 1),  # the only pair is across the boundary
    (2, True, 9.0, [[1.0, 2.0, 3.0], [12.0, 14.0, 3.0]], 0),  # no pair inside the cutoff
    (2, False, None, [[1.0, 2.0, 3.0], [4.0, 2.0, 3.0]], 1),
    (3, False, 4.0, [[0.0, 0.0, 0.0], [100.0, 0.0, 0.0], [0.0, 300.0, 0.0]], 0),  # sparse, no box: empty cells everywhere
])
def test_smallest_systems(hostsim, n, periodic, cutoff, coords, npairs):
    from oracle import refmd
    from torchmd_b200 import Forces
    from torchmd_b200.parameters import TopologyParameters

    def par(prec):
        return TopologyParameters(atom_types=np.zeros(n, int), type_sigma=[3.0], type_epsilon=[0.1], charges=np.full(n, 0.3, np.float32),
                                  masses=np.full(n, 12.0, np.float32), precision=prec, device="cpu")

    cfg = dict(cutoff=cutoff, rfa=cutoff is not None)
    terms = ["lj", "electrostatics"]
    f = Forces(par(torch.float32), terms=terms, **cfg)
    p = torch.tensor(coords, dtype=torch.float32)[None]
    box = torch.zeros(1, 3, 3)
    if periodic:
        box[0] = torch.eye(3) * 25.0
    F = torch.full_like(p, 3.0)
    E = f.compute(p, box, F, returnDetails=True)
    F64 = torch.zeros(1, n, 3, dtype=torch.float64)
    E64 = refmd.OracleForces(par(torch.float64), terms, decision_dtype=torch.float32, **cfg).compute(p.double(), box.double(), F64)
    assert tuple(f.neighbour_pairs(p, box).shape) == (npairs, 2)
    assert float((F.double() - F64).abs().max()) < 1e-5
    for k in terms:
        assert abs(E[0][k] - E64[0][k]) < 1e-5


def test_md_steps_two_replicas_in_different_boxes(hostsim):
    """Fused MD steps with two replicas that differ in configuration AND box (own cell grid, own rebuild moments; thin
    skin so that lists are rebuilt inside the run): positions and velocities after 20 NVE steps against the oracle's
    integrator run in fp64 on the reference's fp32 in/out decisions."""
    from conftest import golden_cfg, load_golden, params_from_golden
    from oracle import refmd
    from torchmd_b200 import Forces, Integrator, System

    g, t = load_golden("water291_rf_switch"), load_golden("water291_traj")
    terms = [str(x) for x in g["terms"]]
    cfg = golden_cfg(g)
    n = len(g["coords"])
    L0 = np.asarray(g["box"], np.float64).reshape(-1)[:3]
    scale = np.array([1.0, 1.04])
    coords = np.stack([g["coords"].astype(np.float64) * s for s in scale])  # replica 1: the same waters 4 % further apart
    system = System(n, 2, torch.float32, "cpu")
    system.pos[:] = torch.tensor(coords, dtype=torch.float32)
    for r in range(2):
        system.box[r] = torch.diag(torch.tensor(L0 * scale[r], dtype=torch.float32))
    system.set_velocities(torch.tensor(t["vel0_f32"]))
    forces = Forces(params_from_golden(g, device="cpu"), terms=terms, skin=0.3, **cfg)
    forces.compute(system.pos, system.box, system.forces)
    pos0, vel0, box = system.pos.clone(), system.vel.clone(), system.box.clone()
    integ = Integrator(system, forces, 1.0, "cpu")
    ek, ep, T = integ.step(niter=20)
    assert forces.stats()["rebuilds"] >= 2

    o = refmd.OracleForces(params_from_golden(g, precision=torch.float64), terms, decision_dtype=torch.float32, **cfg)
    p64, v64, F64 = pos0.double(), vel0.double(), torch.zeros(2, n, 3, dtype=torch.float64)
    o.compute(p64, box.double(), F64)
    oi = refmd.OracleIntegrator(p64, v64, box.double(), F64, params_from_golden(g, precision=torch.float64).masses.double(),
                                lambda p, b, f: o.compute(p, b, f), 1.0)
    oek, oep, oT = oi.step(niter=20)
    dp = float((system.pos.double() - p64).abs().max())
    dv = float((system.vel.double() - v64).abs().max())
    print(f"two boxes, 20 NVE steps: dpos {dp:.2e} A, dvel {dv:.2e}")
    assert dp < 1e-4 and dv < 5e-4
    np.testing.assert_allclose(ek, oek, rtol=2e-4)
    assert abs(float(T[0]) - float(T[1])) > 1e-3  # the replicas really ran different trajectories
