"""Host logic of the decomposed (multi-GPU) step on CPU: ownership ranges, the padded
gather layout and the per-step exchange, run with world_size 2 over gloo.  The CUDA
kernels are replaced by the oracle here (forces for the owned atoms, velocity Verlet on
the owned atoms); the GPU run of the same logic is tests/test_gpu_domain.py."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import ROOT


def test_ranges_cover_every_atom_once():
    from torchmd_b200.domain import SlabDecomposition

    for n, w in ((99999, 8), (99999, 4), (10, 3), (7, 8), (291, 2)):
        decs = [SlabDecomposition(n, w, r) for r in range(w)]
        owned = np.zeros(n, int)
        for d in decs:
            owned[d.lo : d.hi] += 1
            assert d.padded == d.chunk * w >= n and 0 <= d.lo <= d.hi <= n
        assert (owned == 1).all()
        assert decs[0].ranges() == [(d.lo, d.hi) for d in decs]


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, out):
    import sys

    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from oracle import refmd
    from torchmd_b200 import testsystems
    from torchmd_b200.domain import SlabDecomposition

    torch.set_num_threads(1)
    sysd = testsystems.water_box(30, seed=2)
    par = testsystems.water_parameters(sysd, precision=torch.float64)
    terms = ["lj", "electrostatics", "bonds", "angles"]
    of = refmd.OracleForces(par, terms, cutoff=4.0, rfa=True, switch_dist=3.0)
    n = len(sysd["coords"])
    box = torch.zeros(1, 3, 3, dtype=torch.float64)
    for k in range(3):
        box[0, k, k] = float(sysd["box"][k])
    torch.manual_seed(0)
    vel0 = refmd.maxwell_boltzmann(par.masses, 300.0, 1)

    def run(decomposed):
        pos = torch.tensor(sysd["coords"], dtype=torch.float64)[None].clone()
        vel = vel0.clone()
        F = torch.zeros_like(pos)
        m = par.masses.view(1, -1, 1)
        dt = 1.0 / refmd.TIMEFACTOR
        if decomposed:
            dec = SlabDecomposition(n, world, rank)
            buf, pos = dec.rehome(pos)
            send = torch.empty(dec.chunk * 3, dtype=pos.dtype)
            sl = slice(dec.lo, dec.hi)
        else:
            sl = slice(0, n)
        of.compute(pos, box, F)
        for _ in range(5):
            acc = F[:, sl] / m[:, sl]
            pos[:, sl] += vel[:, sl] * dt + 0.5 * acc * dt * dt
            vel[:, sl] += 0.5 * dt * acc
            if decomposed:
                dec.gather(buf, send)  # the exchange step
            of.compute(pos, box, F)  # the oracle computes all rows; only the owned ones are used
            vel[:, sl] += 0.5 * dt * (F[:, sl] / m[:, sl])
        return pos.clone(), vel.clone(), sl

    p1, v1, _ = run(False)
    p2, v2, sl = run(True)
    ok = torch.equal(p1, p2) and torch.equal(v1[:, sl], v2[:, sl])
    out.put((rank, bool(ok)))
    dist.destroy_process_group()


def test_decomposed_step_matches_single_process_gloo():
    world = 2
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, out)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=300)
        assert p.exitcode == 0
    results = dict(out.get(timeout=10) for _ in range(world))
    assert results == {0: True, 1: True}


def _worker_integrator(rank, world, port, out):
    """DecomposedIntegrator itself (its real step sequence through the C ABI, gloo all-gather) on the host
    SIMT-interpreter build of the library (tests/simt) against the undecomposed Integrator in the same process."""
    import sys

    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(1)
    import test_simt_kernels as T
    from torchmd_b200 import Forces, Integrator, System, _lib, maxwell_boltzmann, testsystems
    from torchmd_b200.domain import DecomposedIntegrator

    class _Stream:
        cuda_stream = None

    _lib._lib = T.load(os.path.join(T.SIMT_DIR, "libtmd_simt.so"))  # (built by the parent)
    _lib.on_device = lambda t: True
    torch.cuda.current_stream = lambda *a, **k: _Stream()
    torch.cuda.current_device = lambda: 0
    torch.cuda.synchronize = lambda *a, **k: None

    sysd = testsystems.water_box(64, seed=3)
    n = len(sysd["coords"])

    def make():
        par = testsystems.water_parameters(sysd)
        s = System(n, 1, torch.float32, "cpu")
        s.set_positions(sysd["coords"])
        s.set_box(sysd["box"])
        torch.manual_seed(4)
        s.set_velocities(maxwell_boltzmann(par.masses, 300.0, 1))
        f = Forces(par, terms=["lj", "electrostatics", "bonds", "angles"], cutoff=5.0, rfa=True, switch_dist=4.0, skin=0.4)
        return par, s, f

    par, s1, f1 = make()
    f1.compute(s1.pos, s1.box, s1.forces)
    torch.manual_seed(9)
    single = Integrator(s1, f1, 1.0, "cpu", gamma=0.1, T=300.0)
    par, s2, f2 = make()
    f2.compute(s2.pos, s2.box, s2.forces)
    torch.manual_seed(9)
    dec = DecomposedIntegrator(s2, f2, 1.0, "cpu", gamma=0.1, T=300.0, use_graph=False)
    ok = dec.exchange == "allgather" and single.seed == dec.integ.seed
    for niter in (1, 6):
        e1 = single.step(niter)
        e2 = dec.step(niter)
        lo, hi = dec.dec.lo, dec.dec.hi
        ok = ok and torch.equal(s1.pos, s2.pos) and torch.equal(s1.vel[:, lo:hi], s2.vel[:, lo:hi])
        ok = ok and abs(e1[1][0] - e2[1][0]) <= 1e-9 * abs(e1[1][0]) + 1e-9 and abs(float(e1[0][0]) - float(e2[0][0])) <= 1e-4 * abs(float(e1[0][0]))
    ok = ok and f2.stats()["rebuilds"] >= 2
    out.put((rank, bool(ok)))
    dist.destroy_process_group()


def test_decomposed_integrator_on_the_interpreter_matches_single_process_gloo():
    """world_size 2 over gloo: the N>1 host path (owned ranges, exchange, energy all-reduce, shared noise seed)
    follows the single-process trajectory bit for bit."""
    import sys

    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import test_simt_kernels as T

    T.build_simt()
    world = 2
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker_integrator, args=(r, world, port, out)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=300)
        assert p.exitcode == 0
    results = dict(out.get(timeout=10) for _ in range(world))
    assert results == {0: True, 1: True}


def _worker_bench(rank, world, port, out):
    """bench.py's N>1 body (torchmd_b200.domain.bench_decomposed) with two gloo ranks on the interpreter build."""
    import argparse
    import contextlib
    import io
    import json
    import sys
    import time

    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(1)
    import bench
    import test_simt_kernels as T
    from torchmd_b200 import _lib, domain

    class _Stream:
        cuda_stream = None

    class _Event:
        def __init__(self, enable_timing=False):
            self.t = 0.0

        def record(self, *a):
            self.t = time.perf_counter()

        def elapsed_time(self, other):
            return (other.t - self.t) * 1e3

    class _NoSampler:
        def __init__(self, *a):
            pass

        def stop(self):
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}

    _lib._lib = T.load(os.path.join(T.SIMT_DIR, "libtmd_simt.so"))
    _lib.on_device = lambda t: True
    torch.cuda.current_stream = lambda *a, **k: _Stream()
    torch.cuda.current_device = lambda: 0
    torch.cuda.synchronize = lambda *a, **k: None
    torch.cuda.Event = _Event
    bench.DEVICE_OVERRIDE, bench.MIN_DECOMPOSED_WARMUP, bench.N_WATERS = "cpu", 4, 64
    bench.CFG = dict(bench.CFG, cutoff=5.0, switch_dist=4.0)
    bench.ClockSampler = _NoSampler
    args = argparse.Namespace(gpus=world, steps=5, warmup=3, equil=6, e2e_steps=2, no_cpu_baseline=True, impl="ours", dump_outputs=None)
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf), contextlib.redirect_stderr(io.StringIO()):
        domain.bench_decomposed(args, world, rank, 0, bench.workload_config(world))
    lines = [l for l in buf.getvalue().splitlines() if l.startswith("{")]
    out.put((rank, json.loads(lines[-1]) if lines else None))
    dist.destroy_process_group()


def test_bench_decomposed_dry_run_gloo():
    """The N>1 arm of bench.py end to end (equilibration, warm-up, timed steps, eager profiling stretch, pair count,
    end-to-end loop, the JSON line) with two ranks -- rank 0 prints the one line, the others none."""
    import sys

    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import test_simt_kernels as T

    T.build_simt()
    world = 2
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker_bench, args=(r, world, port, out)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=300)
        assert p.exitcode == 0
    results = dict(out.get(timeout=10) for _ in range(world))
    assert results[1] is None
    line = results[0]
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline", "cpu_baseline"):
        assert key in line, key
    assert line["n_gpus"] == 2 and line["value"] > 0 and line["e2e"]["value"] > 0 and line["gpu_launches"] > 0
    assert line["roofline"]["pair_entries_counted"] > 0 and line["scaling"] == "strong"


def _worker_replicas(rank, world, port, out):
    """bench.py's replica-sharded arm (BASELINE config 5 pattern: R replicas over the ranks, no per-step collective, results
    gathered once) with two gloo ranks on the interpreter build, on the two-replica water fixture."""
    import argparse
    import contextlib
    import io
    import json
    import sys
    import time

    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), WORLD_SIZE=str(world), RANK=str(rank), LOCAL_RANK="0")
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(1)
    import bench
    import test_simt_kernels as T
    from torchmd_b200 import _lib

    class _Stream:
        cuda_stream = None

    class _Event:
        def __init__(self, enable_timing=False):
            self.t = 0.0

        def record(self, *a):
            self.t = time.perf_counter()

        def elapsed_time(self, other):
            return (other.t - self.t) * 1e3

    class _NoSampler:
        def __init__(self, *a):
            pass

        def stop(self):
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}

    real_empty = torch.empty

    def empty(*a, **k):
        k.pop("pin_memory", None)
        return real_empty(*a, **k)

    _lib._lib = T.load(os.path.join(T.SIMT_DIR, "libtmd_simt.so"))
    _lib.on_device = lambda t: True
    torch.cuda.current_stream = lambda *a, **k: _Stream()
    torch.cuda.current_device = lambda: 0
    torch.cuda.synchronize = lambda *a, **k: None
    torch.cuda.Event = _Event
    torch.empty = empty
    bench.DEVICE_OVERRIDE = "cpu"
    bench.ClockSampler = _NoSampler
    args = argparse.Namespace(gpus=world, steps=4, warmup=3, equil=0, e2e_steps=2, no_cpu_baseline=True, impl="ours", dump_outputs=None, workload="water291")
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf), contextlib.redirect_stderr(io.StringIO()):
        bench.gpu_arm(args)
    lines = [l for l in buf.getvalue().splitlines() if l.startswith("{")]
    out.put((rank, json.loads(lines[-1]) if lines else None))


def test_bench_replica_sharding_dry_run_gloo():
    """Two replicas over two ranks: one replica each, no collective inside the steps, one gather at the end; rank 0 prints the
    line with the per-replica temperatures of both ranks folded in."""
    import sys

    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import test_simt_kernels as T

    T.build_simt()
    world = 2
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker_replicas, args=(r, world, port, out)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=300)
        assert p.exitcode == 0
    results = dict(out.get(timeout=10) for _ in range(world))
    assert results[1] is None
    line = results[0]
    assert line["n_gpus"] == 2 and line["value"] > 0 and line["e2e"]["value"] > 0 and line["gpu_launches"] > 0
    assert line["state"]["replicas"] == 2 and line["state"]["replicas_per_gpu"] == 1
    assert "replicas sharded over 2 GPUs" in line["config"]["parallelism"]


def _worker_integrator_cluster(rank, world, port, out):
    """DecomposedIntegrator on the cluster half-list path (lists only for pairs that touch an owned atom) over gloo,
    against the undecomposed Integrator: same trajectory up to the summation order of the force reductions."""
    import sys

    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(1)
    import test_simt_kernels as T
    from test_simt_cluster import CFG, TERMS, tiled_water
    from torchmd_b200 import Forces, Integrator, System, _lib, maxwell_boltzmann, testsystems
    from torchmd_b200.domain import DecomposedIntegrator

    class _Stream:
        cuda_stream = None

    _lib._lib = T.load(os.path.join(T.SIMT_DIR, "libtmd_simt_cl.so"))  # (built by the parent)
    _lib.on_device = lambda t: True
    torch.cuda.current_stream = lambda *a, **k: _Stream()
    torch.cuda.current_device = lambda: 0
    torch.cuda.synchronize = lambda *a, **k: None
    sysd = tiled_water(2)
    n = len(sysd["coords"])

    def make():
        par = testsystems.water_parameters(sysd)
        s = System(n, 1, torch.float32, "cpu")
        s.set_positions(np.array(sysd["coords"], dtype=np.float32))
        s.set_box(sysd["box"])
        torch.manual_seed(4)
        s.set_velocities(maxwell_boltzmann(par.masses, 300.0, 1))
        return par, s, Forces(par, terms=TERMS, **CFG, skin=0.3)

    par, s1, f1 = make()
    f1.compute(s1.pos, s1.box, s1.forces)
    torch.manual_seed(9)
    single = Integrator(s1, f1, 1.0, "cpu", gamma=0.1, T=300.0)
    par, s2, f2 = make()
    f2.compute(s2.pos, s2.box, s2.forces)
    torch.manual_seed(9)
    dec = DecomposedIntegrator(s2, f2, 1.0, "cpu", gamma=0.1, T=300.0, use_graph=False)
    ok = single.seed == dec.integ.seed
    e1 = single.step(8)
    e2 = dec.step(8)
    lo, hi = dec.dec.lo, dec.dec.hi
    ok = ok and _lib.lib().tmd_pair_kernel(f2._ctx) == 4 and _lib.lib().tmd_pair_kernel(f1._ctx) == 4
    ok = ok and (s1.pos - s2.pos).abs().max().item() < 5e-5 and (s1.vel[:, lo:hi] - s2.vel[:, lo:hi]).abs().max().item() < 5e-4
    ok = ok and abs(e1[1][0] - e2[1][0]) <= 1e-5 * abs(e1[1][0]) + 2e-2
    ok = ok and f2.stats()["rebuilds"] >= 2
    out.put((rank, bool(ok)))
    dist.destroy_process_group()


def test_decomposed_integrator_cluster_path_gloo():
    import sys

    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import test_simt_kernels as T

    T.build_simt("_cl", T.VARIANTS["_cl"])
    world = 2
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker_integrator_cluster, args=(r, world, port, out)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=600)
        assert p.exitcode == 0
    results = dict(out.get(timeout=10) for _ in range(world))
    assert results == {0: True, 1: True}
