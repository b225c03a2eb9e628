"""bench.py -- MD steps/s on the synthetic 100k-atom TIP3P water box (BASELINE.json).

    python bench.py --gpus 1 --steps K --warmup W          # our arm
    python bench.py --impl reference --steps K --warmup W  # reference CPU arm (oracle port)

One "step" is one MD step (velocity Verlet + Langevin, LJ + reaction-field
electrostatics + bonds + angles, cutoff 9 / switch 7.5, dt 1 fs) of 33,333 flexible
TIP3P waters (99,999 atoms, fp32).  Rank 0 prints ONE JSON line:

  value      steps/s with the state resident in HBM, K steps enqueued back to back
             through Integrator.step (CUDA events on the launching stream, max over ranks)
  e2e        steps/s through the C-ABI host entry tmd_md_steps_host: pinned HOST
             positions+velocities copied in, one step, positions+velocities+energies
             copied back, every step
  roofline   non-bonded pair kernel: algorithmic bytes (32 N + 4 P_rc, SURVEY.md
             section 8d) / its mean duration (CUDA events around each launch inside the
             timed region) against the measured HBM peak (MEASURED_PEAKS.json)
  cpu_baseline  the oracle port of the reference's all-pairs PyTorch-CPU path timed on
             this box's host cores on a bounded sample (smaller box, O(N^2) scaled)

--dump-outputs DIR (one GPU) writes what the last timed step left to a caller of Integrator.step, as
DIR/<name>.npy: positions, velocities, forces (replicas, atoms, 3) float32 and the per-replica
kinetic_energy, potential_energy and temperature.  So that the same arguments give the same inputs on
every run and two builds can be compared output for output, the warm-up then runs a fixed number of
steps (not "at least 0.6 s") and the relaxation of the water boxes runs on the full Verlet rows, whose
force sums have a fixed order.  The warm-up and the timed steps stay on the default path: where that is
the cluster path, whose force sums depend on the order of arrival, two runs differ by rounding that the
dynamics amplify with every step, so per-atom arrays are comparable over short runs only.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_WATERS = 33333
TERMS = ["lj", "electrostatics", "bonds", "angles"]
CFG = dict(cutoff=9.0, rfa=True, switch_dist=7.5)
TIMESTEP_FS = 1.0
GAMMA_PS = 0.1
TEMPERATURE = 300.0
FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md

# BASELINE.json configs as bench workloads.  The headline (and the default) is water100k.
WORKLOADS = {
    "water100k": "synthetic TIP3P water box, 33333 waters = 99999 atoms, L=99.93 A, LJ(switch 7.5)+RF electrostatics cutoff 9 A, "
                 "flexible bonds+angles, Langevin 300 K gamma 0.1/ps, dt 1 fs, 1 replica (BASELINE config 4)",
    "water800k": "synthetic TIP3P water box, 266664 waters = 799992 atoms, L=199.87 A, same settings as water100k: eight times the "
                 "headline box, the weak-scaling companion of the 8-GPU line (about one headline box of work per GPU)",
    "water10k": "synthetic TIP3P water box, 3333 waters = 9999 atoms, L=46.39 A, same settings as water100k: the largest size "
                "the reference's all-pairs path runs in seconds per step, so BOTH arms are timed on it",
    "water291": "the reference's tests/water fixture: 97 waters = 291 atoms, L=16.9 A, 2 replicas, LJ(switch 6.0)+RF cutoff 7.3 A, "
                "bonds+angles, Langevin 300 K (BASELINE config 2)",
    "ala2": "the reference's tests/prod_alanine_dipeptide_amber: 688 atoms in a 19.8 A box, AMBER bonds/angles/dihedrals/impropers/1-4 + "
            "LJ(switch 7.5)+RF cutoff 9 A, Langevin 300 K (BASELINE config 3)",
    "thrombin16": "the reference's tests/thrombin-ligand-amber: 4676 atoms, no box, all AMBER terms, RF cutoff 7.3 A, 16 replicas "
                  "(sharded over the GPUs when --gpus > 1), Langevin 300 K (BASELINE config 5)",
}


def build_workload(name, device, precision=None, nrep=None):
    """(par, coords (N,3), box (3,), terms, cfg, nrep, needs_equilibration) of a workload."""
    import numpy as np
    import torch

    from torchmd_b200 import testsystems

    precision = precision or torch.float32
    if name in ("water100k", "water10k", "water800k"):
        sysd = testsystems.water_box({"water100k": N_WATERS, "water10k": 3333, "water800k": 266664}[name], seed=0)
        par = testsystems.water_parameters(sysd, precision=precision, device=device)
        return par, np.asarray(sysd["coords"], np.float32), np.asarray(sysd["box"], np.float32), list(TERMS), dict(CFG), nrep or 1, True
    golden = {"water291": ("water291_rf_switch", 2), "ala2": ("ala2_xsc_rf", 1), "thrombin16": ("thrombin_nobox_rf", 16)}[name]
    par, coords, box, terms, cfg = testsystems.golden_system(golden[0], precision=precision, device=device)
    return par, coords, box, terms, cfg, nrep or golden[1], False


# ------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the oracle port of the reference's CPU path
# ------------------------------------------------------------------------------------
def _probe_threads():
    """ATen's elementwise kernels stop scaling (and degrade) on very wide hosts: probe a few thread counts on a
    3,000-atom box and give the reference the fastest one."""
    import torch

    from oracle import refmd
    from torchmd_b200 import testsystems

    ncores = os.cpu_count() or 1
    best = (float("inf"), ncores)
    try:
        probe = testsystems.water_box(1000, seed=0)
        ppar = testsystems.water_parameters(probe, precision=torch.float32)
        pof = refmd.OracleForces(ppar, TERMS, **CFG)
        ppos = torch.tensor(probe["coords"])[None].clone()
        pbox = torch.zeros(1, 3, 3)
        for k in range(3):
            pbox[0, k, k] = float(probe["box"][k])
        pF = torch.zeros_like(ppos)
        for nt in sorted({min(ncores, c) for c in (8, 16, 32, 64, ncores)}):
            torch.set_num_threads(nt)
            pof.compute(ppos, pbox, pF)
            t0 = time.perf_counter()
            pof.compute(ppos, pbox, pF)
            dt = time.perf_counter() - t0
            if dt < best[0]:
                best = (dt, nt)
    except Exception:
        pass
    torch.set_num_threads(best[1])
    return best[1], ncores


def cpu_reference_run(workload, steps, warmup, budget_s=150.0):
    """Time the reference algorithm (all-pairs table + cutoff mask, torch CPU ops, all useful host threads) through the
    oracle port.  water100k cannot run there at all (the pair table alone is 80 GB, BASELINE.md section 2): the arm then
    times a BOUNDED SAMPLE -- the same generator and settings at a box size whose steps fit the budget -- and
    reports what it MEASURED at that size; an O(N^2) extrapolation to 99,999 atoms is given separately and labelled.
    Every other workload is timed as it is (thrombin16: fewer replicas if 16 do not fit the budget)."""
    import numpy as np
    import torch

    from oracle import refmd

    nthreads, ncores = _probe_threads()
    sample_note = ""
    name = workload
    nrep_full = None
    if workload == "water100k":
        est = {3333: 1.6, 1000: 0.22, 333: 0.05}  # s/step measured on 8 cores (BASELINE.md)
        scale = 8.0 / max(1, min(ncores, 32))
        nw = 333
        for cand in (3333, 1000, 333):
            if (steps + warmup) * est[cand] * max(scale, 0.25) <= budget_s:
                nw = cand
                break
        from torchmd_b200 import testsystems

        sysd = testsystems.water_box(nw, seed=0)
        par = testsystems.water_parameters(sysd, precision=torch.float32)
        coords, boxd, terms, cfg, nrep = np.asarray(sysd["coords"], np.float32), np.asarray(sysd["box"], np.float32), list(TERMS), dict(CFG), 1
        sample_note = f"bounded sample of water100k: the same generator and settings at {3 * nw} atoms; "
    else:
        par, coords, boxd, terms, cfg, nrep, _ = build_workload(workload, "cpu")
        if workload == "thrombin16":
            nrep_full = nrep
            nrep = 2 if (steps + warmup) * 16 * 2.0 > budget_s else 16
            if nrep != nrep_full:
                sample_note = f"bounded sample of thrombin16: {nrep} of the {nrep_full} replicas (the reference loops over replicas serially, forces.py:116); "
    n = len(coords)
    t0 = time.perf_counter()
    of = refmd.OracleForces(par, terms, **cfg)
    t_init = time.perf_counter() - t0
    pos = torch.tensor(coords)[None].repeat(nrep, 1, 1).contiguous()
    box = torch.zeros(nrep, 3, 3)
    for k in range(3):
        box[:, k, k] = float(boxd[k])
    torch.manual_seed(1)
    vel = refmd.maxwell_boltzmann(par.masses, TEMPERATURE, nrep)
    F = torch.zeros_like(pos)
    fn = lambda p, b, f: [sum(e.values()) for e in of.compute(p, b, f)]  # noqa: E731
    fn(pos, box, F)
    integ = refmd.OracleIntegrator(pos, vel, box, F, par.masses, fn, TIMESTEP_FS, gamma_ps=GAMMA_PS, T=TEMPERATURE)
    integ.step(warmup)
    t0 = time.perf_counter()
    integ.step(steps)
    dt = time.perf_counter() - t0
    measured = steps / dt
    out = {
        "value": measured,
        "unit": "steps/s",
        "cores": nthreads,
        "kind": "port",
        "sample": (
            f"{sample_note}oracle/refmd.py (torch-CPU restatement of the reference; {nthreads} torch threads, the fastest of a probe "
            f"over 8..{ncores} on this {ncores}-core host), {n} atoms x {nrep} replica(s), {steps} steps after {warmup} warm-up: "
            f"{measured:.4g} steps/s measured ({dt / steps:.3f} s/step, pair-table init {t_init:.1f} s)"
        ),
        "measured_natoms": n,
        "measured_replicas": nrep,
        "ms_per_step_measured": 1e3 * dt / steps,
    }
    if workload == "water100k":
        out["extrapolated_99999_atoms_steps_per_s"] = measured * (n / (3.0 * N_WATERS)) ** 2
        out["extrapolation_note"] = "measured x (natoms/99999)^2, the all-pairs O(N^2) law; NOT a measurement: 99,999 atoms are infeasible for the reference (O(N^2) memory)"
    if nrep_full and nrep != nrep_full:
        out["extrapolated_16_replicas_steps_per_s"] = measured * nrep / nrep_full
    return out


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = max(1, args.steps)
    base = cpu_reference_run(args.workload, steps, max(0, args.warmup))
    cfg = workload_config(args.gpus, args.workload)
    cfg["natoms"] = base["measured_natoms"]  # what this arm actually ran
    cfg["replicas"] = base["measured_replicas"]
    if args.workload == "water100k":
        cfg["workload"] = ("REFERENCE ARM SAMPLE of: " + cfg["workload"] + f" -- timed at {base['measured_natoms']} atoms "
                           "(the reference cannot hold the 99,999-atom pair table); `value` is the measured steps/s at that size")
    line = {
        "impl": "reference",
        "metric": METRICS[args.workload],
        "value": base["value"],
        "unit": "steps/s",
        "n_gpus": args.gpus,
        "steps": steps,
        "warmup": args.warmup,
        "ms_per_step": 1e3 / base["value"],
        "higher_is_better": True,
        "scaling": "strong",
        "vs_baseline": None,
        "dtype": "f32",
        "data": "synthetic",
        "config": cfg,
        "cpu_baseline": base,
        "e2e": {"value": base["value"], "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


METRICS = {
    "water100k": "MD steps/sec (100k-atom water, fp32)",
    "water10k": "MD steps/sec (9,999-atom water, fp32)",
    "water800k": "MD steps/sec (799,992-atom water, fp32)",
    "water291": "MD steps/sec (tests/water fixture, 291 atoms x 2 replicas, fp32)",
    "ala2": "MD steps/sec (alanine dipeptide in water, 688 atoms, AMBER, fp32)",
    "thrombin16": "MD steps/sec (thrombin-ligand, 4676 atoms x 16 replicas, fp32)",
}


def workload_config(ngpus, workload="water100k"):
    replicated = workload in ("thrombin16", "water291")
    return {
        "workload": WORKLOADS[workload],
        "natoms": {"water100k": 3 * N_WATERS, "water800k": 799992, "water10k": 9999, "water291": 291, "ala2": 688, "thrombin16": 4676}[workload],
        "pair_kernel": "cluster half list, packed fp32x2 arithmetic on fixed-point separations (cluster.cuh) where it applies; "
                       "TMD_B200_CLUSTER=0: full Verlet rows",
        "parallelism": "single GPU" if ngpus == 1 else (
            f"replicas sharded over {ngpus} GPUs, no per-step collective" if replicated else
            f"spatial slabs over {ngpus} GPUs, " + ("positions pushed to all ranks over NVLink peer memory by the integration kernel"
                                                   if os.environ.get("TMD_B200_EXCHANGE", "").lower() == "p2p" else "position all-gather")),
        "l2": "no flush between steps: consecutive MD steps are data-dependent (each step's positions are the previous step's "
        "output); the state is re-read from L2/HBM as a real run does",
    }


# ------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------
class ClockSampler:
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index=0):
        self.tmp = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(gpu_index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=self.tmp, stderr=subprocess.DEVNULL,
            )
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.tmp.flush()
        self.tmp.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.tmp.read().splitlines():
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.tmp.name)
        if sm:
            sm.sort()
            out.update(sm_mhz=sm[len(sm) // 2], sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


# ------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------
DEVICE_OVERRIDE = None  # tests/test_mirrors_on_interpreter.py dry-runs gpu_arm on the host interpreter build with "cpu"
MIN_DECOMPOSED_WARMUP = 5000  # N > 1: steps before the timed region (>= 0.4 s under load for the clock sampler)


def gpu_arm(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from torchmd_b200 import Forces, Integrator, System, _lib, maxwell_boltzmann

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    wl = args.workload
    replicated = wl in ("thrombin16", "water291")
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs runs with one GPU")
    if world > 1:
        # (NCCL's own log, if NCCL_DEBUG is set, goes to stderr / NCCL_DEBUG_FILE; rank 0 prints the JSON line last)
        if not dist.is_initialized():  # (tests/test_domain_host.py brings its own gloo group)
            dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    dev = DEVICE_OVERRIDE or f"cuda:{local}"
    if DEVICE_OVERRIDE is None:
        torch.cuda.set_device(local)
    if world > 1 and not replicated:
        if wl not in ("water100k", "water800k"):
            raise SystemExit(f"--gpus > 1 runs water100k / water800k (spatial decomposition) or the replicated workloads, not {wl}")
        from torchmd_b200 import domain  # spatial decomposition driver

        try:
            return domain.bench_decomposed(args, world, rank, local, workload_config(world, wl))
        finally:
            dist.destroy_process_group()

    par, coords, boxd, terms, cfg, nrep_total, needs_eq = build_workload(wl, dev)
    # replicas are independent (forces.py:116 loops over them): shard them over the ranks, no per-step collective
    if nrep_total % world:
        raise SystemExit(f"{nrep_total} replicas do not divide over {world} ranks")
    nrep = nrep_total // world
    n = len(coords)
    system = System(n, nrep, torch.float32, dev)
    system.set_positions(coords)
    system.set_box(boxd)
    torch.manual_seed(1 + rank)
    system.set_velocities(maxwell_boltzmann(par.masses, TEMPERATURE, nrep))
    # --dump-outputs: the relaxation runs on the full Verlet rows, whose force sums have a fixed order, so that every run
    # enters the warm-up from the same state (the cluster path adds forces in arrival order, and MD amplifies the last bits)
    relax_env = {"TMD_B200_CLUSTER": "0"} if args.dump_outputs and needs_eq else {}
    env_before = {k: os.environ.get(k) for k in relax_env}
    os.environ.update(relax_env)
    forces = Forces(par, terms=terms, **cfg)
    forces.compute(system.pos, system.box, system.forces)

    # relax a lattice start into a liquid: strong coupling, then the production thermostat
    equil_done = 0
    if needs_eq:
        eq = Integrator(system, forces, TIMESTEP_FS, dev, gamma=10.0, T=TEMPERATURE)
        for _ in range(args.equil // 100):
            eq.step(niter=100)
            equil_done += 100
        for k, v in env_before.items():  # the warm-up and the timed steps run the default path
            if v is None:
                os.environ.pop(k)
            else:
                os.environ[k] = v
        if equil_done or relax_env:
            # A lattice start can be refused by the cluster lists (its 4-atom clusters are too long for a small box) and the
            # context then waits >= 1000 force calls before it tries them again: the melted configuration gets a fresh one.
            forces = Forces(par, terms=terms, **cfg)
            forces.compute(system.pos, system.box, system.forces)
    integ = Integrator(system, forces, TIMESTEP_FS, dev, gamma=GAMMA_PS, T=TEMPERATURE)
    sampler = ClockSampler(local) if rank == 0 else None  # runs through the warm-up too (same load)
    t_w = time.perf_counter()
    chunk = 50 if n > 20000 else 500
    nwarm = max(3, args.warmup, chunk if world == 1 else 4 * chunk)
    done = 0
    # >= 0.6 s under load for the sampler; a fixed step count when the outputs are dumped (a reproducible start)
    while done < nwarm or (world == 1 and not args.dump_outputs and time.perf_counter() - t_w < 0.6):
        ekin, pot, T = integ.step(niter=chunk)
        done += chunk

    L = _lib.lib()
    stream = torch.cuda.current_stream().cuda_stream
    st0 = forces.stats()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    ekin, pot, T = integ.step(niter=args.steps)
    ev1.record()
    torch.cuda.synchronize()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, system, ekin, pot, T)
    import ctypes as C

    # The timed steps are replays of a captured step (one graph launch per step); a kernel inside a replay cannot be
    # bracketed by events, so the pair kernel is timed with CUDA events around each of its launches in a stretch of
    # the SAME run right after the timed region, launched kernel by kernel on the same stream.
    nprof = min(200, args.steps)
    st_p0 = forces.stats()
    _lib.check(L.tmd_profile_begin(forces._ctx, nprof))
    integ.step(niter=nprof)
    pair_ms, pair_n = C.c_double(), C.c_int()
    _lib.check(L.tmd_profile_end(forces._ctx, C.byref(pair_ms), C.byref(pair_n), stream))
    st_p1 = forces.stats()
    ms_total = ev0.elapsed_time(ev1)
    if world > 1:
        t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)  # device time, max over ranks
        ms_total = float(t.item())
        dist.barrier()
    clocks = sampler.stop() if sampler else None
    st1 = st_p0
    ms_per_step = ms_total / args.steps
    value = 1e3 / ms_per_step
    pair_kernel_id = int(L.tmd_pair_kernel(forces._ctx))

    # exact number of in-cutoff pairs of the final configuration (reference predicate), replica 0
    p_rc = 0
    if forces.require_distances:
        count = torch.zeros(1, dtype=torch.int64, device=dev)
        dummy = torch.zeros(2, dtype=torch.int32, device=dev)
        scratch = torch.empty_like(system.pos)
        forces.compute(system.pos, system.box, scratch)
        _lib.check(L.tmd_export_pairs(forces._ctx, system.pos.data_ptr(), 0, dummy.data_ptr(), 0, count.data_ptr(), stream))
        p_rc = int(count.item())

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", FALLBACK_HBM_GBS))
    pair_avg_ms = pair_ms.value / max(1, pair_n.value)
    alg_bytes = nrep * (32.0 * n + 4.0 * p_rc)  # SURVEY.md 8d, per force evaluation and replica
    achieved = alg_bytes / (pair_avg_ms * 1e-3) / 1e9 if pair_avg_ms > 0 else 0.0
    kname = {0: "k_pair (full rows, float separations)", 1: "k_pair_fx (full rows, fixed-point separations)",
             2: "k_pair_fx2 (full rows, packed fp32x2)", 3: "k_pair2_open (full rows, packed fp32x2, no box)",
             4: "k_cpair (cluster half list, TMA-staged entries, packed fp32x2)"}.get(pair_kernel_id, str(pair_kernel_id))
    # the pair kernel's other roof: packed or not, the SM issues 128 fp32 FMA lanes per clock
    flops_per_pair = 60.0
    fp32_peak_tflops = 148 * 128 * 2 * (clocks["sm_mhz"] if clocks and clocks.get("sm_mhz") else 1965.0) * 1e6 / 1e12
    roofline = {
        "kernel": kname,
        "bound": "hbm",
        "achieved": achieved,
        "peak": peak,
        "unit": "GB/s",
        "frac": achieved / peak,
        "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)",
        "algorithmic_bytes": alg_bytes,
        "pairs_in_cutoff": p_rc,
        "avg_kernel_ms": pair_avg_ms,
        "launches_sampled": pair_n.value,
        "share_of_step": pair_avg_ms / ms_per_step,
        "timing": f"CUDA events around each of {pair_n.value} launches in {nprof} steps run kernel by kernel right after the timed "
                  "region (the timed steps are graph replays, whose kernels cannot be bracketed)",
        "traffic": None,
        "fp32_useful_tflops": nrep * p_rc * flops_per_pair / (pair_avg_ms * 1e-3) / 1e12 if pair_avg_ms > 0 else 0.0,
        "fp32_peak_tflops": fp32_peak_tflops,
        "note": "the pair loop is bound by the fp32 pipe, not by HBM (DESIGN.md 4): ~60 flop per in-cutoff pair; "
                "fp32_useful_tflops / fp32_peak_tflops is its fraction of that roof",
    }
    try:
        prof = json.load(open(os.path.join(ROOT, "profiles", "pair_kernel_traffic.json")))
        if prof.get("kernel_id") == pair_kernel_id and wl == "water100k":
            roofline["traffic"] = prof.get("dram_bytes_per_launch")
            roofline["traffic_source"] = prof.get("source")
    except Exception:
        pass

    # end to end: host-resident state through the C-ABI host entry, one step per call
    e2e_steps = min(args.steps, args.e2e_steps)
    hpos = torch.empty(system.pos.shape, dtype=torch.float32, pin_memory=True)
    hvel = torch.empty(system.vel.shape, dtype=torch.float32, pin_memory=True)
    hpos.copy_(system.pos)
    hvel.copy_(system.vel)
    hene = np.zeros((nrep, _lib.NUM_ENERGIES), dtype=np.float64)
    hke = np.zeros(nrep, dtype=np.float64)
    gamma_int = GAMMA_PS / (1000.0 / 48.88821)

    def host_step(k):
        _lib.check(
            L.tmd_md_steps_host(
                forces._ctx, 1, hpos.data_ptr(), hvel.data_ptr(), system.forces.data_ptr(), integ.masses.data_ptr(),
                system.pos.data_ptr(), system.vel.data_ptr(), integ.dt, gamma_int, integ.vcoeff.data_ptr(),
                integ.seed, 10_000_000 + k, hene.ctypes.data, hke.ctypes.data, stream,
            )
        )

    for k in range(5):
        host_step(k)
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for k in range(e2e_steps):
        host_step(5 + k)
    t_e2e = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([t_e2e], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t_e2e = float(t.item())
    bytes_each_way = 2 * system.pos.numel() * 4 * world
    e2e = {
        "value": e2e_steps / t_e2e,
        "unit": "steps/s",
        "h2d_bytes_per_step": bytes_each_way,
        "d2h_bytes_per_step": bytes_each_way + (hene.nbytes + hke.nbytes) * world,
        "steps": e2e_steps,
        "api": "tmd_md_steps_host (C ABI, pinned host positions+velocities in and out every step)",
    }
    # replica sharding: the per-replica results gathered once, after the run (run.py:211-216 logs them per replica)
    launches = int(st1["kernel_launches"] - st0["kernel_launches"])
    if world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, (np.asarray(ekin).tolist(), [float(x) for x in pot], np.asarray(T).tolist()))
        T = np.concatenate([np.asarray(g[2]) for g in gathered])
        pot = sum((g[1] for g in gathered), [])
        t = torch.tensor([launches], dtype=torch.int64, device=dev)
        dist.all_reduce(t)
        launches = int(t.item())
        dist.destroy_process_group()
    if rank != 0:
        return
    base = cpu_reference_run(wl, 3, 1, budget_s=40.0) if not args.no_cpu_baseline else None

    line = {
        "metric": METRICS[wl],
        "value": value,
        "unit": "steps/s",
        "n_gpus": world,
        "steps": args.steps,
        "warmup": done,
        "ms_per_step": ms_per_step,
        "higher_is_better": True,
        "scaling": "strong",
        "vs_baseline": None,
        "dtype": "f32",
        "data": "synthetic" if wl in ("water100k", "water10k", "water800k") else "the reference's own test system (coordinates and parameters from its fixtures), random velocities",
        "config": workload_config(world, wl),
        "clocks": clocks,
        "e2e": e2e,
        "gpu_launches": launches,
        "roofline": roofline,
        "cpu_baseline": base,
        "state": {
            "temperature_K": float(np.mean(T)),
            "epot": float(pot[0]),
            "replicas": nrep_total,
            "replicas_per_gpu": nrep,
            "rebuilds_in_timed_region": int(st1["rebuilds"] - st0["rebuilds"]),
            "max_neighbours": int(st1["max_neighbours"]),
            "row_capacity": int(st1["row_capacity"]),
            "skin_A": forces.skin,
            "equilibration_steps": equil_done,
            "warmup_steps_run": done,
            "pair_kernel_id": pair_kernel_id,
        },
    }
    print(json.dumps(line), flush=True)


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, system, ekin, pot, T):
    """The state and the return values of the last timed Integrator.step call, one .npy file each."""
    import numpy as np

    arrays = {
        "positions": system.pos.detach().cpu().numpy(),
        "velocities": system.vel.detach().cpu().numpy(),
        "forces": system.forces.detach().cpu().numpy(),
        "kinetic_energy": np.asarray(ekin, np.float32),
        "potential_energy": np.asarray(pot, np.float64),
        "temperature": np.asarray(T, np.float32),
    }
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes of outputs exceed {DUMP_LIMIT_BYTES}")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3000, help="timed MD steps (>= 1)")
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--equil", type=int, default=600, help="relaxation steps before warm-up (lattice start)")
    ap.add_argument("--e2e-steps", type=int, default=300)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="water100k", choices=sorted(WORKLOADS),
                    help="water100k is BASELINE.json's headline; the others are its configs 2, 3, 5 and the 9,999-atom box both arms can run")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step to DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        return reference_arm(args)
    return gpu_arm(args)


if __name__ == "__main__":
    main()
