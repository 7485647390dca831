#!/usr/bin/env python
"""bench.py -- atom-steps/s of the MD hot path on B200 (BASELINE.json's metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--cells C]

Workload (config C3 of BASELINE.md, the one the metric is quoted on): rocksalt PbTe, 50x50x50
conventional cells = 1 000 000 atoms per GPU, Gaussian rattle 0.02 A (seed 1), velocities at 300 K
(seed 42), NVE, dt = 1 fs, NEP model tests/golden/nep_PbTe.txt (the reference's
tests/gpumd/dump_observer/PbTe_species/PbTe.txt).  One "step" = velocity-Verlet half step ->
Force::compute (position wrap, zero, neighbour maintenance, NEP descriptor / MLP / forces) ->
second half step -> thermo reduction: exactly what Run::perform_a_run does per step
(src/main_gpumd/run.cu:250-318), every kernel from libb200md.so.

Printed JSON (one line, rank 0):
  value      whole-job atom-steps/s, state resident in HBM, CUDA-event timed, max over ranks
  e2e        the same metric through the host-buffer C-ABI call b200md_nep_compute_host
             (positions/types H2D from pinned memory, energies/forces/virials D2H, every step)
  roofline   dominant kernel: SURVEY.md 8(d) algorithmic bytes per atom x atoms / mean launch time
  cpu_baseline  the reference's own CPU implementation (NEP_CPU, oracle/_ref) on the host cores
  reference_gpu the unmodified reference gpumd (oracle/_ref/gpumd_ref) on the same GPU(s), same
                model.xyz / run.in / step count, run after our timed region -- the bar north_star names
  neighbor      cost of one neighbour rebuild and the measured steps per rebuild
--impl reference times NEP_CPU alone on the same crystal/model/metric (bounded sample per step).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
GOLDEN = ROOT / "tests" / "golden"
MODEL = GOLDEN / "nep_PbTe.txt"
METRIC = "atom-steps/sec (1M-atom PbTe NEP NVE per GPU)"
DOMAIN_SKIN = 3.0  # A, multi-GPU ghost-list skin (gpumd_b200/domain.py)


def stage_algorithmic_bytes(nn, model):
    """SURVEY.md 8(d) per-stage algorithmic bytes per atom-step (counting rule stated there).
    Ng/Nr/Na = measured mean skin/radial/angular list lengths; K = steps per list rebuild."""
    Ng, Nr, Na = nn["skin"], nn["radial"], nn["angular"]
    D, Dr, S = model["D"], model["Dr"], model["S"]
    Da = D - Dr
    return {
        # the neighbour-set split (36 + 4(Ng+Nr+Na)) is fused into the radial descriptor pass,
        # which therefore reads the skin list instead of re-reading the radial list
        "descriptor+MLP": 36 + 4 * (Ng + Nr + Na) + 52 + 4 * Na + 4 * D + 4 * S,
        # fused radial force + angular pair reduction + scatter: the radial-force stage
        # (32+4Nr+4Dr+192) plus the list and f12 reads of the pair reduction (16 Na); the second
        # 192-byte force/virial RMW and 28-byte per-atom read of the separate stage are gone
        "k_force_final": 32 + 4 * Nr + 4 * Dr + 192 + 16 * Na,
        "k_force_angular": 32 + 4 * Na + 4 * Da + 4 * S + 12 * Na,
        "VV1": 128, "PBC": 48, "zero": 104, "displacement_check": 48, "VV2": 80, "thermo": 88,
    }


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.proc = None
        self.lines = []
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(gpu_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append((time.time(), ln.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for t, ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                clk, cmax = float(f[1]), float(f[2])
            except ValueError:
                continue
            mx.append(cmax)
            if t0 - 0.05 <= t <= t1 + 0.05:
                sm.append(clk)
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                      "sw_power_cap"), f[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
        if not sm:  # region shorter than the sampling period: use every sample
            sm = [float(ln.split(",")[1]) for _, ln in self.lines if len(ln.split(",")) >= 9] or [0.0]
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


DUMP_ATOMS = 1 << 18  # 152 bytes each over the five per-atom arrays: 38 MB at most


def dump_outputs(out_dir, atom, thermo):
    """--dump-outputs DIR: the state the timed steps leave to a caller, as float64 .npy files --
    thermo[8] and, for every atom or (above DUMP_ATOMS atoms) a fixed seeded sample of atom indices in
    ascending order, position[3][m], velocity[3][m], force[3][m], potential[m], virial[9][m] (GPUMD's
    per-atom layouts).  Inputs are seeded, so two builds run with the same arguments compare array for
    array."""
    import torch
    n = atom.number_of_atoms
    idx = np.arange(n)
    if n > DUMP_ATOMS:
        idx = np.sort(np.random.default_rng(0).choice(n, DUMP_ATOMS, replace=False))
    idx = torch.as_tensor(idx, device=atom.position_per_atom.device)
    out = {"thermo": thermo}
    for name, rows, t in (("position", 3, atom.position_per_atom), ("velocity", 3, atom.velocity_per_atom),
                          ("force", 3, atom.force_per_atom), ("potential", 1, atom.potential_per_atom),
                          ("virial", 9, atom.virial_per_atom)):
        out[name] = t.view(rows, n).index_select(1, idx).squeeze(0)
    os.makedirs(out_dir, exist_ok=True)
    for name, t in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.double().cpu().numpy())


def crystal(cells, workload="pbte"):
    from gpumd_b200.structures import fcc, init_velocities, rocksalt_pbte
    if workload == "lj":  # config C2: fcc argon, a = 5.30 A, 80 K
        s = fcc(cells, 5.30, rattle=0.0, seed=1)
        s["vel"] = init_velocities(s["mass"], 80.0, seed=42)
        return s
    s = rocksalt_pbte(cells, rattle=0.02, seed=1)
    s["vel"] = init_velocities(s["mass"], 300.0, seed=42)
    return s


def reference_gpu(s, vel, n_gpus, steps, potential=MODEL, symbols=None, ensemble="nve", dt_fs=1.0):
    """The bar north_star names: the UNMODIFIED reference gpumd (oracle/_ref/gpumd_ref, built from
    /root/reference by oracle/Makefile.gpumd_ref) on the same model.xyz / run.in for the same number of
    steps, on the same box, OUTSIDE our timed region; with n_gpus > 1 visible devices it takes its own
    NEP_MULTIGPU path (src/force/force.cu:139-160).  Value = its "Speed of this run" line
    (src/main_gpumd/run.cu:321-326).  Returns None when the binary did not travel to this box."""
    import re
    import shutil
    import tempfile
    from gpumd_b200.structures import nep_type_order, write_xyz
    exe = ROOT / "oracle" / "_ref" / "gpumd_ref"
    if not exe.exists():
        return None
    d = Path(tempfile.mkdtemp(prefix="refgpu_"))
    try:
        t0 = time.time()
        write_xyz(d / "model.xyz", s, symbols or nep_type_order(potential), vel)
        shutil.copyfile(potential, d / "potential.txt")
        (d / "run.in").write_text(f"potential potential.txt\nensemble {ensemble}\ntime_step {dt_fs:g}\n"
                                  f"dump_thermo {max(steps, 1)}\nrun {steps}\n")
        t_write = time.time() - t0
        env = dict(os.environ)
        vis = env.get("CUDA_VISIBLE_DEVICES")
        ids = [x for x in vis.split(",") if x] if vis else [str(k) for k in range(n_gpus)]
        env["CUDA_VISIBLE_DEVICES"] = ",".join(ids[:n_gpus])
        t0 = time.time()
        r = subprocess.run([str(exe)], cwd=d, capture_output=True, text=True, timeout=1500, env=env)
        wall = time.time() - t0
        speed = re.findall(r"Speed of this run = ([0-9.eE+-]+) atom\*step/second", r.stdout)
        tail = [ln.strip() for ln in r.stdout.splitlines() if ln.strip() and not ln.startswith("---")][-6:]
        kind = Path(potential).read_text().split(None, 1)[0]
        if kind.startswith("nep"):
            path = "NEP_MULTIGPU" if n_gpus > 1 else "NEP"
        else:  # only NEP has a multi-GPU path in the reference (force.cu:139-160): one device is used
            path = kind + (" (the reference runs this potential on one GPU)" if n_gpus > 1 else "")
        out = {"value": float(speed[-1]) if speed else None, "unit": "atom-steps/s", "steps": steps,
               "n_gpus": n_gpus, "n_atoms": int(s["type"].shape[0]), "returncode": r.returncode,
               "wall_s": round(wall, 2), "input_write_s": round(t_write, 2),
               "binary": "oracle/_ref/gpumd_ref (unmodified reference, nvcc -O3 -arch=sm_100 -DDEBUG)",
               "path": path, "stdout_tail": tail}
        if r.returncode != 0:
            out["stderr_tail"] = r.stderr[-500:]
        return out
    finally:
        shutil.rmtree(d, ignore_errors=True)


def reference_arm(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path (NEP_CPU, compiled from
    /root/reference into oracle/_ref; falls back to the C restatement if the .so is absent)."""
    if rank != 0:
        return
    from oracle import oracle_py
    threads = os.cpu_count() or 1
    os.environ.setdefault("OMP_NUM_THREADS", str(threads))
    kind = "reference" if oracle_py.ref_available() else "port"
    if kind == "reference":
        eng = oracle_py.RefNepCpu(MODEL)
        call = lambda s: eng.compute(s["type"], s["h"], s["pos"])
    else:
        eng = oracle_py.NepOracle(MODEL)
        call = lambda s: eng.compute(s["type"], s["h"], s["pbc"], s["pos"], precision=32)
        threads = 1
    # calibrate so that K+W steps take about two minutes at most
    probe = crystal(8)  # 4096 atoms
    t0 = time.time()
    call(probe)
    rate = probe["type"].shape[0] / max(time.time() - t0, 1e-6)
    budget_atoms = rate * 120.0 / (args.steps + args.warmup)
    cells = int(max(4, min(16, np.floor((budget_atoms / 8.0) ** (1.0 / 3.0)))))
    s = crystal(cells)
    n = s["type"].shape[0]
    for _ in range(args.warmup):
        call(s)
    t0 = time.time()
    for _ in range(args.steps):
        call(s)
    dt = time.time() - t0
    value = n * args.steps / dt
    sample = f"{cells}^3 cells = {n} atoms of the same rattled PbTe crystal, one force evaluation per step"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "atom-steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "C3: rocksalt PbTe NEP (nep_PbTe.txt), NVE 1 fs; CPU arm: force "
                               "evaluation on a bounded sample", "sample": sample},
        "cpu_baseline": {"value": value, "unit": "atom-steps/s", "cores": threads, "kind": kind,
                         "sample": sample},
        "e2e": {"value": value, "unit": "atom-steps/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
    }))


def cpu_baseline(seconds=15.0):
    from oracle import oracle_py
    threads = os.cpu_count() or 1
    os.environ.setdefault("OMP_NUM_THREADS", str(threads))
    if oracle_py.ref_available():
        kind, eng = "reference", oracle_py.RefNepCpu(MODEL)
        call = lambda s: eng.compute(s["type"], s["h"], s["pos"])
    else:
        kind, eng, threads = "port", oracle_py.NepOracle(MODEL), 1
        call = lambda s: eng.compute(s["type"], s["h"], s["pbc"], s["pos"], precision=32)
    s = crystal(12)  # 13 824 atoms
    n = s["type"].shape[0]
    call(s)
    t0 = time.time()
    reps = 0
    while time.time() - t0 < seconds and reps < 50:
        call(s)
        reps += 1
    dt = time.time() - t0
    return {"value": n * reps / dt, "unit": "atom-steps/s", "cores": threads, "kind": kind,
            "sample": f"{reps} force evaluations of 12^3 cells = {n} atoms (same crystal and model), "
                      f"{dt:.1f} s"}


SIDE = {
    # name: (description, potential file, ensemble, dt fs, T K, heat-current interval)
    "lj": ("C2: fcc Ar, LJ rc 10 A", "lj_Ar_10A.txt", "nve", 5.0, 80.0, 0),
    "unep": ("C4: fcc 16-metal random alloy a=3.9 A, UNEP-v1 (16 types, ZBL), nvt_ber 300 300 100",
             "nep_UNEP_v1.txt", "nvt_ber", 1.0, 300.0, 0),
    "si": ("C5: diamond Si a=5.431 A, Tersoff-1989 (FP64), NVE + heat current every 20 steps",
           "tersoff_Si_1989.txt", "nve", 1.0, 300.0, 20),
}


def side_structure(workload, world, cells):
    from gpumd_b200.structures import diamond, fcc, init_velocities, nep_type_order
    if workload == "lj":
        c = 63 if cells == 50 else cells
        s = fcc((c * world, c, c), 5.30, rattle=0.0, seed=1)
    elif workload == "unep":  # 16 x 126 x 126 cells per GPU = 1 016 064 atoms; 8 GPUs ~ C4's 8 M
        c = (16, 126, 126) if cells == 50 else (cells, cells, cells)
        s = fcc((c[0] * world, c[1], c[2]), 3.9, rattle=0.0, seed=7, num_types=16,
                symbols=nep_type_order(GOLDEN / "nep_UNEP_v1.txt"))
    else:  # si: 16 x 63 x 63 cells per GPU = 508 032 atoms; 4 GPUs ~ C5's 2 M
        c = (16, 63, 63) if cells == 50 else (cells, cells, cells)
        s = diamond((c[0] * world, c[1], c[2]), a=5.431, rattle=0.0, seed=1)
    s["vel"] = init_velocities(s["mass"], SIDE[workload][4], seed=42)
    return s


def side_bench(args, rank, world, local, torch, dist, engine):
    """--workload lj|unep|si: the other BASELINE configs (C2, C4, C5) as secondary lines -- same
    step definition and timing rules as the headline, single GPU or slab domains."""
    from gpumd_b200.structures import TIME_UNIT_CONVERSION
    desc, potfile, ensemble, dt_fs, T0, heat_every = SIDE[args.workload]
    s = side_structure(args.workload, world, args.cells)
    n_global = s["type"].shape[0]
    dt = dt_fs / TIME_UNIT_CONVERSION
    heat = [None]
    if world == 1:
        atom = engine.Atom(s["type"], s["pos"], s["mass"], s["vel"])
        box = engine.Box(s["h"], s["pbc"])
        force = engine.Force()
        pot = force.parse_potential(GOLDEN / potfile, n_global)
        ens = engine.Ensemble_BER(n_global, T0, 100.0) if ensemble == "nvt_ber" else engine.Ensemble_NVE(n_global)
        thermo = torch.zeros(8, dtype=torch.float64, device="cuda")
        fargs = (box, atom.position_per_atom, atom.type, atom.potential_per_atom, atom.force_per_atom,
                 atom.virial_per_atom)
        count = [0]

        def step():
            ens.compute1(dt, box, atom, thermo)
            force.compute(*fargs)
            ens.compute2(dt, box, atom, thermo)
            count[0] += 1
            if heat_every and count[0] % heat_every == 0:
                heat[0] = engine.compute_heat(atom).view(5, n_global).sum(dim=1)

        force.compute(*fargs)
        get_thermo = lambda: thermo.cpu().numpy()
        check = pot.check
        rebuilds = lambda: pot.num_rebuilds
    else:
        # libb200md_mgpu: C++ / CUDA / NCCL domains (slabs along x by default, --grid for blocks)
        from gpumd_b200 import build, mgpu
        if rank == 0:
            build.build_mgpu()
        dist.barrier()
        grid = parse_grid(args.grid, world)
        g = mgpu.DomainGroup(s["h"], s["pbc"], grid, GOLDEN / potfile, ensemble=ensemble, temperature=T0,
                             temperature_coupling=100.0, time_step=dt, skin=DOMAIN_SKIN, distributed=True,
                             cuda_graph=not args.no_graph)
        g.distribute(s["type"], s["pos"], s["mass"], s["vel"])
        count = [0]

        def step():
            g.run(1, 5)
            count[0] += 1
            if heat_every and count[0] % heat_every == 0:
                heat[0] = torch.as_tensor(g.heat_current())

        get_thermo = lambda: g.thermo()
        check = g.check
        rebuilds = lambda: g.info(4, 0)
    del s
    check()
    for _ in range(max(args.warmup, 3)):
        step()
    if world > 1 and heat_every:
        g.heat_current()
    check()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
    r0 = rebuilds()
    if world == 1:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            step()
        e1.record()
        torch.cuda.synchronize()
        ms_dev = e0.elapsed_time(e1)
    else:
        # the module owns its stream: device time from its own CUDA events, heat-current samples
        # (host reads) between the timed chunks
        ms_dev, done = 0.0, 0
        chunk = heat_every if heat_every else args.steps
        while done < args.steps:
            k = min(chunk, args.steps - done)
            ms_dev += g.run_timed(k, 5)
            done += k
            if heat_every and done % heat_every == 0:
                t0 = time.time()
                heat[0] = torch.as_tensor(g.heat_current())
                ms_dev += (time.time() - t0) * 1e3
    ms_t = torch.tensor([ms_dev], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.barrier()
        dist.all_reduce(ms_t, op=dist.ReduceOp.MAX)
    ms = float(ms_t.item())
    check()
    th = get_thermo()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, atom, thermo)
    stage_ms = None
    if world == 1 and hasattr(pot, "profile"):
        pot.profile(True)
        for _ in range(10):
            step()
        stage_ms = {k: round(v[0] / max(v[1], 1), 4) for k, v in pot.profile_read().items()}
        pot.profile(False)
    ref_gpu = None
    if rank == 0 and not args.no_reference_gpu:
        from gpumd_b200.structures import nep_type_order
        if world == 1:
            del atom, force, pot, ens
            torch.cuda.empty_cache()
        s_ref = side_structure(args.workload, world, args.cells)
        sym = {"lj": ["Ar"], "si": ["Si"]}.get(args.workload) or nep_type_order(GOLDEN / potfile)
        ens_line = "nve" if ensemble == "nve" else f"{ensemble} {T0:g} {T0:g} 100"
        ref_gpu = reference_gpu(s_ref, s_ref["vel"], world, args.steps, potential=GOLDEN / potfile,
                                symbols=sym, ensemble=ens_line, dt_fs=dt_fs)
        del s_ref
    if rank == 0:
        print(json.dumps({
            "reference_gpu": ref_gpu,
            "metric": f"atom-steps/sec ({args.workload}, secondary config)", "value": n_global * args.steps / (ms * 1e-3),
            "unit": "atom-steps/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "dtype": "f64" if args.workload == "si" else "f32", "data": "synthetic",
            "config": {"workload": f"{desc}; {n_global} atoms on {world} GPU(s), dt {dt_fs} fs, {ensemble}",
                       "atoms_per_gpu": n_global // world,
                       "list_rebuilds_in_timed_region_rank0": rebuilds() - r0,
                       "final_T_K": float(th[0]), "nep_stage_ms": stage_ms,
                       "heat_current": None if heat[0] is None else [float(v) for v in heat[0].cpu().numpy()]}}))
    if world > 1:
        dist.barrier(group=args.cpu_group)


def parse_grid(spec, world):
    """--grid PxxPyxPz (default: slabs along x, which is also how the weak-scaling crystal grows)."""
    if not spec:
        return (world, 1, 1)
    g = tuple(int(v) for v in spec.lower().split("x"))
    if len(g) != 3 or g[0] * g[1] * g[2] != world:
        raise SystemExit(f"--grid {spec}: need PxxPyxPz with product {world}")
    return g


def ours_multi(args, rank, world, local, torch, dist, engine):
    """N > 1: weak scaling, cells^3 conventional cells (1 M atoms) per GPU.  The whole multi-GPU step
    is libb200md_mgpu (C++ / CUDA / NCCL, include/b200md_mgpu.h): owned-atom integration, staged
    ncclSend/Recv of FP64 ghost positions per force evaluation, 8-double thermo all-reduce, device-side
    displacement-triggered migration; one CUDA graph replay per step."""
    from gpumd_b200 import build, mgpu
    from gpumd_b200.structures import TIME_UNIT_CONVERSION, init_velocities, rocksalt_pbte
    if rank == 0:
        build.build_mgpu()
    dist.barrier()
    grid = parse_grid(args.grid, world)
    cells = tuple(args.cells * g for g in grid)
    s = rocksalt_pbte(cells, rattle=0.02, seed=1)
    vel = init_velocities(s["mass"], 300.0, seed=42)
    n_global = s["type"].shape[0]
    dt = 1.0 / TIME_UNIT_CONVERSION
    cadence = 5  # displacement check (max displacement, all-reduce MAX, one host read) every 5 steps
    # ghost skin 3 A: ghost lists stay valid until some atom has moved 1.05 A (0.7 * skin / 2), which a
    # solid at 300 K never does -- migrations are for diffusing systems; costs ~1 % more ghosts than 1 A
    g = mgpu.DomainGroup(s["h"], s["pbc"], grid, MODEL, time_step=dt, skin=DOMAIN_SKIN, distributed=True,
                         cuda_graph=not args.no_graph)
    g.distribute(s["type"], s["pos"], s["mass"], vel)
    del s, vel
    g.run(max(args.warmup, 3), cadence)
    g.check()
    sampler = ClockSampler(local) if rank == 0 and not os.environ.get("BENCH_NO_SAMPLER") else None
    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()
    mig0 = g.migrations
    w0 = time.time()
    ms = g.run_timed(args.steps, cadence)  # CUDA events on the launching stream, synchronised
    dist.barrier()
    torch.cuda.synchronize()
    w1 = time.time()
    g.check()
    ms_t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    dist.all_reduce(ms_t, op=dist.ReduceOp.MAX)
    ms = float(ms_t.item())
    clocks = sampler.stop(w0, w1) if sampler else None
    launches = g.launches_per_step * args.steps
    th = g.thermo()
    # phase breakdown: untimed extra steps, eager launches with CUDA events between the phases
    g.profile(True)
    h0 = time.time()
    g.run(10, cadence)
    host_ms = (time.time() - h0) * 100.0
    phase_ms = g.profile(False)
    phase_ms["host_per_step_eager"] = host_ms
    loc = torch.tensor([g.info(1, 0), g.info(2, 0)], dtype=torch.float64, device="cuda")
    loc_max = loc.clone()
    dist.all_reduce(loc_max, op=dist.ReduceOp.MAX)

    # end to end: every rank pushes its own local (owned + ghost) system through the host-buffer entry
    ls = g.local_system(0)
    n = ls["type"].shape[0]
    h_type = torch.from_numpy(ls["type"]).pin_memory()
    h_pos = torch.from_numpy(ls["pos"]).pin_memory()
    h_pe = torch.zeros(n, dtype=torch.float64).pin_memory()
    h_f = torch.zeros(3 * n, dtype=torch.float64).pin_memory()
    h_v = torch.zeros(9 * n, dtype=torch.float64).pin_memory()
    pot2 = engine.NEP(MODEL, n)
    box = engine.Box(ls["h"], ls["pbc"])
    for _ in range(2):
        pot2.compute_host(box, h_type, h_pos, h_pe, h_f, h_v)
    torch.cuda.synchronize()
    dist.barrier()
    t0 = time.time()
    e2e_steps = 5
    for _ in range(e2e_steps):
        pot2.compute_host(box, h_type, h_pos, h_pe, h_f, h_v)
    torch.cuda.synchronize()
    e2e_t = torch.tensor([time.time() - t0], dtype=torch.float64, device="cuda")
    dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    ref_gpu = None
    torch.cuda.synchronize()
    if rank == 0 and not args.no_reference_gpu:
        s_ref = rocksalt_pbte(cells, rattle=0.02, seed=1)
        ref_gpu = reference_gpu(s_ref, init_velocities(s_ref["mass"], 300.0, seed=42), world, args.steps)
        del s_ref
    if rank == 0:
        print(json.dumps({
            "metric": METRIC, "value": n_global * args.steps / (ms * 1e-3), "unit": "atom-steps/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {
                "workload": f"C3 x {world}: rocksalt PbTe {cells[0]}x{cells[1]}x{cells[2]} cells = "
                            f"{n_global} atoms, NEP (nep_PbTe.txt), NVE dt 1 fs, 300 K",
                "atoms_per_gpu": n_global // world,
                "parallelism": f"{grid[0]}x{grid[1]}x{grid[2]} block domains (libb200md_mgpu: C++ host, "
                               f"device-side migration, NCCL), owned-atom integration, staged ncclSend/Recv of "
                               f"FP64 ghost positions (halo 2*rc+skin = {16 + DOMAIN_SKIN:g} A) per force call; "
                               f"descriptor work only for ghosts within rc+skin of the owned block; thermo "
                               f"all-reduce per step; displacement check every {cadence} steps "
                               f"({g.migrations - mig0} migrations in the timed region); "
                               f"{'one CUDA-graph replay per step' if not args.no_graph else 'eager launches'}",
                "max_owned": int(loc_max[0].item()), "max_local_with_ghosts": int(loc_max[1].item()),
                "phase_ms_rank0": {k: round(v, 4) for k, v in (phase_ms or {}).items()},
                "cache": "inputs larger than L2; no flush needed",
                "final_T_K": float(th[0]), "final_U_eV_per_atom": float(th[1]) / n_global},
            "clocks": clocks,
            "e2e": {"value": g.info(1, 0) * world * e2e_steps / float(e2e_t.item()), "unit": "atom-steps/s",
                    "h2d_bytes_per_step": int(28 * n), "d2h_bytes_per_step": int(104 * n),
                    "steps": e2e_steps,
                    "what": "per rank: b200md_nep_compute_host on its local (owned+ghost) system, pinned "
                            "host buffers, H2D+D2H inside the timed region; owned atoms x ranks / max time"},
            "gpu_launches": int(launches), "roofline": None, "cpu_baseline": None,
            "reference_gpu": ref_gpu}))
    dist.barrier(group=args.cpu_group)


def ours(args, rank, world):
    import torch
    import torch.distributed as dist
    from gpumd_b200 import build, engine
    from gpumd_b200.structures import TIME_UNIT_CONVERSION

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU fallback)")
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl")
        # host-side barrier for the wait on rank 0's reference-GPU run (an NCCL barrier would spin on
        # the very GPUs the reference is being timed on)
        args.cpu_group = dist.new_group(backend="gloo")
    if rank == 0:
        build.build_lib()
    if world > 1:
        dist.barrier()

    if args.workload != "pbte":
        return side_bench(args, rank, world, local, torch, dist, engine)
    if world > 1:
        return ours_multi(args, rank, world, local, torch, dist, engine)
    s = crystal(args.cells)
    n = s["type"].shape[0]
    atom = engine.Atom(s["type"], s["pos"], s["mass"], s["vel"])
    box = engine.Box(s["h"], s["pbc"])
    force = engine.Force()
    pot = force.parse_potential(MODEL, n)
    ens = engine.Ensemble_NVE(n)
    thermo = torch.zeros(8, dtype=torch.float64, device="cuda")
    dt = 1.0 / TIME_UNIT_CONVERSION
    fargs = (box, atom.position_per_atom, atom.type, atom.potential_per_atom, atom.force_per_atom,
             atom.virial_per_atom)

    def step():
        ens.compute1(dt, box, atom, thermo)
        force.compute(*fargs)
        ens.compute2(dt, box, atom, thermo)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    force.compute(*fargs)  # first force evaluation is outside the loop, like run.cu:217-248
    pot.check()
    for _ in range(max(args.warmup, 3)):
        step()
    pot.check()

    # ---------------- timed region: K steps, state resident in HBM ----------------
    sampler = ClockSampler(local) if rank == 0 else None
    sync_all()
    launches0 = engine.launch_count()
    rebuilds0 = pot.num_rebuilds
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.time()
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    sync_all()
    w1 = time.time()
    ms = e0.elapsed_time(e1)
    launches = engine.launch_count() - launches0
    rebuilds = pot.num_rebuilds - rebuilds0
    clocks = sampler.stop(w0, w1) if sampler else None
    pot.check()
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = n * world * args.steps / (ms * 1e-3)
    t_final = thermo.cpu().numpy()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, atom, thermo)

    if rank != 0:
        if world > 1:
            dist.barrier()
        return

    # ---------------- per-stage device timing for the roofline block ----------------
    prof_steps = min(args.steps, 64)
    pot.profile(True)
    ev = {k: [torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)]
          for k in ("VV1", "force_call", "VV2+thermo")}
    acc = {k: 0.0 for k in ev}
    for _ in range(prof_steps):
        ev["VV1"][0].record(); ens.compute1(dt, box, atom, thermo); ev["VV1"][1].record()
        ev["force_call"][0].record(); force.compute(*fargs); ev["force_call"][1].record()
        ev["VV2+thermo"][0].record(); ens.compute2(dt, box, atom, thermo); ev["VV2+thermo"][1].record()
        torch.cuda.synchronize()
        for k in ev:
            acc[k] += ev[k][0].elapsed_time(ev[k][1])
    stages = pot.profile_read()
    pot.profile(False)
    nn = pot.mean_neighbors()
    per_stage_ms = {k: v[0] / max(v[1], 1) for k, v in stages.items()}
    step_ms_prof = sum(acc.values()) / prof_steps
    model = {"D": pot.dim, "Dr": 5, "S": 120}
    abytes = stage_algorithmic_bytes(nn, model)
    top = max(per_stage_ms, key=per_stage_ms.get)
    key = top if top in abytes else "descriptor+MLP"
    top_ms = per_stage_ms[top] if key == top else sum(
        per_stage_ms.get(k, 0.0) for k in ("k_desc_radial", "k_desc_angular", "k_mlp"))
    peaks_file = ROOT / "MEASURED_PEAKS.json"
    if peaks_file.exists():
        peak, peak_src = json.loads(peaks_file.read_text())["hbm_gbs"], "MEASURED_PEAKS.json hbm_gbs (measured)"
    else:
        peak, peak_src = 6650.0, "B200_PROFILING.md fallback"
    achieved = abytes[key] * n / (top_ms * 1e-3) / 1e9
    traffic = None
    tf = ROOT / "profiles" / "ncu_traffic.json"
    if tf.exists():
        traffic = json.loads(tf.read_text()).get(top)
    ncu_metrics = None
    mf = ROOT / "profiles" / "ncu_metrics.json"
    if mf.exists():  # issue / FMA / L1 utilisation of the same kernel from the committed ncu capture:
        ncu_metrics = json.loads(mf.read_text()).get(top)  # the NEP kernels are not HBM-bound
    total_bytes = sum(abytes.values()) - abytes["descriptor+MLP"] + abytes["descriptor+MLP"]
    roofline = {
        "bound": "hbm", "kernel": top, "achieved": achieved, "peak": peak, "unit": "GB/s",
        "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src, "ncu": ncu_metrics,
        "algorithmic_bytes_per_atom": abytes[key], "kernel_ms": top_ms,
        "step_algorithmic_bytes_per_atom": total_bytes,
        "step_hbm_frac": total_bytes * n / (ms / args.steps * 1e-3) / 1e9 / peak,
        "mean_neighbors": nn,
        "stage_ms": {**{k: round(v, 4) for k, v in per_stage_ms.items()},
                     **{k: round(v / prof_steps, 4) for k, v in acc.items()}},
        "stage_share_of_step": {k: round(v / step_ms_prof, 4) for k, v in per_stage_ms.items()},
    }

    # ---------------- cost of one neighbour rebuild (outside the headline: a 300 K solid does not
    # trigger one in K steps, and neither does the reference, neighbor.cu:741-776) ----------------
    rb = [torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)]
    rebuild_ms = []
    for _ in range(3):
        pot.invalidate(n)  # forget the ordering and lists: the next force call rebuilds everything
        torch.cuda.synchronize()
        rb[0].record(); force.compute(*fargs); rb[1].record()
        torch.cuda.synchronize()
        rebuild_ms.append(rb[0].elapsed_time(rb[1]) - acc["force_call"] / prof_steps)
    neighbor = {
        "rebuild_ms": round(float(np.median(rebuild_ms)), 4),
        "what": "extra device time of a force call that rebuilds cell sort + skin list + type tiles "
                "(median of 3 forced rebuilds) over a force call that reuses them",
        "rebuilds_in_timed_region": rebuilds,
        "steps_per_rebuild_measured": (args.steps / rebuilds) if rebuilds else None,
        "ms_per_step_if_rebuilt_every_20_steps": round(ms / args.steps + float(np.median(rebuild_ms)) / 20.0, 4),
    }

    # ---------------- end to end: host buffers through b200md_nep_compute_host ----------------
    e2e_steps = max(3, min(args.steps, 10))
    h_type = torch.from_numpy(s["type"].copy()).pin_memory()
    h_pos = torch.from_numpy(np.ascontiguousarray(s["pos"]).reshape(-1).copy()).pin_memory()
    h_pe = torch.zeros(n, dtype=torch.float64).pin_memory()
    h_f = torch.zeros(3 * n, dtype=torch.float64).pin_memory()
    h_v = torch.zeros(9 * n, dtype=torch.float64).pin_memory()
    pot2 = engine.NEP(MODEL, n)
    for _ in range(2):
        pot2.compute_host(box, h_type, h_pos, h_pe, h_f, h_v)
    torch.cuda.synchronize()
    t0 = time.time()
    for _ in range(e2e_steps):
        pot2.compute_host(box, h_type, h_pos, h_pe, h_f, h_v)
    torch.cuda.synchronize()
    e2e_dt = time.time() - t0
    e2e = {"value": n * e2e_steps / e2e_dt, "unit": "atom-steps/s",
           "h2d_bytes_per_step": int(h_type.numel() * 4 + h_pos.numel() * 8),
           "d2h_bytes_per_step": int((h_pe.numel() + h_f.numel() + h_v.numel()) * 8),
           "steps": e2e_steps,
           "what": "b200md_nep_compute_host: one full force evaluation per step (wrap-free input), "
                   "pinned host buffers, H2D+D2H inside the timed region; 1 GPU"}
    del pot2

    cpu = cpu_baseline() if not args.no_cpu_baseline else None
    ref_gpu = None
    if not args.no_reference_gpu:
        del atom, force, pot, ens
        torch.cuda.empty_cache()
        ref_gpu = reference_gpu(s, s["vel"], 1, args.steps)
    out = {
        "metric": METRIC, "value": value, "unit": "atom-steps/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {
            "workload": f"C3: rocksalt PbTe {args.cells}^3 cells = {n} atoms per GPU, NEP "
                        "(nep_PbTe.txt, D=30, 30 neurons, rc 8/4 A), NVE dt 1 fs, 300 K",
            "atoms_per_gpu": n, "state": "FP64 positions/velocities/forces (GPUMD layouts), FP32 pair math",
            "cache": "inputs larger than L2 (per-step working set > 1 GB vs 126 MB L2); no flush needed",
            "list_rebuilds_in_timed_region": rebuilds, "parallelism": f"{world} x 1 GPU domain(s)",
            "final_T_K": float(t_final[0]), "final_U_eV_per_atom": float(t_final[1]) / n,
        },
        "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline,
        "cpu_baseline": cpu, "neighbor": neighbor, "reference_gpu": ref_gpu,
    }
    print(json.dumps(out))
    if world > 1:
        dist.barrier()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cells", type=int, default=50, help="conventional cells per edge (50 -> 1M atoms)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--grid", default="", help="multi-GPU block grid PxxPyxPz (default: Nx1x1 slabs)")
    ap.add_argument("--no-graph", action="store_true", help="multi-GPU: eager launches instead of a CUDA graph per step")
    ap.add_argument("--no-reference-gpu", action="store_true",
                    help="skip the run of oracle/_ref/gpumd_ref (the reference on the same GPU) after the bench")
    ap.add_argument("--workload", default="pbte", choices=["pbte", "lj", "unep", "si"],
                    help="pbte = the BASELINE metric (C3); lj / unep / si = secondary lines for C2 / C4 / C5")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write the state they computed as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.dump_outputs and (world > 1 or args.impl != "ours"):
        raise SystemExit("bench.py: --dump-outputs is for single-GPU runs of --impl ours")
    if args.impl == "reference":
        reference_arm(args, rank, world)
    else:
        ours(args, rank, world)


if __name__ == "__main__":
    main()
