#!/usr/bin/env python
"""bench.py -- cell-updates/s of the fused per-level Godunov sweep (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on the host cores

A "step" is one level step of a levelmin=levelmax run: courant_fine -> set_unew -> godunov_fine -> set_uold
(-> ghost exchange -> boundaries), amr/amr_step.f90:326-514.  Default workload: BASELINE.json configs[2], "sedov3d uniform
512^3, HLLC" (namelist/sedov3d.nml with riemann='hllc'), the size north_star quotes its roofline target on; at N=1 the
line also carries configs[1] (256^3, exact Riemann) under "secondary".  With N ranks every rank owns one 512^3 coarse cell
of an (nx,ny,nz) periodic coarse grid holding a copy of the same blast (weak scaling; 1024^3 at N=8), ghost octs exchanged
over NCCL.  After the timed steps the state is compared, bit for bit, with the single-GPU run ("check").
Prints ONE JSON line on rank 0.
"""
import os
os.environ.setdefault("OMP_WAIT_POLICY", "passive")   # CPU baseline: idle OpenMP threads must not spin on a shared host
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GAMMA = 1.4
WORKLOADS = {
    # name: (levelmax per rank cube, riemann, slope_type, ic)
    "sedov3d_256_exact": dict(level=8, riemann="exact", slope_type=1, ic="sedov"),
    "sedov3d_512_hllc": dict(level=9, riemann="hllc", slope_type=1, ic="sedov"),
    "sedov3d_256_hllc": dict(level=8, riemann="hllc", slope_type=1, ic="sedov"),
    "sedov3d_128_hllc": dict(level=7, riemann="hllc", slope_type=1, ic="sedov"),
    "smooth_256_hllc": dict(level=8, riemann="hllc", slope_type=1, ic="smooth"),
    "smooth_256_exact": dict(level=8, riemann="exact", slope_type=1, ic="smooth"),
    "smooth_256_llf": dict(level=8, riemann="llf", slope_type=1, ic="smooth"),
    "sedov3d_128_exact": dict(level=7, riemann="exact", slope_type=1, ic="sedov"),
    "sedov3d_64_exact": dict(level=6, riemann="exact", slope_type=1, ic="sedov"),
    # BASELINE.json configs[4] (M4): namelist/tube_mhd.nml on 256^3, ideal MHD, riemann='roe', riemann2d='llf', slope_type=0
    "tube_mhd_256_roe": dict(level=8, riemann="roe", riemann2d="llf", slope_type=0, ic="tube_mhd", mhd=True),
    "tube_mhd_256_hlld": dict(level=8, riemann="hlld", riemann2d="hlld", slope_type=1, ic="tube_mhd", mhd=True),
    "tube_mhd_128_roe": dict(level=7, riemann="roe", riemann2d="llf", slope_type=0, ic="tube_mhd", mhd=True),
    "tube_mhd_64_roe": dict(level=6, riemann="roe", riemann2d="llf", slope_type=0, ic="tube_mhd", mhd=True),
    # BASELINE.json configs[3]: sedov3d AMR levelmin=7 levelmax=10 (statically nested refinement around the blast, oct-batch kernel)
    "sedov3d_amr_7_10_hllc": dict(level=10, levelmin=7, half_width=16, riemann="hllc", slope_type=1, ic="sedov_centre", amr=True),
    "sedov3d_amr_5_8_hllc": dict(level=8, levelmin=5, half_width=8, riemann="hllc", slope_type=1, ic="sedov_centre", amr=True),
}
MHD_GAMMA = 1.6666667
TUBE_L = (1.0, 0.0, 0.0, 0.0, 2.0, 1.0, 0.0, 0.0)               # namelist/tube_mhd.nml:25-38 (d,u,v,w,P,A,B,C)
TUBE_R = (0.2, 1.186, 2.967, 0.0, 0.1368, 1.0, 1.6405, 0.0)
MHD_BYTES_PER_CELL = 176.0   # 2 * 11 stored variables * 8 B (SURVEY 8d)
BYTES_PER_CELL = 80.0   # algorithmic: read uold once + write unew once = 2*nvar*8 B (SURVEY 8d)
# --dump-outputs: cells of the state sample per workload; the default line runs four workloads: (5+5+11+5) * 8 B * 2^17 = 27 MB
DUMP_CELLS = 1 << 17
DUMP_SEED = 20240611


def dump_outputs(outdir, workload, uold, cells, dts):
    """--dump-outputs: what the timed steps of `workload` hand back to the caller, after the last of them.
    <workload>_state.npy: the conserved state uold[:, c] (float64, [nvar][n]) of a fixed, seeded sample of n <= DUMP_CELLS of the
    active cells `cells` (all of them when fewer); <workload>_dt.npy: the time step of every timed step.  Same arguments, same
    inputs and same sample, so two builds can be compared array for array."""
    os.makedirs(outdir, exist_ok=True)
    cells = np.asarray(cells, dtype=np.int64)
    if len(cells) > DUMP_CELLS:
        cells = cells[np.sort(np.random.default_rng(DUMP_SEED).choice(len(cells), DUMP_CELLS, replace=False))]
    np.save(os.path.join(outdir, f"{workload}_state.npy"), np.ascontiguousarray(uold[:, cells], dtype=np.float64))
    np.save(os.path.join(outdir, f"{workload}_dt.npy"), np.asarray(dts, dtype=np.float64))


def active_cells(a, levels):
    """0-based indices into the ncell axis of uold of the active cells of `levels` (oct order, then the 2^ndim cells)"""
    T = 1 << a.ndim
    return np.concatenate([(a.ncoarse + np.arange(T)[None, :] * a.ngridmax + a.active[l].astype(np.int64)[:, None] - 1).ravel()
                           for l in levels])


def sedov_ic(boxlen, nx, level):
    """namelist/sedov3d.nml:19-34 evaluated like region_condinit (hydro/init_flow_fine.f90:475-596)."""
    scale = boxlen / nx
    dx = 0.5 ** level * scale

    def fn(x, y, z):                      # x,y,z in coarse-cell units
        xs, ys, zs = x * scale, y * scale, z * scale
        r = (np.maximum(1.0 - np.abs(xs) / dx, 0.0) * np.maximum(1.0 - np.abs(ys) / dx, 0.0)
             * np.maximum(1.0 - np.abs(zs) / dx, 0.0))
        p = 1e-5 + 0.4 * r / dx ** 3
        u = np.zeros((5, len(x)))
        u[0] = 1.0
        u[4] = p / (GAMMA - 1.0)
        return u
    return fn


def smooth_ic(nxyz):
    """SURVEY 8d M2b: smooth, everywhere non-trivial periodic state."""
    def fn(x, y, z):
        tw = 2 * np.pi
        xs, ys, zs = x / nxyz[0], y / nxyz[1], z / nxyz[2]
        rho = 1 + 0.2 * np.sin(tw * xs) * np.cos(tw * ys)
        vx, vy, vz = 0.3 * np.sin(tw * ys), 0.3 * np.sin(tw * zs), 0.3 * np.sin(tw * xs)
        p = 1 + 0.1 * np.cos(tw * (xs + ys + zs))
        u = np.zeros((5, len(x)))
        u[0] = rho
        u[1], u[2], u[3] = rho * vx, rho * vy, rho * vz
        u[4] = p / (GAMMA - 1) + 0.5 * rho * (vx ** 2 + vy ** 2 + vz ** 2)
        return u
    return fn


def cpu_reference_run_amr(workload, steps, warmup):
    """AMR workloads on the host cores: the oracle's amr_step (oracle/amr.py driving oracle/ramses_oracle.c, one thread: the
    reference's serial build) on a bounded sample of the same statically nested mesh (levelmin=5, levelmax=8, 16^3-oct cubes)."""
    from oracle.amr import AmrRun
    from ramses_b200.tree import build_nested_tree, cell_centers
    w = WORKLOADS[workload]
    levelmin, levelmax, hw = 5, 8, 8
    a = build_nested_tree(levelmin, levelmax, half_width=hw, boxlen=1.0)
    dxf = 0.5 ** levelmax
    for l in range(levelmin, levelmax + 1):
        ig, cc = cell_centers(a, l)
        for ind in range(8):
            x, y, z = cc[ind][:, 0] - 0.5, cc[ind][:, 1] - 0.5, cc[ind][:, 2] - 0.5
            r = (np.maximum(1.0 - np.abs(x) / dxf, 0.0) * np.maximum(1.0 - np.abs(y) / dxf, 0.0) * np.maximum(1.0 - np.abs(z) / dxf, 0.0))
            u = np.zeros((5, len(x)))
            u[0] = 1.0
            u[4] = (1e-5 + 0.4 * r / dxf ** 3) / (GAMMA - 1.0)
            a.uold[:, a.ncoarse + ind * a.ngridmax + ig - 1] = u
    r = AmrRun(3, levelmin, levelmax, (0,) * 6, 1.0, nsubcycle=[2, 2, 2, 2], ngridmax=a.ngridmax, riemann=w["riemann"],
               slope_type=w["slope_type"], gamma=GAMMA, interpol_type=1, tout=[1e9])
    r.son[1:] = a.son; r.father[1:] = a.father; r.nbor[:, 1:] = a.nbor
    for l in range(1, levelmax + 1):
        r.active[l] = [int(g) for g in a.active[l]]
    r.push_all()
    r.uold[:] = a.uold.ravel()
    for l in range(levelmax - 1, 0, -1):
        r.upload_fine(l)
    r.static = True
    updates = sum(8 * len(a.active[l]) * 2 ** (l - levelmin) for l in range(levelmin, levelmax + 1))
    for _ in range(warmup):
        r.amr_step(levelmin, 1)
    t0 = time.perf_counter()
    for _ in range(steps):
        r.amr_step(levelmin, 1)
    el = time.perf_counter() - t0
    return {"value": updates * steps / el, "unit": "cell-updates/s", "cores": 1, "kind": "port",
            "sample": f"statically nested AMR mesh levelmin={levelmin} levelmax={levelmax} ({(2 * hw) ** 3} octs per refined level), "
                      f"riemann={w['riemann']}, {steps} coarse steps with sub-cycling (1+2+4+8 level steps), the oracle's amr_step "
                      f"(oracle/amr.py + oracle/ramses_oracle.c: godfine1 with interpol_hydro, refluxing, upload_fine), 1 host thread",
            "seconds": el}, el / steps


def amr_bench(args, w, rank, world, local_rank, workload=None, embedded=False):
    """configs[3]: one GPU, AMR mode.  A `step` is one coarse step of amr_step (levelmin .. levelmax with sub-cycling 2 per
    level: 1+2+4+8 level steps), every per-level routine through the C-ABI in the reference's order (hydro.amr_step)."""
    import torch
    from ramses_b200.hydro import HydroGPU, amr_step
    from ramses_b200.tree import build_nested_tree, cell_centers
    if world > 1:
        raise SystemExit("the AMR workloads are single-GPU in this round (multi-rank AMR is covered by tests/mgpu_amr_check.py)")
    levelmin, levelmax = w["levelmin"], w["level"]
    a = build_nested_tree(levelmin, levelmax, half_width=w["half_width"], boxlen=1.0)
    a.gamma, a.courant_factor, a.slope_type, a.riemann = GAMMA, 0.8, w["slope_type"], w["riemann"]
    dxf = 0.5 ** levelmax
    for l in range(levelmin, levelmax + 1):       # sedov3d.nml regions with the point source moved to the box centre
        ig, cc = cell_centers(a, l)
        for ind in range(8):
            x, y, z = cc[ind][:, 0] - 0.5, cc[ind][:, 1] - 0.5, cc[ind][:, 2] - 0.5
            r = (np.maximum(1.0 - np.abs(x) / dxf, 0.0) * np.maximum(1.0 - np.abs(y) / dxf, 0.0) * np.maximum(1.0 - np.abs(z) / dxf, 0.0))
            u = np.zeros((5, len(x)))
            u[0] = 1.0
            u[4] = (1e-5 + 0.4 * r / dxf ** 3) / (GAMMA - 1.0)
            a.uold[:, a.ncoarse + ind * a.ngridmax + ig - 1] = u
    h = HydroGPU(a, device=local_rank, amr_mode=True, interpol_type=1)
    for l in range(1, levelmax + 1):
        h.bind_level(l)
    h.host_register(a.uold)
    h.upload_state(0)
    for l in range(levelmax - 1, 0, -1):
        h.upload_fine(l)
    nsub = [1] * levelmin + [2] * 64     # by level: nsubcycle(levelmin:) = 2 as in the reference's default (amr/read_params.f90)
    dtnew = {l: 0.0 for l in range(0, levelmax + 2)}
    dtold = {l: 0.0 for l in range(0, levelmax + 2)}
    ncell = {l: 8 * len(a.active[l]) for l in range(levelmin, levelmax + 1)}
    updates = sum(ncell[l] * 2 ** (l - levelmin) for l in ncell)
    launches0 = lambda: sum(h.level_info(l).kernel_launches for l in range(1, levelmax + 1))
    steps, warmup = args.steps, max(args.warmup, 3)
    h.amr_steps(levelmin, nsub, warmup)
    h.synchronize(); torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    sampler.start(); time.sleep(0.3)
    l0 = launches0()
    h.synchronize(); torch.cuda.synchronize()
    t0 = time.perf_counter()
    dts = h.amr_steps(levelmin, nsub, steps)  # rgpu_amr_steps: time steps stay on the device, one host sync at the end
    h.synchronize(); torch.cuda.synchronize()
    wall_host = time.perf_counter() - t0
    wall = h.level_info(levelmin).last_steps_ms * 1e-3      # CUDA events on the launching stream around the K coarse steps
    launches = launches0() - l0
    clocks = sampler.stop()
    if args.dump_outputs:
        initial = a.uold.copy()           # the end-to-end pass below starts from the initial state, as without the dump
        h.download_state(0)
        dump_outputs(args.dump_outputs, workload or args.workload, a.uold, active_cells(a, range(levelmin, levelmax + 1)), dts)
        a.uold[:] = initial
    # end to end: host arrays in, host arrays out around every coarse step
    t0 = time.perf_counter()
    for _ in range(args.e2e_steps):
        h.upload_state(0)
        amr_step(h, levelmin, 1, levelmin, nsub, dtnew, dtold)
        h.download_state(0)
    h.synchronize()
    e2e_t = time.perf_counter() - t0
    nbytes = a.uold.nbytes
    h.finalize()
    peaks_file = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak = json.load(open(peaks_file))["hbm_gbs"] if os.path.exists(peaks_file) else 6650.0
    achieved = BYTES_PER_CELL * updates / (wall / steps) / 1e9
    line = {"metric": "cell_updates_per_s", "value": updates * steps / wall, "unit": "cell-updates/s", "n_gpus": 1, "steps": steps,
            "warmup": warmup, "ms_per_step": wall / steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload or args.workload, "levelmin": levelmin, "levelmax": levelmax, "cells_per_level": ncell,
                       "level_steps_per_coarse_step": {l: 2 ** (l - levelmin) for l in ncell}, "riemann": w["riemann"],
                       "mesh": "static nested refinement (ramses_b200.tree.build_nested_tree), periodic box",
                       "timing": "CUDA events on the launching stream around K coarse steps of rgpu_amr_steps (device-resident time steps)",
                       "wall_ms_per_step": wall_host / steps * 1e3,
                       "l2": "state %.2f GB vs 126 MB L2" % (nbytes / 1e9)},
            "clocks": clocks, "gpu_launches": int(launches),
            "e2e": {"value": updates * args.e2e_steps / e2e_t, "unit": "cell-updates/s", "h2d_bytes_per_step": int(nbytes),
                    "d2h_bytes_per_step": int(nbytes), "steps": args.e2e_steps,
                    "api": "rgpu_upload_state + amr_step order of per-level rgpu_* calls + rgpu_download_state"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                         "kernel": "whole coarse step (amr_godfine_kernel + reflux + list passes)", "kernel_ms": wall / steps * 1e3,
                         "algorithmic_bytes_per_launch": BYTES_PER_CELL * updates},
            "cpu_baseline": None}
    if not args.no_cpu_baseline and not embedded:
        try:
            cb, _ = cpu_reference_run_amr(workload or args.workload, 2, 1)
            cb.pop("seconds", None)
            line["cpu_baseline"] = cb
        except Exception as e:
            line["cpu_baseline"] = {"error": repr(e)}
    if embedded:
        return line
    print(json.dumps(line))
    return 0


def tube_mhd_ic(x_lo, x_mid, x_hi):
    """namelist/tube_mhd.nml INIT_PARAMS: two 'square' regions spanning y,z (mhd/condinit.f90); x in coarse-cell units.
    Cells outside [x_lo, x_hi) (periodic multi-rank variant) repeat the pattern."""
    def fn(x, y, z):
        left = ((x - x_lo) % (x_hi - x_lo)) < (x_mid - x_lo)
        u = np.zeros((11, len(x)))
        for sel, st in ((left, TUBE_L), (~left, TUBE_R)):
            d, vx, vy, vz, P, A, B, Cc = st
            u[0][sel] = d
            u[1][sel], u[2][sel], u[3][sel] = d * vx, d * vy, d * vz
            u[5][sel] = A; u[8][sel] = A
            u[6][sel] = B; u[9][sel] = B
            u[7][sel] = Cc; u[10][sel] = Cc
            u[4][sel] = P / (MHD_GAMMA - 1.0) + 0.5 * d * (vx * vx + vy * vy + vz * vz) + 0.5 * (A * A + B * B + Cc * Cc)
        return u
    return fn


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            pass
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) >= 9:
                for i, nm in enumerate(names):
                    if r[5 + i].lower().startswith("active"):
                        reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_reference_run(workload, steps, warmup, sample_level=None, budget_s=60.0):
    """The reference algorithm on the host cores: oracle/ (C restatement of RAMSES, reference-shaped per-oct
    6^3 patches, nvector=32 batches, OpenMP over batches, gcc -O3 as BASELINE.md states).  The F90 itself cannot be built
    (no gfortran/MPI).  Thread count: the host threads this process may run on, at most 64 (more does not scale on these
    shared hosts; recorded in `cores`).  Grid: the workload's own grid when warmup+steps steps of it fit `budget_s` seconds
    at the rate measured on a 64^3 probe, else the next smaller power of two (`sample` says which)."""
    from oracle import orc
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from helpers import SEDOV3D_REGIONS, smooth_state
    w = WORKLOADS[workload]
    if w.get("mhd"):
        return cpu_reference_run_mhd(workload, steps, warmup, sample_level=6)
    if w.get("amr"):
        return cpu_reference_run_amr(workload, steps, warmup)
    p = orc.make_params(ndim=3, riemann=w["riemann"], slope_type=w["slope_type"], boxlen=0.5, gamma=GAMMA,
                        courant_factor=0.8)

    def setup(level):
        m = orc.Mesh(3, level, order=0)
        u = m.new_state(5)
        if w["ic"] == "sedov":
            orc.condinit_regions(p, m, level, u, SEDOV3D_REGIONS)
        else:
            m.dense_to_level(smooth_state(3, 1 << level), u, level, 5)
        return m, u
    nmax = host_threads()
    nthr = min(nmax, 64)
    mc, uc = setup(6)
    orc.run_uniform(p, mc, 6, 1, uc, nthreads=nthr)
    t0 = time.perf_counter()
    orc.run_uniform(p, mc, 6, 3, uc, nthreads=nthr)
    rate = 3 * 64 ** 3 / (time.perf_counter() - t0)
    if sample_level is None:
        sample_level = w["level"]
        try:
            import psutil
            avail = psutil.virtual_memory().available
        except Exception:
            avail = 64e9
        while sample_level > 6 and ((steps + warmup) * 8 ** sample_level / rate > budget_s or 8 ** sample_level * 40 * 4 > 0.5 * avail):
            sample_level -= 1
    m, u = setup(sample_level)
    ncell = (1 << sample_level) ** 3
    if warmup:
        orc.run_uniform(p, m, sample_level, warmup, u, nthreads=nthr)
    t0 = time.perf_counter()
    orc.run_uniform(p, m, sample_level, steps, u, nthreads=nthr)
    el = time.perf_counter() - t0
    n = 1 << sample_level
    return {"value": ncell * steps / el, "unit": "cell-updates/s", "cores": nthr, "kind": "port",
            "same_grid_as_gpu_arm": sample_level == w["level"],
            "sample": f"{w['ic']} {n}^3 periodic, riemann={w['riemann']}, {steps} level steps "
                      f"(courant_fine+set_unew+godunov_fine+set_uold), C restatement of the RAMSES algorithm "
                      f"(oracle/ramses_oracle.c, gcc -O3 -ffp-contract=off, OpenMP over nvector=32 oct batches); "
                      f"{nthr} of {nmax} host threads",
            "seconds": el}, el / steps


def cpu_reference_run_mhd(workload, steps, warmup, sample_level=6):
    """MHD workloads: oracle/ramses_oracle_mhd.c (per-oct 6^3 patches like mag_unsplit, OpenMP over octs)."""
    from oracle import orc
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from helpers import mhd_tube_state
    w = WORKLOADS[workload]
    p = orc.make_mhd_params(slope_type=w["slope_type"], riemann=w["riemann"], riemann2d=w["riemann2d"], gamma=MHD_GAMMA,
                            courant_factor=0.8, boxlen=2.0)

    def setup(level):
        m = orc.Mesh(3, level, (2, 2, 0, 0, 0, 0), 0, 1)
        u = m.new_state(11)
        n = 1 << level
        m.dense_to_level(mhd_tube_state(n, TUBE_L, TUBE_R, 1.0, 2.0, MHD_GAMMA), u, level, 11)
        return m, u
    nmax = host_threads()
    cands = sorted({min(nmax, c) for c in (8, 16, 32, 64, 128, nmax)})
    mc, uc = setup(5)
    best, best_rate = cands[0], 0.0
    for c in cands:
        orc.mhd_run_uniform(p, mc, 5, 1, uc, nthreads=c)
        t0 = time.perf_counter()
        orc.mhd_run_uniform(p, mc, 5, 2, uc, nthreads=c)
        rate = 2 * 32 ** 3 / (time.perf_counter() - t0)
        if rate > best_rate:
            best, best_rate = c, rate
    nthr = best
    m, u = setup(sample_level)
    n = 1 << sample_level
    if warmup:
        orc.mhd_run_uniform(p, m, sample_level, warmup, u, nthreads=nthr)
    t0 = time.perf_counter()
    orc.mhd_run_uniform(p, m, sample_level, steps, u, nthreads=nthr)
    el = time.perf_counter() - t0
    return {"value": n ** 3 * steps / el, "unit": "cell-updates/s", "cores": nthr, "kind": "port",
            "sample": f"tube_mhd {n}^3 (x zero-gradient, y/z periodic), riemann={w['riemann']}, riemann2d={w['riemann2d']}, "
                      f"slope_type={w['slope_type']}, {steps} level steps (courant_fine+set_unew+godunov_fine+set_uold+"
                      f"make_boundary_hydro), C restatement of the RAMSES MHD algorithm (oracle/ramses_oracle_mhd.c, gcc -O2 "
                      f"-ffp-contract=off, OpenMP over octs); {nthr} of {nmax} host threads (fastest of a calibration sweep)",
            "seconds": el}, el / steps


def pin_to_gpu_numa_node(gpu_index):
    """Bind this process to the CPUs local to its GPU (NVML affinity) BEFORE the host arrays are allocated: first-touch then
    places them on the GPU's NUMA node and the pinned H2D/D2H copies of the Level-0 call do not cross the socket interconnect."""
    try:
        import pynvml
        pynvml.nvmlInit()
        hdl = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(hdl, (ncpu + 63) // 64)
        cpus = {w * 64 + b for w, m in enumerate(words) for b in range(64) if (m >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def canonical_check(a, level, coarse, rank, dts, keep_block=False):
    """Size-independent identity of the run: SHA-1 of the dt history and of the conserved state in the two bottom and two top
    oct planes of the rank's cube (all eight corners: where the periodic images of the blast arrive through the ghost exchange),
    in (z, y, x, cell, variable) order -- independent of the oct numbering and of the decomposition.  Every rank holds the same
    periodic problem (the blast is replicated in every coarse cell), so all ranks of an N-GPU run and the single-GPU run must
    produce the SAME hash: bench.py compares with tests/golden/bench_hashes.json (written by a single-GPU run)."""
    import hashlib
    pos = a._pos[level]
    ig0 = a._igrid0[level]
    ig = a.active[level].astype(np.int64)
    n1 = 1 << (level - 1)
    nx, ny = coarse[0], coarse[1]
    myc = np.array([rank % nx, (rank // nx) % ny, rank // (nx * ny)], dtype=np.int64)
    pl = pos[ig - ig0] - myc[None, :] * n1
    sel = (pl[:, 2] < 2) | (pl[:, 2] >= n1 - 2)
    pl, igs = pl[sel], ig[sel]
    order = np.lexsort((pl[:, 0], pl[:, 1], pl[:, 2]))
    igs = igs[order]
    T = a.twotondim
    cells = (a.ncoarse + np.arange(T)[None, :] * a.ngridmax + igs[:, None] - 1).ravel()
    blk = np.ascontiguousarray(a.uold[:, cells].T)
    act = (a.ncoarse + np.arange(T)[:, None] * a.ngridmax + ig[None, :] - 1).ravel()
    out = {"state_sha1": hashlib.sha1(blk.tobytes()).hexdigest(), "dt_sha1": hashlib.sha1(np.asarray(dts).tobytes()).hexdigest(),
           "mass_sum": float(a.uold[0, act].sum()), "etot_sum": float(a.uold[a.ndim + 1, act].sum()), "cells_hashed": int(len(cells))}
    if keep_block:
        out["_block"] = blk
    return out


GOLDEN_HASHES = os.path.join(ROOT, "tests", "golden", "bench_hashes.json")


def dense_bench(args, workload, rank, world, local_rank, secondary=False):
    """One levelmin=levelmax workload on `world` GPUs (one cube of 2^level cells per rank).  Returns the JSON line (rank 0) or None."""
    import torch
    from ramses_b200.hydro import HydroGPU
    from ramses_b200.tree import build_uniform_tree, coarse_dims_for_ranks, fill_state
    dist = None
    if world > 1:
        import torch.distributed as dist
    w = WORKLOADS[workload]
    steps, warmup = args.steps, max(args.warmup, 3)
    level = w["level"]
    coarse = coarse_dims_for_ranks(3, world)
    mhd = bool(w.get("mhd"))
    nvs = 11 if mhd else 5
    bpc = MHD_BYTES_PER_CELL if mhd else BYTES_PER_CELL
    t_setup = time.perf_counter()
    if mhd:
        # single rank: the namelist's own box (x zero-gradient boundaries, boxlen=2); several ranks: the periodic
        # image of the same tube (one coarse cell per rank, no physical boundary) -- same work per cell
        boxlen = 2.0
        xb = (2, 2) if world == 1 else None
        a = build_uniform_tree(3, level, coarse=coarse, myid=rank + 1, ncpu=world, order=args.order, boxlen=boxlen, mhd=True, xbound=xb)
        a.gamma, a.courant_factor, a.slope_type, a.riemann, a.riemann2d = MHD_GAMMA, 0.8, w["slope_type"], w["riemann"], w["riemann2d"]
        fill_state(a, level, tube_mhd_ic(1.0, 1.5, 2.0) if world == 1 else tube_mhd_ic(0.0, 0.5 * coarse[0], float(coarse[0])))
    else:
        # every rank owns one coarse cell = one copy of the namelist's box (boxlen 0.5 per coarse cell, so dx does not depend on
        # N); the initial condition is replicated in every coarse cell: N copies of the same periodic problem (weak scaling)
        boxlen = 0.5 * coarse[0]
        a = build_uniform_tree(3, level, coarse=coarse, myid=rank + 1, ncpu=world, order=args.order, boxlen=boxlen)
        a.gamma, a.courant_factor, a.slope_type, a.riemann = GAMMA, 0.8, w["slope_type"], w["riemann"]
        base = sedov_ic(0.5, 1, level) if w["ic"] == "sedov" else smooth_ic((1, 1, 1))
        fill_state(a, level, lambda x, y, z: base(np.mod(x, 1.0), np.mod(y, 1.0), np.mod(z, 1.0)))
    t_setup = time.perf_counter() - t_setup
    h = HydroGPU(a, device=local_rank)
    if world > 1:
        uid = torch.zeros(128, dtype=torch.uint8)
        from ramses_b200 import lib as _l
        if rank == 0:
            buf = (C.c_ubyte * 128)()
            _l.check(h.L.rgpu_comm_unique_id(buf))
            uid = torch.tensor(list(buf), dtype=torch.uint8)
        uid = uid.cuda()
        dist.broadcast(uid, 0)
        buf = (C.c_ubyte * 128)(*uid.cpu().tolist())
        _l.check(h.L.rgpu_comm_init(world, rank, buf))
    h.bind_level(level)
    info0 = h.level_info(level)
    assert info0.dense == 1
    h.host_register(a.uold)
    h.host_register(a.unew)
    h.upload_state(level)
    ncell_rank = len(a.active[level]) * 8
    ncell_total = ncell_rank * world

    def barrier():
        h.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # warm-up
    dts_w, _ = h.level_steps(level, warmup)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    l0 = h.level_info(level).kernel_launches
    barrier()
    t0 = time.perf_counter()
    dts, _ = h.level_steps(level, steps)
    barrier()
    wall = time.perf_counter() - t0
    dev_ms = h.level_info(level).last_steps_ms      # CUDA events on the launching stream
    launches = h.level_info(level).kernel_launches - l0
    clocks = sampler.stop() if rank == 0 else None
    t_dev = dev_ms * 1e-3
    if world > 1:
        tt = torch.tensor([t_dev, wall], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t_dev, wall = tt.tolist()
    value = ncell_total * steps / t_dev

    # ---- correctness inside the bench: the state after warmup+steps level steps must be the single-GPU state, bit for bit
    h.download_state(level)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, workload, a.uold, active_cells(a, [level]), dts)
    check = None
    if not mhd:
        check = canonical_check(a, level, coarse, rank, np.concatenate([dts_w, dts]), keep_block=True)
        strict_block = check.pop("_block")
        key = f"{workload}:{warmup + steps}"
        gold = json.load(open(GOLDEN_HASHES)) if os.path.exists(GOLDEN_HASHES) else {}
        g = gold.get(key)
        check["golden_key"] = key
        ok = None if g is None else (g["state_sha1"] == check["state_sha1"] and g["dt_sha1"] == check["dt_sha1"])
        if world > 1:
            mine = torch.tensor([int(check["state_sha1"][:15], 16), int(check["dt_sha1"][:15], 16), -1 if ok is None else int(ok)],
                                dtype=torch.int64, device="cuda")
            allh = [torch.zeros_like(mine) for _ in range(world)]
            dist.all_gather(allh, mine)
            allh = torch.stack(allh).cpu().numpy()
            check["all_ranks_same_bits"] = bool((allh[:, :2] == allh[0, :2]).all())
            ok = None if (allh[:, 2] < 0).any() else bool(allh[:, 2].all())
        check["equals_single_gpu_golden"] = ok
        if args.write_golden and world == 1:
            gold[key] = {k: check[k] for k in ("state_sha1", "dt_sha1", "mass_sum", "etot_sum", "cells_hashed")}
            json.dump(gold, open(GOLDEN_HASHES, "w"), indent=1, sort_keys=True)

    # kernel-only roofline: average duration of the sweep kernel, CUDA events around each launch
    h.set_timing(True)
    ks = []
    for _ in range(5):
        h.level_steps(level, 1)
        ks.append(h.level_info(level).last_sweep_ms)
    h.set_timing(False)
    k_ms = float(np.mean(ks))
    peaks_file = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_file):
        peak, peak_src = json.load(open(peaks_file))["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    achieved = bpc * ncell_rank / (k_ms * 1e-3) / 1e9
    prof = {}
    pf = os.path.join(ROOT, "profiles", "kernel_counters.json")
    if os.path.exists(pf):
        prof = json.load(open(pf)).get(workload, {})
    traffic = prof.get("dram_bytes_per_launch")
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "kernel": ("MHD sweep: 6 kernels (prim, efield, trace, flux<%s>, emf<%s>, update)" % (w["riemann"], w["riemann2d"]))
                if mhd else "%s<3,%s>" % ("sweep3_kernel" if info0.sweep_variant else "sweep_dense_kernel", w["riemann"]),
                "kernel_ms": k_ms, "algorithmic_bytes_per_launch": bpc * ncell_rank, "peak_source": peak_src,
                "note": "FP64 issue rate, not HBM, is the binding roof for this kernel (DESIGN.md); see roofline.fp64"
                        + ("; kernel_ms spans the six passes of the sweep, traffic is the dominant pass (flux)" if mhd else "")}
    if prof.get("fp64_thread_instr_per_cell"):
        # second roof (SURVEY 8d): FP64-pipe instructions per cell-update from the ncu capture of this build (profiles/
        # kernel_counters.json: DADD+DMUL+DFMA thread instructions / cells) against the measured DFMA issue peak of a B200
        ipc = prof["fp64_thread_instr_per_cell"]
        pk = prof.get("fp64_peak_thread_instr_per_s", 16.7e12)
        ach = ipc * ncell_rank / (k_ms * 1e-3)
        roofline["fp64"] = {"instr_per_cell": ipc, "achieved_instr_s": ach, "peak_instr_s": pk, "frac": ach / pk,
                            "source": prof.get("source"), "peak_source": "profiles/microbench/fp64_latency_b200.txt (DFMA, ILP 8, 32 warps/SM)"}

    # end-to-end through the reference-facing call godunov_fine(ilevel) on HOST arrays (H2D + sweep + D2H per step)
    a.dtnew[level] = float(dts[-1])      # a CFL-limited dt of this run
    a.unew[:, :] = a.uold                # boundary / ghost cells of the second host array hold valid states too
    info = h.level_info(level)
    gspan = info.nslot        # contiguous igrid window of the level on this rank

    def time_e2e(nrep):
        h.godunov_fine(level)           # warm
        barrier()
        t0 = time.perf_counter()
        for _ in range(nrep):
            h.godunov_fine(level)
            a.uold, a.unew = a.unew, a.uold
        barrier()
        el = time.perf_counter() - t0
        if world > 1:
            tt = torch.tensor([el], dtype=torch.float64, device="cuda")
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            el = tt.item()
        return ncell_total * nrep / el
    e2e_v = time_e2e(args.e2e_steps)
    e2e = {"value": e2e_v, "unit": "cell-updates/s",
           "h2d_bytes_per_step": int(nvs * 8 * gspan * 8), "d2h_bytes_per_step": int(nvs * 8 * ncell_rank),
           "steps": args.e2e_steps, "api": "rgpu_godunov_fine(ilevel, dt, uold_host, unew_host), pinned host arrays",
           "pipeline_slabs": int(info.pipeline_slabs),
           "mode": ("three-stream z-slab pipeline (H2D | gather+sweep+scatter | D2H), oct numbering '%s'" % args.order)
           if info.pipeline_slabs else "serial H2D -> sweep -> D2H (oct numbering '%s' scatters z-slabs over the igrid window)" % args.order}
    if info.pipeline_slabs and not secondary:
        h.set_pipeline(False)           # what the same call costs when the numbering does not allow the pipeline
        e2e["serial_order_value"] = time_e2e(max(2, args.e2e_steps // 2))
        h.set_pipeline(True)

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and not secondary:
        try:
            cpu_baseline, _ = cpu_reference_run(workload, 2, 1, budget_s=45.0)
            cpu_baseline.pop("seconds", None)
        except Exception as e:      # the checker is optional for the measurement
            cpu_baseline = {"error": repr(e)}
    h.host_unregister(a.uold)
    h.host_unregister(a.unew)
    h.finalize()
    # ---- FAST arithmetic mode (rgpu_params.fast = 1) on the same workload: reported next to the strict headline, never as it
    fast = None
    if not mhd and not args.no_fast:
        a.uold[:, :] = 0.0
        base = sedov_ic(0.5, 1, level) if w["ic"] == "sedov" else smooth_ic((1, 1, 1))
        fill_state(a, level, lambda x, y, z: base(np.mod(x, 1.0), np.mod(y, 1.0), np.mod(z, 1.0)))
        a.fast = True
        hf = HydroGPU(a, device=local_rank)
        if world > 1:
            from ramses_b200 import lib as _l
            uid = torch.zeros(128, dtype=torch.uint8)
            if rank == 0:
                buf = (C.c_ubyte * 128)()
                _l.check(hf.L.rgpu_comm_unique_id(buf))
                uid = torch.tensor(list(buf), dtype=torch.uint8)
            uid = uid.cuda()
            dist.broadcast(uid, 0)
            buf = (C.c_ubyte * 128)(*uid.cpu().tolist())
            _l.check(hf.L.rgpu_comm_init(world, rank, buf))
        hf.bind_level(level)
        hf.upload_state(level)
        fw, _ = hf.level_steps(level, warmup)
        hf.synchronize()
        if world > 1:
            dist.barrier()
        fd, _ = hf.level_steps(level, steps)
        f_ms = hf.level_info(level).last_steps_ms
        if world > 1:
            tt = torch.tensor([f_ms], dtype=torch.float64, device="cuda")
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            f_ms = tt.item()
        hf.download_state(level)
        hf.finalize()
        a.fast = False
        fb = canonical_check(a, level, coarse, rank, np.concatenate([fw, fd]), keep_block=True)["_block"]
        scale = np.abs(strict_block).max(axis=0, keepdims=True)
        scale[scale == 0] = 1.0
        rel = float((np.abs(fb - strict_block) / scale).max())
        fast = {"value": ncell_total * steps / (f_ms * 1e-3), "unit": "cell-updates/s", "ms_per_step": f_ms / steps,
                "max_rel_diff_vs_strict": rel, "tolerance": 1e-12, "within_tolerance": rel <= 1e-12,
                "what": "rgpu_params.fast = 1: FMA contraction, reciprocal-multiply quotients, <= 2 ulp reciprocal / sqrt in the 3-D dense "
                        "sweep; difference on the hashed planes of the conserved state after warmup+steps level steps, per variable maximum"}
    if rank != 0:
        return None
    n = 1 << level
    line = {"metric": "cell_updates_per_s", "value": value, "unit": "cell-updates/s", "n_gpus": world,
            "steps": steps, "warmup": warmup, "ms_per_step": t_dev / steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload, "grid_per_gpu": f"{n}^3", "global_grid":
                       f"{n * coarse[0]}x{n * coarse[1]}x{n * coarse[2]}", "riemann": w["riemann"], "riemann2d": w.get("riemann2d"),
                       "slope_type": w["slope_type"], "decomposition": f"{coarse[0]}x{coarse[1]}x{coarse[2]} coarse cells, one per rank, "
                       "initial condition replicated per coarse cell",
                       "oct_order": args.order, "sweep_variant": int(info0.sweep_variant), "host_setup_s": round(t_setup, 1),
                       "l2": "inputs larger than L2 (state %.2f GB per rank vs 126 MB L2), no flush" % (nvs * 8 * ncell_rank / 1e9)},
            "wall_ms_per_step": wall / steps * 1e3, "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
            "roofline": roofline, "cpu_baseline": cpu_baseline, "check": check, "fast": fast}
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS))
    ap.add_argument("--secondary", default="sedov3d_256_exact", help="second workload reported under 'secondary' at N=1 ('' = none)")
    ap.add_argument("--config5", default="tube_mhd_256_roe", help="MHD workload (BASELINE.json configs[4]) reported under 'config5' at N=1 ('' = none)")
    ap.add_argument("--config4", default="sedov3d_amr_7_10_hllc", help="AMR workload (BASELINE.json configs[3]) reported under 'config4' at N=1 ('' = none)")
    ap.add_argument("--e2e-steps", type=int, default=4)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-fast", action="store_true", help="skip the FAST-arithmetic re-run of the workload")
    ap.add_argument("--order", default="lattice", choices=["lattice", "creation", "random"],
                    help="oct numbering of the fabricated tree; 'creation' = the reference's refine order (nvector = infinity)")
    ap.add_argument("--write-golden", action="store_true", help="single-GPU run: record the state / dt hashes in tests/golden/bench_hashes.json")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps of each workload, write a fixed sample of the state they computed and their time "
                         "steps as DIR/<workload>_{state,dt}.npy (rank 0)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the CUDA path computed (--impl ours)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    default_workload = args.workload is None
    if default_workload:
        # BASELINE.json configs[2]: sedov3d uniform 512^3, HLLC -- the size north_star's roofline target is quoted on.  It needs
        # ~14 GB of host memory per rank (two state arrays + the tree); fall back to 256^3 per GPU when the box is short of it
        args.workload = "sedov3d_512_hllc"
        try:
            import psutil
            if psutil.virtual_memory().available < 20e9 * max(world, 1):
                args.workload = "sedov3d_256_hllc"
        except Exception:
            pass
    w = WORKLOADS[args.workload]
    steps, warmup = args.steps, max(args.warmup, 3)

    # ------------------------------------------------------------------ reference arm (host cores, rank 0 only)
    if args.impl == "reference":
        if rank != 0:
            return 0
        cb, sec_per_step = cpu_reference_run(args.workload, steps, warmup, budget_s=150.0)
        line = {"impl": "reference", "metric": "cell_updates_per_s", "value": cb["value"], "unit": "cell-updates/s",
                "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": sec_per_step * 1e3,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": args.workload, "note": "each step is a bounded sample of the workload (cpu_baseline.sample)"},
                "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "e2e": {"value": cb["value"], "unit": "cell-updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------ our arm
    ncpus_bound = pin_to_gpu_numa_node(local_rank)
    import torch
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if w.get("amr"):
        return amr_bench(args, w, rank, world, local_rank)
    line = dense_bench(args, args.workload, rank, world, local_rank)
    if line is not None:
        line["config"]["host_cpus_bound"] = ncpus_bound
    if world == 1 and default_workload and args.secondary and args.secondary != args.workload:
        try:      # BASELINE.json configs[1] next to the headline workload (same process, N=1 only)
            sec = dense_bench(args, args.secondary, rank, world, local_rank, secondary=True)
            line["secondary"] = {k: sec[k] for k in ("value", "unit", "ms_per_step", "roofline", "e2e", "check", "gpu_launches", "fast")}
            line["secondary"]["config"] = sec["config"]
        except Exception as e:
            line["secondary"] = {"error": repr(e)}
    if world == 1 and default_workload and args.config5:
        try:      # BASELINE.json configs[4]: tube_mhd 256^3, 8-wave MHD path (roe / llf), same process
            sec = dense_bench(args, args.config5, rank, world, local_rank, secondary=True)
            line["config5"] = {k: sec[k] for k in ("value", "unit", "ms_per_step", "roofline", "e2e", "gpu_launches")}
            line["config5"]["config"] = sec["config"]
        except Exception as e:
            line["config5"] = {"error": repr(e)}
    if world == 1 and default_workload and args.config4:
        try:      # BASELINE.json configs[3]: sedov3d AMR levelmin=7 levelmax=10 (one GPU), same process
            sec = amr_bench(args, WORKLOADS[args.config4], rank, world, local_rank, workload=args.config4, embedded=True)
            line["config4"] = {k: sec[k] for k in ("value", "unit", "ms_per_step", "roofline", "e2e", "gpu_launches", "config")}
        except Exception as e:
            line["config4"] = {"error": repr(e)}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    failed = line is not None and line.get("check") and line["check"].get("equals_single_gpu_golden") is False
    return 1 if failed else 0


if __name__ == "__main__":
    sys.exit(main())
