#!/usr/bin/env python
"""bench.py -- MLUPS (fp64 D2Q9) of the B200 collide-stream path, with roofline and CPU baseline.

Contract (one JSON line on stdout from rank 0):
  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload NAME] [--dump-outputs DIR]
  N > 1 is launched by torchrun, one rank per GPU (RANK / LOCAL_RANK / WORLD_SIZE / MASTER_* from
  the environment); each rank owns one x-slab, the halo of a pass is stored into the neighbouring
  GPU's memory by the step kernel itself (CUDA IPC peer memory over NVLink; NCCL where unavailable).

A "step" is one lattice update of the whole channel = one pass of Solver::run's loop body
(reference include/LBMSolver.h:48-64): fused pull + boundary + collide, halo exchange, stability
flag, and on every output_frequency-th step the momentum-exchange reduction.  The default kernels
do THREE such steps per launch and per trip through HBM (temporal blocking, csrc/lbm_tb.cuh).

  value     MLUPS with the state resident in HBM, timed with CUDA events on the engine's compute
            stream, max over ranks.
  e2e       the same metric through the C-ABI with HOST buffers: one segment uploads the padded
            AoS f_current from pinned host memory (lbm_upload_f, H2D), runs max(K, 1000) steps
            the way Solver::run does (lbm_run per output period: forces rows and the stability
            verdict come back to the host; lbm_max_velocity after every output step) and downloads
            rho/ux/uy to pinned host memory (lbm_download_macros, D2H) -- what Solver::initialise +
            run + write_final_results amount to (the reference's own job is 120 000 steps per
            segment).  Timed with CUDA events around the whole segment; the parts are reported too.
  roofline  the dominant kernel: 144 B (9 fp64 loads + 9 fp64 stores, SURVEY.md section 8d) x the
            cells a launch really moves through HBM / its average duration (CUDA events around the
            launch of every 8th step INSIDE the timed region), against MEASURED_PEAKS.json: `frac`
            is the honest traffic fraction; a pass of depth T updates every cell T times on that
            trip, `frac_at_144B_per_update` = frac x T.
  multi_gpu_parity / parity_check
            BEFORE anything is timed: a seeded small case on the job's N slabs == one GPU running
            the one-iteration kernels, bit for bit, and == the SHA-256 of the CPU oracle's result
            committed under tests/golden/ (the oracle itself is not touched here).
  cpu_baseline  oracle/_ref/lbm_ref_fast (the unmodified reference headers built with the
            reference's own flags, all host cores) on a bounded sample of the same workload.

Workloads (BASELINE.json configs): slab = weak-scaling cylinder flow, 4096 x 8192 cells per GPU
(config 5; the default, the one the 1/2/4/8-GPU metric is quoted on); c3 = 8192 x 2048 cylinder
flow at Re = 200; c4 = periodic obstacle-free 16384 x 16384 (adds physics_check: decay rate, mass);
c1 = the reference's default 2048 x 512 (L2-resident on a B200: reported, never the roofline evidence).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

BYTES_PER_UPDATE = 144  # 9 fp64 loads + 9 fp64 stores, A-B double buffer (SURVEY.md 8d)
METRIC = "MLUPS (fp64 D2Q9)"
UNIT = "MLUPS"


def config_of(cfg: dict) -> dict:
    """The `config` object: identical in the B200 arm and the reference arm (the driver compares them)."""
    return {"workload": cfg["label"], "nx": cfg["nx"], "ny": cfg["ny"], "tau": cfg["tau"], "inlet_velocity": cfg["inlet_velocity"],
            "output_frequency": cfg["output_frequency"],
            "l2": "inputs exceed every cache: %.2f GB of populations per buffer, no flush needed" % (
                (cfg["nx"] + 2) * (cfg["ny"] + 2) * 72 / 1e9) if cfg["nx"] * cfg["ny"] * 72 > 400e6 else
            "working set near the L2 size: reported, never the roofline evidence"}


def workload(name: str, n_gpus: int) -> dict:
    if name == "slab":
        return dict(nx=4096 * n_gpus, ny=8192, tau=0.6, inlet_velocity=0.01333, output_frequency=140, flags=0,
                    label="weak-scaling cylinder flow, 4096x8192 cells per GPU (BASELINE config 5; N=8: 32768x8192)")
    if name == "c3":
        # Re = u*D/nu = 200 with D = 2*0.05*2048 = 204.8 and tau = 0.6 (nu = 1/30): u = 0.0325521
        return dict(nx=8192, ny=2048, tau=0.6, inlet_velocity=200.0 * ((0.6 - 0.5) / 3.0) / 204.8, output_frequency=140,
                    flags=0, label="cylinder flow Re=200, 8192x2048 (BASELINE config 3)")
    if name == "c4":
        return dict(nx=16384, ny=16384, tau=0.6, inlet_velocity=0.01, output_frequency=0, flags=1 | 2 | 4 | 8,
                    label="periodic obstacle-free 16384x16384 shear wave (BASELINE config 4)")
    if name == "c1":
        return dict(nx=2048, ny=512, tau=0.6, inlet_velocity=0.01333, output_frequency=140, flags=0,
                    label="default cylinder flow 2048x512 (BASELINE config 1, L2-resident)")
    raise SystemExit("unknown workload %s" % name)


# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """SM clock / throttle reasons sampled DURING the timed region (NVML; nvidia-smi as fallback)."""

    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, device: int, period=0.02):
        super().__init__(daemon=True)
        self.device, self.period = device, period
        self.samples = []  # (t, sm_mhz, reasons_bits, power_w)
        self.sm_max = None
        self._halt = threading.Event()
        self.ok = False
        try:
            import pynvml

            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = device
            if vis:
                try:
                    idx = int(vis.split(",")[device])
                except ValueError:
                    idx = device
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.sm_max = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:  # noqa: BLE001
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        while not self._halt.is_set():
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    bits = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:  # noqa: BLE001
                    bits = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                try:
                    pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                except Exception:  # noqa: BLE001
                    pw = None
                self.samples.append((time.time(), mhz, bits, pw))
            except Exception:  # noqa: BLE001
                pass
            self._halt.wait(self.period)

    def stop(self):
        self._halt.set()

    def summary(self, windows):
        """Median SM clock and the union of reasons over samples inside the (t0, t1) windows."""
        sel = [s for s in self.samples if any(a <= s[0] <= b for a, b in windows)]
        if not sel:
            sel = self.samples[-3:]
        if not sel:
            return smi_clocks_once(self.device)
        mhz = sorted(s[1] for s in sel)
        bits = 0
        for s in sel:
            bits |= s[2]
        reasons = [n for b, n in self.REASONS.items() if bits & b and n != "gpu_idle"]
        pw = [s[3] for s in sel if s[3] is not None]
        return {"sm_mhz": mhz[len(mhz) // 2], "sm_max_mhz": self.sm_max, "reasons": reasons, "samples": len(sel),
                "power_w_max": max(pw) if pw else None, "source": "nvml"}


def smi_clocks_once(device: int) -> dict:
    try:
        out = subprocess.run(
            ["nvidia-smi", "-i", str(device), "--query-gpu=clocks.sm,clocks.max.sm,clocks_event_reasons.active",
             "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=20).stdout.strip().split(",")
        return {"sm_mhz": float(out[0]), "sm_max_mhz": float(out[1]), "reasons": [out[2].strip()], "samples": 1,
                "source": "nvidia-smi (single sample after the timed region)"}
    except Exception as e:  # noqa: BLE001
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable: %s" % e], "samples": 0}


def bind_near_gpu(device: int):
    """Pin this rank to the CPUs NVML lists as local to its GPU (its NUMA node) BEFORE any pinned host buffer is
    allocated: first-touch then places the buffers next to the GPU's PCIe root, and the N ranks of a multi-GPU job stop
    pulling each other's host traffic across the socket interconnect.  Returns (previous affinity, note); harmless where
    every GPU reports the same CPU set."""
    try:
        import pynvml

        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = device
        if vis:
            try:
                idx = int(vis.split(",")[device])
            except ValueError:
                idx = device
        h = pynvml.nvmlDeviceGetHandleByIndex(idx)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (int(word) >> b) & 1}
        before = os.sched_getaffinity(0)
        cpus &= before
        if cpus and cpus != before:
            os.sched_setaffinity(0, cpus)
            return before, "rank pinned to the %d CPUs local to GPU %d (of %d)" % (len(cpus), idx, len(before))
        return before, "GPU %d is local to every CPU of this process (%d)" % (idx, len(before))
    except Exception as e:  # noqa: BLE001
        return None, "no NVML CPU affinity (%s)" % type(e).__name__


# ------------------------------------------------------------------------------------------------
def measured_peak_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    except Exception:  # noqa: BLE001
        return 6650.0, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"


def ncu_traffic_per_launch(workload_name: str):
    """dram read+write bytes per launch of the bulk kernel from the committed ncu --set full
    capture of this workload (profiles/*.json written by tools/ncu_summary.py), else None."""
    path = os.path.join(ROOT, "profiles", "bulk_traffic.json")
    try:
        return float(json.load(open(path))[workload_name]["dram_bytes_per_launch"])
    except Exception:  # noqa: BLE001
        return None


def cpu_model() -> str:
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def reference_binary():
    from oracle import oracle as O  # the ONLY use of oracle/ here: the CPU baseline legs

    if os.path.exists(O.REF_FAST):
        return O.REF_FAST, "reference"
    return None, "port"


def run_reference(cfg: dict, steps: int, warmup: int, budget_s: float):
    """Time the reference's own CPU path (oracle/_ref/lbm_ref_fast: unmodified reference headers,
    reference flags, OpenMP over every host core) on a bounded sample of the workload.  Returns
    (mlups, cores, kind, sample description).  Falls back to the C oracle port (1 thread) where
    the compiled reference is absent."""
    cores = host_cores()
    exe, kind = reference_binary()
    nx, ny = cfg["nx"], cfg["ny"]
    # bounded sample: halve the lattice (ny, then nx) until (steps+warmup) updates fit the budget
    # at a pessimistic 5 MLUPS per core; never below 2048 x 2048 (0.6 GB of populations: still
    # far larger than any host cache), and at most the per-GPU slab.
    assumed = 5.0e6 * (cores if kind == "reference" else 1)
    flip = 0
    while (nx * ny * (steps + warmup) / assumed > budget_s) and (nx * ny > 2048 * 2048):
        if flip % 2 == 0 and ny > 2048 or nx <= 2048:
            ny //= 2
        else:
            nx //= 2
        flip += 1
    if kind == "reference":
        env = dict(os.environ, OMP_NUM_THREADS=str(cores), OMP_PROC_BIND="close", OMP_PLACES="cores")
        cmd = [exe, "--time", "--nx", str(nx), "--ny", str(ny), "--steps", str(steps), "--warmup", str(warmup),
               "--of", str(cfg["output_frequency"] or 140), "--tau", repr(cfg["tau"]), "--uin", repr(cfg["inlet_velocity"])]
        with tempfile.TemporaryDirectory() as cwd:  # IOManager writes forces.csv into cwd; the tree may be read-only
            r = subprocess.run(cmd, capture_output=True, text=True, env=env, cwd=cwd)
        line = [l for l in r.stderr.splitlines() if l.startswith("{")]
        if r.returncode != 0 or not line:
            raise RuntimeError("reference run failed: rc=%d %s" % (r.returncode, r.stderr[-400:]))
        j = json.loads(line[-1])
        sample = "%dx%d cylinder flow, %d timed steps after %d warm-up, Solver::run of the unmodified reference " \
                 "(-O3 -ffast-math -mavx2 -mfma -fopenmp), VTK off, %d OpenMP threads, %.1f s" % (
                     nx, ny, steps, warmup, j["threads"], j["seconds"])
        return j["mlups"], j["threads"], kind, sample, j["seconds"] / steps * 1e3
    from oracle import oracle as O

    case = O.Case(nx=nx, ny=ny, tau=cfg["tau"], inlet_velocity=cfg["inlet_velocity"],
                  output_frequency=cfg["output_frequency"] or 140)
    o = O.Oracle(case)
    o.run(warmup)
    t0 = time.perf_counter()
    o.run(steps)
    dt = time.perf_counter() - t0
    return (nx * ny * steps / dt / 1e6, 1, kind, "%dx%d, %d steps of the scalar C oracle port, %.1f s" % (nx, ny, steps, dt),
            dt / steps * 1e3)


# ------------------------------------------------------------------------------------------------
# Correctness inside the bench run (outside every timed region): a small seeded cylinder-flow case on the job's
# N slabs against (a) the same engine on ONE GPU, bit for bit, and (b) the SHA-256 of the CPU oracle's result
# committed under tests/golden/ (generated by oracle/gen_parity_sha.py; the oracle itself is not touched here).
PARITY_STEPS = 64


def parity_case(n_gpus: int) -> dict:
    """128 columns per slab x 96 rows; the cylinder (r = 19 cells) sits ON the face between slabs 0 and 1."""
    return dict(nx=128 * n_gpus, ny=96, tau=0.6, inlet_velocity=0.04, output_frequency=7,
                cylinder_x=(1.0 / n_gpus if n_gpus > 1 else 0.5), cylinder_y=0.5, cylinder_radius=0.2)


def parity_state(nx: int, ny: int):
    """A deterministic non-equilibrium f_current on the padded grid (AoS): integer hash -> exact fp64, the same
    bits on every platform (no RNG, no libm)."""
    import numpy as np

    gy, gx, i = np.meshgrid(np.arange(ny + 2, dtype=np.int64), np.arange(nx + 2, dtype=np.int64), np.arange(9, dtype=np.int64),
                            indexing="ij")
    hsh = ((gx * 73856093) ^ (gy * 19349663) ^ ((i + 1) * 83492791)) % 1000
    w = np.array([4.0 / 9.0] + [1.0 / 9.0] * 4 + [1.0 / 36.0] * 4)
    return np.ascontiguousarray(w * (1.0 + 0.05 * (hsh.astype(np.float64) / 1000.0 - 0.5)))


def parity_sha(f_next_interior, rows) -> str:
    import hashlib

    import numpy as np

    hh = hashlib.sha256()
    hh.update(np.ascontiguousarray(f_next_interior, dtype=np.float64).tobytes())
    hh.update(np.ascontiguousarray(rows[:, 0], dtype=np.float64).tobytes())  # the output timesteps
    return hh.hexdigest()


def parity_golden(n_gpus: int):
    try:
        return json.load(open(os.path.join(ROOT, "tests", "golden", "bench_parity_sha.json")))[str(n_gpus)]
    except Exception:  # noqa: BLE001
        return None


def parity_check(lbm_b200, dist, rank, world, local_rank, nccl_id, variant=2, depth=None):
    """Returns the dict bench.py prints as "multi_gpu_parity" (rank 0) or None (other ranks)."""
    import numpy as np

    c = parity_case(world)
    p = lbm_b200.SimulationParams(**c)
    state = parity_state(c["nx"], c["ny"])
    s = lbm_b200.Solver(p, device=local_rank, rank=rank, world=world, nccl_id=nccl_id)
    s.set_kernel_variant(variant)  # (a lattice this small would default to the one-iteration kernels)
    if depth is not None:
        s.set_pass_depth(depth)
    s.initialise()
    info = s.info()
    lnx, x0 = info.local_nx, info.x_start
    s.upload_f(np.ascontiguousarray(state[:, x0:x0 + lnx + 2, :]), iteration=0)
    rows, bad = s.run(PARITY_STEPS)
    mine = {"f_next": s.f_next()[1:-1, 1:-1].copy(), "f_current": s.f_current()[1:-1, 1:-1].copy(), "rows": rows, "bad": bad,
            "p2p": info.halo_p2p, "depth": info.pass_depth}
    mine["rho"], mine["ux"], mine["uy"] = (a.copy() for a in s.macros())
    s.close()
    if dist is not None:
        parts = [None] * world if rank == 0 else None
        dist.gather_object(mine, parts, dst=0)
    else:
        parts = [mine]
    if rank != 0:
        return None
    one = lbm_b200.Solver(p, device=local_rank)
    one.set_kernel_variant(1)  # the reference point: one iteration per launch, the round-1 kernels
    one.initialise()
    one.upload_f(state, iteration=0)
    rows1, bad1 = one.run(PARITY_STEPS)
    ref = {"f_next": one.f_next()[1:-1, 1:-1], "f_current": one.f_current()[1:-1, 1:-1]}
    ref["rho"], ref["ux"], ref["uy"] = one.macros()
    one.close()
    same = all(np.array_equal(np.concatenate([q[k] for q in parts], axis=1), ref[k]) for k in ("f_next", "f_current", "rho", "ux", "uy"))
    forces = sum(q["rows"][:, 1:3] for q in parts)
    f_err = float(np.abs(forces - rows1[:, 1:3]).max()) if len(rows1) else 0.0
    sha = parity_sha(np.concatenate([q["f_next"] for q in parts], axis=1), parts[0]["rows"])
    gold = parity_golden(world)
    return {"bit_identical": bool(same and all(q["bad"] == bad1 == -1 for q in parts) and
                                  np.array_equal(parts[0]["rows"][:, 0], rows1[:, 0])),
            "against": "one GPU running the one-iteration kernels (populations, f_current, rho, ux, uy: every cell)",
            "kernel_variant": int(variant),
            "forces_max_abs_diff": f_err, "forces_ok": bool(f_err <= 1e-13),
            "sha256_f_next": sha, "sha_matches_oracle": (None if gold is None else bool(sha == gold["sha256"])),
            "golden": "tests/golden/bench_parity_sha.json (CPU oracle, oracle/gen_parity_sha.py)",
            "case": "%dx%d cylinder on a slab face, %d steps from a seeded state" % (c["nx"], c["ny"], PARITY_STEPS),
            "cells": c["nx"] * c["ny"], "steps": PARITY_STEPS, "halo_p2p": int(min(q["p2p"] for q in parts)),
            "pass_depth": int(parts[0]["depth"])}


def run_like_solver(s, n_steps: int, of: int):
    """Solver::run's loop (include/LBMSolver.h:48-76) over the C-ABI: chunks that end on output steps, the forces
    rows of each chunk, and Grid::max_velocity after every output step (the 'Timestep t: max_vel=' line)."""
    rows_all, t, bad = [], 0, -1
    while t < n_steps:
        nxt = ((t + of - 1) // of) * of if of > 0 else n_steps - 1
        last = min(nxt, n_steps - 1)
        rows, bad = s.run(last - t + 1)
        rows_all.extend(rows)
        if bad >= 0:
            break
        if of > 0 and last > 0 and last % of == 0:
            s.max_velocity()
        t = last + 1
    return rows_all, bad


# ------------------------------------------------------------------------------------------------
# --dump-outputs: the state the timed steps leave behind, what a caller of lbm_step reads back (Grid::rho / ux / uy and
# the populations of f_current and f_next), at a fixed seeded sample of cells so that two builds can be compared
# output for output.  2^18 cells x (3 moments + 2 x 9 populations + 2 coordinates) x 8 B = 48 MB in all.  To get there
# each rank downloads its whole slab once per field: padded f_current and f_next are 2.4 GB each on the default slab
# workload and 19 GB each on c4, held in host memory one at a time.
DUMP_CELLS = 1 << 18
DUMP_SEED = 20251020


def dump_cells(nx: int, ny: int):
    """Sorted global cell indices y * nx + x of the sample: every cell of a lattice that has at most DUMP_CELLS."""
    import numpy as np

    if nx * ny <= DUMP_CELLS:
        return np.arange(nx * ny, dtype=np.int64)
    return np.sort(np.random.default_rng(DUMP_SEED).choice(nx * ny, DUMP_CELLS, replace=False))


def dump_outputs(s, lbm_b200, dist, rank, world, nx, ny, out_dir):
    """Writes out_dir/{rho,ux,uy,f_current,f_next,cell_x,cell_y}.npy (float64) on rank 0; every rank contributes the
    sampled cells of its own slab."""
    import numpy as np

    info = s.info()
    gy, gx = np.divmod(dump_cells(nx, ny), nx)
    mine = np.nonzero((gx >= info.x_start) & (gx < info.x_start + info.local_nx))[0]
    ly, lx = gy[mine], gx[mine] - info.x_start
    part = {"at": mine}
    for k, a in zip(("rho", "ux", "uy"), s.macros()):
        part[k] = a[ly, lx]
    for k, which in (("f_current", lbm_b200.F_CURRENT), ("f_next", lbm_b200.F_NEXT)):
        part[k] = s.f(which)[ly + 1, lx + 1, :]  # padded layout: interior cell (y, x) sits at [y + 1, x + 1]
    if dist is not None:
        parts = [None] * world if rank == 0 else None
        dist.gather_object(part, parts, dst=0)
    else:
        parts = [part]
    if rank != 0:
        return
    out = {"cell_x": gx.astype(np.float64), "cell_y": gy.astype(np.float64)}
    for k in ("rho", "ux", "uy", "f_current", "f_next"):
        a = np.empty((len(gx),) + parts[0][k].shape[1:], dtype=np.float64)
        for q in parts:
            a[q["at"]] = q[k]
        out[k] = a
    os.makedirs(out_dir, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="slab", choices=["slab", "c3", "c4", "c1"])
    ap.add_argument("--variant", type=int, default=None, help="bulk kernel variant (default: engine default)")
    ap.add_argument("--aa", action="store_true", help="in-place AA variant: one population buffer per GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the seeded correctness check outside the timed regions")
    ap.add_argument("--depth", type=int, default=None, help="iterations per temporally blocked pass (variant 2): 1, 2, 3")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the moments and populations they left at a fixed sample of cells "
                         "as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the B200 arm computes")
    if args.warmup < 3:
        args.warmup = 3  # timing hygiene: at least 3 warm-up steps

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            # re-launch under torchrun, one rank per GPU
            port = 29500 + (os.getpid() % 2000)
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
                   "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.abspath(__file__)] + sys.argv[1:]
            raise SystemExit(subprocess.call(cmd))
        raise SystemExit("--gpus %d does not match WORLD_SIZE %d" % (args.gpus, world))

    cfg = workload(args.workload, args.gpus)
    if args.aa:
        cfg["flags"] |= 16  # LBM_FLAG_AA
    # stdout carries exactly one JSON line: anything libraries print there (NCCL's version banner,
    # for one) is sent to stderr instead
    json_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(json_fd, (json.dumps(obj) + "\n").encode())

    # ---------------------------------------------------------------- reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return 0
        t0 = time.perf_counter()
        mlups, cores, kind, sample, ms_step = run_reference(cfg, args.steps, args.warmup, budget_s=150.0)
        out = {
            "impl": "reference", "metric": METRIC, "value": mlups, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_of(cfg),
            "impl_detail": {"layout": "fp64 AoS (reference include/LBMGrid.h:105-107), host DRAM",
                            "partition": "1 process, OpenMP over %d host cores" % cores},
            "cpu_baseline": {"value": mlups, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample, "cpu_model": cpu_model()},
            "e2e": {"value": mlups, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "wall_s": time.perf_counter() - t0,
        }
        emit(out)
        return 0

    # ---------------------------------------------------------------- B200 arm
    import numpy as np

    affinity_before, affinity_note = bind_near_gpu(local_rank)

    import lbm_b200  # raises if liblbm_b200.so is missing: there is no fallback path

    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist

        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        ident = [lbm_b200.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ident, src=0)
        nccl_id = ident[0]
    else:
        nccl_id = None

    def barrier():
        if dist is not None:
            dist.barrier()

    def max_over_ranks(x: float) -> float:
        if dist is None:
            return x
        import torch

        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x: float) -> float:
        if dist is None:
            return x
        import torch

        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    p = lbm_b200.SimulationParams(nx=cfg["nx"], ny=cfg["ny"], tau=cfg["tau"], inlet_velocity=cfg["inlet_velocity"],
                                  output_frequency=cfg["output_frequency"], flags=cfg["flags"])
    # ---- correctness first (outside every timed region): N slabs == 1 GPU == the oracle's SHA
    parity = None
    if not args.no_parity and not args.aa:
        parity = parity_check(lbm_b200, dist, rank, world, local_rank, nccl_id,
                              variant=2 if args.variant is None else args.variant, depth=args.depth)
        if dist is not None:  # a fresh NCCL id for the measured job
            ident = [lbm_b200.nccl_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(ident, src=0)
            nccl_id = ident[0]

    s = lbm_b200.Solver(p, device=local_rank, rank=rank, world=world, nccl_id=nccl_id)
    if args.variant is not None:
        s.set_kernel_variant(args.variant)
    if args.depth is not None:
        s.set_pass_depth(args.depth)
    s.initialise()
    info = s.info()
    lnx, ny = info.local_nx, info.local_ny
    cells_local = lnx * ny
    cells_global = cfg["nx"] * cfg["ny"]

    sampler = ClockSampler(local_rank)
    sampler.start()
    windows = []

    # Untimed: one output period first, so that every kernel of the path (the depth-1 pass of an output step, the
    # force reduction, the macro emission) has been loaded and every lazily allocated buffer exists before anything is
    # timed (CUDA loads kernels lazily; on a fresh box the first output step costs tens of milliseconds).
    if p.output_frequency > 0:
        s.run(p.output_frequency + 2)
        s.max_velocity()
    # warm-up, then K timed steps bracketed by barrier + synchronize on both sides
    s.step(args.warmup)
    s.sync()
    barrier()
    per_kernel = 8 if args.steps >= 64 else 1  # CUDA events around the bulk launch of every 8th step
    launches0 = s.counters()[0]
    w0 = time.time()
    ms_total, ms_bulk, launches = s.time_steps(args.steps, per_kernel)
    s.sync()
    w1 = time.time()
    barrier()
    windows.append((w0, w1))
    ms = max_over_ranks(ms_total)
    ok, bad = s.check_stability()
    physics = None
    if args.workload == "c4" and world == 1:
        # The shear wave u_x = u0 sin(2 pi y / ny) of the periodic obstacle-free lattice decays as exp(-nu k^2 t)
        # (SURVEY.md 8c: the reference has no such mode, so this analytic property is the check at FULL size):
        # the measured decay rate against nu k^2, and the drift of the total mass.
        n_it = s.info().iteration
        rho_f, ux_f, uy_f = s.macros()  # the stored moments belong to f_current of iteration n_it - 1
        kk = 2.0 * np.pi / ny
        prof = ux_f.mean(axis=1)
        amp = 2.0 * float((prof * np.sin(kk * np.arange(ny))).mean()) / cfg["inlet_velocity"]
        nu = (cfg["tau"] - 0.5) / 3.0
        rate = -np.log(amp) / max(n_it - 1, 1)
        physics = {"iterations": int(n_it), "decay_rate_measured": float(rate), "decay_rate_nu_k2": float(nu * kk * kk),
                   "decay_rate_rel_err": float(rate / (nu * kk * kk) - 1.0),
                   "mass_drift": float(rho_f.sum() / (float(ny) * float(lnx)) - 1.0),
                   "max_abs_uy": float(np.abs(uy_f).max())}
        del rho_f, ux_f, uy_f
    value = cells_global * args.steps / (ms * 1e-3) / 1e6
    gpu_launches = s.counters()[0] - launches0
    if args.dump_outputs:  # after the launch count: its downloads launch export kernels of their own
        dump_outputs(s, lbm_b200, dist, rank, world, cfg["nx"], cfg["ny"], args.dump_outputs)

    # roofline of the dominant kernel, from the launches inside the timed region.  bulk_cells are the cells the
    # launches really moved through HBM (obstacle cells whose eight neighbours are solid are never touched), each
    # read once and written once per launch: 144 B per cell per LAUNCH whatever the pass depth.  A temporally blocked
    # launch of depth T updates every cell T times on that one trip, so its 144-B-per-update equivalent is T x higher
    # and may exceed the HBM peak -- that is the point of the scheme; `frac` stays the honest traffic fraction.
    peak, peak_src = measured_peak_gbs()
    _, bulk_launches, bulk_cells = s.counters()
    bulk_updates = s.bulk_updates()
    if per_kernel and bulk_launches:
        bulk_ms = ms_bulk / bulk_launches
        achieved = (bulk_cells / bulk_launches) * BYTES_PER_UPDATE / (bulk_ms * 1e-3) / 1e9
        depth_eff = bulk_updates / max(bulk_cells, 1)
        kname = {0: "k_bulk_scalar + k_fixup (fused pull collide-stream)", 1: "k_bulk_vec2 + k_fixup (fused pull collide-stream)",
                 2: "k_tb (temporally blocked pull collide-stream, boundary rules inside)"}.get(info.kernel_variant, "k_bulk")
        roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": ncu_traffic_per_launch(args.workload + ("_aa" if args.aa else "") + ("_tb%d" % info.pass_depth if info.kernel_variant == 2 else "")),
                "kernel": kname, "bytes_per_launch": (bulk_cells / bulk_launches) * BYTES_PER_UPDATE, "avg_launch_ms": bulk_ms,
                "launches_timed": bulk_launches, "cells_per_launch": bulk_cells / bulk_launches,
                "updates_per_cell_per_launch": depth_eff, "algorithmic_bytes_per_update": BYTES_PER_UPDATE / max(depth_eff, 1e-9),
                "frac_at_144B_per_update": achieved * depth_eff / peak,
                "kernel_share_of_step": bulk_ms * (args.steps / max(depth_eff, 1e-9)) / ms_total,
                "peak_source": peak_src,
                "whole_step_frac_at_144B_per_update": value * 1e6 * BYTES_PER_UPDATE / 1e9 / args.gpus / peak}
        if args.aa:
            # BASELINE.json quotes "72 B for AA" (the resident footprint per cell); an AA update still
            # moves 9 loads + 9 stores = 144 B, which is what `achieved` counts (SURVEY.md 8d)
            roof["kernel"] = "k_aa_even / k_aa_odd (in-place collide-stream)"
            roof["frac_if_72B_per_update"] = roof["frac"] / 2
    else:
        roof = {"bound": "hbm", "achieved": None, "peak": peak, "unit": "GB/s", "frac": None, "traffic": None}

    # ------------------------------------------------------------ e2e through the C-ABI, host buffers
    e2e = None
    if not args.no_e2e:
        shape_f = (ny + 2, lnx + 2, 9)
        host_f, own_f = lbm_b200.pinned_empty(shape_f)
        host_m, own_m = lbm_b200.pinned_empty((3, ny, lnx))
        s.f(lbm_b200.F_CURRENT, out=host_f)  # a valid f_current to restart from (outside the timed region)
        h2d = host_f.nbytes
        n_rows = 0
        best = None
        # One segment = one Solver::initialise + run + write_final_results shaped job.  The fixed host
        # traffic of a segment (state in, fields out) is amortised over its steps, so the segment is never
        # shorter than 1000 steps (the reference's own job runs 120 000 steps per segment).
        seg_steps = max(args.steps, 1000)
        for rep in range(2):  # first repetition warms the staging buffers; the second one is reported
            s.sync()
            barrier()
            w0 = time.time()
            s.event_record(0)
            s.upload_f(host_f, iteration=0)                              # H2D: the segment's input state
            s.event_record(1)
            rows, bad_e2e = run_like_solver(s, seg_steps, p.output_frequency)  # Solver::run: rows, verdicts, max_velocity
            s.event_record(2)
            s.macros(out=(host_m[0], host_m[1], host_m[2]))              # D2H: rho, ux, uy (write_final_results)
            s.event_record(3)
            ms_e2e = s.event_elapsed(0, 3)
            parts = (s.event_elapsed(0, 1), s.event_elapsed(1, 2), s.event_elapsed(2, 3))
            w1 = time.time()
            barrier()
            windows.append((w0, w1))
            best = max_over_ranks(ms_e2e)
            n_rows = len(rows)
            wall_e2e = w1 - w0
        d2h = host_m.nbytes + n_rows * (16 + 8) + 4 * (seg_steps // max(p.output_frequency, 64) + 2)
        e2e = {"value": cells_global * seg_steps / (best * 1e-3) / 1e6, "unit": UNIT,
               "h2d_bytes_per_step": sum_over_ranks(h2d) / seg_steps, "d2h_bytes_per_step": sum_over_ranks(d2h) / seg_steps,
               "segment": "lbm_upload_f(pinned AoS f_current) + Solver::run's loop over the C-ABI (%d steps: lbm_run per output "
                          "period, forces rows, stability verdicts, lbm_max_velocity after every output step) + "
                          "lbm_download_macros(pinned)" % seg_steps,
               "segment_steps": seg_steps, "ms_per_segment": best, "wall_ms_rank0": wall_e2e * 1e3,
               "rank0_ms": {"upload_h2d": parts[0], "run": parts[1], "download_d2h": parts[2]},
               "stable": bad_e2e == -1, "forces_rows": n_rows}
        lbm_b200.pinned_free(own_f)
        lbm_b200.pinned_free(own_m)

    sampler.stop()
    sampler.join(timeout=2.0)
    clocks = sampler.summary(windows) if sampler.ok else smi_clocks_once(local_rank)
    s.close()

    # ------------------------------------------------------------ CPU baseline (rank 0, N = 1 only)
    cpu = None
    if affinity_before:
        try:
            os.sched_setaffinity(0, affinity_before)  # the reference gets every host core again
        except OSError:
            pass
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            v, cores, kind, sample, _ = run_reference(cfg, 20, 3, budget_s=30.0)
            cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample, "cpu_model": cpu_model()}
        except Exception as e:  # noqa: BLE001
            cpu = {"value": None, "unit": UNIT, "cores": host_cores(), "kind": "reference", "sample": "failed: %s" % e}

    if rank == 0:
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_of(cfg),
            "impl_detail": {"layout": "fp64 SoA, in-place AA pattern (one buffer)" if args.aa else "fp64 SoA, A-B double buffer",
                            "kernel_variant": info.kernel_variant, "pass_depth": info.pass_depth,
                            "partition": ("x-slab x%d, halo of %d ghost columns per face %s" % (
                                world, max(info.pass_depth, 2) if info.kernel_variant == 2 else 1,
                                "stored into the neighbour's memory by the step kernel itself (CUDA IPC peer memory over NVLink)"
                                if info.halo_p2p else "by NCCL send/recv")) if world > 1 else "single GPU",
                            "bytes_per_buffer": info.bytes_per_buffer, "deep_solid_cells_skipped": info.deep_solid_cells,
                            "host_affinity": affinity_note},
            "roofline": roof, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(gpu_launches), "clocks": clocks,
            "stable": bool(ok), "roofline_whole_step_frac": value * 1e6 * BYTES_PER_UPDATE / 1e9 / args.gpus / peak,
            ("multi_gpu_parity" if world > 1 else "parity_check"): parity,
        }
        if physics is not None:
            out["physics_check"] = physics
        emit(out)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
