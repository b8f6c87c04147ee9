"""bench.py contract, CPU side: the reference arm prints exactly one JSON line on stdout with the
keys the driver reads, and the B200 arm refuses to run without a GPU instead of falling back."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*args):
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + list(args), capture_output=True, text=True, env=env, timeout=600)


def test_reference_arm_prints_one_json_line():
    """The reference arm times the compiled reference (oracle/_ref) where it is built, the C oracle port otherwise."""
    kind = "reference" if os.path.exists(os.path.join(ROOT, "oracle", "_ref", "lbm_ref_fast")) else "port"
    r = run_bench("--impl", "reference", "--workload", "c1", "--steps", "4", "--warmup", "3")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    j = json.loads(lines[0])
    assert j["impl"] == "reference" and j["metric"] == "MLUPS (fp64 D2Q9)" and j["unit"] == "MLUPS"
    assert j["value"] > 1.0 and j["higher_is_better"] is True and j["n_gpus"] == 1 and j["steps"] == 4 and j["warmup"] == 3
    assert j["dtype"] == "f64" and j["vs_baseline"] is None and "2048x512" in j["config"]["workload"]
    cb = j["cpu_baseline"]
    assert cb["kind"] == kind and cb["cores"] >= 1 and cb["value"] == j["value"] and "2048x512" in cb["sample"]
    assert j["e2e"] == {"value": j["value"], "unit": "MLUPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert j["gpu_launches"] == 0


def test_b200_arm_has_no_cpu_fallback():
    import torch

    if torch.cuda.is_available():
        pytest.skip("a CUDA device is visible")
    r = run_bench("--workload", "c1", "--steps", "4")
    assert r.returncode != 0 and "no CPU path" in (r.stderr + r.stdout)
    assert not [l for l in r.stdout.splitlines() if l.startswith("{")]  # no number without a GPU


def test_both_arms_print_the_same_config_object():
    """The driver compares `config` of the two arms: everything arm-specific lives in `impl_detail`."""
    sys.path.insert(0, ROOT)
    import bench

    for n in (1, 8):
        cfg = bench.workload("slab", n)
        c = bench.config_of(cfg)
        assert set(c) == {"workload", "nx", "ny", "tau", "inlet_velocity", "output_frequency", "l2"}
        assert c["nx"] == 4096 * n and c["ny"] == 8192 and "exceed" in c["l2"]
    src = open(os.path.join(ROOT, "bench.py")).read()
    assert src.count('"config": config_of(cfg)') == 2  # the reference arm and the B200 arm


def test_dump_sample_is_fixed_and_bounded():
    """--dump-outputs samples the same cells on every run, and stays within 64 MB on the largest workload."""
    sys.path.insert(0, ROOT)
    import bench

    a, b = bench.dump_cells(16384, 16384), bench.dump_cells(16384, 16384)
    assert np.array_equal(a, b) and len(a) == bench.DUMP_CELLS and (np.diff(a) > 0).all() and a[-1] < 16384 * 16384
    assert np.array_equal(bench.dump_cells(64, 32), np.arange(64 * 32))
    assert bench.DUMP_CELLS * (3 + 2 * 9 + 2) * 8 <= 64 << 20


DUMP_STEPS, DUMP_WARMUP = 7, 3


@pytest.fixture(scope="module")
def c1_oracle():
    """The CPU oracle on c1 after the iterations bench.py runs before its dump: the untimed output period + 2, the
    warm-up and the timed steps."""
    from oracle import oracle as O

    o = O.Oracle(O.Case(nx=2048, ny=512))
    o.run(140 + 2 + DUMP_WARMUP + DUMP_STEPS)
    return o


@pytest.mark.gpu
@pytest.mark.parametrize("extra", [[], ["--aa"]], ids=["ab", "aa"])
def test_dumped_outputs_are_the_oracles(tmp_path, c1_oracle, extra):
    """bench.py --dump-outputs on the default cylinder flow (c1), A-B buffers and in-place AA: the sampled moments and
    populations its timed steps leave behind are those of the CPU oracle after the same iterations."""
    r = run_bench("--workload", "c1", "--steps", str(DUMP_STEPS), "--warmup", str(DUMP_WARMUP), "--no-cpu-baseline",
                  "--no-e2e", "--no-parity", "--dump-outputs", str(tmp_path), *extra)
    assert r.returncode == 0, r.stderr[-2000:]
    j = json.loads(r.stdout)
    assert j["steps"] == DUMP_STEPS and j["stable"]
    got = {k: np.load(tmp_path / (k + ".npy")) for k in ("cell_x", "cell_y", "rho", "ux", "uy", "f_current", "f_next")}
    assert all(a.dtype == np.float64 for a in got.values())
    assert sum(a.nbytes for a in got.values()) <= 64 << 20
    x, y = got["cell_x"].astype(np.int64), got["cell_y"].astype(np.int64)
    o = c1_oracle
    for k in ("f_current", "f_next"):
        ref = getattr(o, k)[y + 1, x + 1]
        assert got[k].shape == ref.shape and (np.abs(got[k] - ref) <= 1e-12 * np.abs(ref)).all(), k
    assert (np.abs(got["rho"] - o.rho[y, x]) <= 1e-12 * np.abs(o.rho[y, x])).all()
    for k in ("ux", "uy"):
        assert np.abs(got[k] - getattr(o, k)[y, x]).max() <= 1e-12, k


@pytest.mark.parametrize("n", [1, 2, 4, 8])
def test_in_run_parity_golden_is_the_oracles(n):
    """tests/golden/bench_parity_sha.json (what every `bench.py --gpus N` run compares its N-slab result with) is the
    SHA-256 of the CPU oracle's populations for the seeded case, regenerated here."""
    sys.path.insert(0, ROOT)
    import bench
    from oracle import oracle as O

    c = bench.parity_case(n)
    a, b = bench.parity_state(c["nx"], c["ny"]), bench.parity_state(c["nx"], c["ny"])
    assert a.shape == (c["ny"] + 2, c["nx"] + 2, 9) and (a == b).all() and a.min() > 0
    o = O.Oracle(O.Case(**c))
    o.f_current[...] = a
    rows, bad = o.run(bench.PARITY_STEPS)
    assert bad == -1 and len(rows) == 10
    assert bench.parity_sha(o.f_next[1:-1, 1:-1], rows) == bench.parity_golden(n)["sha256"]
    # the cylinder sits on the face between slabs 0 and 1
    if n > 1:
        assert int(c["cylinder_x"] * c["nx"]) == 128
