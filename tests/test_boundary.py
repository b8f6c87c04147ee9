"""CPU-side checks of the drop-in boundary (no GPU, no compute calls):
the C-ABI library loads and exports every symbol include/lbm_b200.h declares; the product never
touches oracle/; the C++ headers keep the reference's surface (its configuration and helper headers print
what the reference's print, tests/golden/reference_pins.json); the host-side writers produce the reference's file
formats."""
import ctypes
import json
import os
import re
import struct
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "highperformancecomputing-latticeboltzmannmethod_b200")
INC = os.path.join(ROOT, "include")
LIB = os.path.join(PKG, "liblbm_b200.so")
REF = "/root/reference"


@pytest.fixture(scope="session")
def built():
    import __graft_entry__ as g

    g.build()
    return True


def declared_symbols():
    text = open(os.path.join(INC, "lbm_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(lbm_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol(built):
    names = declared_symbols()
    assert len(names) >= 30
    lib = ctypes.CDLL(LIB)
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, missing
    import lbm_b200

    assert sorted(lbm_b200.binding.EXPORTS) == names  # the ctypes binding covers the whole header


def test_no_cpu_fallback_without_a_device(built):
    import torch

    if torch.cuda.is_available():
        pytest.skip("a CUDA device is visible")
    import lbm_b200

    with pytest.raises(lbm_b200.LbmError) as e:
        lbm_b200.Solver(lbm_b200.SimulationParams(nx=8, ny=8))
    assert "no CPU path" in str(e.value)


def test_product_never_touches_the_oracle():
    pat = re.compile(r"oracle|liboracle|/root/reference")
    bad = []
    for base in (PKG, INC, os.path.join(ROOT, "examples")):
        for d, _, files in os.walk(base):
            if "build" in d.split(os.sep):
                continue
            for f in files:
                if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp", ".hpp")) or f == "Makefile":
                    text = open(os.path.join(d, f), errors="replace").read()
                    if pat.search(text):
                        bad.append(os.path.join(d, f))
    assert not bad, bad


def test_bootstrap_env_single_and_multi(built, tmp_path):
    """lbm_bootstrap_env: rank discovery and the NCCL-id file hand-off (no NCCL needed for world 1)."""
    code = (
        "import ctypes,sys;L=ctypes.CDLL(%r);r=ctypes.c_int();w=ctypes.c_int();l=ctypes.c_int();"
        "rc=L.lbm_bootstrap_env(ctypes.byref(r),ctypes.byref(w),ctypes.byref(l),None);print(rc,r.value,w.value,l.value)" % LIB)
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    out = subprocess.run(["python", "-c", code], env=env, capture_output=True, text=True).stdout.split()
    assert out == ["0", "0", "1", "0"]
    env.update(RANK="3", WORLD_SIZE="8", LOCAL_RANK="3")
    out = subprocess.run(["python", "-c", code], env=env, capture_output=True, text=True).stdout.split()
    assert out == ["0", "3", "8", "3"]
    env.update(RANK="9", WORLD_SIZE="8")
    out = subprocess.run(["python", "-c", code], env=env, capture_output=True, text=True).stdout.split()
    assert out[0] == "-1"


@pytest.fixture(scope="session")
def host_checks(built, tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("cpp") / "host_checks")
    subprocess.run(["g++", "-std=c++17", "-O2", "-mfma", "-ffp-contract=off", "-pthread", "-I" + INC, os.path.join(ROOT, "tests", "cpp", "host_checks.cpp"),
                    "-o", exe, "-L" + PKG, "-llbm_b200", "-Wl,-rpath," + PKG], check=True)
    return exe


def test_fixed8_matches_printf(host_checks):
    out = subprocess.run([host_checks, "fixed8", "3000000", "7"], capture_output=True, text=True)
    assert out.returncode == 0 and out.stdout.startswith("ok"), out.stdout


def test_vtk_frame_is_byte_identical_to_the_reference_format(host_checks, tmp_path):
    nx, ny, t = 37, 23, 140
    subprocess.run([host_checks, "vtk", str(nx), str(ny), "5", str(t)], cwd=tmp_path, check=True)
    raw = np.fromfile(tmp_path / "field.bin").reshape(3, ny * nx)
    rho, ux, uy = raw
    # independent rendering of reference include/LBMIO.h:70-108
    lines = ["# vtk DataFile Version 3.0", "LBM Flow Timestep %d" % t, "ASCII", "DATASET STRUCTURED_POINTS",
             "DIMENSIONS %d %d 1" % (nx, ny), "ORIGIN 0 0 0", "SPACING 1 1 1", "POINT_DATA %d" % (nx * ny),
             "VECTORS velocity double"]
    lines += ["%.8f %.8f 0.0" % (a, b) for a, b in zip(ux, uy)]
    lines += ["", "SCALARS velocity_magnitude double", "LOOKUP_TABLE default"]
    lines += ["%.8f" % v for v in np.sqrt(ux * ux + uy * uy)]
    lines += ["", "SCALARS density double", "LOOKUP_TABLE default"]
    lines += ["%.8f" % v for v in rho]
    want = ("\n".join(lines) + "\n").encode()
    got = open(tmp_path / "vtk_output" / ("lbm_%06d.vtk" % t), "rb").read()
    assert got == want


def test_binary_vtk_frame_round_trips(host_checks, tmp_path):
    nx, ny, t = 37, 23, 280
    subprocess.run([host_checks, "vtkbin", str(nx), str(ny), "5", str(t)], cwd=tmp_path, check=True)
    rho, ux, uy = np.fromfile(tmp_path / "field.bin").reshape(3, ny * nx)
    raw = open(tmp_path / "vtk_output" / ("lbm_%06d.vtk" % t), "rb").read()
    head = ("# vtk DataFile Version 3.0\nLBM Flow Timestep %d\nBINARY\nDATASET STRUCTURED_POINTS\nDIMENSIONS %d %d 1\n"
            "ORIGIN 0 0 0\nSPACING 1 1 1\nPOINT_DATA %d\nVECTORS velocity double\n" % (t, nx, ny, nx * ny)).encode()
    assert raw.startswith(head)
    n, pos = nx * ny, len(head)
    vec = np.frombuffer(raw, dtype=">f8", count=3 * n, offset=pos).reshape(n, 3)
    assert np.array_equal(vec[:, 0], ux) and np.array_equal(vec[:, 1], uy) and not vec[:, 2].any()
    pos += 24 * n
    tag = b"\nSCALARS velocity_magnitude double\nLOOKUP_TABLE default\n"
    assert raw[pos:pos + len(tag)] == tag
    pos += len(tag)
    # ux*ux + uy*uy may be contracted into an FMA by the C++ compiler: equal to an ulp
    assert np.allclose(np.frombuffer(raw, dtype=">f8", count=n, offset=pos), np.sqrt(ux * ux + uy * uy), rtol=4e-16, atol=0)
    pos += 8 * n
    tag = b"\nSCALARS density double\nLOOKUP_TABLE default\n"
    assert raw[pos:pos + len(tag)] == tag
    assert np.array_equal(np.frombuffer(raw, dtype=">f8", count=n, offset=pos + len(tag)), rho)


def test_forces_csv_rows(host_checks, tmp_path):
    rows = [(0, 1.53739333123, -4.5e-16), (140, 0.21697769, 0.0), (10000, -0.05162555, 1.25e-9)]
    inp = "".join("%d %.17g %.17g\n" % r for r in rows)
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    subprocess.run([host_checks, "forces"], input=inp, text=True, cwd=tmp_path, check=True, env=env)
    q = 0.5 * 0.01333 * 0.01333 * 2 * int(0.05 * 512)
    want = "timestep,drag_force,lift_force,drag_coeff,lift_coeff\n" + "".join(
        "%d,%.8f,%.8f,%.8f,%.8f\n" % (t, fx, fy, fx / q, fy / q) for t, fx, fy in rows)
    assert open(tmp_path / "forces.csv").read() == want


def test_examples_driver_builds(built):
    subprocess.run(["make", "-C", os.path.join(ROOT, "examples")], check=True, capture_output=True)
    assert os.path.exists(os.path.join(ROOT, "examples", "lbm_solver"))


def test_bootstrap_env_hands_the_nccl_id_to_every_rank(built, tmp_path):
    """Two processes of one "launch": rank 0 creates the NCCL unique id, rank 1 receives the same
    128 bytes through the id file (what a C++ driver started by torchrun --no-python relies on)."""
    code = (
        "import ctypes,sys;L=ctypes.CDLL(%r);r=ctypes.c_int();w=ctypes.c_int();l=ctypes.c_int();"
        "b=ctypes.create_string_buffer(128);rc=L.lbm_bootstrap_env(ctypes.byref(r),ctypes.byref(w),ctypes.byref(l),b);"
        "L.lbm_last_error.restype=ctypes.c_char_p;print(rc,r.value,w.value,b.raw.hex(),L.lbm_last_error(None).decode())" % LIB)
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    env.update(WORLD_SIZE="2", LBM_B200_ID_FILE=str(tmp_path / "nccl.id"))
    procs = [subprocess.Popen(["python", "-c", code], env=dict(env, RANK=str(r), LOCAL_RANK=str(r)), stdout=subprocess.PIPE, text=True)
             for r in (1, 0)]  # rank 1 first: it has to wait for the file
    outs = [p.communicate(timeout=120)[0].split(None, 4) for p in procs]
    if any(o[0] == "-3" for o in outs):
        pytest.skip("NCCL library not loadable here: " + outs[0][-1])
    assert [o[0] for o in outs] == ["0", "0"], outs
    assert outs[0][1:3] == ["1", "2"] and outs[1][1:3] == ["0", "2"]
    assert outs[0][3] == outs[1][3] and len(outs[0][3]) == 256 and set(outs[0][3]) != {"0"}


def test_config_header_matches_the_reference_header(tmp_path, golden_dir):
    """LBM::SimulationParams / lattice tables (SURVEY.md row a1): the same program compiled against this
    repo's LBMConfig.h prints what it prints against the reference's (stored, and live where the reference is mounted)."""
    src = os.path.join(ROOT, "tests", "cpp", "params_dump.cpp")
    ours = str(tmp_path / "ours")
    subprocess.run(["g++", "-std=c++17", "-O1", "-ffp-contract=off", "-I" + INC, src, "-o", ours], check=True)
    out = subprocess.run([ours], capture_output=True, text=True, check=True).stdout
    assert "Q 9 D 2" in out and "defaults 0.59999999999999998 0.01333 2048 512 120000 140" in out
    # default case: Re = 20.47 (SURVEY.md F7), cylinder (409, 256), r = 25
    nu = (0.6 - 0.5) / 3.0
    assert "derived %.17g %.17g 409 256 25" % (nu, 0.01333 * (2.0 * 0.05 * 512) / nu) in out
    assert out == json.load(open(os.path.join(golden_dir, "reference_pins.json")))["params_dump"]
    if os.path.exists(os.path.join(REF, "include", "LBMConfig.h")):
        theirs = str(tmp_path / "theirs")
        subprocess.run(["g++", "-std=c++20", "-O1", "-ffp-contract=off", "-I" + os.path.join(REF, "include"), src, "-o", theirs], check=True)
        assert subprocess.run([theirs], capture_output=True, text=True, check=True).stdout == out


def test_utils_header_matches_the_reference_header(tmp_path, golden_dir):
    """equilibrium_scalar / equilibrium_simd (8 outputs for i = 1..8) / is_stable: same values, bit for bit,
    as the reference's AVX2 versions built without FP contraction (stored, and live where the reference is mounted)."""
    src = os.path.join(ROOT, "tests", "cpp", "utils_dump.cpp")
    builds = [("ours", INC, "c++17")]
    if os.path.exists(os.path.join(REF, "include", "LBMUtils.h")):
        builds.append(("theirs", os.path.join(REF, "include"), "c++20"))
    outs = []
    for name, inc, std in builds:
        exe = str(tmp_path / name)
        subprocess.run(["g++", "-std=" + std, "-O1", "-mavx2", "-mfma", "-ffp-contract=off", "-I" + inc, src, "-o", exe], check=True)
        outs.append(subprocess.run([exe], capture_output=True, text=True, check=True).stdout)
    want = json.load(open(os.path.join(golden_dir, "reference_pins.json")))["utils_dump"]
    assert all(o == want for o in outs), "\n".join(outs)
