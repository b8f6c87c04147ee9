"""Multi-GPU parity: N x-slabs with the NCCL halo exchange (overlapped and not) against the
1-rank CPU oracle.  Needs >= 2 GPUs on the box (skipped otherwise); run with -m gpu."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import oracle as O
import parity_util as util
import geometry_cases as G

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# the cylinder straddles the face between slabs 0 and 1 of a 2-slab run (x = 64)
CASES = {
    "even": O.Case(nx=128, ny=48, cylinder_x=0.5, cylinder_radius=0.2, output_frequency=6, inlet_velocity=0.04),
    # odd ny: scalar bulk kernel, halo fused into the fix-up kernel instead of the bulk launch
    "periodic": O.Case(nx=96, ny=40, cylinder_x=0.02, cylinder_radius=0.2, output_frequency=6, inlet_velocity=0.04),  # flags=1 in the worker
    "odd": O.Case(nx=128, ny=47, cylinder_x=0.5, cylinder_radius=0.2, output_frequency=6, inlet_velocity=0.04),
    # several strips: the disc is centred on the face x = 64 (and lies across x = 32 .. 96 of a 4-slab run), and its
    # last row is the first row of the block of strip 1 at depths 2 / 3, B = 128 (tests/geometry_cases.py)
    "strip_edge": G.disc(128, 300, 64, G.block_lo(128, 3, 1) - 20, 20, output_frequency=6, inlet_velocity=0.04),
}


def n_gpus():
    import torch

    return torch.cuda.device_count()


# kernel variant / pass depth: 1/1 = one iteration per launch pair (3-population halo), 2/d = temporally blocked
# passes of depth d (wide halo stored by the pass itself, or sent by NCCL where forced)
@pytest.mark.parametrize("variant,depth", [(2, 2), (2, 3), (2, 1), (1, 1)])
@pytest.mark.parametrize("overlap", ["1", "0", "nccl"])
@pytest.mark.parametrize("world", [2, 4, 8])
@pytest.mark.parametrize("seed,case_name", [(0, "even"), (5, "even"), (5, "odd")])
def test_slabs_match_single_rank_oracle(tmp_path, world, overlap, seed, case_name, variant, depth):
    CASE = CASES[case_name]
    if n_gpus() < world:
        pytest.skip("needs %d GPUs" % world)
    if variant == 2 and overlap == "0":
        pytest.skip("the temporally blocked passes have one NCCL mode (in stream order)")
    steps = 37
    # "1": edge kernel + halo fused over peer memory when CUDA IPC is available (else the NCCL path);
    # "nccl": the overlapped NCCL send/recv path, forced; "0": exchange in stream order, no overlap
    env = dict(os.environ, LBM_B200_OVERLAP="0" if overlap == "0" else "1", LBM_B200_P2P="0" if overlap == "nccl" else "1",
               LBM_B200_VARIANT=str(variant), LBM_B200_TB_DEPTH=str(depth))
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
        env.pop(k, None)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
           "--master-port", str(29800 + os.getpid() % 150 + world), os.path.join(ROOT, "tests", "multi_gpu_worker.py"), str(tmp_path),
           str(steps), str(seed), case_name]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    if seed:
        state = util.random_state(CASE, seed)
        o = util.oracle_with_state(CASE, state)
    else:
        o = O.Oracle(CASE)
    rows, bad = o.run(steps)
    parts = [np.load(tmp_path / ("slab%d.npz" % k)) for k in range(world)]
    for key, want in (("f_next", o.f_next[1:-1, 1:-1]), ("f_current", o.f_current[1:-1, 1:-1]), ("rho", o.rho), ("ux", o.ux), ("uy", o.uy)):
        got = np.concatenate([p[key] for p in parts], axis=1)
        assert np.array_equal(got, want), "%s differs: max %.3e" % (key, np.abs(got - want).max())
    assert np.array_equal(parts[0]["g_rho"], o.rho) and np.array_equal(parts[0]["g_ux"], o.ux) and np.array_equal(parts[0]["g_uy"], o.uy)
    assert all(int(p["bad"]) == bad == -1 for p in parts)
    if overlap == "nccl":
        assert all(int(p["halo_p2p"]) == 0 for p in parts)
    print("halo_p2p:", [int(p["halo_p2p"]) for p in parts])
    total = sum(p["rows"][:, 1:3] for p in parts)
    assert np.array_equal(parts[0]["rows"][:, 0], rows[:, 0]) and np.abs(total - rows[:, 1:3]).max() <= 1e-13
    ofx, ofy = o.forces()
    assert abs(parts[1]["forces_total"][0] - ofx) <= 1e-13 and abs(parts[1]["forces_total"][1] - ofy) <= 1e-13
    assert abs(float(parts[0]["maxvel"][0]) - o.max_velocity()) <= 1e-15


@pytest.mark.parametrize("variant,depth", [(2, 2), (2, 3), (1, 1)])
@pytest.mark.parametrize("p2p", ["1", "0"])
def test_periodic_slabs_match_single_gpu(tmp_path, p2p, variant, depth):
    """Periodic-x channel over 2 slabs: every rank has a neighbour on BOTH sides (the same peer), the
    situation of the middle ranks of a longer chain.  Reference: the same engine on one GPU."""
    if n_gpus() < 2:
        pytest.skip("needs 2 GPUs")
    import lbm_b200

    steps, seed = 29, 3
    env = dict(os.environ, LBM_B200_P2P=p2p, LBM_B200_VARIANT=str(variant), LBM_B200_TB_DEPTH=str(depth))
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
        env.pop(k, None)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(29950 + os.getpid() % 40), os.path.join(ROOT, "tests", "multi_gpu_worker.py"), str(tmp_path),
           str(steps), str(seed), "periodic"]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    case = CASES["periodic"]
    s = lbm_b200.Solver(util.case_to_params(case, flags=1))
    s.initialise()
    s.upload_f(util.random_state(case, seed), 0)
    rows, bad = s.run(steps)
    parts = [np.load(tmp_path / ("slab%d.npz" % k)) for k in range(2)]
    got, want = np.concatenate([p["f_next"] for p in parts], axis=1), s.f_next()[1:-1, 1:-1]
    bad_cells = np.argwhere((got != want).any(axis=2))
    assert len(bad_cells) == 0, "%d cells differ, x range %d..%d, first %s" % (
        len(bad_cells), bad_cells[:, 1].min(), bad_cells[:, 1].max(), bad_cells[:5].tolist())
    assert np.array_equal(np.concatenate([p["f_current"] for p in parts], axis=1), s.f_current()[1:-1, 1:-1])
    rho, ux, uy = s.macros()
    assert np.array_equal(parts[0]["g_rho"], rho) and np.array_equal(parts[0]["g_ux"], ux) and np.array_equal(parts[0]["g_uy"], uy)
    print("halo_p2p:", [int(p["halo_p2p"]) for p in parts])
    s.close()


def _torchrun(world, script_args, env, port_base, timeout=600):
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
        env.pop(k, None)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
           "--master-port", str(port_base + os.getpid() % 40), os.path.join(ROOT, "tests", "multi_gpu_worker.py")] + script_args
    return subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=timeout)


@pytest.mark.parametrize("variant,depth", [(2, 2), (1, 1)])
def test_observers_between_steps_with_skewed_ranks(tmp_path, variant, depth):
    """rho / u are read in the middle of a run while the ranks are deliberately out of step (odd ranks sleep before
    every observation, even ranks right after it): an observer that pulls from the previous buffer's ghost columns
    must not see the halo of a neighbour that is already one pass ahead (ADVICE r1: the peer-store protocol has to
    cover observers)."""
    world = 2
    if n_gpus() < world:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ, LBM_B200_VARIANT=str(variant), LBM_B200_TB_DEPTH=str(depth))
    r = _torchrun(world, [str(tmp_path), "0", "5", "even", "skewed"], env, 30050)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    CASE = CASES["even"]
    o = util.oracle_with_state(CASE, util.random_state(CASE, 5))
    parts = [np.load(tmp_path / ("skew%d.npz" % k)) for k in range(world)]
    done = 0
    for k, n in enumerate((1, 3, 4, 7, 2, 5)):
        o.run(n)
        done += n
        for key, want in (("rho", o.rho), ("ux", o.ux), ("uy", o.uy)):
            got = np.concatenate([p["%s_%d" % (key, k)] for p in parts], axis=1)
            assert np.array_equal(got, want), "%s after %d iterations differs: max %.3e" % (key, done, np.abs(got - want).max())
    got = np.concatenate([p["f_next"] for p in parts], axis=1)
    assert np.array_equal(got, o.f_next[1:-1, 1:-1])


def test_a_silent_neighbour_is_an_error_not_a_hang(tmp_path):
    """Rank 1 stops stepping; rank 0's step kernels wait for its halo, run into the bound
    (LBM_B200_HALO_TIMEOUT_MS) and every synchronising call on rank 0 returns LBM_ERR_NCCL within seconds."""
    if n_gpus() < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ, LBM_B200_HALO_TIMEOUT_MS="1500")
    r = _torchrun(2, [str(tmp_path), "0", "0", "even", "silent"], env, 30100, timeout=300)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    res = np.load(tmp_path / "silent0.npz")
    assert int(res["halo_p2p"]) == 0 or (int(res["code"]) == -3 and float(res["seconds"]) < 60.0), (int(res["code"]), float(res["seconds"]))
    if int(res["halo_p2p"]):
        assert b"timed out" in bytes(res["message"])


@pytest.mark.parametrize("world", [2, 4, 8])
@pytest.mark.parametrize("seed,case_name,steps", [(5, "even", 37), (5, "even", 36), (0, "even", 21), (5, "odd", 37)])
def test_in_place_aa_variant_over_slabs(tmp_path, world, seed, case_name, steps):
    """LBM_FLAG_AA (ONE population buffer per GPU) over x-slabs: after every E-step the edge columns go to the
    neighbours' ghost columns, after every O-step what was pushed across a face goes into the neighbours' edge
    columns -- plain stores into peer memory plus the step-counter hand-shake.  Populations, f_current, forces rows
    and the verdict bit-identical to the 1-rank oracle at both parities; rho / u to rounding (the single buffer
    cannot keep them, tests/test_gpu_aa.py)."""
    CASE = CASES[case_name]
    if n_gpus() < world:
        pytest.skip("needs %d GPUs" % world)
    env = dict(os.environ, LBM_TEST_AA="1")
    r = _torchrun(world, [str(tmp_path), str(steps), str(seed), case_name], env, 30200)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    o = util.oracle_with_state(CASE, util.random_state(CASE, seed)) if seed else O.Oracle(CASE)
    rows, bad = o.run(steps)
    parts = [np.load(tmp_path / ("slab%d.npz" % k)) for k in range(world)]
    for key, want in (("f_next", o.f_next[1:-1, 1:-1]), ("f_current", o.f_current[1:-1, 1:-1])):
        got = np.concatenate([p[key] for p in parts], axis=1)
        diff = (got != want).any(axis=2)
        assert not diff.any(), "%s differs in %d cells, columns %s" % (key, int(diff.sum()), np.unique(np.nonzero(diff)[1])[:12])
    for key, want, tol in (("rho", o.rho, 1e-14), ("ux", o.ux, 1e-14), ("uy", o.uy, 1e-14)):
        got = np.concatenate([p[key] for p in parts], axis=1)
        assert np.abs(got - want).max() <= tol, key
    assert all(int(p["bad"]) == bad == -1 for p in parts)
    assert all(int(p["halo_p2p"]) == 1 for p in parts)
    total = sum(p["rows"][:, 1:3] for p in parts)
    assert np.array_equal(parts[0]["rows"][:, 0], rows[:, 0]) and np.abs(total - rows[:, 1:3]).max() <= 1e-13
