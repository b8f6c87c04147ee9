"""GPU parity at strip, block and chunk edges: the lattices of tests/geometry_cases.py (derived from the launch geometry
of k_tb), seeded random states, step sequences that mix pass depths, every observable bit for bit against the CPU
oracle -- f_next, f_current, rho / ux / uy, the forces rows of run(), the forces and the stability verdict.

A. k_tb at depths 1, 2, 3 over the whole chunk-width sweep (LBM_B200_TB_XC, read at every launch).
B. The one-iteration kernels (variants 0 and 1, A-B and in place) on heights around their 256-row blocks and on the
   shapes past 65 535 columns / rows (their grid-stride loops).
C. The settings read once per process (block height 64 / 256, the one-column-lag march, no fast lane, the fused later
   stages): A's chunk width 16 in a child process each.
D. Body force and periodic y on a multi-strip lattice: k_tb against variants 0 and 1 of this engine (no reference).
E. The multi-strip case of tests/test_gpu_multi.py over 2 and 4 GPUs (skipped with fewer).
On a difference the message names the first differing (y, x), its strip (y // H) and its chunk (x // xc)."""
import os
import subprocess
import sys
from functools import lru_cache
from types import SimpleNamespace

import numpy as np
import pytest

import geometry_cases as G
import parity_util as util

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def block_height():
    """The block height the library runs in this process (lbm_tb.cu block_threads: 64 and 256 are taken, else 128)."""
    try:
        v = int(os.environ.get("LBM_B200_TB_B", "128"))
    except ValueError:
        v = 128
    return v if v in (64, 256) else G.DEFAULT_B


B = block_height()
CASES = G.all_cases(B)
# step(n) splits into passes of up to the solver's depth (odd and even n), run(n) ends a pass at every output step
# (the cases' output frequencies are odd)
PLAN = (("step", 1), ("step", 2), ("run", 7), ("step", 3), ("step", 5), ("run", 4), ("step", 1))
FIELDS = ("f_next", "f_current", "rho", "ux", "uy")


@lru_cache(maxsize=2)
def oracle_snapshots(name, seed=3):
    case = CASES.get(name) or PARTIAL_Y[name]
    o = util.oracle_with_state(case, util.random_state(case, seed))
    snaps = []
    for kind, n in PLAN:
        rows, bad = o.run(n)
        snaps.append(SimpleNamespace(rows=rows, bad=bad, forces=o.forces(), **{k: getattr(o, k).copy() for k in FIELDS}))
    assert all(s.bad == -1 for s in snaps)
    o.close()
    return snaps


def first_difference(s, want, H, xc):
    got = {"f_next": s.f_next(), "f_current": s.f_current()}
    got["rho"], got["ux"], got["uy"] = s.macros()
    for k in FIELDS:
        d = got[k] != getattr(want, k)
        if d.ndim == 3:
            d = d.any(axis=2)[1:-1, 1:-1]  # padded -> interior (the ghost ring's differences show up next to it)
        if d.any():
            y, x = (int(v) for v in np.argwhere(d)[0])
            return "%s differs in %d cells, first at (y, x) = (%d, %d): strip %d, chunk %s" % (
                k, int(d.sum()), y, x, y // H, (x // xc) if xc else "?")
    return "no difference in the interior"


def check(s, want, what, H, xc, macros_exact=True):
    try:
        util.compare_state(s, want, what, exact=True, macros_exact=macros_exact)
    except AssertionError as e:
        raise AssertionError("%s -- %s" % (e, first_difference(s, want, H, xc))) from None


def replay(s, name, what, H, xc, macros_exact=True):
    case = CASES.get(name) or PARTIAL_Y[name]
    s.upload_f(util.random_state(case, 3), iteration=0)
    for (kind, n), want in zip(PLAN, oracle_snapshots(name)):
        if kind == "step":
            s.step(n)
        else:
            rows, bad = s.run(n)
            assert bad == want.bad == -1 and np.array_equal(rows, want.rows), "%s run(%d): forces rows" % (what, n)
        check(s, want, "%s after %s(%d)" % (what, kind, n), H, xc, macros_exact)
        assert s.forces() == want.forces, what
    ok, bad = s.check_stability()
    assert ok and bad == -1


# ---- A ------------------------------------------------------------------------------------------------------------
XCS = [str(x) for x in G.XC_SWEEP] + ["nx"]


@pytest.mark.parametrize("xc", XCS, ids=["xc" + x for x in XCS])
@pytest.mark.parametrize("depth", [1, 2, 3], ids=["d1", "d2", "d3"])
@pytest.mark.parametrize("name", list(CASES))
def test_tb_passes_at_strip_and_chunk_edges(name, depth, xc, monkeypatch):
    import lbm_b200

    case = CASES[name]
    width = case.nx + 3 if xc == "nx" else int(xc)
    monkeypatch.setenv("LBM_B200_TB_XC", str(width))
    s = lbm_b200.Solver(util.case_to_params(case))
    s.set_kernel_variant(lbm_b200.VARIANT_TB)
    s.set_pass_depth(depth)
    s.initialise()
    assert s.info().pass_depth == depth
    try:
        replay(s, name, "%s B=%d depth %d xc %d" % (name, B, depth, width), G.rows_per_strip(B, depth), width)
    finally:
        s.close()


# ---- B ------------------------------------------------------------------------------------------------------------
# around the 256-row blocks of k_bulk_vec2 / k_bulk_scalar and the AA kernels (lbm_kernels.cu, lbm_aa.cu); the disc
# crosses row 256 (or is cut by the top wall there)
PARTIAL_Y = {"ny%d" % ny: G.disc(40, ny, 15, 252, 6, output_frequency=7, inlet_velocity=0.04)
             for ny in (254, 255, 256, 257, 258, 300, 511, 513)}
PARTIAL_Y.update(G.extreme_cases())


@pytest.mark.parametrize("variant,flags", [(0, 0), (1, 0), (0, 16), (1, 16)], ids=["v0", "v1", "v0_aa", "v1_aa"])
@pytest.mark.parametrize("name", list(PARTIAL_Y))
def test_one_iteration_kernels_at_partial_y_blocks_and_wide_grids(name, variant, flags):
    """rho / ux / uy of the in-place variant are recovered from collision invariants (tests/test_gpu_aa.py): there
    they are held to the tolerance of parity_util, everything else bit for bit."""
    import lbm_b200

    s = lbm_b200.Solver(util.case_to_params(PARTIAL_Y[name], flags=flags))
    s.set_kernel_variant(variant)
    s.initialise()
    try:
        replay(s, name, "%s v%d flags %d" % (name, variant, flags), 256, 0, macros_exact=(flags == 0))
    finally:
        s.close()


# ---- C ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("knob,value", [(k, v) for k in ("LBM_B200_TB_B", "LBM_B200_TB_SKEW", "LBM_B200_TB_FAST", "LBM_B200_TB_FUSED")
                                        for v in G.KNOBS[k]])
def test_settings_read_once_per_process(knob, value):
    """A child pytest over A at chunk width 16 (the extreme shapes left out) with the setting in its environment; the
    strip cases are derived for the block height the child runs."""
    env = dict(os.environ, **{knob: value})
    env.pop("LBM_B200_TB_XC", None)
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-x", "-p", "no:cacheprovider", "-m", "gpu",
                        "-k", "test_tb_passes_at_strip_and_chunk_edges and xc16 and not wide and not tall"],
                       env=env, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-1000:]
    last = r.stdout.strip().splitlines()[-1]
    assert " passed" in last and "skipped" not in last and "failed" not in last, r.stdout[-500:]


# ---- D ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("flags", [0, 2 | 4, 2], ids=["walls_inlet_outlet", "periodic_y_no_cylinder", "periodic_y"])
def test_forced_and_periodic_y_passes_over_several_strips(flags):
    """No reference has these modes (SURVEY.md F11): k_tb at depths 1 / 2 / 3 against the one-iteration kernels,
    variants 0 and 1, bit for bit.  A body force in x and y, three strips, the disc across the first strip edge."""
    import lbm_b200

    H = G.rows_per_strip(B, 3)
    case = G.disc(96, 3 * H - 20, 40, H, 10, output_frequency=7, inlet_velocity=0.03)
    state = util.random_state(case, 4)
    outs = []
    for variant, depth in ((0, 1), (1, 1), (2, 1), (2, 2), (2, 3)):
        s = lbm_b200.Solver(util.case_to_params(case, flags=flags, body_force_x=2e-6, body_force_y=-1.5e-6))
        s.set_kernel_variant(variant)
        s.set_pass_depth(depth)
        s.initialise()
        s.upload_f(state, 0)
        got = []
        for kind, n in PLAN:
            rows = s.run(n) if kind == "run" else None
            if kind == "step":
                s.step(n)
            got.append((s.f_next()[1:-1, 1:-1].copy(), s.f_current()[1:-1, 1:-1].copy()) + tuple(a.copy() for a in s.macros())
                       + (s.forces(), rows))
        got.append(tuple(s.check_stability()))
        outs.append(got)
        s.close()
    assert outs[0][-1] == (True, -1)
    for k, other in enumerate(outs[1:], 1):
        for step, (a, b) in enumerate(zip(outs[0], other)):
            if step == len(PLAN):
                assert a == b, k
                continue
            for j, (x, y) in enumerate(zip(a, b)):
                if j < 5:
                    d = x != y
                    if d.ndim == 3:
                        d = d.any(axis=2)
                    if d.any():
                        yy, xx = (int(v) for v in np.argwhere(d)[0])
                        raise AssertionError("run %d, %s(%d), %s: first difference at (y, x) = (%d, %d), strip %d" % (
                            k, PLAN[step][0], PLAN[step][1], FIELDS[j], yy, xx, yy // H))
                elif j == 5:
                    assert x == y, (k, step, "forces")
                elif x is not None:
                    assert x[1] == y[1] and np.array_equal(x[0], y[0]), (k, step, "rows")


# ---- E ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("world,overlap,variant,depth", [
    (2, "1", 2, 2), (2, "1", 2, 3), (2, "1", 1, 1), (4, "1", 2, 2), (4, "1", 2, 3), (4, "1", 1, 1), (2, "nccl", 2, 3), (4, "nccl", 2, 2)])
def test_multi_strip_slabs(tmp_path, world, overlap, variant, depth):
    """The slab-edge chunks (tb_push) over several strips: tests/test_gpu_multi.py's "strip_edge" case, the disc on
    the slab face with its last row on the edge of strip 1's block, against the 1-rank oracle."""
    import test_gpu_multi as M

    M.test_slabs_match_single_rank_oracle(tmp_path, world, overlap, 5, "strip_edge", variant, depth)
