"""Temporal blocking, pinned on the CPU: the thread program of the sm_100a kernel k_tb
(csrc/lbm_tb.cuh, a __host__ __device__ template) is run thread for thread on the host
(oracle/prototypes/tb_emul.cpp: one std::thread per CUDA thread, std::barrier for __syncthreads) and must
equal the oracle's single steps bit for bit -- for every depth, block height, chunk width, with walls,
inlet, outlet, the corner quirks (SURVEY.md F4), the obstacle inside / across blocks and slabs, and the
wide halo that x-slabs store into each other's ghost columns."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import oracle as O
import geometry_cases as G

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "oracle", "prototypes", "libtbemul.so")

CASES = {
    "64x32": O.Case(nx=64, ny=32, cylinder_x=0.3, cylinder_radius=0.2, output_frequency=3),
    "70x33": O.Case(nx=70, ny=33, cylinder_x=0.3, cylinder_radius=0.15, output_frequency=5, inlet_velocity=0.05),
    "cyl_on_wall": O.Case(nx=80, ny=40, cylinder_x=0.5, cylinder_y=0.1, cylinder_radius=0.2, output_frequency=4),
    "cyl_at_inlet": O.Case(nx=72, ny=36, cylinder_x=0.03, cylinder_y=0.5, cylinder_radius=0.25, output_frequency=5),
    "cyl_at_outlet_corner": O.Case(nx=72, ny=36, cylinder_x=0.97, cylinder_y=0.9, cylinder_radius=0.3, output_frequency=5),
    "tiny_6x4": O.Case(nx=6, ny=4, cylinder_radius=0.3, output_frequency=2),
    "slabs_128x48": O.Case(nx=128, ny=48, cylinder_x=0.5, cylinder_radius=0.2, output_frequency=6, inlet_velocity=0.04),
}


@pytest.fixture(scope="module", params=["skewed", "skewed_fused", "skewed_no_fast_lane", "one_column_lag"])
def emu(request):
    """The marches of lbm_tb.cuh: the skewed one (stage k two columns behind stage k-1, the default) with and without
    its fast lane for plain stretches (and with the later stages of the fast lane fused), and the one-column-lag one with its second cell of prefetched registers."""
    L = C.CDLL(LIB)
    L.tb_set_force.argtypes = [C.c_double, C.c_double]
    L.tb_set_skew({"skewed": 2, "skewed_fused": 3, "skewed_no_fast_lane": 1, "one_column_lag": 0}[request.param])
    L.tb_emulate.restype = C.c_int
    L.tb_emulate.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_double, C.c_int, C.c_int,
                             C.POINTER(C.c_int), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
    return L


def padded_solid(o, case):
    """The global solid mask on the padded grid (ghost cells of a 1-rank job are never solid)."""
    m = np.zeros((case.ny + 2, case.nx + 2), dtype=np.uint8)
    m[1:-1, 1:-1] = o.solid
    return np.ascontiguousarray(m)


def emulate(emu, case, state, solid, depths, world=1, flags=0, B=32, xc=16, edge_cols=4, halo_w=2, first_is_current=0, iter0=1):
    st = np.ascontiguousarray(state.copy())
    d = (C.c_int * len(depths))(*depths)
    bad = emu.tb_emulate(st.ctypes.data, solid.ctypes.data, case.nx, case.ny, case.tau, case.inlet_velocity, world, flags, d,
                         len(depths), B, xc, edge_cols, halo_w, first_is_current, iter0)
    return st, bad


def random_f_current(case, seed, amplitude=0.05):
    rng = np.random.default_rng(seed)
    w = np.array([4 / 9] + [1 / 9] * 4 + [1 / 36] * 4)
    f = w * (1.0 + amplitude * rng.standard_normal((case.ny + 2, case.nx + 2, 9)))
    o = O.Oracle(case)
    init = o.f_current.copy()
    for sl in ((0, slice(None)), (-1, slice(None)), (slice(None), 0), (slice(None), -1)):
        f[sl] = init[sl]
    return np.ascontiguousarray(f)


@pytest.mark.parametrize("name", [n for n in CASES if n != "slabs_128x48"])
@pytest.mark.parametrize("depths,B,xc", [((2,), 32, 16), ((2, 2, 1, 2), 16, 5), ((1, 1), 32, 7), ((3, 2), 32, 1000), ((3, 3), 16, 3)])
def test_passes_equal_oracle_steps(emu, name, depths, B, xc):
    case = CASES[name]
    o = O.Oracle(case)
    o.f_current[...] = random_f_current(case, 5)
    o.run(1)  # a post-collision state whose ghost ring is in its permanent form (F4)
    src, solid = o.f_next.copy(), padded_solid(o, case)
    got, bad = emulate(emu, case, src, solid, depths, B=B, xc=xc)
    o.run(sum(depths))
    assert bad == 0x7fffffff
    assert np.array_equal(got[1:-1, 1:-1], o.f_next[1:-1, 1:-1]), (name, depths, int((got[1:-1, 1:-1] != o.f_next[1:-1, 1:-1]).sum()))


@pytest.mark.parametrize("name", ["64x32", "cyl_at_inlet"])
def test_first_iteration_collides_f_current_in_place(emu, name):
    """Depth 1 with pull = 0 is the iteration after initialise / upload: no pull, no rule, no check."""
    case = CASES[name]
    state = random_f_current(case, 9)
    o = O.Oracle(case)
    o.f_current[...] = state
    solid = padded_solid(o, case)
    got, bad = emulate(emu, case, state, solid, (1, 2, 1), first_is_current=1, iter0=0)
    o.run(4)
    assert bad == 0x7fffffff
    assert np.array_equal(got[1:-1, 1:-1], o.f_next[1:-1, 1:-1])


@pytest.mark.parametrize("world", [2, 4])
@pytest.mark.parametrize("depths,halo_w,edge_cols", [((2, 2, 2), 2, 4), ((1, 2, 1, 1, 2), 2, 2), ((3, 1, 2, 3), 3, 4), ((2, 1), 3, 8)])
def test_slabs_with_the_wide_halo_equal_the_single_rank_oracle(emu, world, depths, halo_w, edge_cols):
    """x-slabs: each pass's last stage stores the halo_w edge columns into the neighbour's ghost columns; ghost
    populations nobody stores are NaN in the emulation, so a pull that reaches for one shows up."""
    case = CASES["slabs_128x48"]  # the cylinder straddles the face between slabs
    o = O.Oracle(case)
    o.f_current[...] = random_f_current(case, 3)
    o.run(1)
    src, solid = o.f_next.copy(), padded_solid(o, case)
    got, bad = emulate(emu, case, src, solid, depths, world=world, B=32, xc=6, edge_cols=edge_cols, halo_w=halo_w)
    o.run(sum(depths))
    assert bad == 0x7fffffff
    diff = (got[1:-1, 1:-1] != o.f_next[1:-1, 1:-1]).any(axis=2)
    assert not diff.any(), ("cells", int(diff.sum()), "columns", np.unique(np.nonzero(diff)[1])[:20])


def test_slabs_first_iteration(emu):
    case = CASES["slabs_128x48"]
    state = random_f_current(case, 4)
    o = O.Oracle(case)
    o.f_current[...] = state
    got, bad = emulate(emu, case, state, padded_solid(o, case), (1, 2, 2, 1), world=2, xc=9, edge_cols=4, first_is_current=1, iter0=0)
    o.run(6)
    assert np.array_equal(got[1:-1, 1:-1], o.f_next[1:-1, 1:-1])


def test_instability_is_flagged_at_the_reference_timestep(emu):
    case = O.Case(nx=96, ny=24, tau=0.52, inlet_velocity=0.1, output_frequency=50)
    o = O.Oracle(case)
    _, obad = o.run(400)
    assert obad > 4
    o2 = O.Oracle(case)
    o2.run(obad - 3)  # iterations 0 .. obad-4 done; the emulation continues with iteration obad-3
    src, solid = o2.f_next.copy(), padded_solid(o2, case)
    for depths in ((2, 2, 2), (1, 2, 2, 1), (3, 3)):
        _, bad = emulate(emu, case, src, solid, depths, iter0=obad - 3)
        assert bad == obad, (depths, bad, obad)


@pytest.mark.parametrize("flags", [1, 2, 3])
def test_periodic_passes_are_self_consistent(emu, flags):
    """The reference has no periodic mode (SURVEY.md F11): depth-2 / depth-3 passes against single depth-1 steps of
    the same code, obstacle included, wrapped addressing instead of ghost copies."""
    case = CASES["64x32"]
    o = O.Oracle(case)
    rng = np.random.default_rng(1)
    w = np.array([4 / 9] + [1 / 9] * 4 + [1 / 36] * 4)
    state = np.ascontiguousarray(w * (1.0 + 0.05 * rng.standard_normal((case.ny + 2, case.nx + 2, 9))))
    solid = padded_solid(o, case)
    state[solid != 0] = w  # solid cells hold w in every reachable post-collision state and are never stored
    ref, _ = emulate(emu, case, state, solid, (1,) * 6, flags=flags, xc=1000)
    for depths in ((2, 2, 2), (3, 3), (2, 1, 3)):
        got, _ = emulate(emu, case, state, solid, depths, flags=flags, B=16, xc=7)
        assert np.array_equal(got[1:-1, 1:-1], ref[1:-1, 1:-1]), depths


def test_the_fast_lane_carries_the_plain_stretches():
    """The skewed march hands every stretch of plain, unmasked columns to tb_fast_lane: on a channel whose cylinder
    sits in one corner of the lattice that is most of the march (and none of it with the lane switched off), so the
    parity cases above do exercise it."""
    L = C.CDLL(LIB)
    L.tb_emulate.restype = C.c_int
    L.tb_emulate.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_double, C.c_int, C.c_int,
                             C.POINTER(C.c_int), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
    case = O.Case(nx=96, ny=64, cylinder_x=0.15, cylinder_y=0.2, cylinder_radius=0.1, output_frequency=5)
    o = O.Oracle(case)
    o.run(1)
    src, solid = o.f_next.copy(), padded_solid(o, case)
    o.run(3)
    counts = {}
    for mode in (2, 1):
        L.tb_set_skew(mode)
        fast, general = C.c_longlong(), C.c_longlong()
        L.tb_step_counts(C.byref(fast), C.byref(general))  # reset
        got, bad = emulate(L, case, src, solid, (3,), B=32, xc=16)
        L.tb_step_counts(C.byref(fast), C.byref(general))
        counts[mode] = (fast.value, general.value)
        assert np.array_equal(got[1:-1, 1:-1], o.f_next[1:-1, 1:-1])
    assert counts[1][0] == 0 and counts[1][1] == sum(counts[2])
    assert counts[2][0] > 3 * counts[2][1], counts


@pytest.mark.parametrize("depths", [(3,), (2, 3), (1,), (3, 2)])
def test_the_last_pass_emits_the_moments_of_its_last_collision(emu, depths):
    """TbArgs::m_rho / m_ux / m_uy (what lbm_run's last pass hands to k_macros_finish): rho, ux, uy exactly as the
    reference's collision stores them (include/LBMSolver.h:112-114), from the general step and from the fast lane;
    obstacle cells keep rho = 1, u = 0 (:260-261).  The inlet / outlet columns get their overrides later
    (k_macros_finish, GPU tests): compared here without them."""
    case = CASES["70x33"]
    o = O.Oracle(case)
    o.f_current[...] = random_f_current(case, 9)
    o.run(1)
    src, solid = o.f_next.copy(), padded_solid(o, case)
    sink = [np.full(case.nx * case.ny, np.nan) for _ in range(3)]
    emu.tb_set_macro_sink.argtypes = [C.c_void_p] * 3
    emu.tb_set_macro_sink(*[a.ctypes.data for a in sink])
    try:
        got, bad = emulate(emu, case, src, solid, depths, B=32, xc=16)
    finally:
        emu.tb_set_macro_sink(None, None, None)
    o.run(sum(depths))
    assert np.array_equal(got[1:-1, 1:-1], o.f_next[1:-1, 1:-1])
    for mine, want in zip(sink, (o.rho, o.ux, o.uy)):
        mine = mine.reshape(case.nx, case.ny).T  # native [x*ny + y] -> [y, x]
        assert np.array_equal(mine[:, 1:-1], np.asarray(want)[:, 1:-1])


def _strip_edge_params():
    """The obstacle-row cases of tests/geometry_cases.py at the shipped block height, B = 128 (strip 1's block edges),
    with the passes of the depths they were derived for."""
    out = []
    for depth, depths in ((1, (1, 1)), (3, (3, 2))):
        for name in G.row_edge_cases(G.DEFAULT_B, depth):
            out.append(pytest.param(depth, name, depths, id=name))
    return out


@pytest.mark.parametrize("depth,name,depths", _strip_edge_params())
def test_strip_edges_at_the_shipped_block_height(emu, depth, name, depths):
    """B = 128 (and xc = 8, so that every block of 128 threads has a short march): the obstacle's rows just inside and
    just outside the block of strip 1, which decides whether that block looks at the mask at all."""
    case = G.row_edge_cases(G.DEFAULT_B, depth)[name]
    assert case.nx <= 40
    o = O.Oracle(case)
    o.f_current[...] = random_f_current(case, 6)
    o.run(1)
    src, solid = o.f_next.copy(), padded_solid(o, case)
    got, bad = emulate(emu, case, src, solid, depths, B=G.DEFAULT_B, xc=8)
    o.run(sum(depths))
    assert bad == 0x7fffffff
    diff = (got[1:-1, 1:-1] != o.f_next[1:-1, 1:-1]).any(axis=2)
    where = np.argwhere(diff)
    assert not diff.any(), "%d cells differ, first (y, x) = %s, strip %d" % (
        len(where), tuple(where[0]), where[0][0] // G.rows_per_strip(G.DEFAULT_B, depth))


@pytest.mark.parametrize("B", [64, 128])
def test_the_default_case_at_block_heights_the_device_runs(B):
    """Multi-strip at B = 64 (ny = 150: three strips) and B = 128, the skewed march with its fast lane."""
    L = C.CDLL(LIB)
    L.tb_emulate.restype = C.c_int
    L.tb_emulate.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_double, C.c_int, C.c_int,
                             C.POINTER(C.c_int), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
    L.tb_set_skew(2)
    case = G.disc(36, 150 if B == 64 else 260, 12, G.rows_per_strip(B, 3), 9, output_frequency=5)
    o = O.Oracle(case)
    o.f_current[...] = random_f_current(case, 8)
    o.run(1)
    src, solid = o.f_next.copy(), padded_solid(o, case)
    got, bad = emulate(L, case, src, solid, (3, 1, 2), B=B, xc=6)
    o.run(6)
    assert bad == 0x7fffffff
    assert np.array_equal(got[1:-1, 1:-1], o.f_next[1:-1, 1:-1])


@pytest.mark.parametrize("flags", [0, 1, 2, 3])
@pytest.mark.parametrize("B,name", [(16, "64x32"), (32, "70x33")])
def test_forced_passes_are_self_consistent(emu, flags, B, name):
    """A body force (Fx and Fy) selects k_tb<T, B, FORCED = true>, which has no reference: depth-2 / depth-3 passes
    against single depth-1 passes of the same code, with the obstacle, walls, inlet and outlet (flags 0) and the
    periodic edges, over several strips and chunks."""
    case = CASES[name]
    o = O.Oracle(case)
    rng = np.random.default_rng(2)
    w = np.array([4 / 9] + [1 / 9] * 4 + [1 / 36] * 4)
    state = np.ascontiguousarray(w * (1.0 + 0.05 * rng.standard_normal((case.ny + 2, case.nx + 2, 9))))
    solid = padded_solid(o, case)
    state[solid != 0] = w
    emu.tb_set_force.argtypes = [C.c_double, C.c_double]
    plain, _ = emulate(emu, case, state, solid, (1,) * 6, flags=flags, B=B, xc=1000)
    emu.tb_set_force(2e-5, -3e-5)
    try:
        ref, _ = emulate(emu, case, state, solid, (1,) * 6, flags=flags, B=B, xc=1000)
        assert not np.array_equal(ref[1:-1, 1:-1], plain[1:-1, 1:-1])  # the force does act
        for depths in ((2, 2, 2), (3, 3), (2, 1, 3)):
            got, _ = emulate(emu, case, state, solid, depths, flags=flags, B=B, xc=7)
            assert np.array_equal(got[1:-1, 1:-1], ref[1:-1, 1:-1]), depths
    finally:
        emu.tb_set_force(0.0, 0.0)
