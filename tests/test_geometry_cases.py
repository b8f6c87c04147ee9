"""The lattices of tests/geometry_cases.py hit the strip, block and chunk edges they claim to, for every block height
the library accepts, every pass depth and every chunk width of the sweep -- checked from the oracle's solid mask, so
the GPU parity cases are known to test those edges before any GPU time is spent.  And the LBM_B200_TB_* settings
those tests set are ones csrc/lbm_tb.cu reads and accepts."""
import os
import re

import pytest

from oracle import oracle as O
import geometry_cases as G

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TB_CU = os.path.join(ROOT, "highperformancecomputing-latticeboltzmannmethod_b200", "csrc", "lbm_tb.cu")

_extent = {}


def extent(name, case):
    if name not in _extent:
        o = O.Oracle(case)
        _extent[name] = (G.solid_extent(o.solid), int(o.solid.sum()))
        o.close()
    return _extent[name]


@pytest.mark.parametrize("B", G.BLOCKS)
def test_heights_fill_one_to_three_strips_and_a_few_rows_more(B):
    cases = G.all_cases(B)
    heights = {c.ny for c in cases.values()}
    for depth in (1, 2, 3):
        H = G.rows_per_strip(B, depth)
        want = {k * H + r for k in (1, 2, 3) for r in range(-1, 4) if k * H + r <= G.NY_MAX}
        assert len(want) >= 10 and want <= heights, (B, depth, sorted(want - heights))
    assert any(ny % 2 for ny in heights)


@pytest.mark.parametrize("depth", [1, 2, 3])
@pytest.mark.parametrize("B", G.BLOCKS)
def test_obstacle_rows_sit_on_either_side_of_a_block_edge(B, depth):
    """For a strip s >= 1 with block rows [lo, lo + B): the obstacle's rows [ylo, yhi) end at yhi = lo - 1, lo, lo + 1
    (the last row just misses the block / is its first row) or start at ylo = lo + B - 1, lo + B, lo + B + 1."""
    H = G.rows_per_strip(B, depth)
    hit = set()
    span = wall = False
    for name, case in G.all_cases(B).items():
        (ylo, yhi, _, _), n = extent(name, case)
        assert n > 0, name
        strips = -(-case.ny // H)
        for s in range(1, strips):
            lo = G.block_lo(B, depth, s)
            if yhi - lo in (-1, 0, 1):
                hit.add(("yhi", yhi - lo))
            if ylo - (lo + B) in (-1, 0, 1):
                hit.add(("ylo", ylo - (lo + B)))
            if ylo < s * H < yhi:  # rows stored by strips s - 1 and s
                span = True
        _, cy, r = G.disc_of(case)
        wall = wall or (cy - r < 0 and ylo == 0) or (cy + r >= case.ny and yhi == case.ny)
    assert hit == {(k, d) for k in ("yhi", "ylo") for d in (-1, 0, 1)}, sorted(hit)
    assert span and wall


@pytest.mark.parametrize("xc", [x for x in G.XC_SWEEP if x > 1])
def test_obstacle_columns_sit_next_to_a_chunk_edge(xc):
    """For every chunk width of the sweep, the obstacle's first and last column at -3 .. +3 from an interior chunk
    edge j xc (0 < j xc < nx); and obstacles touching, next to and cut by the inlet and the outlet column."""
    hit = set()
    inlet, outlet = set(), set()
    for name, case in G.all_cases(G.DEFAULT_B).items():
        (_, _, xf, xl), _ = extent(name, case)
        for j in range(1, -(-case.nx // xc)):
            for which, x in (("first", xf), ("last", xl)):
                if x - j * xc in G.EDGE_OFFSETS:
                    hit.add((which, x - j * xc))
        cx, _, r = G.disc_of(case)
        if xf <= 2:
            inlet.add("cut" if cx - r < 0 else xf)
        if xl >= case.nx - 3:
            outlet.add("cut" if cx + r >= case.nx else case.nx - 1 - xl)
    assert hit == {(w, d) for w in ("first", "last") for d in G.EDGE_OFFSETS}, sorted(hit)
    assert {"cut", 0, 1, 2} <= inlet and {"cut", 0, 1, 2} <= outlet, (inlet, outlet)


def test_extreme_shapes_have_one_solid_cell_past_65535():
    for name, case in G.extreme_cases().items():
        (ylo, yhi, xf, xl), n = extent(name, case)
        assert n == 1 and (case.nx, case.ny) in (G.WIDE, G.TALL)
        assert max(xf, ylo) > 65535


@pytest.mark.parametrize("B", G.BLOCKS)
def test_lattices_stay_small(B):
    for name, case in G.all_cases(B).items():
        if name in G.extreme_cases():
            continue
        assert case.nx <= G.NX_MAX and case.ny <= G.NY_MAX, (name, case.nx, case.ny)


def test_the_settings_the_gpu_tests_use_are_read_and_accepted():
    """A renamed knob would turn a GPU test into a rerun of the default: every LBM_B200_TB_* name the tests set is read
    in lbm_tb.cu, and the values they set select something other than the default."""
    src = open(TB_CU).read()
    for name in G.KNOBS:
        assert re.search(r'env_int\("%s",' % name, src), name
    # block height: 64 and 256 are taken, anything else means 128
    assert re.search(r"v == 256 \? 256 : \(v == 64 \? 64 : 128\)", src)
    assert set(G.KNOBS["LBM_B200_TB_B"]) == {"64", "256"} and G.DEFAULT_B == 128 and set(G.BLOCKS) == {64, 128, 256}
    # chunk width: a positive value is used as it is, <= 0 picks the default
    assert re.search(r'int xc = env_int\("LBM_B200_TB_XC", 0\);\s*if \(xc <= 0\)', src)
    assert all(int(v) > 0 for v in G.KNOBS["LBM_B200_TB_XC"])
    # the one-column-lag march and the march without its fast lane: 0 switches them on; the fused stages: non-zero
    assert re.search(r'env_int\("LBM_B200_TB_SKEW", 1\) != 0', src) and G.KNOBS["LBM_B200_TB_SKEW"] == ["0"]
    assert re.search(r'fast = env_int\("LBM_B200_TB_FAST", 1\)', src) and re.search(r"a\.fast_lane = fast;", src)
    assert G.KNOBS["LBM_B200_TB_FAST"] == ["0"]
    assert re.search(r'env_int\("LBM_B200_TB_FUSED", 0\) != 0', src) and G.KNOBS["LBM_B200_TB_FUSED"] == ["1"]
