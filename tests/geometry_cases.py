"""Lattices derived from the launch geometry of the temporally blocked kernel k_tb (csrc/lbm_tb.cu, lbm_tb.cuh): heights
that fill one, two or three strips up to a few rows, obstacles whose first or last row sits on either side of a block
edge, obstacles whose first or last column sits next to a chunk edge, and the extreme shapes past 65 535 columns or
rows.  Plain functions of (B, depth, xc); tests/test_geometry_cases.py checks on the CPU that the cases hit what they
claim, tests/test_gpu_geometry.py and tests/test_tb_emulation.py run them.

The formulas, restated from the sources:
- TbShape<T, B> (lbm_tb.cuh): ROFF = 0 at depth 1, 2 at depths 2 and 3; a strip stores H = B - 2 ROFF rows; the
  block of strip s holds the rows [lo, lo + B), lo = s H - ROFF (tb_thread: r.y = strip * H - ROFF + tid).
- The row gate (tb_thread, skewed march): a strip whose rows [lo, lo + B) miss the obstacle's rows
  [mask_ylo, mask_yhi) never looks at the mask.
- Chunks (tb_chunk, launch_one): a one-slab lattice is cut into chunks [j xc, (j + 1) xc) of xc columns,
  xc = LBM_B200_TB_XC when set, else 64 halved down to 16 until there are two waves of blocks.
- The obstacle (oracle/lbm_oracle.c:51-53, 104-107): cx = int(cylinder_x nx), cy = int(cylinder_y ny),
  r = int(cylinder_radius ny); cell (x, y) is solid iff (x - cx)^2 + (y - cy)^2 <= r^2, so the disc occupies the
  rows [cy - r, cy + r] and the columns [cx - r, cx + r], cut by the lattice's edges.
"""
from oracle import oracle as O

BLOCKS = (64, 128, 256)        # LBM_B200_TB_B: the block heights the library accepts (lbm_tb.cu block_threads)
DEFAULT_B = 128
XC_SWEEP = (1, 3, 7, 16, 64)   # LBM_B200_TB_XC values; tests add one >= nx (the whole row in one chunk)
EDGE_OFFSETS = range(-3, 4)    # obstacle columns this far from a chunk edge
NY_MAX = 524                   # keeps every lattice but the extreme shapes at ~600 x 520 or below
NX_MAX = 600
WIDE, TALL = (70001, 4), (4, 70000)  # past the 65 535 blocks of a grid's y / z dimension


def roff(depth):
    return 0 if depth == 1 else 2


def rows_per_strip(B, depth):
    return B - 2 * roff(depth)


def block_lo(B, depth, s):
    """First row of the block that works on strip s."""
    return s * rows_per_strip(B, depth) - roff(depth)


def disc(nx, ny, cx, cy, r, output_frequency=7, **kw):
    """The case whose obstacle is the disc of radius r around cell (cx, cy), exactly (int() of the +0.5 points)."""
    return O.Case(nx=nx, ny=ny, cylinder_x=(cx + 0.5) / nx, cylinder_y=(cy + 0.5) / ny, cylinder_radius=(r + 0.5) / ny,
                  output_frequency=output_frequency, **kw)


def disc_of(case):
    """(cx, cy, r) as the oracle derives them."""
    return int(case.cylinder_x * case.nx), int(case.cylinder_y * case.ny), int(case.cylinder_radius * case.ny)


def _depth_class(depth):
    return "t1" if depth == 1 else "t23"


def height_cases(B, depth):
    """ny = k H + r, k = 1, 2, 3, r = -1 .. 3 (odd heights included): full strips, one row short, a few rows over.
    The obstacle crosses the first strip edge."""
    H = rows_per_strip(B, depth)
    out = {}
    for k in (1, 2, 3):
        for r in range(-1, 4):
            ny = k * H + r
            if ny > NY_MAX:
                continue
            name = "h%d_%s_k%d_r%s" % (B, _depth_class(depth), k, ("m1" if r < 0 else str(r)))
            out[name] = disc(48, ny, 15, min(H, ny - 6), 5, output_frequency=7, inlet_velocity=0.04)
    return out


def row_edge_cases(B, depth):
    """The obstacle's rows against the block of strip 1, [lo, lo + B): its last row just below lo (yhi = lo - 1, lo,
    lo + 1) or its first row just above the block's last row (ylo = lo + B - 1, lo + B, lo + B + 1); one obstacle
    across two strips and one cut by each wall."""
    H, lo, r = rows_per_strip(B, depth), block_lo(B, depth, 1), 3
    tag = "%d_%s" % (B, _depth_class(depth))
    out = {}
    for d in (-1, 0, 1):
        ds = "m1" if d < 0 else ("p1" if d > 0 else "0")
        yhi = lo + d                       # the disc's last row is yhi - 1
        out["yhi_%s_lo%s" % (tag, ds)] = disc(40, lo + B + 6, 12, yhi - 1 - r, r, output_frequency=5)
        ylo = lo + B + d                   # ... its first row
        out["ylo_%s_hi%s" % (tag, ds)] = disc(40, ylo + 2 * r + 4, 27, ylo + r, r, output_frequency=5)
    out["span_%s" % tag] = disc(40, 2 * H + 9, 20, H, 6, output_frequency=9)
    out["wall_%s" % tag] = disc(40, H + 5, 18, 1, 5, output_frequency=9)     # cut by the bottom wall
    out["wallN_%s" % tag] = disc(40, H + 5, 18, H + 3, 5, output_frequency=9)  # ... and by the top one
    return out


def column_edge_cases(xc):
    """The obstacle's first and last column at offset d = -3 .. 3 from a chunk edge: a disc of diameter 2r + 1 whose
    width 2r is a multiple of xc puts both at offset d from (different) chunk edges."""
    r = xc // 2 if xc % 2 == 0 else xc
    k = -(-4 // xc) if xc >= 4 else -(-6 // xc)  # the first chunk edge at least 4 columns from the inlet
    out = {}
    for d in EDGE_OFFSETS:
        first = k * xc + d
        nx = first + 2 * r + 9
        ny = 2 * r + 11
        name = "cols_xc%d_d%s" % (xc, ("m%d" % -d) if d < 0 else str(d))
        out[name] = disc(nx, ny, first + r, r + 5, r, output_frequency=5, inlet_velocity=0.03)
    return out


def inlet_outlet_cases():
    """Obstacles touching or next to the inlet and the outlet column (and one cut by each)."""
    out = {}
    for i, first in enumerate((-2, 0, 1, 2)):
        out["inlet_%d" % i] = disc(44, 40, first + 4, 20, 4, output_frequency=5, inlet_velocity=0.04)
    for i, last in enumerate((45, 43, 42, 41)):  # nx = 44: the last column is 43
        out["outlet_%d" % i] = disc(44, 40, last - 4, 19, 4, output_frequency=5, inlet_velocity=0.04)
    return out


def extreme_cases():
    """70 001 x 4 and 4 x 70 000, one solid cell each, past index 65 535."""
    return {
        "wide_70001x4": disc(WIDE[0], WIDE[1], 65540, 1, 0, output_frequency=3, inlet_velocity=0.04),
        "tall_4x70000": disc(TALL[0], TALL[1], 2, 65600, 0, output_frequency=3, inlet_velocity=0.04),
    }


def strip_cases(B):
    """Every height and row-edge case of block height B, depth 1 and depths 2 / 3 (one run mixes both)."""
    out = {}
    for depth in (1, 2):  # depths 2 and 3 share the strip geometry
        out.update(height_cases(B, depth))
        out.update(row_edge_cases(B, depth))
    return out


def chunk_cases():
    out = {}
    for xc in XC_SWEEP:
        if xc > 1:  # every column edge is a chunk edge at xc = 1: any obstacle hits every offset
            out.update(column_edge_cases(xc))
    out.update(inlet_outlet_cases())
    return out


def all_cases(B):
    out = strip_cases(B)
    out.update(chunk_cases())
    out.update(extreme_cases())
    return out


def solid_extent(solid):
    """(ylo, yhi, xfirst, xlast) of a solid mask [ny, nx]: rows [ylo, yhi), columns [xfirst, xlast]."""
    import numpy as np

    ys, xs = np.nonzero(solid)
    return int(ys.min()), int(ys.max()) + 1, int(xs.min()), int(xs.max())


# The LBM_B200_TB_* settings the GPU tests set and the values they use.  lbm_tb.cu reads them with env_int.
KNOBS = {
    "LBM_B200_TB_XC": [str(x) for x in XC_SWEEP],
    "LBM_B200_TB_B": ["64", "256"],
    "LBM_B200_TB_SKEW": ["0"],
    "LBM_B200_TB_FAST": ["0"],
    "LBM_B200_TB_FUSED": ["1"],
}
