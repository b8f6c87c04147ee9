"""Call sequences against the oracle: restarts, edits of f_current / f_next in the middle of a run, parameter changes,
geometry changes, kernel / pass-depth / force-mode switches, re-initialised and reused handles, on every kernel.

The engine updates its per-handle bookkeeping (which buffer holds f_next, how many iterations the last pass covered,
caller-written f_next values, the parameters the last iteration ran with, the geometry tables) by hand in every entry
point.  tests/lifecycle_model.py says what each call does to the reference's arrays; every test here drives an engine
handle and the model with the same calls and compares every observer after each call, on bit patterns (-0.0 is not
0.0).  The exceptions are stated where they occur: rho / u of the in-place AA buffers and right after an upload (to
1e-12 relative / 1e-13 absolute, as tests/test_gpu_aa.py) and the tree force sum (1e-14).  A mismatch names the
sequence, the call and the first differing (y, x, i); the random sequences print their seed and the calls so far.
"""
import os
import subprocess
from dataclasses import replace

import numpy as np
import pytest

from oracle import oracle as O
import geometry_cases as G
import parity_util as util
from lifecycle_model import HandleModel
from test_gpu_parity import CASES as PARITY_CASES

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
AA = 16
NO_CYLINDER = 4

CASES = {n: PARITY_CASES[n] for n in ("64x32", "70x33_odd_ny", "cyl_on_wall", "cyl_at_inlet", "tiny_6x4")}
CASES["span_128_t23"] = G.row_edge_cases(G.DEFAULT_B, 2)["span_128_t23"]  # 40 x 257: three strips, the disc across two

# name: (flags, kernel variant, pass depth)
CONFIGS = {
    "v0": (0, 0, 3), "v1": (0, 1, 3),
    "v2d1": (0, 2, 1), "v2d2": (0, 2, 2), "v2d3": (0, 2, 3),
    "aa_v0": (AA, 0, 3), "aa_v1": (AA, 1, 3),
}
AB_CONFIGS = [c for c in CONFIGS if not CONFIGS[c][0] & AA]
OBSERVERS = ("f_current", "f_next", "macros", "forces", "max_velocity", "stability", "solid", "iteration")


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def first_diff(got, want):
    return tuple(int(v) for v in np.argwhere(bits(got) != bits(want))[0])


class Pair:
    """One engine handle and its model, driven by the same calls."""

    def __init__(self, label, case, config, initialise=True):
        import lbm_b200

        self.label, self.config = label, config
        self.flags, variant, depth = CONFIGS[config]
        self.aa = bool(self.flags & AA)
        self.case = case
        self.s = lbm_b200.Solver(util.case_to_params(case, flags=self.flags))
        self.s.set_kernel_variant(variant)
        self.s.set_pass_depth(depth)
        self.m = HandleModel(case)
        self.tree = False
        self.unstable = False
        self.log = []
        if initialise:
            self.initialise()

    def close(self):
        self.s.close()

    def _note(self, what):
        self.log.append(what)

    def where(self):
        return "%s [%s], call %d (%s); calls so far: %s" % (self.label, self.config, len(self.log) - 1,
                                                           self.log[-1] if self.log else "-", "; ".join(self.log))

    # --- calls -----------------------------------------------------------------------------------
    def initialise(self, u=None):
        self._note("initialise(%s)" % u)
        self.s.initialise(u)
        self.m.initialise(u)
        self.unstable = False

    def upload_f(self, state, k):
        self._note("upload_f(k=%d)" % k)
        self.s.upload_f(state, k)
        self.m.upload_f(state, k)

    def upload_f_next(self, img):
        self._note("upload_f_next")
        self.s.upload_f_next(img)
        self.m.upload_f_next(img)

    def set_params(self, case, flags=None):
        self._note("set_params(tau=%r, u_in=%r, of=%d, cyl=(%r, %r, %r), flags=%s)" % (
            case.tau, case.inlet_velocity, case.output_frequency, case.cylinder_x, case.cylinder_y,
            case.cylinder_radius, flags))
        self.s.set_params(util.case_to_params(case, flags=self.flags if flags is None else flags))
        self.case = case
        self.m.set_params(case)

    def setup_geometry(self):
        self._note("setup_geometry")
        n = self.s.setup_geometry()
        self.m.setup_geometry()
        return n

    def step(self, n):
        self._note("step(%d)" % n)
        self.s.step(n)
        self.m.step(n)

    def run(self, n):
        self._note("run(%d)" % n)
        rows, bad = self.s.run(n)
        want, wbad = self.m.run(n)
        assert bad == wbad, "%s: unstable_at %d, the reference %d" % (self.where(), bad, wbad)
        self.compare_rows(rows, want)
        self.unstable = bad >= 0
        return rows, bad

    def variant(self, v):
        self._note("set_kernel_variant(%d)" % v)
        self.s.set_kernel_variant(v)

    def depth(self, d):
        self._note("set_pass_depth(%d)" % d)
        self.s.set_pass_depth(d)

    def force_mode(self, tree):
        self._note("set_force_mode(%d)" % tree)
        self.s.set_force_mode(tree)
        self.tree = bool(tree)

    # --- comparisons -------------------------------------------------------------------------------
    def compare_rows(self, rows, want):
        assert rows.shape == want.shape, "%s: %d forces rows, the reference %d" % (self.where(), len(rows), len(want))
        if not self.tree:
            assert np.array_equal(bits(rows), bits(want)), "%s: forces rows differ: %s vs %s" % (self.where(), rows, want)
            return
        assert np.array_equal(rows[:, 0], want[:, 0]), self.where()
        assert np.abs(rows[:, 1:3] - want[:, 1:3]).max(initial=0.0) <= 1e-14 * max(np.abs(want[:, 1:3]).max(initial=0.0), 1.0), \
            "%s: tree-summed forces rows beyond 1e-14" % self.where()
        q = 0.5 * 1.0 * self.case.inlet_velocity * self.case.inlet_velocity * (2.0 * int(self.case.cylinder_radius * self.case.ny))
        coef = rows[:, 1:3] / q if q > 1e-12 else np.zeros_like(rows[:, 1:3])
        assert np.array_equal(rows[:, 3:5], coef), self.where()

    def _field(self, name, got, want, tolerant=False):
        if tolerant:
            if name == "rho":
                util.assert_close_f(got, want, "%s: %s" % (self.where(), name))
            else:
                util.assert_close_u(got, want, "%s: %s" % (self.where(), name))
            return
        if not np.array_equal(bits(got), bits(want)):
            at = first_diff(got, want)
            raise AssertionError("%s: %s differs first at (y, x%s) = %s: got %r, the reference %r" % (
                self.where(), name, ", i" if len(at) == 3 else "", at, got[at], want[at]))

    def check(self, order=OBSERVERS):
        """Every observer, in the given order (the engine caches some of them)."""
        if self.unstable:  # the engine finishes its chunk past the failing iteration: only the verdict is defined
            ok, bad = self.s.check_stability()
            assert (ok, bad) == self.m.observed()["stability"], self.where()
            return
        want = self.m.observed()
        loose = self.aa or self.m.uploaded
        for k in order:
            if k in ("f_current", "f_next"):
                self._field(k, self.s.f(0 if k == "f_current" else 1), want[k])
            elif k == "macros":
                rho, ux, uy = self.s.macros()
                for name, got in (("rho", rho), ("ux", ux), ("uy", uy)):
                    self._field(name, got, want[name], tolerant=loose)
            elif k == "forces":
                got = self.s.forces()
                if self.tree:
                    assert np.abs(np.subtract(got, want["forces"])).max() <= 1e-14 * max(np.abs(want["forces"]).max(), 1.0), self.where()
                else:
                    assert bits(np.array(got)).tolist() == bits(np.array(want["forces"])).tolist(), \
                        "%s: forces %r, the reference %r" % (self.where(), got, want["forces"])
            elif k == "max_velocity":
                assert abs(self.s.max_velocity() - want["max_velocity"]) <= 1e-13, self.where()
            elif k == "stability":
                assert self.s.check_stability() == want["stability"], self.where()
            elif k == "solid":
                assert np.array_equal(self.s.solid() != 0, self.m.solid != 0), "%s: solid mask" % self.where()
            elif k == "iteration":
                assert self.s.info().iteration == self.m.t, "%s: iteration %d, the reference %d" % (
                    self.where(), self.s.info().iteration, self.m.t)


def edited(f, rng, scale=1e-3):
    """f times (1 + scale N(0,1)) in every entry."""
    return np.ascontiguousarray(f * (1.0 + scale * rng.standard_normal(f.shape)))


def moved(case):
    """The same lattice with another obstacle: across the inlet, in another strip of a tall lattice."""
    return replace(case, cylinder_x=0.04, cylinder_y=0.3 if case.ny < 200 else 0.8, cylinder_radius=0.2 if case.ny < 200 else 0.08)


# ---- a. named sequences -------------------------------------------------------------------------------

@pytest.mark.parametrize("name", list(CASES))
@pytest.mark.parametrize("config", list(CONFIGS))
def test_restart_at_iterations_around_output_steps_and_pass_edges(config, name):
    """lbm_upload_f(f_current, k) -- Grid::load_checkpoint -- at k = of m - 1, of m, of m + 1 and k = 0, 1, 2 mod 3, on
    the running handle and on a new one: the run goes on as the straight run does."""
    case = CASES[name]
    of = case.output_frequency
    ks = sorted({of * 2 - 1, of * 2, of * 2 + 1, 9, 10, 11})
    for k in ks:
        p = Pair("restart %s k=%d" % (name, k), case, config)
        p.run(k)
        p.check()
        saved = p.s.f_current()
        p.step(3)
        p.upload_f(saved, k)  # back to iteration k on the same handle
        p.check()
        p.step(1)
        p.check()
        p.run(of + 2)
        p.check()
        fresh = Pair("restart %s k=%d, new handle" % (name, k), case, config)
        fresh.upload_f(saved, k)
        fresh.run(2 * of + 1)
        fresh.check()
        p.close()
        fresh.close()


def poke(f, case):
    f = f.copy()
    f[4, 3, 1] *= 1.25
    f[case.ny, case.nx, 8] *= 0.5
    f[case.ny // 2 + 1, 1, 6] += 0.001
    return f


def f_next_edit(f, solid):
    f = f.copy()
    ys, xs = np.nonzero(solid)
    f[ys + 1, xs + 1, :] *= 1.0 + 0.01 * np.arange(9)
    f[0, :, :] *= 0.97
    f[-1, 2:, 3] += 0.002
    f[1:-1, 1:-1][~solid.astype(bool)] = 123.0  # fluid cells: dead values
    return f


@pytest.mark.parametrize("name", list(CASES))
@pytest.mark.parametrize("config", list(CONFIGS))
@pytest.mark.parametrize("what", ["f_current", "f_next", "both"])
def test_edit_in_the_middle_of_a_run(config, name, what):
    """Grid::f_current / Grid::f_next written at iteration k > 0 (Grid::flush_edits: upload_f, then upload_f_next)."""
    if what != "f_current" and CONFIGS[config][0] & AA:
        pytest.skip("the in-place buffer keeps no f_next to write into")
    case = CASES[name]
    p = Pair("edit %s mid-run" % what, case, config)
    p.run(case.output_frequency + 2)
    if what in ("f_current", "both"):
        p.upload_f(poke(p.s.f_current(), case), p.m.t)
    if what in ("f_next", "both"):
        p.upload_f_next(f_next_edit(p.s.f_next() if what == "f_next" else p.m.o.f_next, p.m.solid))
    p.check()
    for n in (1, 1, 2, 7):
        p.step(n)
        p.check()
    p.run(2 * case.output_frequency + 1)
    p.check()
    p.close()


@pytest.mark.parametrize("name", list(CASES))
@pytest.mark.parametrize("config", AB_CONFIGS)
def test_written_f_next_survives_a_later_f_current_upload(config, name):
    """Lead: f_next's solid cells and ghost rows written, two or more iterations, then f_current written.  The reference
    keeps the written f_next values (its collision skips solid cells, nothing rewrites the ghost rows)."""
    case = CASES[name]
    p = Pair("f_next then f_current", case, config)
    p.step(5)
    p.upload_f_next(f_next_edit(p.s.f_next(), p.m.solid))
    p.step(2)
    p.check()
    p.step(1)
    p.upload_f(poke(p.s.f_current(), case), p.m.t)
    for n in (1, 1, 3):
        p.step(n)
        p.check()
    p.upload_f(p.s.f_current(), p.m.t + 4)  # a restart at another iteration keeps them too
    p.run(2 * case.output_frequency)
    p.check()
    p.close()


@pytest.mark.parametrize("first", OBSERVERS)
@pytest.mark.parametrize("name", ["64x32", "70x33_odd_ny", "cyl_at_inlet", "span_128_t23"])
@pytest.mark.parametrize("config", list(CONFIGS))
def test_set_params_between_step_and_observer(config, name, first):
    """Lead: lbm_set_params (tau, u_in, output_frequency) after a step and before an observer.  The observers show the
    state the last iteration left, computed with the parameters it ran with; the next iterations use the new ones."""
    case = CASES[name]
    p = Pair("set_params before %s" % first, case, config)
    p.step(case.output_frequency + 4)  # a pass of several iterations that did not emit its moments
    p.set_params(replace(case, tau=case.tau + 0.15, inlet_velocity=case.inlet_velocity * 2.5,
                         output_frequency=case.output_frequency + 1))
    p.check((first,) + tuple(o for o in OBSERVERS if o != first))
    p.step(1)
    p.check()
    p.step(4)
    p.check()
    p.set_params(replace(p.case, output_frequency=2))
    p.run(9)
    p.check()
    p.close()


@pytest.mark.parametrize("name", list(CASES))
@pytest.mark.parametrize("config", list(CONFIGS))
def test_setup_geometry_on_a_running_handle_needs_a_new_state(config, name):
    """Lead: lbm_setup_geometry with a moved obstacle on a running handle leaves it uninitialised (the buffers hold the
    old geometry's state); lbm_initialise then gives the new case's fresh state."""
    import lbm_b200

    case = CASES[name]
    p = Pair("setup_geometry mid-run", case, config)
    p.run(6)
    p.set_params(moved(case))
    assert p.setup_geometry() == int(O.Oracle(moved(case)).n_solid)
    with pytest.raises(lbm_b200.LbmError):
        p.s.step(1)
    with pytest.raises(lbm_b200.LbmError):
        p.s.run(1)
    p.initialise()
    p.check()
    p.run(2 * case.output_frequency + 3)
    p.check()
    p.close()


@pytest.mark.parametrize("name", list(CASES))
def test_variant_depth_and_force_mode_switches_in_one_run(name):
    """Variant 2 -> 1 -> 0 -> 2, pass depth 3 -> 2 -> 1 -> 3 and ordered <-> tree forces between steps of one run."""
    case = CASES[name]
    p = Pair("switches", case, "v2d3")
    plan = [("variant", 1), ("variant", 0), ("variant", 2), ("depth", 2), ("depth", 1), ("depth", 3),
            ("force_mode", 1), ("variant", 1), ("force_mode", 0), ("depth", 2), ("variant", 2)]
    p.step(4)
    for what, v in plan:
        getattr(p, what)(v)
        p.step(case.output_frequency + 1)
        p.check()
        p.run(case.output_frequency)
        p.check()
    p.close()


@pytest.mark.parametrize("config", list(CONFIGS))
def test_reinitialise_after_an_unstable_run(config):
    """tau = 0.52: the run stops at the reference's timestep; lbm_initialise starts over (iteration 0, no verdict,
    the same rows and the same failing timestep again)."""
    case = O.Case(nx=512, ny=128, tau=0.52, inlet_velocity=0.1, output_frequency=50)
    p = Pair("unstable, re-initialised", case, config)
    first, bad = p.run(400)
    assert bad >= 0
    p.check()
    assert p.s.check_stability() == (False, bad)
    p.initialise()
    p.check()
    again, bad2 = p.run(400)
    assert bad2 == bad and np.array_equal(bits(again), bits(first))
    p.initialise()
    p.step(3)
    p.check()
    p.close()


@pytest.mark.parametrize("name", list(CASES))
@pytest.mark.parametrize("config", AB_CONFIGS)
def test_reinitialise_after_upload_f_next(config, name):
    case = CASES[name]
    p = Pair("re-initialised after upload_f_next", case, config)
    p.step(3)
    p.upload_f_next(f_next_edit(p.s.f_next(), p.m.solid))
    p.step(2)
    p.initialise()
    p.check()
    p.run(2 * case.output_frequency + 2)
    p.check()
    p.close()


@pytest.mark.parametrize("name", list(CASES))
@pytest.mark.parametrize("config", list(CONFIGS))
def test_handle_reuse_for_another_case(config, name):
    """Grid::setup_geometry(params) + initialise on a used handle (set_params, setup_geometry, initialise) equals a
    fresh handle and a fresh oracle: another tau, u_in and output frequency, the obstacle moved, then removed
    (LBM_FLAG_NO_CYLINDER), then back elsewhere.  Pins that build_geometry rebuilds every table the kernels read."""
    case = CASES[name]
    p = Pair("reuse", case, config)
    p.run(case.output_frequency + 3)
    b = replace(moved(case), tau=case.tau + 0.1, inlet_velocity=0.035, output_frequency=case.output_frequency + 2)
    nocyl = replace(b, cylinder_x=100.0)  # the oracle's obstacle-free channel: the disc far outside
    c = replace(case, cylinder_x=0.6, cylinder_y=0.75, cylinder_radius=0.15, output_frequency=3, tau=0.65)
    for label, nxt, flags in (("moved", b, None), ("no cylinder", nocyl, NO_CYLINDER), ("back", c, None)):
        p.set_params(nxt, flags=None if flags is None else p.flags | flags)
        p.setup_geometry()
        p.initialise()
        p.check()
        fresh = Pair("fresh handle: " + label, nxt, config, initialise=False)
        if flags:
            fresh.s.set_params(util.case_to_params(nxt, flags=fresh.flags | flags))
        fresh.initialise()
        for n in (1, 2, 2 * nxt.output_frequency + 1):
            p.step(n) if n < 3 else p.run(n)
            fresh.step(n) if n < 3 else fresh.run(n)
            p.check()
            fresh.check()
        assert np.array_equal(bits(p.s.f_next()), bits(fresh.s.f_next()))
        fresh.close()
    p.close()


# ---- b. seeded random sequences -------------------------------------------------------------------------

SEEDS = 30
CALLS = 15


def random_call(p, rng):
    ops = ["step", "run", "upload_f", "upload_f_next", "switch", "observe", "initialise", "set_params"]
    weights = [4, 3, 2, 2, 2, 2, 1, 1]
    if p.aa:
        ops, weights = zip(*[(o, w) for o, w in zip(ops, weights) if o not in ("upload_f_next", "switch")])
    op = rng.choice(list(ops), p=np.array(weights, dtype=float) / sum(weights))
    if op == "step":
        p.step(int(rng.integers(1, 8)))
    elif op == "run":
        p.run(int(rng.integers(1, 13)))
    elif op == "upload_f":
        state = p.m.o.f_current.copy()
        state[1:-1, 1:-1] = edited(state[1:-1, 1:-1], rng)
        k = p.m.t if rng.random() < 0.5 else int(rng.integers(0, 40))
        p.upload_f(state, k)
    elif op == "upload_f_next":
        p.upload_f_next(edited(p.m.observed()["f_next"], rng))
    elif op == "switch":
        what = rng.choice(["variant", "depth", "force_mode"])
        getattr(p, str(what))(int(rng.integers(0, 3)) if what == "variant" else
                              int(rng.integers(1, 4)) if what == "depth" else int(rng.integers(0, 2)))
    elif op == "observe":
        p._note("observe")
    elif op == "initialise":
        p.initialise(None if rng.random() < 0.5 else float(rng.choice([0.02, 0.035])))
    elif op == "set_params":
        p.set_params(replace(p.case, tau=float(rng.choice([0.55, 0.6, 0.7, 0.9])),
                             inlet_velocity=float(rng.choice([0.01, 0.02, 0.04])),
                             output_frequency=int(rng.integers(1, 10))))


@pytest.mark.parametrize("seed", range(SEEDS))
@pytest.mark.parametrize("config", list(CONFIGS))
def test_random_call_sequence(config, seed):
    names = list(CASES)
    name = names[seed % len(names)]
    rng = np.random.default_rng(1000 * seed + list(CONFIGS).index(config))
    p = Pair("random seed %d on %s" % (seed, name), CASES[name], config)
    for _ in range(CALLS):
        if p.unstable:  # (the engine ran past the failing iteration; only a new state continues the comparison)
            p.initialise()
        random_call(p, rng)
        p.check(tuple(rng.permutation(OBSERVERS)))
    p.close()


# ---- c. the C++ surface ---------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def lifecycle_exe(tmp_path_factory):
    pkg = os.path.join(ROOT, "highperformancecomputing-latticeboltzmannmethod_b200")
    exe = str(tmp_path_factory.mktemp("cpp") / "grid_lifecycle_dump")
    subprocess.run(["g++", "-std=c++17", "-O1", "-mfma", "-ffp-contract=off", "-pthread", "-I" + os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "tests", "cpp", "grid_lifecycle_dump.cpp"), "-o", exe, "-L" + pkg, "-llbm_b200",
                    "-Wl,-rpath," + pkg], check=True)
    return exe


CPP_CASE = O.Case(nx=48, ny=20, output_frequency=5, cylinder_radius=0.15)


def run_cpp(exe, tmp_path, *args):
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    r = subprocess.run([exe] + [str(a) for a in args] + [str(tmp_path)], cwd=tmp_path, capture_output=True, text=True, env=env,
                       timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr


def compare_dump(tmp_path, o, aa):
    ny, nx = CPP_CASE.ny, CPP_CASE.nx
    for k, shape in (("f_current", (ny + 2, nx + 2, 9)), ("f_next", (ny + 2, nx + 2, 9)), ("rho", (ny, nx)), ("ux", (ny, nx)),
                     ("uy", (ny, nx))):
        got = np.fromfile(tmp_path / (k + ".bin")).reshape(shape)
        if k in ("rho", "ux", "uy") and aa:
            (util.assert_close_f if k == "rho" else util.assert_close_u)(got, getattr(o, k), k)
        elif not np.array_equal(bits(got), bits(getattr(o, k))):
            raise AssertionError("%s differs first at %s" % (k, first_diff(got, getattr(o, k))))


@pytest.mark.parametrize("flags,variant,depth", [(0, 2, 3), (0, 0, 1), (AA, 0, 1)])
def test_grid_edits_at_a_later_iteration(lifecycle_exe, tmp_path, flags, variant, depth):
    """Grid::f_current and Grid::f_next written at iteration 7, between two Grid::advance calls."""
    run_cpp(lifecycle_exe, tmp_path, "edit", flags, variant, depth)
    o = O.Oracle(CPP_CASE)
    o.run(7)
    nx, ny = CPP_CASE.nx, CPP_CASE.ny
    o.f_current[4, 3, 1] *= 1.25
    o.f_current[ny, nx, 8] *= 0.5
    if not flags & AA:
        cx, cy = int(CPP_CASE.cylinder_x * nx), int(CPP_CASE.cylinder_y * ny)
        assert o.solid[cy, cx]
        o.f_next[cy + 1, cx + 1, 5] *= 1.5
        o.f_next[0, 10, 2] += 0.001
        o.f_next[ny + 1, nx + 1, 7] *= 0.75
    o.run(9)
    compare_dump(tmp_path, o, bool(flags & AA))


@pytest.mark.parametrize("flags,variant,depth", [(AA, 0, 1), (AA, 1, 1), (0, 2, 3), (0, 1, 1)])
def test_checkpoint_restart_at_a_non_output_iteration(lifecycle_exe, tmp_path, flags, variant, depth):
    """Solver::run to 13, save_checkpoint; a second Solver load_checkpoint()s and runs to 31: forces.csv from 15 on and
    the final fields are the straight run's."""
    run_cpp(lifecycle_exe, tmp_path, "restart", flags, variant, depth)
    o = O.Oracle(CPP_CASE)
    o.run(13)
    rows, bad = o.run(31 - 13)
    assert bad == -1
    compare_dump(tmp_path, o, bool(flags & AA))
    assert open(tmp_path / "forces.csv").read() == O.format_forces_csv(rows)
