"""What one engine handle (include/lbm_b200.h) computes over any sequence of calls, restated on the oracle.

The engine keeps per-handle state between calls (which buffer holds f_next, how many iterations the last pass
covered, caller-written f_next values, the parameters the last iteration ran with, ...).  This class keeps only what
the reference keeps -- one oracle.Oracle, i.e. the arrays of LBM::Grid, and the iteration counter of Solver::run --
and says for each entry point what that call does to them:

  initialise(u)       fresh Oracle(case); with u != case.inlet_velocity the arrays of Oracle(case with inlet u)
                      (Grid::initialise(u): ghost rows eq(1,u,0), fluid ux = u) while Zou-He keeps the params' value
  upload_f(state, k)  interior of f_current := state; the ghost ring and f_next keep their values; t = k
  upload_f_next(img)  solid cells and S/N ghost rows (corners included) of f_next := img; fluid cells and the W/E
                      ghost columns are ignored (the next collision / exchange rewrites them)
  set_params(case')   Oracle(case') holding the same arrays and t: later iterations use case', what the earlier ones
                      stored stays
  setup_geometry()    the handle needs initialise or upload_f before it steps again
  step(n), run(n)     Oracle.run(n)
  kernel variant, pass depth, force mode: nothing (the tree force sum equals the ordered one to 1e-14)

Between upload_f and the next iteration the engine defines what the observers derived from f_next show: the uploaded
state, as right after Grid::initialise (f_next reads as f_current, the forces are taken from it, rho / u are its
moments, solid cells 1 / 0 / 0).  `uploaded` marks that state; `observed()` returns it.  Likewise the values
upload_f_next writes show in the downloaded f_next from the next iteration on (`shown_f_next` until then).

CPU only: tests/test_lifecycle_model.py checks the model against straight oracle runs, tests/test_gpu_lifecycle.py
checks the engine against the model.
"""
from __future__ import annotations

from dataclasses import replace

import numpy as np

from oracle import oracle as O

FIELDS = ("f_current", "f_next", "rho", "ux", "uy")


def adopt(case: O.Case, src: O.Oracle) -> O.Oracle:
    """Oracle(case) holding src's arrays and iteration."""
    o = O.Oracle(case)
    for k in FIELDS:
        getattr(o, k)[...] = getattr(src, k)
    o.t = src.t
    return o


def moments(f):
    """rho, ux, uy of an interior block of populations [ny, nx, 9]."""
    cx = np.array([0, 1, 0, -1, 0, 1, -1, -1, 1], dtype=np.float64)
    cy = np.array([0, 0, 1, 0, -1, 1, 1, -1, -1], dtype=np.float64)
    rho = f.sum(axis=-1)
    return rho, (f * cx).sum(axis=-1) / rho, (f * cy).sum(axis=-1) / rho


class HandleModel:
    def __init__(self, case: O.Case):
        self.case = case
        self.o: O.Oracle | None = None
        self.initialised = False
        self.uploaded = False
        self.first_bad = -1
        self.shown_f_next = None

    @property
    def t(self) -> int:
        return self.o.t

    @property
    def solid(self):
        return self.o.solid

    # --- the entry points ------------------------------------------------------------------
    def initialise(self, u: float | None = None):
        o = O.Oracle(self.case)
        if u is not None and u != self.case.inlet_velocity:
            src = O.Oracle(replace(self.case, inlet_velocity=u))
            for k in FIELDS:
                getattr(o, k)[...] = getattr(src, k)
        self.o = o
        self.initialised = True
        self.uploaded = False
        self.first_bad = -1
        self.shown_f_next = None

    def upload_f(self, state, iteration: int):
        self.o.f_current[1:-1, 1:-1] = np.asarray(state)[1:-1, 1:-1]
        self.o.t = iteration
        self.initialised = True
        self.uploaded = True
        self.first_bad = -1

    def upload_f_next(self, img):
        img = np.asarray(img)
        ys, xs = np.nonzero(self.o.solid)
        fn = self.o.f_next
        if self.shown_f_next is None:
            self.shown_f_next = fn.copy()
        fn[ys + 1, xs + 1, :] = img[ys + 1, xs + 1, :]
        fn[0, :, :] = img[0, :, :]
        fn[-1, :, :] = img[-1, :, :]

    def set_params(self, case: O.Case):
        self.case = case
        if self.o is not None:
            self.o = adopt(case, self.o)

    def setup_geometry(self):
        self.initialised = False

    def run(self, n: int):
        assert self.initialised, "the engine refuses to step before initialise / upload_f"
        rows, bad = self.o.run(n)
        self.uploaded = False
        self.shown_f_next = None
        if bad >= 0 and self.first_bad < 0:
            self.first_bad = bad
        return rows, bad

    step = run

    # --- observers ---------------------------------------------------------------------------
    def observed(self):
        """{name: value} of every observer: the five arrays, forces, max_velocity, check_stability (ok, first bad)."""
        o = self.o
        out = {k: getattr(o, k).copy() for k in FIELDS}
        if self.shown_f_next is not None:
            out["f_next"] = self.shown_f_next.copy()
        if self.uploaded:
            out["f_next"] = out["f_current"].copy()
            rho, ux, uy = moments(out["f_current"][1:-1, 1:-1])
            solid = o.solid != 0
            rho[solid], ux[solid], uy[solid] = 1.0, 0.0, 0.0
            out["rho"], out["ux"], out["uy"] = rho, ux, uy
            tmp = adopt(self.case, o)
            tmp.f_next[...] = out["f_current"]
            out["forces"] = tmp.forces()
            out["max_velocity"] = float(np.sqrt((ux * ux + uy * uy).max()))
        else:
            out["forces"] = o.forces()
            out["max_velocity"] = o.max_velocity()
        ok = o.check_stability() and self.first_bad < 0
        out["stability"] = (ok, self.first_bad)
        return out
