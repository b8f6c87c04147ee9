"""CPU checks of tests/lifecycle_model.py: where a call sequence means the same as a straight run, the model says so
bit for bit."""
from dataclasses import replace

import numpy as np
import pytest

from oracle import oracle as O
from lifecycle_model import FIELDS, HandleModel

CASE = O.Case(nx=64, ny=32, cylinder_x=0.3, cylinder_radius=0.2, output_frequency=3)


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def same_state(model, o):
    assert model.t == o.t
    for k in FIELDS:
        assert np.array_equal(bits(getattr(model.o, k)), bits(getattr(o, k))), k


def test_fresh_model_is_a_fresh_oracle():
    m = HandleModel(CASE)
    m.initialise()
    same_state(m, O.Oracle(CASE))
    m2 = HandleModel(CASE)
    m2.initialise(CASE.inlet_velocity)
    same_state(m2, O.Oracle(CASE))


def test_initialise_with_another_velocity_keeps_the_params_inlet():
    m = HandleModel(CASE)
    m.initialise(0.03)
    other = O.Oracle(replace(CASE, inlet_velocity=0.03))
    same_state(m, other)
    m.run(5)
    other.run(5)
    # same start, different Zou-He inlet: the states part
    assert not np.array_equal(m.o.f_current, other.f_current)


@pytest.mark.parametrize("k", [1, 2, 3, 7])
def test_uploading_the_own_f_current_continues_the_straight_run(k):
    straight = O.Oracle(CASE)
    straight.run(k + 6)
    m = HandleModel(CASE)
    m.initialise()
    m.run(k)
    m.upload_f(m.o.f_current.copy(), k)
    assert m.uploaded and m.t == k
    rows, bad = m.run(6)
    assert bad == -1 and not m.uploaded
    same_state(m, straight)


def test_set_params_to_the_same_params_changes_nothing():
    straight = O.Oracle(CASE)
    want, _ = straight.run(11)
    m = HandleModel(CASE)
    m.initialise()
    rows_a, _ = m.run(4)
    m.set_params(replace(CASE))
    rows_b, _ = m.run(7)
    same_state(m, straight)
    assert np.array_equal(np.concatenate([rows_a, rows_b]), want)


def test_set_params_keeps_what_earlier_iterations_stored():
    m = HandleModel(CASE)
    m.initialise()
    m.run(4)
    before = {k: getattr(m.o, k).copy() for k in FIELDS}
    m.set_params(replace(CASE, tau=0.7, inlet_velocity=0.02, output_frequency=2))
    for k in FIELDS:
        assert np.array_equal(getattr(m.o, k), before[k]), k
    rows, _ = m.run(3)
    assert [int(r[0]) for r in rows] == [4, 6]


def test_upload_f_next_takes_solid_cells_and_ghost_rows_only():
    m = HandleModel(CASE)
    m.initialise()
    m.run(3)
    before = m.o.f_next.copy()
    img = before * 1.5
    m.upload_f_next(img)
    fn = m.o.f_next
    solid = np.zeros(fn.shape[:2], dtype=bool)
    solid[1:-1, 1:-1] = m.solid != 0
    solid[0, :] = solid[-1, :] = True
    assert np.array_equal(fn[solid], img[solid])
    assert np.array_equal(fn[~solid], before[~solid])


def test_observers_right_after_an_upload_describe_the_uploaded_state():
    m = HandleModel(CASE)
    m.initialise()
    m.run(5)
    state = m.o.f_current.copy()
    m.upload_f(state, 5)
    obs = m.observed()
    assert np.array_equal(obs["f_next"], state)
    assert obs["rho"][m.solid != 0].tolist() == [1.0] * int(m.solid.sum())
    assert np.allclose(obs["rho"][m.solid == 0], state[1:-1, 1:-1].sum(axis=-1)[m.solid == 0], rtol=1e-15, atol=0)
    assert obs["stability"] == (True, -1)


def test_setup_geometry_requires_a_new_state():
    m = HandleModel(CASE)
    m.initialise()
    m.setup_geometry()
    with pytest.raises(AssertionError):
        m.run(1)
    m.initialise()
    m.run(1)
