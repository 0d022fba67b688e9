"""Pins the oracle's contact-spline restatement (oracle/foot_spline.cpp).

Every check of the reference's own test/splines_tests.cpp is restated here (known answers :66-105, coefficient
reconstruction :109-158, add/remove polys :160-237, finite-difference partials :239-444) and run against
  * 'oracle' -- the restatement, always;
  * 'ref'    -- the reference's own end_effector_splines.cpp compiled from BGG_REFERENCE_DIR (oracle/_ref), when built.
A third group compares restatement and compiled reference on seeded random splines, bit for bit; without the compiled
reference, against the reference's values stored in tests/golden/reference_outputs.json (common.Recorded).
"""
import math

import hashlib

import numpy as np
import pytest

import common
import pyoracle as po
from pyoracle import FORCE, POSITION

MARGIN = 1e-3
FORCE_MULT = 100.0
WHICH = ["oracle"] + (["ref"] if po.have_ref() else [])


def make_pair(which):
    times = [0.2 * i for i in range(5)]
    return [po.FootSpline(times, False, 3, which), po.FootSpline(times, True, 3, which)], times


@pytest.mark.parametrize("which", WHICH)
def test_setting_vars(which):   # splines_tests.cpp:34-56
    splines, _ = make_pair(which)
    for s in splines:
        for coord in range(3):
            t = s.times()
            for it in s.mutable_nodes(POSITION, coord):
                s.set_vars(POSITION, coord, it, it, 2.0)
                assert s.value(POSITION, coord, t[it]) == it
            for it in s.mutable_nodes(FORCE, coord):
                s.set_vars(FORCE, coord, it, it, 2.0 / FORCE_MULT)
                assert s.value(FORCE, coord, t[it]) == it


@pytest.mark.parametrize("which", WHICH)
def test_known_answers(which):   # splines_tests.cpp:58-106
    splines, _ = make_pair(which)
    s0, s1 = splines
    for coord in range(3):
        for it in s0.mutable_nodes(POSITION, coord):
            s0.set_vars(POSITION, coord, it, it, it - 1)
        assert s0.value(POSITION, coord, 0) == 0
        if coord != 2:
            assert abs(s0.value(POSITION, coord, 0.103448) - 1.0517) < MARGIN
            assert abs(s0.value(POSITION, coord, 0.503448) - 4.62926) < MARGIN
        else:
            assert abs(s0.value(POSITION, coord, 0.162069) - 1.67752) < MARGIN
            assert abs(s0.value(POSITION, coord, 0.5) - 6) < MARGIN
        for it in s1.mutable_nodes(POSITION, coord):
            s1.set_vars(POSITION, coord, it, it, it - 1)
        assert s1.value(POSITION, coord, 0) == 0
        if coord != 2:
            assert abs(s1.value(POSITION, coord, 0.103448) - 0.0) < MARGIN
            assert abs(s1.value(POSITION, coord, 0.25517) - 0.93156) < MARGIN
        else:
            assert abs(s1.value(POSITION, coord, 0.162069) - 0) < MARGIN
            assert abs(s1.value(POSITION, coord, 0.25517) - 2.2683) < MARGIN
        for it in s0.mutable_nodes(FORCE, coord):
            s0.set_vars(FORCE, coord, it, it, (it - 1) / FORCE_MULT)
        assert s0.value(FORCE, coord, 0) == 0
        assert abs(s0.value(FORCE, coord, 0.103448)) < MARGIN
        assert abs(s0.value(FORCE, coord, 0.26666 + 0.0229885) - 3.27887) < MARGIN


def _check_force_reconstruction(s, coord, t0, t1, n=100):
    vec = s.as_qp_vec(FORCE, coord)
    for i in range(n):
        time = i * ((t1 - t0) / n) + t0
        if s.is_force_mutable(time):
            idx, cnt = s.vars_idx(FORCE, coord, time)
            w = s.lin(FORCE, coord, time)
            assert len(w) == cnt
            assert abs(s.value(FORCE, coord, time) - float(vec[idx:idx + cnt] @ w)) < MARGIN
        else:
            assert s.value(FORCE, coord, time) == 0


@pytest.mark.parametrize("which", WHICH)
def test_linearisation_reconstructs_value(which):   # splines_tests.cpp:108-158
    splines, _ = make_pair(which)
    for s in splines:
        for coord in range(3):
            total = s.end_time()
            for it in s.mutable_nodes(POSITION, coord):
                s.set_vars(POSITION, coord, it, it, 3.1)
            vec = s.as_qp_vec(POSITION, coord)
            for i in range(100):
                time = i * (total / 100.0)
                idx, cnt = s.vars_idx(POSITION, coord, time)
                w = s.lin(POSITION, coord, time)
                assert len(w) == cnt
                assert abs(s.value(POSITION, coord, time) - float(vec[idx:idx + cnt] @ w)) < MARGIN
            for it in s.mutable_nodes(FORCE, coord):
                s.set_vars(FORCE, coord, it, it, 1.4 / FORCE_MULT)
            _check_force_reconstruction(s, coord, 0.0, total)


@pytest.mark.parametrize("which", WHICH)
def test_add_remove_polys(which):   # splines_tests.cpp:160-237
    splines, times = make_pair(which)
    addt = 0.2
    for s in splines:
        for i in range(3):
            s.add_poly(addt)
            assert abs(s.end_time() - (times[-1] + (i + 1) * addt)) < MARGIN
        for coord in range(3):
            for it in s.mutable_nodes(FORCE, coord):
                s.set_vars(FORCE, coord, it, it - 1, 0.75 / FORCE_MULT)
            _check_force_reconstruction(s, coord, 0.0, s.end_time())
    for s in splines:
        s.remove_poly(0.5)
        assert abs(s.end_time() - (times[-1] + 3 * addt)) < MARGIN
        for coord in range(3):
            for it in s.mutable_nodes(FORCE, coord):
                s.set_vars(FORCE, coord, it, 2 * it - 1, 0.5 / FORCE_MULT)
            _check_force_reconstruction(s, coord, s.start_time(), s.end_time())
            # The reference's (unregistered, test/CMakeLists.txt:17-20) test keeps calling RemovePoly(0.5 + i*0.1) for
            # every coord; once the start has moved past the requested time its own code throws "Time requested is too
            # small." (end_effector_splines.cpp:1065-1066) -- observed with oracle/_ref.  Same behaviour is required.
            for i in range(20):
                try:
                    s.remove_poly(0.5 + i * 0.1)
                except po.OracleError as e:
                    assert "too small" in str(e)
                    assert 0.5 + i * 0.1 < s.start_time() - 1e-4
                    break


def _fd_failures_value(s, typ, ncoord):
    """(time, contact, coord, partial, fd) where |partial - fd| > 1e-4, as in splines_tests.cpp:253-325."""
    dt = math.sqrt(1e-16)
    bad = []
    ctimes = _contact_times(s)
    s2 = s.clone()
    time = 0.0
    while time < s.end_time():
        for contact in range(len(ctimes)):
            for coord in range(ncoord):
                v1 = s.value(typ, coord, time)
                c2 = ctimes.copy()
                c2[contact] += dt
                s2.set_contact_times(c2)
                v2 = s2.value(typ, coord, time)
                fd = (v2 - v1) / dt
                p = s.partial(typ, coord, time, contact)
                if abs(p - fd) > 1e-4:
                    bad.append((time, contact, coord, p, fd))
                s2.set_contact_times(ctimes)
        time += 0.01
    return bad


def _contact_times(s):
    """Contact (lift-off / touch-down) times: the knots where the x-position spline has a non-empty knot."""
    t = s.times()
    return np.array([t[i] for i in range(s.num_nodes()) if s.node_type(POSITION, 0, i) != po.EMPTY])


@pytest.mark.parametrize("which", WHICH)
def test_value_partials_fd(which):   # splines_tests.cpp:239-325
    splines, _ = make_pair(which)
    for s in splines:
        for coord in range(3):
            for it in s.mutable_nodes(FORCE, coord):
                s.set_vars(FORCE, coord, it, 2 * it - 1, 0.5 / FORCE_MULT)
        assert _fd_failures_value(s, FORCE, 3) == []
        for coord in range(2):
            for it in s.mutable_nodes(POSITION, coord):
                s.set_vars(POSITION, coord, it, 2 * it - 1, 0.5)
        assert _fd_failures_value(s, POSITION, 2) == []


@pytest.mark.parametrize("which", WHICH)
def test_coefficient_partials_fd(which):   # splines_tests.cpp:327-444
    splines, _ = make_pair(which)
    dt = math.sqrt(1e-16)
    for s in splines:
        for coord in range(3):
            for it in s.mutable_nodes(FORCE, coord):
                s.set_vars(FORCE, coord, it, 2 * it - 1, 0.5 / FORCE_MULT)
        ctimes = _contact_times(s)
        s2 = s.clone()
        time = 0.0
        while time < s.end_time():
            if s.is_force_mutable(time):
                for contact in range(len(ctimes)):
                    for coord in range(3):
                        w = s.lin(FORCE, coord, time)
                        c2 = ctimes.copy()
                        c2[contact] += dt
                        s2.set_contact_times(c2)
                        if s2.is_force_mutable(time):
                            w2 = s2.lin(FORCE, coord, time)
                            assert len(w) == len(w2)
                            dw = s.coef_partial(FORCE, coord, time, contact)
                            assert len(dw) == len(w)
                            assert np.all(np.abs(dw - (w2 - w) / dt) < 1e-4), (time, contact, coord)
                        s2.set_contact_times(ctimes)
            time += 0.01
        for coord in range(3):
            for it in s.mutable_nodes(POSITION, coord):
                s.set_vars(POSITION, coord, it, 2 * it - 1, 0.5 / FORCE_MULT)
        s2 = s.clone()
        time = 0.0
        while time < s.end_time():
            for contact in range(len(ctimes)):
                for coord in range(2):
                    w = s.lin(POSITION, coord, time)
                    c2 = ctimes.copy()
                    c2[contact] += dt
                    s2.set_contact_times(c2)
                    w2 = s2.lin(POSITION, coord, time)
                    if len(w) == len(w2):
                        dw = s.coef_partial(POSITION, coord, time, contact)
                        assert len(dw) == len(w)
                        assert np.all(np.abs(dw - (w2 - w) / dt) < 1e-4), (time, contact, coord)
                    s2.set_contact_times(ctimes)
            time += 0.01


# ---------------------------------------------------------------------------------------- restatement vs reference
def _ref_spline(times, sic, digest):
    """The reference's compiled spline, or the restatement standing in for it; what it returns goes into `digest`."""
    return common.Recorded(po.FootSpline(times, sic, 3, "ref" if po.have_ref() else "oracle"), digest)


def _random_spline_pair(rng, digest):
    n = int(rng.integers(3, 8))
    gaps = rng.uniform(0.15, 0.45, size=n - 1)
    times = np.concatenate([[0.0], np.cumsum(gaps)])
    sic = bool(rng.integers(0, 2))
    a, b = po.FootSpline(times, sic, 3, "oracle"), _ref_spline(times, sic, digest)
    for _ in range(int(rng.integers(0, 3))):
        d = float(rng.uniform(0.2, 0.4))
        a.add_poly(d)
        b.add_poly(d)
    for coord in range(3):
        for it in a.mutable_nodes(FORCE, coord):
            v = rng.normal(size=2) * [50.0, 1.0]
            a.set_vars(FORCE, coord, it, *v)
            b.set_vars(FORCE, coord, it, *v)
        for it in a.mutable_nodes(POSITION, coord):
            v = rng.normal(size=2) * [0.3, 0.5]
            a.set_vars(POSITION, coord, it, *v)
            b.set_vars(POSITION, coord, it, *v)
    return a, b


def test_restatement_matches_compiled_reference_bitwise():
    rng = np.random.default_rng(0)
    digest = hashlib.sha256()
    for trial in range(40):
        a, b = _random_spline_pair(rng, digest)
        if trial % 3 == 0:
            t_rm = float(rng.uniform(a.start_time(), 0.5 * a.end_time()))
            a.remove_poly(t_rm)
            b.remove_poly(t_rm)
        assert a.num_nodes() == b.num_nodes()
        assert np.array_equal(a.times(), b.times())
        nct = a.num_contacts()
        assert nct == b.num_contacts()
        for typ in (FORCE, POSITION):
            for coord in range(3):
                assert a.mutable_nodes(typ, coord) == b.mutable_nodes(typ, coord)
                assert np.array_equal(a.as_qp_vec(typ, coord), b.as_qp_vec(typ, coord))
        ts = np.concatenate([rng.uniform(a.start_time(), a.end_time(), size=60), a.times()])
        for t in ts:
            t = float(t)
            assert a.is_force_mutable(t) == b.is_force_mutable(t)
            assert a.is_in_contact(t) == b.is_in_contact(t)
            assert a.next_td(t) == b.next_td(t) or (math.isnan(a.next_td(t)) and math.isnan(b.next_td(t)))
            assert a.swing_time(t) == b.swing_time(t)
            for coord in range(3):
                assert a.value(FORCE, coord, t) == b.value(FORCE, coord, t)
                assert a.value(POSITION, coord, t) == b.value(POSITION, coord, t)
                assert a.vars_idx(POSITION, coord, t) == b.vars_idx(POSITION, coord, t)
                assert np.array_equal(a.lin(POSITION, coord, t), b.lin(POSITION, coord, t))
                if a.is_force_mutable(t):
                    assert a.vars_idx(FORCE, coord, t) == b.vars_idx(FORCE, coord, t)
                    assert np.array_equal(a.lin(FORCE, coord, t), b.lin(FORCE, coord, t))
                for c in range(nct):
                    try:
                        pa = a.partial(FORCE, coord, t, c)
                    except po.OracleError:
                        with pytest.raises(po.OracleError):
                            b.partial(FORCE, coord, t, c)
                        continue
                    pb = b.partial(FORCE, coord, t, c)
                    assert pa == pb or (math.isnan(pa) and math.isnan(pb)) or (math.isinf(pa) and math.isinf(pb))
                    if coord < 2:
                        pa, pb = a.partial(POSITION, coord, t, c), b.partial(POSITION, coord, t, c)
                        assert pa == pb or (not math.isfinite(pa) and not math.isfinite(pb))
                    if a.is_force_mutable(t) and t < a.end_time():
                        for dtw in (0.0, 0.3):
                            assert np.array_equal(a.coef_partial(FORCE, coord, t, c, dtw),
                                                  b.coef_partial(FORCE, coord, t, c, dtw), equal_nan=True)
                    if coord < 2 and t < a.end_time():
                        assert np.array_equal(a.coef_partial(POSITION, coord, t, c), b.coef_partial(POSITION, coord, t, c),
                                              equal_nan=True)
        # contact-time edits
        ct = _contact_times(a)
        ct2 = ct + np.concatenate([[0.0], np.sort(rng.uniform(-0.03, 0.03, size=len(ct) - 1))])
        ct2 = np.maximum.accumulate(ct2)
        a.set_contact_times(ct2)
        b.set_contact_times(ct2)
        assert np.array_equal(a.times(), b.times())
    common.check_golden_reference("splines_random", digest)


def test_set_to_touchdown_matches_reference():
    times = [0, 0.3, 0.6, 0.9, 1.2]
    digest = hashlib.sha256()
    for sic in (False, True):
        a, b = po.FootSpline(times, sic, 3, "oracle"), _ref_spline(times, sic, digest)
        td = a.next_td(0.05)
        assert td == b.next_td(0.05)
        a.set_to_touchdown(td - 0.04)
        b.set_to_touchdown(td - 0.04)
        assert np.array_equal(a.times(), b.times())
        for bad in (td + 5.0,):
            with pytest.raises(po.OracleError):
                a.set_to_touchdown(bad)
            with pytest.raises(po.OracleError):
                b.set_to_touchdown(bad)
    common.check_golden_reference("splines_set_to_touchdown", digest)
