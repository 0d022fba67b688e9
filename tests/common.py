"""Shared helpers for the parity tests: build oracle / CUDA solvers for a named config and mirror a trajectory from
the oracle into the CUDA path's instance POD so both sides start a solve from bit-identical inputs."""
import hashlib
import json
import os
import struct
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "bilevel-gait-gen_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import workloads as wl  # noqa: E402


def make_oracle(cfg_name, init_state=None):
    import pyoracle as po
    cfg = wl.CONFIGS[cfg_name]
    o = po.SrbMpc(cfg["num_nodes"], cfg["integrator_dt"], wl.robot(), **wl.mpc_kwargs(cfg))
    o.set_costs(wl.target_tangent(cfg), np.asarray(cfg["Q"], float))
    s = np.asarray(cfg["srb_init"] if init_state is None else init_state, float)
    o.set_warm_states(np.tile(s, (cfg["num_nodes"] + 1, 1)))
    return o


def make_gpu(cfg_name, batch, init_states=None, **kw):
    import bgg_b200 as bg
    cfg = wl.CONFIGS[cfg_name]
    m = bg.BatchedMPC(cfg["num_nodes"], cfg["integrator_dt"], wl.robot(), **wl.mpc_kwargs(cfg), **kw)
    m.AddQuadraticTrackingCost(wl.target_tangent(cfg), np.asarray(cfg["Q"], float))
    m.Reset(batch)
    s = np.tile(np.asarray(cfg["srb_init"], float), (batch, 1)) if init_states is None else np.asarray(init_states, float)
    m.SetStateTrajectoryWarmStart(s)
    return m


def mirror_oracle_to_gpu(o, gpu, b):
    """Copy the oracle's current trajectory (states, four feet's knots, foot-box size, init time) into GPU instance b."""
    import pyoracle as po
    inst = gpu.get_instance(b)
    st = o.states()
    inst["states"][:st.shape[0]] = st
    for e in range(4):
        f = o.foot(e)
        n = f.num_nodes()
        ft = inst["foot"][e]
        ft["n"] = n
        ft["t"][:n] = f.times()
        ft["ttype"][:n] = f.time_types()
        for c in range(3):
            ty, va = f.knots(po.FORCE, c)
            if c == 0:
                ft["ftype"][:n] = ty
            ft["f"][c, :n] = va
            ty, va = f.knots(po.POSITION, c)
            if c == 0:
                ft["ptype"][:n] = ty
            if c == 2:
                ft["ztype"][:n] = ty
            ft["p"][c, :n] = va
    stt = o.stats()
    inst["ee_box"][:] = [stt["ee_box_x"], stt["ee_box_y"]]
    inst["init_time"] = o.init_time()
    gpu.set_instance(b, inst)


def gpu_rows_to_reference_order(sol, N):
    """Map the kernel's inequality-row order (csrc/bgg_ipm.cu) to the reference's stacked Clarabel rows
    [force box (+ then -) | friction cone | foot box (+ then -)] (mpc.cpp:166-209,352-414; mpc_single_rigid_body.cpp:381-443)."""
    sz = sol["sizes"]
    ns, ne = sz["n_samples"], sz["n_eebox"]
    idx = []
    idx += [6 * j + 0 for j in range(ns)] + [6 * j + 1 for j in range(ns)]
    idx += [6 * j + 2 + r for j in range(ns) for r in range(4)]
    idx += [6 * ns + 2 * e for e in range(ne)] + [6 * ns + 2 * e + 1 for e in range(ne)]
    return np.array(idx)


# Digests of what the reference's own code returned in the bit-for-bit comparisons (tests/test_oracle_vs_reference_mpc.py,
# test_oracle_splines.py, test_oracle_ik.py, test_gpu_parity.py): with the reference's sources absent the comparisons run against
# these, and BGG_RECORD_GOLDEN=1 rewrites them.
GOLDEN_REFERENCE = os.path.join(ROOT, "tests", "golden", "reference_outputs.json")


def _feed(h, v):
    """Hash a value exactly: arrays by dtype, shape and bytes, floats by their IEEE bits."""
    if isinstance(v, np.ndarray):
        h.update(f"a{v.dtype.str}{v.shape}".encode())
        h.update(np.ascontiguousarray(v).tobytes())
    elif isinstance(v, (bool, np.bool_)):
        h.update(b"b1" if v else b"b0")
    elif isinstance(v, (int, np.integer)):
        h.update(f"i{int(v)}".encode())
    elif isinstance(v, (float, np.floating)):
        h.update(b"f" + struct.pack("<d", float(v)))
    elif isinstance(v, str):
        h.update(b"s" + v.encode())
    elif v is None:
        h.update(b"n")
    elif isinstance(v, dict):
        h.update(f"d{len(v)}".encode())
        for k in sorted(v):
            _feed(h, k)
            _feed(h, v[k])
    elif isinstance(v, (list, tuple)):
        h.update(f"l{len(v)}".encode())
        for x in v:
            _feed(h, x)
    elif hasattr(v, "tocsc"):
        m = v.tocsc()
        _feed(h, (m.shape, m.indptr, m.indices, m.data))
    else:
        h.update(b"o" + type(v).__name__.encode())


class Recorded:
    """Wraps the reference side of a comparison and digests every value its methods return (or the exception they raise),
    in call order.  Where the reference's compiled sources are absent the restatement plays that side: the test's own
    assertions then hold trivially, and the digest, compared with the stored one, is what pins the values to the reference's."""

    def __init__(self, obj, digest=None):
        self._obj, self.digest = obj, digest or hashlib.sha256()

    def __getattr__(self, name):
        a = getattr(self._obj, name)
        if not callable(a):
            return a

        def call(*args, **kw):
            try:
                r = a(*args, **kw)
            except Exception as e:
                _feed(self.digest, name + "!" + type(e).__name__)
                raise
            _feed(self.digest, name)
            _feed(self.digest, r)
            return r
        return call


def golden_reference(key):
    with open(GOLDEN_REFERENCE) as f:
        return json.load(f)[key]


def check_golden_reference(key, value):
    """value: a hashlib digest (compared as hex) or a JSON-able value (compared exactly)."""
    v = value.hexdigest() if hasattr(value, "hexdigest") else value
    if os.environ.get("BGG_RECORD_GOLDEN"):
        gold = json.load(open(GOLDEN_REFERENCE)) if os.path.exists(GOLDEN_REFERENCE) else {}
        gold[key] = v
        with open(GOLDEN_REFERENCE, "w") as f:
            json.dump(gold, f, indent=1, sort_keys=True)
        return
    assert golden_reference(key) == v, f"{key}: the values differ from the reference's stored ones"
