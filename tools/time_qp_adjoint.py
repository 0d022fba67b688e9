"""Wall time of the generic QP solve (bgg_qp_solve_batch) and of its derivative (bgg_qp_adjoint_batch) on batches of QPs.

For each (n, me, mi) a batch of QPs on one pattern (A at the density printed, built around a known optimum as in
tests/test_oracle_qp_adjoint.py; q and b differ per QP) is solved, and the adjoint is taken at the solutions with dx = P x + q,
as the reference passes it.  Both calls are synchronous and include their host <-> device copies (pattern, values, points,
outputs), which is what a caller of the C ABI pays.  Warm-up first, then the two calls alternate; the median of the repetitions
is printed.  The card's name and power limit are read in the same run.

    python tools/time_qp_adjoint.py [--count 4096] [--reps 20]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import scipy.sparse as sp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "bilevel-gait-gen_b200"), os.path.join(ROOT, "tests"), os.path.join(ROOT, "oracle")):
    sys.path.insert(0, p)

import bgg_b200 as bg  # noqa: E402
import common  # noqa: E402
from test_oracle_qp_adjoint import margin_qps  # noqa: E402

SHAPES = [(3, 2, 4, 1.0), (42, 18, 60, 0.5), (128, 32, 256, 0.5)]   # n, me, mi, density of A


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                              timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--count", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    gpu = common.make_gpu("a1_configuration", 1)
    L, h = gpu.L, gpu.h
    print(f"# card: {card()}")
    print("# both calls synchronous, host<->device copies included; median of", args.reps, "repetitions after", args.warmup, "warm-up calls")
    for n, me, mi, dens in SHAPES:
        Q = margin_qps(7, n, me, mi // 2, mi - mi // 2, 0, count=1, density=dens)
        P, A, is_eq = sp.csc_matrix(np.triu(Q["P"][0])), sp.csc_matrix(Q["A"][0]), Q["is_eq"]
        P.sort_indices()
        A.sort_indices()
        m, cnt = A.shape[0], args.count
        rng = np.random.default_rng(1)
        pc, pr = P.indptr.astype(np.int32), P.indices.astype(np.int32)
        ac, ar = A.indptr.astype(np.int32), A.indices.astype(np.int32)
        pv = np.ascontiguousarray(np.tile(P.data, (cnt, 1)))
        av = np.ascontiguousarray(np.tile(A.data, (cnt, 1)))
        q = np.ascontiguousarray(Q["q"][0] + 0.01 * rng.normal(size=(cnt, n)))
        b = np.ascontiguousarray(Q["b"][0] + 0.01 * rng.uniform(size=(cnt, m)))
        eq = np.ascontiguousarray(is_eq.astype(np.uint8))
        x, y, s = np.zeros((cnt, n)), np.zeros((cnt, m)), np.zeros((cnt, m))
        st, it = np.zeros(cnt, np.int32), np.zeros(cnt, np.int32)
        dz, dy, db, dA, ast = np.zeros((cnt, n)), np.zeros((cnt, m)), np.zeros((cnt, m)), np.zeros((cnt, len(ar))), np.zeros(cnt, np.int32)
        u8 = eq.ctypes.data_as(C.POINTER(C.c_uint8))
        I, D = bg._i, bg._d

        def solve():
            gpu._chk(L.bgg_qp_solve_batch(h, cnt, n, m, I(pc), I(pr), D(pv), I(ac), I(ar), D(av), D(q), D(b), u8, D(x), D(y), D(s), I(st), I(it)))

        dxv = None

        def adjoint():
            gpu._chk(L.bgg_qp_adjoint_batch(h, cnt, n, m, I(pc), I(pr), D(pv), I(ac), I(ar), D(av), u8, D(x), D(y), D(s), D(dxv), D(dz), D(dy),
                                            D(db), D(dA), I(ast)))

        solve()
        Pf = Q["P"][0]
        dxv = np.ascontiguousarray(x @ Pf.T + q)   # Computedx
        for _ in range(args.warmup):
            solve()
            adjoint()
        ts, ta = [], []
        for _ in range(args.reps):
            t0 = time.perf_counter()
            solve()
            ts.append(time.perf_counter() - t0)
            t0 = time.perf_counter()
            adjoint()
            ta.append(time.perf_counter() - t0)
        res = dict(n=n, me=me, mi=mi, A_density=dens, nnzA=int(len(ar)), count=cnt, solve_ms=1e3 * float(np.median(ts)),
                   adjoint_ms=1e3 * float(np.median(ta)), solve_status0=int((st == 0).sum()), adjoint_status0=int((ast == 0).sum()),
                   median_iters=float(np.median(it)))
        res["adjoint_over_solve"] = res["adjoint_ms"] / res["solve_ms"]
        print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
