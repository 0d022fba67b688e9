"""k_ipm's fused block reduction (bgg::block_reduce_multi, csrc/bgg_kernels.cuh) through a test-only kernel
(tests/cuda/reduce_harness.cu), against a restatement of the rounding it must keep: per value the 5-level XOR butterfly
of warp_sum / warp_max (at each level lane l adds lane l ^ o's partial), then the warps' results combined in warp order
0, 1, 2, ...  Sums must equal it bit for bit; maxima must equal it as numbers (the order of fmax may change which zero
of +0 / -0 survives, nothing else).  Partials span 1e-300 to 1e300 with heavy cancellation, zeros and negative zeros,
so a sum taken in any other order differs in its bits.
"""
import os
import shutil
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHAPES = [(4, 4), (3, 0), (0, 2)]   # (sums, maxima) as k_ipm reduces them: residual norms, pass scalars, starting point
COUNT = 64


def _harness_path(tmp_dir):
    src = os.path.join(ROOT, "tests", "cuda", "reduce_harness.cu")
    prebuilt = os.path.join(ROOT, "tools", "bin", "libreduce_harness.so")
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        if os.path.exists(prebuilt):
            return prebuilt
        pytest.skip("nvcc not found and the reduction harness is not built (python -c 'import __graft_entry__ as g; g.build()')")
    out = os.path.join(tmp_dir, "libreduce_harness.so")
    subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-maxrregcount=128", "-Xcompiler", "-fPIC", "-shared",
                    "-I", os.path.join(ROOT, "bilevel-gait-gen_b200", "csrc"), "-o", out, src], check=True)
    return out


@pytest.fixture(scope="module")
def reduce(tmp_path_factory):
    import ctypes as C
    lib = C.CDLL(_harness_path(str(tmp_path_factory.mktemp("reduce_harness"))))
    dp = C.POINTER(C.c_double)
    lib.reduce_harness_run.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, dp, dp]

    def run(ns, nm, threads, x):
        x = np.ascontiguousarray(x, np.float64)
        out = np.empty_like(x)
        rc = lib.reduce_harness_run(ns, nm, threads, x.shape[0], x.ctypes.data_as(dp), out.ctypes.data_as(dp))
        assert rc == 0, f"reduce_harness_run: error {rc}"
        return out
    return run


def _partials(rng, count, threads, k):
    """[count][threads][k]: magnitudes 1e-300 .. 1e300, every value followed somewhere in its warp by its negation or a near
    negation, plus runs of +0 and -0.  The sum of 512 of them stays below the overflow threshold."""
    x = np.sign(rng.standard_normal((count, threads, k))) * 10.0 ** rng.uniform(-300, 300, (count, threads, k))
    near = x * (1 + rng.uniform(-1e-12, 1e-12, x.shape))
    perm = rng.permuted(np.arange(threads).reshape(threads // 32, 32), axis=1).reshape(-1)   # partner within the same warp
    half = rng.random(x.shape) < 0.5
    x = np.where(half, x, -near[:, perm, :])
    z = rng.random(x.shape)
    x[z < 0.05] = 0.0
    x[(z >= 0.05) & (z < 0.10)] = -0.0
    return x


def _butterfly(x, op):
    """Per warp, the value lane 0 holds after warp_sum / warp_max: at o = 16, 8, 4, 2, 1 lane l computes op(a_l, a_{l ^ o})."""
    a = x.reshape(x.shape[0], x.shape[1] // 32, 32, x.shape[-1])
    lanes = np.arange(32)
    for o in (16, 8, 4, 2, 1):
        a = op(a, a[:, :, lanes ^ o, :])
    return a[:, :, 0, :]   # [count][warps][k]


def _reference(x, ns):
    s = _butterfly(x[..., :ns], np.add)
    m = _butterfly(x[..., ns:], np.fmax)
    rs, rm = s[:, 0, :].copy(), m[:, 0, :].copy()
    for w in range(1, s.shape[1]):   # warp order, one value at a time
        rs = rs + s[:, w, :]
        rm = np.fmax(rm, m[:, w, :])
    return rs, rm


@pytest.mark.parametrize("threads", [256, 512])
@pytest.mark.parametrize("ns,nm", SHAPES)
def test_block_reduce_multi_keeps_the_butterfly_rounding(reduce, ns, nm, threads):
    rng = np.random.default_rng(1000 * ns + 10 * nm + threads)
    x = _partials(rng, COUNT, threads, ns + nm)
    out = reduce(ns, nm, threads, x)
    rs, rm = _reference(x, ns)
    # every thread holds the result
    assert (out.view(np.uint64) == out[:, :1, :].view(np.uint64)).all(), "the result is not the same in every thread"
    got = out[:, 0, :]
    assert np.isfinite(rs).all() and np.isfinite(rm).all()
    assert np.array_equal(got[:, :ns].view(np.uint64), rs.view(np.uint64)), "sums differ in their bits from the butterfly's"
    assert np.array_equal(got[:, ns:], rm), "maxima differ from the butterfly's"
    # the restatement is order-sensitive on these inputs: a plain sequential sum over all threads rounds differently
    if ns:
        seq = x[..., :ns].copy()
        acc = seq[:, 0, :].copy()
        for t in range(1, threads):
            acc = acc + seq[:, t, :]
        assert not np.array_equal(acc.view(np.uint64), rs.view(np.uint64))
