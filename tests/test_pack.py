"""CPU checks of the host-side packing loops of the ``*_host`` entry points (csrc/ml_pack.cpp).

``ml_pack_index_rows`` / ``ml_pack_rows`` compress a level row to the cells where the reference volcello
is present -- the only cells the reference reads (src/momlevel/steric.py:151-153, 163).  They are plain
host code, so they are checked here against numpy boolean indexing; the transfer built on them is checked
on the GPU (tests/test_gpu_steric.py::test_host_packed_transfer_*).
"""

import ctypes

import numpy as np
import pytest


@pytest.fixture(scope="module")
def L():
    from momlevel_b200 import _lib

    return _lib.lib()


def _ptr(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _index(L, V):
    nrows, ncol = V.shape
    ngrp = (ncol + 31) // 32
    words = np.zeros((nrows, ngrp), dtype=np.uint32)
    before = np.zeros((nrows, ngrp), dtype=np.uint32)
    count = np.zeros(nrows, dtype=np.uint64)
    total = L.ml_pack_index_rows(_ptr(V), nrows, ncol, _ptr(words), _ptr(before), _ptr(count))
    return words, before, count, total


@pytest.mark.parametrize("ncol", [1, 25, 31, 32, 33, 64, 1000, 4099])
@pytest.mark.parametrize("wet", [0.0, 0.07, 0.5, 0.93, 1.0])
def test_index_and_pack_match_numpy(L, ncol, wet):
    rng = np.random.default_rng(ncol * 7 + int(wet * 100))
    nrows = 3
    V = rng.uniform(1.0, 2.0, (nrows, ncol)).astype(np.float32)
    V[rng.uniform(size=V.shape) >= wet] = np.nan
    if wet == 0.5:  # other NaN payloads and infinities: only "is NaN" decides
        V.view(np.uint32)[0, 0] = 0xFFC00001
        V[1, 0] = np.inf
    T = rng.normal(10, 5, (nrows, ncol)).astype(np.float32)
    S = rng.normal(35, 1, (nrows, ncol)).astype(np.float32)
    T[rng.uniform(size=T.shape) < 0.1] = np.nan  # holes in the fields travel as they are
    words, before, count, total = _index(L, V)
    present = ~np.isnan(V)
    assert total == present.sum()
    assert np.array_equal(count, present.sum(axis=1).astype(np.uint64))
    ngrp = (ncol + 31) // 32
    padded = np.zeros((nrows, ngrp * 32), dtype=bool)
    padded[:, :ncol] = present
    bits = padded.reshape(nrows, ngrp, 32)
    assert np.array_equal(words, (bits.astype(np.uint64) << np.arange(32, dtype=np.uint64)).sum(axis=2).astype(np.uint32))
    assert np.array_equal(before, np.cumsum(bits.sum(axis=2), axis=1) - bits.sum(axis=2))
    for r in range(nrows):
        n = int(count[r])
        for cuts in ([0, ngrp], [0, ngrp // 2, ngrp], list(range(ngrp + 1))[:: max(1, ngrp // 5)] + [ngrp]):
            guard = np.float32(-777.0)
            t_out = np.full(n + 40, guard, dtype=np.float32)
            s_out = np.full(n + 40, guard, dtype=np.float32)
            pack = L.ml_pack_rows if len(cuts) % 2 else L.ml_pack_rows_cached  # non-temporal / ordinary stores
            for g0, g1 in zip(cuts[:-1], cuts[1:]):
                pack(_ptr(T[r]), _ptr(S[r]), _ptr(words[r]), _ptr(before[r]), g0, g1, ncol, _ptr(t_out), _ptr(s_out))
            assert np.array_equal(t_out[:n].view(np.uint32), T[r][present[r]].view(np.uint32))
            assert np.array_equal(s_out[:n].view(np.uint32), S[r][present[r]].view(np.uint32))
            assert np.all(t_out[n:] == guard) and np.all(s_out[n:] == guard), "wrote past the row's share"


def test_simd_body_is_reported(L):
    assert L.ml_pack_simd() in (0, 512)


def test_scalar_bodies_give_the_same_rows():
    """A CPU without AVX-512 runs the scalar loops; force them in a fresh process and repeat one case."""
    import os
    import subprocess
    import sys

    code = (
        "import ctypes, numpy as np\n"
        "from momlevel_b200 import _lib\n"
        "L = _lib.lib()\n"
        "assert L.ml_pack_simd() == 0\n"
        "p = lambda a: a.ctypes.data_as(ctypes.c_void_p)\n"
        "rng = np.random.default_rng(4)\n"
        "ncol = 1003; ngrp = (ncol + 31) // 32\n"
        "V = rng.uniform(1, 2, (2, ncol)).astype(np.float32); V[rng.uniform(size=V.shape) < 0.6] = np.nan\n"
        "T = rng.normal(size=(2, ncol)).astype(np.float32); S = rng.normal(size=(2, ncol)).astype(np.float32)\n"
        "w = np.zeros((2, ngrp), np.uint32); b = np.zeros((2, ngrp), np.uint32); c = np.zeros(2, np.uint64)\n"
        "assert L.ml_pack_index_rows(p(V), 2, ncol, p(w), p(b), p(c)) == (~np.isnan(V)).sum()\n"
        "for r in range(2):\n"
        "    n = int(c[r]); to = np.zeros(n + 8, np.float32); so = np.zeros(n + 8, np.float32)\n"
        "    L.ml_pack_rows(p(T[r]), p(S[r]), p(w[r]), p(b[r]), 0, ngrp // 2, ncol, p(to), p(so))\n"
        "    L.ml_pack_rows(p(T[r]), p(S[r]), p(w[r]), p(b[r]), ngrp // 2, ngrp, ncol, p(to), p(so))\n"
        "    m = ~np.isnan(V[r])\n"
        "    assert np.array_equal(to[:n], T[r][m]) and np.array_equal(so[:n], S[r][m]) and not to[n:].any()\n"
        "print('scalar ok')\n"
    )
    env = dict(os.environ, ML_PACK_FORCE_SCALAR="1")
    root = str(__import__("pathlib").Path(__file__).resolve().parent.parent)
    out = subprocess.run([sys.executable, "-c", code], cwd=root, env=env, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "scalar ok" in out.stdout, out.stderr[-2000:]


def test_packing_mode_argument(L):
    # the packing settings and the accounting of the last host call belong to the calling host thread: a fresh
    # thread starts from the defaults whatever host calls other tests made on theirs
    from concurrent.futures import ThreadPoolExecutor

    def body():
        assert L.ml_host_set_packing(5, 0) == -5 and b"packing mode" in L.ml_last_error()
        assert L.ml_host_set_packing(-1, 0) == -5
        for mode in (0, 2, 3, 4, 1):
            assert L.ml_host_set_packing(mode, 0) == 0
        assert L.ml_host_last_packed_fraction() == 0.0

    with ThreadPoolExecutor(max_workers=1) as ex:
        ex.submit(body).result()
