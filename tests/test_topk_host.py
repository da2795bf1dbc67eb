"""Host side of q3_score_topk: the Python wrappers' shapes, dtypes and argument checks over a fake library (CPU), and the C++
header's Transformer::score_topk (compiled here; on the GPU its results equal the Python binding's bit for bit)."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

from qwen3_rs_b200 import build
from qwen3_rs_b200 import transformer as T

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _view(ptr, dtype, n):
    ct = C.c_int32 if dtype == np.int32 else C.c_float
    return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(ct)), shape=(n,))


class _FakeLib:
    """Records the top-k calls and fills every output: ids[i][j] = 10 i + j, lps[i][j] = -j, lp[i] = -0.5, argmax[i] = 10 i."""

    def __init__(self):
        self.calls = []

    def _fill(self, rows, k, ids, lps, lp, am):
        _view(ids, np.int32, rows * k)[:] = (10 * np.arange(rows)[:, None] + np.arange(k)).reshape(-1)
        _view(lps, np.float32, rows * k)[:] = np.tile(-np.arange(k, dtype=np.float32), rows)
        if lp is not None:
            _view(lp, np.float32, rows)[:] = -0.5
        if am is not None:
            _view(am, np.int32, rows)[:] = 10 * np.arange(rows)
        return 0

    def q3_score_topk(self, h, tokens, n, pos0, k, ids, lps, targets, lp, am):
        self.calls.append(("score_topk", n, pos0, k, targets is not None, lp is not None, am is not None))
        return self._fill(n, k, ids, lps, lp, am)

    def q3_op_topk_logprobs(self, device, logits, rows, n, k, targets, ids, lps, lp, am):
        self.calls.append(("op", rows, n, k, targets is not None, lp is not None, am is not None))
        return self._fill(rows, k, ids, lps, lp, am)


@pytest.fixture
def fake(monkeypatch):
    lib = _FakeLib()
    monkeypatch.setattr(T, "_lib", lib)
    return lib


def _fake_transformer():
    m = object.__new__(T.Transformer)
    m._h = 1
    return m


def test_score_topk_shapes_and_outputs(fake):
    m = _fake_transformer()
    ids, lps, lp, am = m.score_topk([5, 6, 7], 4, targets=[6, 7, 8], pos0=9)
    assert fake.calls == [("score_topk", 3, 9, 4, True, True, True)]
    assert ids.shape == (3, 4) and ids.dtype == np.int32 and lps.shape == (3, 4) and lps.dtype == np.float32
    assert ids[2].tolist() == [20, 21, 22, 23] and lps[1].tolist() == [0.0, -1.0, -2.0, -3.0]
    assert lp.tolist() == [-0.5] * 3 and am.tolist() == [0, 10, 20]
    ids, lps, lp, am = m.score_topk(np.array([1, 2]), 64, want_argmax=False)
    assert fake.calls[-1] == ("score_topk", 2, 0, 64, False, False, False)
    assert ids.shape == (2, 64) and lp is None and am is None


def test_op_topk_logprobs_shapes_and_outputs(fake):
    ids, lps, lp, am = T.op_topk_logprobs(np.zeros((3, 100), np.float32), 2, targets=[0, 1, 2])
    assert fake.calls == [("op", 3, 100, 2, True, True, True)]
    assert ids.shape == (3, 2) and lps.shape == (3, 2) and lp.shape == (3,) and am.shape == (3,)
    ids, _, lp, am = T.op_topk_logprobs(np.zeros(50), 1, want_argmax=False)  # one row; float64 input converted
    assert fake.calls[-1] == ("op", 1, 50, 1, False, False, False)
    assert ids.shape == (1, 1) and lp is None and am is None


@pytest.mark.parametrize("k", [0, -1, 65, 2.5, True, None])
def test_bad_k_is_refused_before_the_library(fake, k):
    with pytest.raises((ValueError, TypeError)):
        _fake_transformer().score_topk([1, 2], k)
    with pytest.raises((ValueError, TypeError)):
        T.op_topk_logprobs(np.zeros((2, 100), np.float32), k)
    assert fake.calls == []


def test_target_count_must_match(fake):
    with pytest.raises(ValueError):
        _fake_transformer().score_topk([1, 2, 3], 2, targets=[1, 2])
    with pytest.raises(ValueError):
        T.op_topk_logprobs(np.zeros((2, 100), np.float32), 2, targets=[1, 2, 3])
    assert fake.calls == []


def test_topk_max_matches_the_header():
    src = open(os.path.join(ROOT, "include", "qwen3_cuda.h")).read()
    assert f"#define Q3_TOPK_MAX {T.TOPK_MAX}\n" in src


@pytest.fixture(scope="module")
def topk_check(tmp_path_factory):
    cxx = shutil.which("g++")
    if cxx is None:
        pytest.skip("g++ not available")
    lib = build.build()
    out = str(tmp_path_factory.mktemp("cpp") / "topk_check")
    libdir = os.path.dirname(lib)
    subprocess.check_call([cxx, "-std=c++17", "-O1", "-ffp-contract=off", "-Wall", "-Wextra", "-Werror",
                           os.path.join(ROOT, "tests", "cpp", "topk_check.cpp"), "-I", os.path.join(ROOT, "include"),
                           "-L", libdir, "-lqwen3cuda", "-Wl,-rpath," + libdir, "-o", out])
    return out


def test_cpp_topk_compiles(topk_check):
    assert os.access(topk_check, os.X_OK)


@pytest.mark.gpu
def test_cpp_topk_matches_the_python_binding(topk_check, ckpt):
    path = ckpt("small", 64, 3)
    k = 20
    toks = np.random.default_rng(5).integers(0, 4096, 81).tolist()
    r = subprocess.run([topk_check, path, *map(str, [7, k, *toks[:80], "--", *toks[1:]])], capture_output=True, text=True,
                       timeout=120)
    assert r.returncode == 0, r.stderr
    lines = r.stdout.split("\n")
    ids_cpp = [int(x) for x in lines[0].split()]
    lps_cpp = np.array([int(x, 16) for x in lines[1].split()], np.uint32)
    lp_cpp = np.array([int(x, 16) for x in lines[2].split()], np.uint32)
    am_cpp = [int(x) for x in lines[3].split()]
    assert lines[4].strip() == "-1"  # Q3_EINVAL for an out-of-range target, thrown as qwen3::Error
    m = T.TransformerBuilder.new(path).build()
    try:
        ids, lps, lp, am = m.score_topk(toks[:80], k, targets=toks[1:], pos0=7)
    finally:
        m.close()
    assert ids_cpp == ids.reshape(-1).tolist() and np.array_equal(lps_cpp, lps.reshape(-1).view(np.uint32))
    assert np.array_equal(lp_cpp, lp.view(np.uint32)) and am_cpp == am.tolist()
