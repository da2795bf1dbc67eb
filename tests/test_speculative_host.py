"""Host side of q3_forward_multi / q3_decode_speculative: the Python wrappers' shapes and argument checks over a fake library
(CPU), and the C++ header's Transformer::forward_multi / decode_speculative (compiled and linked here)."""
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
    """Records the calls; forward_multi writes argmax[i] = tokens[i] + 1 and logits[i][j] = i; decode_speculative writes
    tokens_out[i] = first + i and the statistics (1, 2, 3)."""

    def __init__(self):
        self.calls = []

    def q3_forward_multi(self, h, tokens, n, pos0, am, lg):
        self.calls.append(("multi", h, n, pos0, lg is not None))
        _view(am, np.int32, n)[:] = _view(tokens, np.int32, n) + 1
        if lg is not None:
            _view(lg, np.float32, n * 10)[:] = np.repeat(np.arange(n, dtype=np.float32), 10)
        return 0

    def q3_decode_speculative(self, h, d, first, pos0, n, k, out, r, dr, a):
        self.calls.append(("spec", h, d, first, pos0, n, k))
        if n:
            _view(out, np.int32, n)[:] = first + np.arange(n)
        for p, v in ((r, 1), (dr, 2), (a, 3)):
            C.cast(p, C.POINTER(C.c_int)).contents.value = v
        return 0


@pytest.fixture
def fake(monkeypatch):
    lib = _FakeLib()
    monkeypatch.setattr(T, "_lib", lib)
    return lib


def _fake_transformer(h=1):
    m = object.__new__(T.Transformer)
    m._h = h
    m._config = T.ModelConfig(1, 128, 384, 2, 2, 1, 128, 64, 10, 32, False)
    return m


def test_forward_multi_shapes_and_outputs(fake):
    am, lg = _fake_transformer().forward_multi([4, 5, 6], 7, want_logits=True)
    assert fake.calls == [("multi", 1, 3, 7, True)]
    assert am.dtype == np.int32 and am.tolist() == [5, 6, 7]
    assert lg.shape == (3, 10) and lg.dtype == np.float32 and lg[2].tolist() == [2.0] * 10
    am, lg = _fake_transformer().forward_multi(np.arange(T.MULTI_MAX), 0)
    assert fake.calls[-1] == ("multi", 1, T.MULTI_MAX, 0, False) and lg is None and am.size == T.MULTI_MAX


@pytest.mark.parametrize("tokens", [[], list(range(T.MULTI_MAX + 1))])
def test_forward_multi_token_count_is_checked_before_the_library(fake, tokens):
    with pytest.raises(ValueError):
        _fake_transformer().forward_multi(tokens, 0)
    assert fake.calls == []


def test_decode_speculative_outputs(fake):
    tgt, draft = _fake_transformer(1), _fake_transformer(2)
    toks, st = tgt.decode_speculative(draft, 9, 3, 5, 7)
    assert fake.calls == [("spec", 1, 2, 9, 3, 5, 7)]
    assert toks == [9, 10, 11, 12, 13] and st == {"rounds": 1, "drafted": 2, "accepted": 3}
    toks, _ = tgt.decode_speculative(draft, 9, 3, 0, 1)
    assert toks == []


@pytest.mark.parametrize("k", [0, -1, T.MULTI_MAX, 2.5, True])
def test_decode_speculative_bad_k_is_refused_before_the_library(fake, k):
    with pytest.raises((ValueError, TypeError)):
        _fake_transformer(1).decode_speculative(_fake_transformer(2), 1, 0, 4, k)
    assert fake.calls == []


@pytest.mark.parametrize("n", [-1, 2.5])
def test_decode_speculative_bad_n_is_refused_before_the_library(fake, n):
    with pytest.raises(ValueError):
        _fake_transformer(1).decode_speculative(_fake_transformer(2), 1, 0, n, 3)
    assert fake.calls == []


def test_decode_speculative_draft_must_be_a_transformer(fake):
    with pytest.raises(TypeError):
        _fake_transformer().decode_speculative(object(), 1, 0, 4, 3)
    assert fake.calls == []


def test_multi_max_matches_the_header():
    src = open(os.path.join(ROOT, "include", "qwen3_cuda.h")).read()
    assert f"#define Q3_MULTI_MAX {T.MULTI_MAX}\n" in src


CPP = r"""
#include "qwen3_transformer.hpp"
#include <cstdio>
int main(int argc, char **argv) {
    if (argc < 3) return 2;  // never run: compiled and linked only
    qwen3::Transformer t = qwen3::TransformerBuilder(argv[1]).build();
    qwen3::Transformer d = qwen3::TransformerBuilder(argv[2]).build();
    auto m = t.forward_multi({1, 2, 3}, 0, true);
    qwen3::Transformer::SpecStats st;
    auto toks = t.decode_speculative(d, 1, 0, 8, 3, &st);
    std::printf("%d %zu %zu %d\n", m.argmax[0], m.logits.size(), toks.size(), st.rounds);
    return 0;
}
"""


def test_cpp_header_methods_compile_and_link(tmp_path):
    cxx = shutil.which("g++")
    if cxx is None:
        pytest.skip("g++ not available")
    lib = build.build()
    src = tmp_path / "spec.cpp"
    src.write_text(CPP)
    libdir = os.path.dirname(lib)
    subprocess.check_call([cxx, "-std=c++17", "-O1", "-ffp-contract=off", "-Wall", "-Wextra", "-Werror", str(src), "-I",
                           os.path.join(ROOT, "include"), "-L", libdir, "-lqwen3cuda", "-Wl,-rpath," + libdir, "-o",
                           str(tmp_path / "spec")])
