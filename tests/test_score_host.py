"""Host side of q3_score: generation.perplexity over a fake transformer (CPU), and the C++ header's Transformer::score (built
like tests/test_cpp_host.py's check; on the GPU its results equal the Python binding's bit for bit)."""
import math
import os
import shutil
import subprocess

import numpy as np
import pytest

from qwen3_rs_b200 import build, generation

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class _FakeScorer:
    """Records the score() calls; log p(target at position p) = -(target + p) / 100."""

    class _Cfg:
        seq_len, vocab_size = 16, 64

    def __init__(self):
        self.calls = []

    def get_config(self):
        return self._Cfg

    def score(self, tokens, targets=None, pos0=0, want_argmax=True):
        self.calls.append((list(tokens), list(targets), pos0, want_argmax))
        lp = np.array([-(t + pos0 + i) / 100.0 for i, t in enumerate(targets)], np.float32)
        return lp, (np.zeros(len(tokens), np.int32) if want_argmax else None)


def test_perplexity_scores_the_next_token_at_each_position():
    f = _FakeScorer()
    toks = [5, 9, 2, 7, 1]
    ppl, total = generation.perplexity(f, toks, pos0=3)
    assert f.calls == [([5, 9, 2, 7], [9, 2, 7, 1], 3, False)]  # one call: targets shifted by one, at pos0
    want = [-(t + 3 + i) / 100.0 for i, t in enumerate([9, 2, 7, 1])]
    assert total == pytest.approx(sum(want), rel=1e-6)
    assert ppl == pytest.approx(math.exp(-sum(want) / 4), rel=1e-6)


def test_perplexity_length_limit():
    f = _FakeScorer()
    generation.perplexity(f, list(range(17)))            # 16 scored positions: exactly seq_len
    generation.perplexity(f, list(range(11)), pos0=6)    # positions 6 .. 15
    for toks, pos0 in ((list(range(18)), 0), (list(range(12)), 6), ([3], 0), ([], 0), ([1, 2], -1)):
        with pytest.raises(ValueError):
            generation.perplexity(f, toks, pos0=pos0)
    assert len(f.calls) == 2


@pytest.fixture(scope="module")
def score_check(tmp_path_factory):
    cxx = shutil.which("g++")
    if cxx is None:
        pytest.skip("g++ not available")
    lib = build.build()
    out = str(tmp_path_factory.mktemp("cpp") / "score_check")
    libdir = os.path.dirname(lib)
    subprocess.check_call([cxx, "-std=c++17", "-O1", "-ffp-contract=off", "-Wall", "-Wextra", "-Werror",
                           os.path.join(ROOT, "tests", "cpp", "score_check.cpp"), "-I", os.path.join(ROOT, "include"),
                           "-L", libdir, "-lqwen3cuda", "-Wl,-rpath," + libdir, "-o", out])
    return out


def test_cpp_score_compiles(score_check):
    assert os.access(score_check, os.X_OK)


@pytest.mark.gpu
def test_cpp_score_matches_the_python_binding(score_check, ckpt):
    from qwen3_rs_b200 import transformer as T

    path = ckpt("small", 64, 3)
    toks = np.random.default_rng(4).integers(0, 4096, 81).tolist()
    r = subprocess.run([score_check, path, *map(str, [7, *toks[:80], "--", *toks[1:]])], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    lines = r.stdout.split("\n")
    lp_cpp = np.array([int(x, 16) for x in lines[0].split()], np.uint32)
    am_cpp = [int(x) for x in lines[1].split()]
    assert lines[2].strip() == "-1"  # Q3_EINVAL for an out-of-range target, thrown as qwen3::Error
    m = T.TransformerBuilder.new(path).build()
    try:
        lp, am = m.score(toks[:80], targets=toks[1:], pos0=7)
    finally:
        m.close()
    assert np.array_equal(lp_cpp, lp.view(np.uint32)) and am_cpp == am.tolist()
