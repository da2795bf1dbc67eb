"""Every decode weight stream against an int64 reference, bit for bit: exact-arithmetic GEMV probes across group sizes, K
tilings and row splits.

A GEMV here is y = sum_g fl(fl(float(dot_g) ws_g) xs_g) with dot_g an exact int32; the implementations differ only in the
order of the f32 sum.  When every term is a multiple of one power of two u and sum_g |term_g| < 2^24 u, every partial sum of
every order is exact, so every path returns the same bits, and those bits follow from an int64 numpy reference
(`exact_gemv`).  A wrong term, scale, chunk, K tile or row then changes the result instead of hiding in round-off.  The
probes (`export_gemv_probe`) are built so that every GEMV the decode step observes is such a sum:

  * probe activation x = c 2^(e_g - 2): integer codes c, one exponent e_g in {-1, 0, 1} per quantisation group, varying
    between groups.  Each group holds a +-127 and a code 64, each 32-element block two reserved zero codes; the free codes
    are fitted so that sum x^2 = 64 dim exactly (`probe_x`), with every partial sum exact.  The RMSNorm factor is then
    exactly 1/8 and (norm weights 1) quantize(rmsnorm(x)) gives the codes c and the scales 2^(e_g - 5) exactly.
  * observed rows ("dense"): codes in [-A, A] with a +-127 in every group, scale 2^-k_g, k_g random in {6, 7, 8} (the
    exporter reproduces them exactly); A is halved for a row until the row's exactness bound holds for every probe vector.
  * layer 0 observes o_proj: down_proj = 0, and at pos 0 attention returns v0 exactly.  The v rows are "selections": code 1
    at column pi(i), the scale-setting 127 and random codes at reserved zero columns, so v0_i = c_pi(i) 2^(-k_j + e - 5)
    with one k_j per output group j and pi mapping that group onto one group of x: v0 quantises exactly, and x_out =
    fl(x + o_proj(v0)) with o_proj(v0) exact.
  * layer 1 observes the gate/up pair stream, down_proj and the qkv tail: o_proj = 0; the gate rows hit the reserved 64
    codes of up to 32 groups, so gate = 32 exactly and silu(32) = 32 (glibc's expf and the device's); the up rows are
    selections, so h = 32 up quantises exactly; down rows are dense, x_out = fl(x + down(h)).  The v rows are dense: the V
    cache row is the raw v GEMV, exact.  The k rows are dense too: the K cache row (after QK-norm) is checked against
    float64 at 1e-6.
  * the lm_head rows are dense: forward_layers(x, 0, 0, 0, run_head=True) returns exact logits.
  * head probes (`HeadProbe`): every layer is a pass-through (o_proj = 0, down = 0), embedding rows are probe
    vectors, the untied lm_head carries planted ties -- two identical rows per token with its maximum logit, across a CTA
    boundary of the head split, across the two consumer groups of a stage, across a 32-row batch -- and the tied rows form a
    cycle of tokens, so greedy decoding stays on probe vectors.  One head probe has vocab < the SM count and only negative
    logits.

Regimes: the K tiling (`pick_n_kt`), the per-CTA row split (`cta_share`) and whether the persistent kernel takes a shape
(`mega_decline`) are mirrored here from q3_engine.cu / q3_mega.cuh; `test_matrix_hits_every_regime` keeps MATRIX on every
regime at the B200's 148 SMs, and the GPU test asserts that the persistent path is offered exactly when the mirror says so.
"""
from __future__ import annotations

import math
import os
from dataclasses import dataclass

import numpy as np
import pytest

from oracle import binding as orc
from qwen3_rs_b200 import transformer as T
from qwen3_rs_b200.export import EMBED_TOKENS_KEY, ExportConfig, export_from_loader, quantize_q80

HD = 128
N_LAYERS = 2
SEQ = 64
B200_SMS = 148
MEGA_MAX_KT, MEGA_GW, MEGA_BATCH = 4096, 8, 32   # q3_mega.cuh
MEGA_MAX_ACT = 16384                             # build_mega: activation vectors up to 16384
K_CHOICES = (6, 7, 8)                            # weight scales 2^-k of the observed rows
EXACT = 1 << 24
N_X = 2                                          # probe vectors per checkpoint
Q3_EUNSUPPORTED = -5
GS_ALL = (32, 64, 128)


@dataclass(frozen=True)
class Shape:
    dim: int
    hidden: int
    n_heads: int
    n_kv: int
    vocab: int
    gs: int

    @property
    def AH(self) -> int:
        return self.n_heads * HD

    @property
    def KV(self) -> int:
        return self.n_kv * HD

    @property
    def qkv_rows(self) -> int:
        return self.AH + 2 * self.KV

    def __str__(self):
        return f"d{self.dim}_h{self.hidden}_a{self.n_heads}kv{self.n_kv}_v{self.vocab}_gs{self.gs}"


# ---- mirrors of the persistent kernel's stream layout (q3_engine.cu pick_n_kt / build_mega, q3_mega.cuh cta_share) ----
def pick_n_kt(K: int, gs: int) -> int:
    for n in range(-(-K // MEGA_MAX_KT), 65):
        if K % (n * gs) == 0 and (K // n) % 16 == 0 and K // n <= MEGA_MAX_KT:
            return n
    return 0


def cta_share(units: int, nctas: int, c: int):
    base, rem = divmod(units, nctas)
    return c * base + min(c, rem), base + (1 if c < rem else 0)


def mega_decline(s: Shape, num_sms: int):
    """Why build_mega declines the shape, or None when the persistent kernel takes it."""
    if s.dim > MEGA_MAX_KT:
        return "dim > 4096"
    if not pick_n_kt(s.AH, s.gs) or not pick_n_kt(s.hidden, s.gs):
        return "no K tiling for o_proj/down"
    if max(s.AH, s.hidden, s.dim) > MEGA_MAX_ACT:
        return "activation vector > 16384"
    if s.qkv_rows < num_sms or s.hidden < num_sms:
        return "fewer qkv rows / FFN units than SMs"
    return None


def phases(s: Shape):
    """(phase, units, K): gate/up units are (gate, up) pairs."""
    return (("qkv", s.qkv_rows, s.dim), ("o", s.dim, s.AH), ("gu", s.hidden, s.dim), ("down", s.dim, s.hidden),
            ("head", s.vocab, s.dim))


def regimes(s: Shape, num_sms: int) -> dict:
    out = {}
    for ph, units, K in phases(s):
        n = pick_n_kt(K, s.gs)
        KT = K // n if n else 0
        G = KT // s.gs
        counts = [cta_share(units, num_sms, c)[1] for c in range(num_sms)]
        out[ph] = dict(n_kt=n, KT=KT, G=G, full=bool(n) and G % 32 == 0, padded=bool(n) and (4 * G) % 16 != 0,
                       rows_min=min(counts), rows_max=max(counts))
    return out


def regime_line(s: Shape, num_sms: int, paths) -> str:
    r = regimes(s, num_sms)
    cells = []
    for ph, v in r.items():
        t = f"{ph}: n_kt {v['n_kt']} G {v['G']}{' FULL' if v['full'] else ''}{' pad' if v['padded'] else ''}"
        cells.append(t + f" rows/CTA {v['rows_min']}-{v['rows_max']}")
    why = mega_decline(s, num_sms)
    return f"{s}: " + " | ".join(cells) + f" | paths {list(paths)}" + (f" (persistent declined: {why})" if why else "")


# ---- the probe matrix ---------------------------------------------------------------------------------------------------
MATRIX = (
    [Shape(256, 6144, 4, 2, 512, gs) for gs in GS_ALL]       # down n_kt 2 (G 96 FULL / 48 / 24); < 8 qkv and head rows per CTA
    + [Shape(256, 9728, 4, 2, 6000, gs) for gs in GS_ALL]    # Qwen3-4B down_proj: n_kt 4, G 76 / 38 / 19 (padded scale areas); > 32 head rows
    + [Shape(256, 12160, 4, 2, 100, gs) for gs in GS_ALL]    # n_kt 4 / 5 / 5; vocab < SMs: CTAs without head rows
    + [Shape(256, 14080, 4, 2, 512, 128)]                    # n_kt 5, G 22
    + [Shape(256, 16256, 4, 2, 512, gs) for gs in GS_ALL]    # gs 32: n_kt 4, G 127; gs 64 / 128: no K tiling (declined)
    + [Shape(512, 1536, 40, 5, 4736, gs) for gs in GS_ALL]   # o_proj K 5120: n_kt 2; exactly 32 head rows per CTA
    + [Shape(256, 512, 64, 8, 512, gs) for gs in (64, 128)]  # o_proj K 8192: n_kt 2, FULL blocks
    + [Shape(512, 768, 24, 6, 512, 64)]                      # 4608 qkv rows: 31 / 32 per CTA
    + [Shape(256, 13952, 4, 2, 512, 64)]                     # declined: no K tiling for down (K 13952)
    + [Shape(256, 128, 4, 2, 512, 64)]                       # declined: hidden < SMs
)
BENCH_SHAPE = Shape(4096, 12288, 32, 8, 6000, 64)            # the bench's tiling (Qwen3-8B): FULL blocks, down n_kt 3


def _pairs_not_mult8(r):
    return r["gu"]["rows_min"] % 8 != 0 or r["gu"]["rows_max"] % 8 != 0


REQUIRED_REGIMES = {
    **{f"down_proj with more than one K tile at gs {g}": (lambda g: lambda s, r: s.gs == g and r["down"]["n_kt"] > 1)(g)
       for g in GS_ALL},
    **{f"o_proj with more than one K tile at gs {g}": (lambda g: lambda s, r: s.gs == g and r["o"]["n_kt"] > 1)(g)
       for g in GS_ALL},
    "n_kt 2 at gs 64, G 48 (Qwen3-1.7B down_proj)": lambda s, r: s.gs == 64 and (r["down"]["n_kt"], r["down"]["G"]) == (2, 48),
    "padded scale area at gs 128, G 19": lambda s, r: s.gs == 128 and r["down"]["padded"] and r["down"]["G"] == 19,
    "padded scale area at gs 64": lambda s, r: s.gs == 64 and r["down"]["padded"] and r["down"]["n_kt"] > 1,
    "n_kt 5 at gs 64": lambda s, r: s.gs == 64 and r["down"]["n_kt"] == 5,
    "n_kt 5 at gs 128": lambda s, r: s.gs == 128 and r["down"]["n_kt"] == 5 and s.hidden == 12160,
    "n_kt 5 at gs 128, K 14080": lambda s, r: s.gs == 128 and r["down"]["n_kt"] == 5 and s.hidden == 14080,
    "G 127 (K 16256 gs 32)": lambda s, r: r["down"]["G"] == 127,
    "FULL blocks with more than one K tile": lambda s, r: r["down"]["full"] and r["down"]["n_kt"] > 1,
    "FULL o_proj blocks with two K tiles": lambda s, r: r["o"]["full"] and r["o"]["n_kt"] == 2,
    "the bench's tiling (dim 4096, hidden 12288, gs 64)": lambda s, r: (s.dim, s.hidden, s.gs) == (4096, 12288, 64)
    and r["qkv"]["full"] and r["down"]["full"] and r["down"]["n_kt"] == 3,
    "qkv: < 8 rows per CTA": lambda s, r: r["qkv"]["rows_max"] < 8,
    "qkv: 32 rows per CTA": lambda s, r: r["qkv"]["rows_min"] <= 32 <= r["qkv"]["rows_max"],
    "qkv: > 32 rows per CTA": lambda s, r: r["qkv"]["rows_min"] > 32,
    "head: CTAs with no rows (vocab < SMs)": lambda s, r: r["head"]["rows_min"] == 0,
    "head: < 8 rows per CTA": lambda s, r: 0 < r["head"]["rows_min"] and r["head"]["rows_max"] < 8,
    "head: exactly 32 rows per CTA": lambda s, r: r["head"]["rows_min"] == r["head"]["rows_max"] == 32,
    "head: > 32 rows per CTA": lambda s, r: r["head"]["rows_min"] > 32,
    "gate/up pair blocks not a multiple of 8": lambda s, r: _pairs_not_mult8(r),
}
REQUIRED_DECLINES = {
    "no K tiling for down_proj (K 13952 gs 64)": lambda s: s.hidden == 13952,
    "no K tiling for down_proj (K 16256 gs 64 / 128)": lambda s: s.hidden == 16256 and s.gs != 32,
    "hidden < SMs": lambda s: s.hidden < B200_SMS,
}


# ---- the generator ------------------------------------------------------------------------------------------------------
@dataclass
class Layout:
    """What every probe vector of one checkpoint shares: group exponents and the reserved columns."""
    dim: int
    gs: int
    e: np.ndarray       # [G] activation exponent of each group
    p127: np.ndarray    # [G] column of the group's +-127
    p64: np.ndarray     # [G] column of the group's 64
    zeros: np.ndarray   # [G, 2 gs / 32] reserved zero columns

    @property
    def G(self) -> int:
        return self.dim // self.gs

    @property
    def e_elem(self) -> np.ndarray:
        return np.repeat(self.e, self.gs)


def make_layout(rng, dim: int, gs: int) -> Layout:
    G = dim // gs
    e = np.resize(np.array([-1, 0, 1, -1, 0, -1]), G)
    e[1:] = rng.permutation(e[1:])
    p127, p64, zeros = np.empty(G, np.int64), np.empty(G, np.int64), []
    for g in range(G):
        perm = g * gs + rng.permutation(gs)
        p127[g], p64[g] = perm[0], perm[1]
        z = []
        for b in range(gs // 32):
            cols = [c for c in g * gs + 32 * b + rng.permutation(32) if c not in (p127[g], p64[g])]
            z += cols[:2]
        zeros.append(z)
    lay = Layout(dim, gs, e, p127, p64, np.array(zeros, np.int64))
    assert len(np.unique(np.concatenate([p127, p64, lay.zeros.ravel()]))) == 2 * G + lay.zeros.size
    return lay


def four_squares(D: int):
    """a^2 + b^2 + c^2 + d^2 = D with every term <= 126^2."""
    for a in range(min(126, math.isqrt(D)), -1, -1):
        r = D - a * a
        if r > 3 * 126 * 126:
            break
        for b in range(min(126, math.isqrt(r)), -1, -1):
            r2 = r - b * b
            if r2 > 2 * 126 * 126:
                break
            for c in range(min(126, math.isqrt(r2)), -1, -1):
                r3 = r2 - c * c
                if r3 > 126 * 126:
                    break
                d = math.isqrt(r3)
                if d * d == r3:
                    return a, b, c, d
    raise AssertionError(f"no four squares <= 126^2 sum to {D}")


def probe_x(rng, lay: Layout, nonneg: bool = False, sparse: float = 0.0):
    """-> (codes c [dim] int64, x = c 2^(e - 2) [dim] f32) with sum x^2 = 64 dim exactly."""
    dim, G = lay.dim, lay.G
    w = 4 ** (lay.e_elem + 1)                   # x^2 in units of 2^-6: c^2 4^(e + 1)
    U = 4096 * dim                              # = 64 dim / 2^-6
    c = np.zeros(dim, np.int64)
    c[lay.p127] = 127 if nonneg else 127 * rng.choice([-1, 1], G)
    c[lay.p64] = 64
    reserved = np.zeros(dim, bool)
    reserved[lay.p127] = reserved[lay.p64] = True
    reserved[lay.zeros.ravel()] = True
    free = np.flatnonzero(~reserved)
    f0 = rng.uniform(-1.0, 1.0, free.size)
    if nonneg:
        f0 = np.abs(f0)
    if sparse:
        f0[rng.random(free.size) < sparse] = 0.0
    fix = rng.choice(free[(lay.e_elem[free] == -1) & (f0 != 0)], 4, replace=False)  # the last four squares go here
    f0[np.searchsorted(free, fix)] = 0.0
    B = U - int((c * c * w).sum())
    fw = w[free]
    assert B > 0, "reserved codes alone exceed the mean square: rebalance the exponents"
    s = math.sqrt((B - 30000) / float((f0 * f0 * fw).sum()))
    for _ in range(100):
        f = np.clip(np.rint(s * f0), -126, 126).astype(np.int64)
        D = B - int((f * f * fw).sum())
        if 0 <= D <= 4 * 126 * 126 - 1000:
            break
        s *= math.sqrt((B - 30000) / max(float((f * f * fw).sum()), 1.0))
    else:
        raise AssertionError("could not fit the probe vector's mean square")
    c[free] = f
    sq = np.array(four_squares(D), np.int64)
    c[fix] = sq * (1 if nonneg else rng.choice([-1, 1], 4))
    assert int((c * c * w).sum()) == U
    assert np.abs(c).max() <= 127 and (c[lay.zeros.ravel()] == 0).all() and (np.abs(c[lay.p127]) == 127).all()
    assert all((np.abs(c[g * lay.gs:(g + 1) * lay.gs]) <= 126).sum() == lay.gs - 1 for g in range(G))
    return c, np.ldexp(c.astype(np.float32), (lay.e_elem - 2).astype(np.int32)).astype(np.float32)


def exact_gemv(codes: np.ndarray, kexp: np.ndarray, acodes: np.ndarray, aexp: np.ndarray, gs: int, chunk: int = 1024):
    """sum_g dot_g 2^(aexp_g - kexp_rg) per row -> (y f32 [rows], bound [rows]): y is exact when bound < 2^24 (units of the
    row's smallest term exponent, so every partial sum of every order is an exact f32)."""
    rows, K = codes.shape
    G = K // gs
    a = acodes.astype(np.int32).reshape(G, gs)
    y = np.empty(rows, np.float32)
    bound = np.empty(rows, np.int64)
    for r0 in range(0, rows, chunk):
        d = (codes[r0:r0 + chunk].astype(np.int32).reshape(-1, G, gs) * a).sum(-1, dtype=np.int64)
        y[r0:r0 + chunk], bound[r0:r0 + chunk] = units_to_f32(d, aexp[None, :] - kexp[r0:r0 + chunk].astype(np.int64))
    return y, bound


def units_to_f32(d: np.ndarray, t: np.ndarray):
    tmin = t.min(axis=1, keepdims=True)
    sh = t - tmin
    units = (d << sh).sum(axis=1)
    bound = (np.abs(d) << sh).sum(axis=1)
    return np.ldexp(units.astype(np.float64), tmin[:, 0].astype(np.int32)).astype(np.float32), bound


def group_dots(codes, acodes, gs):
    G = codes.shape[1] // gs
    return (codes.astype(np.int32).reshape(-1, G, gs) * acodes.astype(np.int32).reshape(G, gs)).sum(-1, dtype=np.int64)


def _pm127(rng, codes: np.ndarray, gs: int, sign=None):
    rows, K = codes.shape
    G = K // gs
    pos = np.arange(G) * gs + rng.integers(0, gs, (rows, G))
    sgn = rng.choice([-1, 1], (rows, G)) if sign is None else sign
    codes[np.arange(rows)[:, None], pos] = 127 * sgn


def dense_rows(rng, rows: int, K: int, gs: int, acts=(), lo: int = -126, hi: int = 126, sign=None):
    """Codes in [lo, hi] (scaled down per row until exact for every activation in acts) with a +-127 in every group,
    scales 2^-k, k in K_CHOICES."""
    G = K // gs
    codes = rng.integers(lo, hi + 1, (rows, K)).astype(np.int8)
    _pm127(rng, codes, gs, sign)
    kexp = rng.choice(K_CHOICES, (rows, G)).astype(np.int64)
    for _ in range(8):
        bad = np.zeros(rows, bool)
        for ac, ae in acts:
            bad |= exact_gemv(codes, kexp, ac, ae, gs)[1] >= EXACT
        if not bad.any():
            return codes, kexp
        idx = np.flatnonzero(bad)
        lo, hi = lo // 2, (hi + 1) // 2
        sub = rng.integers(lo, hi + 1, (idx.size, K)).astype(np.int8)
        _pm127(rng, sub, gs, None if sign is None else sign[:idx.size])
        codes[idx] = sub
    raise AssertionError("could not draw exact rows")


def zero_col_noise(rng, lay: Layout, rows: int):
    """Rows that are zero except at the reserved zero columns of x (a +-127 and random codes there): they add exactly 0
    against every probe vector, unless a kernel pairs them with the wrong activation chunk."""
    codes = np.zeros((rows, lay.dim), np.int8)
    Z = lay.zeros
    codes[:, Z.ravel()] = rng.integers(-126, 127, (rows, Z.size))
    codes[:, Z[:, 0]] = 127 * rng.choice([-1, 1], (rows, lay.G))
    return codes, rng.choice(K_CHOICES, (rows, lay.G)).astype(np.int64)


def selection_rows(rng, lay: Layout, n_out: int):
    """Row i: code 1 at column pi(i), pi mapping output group j onto x group sigma_j, weight scale 2^-k_j there ->
    (codes, kexp, pi [n_out], out_exp [n_out / gs]): output i is c[pi(i)] 2^(out_exp_j) exactly, out_exp_j = -k_j + e - 5."""
    gs = lay.gs
    Gout = n_out // gs
    sigma = rng.integers(0, lay.G, Gout)
    kout = rng.choice(K_CHOICES, Gout)
    pi = np.concatenate([sg * gs + rng.permutation(gs) for sg in sigma])
    codes, kexp = zero_col_noise(rng, lay, n_out)
    r = np.arange(n_out)
    sg = sigma[r // gs]
    z0, z1 = lay.zeros[sg, 0], lay.zeros[sg, 1]
    z = np.where(z0 == pi, z1, z0)
    codes[r, z] = 127 * rng.choice([-1, 1], n_out)
    codes[r, pi] = 1
    kexp[r, sg] = kout[r // gs]
    return codes, kexp, pi, -kout + lay.e[sigma] - 5


def gate_rows(rng, lay: Layout, rows: int):
    """Code 1 at the 64 column of n_hit groups per row, weight scale 2^(4 - log2 n_hit - e) there, so that each hit adds
    64 2^(4 - log2 n_hit - e) 2^(e - 5) = 32 / n_hit: gate = 32 exactly."""
    n_hit = 1 << int(math.log2(min(32, lay.G)))
    codes, kexp = zero_col_noise(rng, lay, rows)
    hits = np.argsort(rng.random((rows, lay.G)), axis=1)[:, :n_hit]
    r = np.arange(rows)[:, None]
    codes[r, lay.p64[hits]] = 1
    kexp[r, hits] = lay.e[hits] - 4 + int(math.log2(n_hit))
    return codes, kexp


def to_float(codes: np.ndarray, kexp: np.ndarray, gs: int) -> np.ndarray:
    rows, K = codes.shape
    return np.ldexp(codes.astype(np.float32).reshape(rows, K // gs, gs), -kexp[:, :, None].astype(np.int32)).reshape(rows, K).astype(np.float32)


def _export(s: Shape, n_layers: int, path: str, tensors: dict, embed: np.ndarray):
    """Writes the checkpoint; every quantised tensor must come back with exactly the intended codes and scales."""
    cfg = ExportConfig(s.dim, s.hidden, n_layers, s.n_heads, s.n_kv, s.vocab, SEQ, HD)
    current = {}

    def load(name: str):
        if name.endswith("layernorm.weight") or name == "model.norm.weight":
            return np.ones(s.dim, np.float32)
        if name.endswith("q_norm.weight") or name.endswith("k_norm.weight"):
            return np.ones(HD, np.float32)
        if name == EMBED_TOKENS_KEY:
            current["want"] = None
            return embed
        key = name.rsplit(".", 1)[0]
        t = tensors[key]
        current["want"] = t
        if isinstance(t, tuple) and len(t) == 2 and isinstance(t[0], int):
            return np.zeros(t, np.float32)
        return to_float(t[0], t[1], s.gs)

    def checked(w, gs):
        q, sc, err = quantize_q80(w, gs)
        t = current["want"]
        if t is not None and not isinstance(t[0], int):
            assert np.array_equal(q, t[0].reshape(-1)), "exporter changed the codes"
            assert np.array_equal(sc, np.ldexp(np.float32(1), -t[1]).astype(np.float32).reshape(-1)), "exporter changed the scales"
        return q, sc, err

    info = export_from_loader(load, cfg, path, s.gs, shared_classifier=False, quantizer=checked)
    assert info["group_size"] == s.gs


class GemvProbe:
    """A probe checkpoint with its probe vectors and int64 references (see the module docstring)."""

    def __init__(self, s: Shape, path: str, seed: int = 0):
        self.s, self.path = s, path
        rng = np.random.default_rng(seed * 7919 + s.dim * 31 + s.hidden * 7 + s.gs + s.n_heads)
        lay = self.lay = make_layout(rng, s.dim, s.gs)
        gs = s.gs
        self.xs = [probe_x(rng, lay) for _ in range(N_X)]
        xacts = [(c, lay.e - 5) for c, _ in self.xs]          # quantize(rmsnorm(x)): codes c, scales 2^(e - 5)
        # layer 0: o_proj observed through v0 = selections of x
        vsel = selection_rows(rng, lay, s.KV)
        self.v0_pi, self.v0_exp = vsel[2], vsel[3]
        att = [self.att_codes(c) for c, _ in self.xs]
        o0 = dense_rows(rng, s.dim, s.AH, gs, att)
        # layer 1: gate = 32, up selections, down observed; v / k rows observed raw
        usel = selection_rows(rng, lay, s.hidden)
        self.up_pi, self.up_exp = usel[2], usel[3]
        hact = [self.h_codes(c) for c, _ in self.xs]
        dn1 = dense_rows(rng, s.dim, s.hidden, gs, hact)
        v1 = dense_rows(rng, s.KV, s.dim, gs, xacts)
        k1 = dense_rows(rng, s.KV, s.dim, gs, xacts)
        head = dense_rows(rng, s.vocab, s.dim, gs, xacts)
        free = lambda rows, K: dense_rows(rng, rows, K, gs)   # noqa: E731 -- rows no test observes exactly
        self.tensors = {
            "model.layers.0.self_attn.q_proj": free(s.AH, s.dim), "model.layers.0.self_attn.k_proj": free(s.KV, s.dim),
            "model.layers.0.self_attn.v_proj": vsel[:2], "model.layers.0.self_attn.o_proj": o0,
            "model.layers.0.mlp.gate_proj": free(s.hidden, s.dim), "model.layers.0.mlp.up_proj": free(s.hidden, s.dim),
            "model.layers.0.mlp.down_proj": (s.dim, s.hidden),
            "model.layers.1.self_attn.q_proj": free(s.AH, s.dim), "model.layers.1.self_attn.k_proj": k1,
            "model.layers.1.self_attn.v_proj": v1, "model.layers.1.self_attn.o_proj": (s.dim, s.AH),
            "model.layers.1.mlp.gate_proj": gate_rows(rng, lay, s.hidden), "model.layers.1.mlp.up_proj": usel[:2],
            "model.layers.1.mlp.down_proj": dn1, "lm_head": head,
        }
        self.want = [self.reference(c, x) for c, x in self.xs]

    def att_codes(self, c):
        """o_proj input: v0 = c[pi] 2^v0_exp, repeated for every query head of a kv head."""
        s = self.s
        v0 = c[self.v0_pi].reshape(s.n_kv, HD)
        codes = np.repeat(v0, s.n_heads // s.n_kv, axis=0).reshape(-1)
        e = np.repeat(self.v0_exp.reshape(s.n_kv, HD // s.gs), s.n_heads // s.n_kv, axis=0).reshape(-1)
        return codes, e

    def h_codes(self, c):
        """down_proj input: h = 32 up = c[pi] 2^(up_exp + 5)."""
        return c[self.up_pi], self.up_exp + 5

    def reference(self, c, x) -> dict:
        s, gs, t = self.s, self.s.gs, self.tensors
        xa = (c, self.lay.e - 5)
        ac, ae = self.att_codes(c)
        hc, he = self.h_codes(c)
        y_o, b_o = exact_gemv(*t["model.layers.0.self_attn.o_proj"], ac, ae, gs)
        y_d, b_d = exact_gemv(*t["model.layers.1.mlp.down_proj"], hc, he, gs)
        v1, b_v = exact_gemv(*t["model.layers.1.self_attn.v_proj"], *xa, gs)
        k1, b_k = exact_gemv(*t["model.layers.1.self_attn.k_proj"], *xa, gs)
        lg, b_h = exact_gemv(*t["lm_head"], *xa, gs)
        v0, b_v0 = exact_gemv(*t["model.layers.0.self_attn.v_proj"][:2], *xa, gs)
        up, b_u = exact_gemv(*t["model.layers.1.mlp.up_proj"][:2], *xa, gs)
        gate, b_g = exact_gemv(*t["model.layers.1.mlp.gate_proj"], *xa, gs)
        for b in (b_o, b_d, b_v, b_k, b_h, b_v0, b_u, b_g):
            assert (b < EXACT).all()
        assert (gate == 32.0).all()
        assert np.array_equal(v0, np.ldexp(c[self.v0_pi].astype(np.float32), np.repeat(self.v0_exp, gs)))
        assert np.array_equal(np.float32(32.0) * up, np.ldexp(hc.astype(np.float32), np.repeat(he, gs)))
        return dict(x0=(x + y_o).astype(np.float32), v0=v0, x1=(x + y_d).astype(np.float32), v1=v1, k1_raw=k1, logits=lg,
                    y_o=y_o, y_d=y_d)

    def export(self):
        _export(self.s, N_LAYERS, self.path, self.tensors, np.zeros((self.s.vocab, self.s.dim), np.float32))
        return self


def export_gemv_probe(s: Shape, path: str, seed: int = 0) -> GemvProbe:
    return GemvProbe(s, path, seed).export()


# ---- head probes --------------------------------------------------------------------------------------------------------
HEAD_SHAPE = (256, 256, 4, 2, 64)   # dim, hidden, n_heads, n_kv, gs


def head_pairs(vocab: int, num_sms: int):
    """Planted (r1, r2) ties: across CTA boundaries of the head split, across the two consumer groups of a stage (rows 7 / 8
    of a CTA's share), across a 32-row batch (rows 31 / 32), and (small vocabularies) wherever rows are free."""
    if vocab < num_sms:
        return [(0, 1), (11, 12), (30, 57), (63, 64), (72, 73), (85, 98), (96, 97), (90, 99)]
    st = [cta_share(vocab, num_sms, c)[0] for c in range(num_sms)]
    n = num_sms
    pairs = [(st[c] - 1, st[c]) for c in (1, n // 4, n // 2, n - 1)]
    pairs += [(st[c] + MEGA_GW - 1, st[c] + MEGA_GW) for c in (3, n // 3)]
    pairs += [(st[c] + MEGA_BATCH - 1, st[c] + MEGA_BATCH) for c in (5, 2 * n // 3)]
    return pairs


class HeadProbe:
    """Pass-through layers, probe-vector embeddings and planted ties in an untied lm_head (module docstring)."""

    def __init__(self, vocab: int, num_sms: int, path: str, negative: bool, seed: int = 0):
        dim, hidden, nh, nkv, gs = HEAD_SHAPE
        s = self.s = Shape(dim, hidden, nh, nkv, vocab, gs)
        self.path, self.negative = path, negative
        rng = np.random.default_rng(seed + vocab)
        lay = make_layout(rng, dim, gs)
        self.pairs = head_pairs(vocab, num_sms)
        rows = np.array(self.pairs).ravel()
        assert len(set(rows.tolist())) == rows.size and rows.min() >= 0 and rows.max() < vocab
        N = len(self.pairs)
        self.tokens = [self.pairs[i - 1][1] for i in range(N)]       # token i's maximum is at pairs[i]: the next token
        xs = [probe_x(rng, lay, nonneg=negative, sparse=0.3 if negative else 0.0) for _ in range(N)]
        xacts = [(c, lay.e - 5) for c, _ in xs]
        embed = np.zeros((vocab, dim), np.float32)
        for tok, (_, x) in zip(self.tokens, xs):
            embed[tok] = x
        if negative:  # non-positive rows against non-negative codes: every logit < 0
            head = dense_rows(rng, vocab, dim, gs, xacts, lo=-126, hi=0, sign=-np.ones((vocab, dim // gs), np.int64))
        else:
            head = dense_rows(rng, vocab, dim, gs, xacts)
        hc, hk = head
        for i, (c, _) in enumerate(xs):
            row = np.zeros(dim, np.int8)
            if negative:  # -126 where this vector is 0, -1 at one 64: small negative for it, far below for the others
                row[c == 0] = -126
                row[lay.zeros[:, 0]] = -127
                row[lay.p64[0]] = -1
            else:         # sign-matched: far above every dense row
                row[:] = np.sign(c) * 100
                row[lay.p127] = np.sign(c[lay.p127]) * 127
            for r in self.pairs[i]:
                hc[r], hk[r] = row, 8
        self.v_rows = [dense_rows(rng, s.KV, dim, gs, xacts) for _ in range(N_LAYERS)]
        free = lambda r, K: dense_rows(rng, r, K, gs)  # noqa: E731
        self.tensors = {"lm_head": (hc, hk)}
        for l in range(N_LAYERS):
            self.tensors.update({
                f"model.layers.{l}.self_attn.q_proj": free(s.AH, dim), f"model.layers.{l}.self_attn.k_proj": free(s.KV, dim),
                f"model.layers.{l}.self_attn.v_proj": self.v_rows[l], f"model.layers.{l}.self_attn.o_proj": (dim, s.AH),
                f"model.layers.{l}.mlp.gate_proj": free(hidden, dim), f"model.layers.{l}.mlp.up_proj": free(hidden, dim),
                f"model.layers.{l}.mlp.down_proj": (dim, hidden)})
        self.logits, self.v = {}, {}
        for i, (tok, (c, _)) in enumerate(zip(self.tokens, xs)):
            lg, b = exact_gemv(hc, hk, c, lay.e - 5, gs)
            assert (b < EXACT).all()
            top = np.flatnonzero(lg == lg.max())
            assert top.tolist() == sorted(self.pairs[i]), f"token {tok}: maximum at {top}, planted at {self.pairs[i]}"
            assert (lg < 0).all() if negative else lg.max() > 0
            self.logits[tok] = lg
            self.v[tok] = [exact_gemv(*self.v_rows[l], c, lay.e - 5, gs)[0] for l in range(N_LAYERS)]
        _export(s, N_LAYERS, path, self.tensors, embed)

    def next_token(self, tok: int) -> int:
        lg = self.logits[tok]
        return int(np.flatnonzero(lg == lg.max())[-1])


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def assert_bits(got, want, label):
    bad = np.flatnonzero(bits(got) != bits(want))
    assert bad.size == 0, (f"{label}: {bad.size} of {np.size(want)} outputs differ from the exact reference, first at "
                           f"{bad[:8].tolist()}: got {np.asarray(got).reshape(-1)[bad[:4]]}, want {np.asarray(want).reshape(-1)[bad[:4]]}")


def k_post64(k_raw: np.ndarray) -> np.ndarray:
    """QK-norm (weights 1) in float64; RoPE at pos 0 is the identity."""
    k = k_raw.astype(np.float64).reshape(-1, HD)
    return (k / np.sqrt((k * k).mean(axis=1, keepdims=True) + 1e-6)).reshape(-1)


# ---- fixtures -----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def gemv_probe(tmp_path_factory):
    d = tmp_path_factory.mktemp("gemv")
    cache = {}

    def get(s: Shape) -> GemvProbe:
        if s not in cache:
            for old in cache.values():  # one checkpoint at a time: the bench-sized one is ~0.4 GB
                os.remove(old.path)
            cache.clear()
            cache[s] = export_gemv_probe(s, str(d / f"{s}.bin"))
        return cache[s]

    return get


def _decode_path_offered(m) -> bool:
    try:
        m.set_decode_path(1)
        return True
    except T.Q3Error as e:
        assert e.code == Q3_EUNSUPPORTED, e
        return False


def check_probe_on_device(P: GemvProbe, m, label: str):
    for i, ((c, x), w) in enumerate(zip(P.xs, P.want)):
        lab = f"{label} x{i}"
        xo = m.forward_layers(x, 0, 0, 1)
        _, v = m.kv_read(0, 0, 1)
        assert_bits(v[0], w["v0"], f"{lab} layer 0 v row (selections)")
        assert_bits(xo, w["x0"], f"{lab} layer 0 x + o_proj(v0)")
        xo = m.forward_layers(x, 0, 1, 2)
        k, v = m.kv_read(1, 0, 1)
        assert_bits(v[0], w["v1"], f"{lab} layer 1 v row")
        assert_bits(xo, w["x1"], f"{lab} layer 1 x + down(32 up)")
        k64 = k_post64(w["k1_raw"])
        err = np.abs(k[0].astype(np.float64) - k64).reshape(-1, HD).max(axis=1) / np.abs(k64).reshape(-1, HD).max(axis=1)
        assert err.max() <= 1e-6, f"{lab} layer 1 k row after QK-norm off float64 by {err.max():.2e} (relative)"
        _, lg = m.forward_layers(x, 0, 0, 0, run_head=True)
        assert_bits(lg, w["logits"], f"{lab} lm_head")


# ---- on the GPU ---------------------------------------------------------------------------------------------------------
def _run_gpu(P: GemvProbe):
    s = P.s
    m = T.TransformerBuilder.new(P.path).build()
    try:
        ns = m.num_sms
        why = mega_decline(s, ns)
        check_probe_on_device(P, m, f"{s} default path")
        offered = _decode_path_offered(m)
        assert offered == (why is None), f"{s}: persistent kernel offered {offered}, the mirror predicts {why or 'offered'}"
        paths = (0, 1) if offered else (0,)
        for path in paths:
            m.set_decode_path(path)
            check_probe_on_device(P, m, f"{s} path {path}")
        print(regime_line(s, ns, paths))
    finally:
        m.close()


@pytest.mark.gpu
@pytest.mark.parametrize("s", MATRIX, ids=str)
def test_decode_gemv_bit_exact(gemv_probe, s):
    """Every observed GEMV output (o_proj, down_proj via the gate/up pairs, the qkv tail, lm_head) bit-identical to the
    int64 reference on every decode path the handle offers; the persistent path offered exactly when the mirror says."""
    _run_gpu(gemv_probe(s))


@pytest.mark.gpu
@pytest.mark.slow
def test_decode_gemv_bit_exact_bench_tiling(gemv_probe):
    """The same at the bench's tiling: dim 4096, hidden 12288, 32 / 8 heads, gs 64 (FULL blocks, down_proj n_kt 3)."""
    _run_gpu(gemv_probe(BENCH_SHAPE))


def _sms() -> int:
    import torch

    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.mark.gpu
@pytest.mark.parametrize("negative", [False, True], ids=["ties", "negative_small_vocab"])
def test_head_argmax_and_multi_token_paths_bit_exact(tmp_path, negative):
    """Planted ties: forward / forward_argmax / decode_greedy on both paths, forward_multi n = 1..8, prefill and score all
    give the exact logits and V rows and the last maximum.  negative: vocab < SM count and every logit < 0."""
    ns = _sms()
    vocab = 100 if negative else 40 * ns
    H = HeadProbe(vocab, ns, str(tmp_path / "head.bin"), negative)
    assert not negative or vocab < ns
    m = T.TransformerBuilder.new(H.path).build()
    try:
        assert m.num_sms == ns
        assert mega_decline(H.s, ns) is None and _decode_path_offered(m), "the head probes are persistent-kernel shapes"
        toks, N = H.tokens, len(H.tokens)
        nxt = [H.next_token(t) for t in toks]
        assert nxt == toks[1:] + toks[:1]
        for path in (0, 1):
            m.set_decode_path(path)
            for i, t in enumerate(toks):
                assert_bits(m.forward(t, i), H.logits[t], f"path {path} forward({t})")
                for l in range(N_LAYERS):
                    assert_bits(m.kv_read(l, i, 1)[1][0], H.v[t][l], f"path {path} layer {l} v row of token {t}")
                got = m.forward_argmax(t, i)
                assert got == nxt[i], f"path {path} forward_argmax({t}) = {got}, planted last maximum {nxt[i]} (tie {H.pairs[i]})"
            got = m.decode_greedy(toks[0], 0, N)
            assert got == nxt, f"path {path} decode_greedy: {got}, want {nxt}"
            for n in range(1, 9):
                am, lg = m.forward_multi(toks[:n], 0, want_logits=True)
                assert am.tolist() == nxt[:n], f"path {path} forward_multi n {n}: argmax {am.tolist()}, want {nxt[:n]}"
                for j in range(n):
                    assert_bits(lg[j], H.logits[toks[j]], f"path {path} forward_multi n {n} token {j} logits")
                for l in range(N_LAYERS):
                    v = m.kv_read(l, 0, n)[1]
                    for j in range(n):
                        assert_bits(v[j], H.v[toks[j]][l], f"path {path} forward_multi n {n} layer {l} v row {j}")
        seq = (toks * 3)[:2 * N + 3]
        lg = m.prefill(seq, 0)  # dims are multiples of 128 with even group counts: the batched path must take this shape
        assert_bits(lg, H.logits[seq[-1]], "prefill last logits")
        for l in range(N_LAYERS):
            v = m.kv_read(l, 0, len(seq))[1]
            for j, t in enumerate(seq):
                assert_bits(v[j], H.v[t][l], f"prefill layer {l} v row {j}")
        _, am = m.score(seq)
        want = [H.next_token(t) for t in seq]
        assert am.tolist() == want, f"score argmax {am.tolist()}, want {want}"
        print(f"head probe vocab {vocab} ({ns} SMs): ties at {H.pairs}, head rows per CTA "
              f"{regimes(H.s, ns)['head']['rows_min']}-{regimes(H.s, ns)['head']['rows_max']}")
    finally:
        m.close()


# ---- without a GPU ------------------------------------------------------------------------------------------------------
def test_matrix_hits_every_regime():
    """MATRIX (with the bench-tiling case) reaches every regime at the B200's 148 SMs, and declines where it should."""
    allp = MATRIX + [BENCH_SHAPE]
    for name, pred in REQUIRED_REGIMES.items():
        hit = [s for s in allp if mega_decline(s, B200_SMS) is None and pred(s, regimes(s, B200_SMS))]
        assert hit, f"no probe hits: {name}"
    for name, pred in REQUIRED_DECLINES.items():
        hit = [s for s in allp if pred(s)]
        assert hit and all(mega_decline(s, B200_SMS) for s in hit), f"declined regime not covered: {name}"
    for s in allp:
        print(regime_line(s, B200_SMS, (0, 1) if mega_decline(s, B200_SMS) is None else (0,)))


def test_pick_n_kt_examples():
    """The tilings the matrix is built around (from the engine's rule)."""
    assert (pick_n_kt(6144, 64), 6144 // 2 // 64) == (2, 48)
    assert (pick_n_kt(9728, 128), 9728 // 4 // 128) == (4, 19)
    assert pick_n_kt(12160, 64) == pick_n_kt(12160, 128) == pick_n_kt(14080, 128) == 5
    assert (pick_n_kt(16256, 32), 16256 // 4 // 32) == (4, 127)
    assert pick_n_kt(13952, 64) == pick_n_kt(16256, 64) == pick_n_kt(16256, 128) == 0
    assert pick_n_kt(12288, 64) == 3 and pick_n_kt(4096, 64) == 1


HOST_SHAPES = [Shape(256, 6144, 4, 2, 512, 32), Shape(512, 1536, 8, 4, 512, 64), Shape(256, 512, 4, 2, 512, 128)]


@pytest.fixture(scope="module")
def host_probes(tmp_path_factory):
    d = tmp_path_factory.mktemp("gemv_host")
    return {s: export_gemv_probe(s, str(d / f"{s}.bin"), seed=3) for s in HOST_SHAPES}


@pytest.mark.parametrize("s", HOST_SHAPES, ids=str)
def test_oracle_reproduces_reference(host_probes, s):
    """The CPU oracle (the reference semantics) gives the int64 reference bit for bit in every role."""
    P = host_probes[s]
    o = orc.Model(P.path)
    try:
        for i, ((c, x), w) in enumerate(zip(P.xs, P.want)):
            assert_bits(o.forward_layers(x, 0, 0, 1), w["x0"], f"oracle x{i} layer 0")
            assert_bits(o.forward_layers(x, 0, 1, 2), w["x1"], f"oracle x{i} layer 1")
            kc, vc = o.kv_cache()
            assert_bits(vc[0, 0].reshape(-1), w["v0"], f"oracle x{i} layer 0 v row")
            assert_bits(vc[1, 0].reshape(-1), w["v1"], f"oracle x{i} layer 1 v row")
            assert np.abs(kc[1, 0].reshape(-1) - k_post64(w["k1_raw"])).max() <= 1e-6 * 4
            _, lg = o.forward_layers(x, 0, 0, 0, run_head=True)
            assert_bits(lg, w["logits"], f"oracle x{i} lm_head")
    finally:
        o.close()


def _fold_shuffled(terms: np.ndarray, rng) -> np.ndarray:
    """Left fold in f32 of each row's terms in a random order of its own."""
    perm = np.argsort(rng.random(terms.shape), axis=1)
    t = np.take_along_axis(terms, perm, axis=1)
    acc = np.zeros(terms.shape[0], np.float32)
    for g in range(t.shape[1]):
        acc = (acc + t[:, g]).astype(np.float32)
    return acc


def _terms(codes, kexp, acodes, aexp, gs):
    d = group_dots(codes, acodes, gs).astype(np.float32)
    return ((d * np.ldexp(np.float32(1), -kexp).astype(np.float32)).astype(np.float32)
            * np.ldexp(np.float32(1), aexp).astype(np.float32)[None, :]).astype(np.float32)


@pytest.mark.parametrize("s", HOST_SHAPES, ids=str)
def test_generator_claims_hold_in_float32(host_probes, s):
    """In float32 numpy: sum x^2 = 64 dim in any order, the RMSNorm factor is 1/8, quantize gives the codes and 2^(e - 5);
    gate = 32 and silu(32) = 32 with glibc's expf; every observed GEMV summed in shuffled orders equals the reference."""
    P, rng = host_probes[s], np.random.default_rng(17)
    lay, gs, t = P.lay, s.gs, P.tensors
    for (c, x), w in zip(P.xs, P.want):
        for _ in range(3):
            ss = np.float32(0)
            for v in x[rng.permutation(s.dim)]:
                ss = np.float32(ss + v * v)
            assert ss == np.float32(64 * s.dim)
            f = np.float32(1) / np.sqrt(np.float32(ss / np.float32(s.dim)) + np.float32(1e-6))
            assert f == np.float32(0.125)
        xn = (x * np.float32(0.125)).astype(np.float32)
        q, sc = orc.quantize(xn, gs)
        assert np.array_equal(q.astype(np.int64), c)
        assert np.array_equal(sc, np.ldexp(np.float32(1), lay.e - 5).astype(np.float32))
        g = np.float32(32)
        assert np.float32(g * (np.float32(1) / (np.float32(1) + orc.expf(np.array([-g], np.float32))[0]))) == g
        xa = (c, lay.e - 5)
        cases = [("o_proj", t["model.layers.0.self_attn.o_proj"], P.att_codes(c), w["y_o"]),
                 ("down", t["model.layers.1.mlp.down_proj"], P.h_codes(c), w["y_d"]),
                 ("v", t["model.layers.1.self_attn.v_proj"], xa, w["v1"]),
                 ("lm_head", t["lm_head"], xa, w["logits"]),
                 ("gate", t["model.layers.1.mlp.gate_proj"], xa, np.full(s.hidden, 32, np.float32))]
        for name, (codes, kexp), (ac, ae), want in cases:
            terms = _terms(codes, kexp, ac, ae, gs)
            for _ in range(2):
                assert_bits(_fold_shuffled(terms, rng), want, f"{name} in a shuffled f32 order")
        vsel = t["model.layers.0.self_attn.v_proj"][:2]
        assert_bits(_fold_shuffled(_terms(*vsel, *xa, gs), rng), w["v0"], "v selections")


def test_criterion_sees_single_faults(host_probes):
    """In the reference: dropping one group term, taking the neighbouring group's weight or activation scale, or swapping
    two K tiles' activations changes >= 99 % of the observed outputs (x_out of o_proj / down_proj, the logits)."""
    s = HOST_SHAPES[0]
    P = host_probes[s]
    gs, t = s.gs, P.tensors
    n_kt = pick_n_kt(s.hidden, gs)
    assert n_kt >= 2
    c, x = P.xs[0]
    w = P.want[0]
    cases = [("o_proj", t["model.layers.0.self_attn.o_proj"], P.att_codes(c), x, w["x0"]),
             ("down", t["model.layers.1.mlp.down_proj"], P.h_codes(c), x, w["x1"]),
             ("lm_head", t["lm_head"], (c, P.lay.e - 5), None, w["logits"])]
    report = []
    for name, (codes, kexp), (ac, ae), xres, want in cases:
        G = codes.shape[1] // gs

        def out(d, te):
            y, _ = units_to_f32(d, te)
            return y if xres is None else (xres + y).astype(np.float32)

        d = group_dots(codes, ac, gs)
        te = ae[None, :] - kexp
        assert_bits(out(d, te), want, name)
        faults = {}
        for g in (0, G // 2, G - 1):
            dd = d.copy()
            dd[:, g] = 0
            faults[f"drop group {g}"] = out(dd, te)
        faults["neighbour weight scale"] = out(d, ae[None, :] - np.roll(kexp, -1, axis=1))
        faults["neighbour activation scale"] = out(d, np.roll(ae, -1)[None, :] - kexp)
        if name == "down":
            KT, Gt = s.hidden // n_kt, s.hidden // n_kt // gs
            ac2, ae2 = ac.copy(), ae.copy()
            ac2[:KT], ac2[KT:2 * KT] = ac[KT:2 * KT], ac[:KT]
            ae2[:Gt], ae2[Gt:2 * Gt] = ae[Gt:2 * Gt], ae[:Gt]
            faults["K tiles 0 and 1 swapped"] = out(group_dots(codes, ac2, gs), ae2[None, :] - kexp)
        for f, got in faults.items():
            frac = float((bits(got) != bits(want)).mean())
            report.append(f"{name} {f}: {frac:.4f}")
            assert frac >= 0.99, f"{name}: '{f}' changes only {frac:.2%} of the outputs"
    print("; ".join(report))
