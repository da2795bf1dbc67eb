"""Decode attention of every (group size, GQA factor) kernel instance against a float64 reference, on both decode paths.

Decode attention -- the graph path's k_attn_partial<KVM> + k_attn_combine_quant<GS>, the persistent kernel's
attention_item<GS, KVM> -- is otherwise seen only through whole layers, where its output is re-quantised to int8 and an
FFN follows, so an error below one int8 step is invisible.  Here it is made observable through q3_forward_layers on
"attention probe" checkpoints (`export_probe`):

  * head_dim 128 and n_heads * 128 == dim; o_proj is the identity held exactly: row i has 127 * 2^-7 at column i (group
    scale 2^-7, code 127), every all-zero group has scale 1 and code 0;
  * down_proj is zero, so the FFN adds exactly 0; input_layernorm is 1.0; q / k / v projections and QK-norms are random;
  * the residual x holds integers * 2^-10 with a +-127 in every 32-element group (`probe_x`): rmsnorm is scale-invariant and
    every normalised value lands within a few ulps of an integer code, so quantize(rmsnorm(x)) gives the same codes
    whatever the order of the sums.
  So x_out - x is fl(fl(127 code_i 2^-7) xs_g), the dequantised int8 attention output o, up to the round-off of one f32
  addition.  q (after QK-norm and RoPE) is taken from the oracle (trace_layer): the reference's own f32 semantics,
  including its f32 RoPE angle.  The attended rows are read back from the device cache after the step, row `pos` (which
  the kernel wrote) included, so the float64 reference attends over exactly what the kernel attended over; that row is
  checked against the oracle's k / v on its own.

Regimes:
  needle  every query head h has a key alpha_h q_h / |q_h| at its own row p_h that beats every other score h sees by
          >= EXP_MARGIN (asserted): both exp implementations give exactly 0 for every other row and exp(0) = 1, so the
          output is V[p_h], integers * 2^-6 with a +-127 in every group -- exact in int8.  x_out must be bit-identical to
          the oracle's on both paths.  p_h: row 0 and pos - 1, first / last row of every split of both paths and of the
          persistent kernel's 32-row stages; heads sharing a kv head get different rows, so a wrong query head -> kv head
          mapping returns another head's needle.  One group of one head's needle row is zero (the zero-scale edge of
          quantize): its output must be exactly 0.
  dense   K rows N(0, 0.3^2), V rows N(0, 1): thousands of rows carry weight.
  peaky   dense with PEAKY_ROWS rows (boundary rows among them) scaled by PEAKY_GAIN: a few dozen rows carry most weight.
          Criterion for dense and peaky: |o_i - att64_i| <= (0.5 + tau) s_g for every element, s_g = max |att64| over the
          element's group / 127: the int8 rounding of the kernel's output is consistent with float64.  A correct f32
          kernel never violates it; an error of e codes violates it in about a fraction e - tau of the elements.  Each
          group's largest |o| must be 127 s_g within tau s_g.  The graph path repeats dense with exact mask 0b00111
          (norms, GEMV fold and QK-norm in reference order, attention still fast): q and the new K / V row are then
          bit-identical to the oracle's and only the attention kernel is under test.

tau, in codes (units of s_g); u = 2^-24.  Scales: |q_h| = |k_pos| ~ sqrt(128) = 11.3 (QK-norm), dense |k| ~ 0.3 * 11.3
= 3.4, boosted peaky rows |k| ~ 58, |v| ~ 1.  Sources of |att32 - att64|:
  * a score is a 128-term f32 dot: |ds| <~ u sqrt(128) |q| |k| / sqrt(128) = u |q| |k| (random-walk round-off of partial
    sums of size ~ |q| |k| / sqrt(128)); fast-mode q differs from the oracle's by |dq| / |q| ~ 3e-7 (a fold of dim / gs
    <= 64 group terms, the rmsnorm / QK-norm scales, RoPE), which adds ~ |dq| |k| / sqrt(128) per score.  A score error ds
    is a relative error ds of that row's weight.
      dense: ds ~ 2.5e-6, independent across the n rows that each carry ~1/n of the weight: o moves by ~ ds / sqrt(n),
      against s_g ~ 2.5 / (127 sqrt(n)): 127 * 2.5e-6 / 2.5 ~ 1.3e-4 codes, whatever n;
      peaky: the few rows that carry the weight have |ds| ~ u |q| |k| ~ 4e-5 and max |att| ~ |v|: 127 * 4e-5 ~ 5e-3 codes
      per unit of |v| / max |att|, which reaches 2-3.
  * exp (<= 2 ulp), the weighted sums (for the zero-mean dense V the partial sums stay of size ~ |att|) and 1 / L: a few
    u relative to max |att|; the softmax denominator, n positive terms: relative ~ u sqrt(m / 3) for sums of m terms --
    127 u sqrt(n / 3) = 9e-4 codes for one left fold over n = 40960 rows, far less in the kernels' split sums;
  * recovering o from fl(x + o): ulp(|x| + |o|) / 2 <= u (0.125 + 127 s_g), s_g >= 1e-4 here: < 1e-4 codes.
  TAU = 2e-3 (dense: ~1e-3 at worst); TAU_PEAKY = 3e-2 (~1.5e-2 at worst).  The oracle's f32 attention, whose left folds
  over all rows are the worst order there is, measures 4.9e-4 (dense) and 3.8e-3 (peaky) codes against float64 over up to
  4224 rows (`test_harness_float64_matches_oracle`), ~1e-2 codes on a peaky group maximum and 1.1e-3 on a dense one at
  40960 rows.  Dropping one cached row at the largest n tested (40960, dense) moves its head by ~0.6 codes, >= 10 TAU
  (`test_dropped_row_is_far_above_tau`); dropping a boosted peaky row moves it by tens of codes.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np
import pytest

from oracle import binding as orc
from qwen3_rs_b200 import transformer as T
from qwen3_rs_b200.export import EMBED_TOKENS_KEY, ExportConfig, export_from_loader
from qwen3_rs_b200.synth import make_tensor

HD = 128
N_LAYERS = 2
VOCAB = 256
HIDDEN = 256          # a multiple of 128 and >= the SM count: the persistent kernel gives every CTA an FFN unit
SEQ = 4224            # past the graph path's 32 splits x 128 rows
SEQ_LONG = 40960
GRAPH_CHUNK, GRAPH_MAX_SPLITS = 128, 32   # ATTN_MIN_CHUNK, ATTN_MAX_SPLITS (q3_kernels.cuh)
MEGA_CHUNK, MEGA_MAX_SPLITS = 32, 32      # MEGA_ATTN_CHUNK = MEGA_KV_ROWS, MEGA_MAX_SPLITS (q3_mega.cuh)
STAGE = 32
EXP_MARGIN = 120.0    # exp(-120) is 0 in f32 for glibc's expf and the device's
NEEDLE_SCORE = 300.0  # the scaled score of a head's own needle
TAU = 2e-3
TAU_PEAKY = 3e-2
DENSE_K_STD = 0.3
PEAKY_GAIN, PEAKY_ROWS = 17.0, 48
NEEDLE_ROUNDS = 3     # needle layouts per position (each plants one needle per query head)
EXACT_QKV_MASK = 0b00111
SCALE32 = float(np.float32(1.0) / np.sqrt(np.float32(HD)))  # the f32 1/sqrt(128) both implementations multiply by


@dataclass(frozen=True)
class Probe:
    n_heads: int
    n_kv: int
    gs: int
    seq_len: int = SEQ

    @property
    def dim(self) -> int:
        return self.n_heads * HD

    @property
    def kvm(self) -> int:
        return self.n_heads // self.n_kv

    @property
    def kv(self) -> int:
        return self.n_kv * HD

    def __str__(self):
        return f"h{self.n_heads}kv{self.n_kv}_gs{self.gs}_s{self.seq_len}"


# one shape per GQA factor at every group size, 8 kv heads (persistent split cap 148 // 8 = 18) and GQA 8 over 2 kv heads
# (a wrong query head -> kv head mapping reads the other kv head's query): all 12 k_mega_decode<GS, KVM> and all 4
# k_attn_partial<KVM> instances
PROBES = ([Probe(4, 4, gs) for gs in (32, 64, 128)] + [Probe(8, 8, 64)]
          + [Probe(8, kv, gs) for kv in (4, 2, 1) for gs in (32, 64, 128)] + [Probe(16, 2, 64)])
LONG_PROBE = Probe(8, 2, 64, SEQ_LONG)


def export_probe(p: Probe, path: str, seed: int = 0) -> dict:
    """An attention-probe checkpoint in the normal format (see the module docstring)."""
    cfg = ExportConfig(p.dim, HIDDEN, N_LAYERS, p.n_heads, p.n_kv, VOCAB, p.seq_len, HD)
    eye = (np.eye(p.dim, dtype=np.float32) * np.float32(127.0 / 128.0))
    shapes = {"self_attn.q_proj": (p.dim, p.dim), "self_attn.k_proj": (p.kv, p.dim), "self_attn.v_proj": (p.kv, p.dim),
              "mlp.gate_proj": (HIDDEN, p.dim), "mlp.up_proj": (HIDDEN, p.dim)}

    def load(name: str):
        if name == EMBED_TOKENS_KEY:
            return make_tensor(name, (VOCAB, p.dim), "embed", seed).numpy()
        if name.endswith("input_layernorm.weight") or name == "model.norm.weight":
            return np.ones(p.dim, np.float32)
        if name.endswith("post_attention_layernorm.weight"):
            return make_tensor(name, (p.dim,), "norm", seed).numpy()
        if name.endswith("q_norm.weight") or name.endswith("k_norm.weight"):
            return make_tensor(name, (HD,), "norm", seed).numpy()
        comp = name.split(".", 3)[3].rsplit(".", 1)[0] if name.startswith("model.layers.") else None
        if comp == "self_attn.o_proj":
            return eye
        if comp == "mlp.down_proj":
            return np.zeros((p.dim, HIDDEN), np.float32)
        if comp in shapes:
            return make_tensor(name, shapes[comp], "linear", seed).numpy()
        return None

    info = export_from_loader(load, cfg, path, p.gs, shared_classifier=True)
    assert info["group_size"] == p.gs, info
    return info


def _with_pm127(k: np.ndarray, rng) -> np.ndarray:
    """Integer codes in [-126, 126] with one +-127 in every 32-element group."""
    g = k.reshape(-1, 32)
    g[np.arange(g.shape[0]), rng.integers(0, 32, g.shape[0])] = rng.choice([-127, 127], g.shape[0])
    return g.reshape(k.shape)


def probe_x(rng, dim: int) -> np.ndarray:
    return (_with_pm127(rng.integers(-126, 127, dim), rng) * 2.0 ** -10).astype(np.float32)


def needle_v(rng) -> np.ndarray:
    return (_with_pm127(rng.integers(-126, 127, HD), rng) * 2.0 ** -6).astype(np.float32)


# ---- split / stage maps of the two paths (mirrors of attn_split_range and mega_nsplit + attention_item) ----------------
def graph_splits(pos: int):
    n = pos + 1
    ns = min(-(-n // GRAPH_CHUNK), GRAPH_MAX_SPLITS)
    per = -(-n // ns)
    return [(s * per, min(s * per + per, n)) for s in range(ns) if s * per < n]


def mega_splits(pos: int, n_kv: int, num_sms: int):
    n = pos + 1
    ns = min(-(-n // MEGA_CHUNK), max(1, min(num_sms // n_kv, MEGA_MAX_SPLITS)))
    per = -(-n // ns)
    return [(s * per, min(s * per + per, n)) for s in range(ns) if s * per < n]


def positions(p: Probe, num_sms: int):
    """Every split-count boundary of both paths +-1 (including both caps), plus the last position."""
    cap = max(1, min(num_sms // p.n_kv, MEGA_MAX_SPLITS))
    edges = {32, 128, cap * MEGA_CHUNK, GRAPH_CHUNK * GRAPH_MAX_SPLITS}
    if p.seq_len > SEQ:
        edges = {GRAPH_CHUNK * GRAPH_MAX_SPLITS, 32768}
    ps = sorted({e + d for e in edges for d in (-1, 0, 1)} | {p.seq_len - 1})
    return [q for q in ps if 0 < q < p.seq_len]


def needle_candidates(pos: int, n_kv: int, num_sms: int, rng):
    """Rows where decode attention goes wrong, categories interleaved so every layout mixes them."""
    ms, gsp = mega_splits(pos, n_kv, num_sms), graph_splits(pos)
    stages = [(b, min(b + STAGE, t1) - 1) for t0, t1 in ms for b in range(t0, t1, STAGE)]
    cats = [[0, pos - 1], [t1 - 1 for _, t1 in ms], [t1 - 1 for _, t1 in gsp], [t0 for t0, _ in ms], [t0 for t0, _ in gsp],
            [a for a, _ in stages], [b for _, b in stages]]
    cats = [[c for c in cat if 0 <= c < pos] for cat in cats]
    for cat in cats[1:]:
        rng.shuffle(cat)
    out, seen = [], set()
    while any(cats):
        for cat in cats:
            while cat:
                c = cat.pop(0)
                if c not in seen:
                    seen.add(c)
                    out.append(c)
                    break
    return out


# ---- float64 reference ------------------------------------------------------------------------------------------------
def attend64(q: np.ndarray, k: np.ndarray, v: np.ndarray, n_heads: int, n_kv: int):
    """softmax(q k^T / sqrt(128)) v per query head in float64 over the rows k / v [n][n_kv * 128] -> (att [AH],
    scores [n_heads][n])."""
    n, kvm = k.shape[0], n_heads // n_kv
    qh = q.astype(np.float64).reshape(n_heads, HD)
    kk = k.astype(np.float64).reshape(n, n_kv, HD)
    vv = v.astype(np.float64).reshape(n, n_kv, HD)
    att, sc = np.empty((n_heads, HD)), np.empty((n_heads, n))
    for g in range(n_kv):
        s = qh[g * kvm:(g + 1) * kvm] @ kk[:, g].T * SCALE32
        w = np.exp(s - s.max(axis=1, keepdims=True))
        att[g * kvm:(g + 1) * kvm] = (w @ vv[:, g]) / w.sum(axis=1, keepdims=True)
        sc[g * kvm:(g + 1) * kvm] = s
    return att.reshape(-1), sc


def o_of(x: np.ndarray, x_out: np.ndarray) -> np.ndarray:
    """The dequantised int8 attention output code_i xs_g from a probe layer's residual update 127/128 code_i xs_g."""
    return (x_out.astype(np.float64) - x.astype(np.float64)) * (128.0 / 127.0)


def judge(o: np.ndarray, att64: np.ndarray, gs: int):
    """-> (worst excess over half a code, worst |largest |o| of a group - 127 s_g|), both in codes."""
    og, ag = o.reshape(-1, gs), att64.reshape(-1, gs)
    s = np.abs(ag).max(axis=1) / 127.0
    assert (s > 0).all()
    excess = float((np.abs(og - ag) / s[:, None]).max() - 0.5)
    top = float((np.abs(np.abs(og).max(axis=1) - 127.0 * s) / s).max())
    return excess, top


# ---- the harness: one probe checkpoint with its CPU oracle and host mirror of the cache --------------------------------
class Harness:
    def __init__(self, p: Probe, path: str, seed: int = 0):
        self.p = p
        self.o = orc.Model(path)
        c = self.o.config
        assert (c["dim"], c["n_heads"], c["n_kv_heads"], c["group_size"], c["seq_len"]) == (p.dim, p.n_heads, p.n_kv, p.gs, p.seq_len)
        self.rng = np.random.default_rng(seed + 1000 * p.n_heads + 100 * p.n_kv + p.gs)
        self.K = np.empty((N_LAYERS, p.seq_len, p.kv), np.float32)
        self.V = np.empty((N_LAYERS, p.seq_len, p.kv), np.float32)
        self.ko, self.vo = self.o.kv_cache()
        self.devices = []

    def fill_dense(self):
        for l in range(N_LAYERS):
            self.K[l] = (self.rng.standard_normal((self.p.seq_len, self.p.kv)) * DENSE_K_STD).astype(np.float32)
            self.V[l] = self.rng.standard_normal((self.p.seq_len, self.p.kv)).astype(np.float32)
            self.sync_rows(l, 0, self.p.seq_len)

    def sync_rows(self, l: int, r0: int, r1: int):
        """Host mirror rows [r0, r1) of layer l -> the oracle's cache and every attached device handle."""
        self.ko[l, r0:r1] = self.K[l, r0:r1].reshape(r1 - r0, self.p.n_kv, HD)
        self.vo[l, r0:r1] = self.V[l, r0:r1].reshape(r1 - r0, self.p.n_kv, HD)
        for m in self.devices:
            m.kv_write(l, r0, self.K[l, r0:r1], self.V[l, r0:r1])

    def oracle(self, x: np.ndarray, pos: int, l: int):
        """The oracle's layer l at pos -> (x_out, trace); its cache row pos is restored afterwards."""
        tr = self.o.trace_layer(l)
        xo = self.o.forward_layers(x, pos, l, l + 1)
        tr = {k: v.copy() for k, v in tr.items()}
        self.sync_rows(l, pos, pos + 1)
        return xo, tr

    def device(self, m, x: np.ndarray, pos: int, l: int):
        """The device's layer l at pos -> (x_out, K rows [0, pos], V rows [0, pos] as the kernel attended over them);
        its cache row pos is restored afterwards."""
        xo = m.forward_layers(x, pos, l, l + 1)
        k, v = m.kv_read(l, 0, pos + 1)
        m.kv_write(l, pos, self.K[l, pos:pos + 1], self.V[l, pos:pos + 1])
        return xo, k, v

    def plant_needles(self, l: int, q: np.ndarray, rows, zero_head: int):
        """Head h's needle at rows[h] of layer l; one GS group of head zero_head's needle V row is zero."""
        p = self.p
        for h, r in enumerate(rows):
            g = h // p.kvm
            qh = q[h * HD:(h + 1) * HD].astype(np.float64)
            alpha = NEEDLE_SCORE / SCALE32 / np.linalg.norm(qh)
            self.K[l, r, g * HD:(g + 1) * HD] = (alpha * qh / np.linalg.norm(qh)).astype(np.float32)
            vn = needle_v(self.rng)
            if h == zero_head:
                z = self.rng.integers(0, HD // p.gs) if p.gs < HD else 0
                vn[z * p.gs:(z + 1) * p.gs] = 0.0
            self.V[l, r, g * HD:(g + 1) * HD] = vn
            self.sync_rows(l, r, r + 1)

    def close(self):
        self.o.close()


def needle_rows(cands, r: int, n_heads: int, pos: int, rng):
    """Layout r: one row per query head, all different (so heads sharing a kv head never share a needle)."""
    rows = list(cands[r * n_heads:(r + 1) * n_heads])
    free = np.setdiff1d(np.arange(pos), rows)
    rows += rng.choice(free, n_heads - len(rows), replace=False).tolist()
    return rows


def assert_needle_margins(H: Harness, q, k, v, rows, label):
    """Over the rows the kernel attended (read back), each head's needle beats its every other score by EXP_MARGIN."""
    _, sc = attend64(q, k, v, H.p.n_heads, H.p.n_kv)
    for h, r in enumerate(rows):
        margin = sc[h, r] - np.delete(sc[h], r).max()
        assert margin >= EXP_MARGIN, f"{label}: head {h} needle at {r}: margin {margin:.1f}"


def needle_expected(H: Harness, x, l: int, rows):
    """x + o with o = 127/128 V[p_h] per head: every operation exact (V holds integers * 2^-6)."""
    p = H.p
    o = np.concatenate([H.V[l, r, (h // p.kvm) * HD:(h // p.kvm + 1) * HD] for h, r in enumerate(rows)])
    return x + o * np.float32(127.0 / 128.0)


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def assert_new_row(H: Harness, k, v, tr, pos, label, exact=False):
    """The row the kernel wrote at pos against the oracle's k (after QK-norm + RoPE) and v."""
    for got, want, what in ((k[pos], tr["k_post"], "k"), (v[pos], tr["v_row"], "v")):
        if exact:
            assert np.array_equal(bits(got), bits(want)), f"{label}: new {what} row differs"
        else:
            err = float(np.abs(got - want).max())
            assert err <= 1e-5 * max(1.0, float(np.abs(want).max())), f"{label}: new {what} row off by {err:.2e}"


def peaky_rows(p: Probe, pos_list, rng):
    """PEAKY_ROWS rows: split / stage boundaries below the positions tested, the rest random."""
    b = sorted({e + d for e in (32, 128, 576, 1024, 4096, 32768) for d in (-1, 0)} | {0})
    b = [r for r in b if r < max(pos_list)]
    return sorted(set(b) | set(rng.choice(np.setdiff1d(np.arange(max(pos_list)), b), PEAKY_ROWS - len(b), replace=False).tolist()))


def run_probe(H: Harness, m, pos_list):
    """Every regime on both paths at every position of pos_list, layer alternating with the position; exact mode last.
    Returns the per-regime statistics that the test prints."""
    p = H.p
    num_sms = m.num_sms
    st = {"needles": 0, "dense": -1.0, "peaky": -1.0, "dense_q_exact": -1.0, "top": 0.0, "exact_steps": 0}
    H.devices = [m]
    H.fill_dense()

    def judged(key, x, xo, q, k, v, label, tau=TAU):
        att64, _ = attend64(q, k, v, p.n_heads, p.n_kv)
        excess, top = judge(o_of(x, xo), att64, p.gs)
        st[key] = max(st[key], excess)
        st["top"] = max(st["top"], top)
        assert excess <= tau, f"{label}: int8 output off float64 by {0.5 + excess:.4f} codes (allowed {0.5 + tau})"
        assert top <= tau, f"{label}: a group's largest output is {top:.4f} codes off 127 s_g"

    for i, pos in enumerate(pos_list):
        l = i % N_LAYERS
        x = probe_x(H.rng, p.dim)
        _, tr = H.oracle(x, pos, l)
        q = tr["q_post"]
        for path in (0, 1):
            m.set_decode_path(path)
            label = f"{p} path {path} layer {l} pos {pos} dense"
            xo, k, v = H.device(m, x, pos, l)
            assert_new_row(H, k, v, tr, pos, label)
            judged("dense", x, xo, q, k, v, label)
        m.set_exact_mask(EXACT_QKV_MASK)  # any non-zero mask runs the graph path
        try:
            label = f"{p} graph path, exact q/k/v, layer {l} pos {pos} dense"
            xo, k, v = H.device(m, x, pos, l)
            assert_new_row(H, k, v, tr, pos, label, exact=True)
            judged("dense_q_exact", x, xo, q, k, v, label)
        finally:
            m.set_exact_mask(0)
        cands = needle_candidates(pos, p.n_kv, num_sms, H.rng)
        for r in range(min(NEEDLE_ROUNDS, -(-len(cands) // p.n_heads))):
            rows = needle_rows(cands, r, p.n_heads, pos, H.rng)
            saved = H.K[l, rows].copy(), H.V[l, rows].copy()
            zero_head = (i + r) % p.n_heads
            H.plant_needles(l, q, rows, zero_head)
            want = needle_expected(H, x, l, rows)
            xo_ref, tr_n = H.oracle(x, pos, l)
            assert np.array_equal(bits(tr_n["q_post"]), bits(q))
            for path in (0, 1):
                m.set_decode_path(path)
                label = f"{p} path {path} layer {l} pos {pos} needles at {rows}"
                xo, k, v = H.device(m, x, pos, l)
                assert_needle_margins(H, q, k, v, rows, label)
                z = slice(zero_head * HD, (zero_head + 1) * HD)
                zg = np.nonzero(want[z] == x[z])[0]
                assert np.array_equal(bits(xo[z][zg]), bits(x[z][zg])), f"{label}: zero group of head {zero_head} not 0"
                bad = np.nonzero(bits(xo) != bits(want))[0]
                assert bad.size == 0, f"{label}: heads {sorted(set((bad // HD).tolist()))} differ from their needle rows"
                assert np.array_equal(bits(xo), bits(xo_ref)), f"{label}: differs from the oracle"
            st["needles"] += len(rows)
            H.K[l, rows], H.V[l, rows] = saved
            for row in rows:
                H.sync_rows(l, row, row + 1)

    boost = peaky_rows(p, pos_list, H.rng)
    for l in range(N_LAYERS):
        H.K[l, boost] *= np.float32(PEAKY_GAIN)
        for row in boost:
            H.sync_rows(l, row, row + 1)
    for i, pos in enumerate(pos_list):
        l = (i + 1) % N_LAYERS
        x = probe_x(H.rng, p.dim)
        _, tr = H.oracle(x, pos, l)
        for path in (0, 1):
            m.set_decode_path(path)
            label = f"{p} path {path} layer {l} pos {pos} peaky"
            xo, k, v = H.device(m, x, pos, l)
            assert_new_row(H, k, v, tr, pos, label)
            judged("peaky", x, xo, tr["q_post"], k, v, label, TAU_PEAKY)

    # exact mode: the whole step (both layers) bit-identical to the oracle on both sides of 128
    m.set_exact(True)
    try:
        for pos in [q for q in (126, 127, 128, 129, 130) if q < p.seq_len]:
            x = probe_x(H.rng, p.dim)
            xo = m.forward_layers(x, pos, 0, N_LAYERS)
            xr = H.o.forward_layers(x, pos, 0, N_LAYERS)
            assert np.array_equal(bits(xo), bits(xr)), f"{p} exact mode pos {pos}: differs from the oracle"
            for l in range(N_LAYERS):
                H.sync_rows(l, pos, pos + 1)
            st["exact_steps"] += 1
    finally:
        m.set_exact(False)
        m.set_decode_path(1)
    H.devices = []
    return st


@pytest.fixture(scope="module")
def probe_path(tmp_path_factory):
    d = tmp_path_factory.mktemp("probe")
    cache = {}

    def get(p: Probe) -> str:
        if p not in cache:
            cache[p] = str(d / f"{p}.bin")
            export_probe(p, cache[p])
        return cache[p]

    return get


def _run_gpu(p: Probe, path: str, pos_for):
    H = Harness(p, path)
    m = T.TransformerBuilder.new(path).build()
    try:
        m.set_decode_path(1)  # the persistent kernel must take every probe shape: refused is a failure, not a skip
        pos_list = pos_for(m.num_sms)
        st = run_probe(H, m, pos_list)
        print(f"{p} ({m.num_sms} SMs) positions {pos_list}: worst excess over half a code: dense {st['dense']:+.2e}, "
              f"peaky {st['peaky']:+.2e}, dense with exact q/k/v {st['dense_q_exact']:+.2e}; worst group-max error "
              f"{st['top']:.2e} codes; {st['needles']} needles per path; {st['exact_steps']} exact-mode steps")
    finally:
        m.close()
        H.close()


# ---- on the GPU -------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("p", PROBES, ids=str)
def test_decode_attention_against_float64(probe_path, p):
    """Every decode attention instance (persistent <GS, KVM>, graph <KVM> + combine <GS>) against float64 at every
    split-count boundary of both paths, past both split caps."""
    _run_gpu(p, probe_path(p), lambda num_sms: positions(p, num_sms))


@pytest.mark.gpu
def test_decode_attention_long_context_against_float64(probe_path):
    """The same at 40960 cached rows: past 32K positions (the f32 RoPE angle of the reference, taken from the oracle) and at
    the last position of a 40960-row context."""
    p = LONG_PROBE
    _run_gpu(p, probe_path(p), lambda num_sms: positions(p, num_sms))


# ---- host-only checks of the harness itself (CPU oracle) ------------------------------------------------------------------
HOST_PROBE = Probe(8, 2, 32)


@pytest.fixture(scope="module")
def host_harness(probe_path):
    H = Harness(HOST_PROBE, probe_path(HOST_PROBE), seed=5)
    H.fill_dense()
    yield H
    H.close()


def test_probe_layer_adds_exactly_the_quantised_attention(host_harness):
    """x_out - x is the dequantised int8 attention output, bit for bit: o_proj is the identity, the FFN adds 0."""
    H, p = host_harness, HOST_PROBE
    for pos, l in ((77, 0), (1500, 1)):
        x = probe_x(H.rng, p.dim)
        xo, tr = H.oracle(x, pos, l)
        qa, sa = orc.quantize(tr["att_out"], p.gs)
        o = (qa.astype(np.float32) * np.float32(127.0 / 128.0)) * np.repeat(sa, p.gs)
        assert np.array_equal(bits(xo), bits(x + o))
        assert np.array_equal(bits(tr["x_after_attn"]), bits(xo))  # the FFN added exactly 0


def test_needle_construction_gives_exact_attention(host_harness):
    """With the needles planted the oracle's attention output is each head's needle V row, exactly (zero group included)."""
    H, p = host_harness, HOST_PROBE
    pos, l = 700, 1
    x = probe_x(H.rng, p.dim)
    _, tr = H.oracle(x, pos, l)
    q = tr["q_post"]
    rows = needle_rows(needle_candidates(pos, p.n_kv, 148, H.rng), 0, p.n_heads, pos, H.rng)
    saved = H.K[l, rows].copy(), H.V[l, rows].copy()
    H.plant_needles(l, q, rows, zero_head=3)
    try:
        xo, tr = H.oracle(x, pos, l)
        k, v = H.K[l, :pos + 1].copy(), H.V[l, :pos + 1].copy()
        k[pos], v[pos] = tr["k_post"], tr["v_row"]
        assert_needle_margins(H, q, k, v, rows, "oracle")
        for h, r in enumerate(rows):
            g = h // p.kvm
            assert np.array_equal(bits(tr["att_out"][h * HD:(h + 1) * HD]), bits(H.V[l, r, g * HD:(g + 1) * HD])), h
        assert np.array_equal(bits(xo), bits(needle_expected(H, x, l, rows)))
        assert np.isfinite(xo).all()
    finally:
        H.K[l, rows], H.V[l, rows] = saved
        for row in rows:
            H.sync_rows(l, row, row + 1)


@pytest.mark.parametrize("regime", ["dense", "peaky"])
def test_harness_float64_matches_oracle(host_harness, regime):
    """The float64 reference agrees with the oracle's f32 attention (left folds over up to 4224 rows) within the regime's
    tolerance in codes."""
    H, p = host_harness, HOST_PROBE
    pos_list = [129, 1025, 4097, p.seq_len - 1]
    boost = peaky_rows(p, pos_list, H.rng) if regime == "peaky" else []
    saved = H.K[:, boost].copy()
    for l in range(N_LAYERS):
        H.K[l, boost] *= np.float32(PEAKY_GAIN)
        for row in boost:
            H.sync_rows(l, row, row + 1)
    try:
        worst = 0.0
        for i, pos in enumerate(pos_list):
            l = i % N_LAYERS
            x = probe_x(H.rng, p.dim)
            _, tr = H.oracle(x, pos, l)
            k, v = H.K[l, :pos + 1].copy(), H.V[l, :pos + 1].copy()
            k[pos], v[pos] = tr["k_post"], tr["v_row"]
            att64, sc = attend64(tr["q_post"], k, v, p.n_heads, p.n_kv)
            s = np.abs(att64.reshape(-1, p.gs)).max(axis=1) / 127.0
            err = np.abs(tr["att_out"].astype(np.float64) - att64).reshape(-1, p.gs) / s[:, None]
            worst = max(worst, float(err.max()))
            if regime == "peaky":  # a few dozen rows carry most of the weight
                w = np.exp(sc - sc.max(axis=1, keepdims=True))
                w /= w.sum(axis=1, keepdims=True)
                assert (np.sort(w, axis=1)[:, -PEAKY_ROWS:].sum(axis=1) >= 0.5).all()
        print(f"{regime}: oracle f32 attention vs float64, worst {worst:.2e} codes")
        assert worst <= (TAU_PEAKY if regime == "peaky" else TAU)
    finally:
        for l in range(N_LAYERS):
            H.K[l, boost] = saved[l]
            for row in boost:
                H.sync_rows(l, row, row + 1)


def test_dropped_row_is_far_above_tau():
    """At the largest n tested (40960, dense) dropping one cached row moves its head's int8-scaled output by >= 10 TAU:
    the criterion sees the fault it is meant to see."""
    rng = np.random.default_rng(11)
    n = SEQ_LONG
    q = rng.standard_normal(HD)
    k = rng.standard_normal((n, HD)) * DENSE_K_STD
    v = rng.standard_normal((n, HD))
    s = (k @ q) * SCALE32
    w = np.exp(s - s.max())
    full = (w @ v) / w.sum()
    sg = np.abs(full).max() / 127.0
    moved = []
    for t in rng.choice(n, 64, replace=False):
        keep = np.ones(n, bool)
        keep[t] = False
        moved.append(np.abs((w[keep] @ v[keep]) / w[keep].sum() - full).max() / sg)
    print(f"dropping one of {n} dense rows moves the head by {np.median(moved):.3f} codes (median of 64 rows)")
    assert np.median(moved) >= 10 * TAU
