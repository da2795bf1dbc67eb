"""The gate/up unit map of the persistent decode kernel (q3_mega.cuh gu_map / gu_unit), mirrored on the host.

Each CTA streams cta_share's number of (gate, up) pairs, in blocks of MEGA_GW = 8.  Block s < F of CTA c holds units
s * 8 * nctas + 8 c .. + 7, and the tail past F * 8 * nctas is split with cta_share as each CTA's last block, so the
SwiGLU outputs below (s + 1) * 8 * nctas -- and every quantisation group of the down_proj input below that bound -- are
final once every CTA has finished its block s.  No GPU needed."""
import pytest

MEGA_GW = 8


def cta_share(units, nctas, c):
    base, rem = divmod(units, nctas)
    return c * base + min(c, rem), base + (1 if c < rem else 0)


def gu_map(units, nctas, c):
    full = units // nctas // MEGA_GW
    stride = MEGA_GW * nctas
    ts, _ = cta_share(units - full * stride, nctas, c)
    return full, stride, MEGA_GW * c, full * stride + ts


def gu_unit(m, j):
    full, stride, first, tail0 = m
    if j < MEGA_GW * full:
        return (j // MEGA_GW) * stride + first + j % MEGA_GW
    return tail0 + j - MEGA_GW * full


def segments(units, nctas):
    return [[gu_unit(gu_map(units, nctas, c), j) for j in range(cta_share(units, nctas, c)[1])] for c in range(nctas)]


# H_l of Qwen3-0.6B / 1.7B / 4B / 8B, the synthetic test shapes and the decode probes' hidden sizes
HIDDEN = [3072, 6144, 9728, 12288, 768, 512, 1536, 384, 2048, 3584, 4864, 12160, 14080, 16256]
CASES = sorted({(h // tp, n) for h in HIDDEN for tp in (1, 2, 4, 8) for n in (148, 132, 97, 13, 7, 1) if h // tp >= n})


@pytest.mark.parametrize("units,nctas", CASES)
def test_every_unit_once_and_counts_are_cta_share(units, nctas):
    seg = segments(units, nctas)
    assert [len(s) for s in seg] == [cta_share(units, nctas, c)[1] for c in range(nctas)]
    flat = sorted(u for s in seg for u in s)
    assert flat == list(range(units))


@pytest.mark.parametrize("units,nctas", CASES)
def test_slot_s_is_block_s_of_every_cta(units, nctas):
    """Unit u < F * stride sits in block u // stride of CTA (u % stride) // 8: the first (s + 1) * stride units, and with
    them every quantisation group below that bound, are final after block s of every CTA."""
    full, stride = units // nctas // MEGA_GW, MEGA_GW * nctas
    where = {}
    for c, s in enumerate(segments(units, nctas)):
        for j, u in enumerate(s):
            where[u] = (c, j // MEGA_GW)
    for u in range(full * stride):
        assert where[u] == ((u % stride) // MEGA_GW, u // stride)
    for u in range(full * stride, units):  # the tail: each CTA's last block
        c, blk = where[u]
        assert blk == full
    for gs in (32, 64, 128):
        for g in range(units // gs):
            last = max(where[u][1] for u in range(g * gs, (g + 1) * gs))
            if (g + 1) * gs <= full * stride:
                assert last == ((g + 1) * gs - 1) // stride
            else:
                assert last == full


@pytest.mark.parametrize("units,nctas", CASES)
def test_fewer_than_eight_units_per_cta_is_the_contiguous_map(units, nctas):
    if units // nctas >= MEGA_GW:
        assert gu_map(units, nctas, 0)[0] >= 1
        return
    for c in range(nctas):
        st, n = cta_share(units, nctas, c)
        m = gu_map(units, nctas, c)
        assert m[0] == 0
        assert [gu_unit(m, j) for j in range(n)] == list(range(st, st + n))


def test_bench_shape_regime():
    """Qwen3-8B on 148 SMs: 10 rounds of 1184 units and a tail of 448, so groups 0 .. 184 (of 64) are final after block 9
    of every CTA and only the last 7 groups wait for the tail blocks."""
    units, nctas = 12288, 148
    m = gu_map(units, nctas, 0)
    assert m[:2] == (10, 1184) and units - 10 * 1184 == 448
    assert 10 * 1184 // 64 == 185 and units // 64 - 185 == 7
