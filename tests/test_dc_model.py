"""The integer model of the DC recursion, pinned against the real float recursion (CPU only).

The DC-removal stage (sdrj.cpp:277-283) is the one place where the kernels claim bit-identity with the reference:
avept = fl(fl(avept * a) + fl(c * x)) with a = 1 - 1e-6f, c = 1e-6f. k0_dc_walk replaces most of those float steps by
integer translations and integer solves in units of the state's ulp. That is exact only because of facts about float32
that k0_dc_anchor and k0_dc_qtab rely on without checking them at run time. This file restates the two kernels in numpy,
with the float32 operations in the kernels' order, and checks those facts over every state a uint8 input can drive the
recursion to with a usable ("ok") anchor:

  1. inside the anchor's window (lo, hi) the rounded product removes r0 ulps below T and r0 + 1 from T on, and T is the
     true first mantissa of r0 + 1 wherever the walk can see it;
  2. one real step from a state in the window moves its bit pattern by exactly Q(byte) - r0 - [bits >= T];
  3. no byte is a rounding tie for an ok anchor, which is why k0_dc_qtab, k0_dc_blocks and the walk have no tie
     handling -- while ties do exist for states below 2^-6, where no anchor is ok;
  4. the largest dip one block can make from the window's low edge keeps r in {r0, r0 + 1}: the low side needs no
     per-block check (only the high side has one, DcStats::tb_hi).

Restated: kernels.cuh dc_step / dc_incr (lines 250-258), k0_dc_anchor (260-312), k0_dc_qtab (320-326)."""
import math

import numpy as np
import pytest

F32 = np.float32
DC_A = F32(1.0) - F32(0.000001)          # kernels.cuh:48, folded in float like the reference
DC_C = F32(0.000001)
DC_MAGIC = F32(12582912.0)
DC_BLK = 128
STEP = 16777216.0 / 17.0                   # mantissa distance between steps of r
EF_LO, EF_HI = 127 - 8, 127 + 7            # binades 2^-8 .. 2^7: |avept| <= 128 for uint8 input, and the binade above
EF_OK_MIN = 127 - 3                        # anchors are ok from 2^-3 up


def f32(bits):
    return np.asarray(bits, np.uint32).view(np.float32)


def bits_of(x):
    return np.asarray(x, np.float32).view(np.uint32)


def dc_step(s, x):
    """kernels.cuh:250-252, elementwise in float32."""
    s, x = np.asarray(s, F32), np.asarray(x, F32)
    return (s * DC_A) + (DC_C * x)


def anchor(s0):
    """k0_dc_anchor (kernels.cuh:260-312) for one state; float32 operations in the kernel's order, doubles where it
    uses doubles. Returns a dict with the DcAnchor fields."""
    s0 = F32(s0)
    A = dict(sgn=-1.0 if s0 < 0 else 1.0, inv_u=F32(0), r0=0, ok=0, T=0, lo=0, hi=0, pinned=True)
    m = F32(abs(s0))
    bits = int(bits_of(m))
    ef = bits >> 23
    if not 40 <= ef <= 200:
        return A
    base = bits & 0xFF800000
    inv_u = f32((254 - (ef - 23)) << 23)
    A["inv_u"] = inv_u
    dec = F32(m - F32(m * DC_A))
    r = int(np.rint(F32(dec * inv_u)))
    m_cur = float((bits & 0x7FFFFF) + 0x800000)
    m_up, m_dn = math.ceil((r + 0.5) * STEP), math.ceil((r - 0.5) * STEP)
    if abs(m_up - m_cur) <= abs(m_cur - m_dn):
        r0, m_t = r, m_up
    else:
        r0, m_t = r - 1, m_dn
    if m_t >= 16777216.0:
        T = base + 0x800000
    elif m_t < 8388608.0:
        T = base
    else:
        T = base + (int(m_t) - 8388608)
        A["pinned"] = False
        for _ in range(6):
            a1, a0 = f32(T), f32(T - 1)
            d1 = F32(F32(a1 - F32(a1 * DC_A)) * inv_u)
            d0 = F32(F32(a0 - F32(a0 * DC_A)) * inv_u)
            if d1 >= F32(r0 + 1) and d0 <= F32(r0):
                A["pinned"] = True
                break
            T += 1 if d1 < F32(r0 + 1) else -1
    lo, hi = 8388608.0 + 4096.0, 16777216.0 - 65536.0
    lo = max(lo, math.ceil((r0 - 0.5) * STEP) + 2.0)
    hi = min(hi, math.ceil((r0 + 1.5) * STEP) - 2.0)
    qmax = math.ceil(128.0 * float(DC_C) * float(inv_u)) + 18.0
    lo += DC_BLK * qmax
    A.update(ef=ef, base=base, qmax=qmax)
    if hi > lo and qmax < 1.0e5:
        A.update(lo=base + (int(lo) - 8388608), hi=base + (int(hi) - 8388608), r0=r0, T=T, ok=1)
    return A


def qtab(A):
    """k0_dc_qtab (kernels.cuh:320-326) with dc_incr (255-258): increment d = Q - r0 of each byte. Also returns
    which bytes are rounding ties, fl(c * x) / ulp an exact half: the kernel assumes there are none."""
    x = (np.arange(256) - 127).astype(F32)
    y = F32(DC_C) * (F32(A["sgn"]) * x)
    y = (y * F32(A["inv_u"])).astype(F32)
    q = ((y + DC_MAGIC).astype(F32) - DC_MAGIC).astype(F32)
    tie = np.abs((y - q).astype(F32)) == F32(0.5)
    d = q.astype(np.int64) - A["r0"]
    return (d if A["ok"] else np.zeros_like(d)), tie


def r_of_binade(ef):
    """r(M) = (m - fl(m * a)) / ulp for every mantissa M of binade `ef` (exact: Sterbenz, and ulp is a power of 2).
    Values 8..17, kept as int8: the module keeps sixteen binades of them."""
    base = ef << 23
    m = f32(np.arange(base, base + 0x800000, dtype=np.uint32))
    dec = m - m * DC_A
    inv_u = f32((254 - (ef - 23)) << 23)
    return (dec * inv_u).astype(np.int8)


def anchors_of_binade(ef, r):
    """Every anchor k0_dc_anchor can produce for a state in binade `ef`: it depends on the state only through r0, so
    one state per distinct r0 stands for all."""
    M = np.arange(0x800000, 0x1000000, dtype=np.float64)
    m_up, m_dn = np.ceil((r + 0.5) * STEP), np.ceil((r - 0.5) * STEP)
    r0 = np.where(np.abs(m_up - M) <= np.abs(M - m_dn), r, r - 1)
    vals, first = np.unique(r0, return_index=True)
    out = []
    for v, i in zip(vals, first):
        A = anchor(f32((ef << 23) + int(i)))
        assert A["ok"] == 0 or A["r0"] == v
        out.append(A)
    return out


@pytest.fixture(scope="module")
def binades():
    """{ef: (r of every mantissa, [anchors])} for the binades 2^-8 .. 2^7."""
    out = {}
    for ef in range(EF_LO, EF_HI + 1):
        r = r_of_binade(ef)
        out[ef] = (r, anchors_of_binade(ef, r))
    return out


@pytest.fixture(scope="module")
def ok_anchors(binades):
    return [A for ef in binades for A in binades[ef][1] if A["ok"]]


def test_anchor_is_ok_exactly_from_two_to_the_minus_three(binades):
    """The window exists only where one block's largest excursion fits between two steps of r: from 2^-3 up, at every
    r0 a state of the binade can select."""
    for ef, (r, anchors) in binades.items():
        assert {9, 16} <= {int(v) for v in np.unique(r)} <= set(range(8, 18)), ef
        ok = [A["ok"] for A in anchors]
        if ef < EF_OK_MIN:
            assert not any(ok), ef
        else:
            assert sum(ok) >= 8, (ef, [(A["r0"], A["ok"]) for A in anchors])
    for ef in range(40, EF_LO):                      # far below: never ok (qmax grows as the binade shrinks)
        assert not anchor(f32((ef << 23) + 0x400000))["ok"]


def test_anchor_invariant_exhaustive(binades):
    """For every ok anchor of every binade up to |avept| = 128: every mantissa strictly inside (lo, hi) has
    r = r0 + [bits >= T], and the pinned T is the true first mantissa of r0 + 1 or lies outside (lo, hi)."""
    n_checked = n_t_inside = 0
    for ef, (r, anchors) in binades.items():
        base = ef << 23
        for A in anchors:
            if not A["ok"]:
                continue
            lo, hi, T, r0 = A["lo"] - base, A["hi"] - base, A["T"] - base, A["r0"]
            assert 0 < lo < hi < 0x800000
            idx = np.arange(lo + 1, hi)
            want = r0 + (idx >= T)
            bad = np.flatnonzero(r[lo + 1:hi] != want)
            assert bad.size == 0, (ef, r0, "mantissa", int(idx[bad[0]]), int(r[lo + 1 + bad[0]]), int(want[bad[0]]))
            n_checked += idx.size
            if lo < T < hi:
                n_t_inside += 1
                first = int(np.flatnonzero(r == r0 + 1)[0])
                assert T == first, (ef, r0, T, first)
                assert A["pinned"], (ef, r0)
    assert n_checked > 50_000_000 and n_t_inside >= 50


def test_increment_model_sampled(ok_anchors):
    """10^6 random (anchor, sign, byte, in-window state): one real float step moves the bit pattern of |state| by
    exactly Q(byte) - r0 - [bits >= T] -- the translation every walk path (run, solve, k1 re-derivation) relies on."""
    rng = np.random.default_rng(20261020)
    n = 1_000_000
    k = rng.integers(0, len(ok_anchors), n)
    sgn = np.where(rng.integers(0, 2, n) == 1, -1.0, 1.0)
    byte = rng.integers(0, 256, n)
    lo = np.array([A["lo"] for A in ok_anchors], np.int64)[k]
    hi = np.array([A["hi"] for A in ok_anchors], np.int64)[k]
    T = np.array([A["T"] for A in ok_anchors], np.int64)[k]
    bits = lo + 1 + (rng.random(n) * (hi - lo - 1)).astype(np.int64)
    # half of the draws within 200 mantissas of T, where r changes
    near = rng.random(n) < 0.5
    bits = np.where(near, np.clip(T + rng.integers(-200, 200, n), lo + 1, hi - 1), bits)
    tabs = {}
    for i, A in enumerate(ok_anchors):
        for sg in (1.0, -1.0):
            d, tie = qtab(dict(A, sgn=sg))
            assert not tie.any()
            tabs[(i, sg)] = d
    d = np.empty(n, np.int64)
    for i in range(len(ok_anchors)):
        for sg in (1.0, -1.0):
            sel = (k == i) & (sgn == sg)
            d[sel] = tabs[(i, sg)][byte[sel]]
    s = f32(bits.astype(np.uint32)) * sgn.astype(F32)
    x = (byte - 127).astype(F32)
    real = dc_step(s, x)
    model = f32((bits + d - (bits >= T)).astype(np.uint32)) * sgn.astype(F32)
    bad = np.flatnonzero(bits_of(real) != bits_of(model))
    assert bad.size == 0, (int(bad.size), float(s[bad[0]]), int(byte[bad[0]]), float(real[bad[0]]), float(model[bad[0]]))
    assert (bits >= T).any() and (bits < T).any()


def test_no_rounding_tie_is_reachable(binades, ok_anchors):
    """fl(c * x) / ulp is never an exact half for an ok anchor, whatever the byte and sign: this is why k0_dc_qtab
    stores Q - r0 without marking ties, and k0_dc_blocks and the walk's integer solves have no tie branch. Ties do occur
    for |avept| < 2^-6, where the anchor is never ok and every block is stepped in float."""
    for A in ok_anchors:
        for sg in (1.0, -1.0):
            _, tie = qtab(dict(A, sgn=sg))
            assert not tie.any(), (A["ef"], A["r0"], sg, np.flatnonzero(tie))
    tie_binades = set()
    for ef, (_, anchors) in binades.items():
        for sg in (1.0, -1.0):
            _, tie = qtab(dict(anchors[0], sgn=sg, ok=1))
            if tie.any():
                tie_binades.add(ef)
    assert tie_binades and max(tie_binades) < 127 - 6, sorted(tie_binades)
    assert not any(A["ok"] for ef in tie_binades for A in binades[ef][1])


@pytest.mark.parametrize("x", [-127.0, -128.0])
def test_one_block_dip_from_the_window_low_edge(ok_anchors, x):
    """128 real float steps of the largest pull towards zero (byte 0 for a positive state, byte 255 for a negative
    one; in magnitude x = -127 or -128), starting at bits lo + 1: every state passed through keeps the anchor's binade
    and r in {r0, r0 + 1}. This is the margin `lo += DC_BLK * qmax` buys; checked with the recursion, not the formula."""
    lo = np.array([A["lo"] for A in ok_anchors], np.uint32)
    ef = np.array([A["ef"] for A in ok_anchors], np.uint32)
    r0 = np.array([A["r0"] for A in ok_anchors], np.int64)
    inv_u = f32((254 - (ef - 23)) << 23)
    s = f32(lo + 1)
    xs = np.full(s.shape, x, F32)
    for step in range(DC_BLK + 1):
        assert np.all(bits_of(s) >> 23 == ef), step
        r = ((s - s * DC_A) * inv_u).astype(np.int64)
        bad = np.flatnonzero((r < r0) | (r > r0 + 1))
        assert bad.size == 0, (step, int(ef[bad[0]]), int(r0[bad[0]]), int(r[bad[0]]))
        s = dc_step(s, xs)
    assert np.all(s < f32(lo + 1))
