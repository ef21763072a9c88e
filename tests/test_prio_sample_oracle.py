"""tests/prio_sample_oracle.py on the host: the Philox stream against known answers, and the exact inverse CDF against
hand-worked cases and a rational-arithmetic restatement."""
import math
from fractions import Fraction

import numpy as np
import pytest

from tests import prio_sample_oracle as so


# ---------------------------------------------------------------------------------------------- the random stream
@pytest.mark.parametrize("ctr, key, want", [
    ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
     (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
])
def test_philox_known_answers(ctr, key, want):
    got = so.philox4x32_10(ctr, key)
    assert tuple(int(x) for x in got) == want


def test_philox_is_vectorised_over_the_counter():
    ctr = (np.array([0, 0xFFFFFFFF, 7], dtype=np.uint32), 0, np.uint32(3), 0)
    got = so.philox4x32_10(ctr, (11, 12))
    for i, c0 in enumerate((0, 0xFFFFFFFF, 7)):
        one = so.philox4x32_10((c0, 0, 3, 0), (11, 12))
        assert [int(w[i]) for w in got] == [int(w) for w in one]


def test_uniforms_pinned():
    U = so.uniforms(5, 0, 3)
    assert U.tolist() == [0.56139832071044049, 0.42204616608819734, 0.90786815416357824]
    assert so.uniforms(5, 0, 1).tolist() == U[:1].tolist()              # draw b does not depend on B
    hi = so.uniforms(5, 1 << 32, 3)                                      # the counter's high word is in the stream
    assert not np.array_equal(hi, U) and not np.array_equal(hi, so.uniforms(5, 1, 3))
    big = so.uniforms(2 ** 64 - 1, 2 ** 40 + 3, 4096)
    assert bool(((big >= 0.0) & (big < 1.0)).all())


# ---------------------------------------------------------------------------------------------- the inverse CDF
def _rational_pick(masses, v):
    """First candidate whose inclusive prefix exceeds v, in exact rationals; the last non-zero one past the total."""
    v, run = Fraction(max(v, 0.0)), Fraction(0)
    for i, m in enumerate(masses):
        run += Fraction(float(np.float32(m)))
        if run > v:
            return i
    return max(i for i, m in enumerate(masses) if m > 0)


def test_zeros_leading_interior_and_trailing_are_never_drawn():
    m = [0, 0, 1, 0, 0, 2, 0, 3, 0, 0]
    d, w = so.draw(m, 6.0, np.full(6, 0.5), 6, 0.5)                    # u = 0.5, 1.5, ..., 5.5
    assert d.pos.tolist() == [2, 5, 5, 7, 7, 7]
    assert not d.ambiguous.any()
    assert np.allclose(w, [1.0, 2 ** -0.5, 2 ** -0.5, 3 ** -0.5, 3 ** -0.5, 3 ** -0.5], rtol=1e-15)
    d, _ = so.draw(m, 6.0, np.zeros(6), 6, 0.5)                         # u = 0 .. 5: on the boundaries 1 and 3
    assert d.pos.tolist() == [2, 5, 5, 7, 7, 7]
    assert d.ambiguous.tolist() == [False, True, False, True, False, False]
    assert d.lo.tolist() == [2, 2, 5, 5, 7, 7] and d.hi.tolist() == [2, 5, 5, 7, 7, 7]


def test_a_single_non_zero_candidate_takes_every_draw():
    m = np.zeros(5000, dtype=np.float32)
    m[4321] = 0.25
    U = so.uniforms(9, 3, 256)
    d, w = so.draw(m, 0.25, U, 256, 0.7)
    assert (d.pos == 4321).all() and (w == 1.0).all()
    assert not d.ambiguous[1:].any()
    ref = so.Reference(m)
    assert ref.n_valid == 1 and ref.m_min == 0.25 and ref.last == 4321


def test_u_at_or_past_the_exact_total_takes_the_last_non_zero_candidate():
    m = [1.0, 2.0, 0.0, 0.0]
    total_k = 3.0 * (1 + 2.0 ** -50)                                    # a kernel total rounded above the exact 3
    U = np.array([1.0 - 2.0 ** -53])
    d, _ = so.draw(m, total_k, U, 1, 1.0)
    assert d.u[0] > 3.0
    assert d.pos.tolist() == [1] and d.ambiguous.tolist() == [False]    # both sides of the window are past the total
    ref = so.Reference(m)
    assert ref.pick([3.0, 1e300]).tolist() == [1, 1]
    assert ref.pick([2.9999999999999996]).tolist() == [1]
    assert ref.pick([-1.0, 0.0, 0.99999999]).tolist() == [0, 0, 0]
    assert ref.pick([1.0]).tolist() == [1]


def test_the_ambiguity_window():
    m = [1.0, 1.0, 1.0, 1.0]
    d, _ = so.draw(m, 4.0, np.zeros(4), 4, 0.0)                         # u = 0, 1, 2, 3: exactly on the boundaries
    assert d.pos.tolist() == [0, 1, 2, 3]
    assert d.ambiguous.tolist() == [False, True, True, True]            # (nothing lies before the first candidate)
    assert d.lo.tolist() == [0, 0, 1, 2] and d.hi.tolist() == [0, 1, 2, 3]
    w = so.WINDOW * 4.0                                                 # 2^-42
    d, _ = so.draw(m, 4.0, np.full(4, w / 2), 4, 0.0)                   # u = b + w / 2: inside the window
    assert d.ambiguous.tolist() == [False, True, True, True]
    d, _ = so.draw(m, 4.0, np.full(4, 2 * w), 4, 0.0)                   # u = b + 2 w: outside
    assert not d.ambiguous.any() and d.pos.tolist() == [0, 1, 2, 3]


def test_the_boundary_is_decided_exactly_where_a_float64_prefix_rounds():
    m = [2.0 ** 53, 1.0, 1.0]                                           # float64 cumsum: 2^53, 2^53, 2^53 + 2
    assert np.cumsum(m)[1] == 2.0 ** 53
    ref = so.Reference(m)
    assert ref.pick([2.0 ** 53]).tolist() == [1]                        # exact prefix 2^53 + 1 > 2^53
    assert ref.pick([2.0 ** 53 + 2]).tolist() == [2]
    assert ref.excess(1, 2.0 ** 53) == 1.0 and ref.excess(-1, 5.0) == -5.0
    # 1e30 swallows 1 in float64, not in the exact prefix
    ref = so.Reference([1e30, 1.0, 0.0, 3.0], block=2)
    t = float(np.float32(1e30))
    assert ref.pick([t, t + 0.5]).tolist() == [1, 1]


@pytest.mark.parametrize("seed", range(6))
@pytest.mark.parametrize("block", [1, 3, 2048])
def test_draws_match_rational_arithmetic(seed, block):
    rng = np.random.default_rng(seed)
    n = 60
    m = (10.0 ** rng.uniform(-40, 38, n)).astype(np.float32)
    m[rng.random(n) < 0.3] = 0
    m[:seed] = 0                                                        # leading zeros
    m[-seed - 1:] = 0                                                   # trailing zeros
    if seed % 2:
        m[rng.integers(0, n, 3)] = np.float32(1e-42)                    # subnormals
    if seed == 4:
        m[:] = 0
        m[17] = 3e38
        m[18] = 1e-42
    ref = so.Reference(m, block=block)
    exact = sum(Fraction(float(x)) for x in m.astype(np.float64))
    assert ref.total == float(exact)
    total_k = ref.total * (1 + 40 * 2.0 ** -53)
    U = rng.random(64)
    U[:4] = [0.0, 1.0 - 2.0 ** -53, 0.5, 0.25]
    d = ref.draw(total_k, U, 64)
    for b in range(64):
        u = float(d.u[b])
        assert d.pos[b] == _rational_pick(m, u)
        assert d.lo[b] == _rational_pick(m, u - so.WINDOW * total_k)
        assert d.hi[b] == _rational_pick(m, u + so.WINDOW * total_k)
    # v on the float64 prefixes themselves, each within rounding of a boundary: decided exactly
    inc = np.cumsum(m.astype(np.float64))
    got = ref.pick(inc)
    assert got.tolist() == [_rational_pick(m, float(x)) for x in inc]


def test_weights_are_at_most_one_and_survive_float_range_ratios():
    m = np.array([0.0, 3e38, 1e-42, 1.0, 0.5, 2.5e-4, 0.0], dtype=np.float32)
    ref = so.Reference(m)
    assert ref.m_min == float(np.float32(1e-42)) and ref.n_valid == 5
    for beta in (0.0, 0.4, 1.0, 2.5):
        w = ref.weights(np.flatnonzero(m), beta)
        assert bool((w <= 1.0).all()) and bool((w > 0.0).all())
        assert w[1] == 1.0                                              # the smallest mass
    w = ref.weights([1], 0.4)[0]                                        # ratio ~ 2e80, far past FLT_MAX
    want = (float(np.float32(3e38)) / float(np.float32(1e-42))) ** -0.4
    assert w == want and 1e-33 < w < 1e-31
    assert math.isclose(ref.weights([3], 1.0)[0], float(np.float32(1e-42)), rel_tol=1e-15)
