"""CPU: the polynomial maps of csrc/rod_math.cuh (fast-math paths of the CUDA kernels) against high-precision
references on their stated ranges.  The tables are parsed from the header, so a typo in a coefficient or a range
constant fails here, without a GPU."""
import math
import os
import re

import numpy as np
import pytest

mp = pytest.importorskip("mpmath")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HDR = open(os.path.join(ROOT, "gym_softrobot_b200", "csrc", "rod_math.cuh")).read()


def table(name):
    m = re.search(r"#define\s+" + name + r"\s+\{(.*?)\}", HDR, re.S)
    assert m, name
    return [float(x) for x in m.group(1).replace("\\", " ").split(",")]


def const(name):
    m = re.search(name + r"\s*=\s*([0-9.eE+-]+)", HDR)
    assert m, name
    return float(m.group(1))


def horner(c, x):
    p = np.full_like(x, c[-1])
    for k in range(len(c) - 2, -1, -1):
        p = p * x + c[k]
    return p


mp.mp.dps = 40
SINC = lambda q: mp.sin(mp.sqrt(q)) / mp.sqrt(q) if q else mp.mpf(1)
COSC = lambda q: (1 - mp.cos(mp.sqrt(q))) / q if q else mp.mpf(1) / 2


def BEND(u):
    if not u:
        return mp.mpf(1)
    th = 2 * mp.asin(mp.sqrt(u))
    return th / mp.sin(th)


CASES = [  # (table, reference, lo, hi-constant, degree)
    ("SR_COEF_SINC", SINC, 0.0, "kSmallRotQ", 5), ("SR_COEF_COSC", COSC, 0.0, "kSmallRotQ", 5),
    ("SR_COEF_BEND", BEND, 0.0, "kSmallBendU", 13), ("SR_COEF_EXP", mp.exp, None, "kSmallExpZ", 5),
    ("SR_COEF_SINC3", SINC, 0.0, "kNarrowRotQ", 3), ("SR_COEF_COSC3", COSC, 0.0, "kNarrowRotQ", 3),
    ("SR_COEF_BEND7", BEND, 0.0, "kNarrowBendU", 7), ("SR_COEF_BEND9", BEND, 0.0, "kMidBendU", 9),
    ("SR_COEF_EXP3", mp.exp, None, "kNarrowExpZ", 3),
]


@pytest.mark.parametrize("name,ref,lo,hi_name,degree", CASES, ids=[c[0] for c in CASES])
def test_polynomial_map_is_accurate_on_its_range(name, ref, lo, hi_name, degree):
    c = table(name)
    hi = const(hi_name)
    assert len(c) == degree + 1
    lo = -hi if lo is None else lo
    rng = np.random.default_rng(0)
    x = np.concatenate([rng.uniform(lo, hi, 1500), [hi, lo if lo else hi * 1e-12, 0.5 * (lo + hi)]])
    got = horner(c, x)
    want = np.array([float(ref(mp.mpf(float(v)))) for v in x])
    # <= 1 ulp of fit error (header claim) + the rounding of a plain double Horner evaluation without FMA
    assert np.abs(got / want - 1.0).max() < 6e-16, (name, np.abs(got / want - 1.0).max())


def test_ranges_are_nested_and_match_the_documented_angles():
    assert const("kNarrowRotQ") < const("kSmallRotQ") and const("kNarrowBendU") < const("kMidBendU") < const("kSmallBendU")
    assert const("kNarrowExpZ") < const("kSmallExpZ")
    deg = lambda u: math.degrees(2 * math.asin(math.sqrt(u)))
    assert abs(deg(const("kNarrowBendU")) - 23.1) < 0.1 and abs(deg(const("kMidBendU")) - 36.9) < 0.1 and abs(deg(const("kSmallBendU")) - 60.0) < 1e-9


def test_lean_kernel_maps():
    """Tables of the lean kernel (rod_kernel_lean.cuh): the trace-free bend map in w2 = 4 sin^2(theta) with the
    reference's 1e-10 guard inside, and sin(t)/t, (1 - cos t)/t^2 with exact leading constants."""
    rng = np.random.default_rng(1)
    # bend: theta'/sin(theta'), theta' = acos(cos(theta) - 1e-10), as a function of w2
    c, hi = table("SR_COEF_BENDW"), const("kNarrowBendW2")
    assert len(c) == 10
    w2 = np.concatenate([rng.uniform(0, hi, 1500), [0.0, hi, 1e-12, 1e-6]])
    def ref(w):
        th = mp.acos(mp.sqrt(1 - mp.mpf(float(w)) / 4) - mp.mpf("1e-10"))
        return float(th / mp.sin(th))
    want = np.array([ref(w) for w in w2])
    assert np.abs(horner(c, w2) / want - 1.0).max() < 8e-16
    cm, him = table("SR_COEF_BENDW_MID"), const("kMidBendW2")        # plane models: 37 degrees, degree 13
    assert len(cm) == 14 and abs(him - 4 * np.sin(np.deg2rad(37.0)) ** 2) < 1e-3
    w2m = np.concatenate([rng.uniform(0, him, 1500), [0.0, him, 1e-12, 1e-6]])
    assert np.abs(horner(cm, w2m) / np.array([ref(w) for w in w2m]) - 1.0).max() < 1.5e-15
    # the range is the same 23.07 degrees as the u-based narrow map: w2 = 4 sin^2(theta) = 16 u (1 - u)
    u = const("kNarrowBendU")
    assert abs(16 * u * (1 - u) - hi) < 1e-12
    # rotation maps
    q = np.concatenate([rng.uniform(0, const("kNarrowRotQ"), 1500), [const("kNarrowRotQ"), 1e-14]])
    g, h = table("SR_COEF_SINCG"), table("SR_COEF_COSCH")
    assert len(g) == 3 and len(h) == 3
    A = 1.0 + q * horner(g, q)
    B = 0.5 + q * horner(h, q)
    wantA = np.array([float(SINC(mp.mpf(float(v)))) for v in q])
    wantB = np.array([float(COSC(mp.mpf(float(v)))) for v in q])
    assert np.abs(A / wantA - 1.0).max() < 1.5e-15 and np.abs(B / wantB - 1.0).max() < 6e-16
    # the damper's quadratic drops z^3 / 6
    assert const("kLeanExpZ") ** 3 / 6 < 1.5e-15
    # the lean kernels test a range on the high 32 bits of the argument only (hi_abs(x) > lim_hi, rod_kernel_lean.cuh),
    # so the polynomials also run on the largest double that shares the limit's high word (2^-20 relative beyond it)
    q = top_of_high_word(const("kNarrowRotQ"))
    assert abs(1.0 + q * horner(g, q) - float(SINC(mp.mpf(q)))) / float(SINC(mp.mpf(q))) < 1.5e-15
    assert abs(0.5 + q * horner(h, q) - float(COSC(mp.mpf(q)))) / float(COSC(mp.mpf(q))) < 6e-16
    w = top_of_high_word(hi)
    assert abs(horner(c, w) / ref(w) - 1.0) < 8e-16
    w = top_of_high_word(him)
    assert abs(horner(cm, w) / ref(w) - 1.0) < 1.5e-15


def top_of_high_word(x):
    """The largest double whose high 32 bits are those of x (x > 0)."""
    b = np.array([x]).view(np.uint64) | np.uint64(0xFFFFFFFF)
    return float(b.view(np.float64)[0])
