"""The exact aggregation oracle (``oracle_csr_aggregate_ex_f32``) on the CPU: its fused multiply-adds are correctly rounded
(checked against exact rational arithmetic, including products where fp64-then-fp32 rounds twice), and every form stays
within the fp32 error bound of an fp64 sum.  tests/test_gpu_aggregate_exact.py holds the gather kernel to this oracle bit
for bit, so the oracle itself must be right."""
import zlib
from fractions import Fraction

import numpy as np
import pytest

from oracle import csr_aggregate_c, csr_aggregate_ex

U = 2.0 ** -24


def _round_f32(q: Fraction) -> np.float32:
    """Round an exact rational to fp32, nearest with ties to even (normal range)."""
    f = np.float32(float(q))  # within one fp32 ulp: the answer is f or a neighbour
    cands = [np.nextafter(f, np.float32(-np.inf)), f, np.nextafter(f, np.float32(np.inf))]
    best = min(abs(Fraction(float(c)) - q) for c in cands)
    ties = [c for c in cands if abs(Fraction(float(c)) - q) == best]
    return ties[0] if len(ties) == 1 else next(c for c in ties if int(np.array(c).view(np.uint32)) % 2 == 0)


def _oracle_fma(a, b, c):
    """fmaf(a, b, c) elementwise through the oracle's flush: one edge (acc = 0 + a exactly), row_scale b, addend c."""
    a, b, c = (np.asarray(v, np.float32) for v in (a, b, c))
    n = a.size
    rowptr = np.arange(n + 1, dtype=np.int32)
    col = np.arange(n, dtype=np.int32)
    return csr_aggregate_ex(rowptr, col, a.reshape(n, 1), row_scale=b, addend=c.reshape(n, 1))[:, 0]


def _double_rounding_cases():
    """(a, b, c) whose exact a*b + c lies just off an fp32 midpoint that fp64 rounds onto: float32(float64(a*b + c))
    then breaks the tie the wrong way."""
    out = []
    for i in range(1, 40):
        for sgn in (1.0, -1.0):
            # a*b = 1 + k 2^-12 ... with the 2^-24 bit set: an exact fp32 midpoint; c pushes it off by far less than fp64's ulp
            a = np.float32(1 + i * 2.0 ** -12)
            b = np.float32(1 + 2.0 ** -12)
            p = Fraction(float(a)) * Fraction(float(b))
            for c in (np.float32(2.0 ** -80), np.float32(-(2.0 ** -80))):
                q = p + Fraction(float(c))
                if np.float32(float(q)) != _round_f32(q):
                    out.append((np.float32(sgn * a), b, np.float32(sgn * c)))
    return out


def test_oracle_fma_is_correctly_rounded_on_random_triples():
    rng = np.random.default_rng(0)
    n = 20000
    a = (rng.standard_normal(n) * np.exp2(rng.integers(-20, 20, n))).astype(np.float32)
    b = (rng.standard_normal(n) * np.exp2(rng.integers(-20, 20, n))).astype(np.float32)
    c = (rng.standard_normal(n) * np.exp2(rng.integers(-40, 40, n))).astype(np.float32)
    c[::7] = -(a[::7].astype(np.float64) * b[::7]).astype(np.float32)  # near-total cancellation
    got = _oracle_fma(a, b, c)
    want = np.array([_round_f32(Fraction(float(x)) * Fraction(float(y)) + Fraction(float(z))) for x, y, z in zip(a, b, c)])
    assert np.array_equal(got.view(np.uint32), want.astype(np.float32).view(np.uint32))


def test_oracle_fma_is_not_fooled_by_double_rounding():
    cases = _double_rounding_cases()
    assert len(cases) >= 20
    a, b, c = (np.array(v, np.float32) for v in zip(*cases))
    got = _oracle_fma(a, b, c)
    exact = [Fraction(float(x)) * Fraction(float(y)) + Fraction(float(z)) for x, y, z in cases]
    want = np.array([_round_f32(q) for q in exact], np.float32)
    twice = (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(np.float32)
    assert np.all(twice != want)  # the construction works: fp64 then fp32 is wrong on every case
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


def _random_csr(rng, n_rows, n_src, max_deg):
    deg = rng.integers(0, max_deg + 1, n_rows)
    rowptr = np.concatenate([[0], np.cumsum(deg)]).astype(np.int32)
    col = rng.integers(0, n_src, int(rowptr[-1])).astype(np.int32)
    return rowptr, col


@pytest.mark.parametrize("form", ["sum", "mean", "addend", "scaled_addend", "src_scale", "rectangular"])
def test_oracle_is_within_the_fp32_bound_of_an_fp64_sum(form):
    rng = np.random.default_rng(zlib.crc32(form.encode()))
    n, H = 3000, 24
    n_src = n + 500 if form == "rectangular" else n
    rowptr, col = _random_csr(rng, n, n_src, 40)
    x = rng.standard_normal((n_src, H)).astype(np.float32)
    rs = (rng.standard_normal(n) * 3).astype(np.float32) if form in ("mean", "scaled_addend", "rectangular") else None
    ss = rng.standard_normal(n_src).astype(np.float32) if form == "src_scale" else None
    add = rng.standard_normal((n, H)).astype(np.float32) if form in ("addend", "scaled_addend") else None
    got = csr_aggregate_ex(rowptr, col, x, row_scale=rs, src_scale=ss, addend=add, n_rows=n).astype(np.float64)
    terms = x.astype(np.float64)[col] * (ss.astype(np.float64)[col, None] if ss is not None else 1.0)
    seg = np.repeat(np.arange(n), np.diff(rowptr))
    r = np.zeros((n, H))
    A = np.zeros((n, H))
    np.add.at(r, seg, terms)
    np.add.at(A, seg, np.abs(terms))
    sc = rs.astype(np.float64)[:, None] if rs is not None else 1.0
    r, S = r * sc, A * np.abs(sc)
    if add is not None:
        r, S = r + add, S + np.abs(add)
    deg = np.diff(rowptr).astype(np.float64)[:, None]
    assert np.all(np.abs(got - r) <= (deg + 2) * U * S)
    if form in ("sum", "mean"):  # the plain entry point is the same arithmetic
        assert np.array_equal(csr_aggregate_c(rowptr, col, rs, x), got.astype(np.float32))
