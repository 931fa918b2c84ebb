"""CPU restatement of the exact fixed-point contraction of the integer statistics path.  TEST INFRASTRUCTURE.

The engine (functionalmf_b200/csrc/stats_i8.cu + i8gemm2.cu) computes the product block of the
sufficient statistics

    out[m, c] = sum_k cnt[m, k] * Z[k, c],      Z[k, (k1, k2)] = F[k, k1] * F[k, k2]   (k2 <= k1, packed)

(the `c * v v^T` sums of factor.py:351-356 and 396-400 with the integer replicate counts as weights)
by writing every column of Z as a fixed-point number against a power-of-two column scale,

    e_c = smallest integer with max_k |Z[k, c]| < 2^e_c,     q[k, c] = rint(Z[k, c] * 2^(54 - e_c)),

splitting q into seven signed base-256 digits (round 1: eight base-128 digits; q and therefore the result are the
same), contracting the digit planes with the counts in exact int32 arithmetic on the int8 tensor cores and
recombining them with ONE rounding:

    out[m, c] = RN( (sum_k cnt[m, k] * q[k, c]) * 2^(e_c - 54) ).

This module states that definition in Python integers, so the device result can be compared bit for bit
(tests/test_gpu_i8.py) and its distance to the exact rational sum bounded (tests/test_fixed_point_oracle.py).
"""
from fractions import Fraction
import numpy as np

FIXBITS = 54
NPLANES = 7
DIGIT_OFFSET = sum(128 * 256 ** s for s in range(NPLANES))      # 0x0080808080808080


def column_exponent(z):
    """smallest e with max|z| < 2^e (0 for an all-zero column)"""
    mx = float(np.abs(z).max()) if len(z) else 0.0
    if mx == 0.0:
        return 0
    m, e = np.frexp(mx)            # mx = m * 2^e, 0.5 <= m < 1  ->  mx < 2^e
    return int(e)


def quantise(z, e):
    """q = rint(z * 2^(54 - e)) as Python integers (ties to even, like the device's cvt.rni)"""
    return [int(np.rint(np.ldexp(float(v), FIXBITS - e))) for v in z]


def digits(q):
    """the seven signed base-256 digits of q, carry-free as on the device: fields of q + sum_s 128 * 256^s, minus 128"""
    qq = q + DIGIT_OFFSET
    assert 0 < qq < 256 ** NPLANES
    return [((qq >> (8 * s)) & 255) - 128 for s in range(NPLANES)]


def recombine(planes):
    """the device's recombination: two int64 Horner sums hi = (D6, D5, D4), lo = (D3..D0), re-split into
    H = hi 2^5 + (lo >> 27) and the low 27 bits of lo - both exactly representable in a double - and ONE rounding
    fma(H, 2^27, l27)"""
    hi = (planes[6] * 256 + planes[5]) * 256 + planes[4]
    lo = ((planes[3] * 256 + planes[2]) * 256 + planes[1]) * 256 + planes[0]
    assert abs(hi) < 2 ** 63 and abs(lo) < 2 ** 63
    H, l27 = hi * 32 + (lo >> 27), lo & (2 ** 27 - 1)          # (Python's >> floors like the device's arithmetic shift)
    assert abs(H) < 2 ** 53 and 0 <= l27 < 2 ** 27
    return H * 2 ** 27 + l27          # exact integer (= hi 2^32 + lo); the device rounds it once when converting


def product_block(F, counts, check_digits=False):
    """counts [m, k] (non-negative integers), F [k, K]  ->  out [m, L] float64, L = K (K + 1) / 2 packed (k1 >= k2).
    check_digits: also go through the seven digit planes and their recombination (slow; the CPU test does)."""
    F = np.asarray(F, dtype=np.float64)
    counts = np.asarray(counts)
    K = F.shape[1]
    out = np.zeros((counts.shape[0], K * (K + 1) // 2))
    c = 0
    for k1 in range(K):
        for k2 in range(k1 + 1):
            z = F[:, k1] * F[:, k2]
            e = column_exponent(z)
            q = quantise(z, e)
            dig = [digits(v) for v in q] if check_digits else None
            for m in range(counts.shape[0]):
                tot = sum(int(cc) * v for cc, v in zip(counts[m], q) if cc)
                if check_digits:
                    planes = [sum(int(cc) * d[s] for cc, d in zip(counts[m], dig) if cc) for s in range(NPLANES)]
                    assert recombine(planes) == tot
                # one rounding: integer -> nearest double (Python's int -> float conversion rounds to nearest even),
                # then an exact power-of-two scaling
                out[m, c] = float(np.ldexp(np.float64(float(tot)), e - FIXBITS))
            c += 1
    return out


def product_block_fast(F, counts):
    """The same definition as product_block for large shapes: q is split as qh 2^27 + ql, the two integer contractions are
    done by float64 BLAS (every partial sum stays far below 2^53, so they are exact), recombined as Python integers and
    rounded once.  tests/test_fixed_point_oracle.py checks it against product_block."""
    F = np.asarray(F, dtype=np.float64)
    cf = np.asarray(counts, dtype=np.float64)
    assert cf.sum(axis=1).max() < 2 ** 24
    K = F.shape[1]
    il = np.tril_indices(K)
    Z = F[:, il[0]] * F[:, il[1]]
    mx = np.abs(Z).max(axis=0)
    e = np.where(mx > 0, np.frexp(np.where(mx > 0, mx, 1.0))[1], 0).astype(np.int64)
    q = np.rint(np.ldexp(Z, (FIXBITS - e)[None, :].astype(np.int32))).astype(np.int64)
    qh, ql = q >> 27, q & (2 ** 27 - 1)
    Sh = (cf @ qh.astype(np.float64)).astype(np.int64)
    Sl = (cf @ ql.astype(np.float64)).astype(np.int64)
    out = np.empty(Sh.shape)
    for m in range(Sh.shape[0]):
        for c in range(Sh.shape[1]):
            tot = int(Sh[m, c]) * 2 ** 27 + int(Sl[m, c])
            out[m, c] = float(np.ldexp(np.float64(float(tot)), int(e[c]) - FIXBITS))
    return out


def exact_product_block(F, counts):
    """the same sums in exact rational arithmetic (list of lists of Fraction)"""
    F = np.asarray(F, dtype=np.float64)
    K = F.shape[1]
    rows = []
    for m in range(len(counts)):
        row = []
        for k1 in range(K):
            for k2 in range(k1 + 1):
                row.append(sum(int(cc) * Fraction(float(a)) * Fraction(float(b))
                               for cc, a, b in zip(counts[m], F[:, k1], F[:, k2]) if cc))
        rows.append(row)
    return rows
