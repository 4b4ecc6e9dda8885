"""An exact model of the one-GPU fused update's two-operation quotient (csrc/spx_fused.cu, two_op_flag) — test
infrastructure only.

A binary format with a `t`-bit significand and an unbounded exponent; every operation is exact in `Fraction` and
rounded once to nearest-even by ``rn``.  For a divisor p: yh = RN(1/p), yl = RN((1 - p yh) yh) (the device forms the
residual with one fma, which is exact), and q = RN(a yh + RN(a yl)) is the two-operation quotient of a.

``candidates`` lists the numerators in [1, 2) that the device checks, by the device's method (the inverse of the odd
part of the significand modulo a power of two); ``candidates_brute`` lists the same set from the definition.
``device_flag`` restates the device check in double precision (t = 53) step by step.
"""
from fractions import Fraction


def rn(x: Fraction, t: int) -> Fraction:
    """x rounded to nearest-even with a t-bit significand (no exponent range)."""
    if x == 0:
        return Fraction(0)
    s = -1 if x < 0 else 1
    x = abs(x)
    num, den = x.numerator, x.denominator
    e = num.bit_length() - den.bit_length()          # 2^e <= x < 2^(e+2)
    if (num << max(0, -e)) < (den << max(0, e)):
        e -= 1                                      # now 2^e <= x < 2^(e+1)
    sh = t - 1 - e                                  # x * 2^sh in [2^(t-1), 2^t)
    n2, d2 = (num << sh, den) if sh >= 0 else (num, den << -sh)
    qi, r = divmod(n2, d2)
    if 2 * r > d2 or (2 * r == d2 and qi & 1):
        qi += 1
    return s * (Fraction(qi) / (Fraction(2) ** sh) if sh >= 0 else Fraction(qi) * (Fraction(2) ** -sh))


def reciprocal_pair(p: Fraction, t: int):
    yh = rn(1 / p, t)
    e = 1 - p * yh
    assert rn(e, t) == e, "the residual 1 - p yh must be exact"
    return yh, rn(e * yh, t)


def two_op(a: Fraction, yh: Fraction, yl: Fraction, t: int) -> Fraction:
    return rn(a * yh + rn(a * yl, t), t)


def significand(p: Fraction, t: int) -> int:
    """|p| = P 2^k with P in [2^(t-1), 2^t)."""
    p = abs(p)
    P = p
    while P >= 2 ** t:
        P /= 2
    while P < 2 ** (t - 1):
        P *= 2
    assert P.denominator == 1
    return int(P)


def n_of(A: int, P: int, t: int, q_lo: Fraction, q_hi: Fraction):
    """N = 2^S A - (2M + 1) P for the midpoint between the adjacent quotients q_lo < q_hi of A / P."""
    S = t if A >= P else t + 1
    mid = (q_lo + q_hi) / 2
    odd = mid * 2 ** S
    assert odd.denominator == 1 and int(odd) % 2 == 1
    return 2 ** S * A - int(odd) * P


def candidates(P: int, t: int, K: int):
    """The device's enumeration (two_op_candidates) for a t-bit significand P: the A with 0 < |N| <= K."""
    s = (P & -P).bit_length() - 1
    Po = P >> s
    inv = Po
    for _ in range(7):
        inv = (inv * (2 - Po * inv)) % (1 << 128)
    out = set()
    for N in range(-K, K + 1):
        if N == 0 or ((abs(N) & -abs(N)).bit_length() - 1) != s:
            continue
        No = N >> s
        for S in (t, t + 1):
            w = S - s
            mask = (1 << w) - 1
            r = (-No * inv) & mask
            mm = (1 << t) + ((r - (1 << t)) & mask)
            while mm < (1 << (t + 1)):
                num = mm * Po + No
                assert num % (1 << w) == 0
                A = num >> w
                if (1 << (t - 1)) <= A < (1 << t) and (S == t) == (A >= P):
                    out.add(A)
                mm += 1 << w
    return out


def candidates_brute(P: int, t: int, K: int):
    """The same set from the definition: every A, its nearest midpoint of A / P."""
    out = set()
    for A in range(1 << (t - 1), 1 << t):
        S = t if A >= P else t + 1
        x = Fraction(2 ** S * A, P)                 # the quotient in units of 2^-S; midpoints at odd integers
        odd = int(x)
        if odd % 2 == 0:
            odd = odd + 1 if x - odd > 0 else odd - 1
        if not (1 << t) <= odd < (1 << (t + 1)):
            continue
        N = 2 ** S * A - odd * P
        if 0 < abs(N) <= K:
            out.add(A)
    return out


def device_flag(p: float, K: int = 16, span: int = 100) -> bool:
    """two_op_flag restated on the host in double precision: the two-operation quotient against RN(a / p) (what
    pivot_div returns) on every candidate of the device's enumeration."""
    t = 53
    if not 2.0 ** -span <= abs(p) < 2.0 ** (span + 1):         # the lazy guard's span (NaN fails it too)
        return False
    pf = Fraction(p)
    yh, yl = reciprocal_pair(pf, t)
    for A in candidates(significand(pf, t), t, K):
        a = Fraction(A, 1 << 52)
        if two_op(a, yh, yl, t) != rn(a / pf, t):
            return False
    return True
