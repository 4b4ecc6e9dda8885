"""The two-operation quotient of the one-GPU fused update (csrc/spx_fused.cu, two_op_flag and lazy_level_two_np).

CPU: in reduced precisions every (a, p) pair is checked exhaustively against the exact model (tests/two_op_model.py):
every pair whose two-operation quotient is not RN(a / p) must be a candidate at the K the device uses, and the
device's enumeration of candidates must equal the definition's.  In double precision a seeded sample of divisors gets
the same flags from the host restatement of the device check as from an independent statement.
GPU: the device flags against the host restatement, and the flagged quotients against div.rn.f64.
"""
import ctypes
import random
from fractions import Fraction

import numpy as np
import pytest

import two_op_model as M

K_DEVICE = 16


@pytest.mark.parametrize("t", [7, 8, 9, 10])
def test_every_failing_pair_is_a_candidate(t):
    fails = flagged = 0
    for P in range(1 << (t - 1), 1 << t):
        p = Fraction(P)
        yh, yl = M.reciprocal_pair(p, t)
        cand = M.candidates(P, t, K_DEVICE)
        assert cand == M.candidates_brute(P, t, K_DEVICE), P
        bad = set()
        for A in range(1 << (t - 1), 1 << t):
            q2, q = M.two_op(Fraction(A), yh, yl, t), M.rn(Fraction(A, P), t)
            if q2 != q:
                lo, hi = min(q, q2), max(q, q2)
                N = M.n_of(A, P, t, lo, hi)                                  # asserts they are adjacent
                assert 0 < abs(N) <= 6, (P, A, N)                           # the error bound: |N| < 6
                bad.add(A)
        assert bad <= cand, (P, sorted(bad - cand))
        fails += len(bad)
        # the flag: every candidate agrees  =>  no pair of this divisor fails
        ok = all(M.two_op(Fraction(A), yh, yl, t) == M.rn(Fraction(A, P), t) for A in cand)
        assert not (ok and bad)
        flagged += ok
    assert fails > 0 and flagged > 0


def _sample_divisors(rng, count):
    out = []
    for k in range(count):
        mant = rng.getrandbits(52)
        if k % 4 == 1:
            mant &= ~((1 << rng.randrange(1, 53)) - 1)      # trailing zeros, down to powers of two
        e = rng.randrange(1023 - 100, 1023 + 101)
        bits = (rng.getrandbits(1) << 63) | (e << 52) | mant
        out.append(float(np.array([bits], dtype=np.uint64).view(np.float64)[0]))
    return out


def _independent_flag(p, K=K_DEVICE):
    """The flag from the definition: pow() for the inverse, candidates from the congruence per odd N', and the
    exact quotient."""
    t = 53
    if not 2.0 ** -100 <= abs(p) < 2.0 ** 101:
        return False
    pf = Fraction(p)
    P = M.significand(pf, t)
    s = (P & -P).bit_length() - 1
    Po = P >> s
    yh, yl = M.reciprocal_pair(pf, t)
    for No in range(-(K >> s) | 1, (K >> s) + 1, 2):
        if No == 0 or abs(No << s) > K:
            continue
        for S in (t, t + 1):
            w = S - s
            r = (-No * pow(Po, -1, 1 << w)) % (1 << w)
            for mm in range(r, 1 << (t + 1), 1 << w):
                if mm < (1 << t):
                    continue
                A, rem = divmod(mm * Po + No, 1 << w)
                assert rem == 0
                if (1 << (t - 1)) <= A < (1 << t) and (S == t) == (A >= P):
                    a = Fraction(A, 1 << 52)
                    if M.two_op(a, yh, yl, t) != M.rn(a / pf, t):
                        return False
    return True


def test_double_precision_flags_match_the_statement():
    rng = random.Random(20261022)
    ps = _sample_divisors(rng, 600) + [1.0, -2.0, 0.75, 3.0, 2.0 ** -100, -(2.0 ** 100), 2.0 ** 101, 2.0 ** -101]
    flags = [M.device_flag(p) for p in ps]
    assert flags == [_independent_flag(p) for p in ps]
    share = sum(flags[:600]) / 600
    assert share > 0.9, share                                 # the model: about 97 % of random divisors
    assert M.device_flag(1.0) and not M.device_flag(2.0 ** 101)


@pytest.fixture(scope="module")
def cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("GPU tests need a CUDA device")
    from simplex_method_solver_b200 import _native
    return torch, _native.lib()


@pytest.mark.gpu
def test_device_flags_and_quotients(cuda):
    """About 10^6 divisors (random, trailing zeros, powers of two, both signs, exponents within 2^+-100 and just
    outside): the device flags of a seeded subset equal the host restatement's, and every flagged divisor's quotient
    equals div.rn.f64 on every candidate at K = 64 and on 1,200 pseudo-random numerators (over 2^30 in all)."""
    torch, L = cuda
    rng = random.Random(7)
    host = _sample_divisors(rng, 4000) + [2.0 ** k for k in range(-102, 103)] + [-(2.0 ** k) for k in range(-102, 103)]
    g = torch.Generator(device="cuda")
    g.manual_seed(20261022)
    cnt = 1 << 20
    mant = torch.randint(0, 1 << 52, (cnt,), generator=g, device="cuda", dtype=torch.int64)
    tz = torch.randint(0, 53, (cnt,), generator=g, device="cuda", dtype=torch.int64)
    mant = torch.where(torch.arange(cnt, device="cuda") % 4 == 1, (mant >> tz) << tz, mant)
    exp = torch.randint(1023 - 100, 1023 + 101, (cnt,), generator=g, device="cuda", dtype=torch.int64)
    sign = torch.randint(0, 2, (cnt,), generator=g, device="cuda", dtype=torch.int64) << 63
    rnd = (mant | (exp << 52) | sign).view(torch.float64)
    p = torch.cat([torch.tensor(host, dtype=torch.float64, device="cuda"), rnd])
    flags = torch.empty(p.numel(), dtype=torch.int32, device="cuda")
    bad = ctypes.c_uint64(0)
    rc = L.spx_selftest_two_op(p.data_ptr(), p.numel(), 1200, flags.data_ptr(), ctypes.byref(bad),
                               torch.cuda.current_stream().cuda_stream)
    assert rc == 0
    assert bad.value == 0
    f = flags.cpu().numpy()
    assert f[:len(host)].tolist() == [int(M.device_flag(x)) for x in host]
    share = float(f[len(host):].mean())
    assert share > 0.9, share
