"""The one-GPU fused loop at 16 levels per pass (csrc/spx_fused.cu): two groups of 8 levels per pass, one lazy range
test per group, and an in-place first pass when a call's pass count would otherwise leave table k outside buffer
k & 1."""
import ctypes

import numpy as np
import pytest

import oracle
from simplex_method_solver_b200 import workloads as W
from util import END_TO_STATUS, bits, case_inputs, flat_of, table_sha

pytestmark = pytest.mark.gpu

OPT_FUSE_DEPTH, OPT_FUSE_PRICING = 6, 8


@pytest.fixture(scope="module")
def spx():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("GPU tests need a CUDA device")
    from simplex_method_solver_b200 import _native, engine
    _native.lib()

    class NS:
        pass
    ns = NS()
    from simplex_method_solver_b200 import simplex
    ns.torch, ns.N, ns.engine, ns.simplex = torch, _native, engine, simplex
    return ns


def test_depth_option_reads_the_depth_the_loop_uses(spx):
    L = spx.N.lib()
    try:
        assert L.spx_get_option(OPT_FUSE_DEPTH) == 16                       # the default
        assert L.spx_set_option(OPT_FUSE_DEPTH, 8) == 0 and L.spx_get_option(OPT_FUSE_DEPTH) == 8
        for bad in (9, 12, 15, 17, 24, 32, -1):
            assert L.spx_set_option(OPT_FUSE_DEPTH, bad) != 0
        assert L.spx_set_option(OPT_FUSE_DEPTH, 16) == 0 and L.spx_get_option(OPT_FUSE_DEPTH) == 16
    finally:
        L.spx_set_option(OPT_FUSE_DEPTH, 0)
    assert L.spx_get_option(OPT_FUSE_DEPTH) == 16


@pytest.mark.parametrize("pricing", [1, 2])           # the one-CTA and the whole-GPU cooperative pricing kernels
@pytest.mark.parametrize("n,m", [(3, 1), (9, 17), (40, 70), (65, 513), (130, 1030), (257, 100), (40, 2049)])
def test_fused_loop_depth16_bit_exact_ragged_shapes(spx, n, m, pricing):
    """Calls of 1..40 pivots against the oracle: pivot sequence, status and every bit of the whole table after each
    call.  The calls give passes of every length 1..16, odd and even pass counts and in-place first passes (17, 40,
    33 pivots).  5 % exact zeros; small n starts in phase 1."""
    L = spx.N.lib()
    rng = np.random.default_rng(n * 7 + m)
    rows, c = W.dense_lp(n, m, seed=3 * n + m)
    rows[rng.random(rows.shape) < 0.05] = 0.0
    if n >= 9:
        rows[: n // 3, -1] = -np.abs(rows[: n // 3, -1]) - 1.0          # negative b: phase 1 first
    cap = 600
    dev = spx.engine.DeviceTableau(n, m, trace_capacity=cap)
    dev.load(rows, c, max_pivots=cap)
    T = flat_of(rows, c)
    npiv = 0
    assert L.spx_set_option(OPT_FUSE_PRICING, pricing) == 0
    try:
        for k in (16, 1, 17, 40, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 32, 33, 16):
            want = []
            for _ in range(k):
                st, r, cc, e = oracle.pick(T, n, m)
                if st != oracle.PIVOT:
                    break
                want.append([r, cc])
                T = oracle.update(T, n, m, r, cc)
            status, got = dev.solve(stop_after=k, chunk=k, lookahead="fused")
            assert got == npiv + len(want)
            assert dev.trace[npiv:got].cpu().numpy().tolist() == want
            npiv = got
            assert np.array_equal(bits(dev.export_flat(npiv)), bits(T)), (n, m, npiv, k)
            st, r, cc, e = oracle.pick(T, n, m)
            if status == oracle.PIVOT and st != oracle.PIVOT and len(want) == k:
                continue                                 # fused stops unpriced: the next call reports the ending
            assert status == st
            if st != oracle.PIVOT:
                break
    finally:
        L.spx_set_option(OPT_FUSE_PRICING, 0)


@pytest.mark.parametrize("chunk", [16, 17, 40])
@pytest.mark.parametrize("pricing", [1, 2])
def test_reference_cases_fused_depth16(spx, ref_cases, chunk, pricing):
    """The reference's golden cases through the fused loop at depth 16: trace, ending, labels, final table bits."""
    L = spx.N.lib()
    assert L.spx_set_option(OPT_FUSE_PRICING, pricing) == 0
    try:
        for case in ref_cases:
            rows, c = case_inputs(case)
            sm = spx.simplex.SimplexMethod(rows, c, engine="stream")
            sol = sm.solve(max_pivots=case["cap"], chunk=chunk, lookahead="fused")
            assert sol.status == END_TO_STATUS[case["end"]], case["name"]
            assert sol.trace.tolist() == case["trace"], case["name"]
            assert table_sha(sm._dev.export_flat(sm._npiv)) == case["final_table_sha256"], case["name"]
            assert sm.row == case["row_labels"] and sm.column == case["column_labels"], case["name"]
    finally:
        L.spx_set_option(OPT_FUSE_PRICING, 0)


def test_lazy_range_guard_16_level_chains(spx):
    """16-level chains through the self-test kernel's copy of the update kernel's policy (a range test after each group
    of 8 levels, csrc/spx_fused.cu) against the per-level guarded chain, every bit equal.  The growth suites start from
    tiny cells whose multipliers grow by 2^54..2^128 per level: the proof's error bound after 8 levels (2^-484) is
    below the test's 2^-400, after 16 (2^-44) it is not.

    These suites do NOT show that one test at the end of the pass would let a wrong value through: no chain is known
    that does.  The division error of an underflowing level is absolute and stays below 2^-969 / |p|; a level either
    absorbs it or carries it unchanged, so a wrong value that grows past 2^-400 would need every level to land its
    two candidate results on opposite sides of a rounding boundary.  The per-group test is kept because it is what
    the proof covers; these suites check that the policy stays exact."""
    torch = spx.torch
    L = spx.N.lib()
    g = torch.Generator(device="cuda")
    g.manual_seed(20261021)
    F, cnt = 16, 1 << 19

    def rnd(lo_exp, hi_exp, shape):
        numel = int(np.prod(shape))
        mant = torch.randint(0, 1 << 52, (numel,), generator=g, device="cuda", dtype=torch.int64)
        exp = torch.randint(lo_exp, hi_exp + 1, (numel,), generator=g, device="cuda", dtype=torch.int64)
        sign = torch.randint(0, 2, (numel,), generator=g, device="cuda", dtype=torch.int64) << 63
        return (mant | (exp << 52) | sign).view(torch.float64).reshape(shape)

    def growth(e0, step):
        base = torch.arange(F, device="cuda", dtype=torch.int64)[None, :] * step + e0
        jit = torch.randint(-3, 4, (cnt, F), generator=g, device="cuda", dtype=torch.int64)
        e = (base + jit).clamp(1, 2046)
        mant = torch.randint(0, 1 << 52, (cnt, F), generator=g, device="cuda", dtype=torch.int64)
        sign = torch.randint(0, 2, (cnt, F), generator=g, device="cuda", dtype=torch.int64) << 63
        return (mant | (e << 52) | sign).view(torch.float64)

    one = torch.ones((cnt, F), dtype=torch.float64, device="cuda")
    pivots = [rnd(1023 - 2, 1023 + 2, (F,)), rnd(1023 - 100, 1023 + 100, (F,))]
    suites = [(rnd(1023 - 30, 1023 + 30, (cnt,)), rnd(1023 - 30, 1023 + 30, (cnt, F)), rnd(1023 - 30, 1023 + 30, (cnt, F))),
              (rnd(0, 2046, (cnt,)), rnd(0, 2046, (cnt, F)), rnd(0, 2046, (cnt, F)))]
    for e0, step in [(1, 54), (1, 55), (30, 55), (1, 56), (10, 60), (1, 128)]:
        suites.append((rnd(0, 123, (cnt,)), growth(e0, step), one))
    redo_total = 0
    for t0, rj, ci in suites:
        for p in pivots:
            lz = torch.empty(cnt, dtype=torch.float64, device="cuda")
            ref = torch.empty_like(lz)
            redo = ctypes.c_uint64(0)
            rc = L.spx_selftest_lazy_guard(t0.data_ptr(), p.data_ptr(), rj.contiguous().data_ptr(), ci.contiguous().data_ptr(),
                                           F, cnt, lz.data_ptr(), ref.data_ptr(), ctypes.byref(redo),
                                           torch.cuda.current_stream().cuda_stream)
            assert rc == 0
            bad = (lz.view(torch.int64) != ref.view(torch.int64)).nonzero()
            assert bad.numel() == 0, (int(bad.numel()), int(bad[0]))
            redo_total += redo.value
    assert redo_total > 0
