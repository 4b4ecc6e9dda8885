"""CPU tests of the oracle (oracle/spx_oracle.c): it must reproduce every golden vector that
tests/golden/make_golden.py recorded from the original project's src/simplex.py, the record of
tests/golden/fresh_cases.json on further seeded LPs and, where $SIMPLEX_REF points at the
original's sources, the original itself on those LPs.  Bit-exact: pivot sequences, labels and
every fp64 cell.
"""
import hashlib
import json
import os

import numpy as np
import pytest

import oracle
from simplex_method_solver_b200 import workloads as W
from util import (END_TO_STATUS, FRESH_SHARDED_LPS, bits, case_inputs, drive_reference, flat_of, fresh_dantzig_lps,
                  fresh_lps, label_codes, make_lp, table_sha, unhex)


def test_oracle_builds_and_reports_threads():
    oracle.build()
    assert oracle.num_threads() >= 1


def test_all_golden_cases(ref_cases):
    """381 cases: reference examples (simplex.py:205-238), quirks, three random families."""
    assert len(ref_cases) >= 300
    ends = set()
    for case in ref_cases:
        rows, c = case_inputs(case)
        n, m = rows.shape[0], rows.shape[1] - 1
        o = oracle.solve(rows, c, max_pivots=case["cap"])
        ends.add(case["end"])
        assert o.status == END_TO_STATUS[case["end"]], case["name"]
        assert o.trace.tolist() == case["trace"], case["name"]
        assert table_sha(o.table) == case["final_table_sha256"], case["name"]
        rl, cl = oracle.label_strings(o.rowlab, o.collab, m)
        assert rl == case["row_labels"] and cl == case["column_labels"], case["name"]
        if "x1" in case:
            assert float(o.x[0]).hex() == float(float.fromhex(case["x1"])).hex(), case["name"]
            assert float(o.x[1]).hex() == float(float.fromhex(case["x2"])).hex(), case["name"]
            assert float(o.obj2).hex() == case["f"], case["name"]
    assert ends == {"optimal", "incorrect system", "simplex method does not converge", "cap"}


def test_snapshots_match_get_solution(ref_cases):
    """Info.table sequence of get_solution() (simplex.py:181,198) == the oracle's snapshot trace."""
    cases = [c for c in ref_cases if "get_solution" in c]
    assert len(cases) >= 15
    for case in cases:
        rows, c = case_inputs(case)
        o = oracle.solve(rows, c, max_pivots=case["cap"], snapshots=True)
        infos = [e for e in case["get_solution"] if "error" not in e]
        assert len(infos) == o.npiv + 1, case["name"]
        for k, e in enumerate(infos):
            exp = np.concatenate([unhex(e["table"][:-1]).reshape(-1),
                                  np.asarray([float.fromhex(v) for v in e["table"][-1]])])
            assert np.array_equal(bits(o.snaps[k]), bits(exp)), (case["name"], k)
            if e["i"] is not None:
                assert (e["i"], e["j"]) == tuple(o.trace[k]), case["name"]


def test_cfg1_digest(ref_cases):
    case = next(c for c in ref_cases if c["name"] == "ref_example_cfg1_205")
    o = oracle.solve(W.CFG1_ROWS, W.CFG1_C, snapshots=True)
    assert o.trace.tolist() == [[2, 0], [3, 0], [1, 1], [0, 0]]
    n, m = 4, 2
    assert W.snapshot_digest([oracle.unflatten(s, n, m) for s in o.snaps]) == \
        "0599fb0b6881268191a0d0490575cbe5891d0e5f5f7148bd4124e07a0a853183" == case["snapshot_sha256"]
    assert (o.x[0], o.x[1], o.obj2) == (39.18192919380969, 26.096639697976617, -65.2785688917863)


def test_cfg2_prefix(cfg_digests):
    """1000 x 2000: the reference's own first 12 pivots + its table, then the first 100 pivots."""
    g = cfg_digests["cfg2"]
    rows, c = W.dense_lp(1000, 2000, 0)
    assert W.input_digest(rows, c) == g["input_sha256"]
    o = oracle.solve(rows, c, max_pivots=12)
    assert o.trace.tolist() == g["reference_first12"]["trace"]
    assert table_sha(o.table) == g["reference_first12"]["table_sha256_after12"]
    o = oracle.solve(rows, c, max_pivots=100)
    assert o.status == oracle.CAP
    assert W.pivot_digest(o.trace) == g["oracle_full"]["pivot_sha256_after100"]


def test_cfg3_batch(cfg_digests):
    g = cfg_digests["cfg3"]
    T, C = W.gui_batch(65536, 0)
    assert W.input_digest(T, C) == g["input_sha256"]
    res = oracle.solve_batched(W.batch_flat(T, C), 8, 2, max_pivots=64)
    assert (res.status == 0).all() and int(res.npiv.sum()) == g["total_pivots"] == 408212
    hist = {str(k): int(v) for k, v in zip(*np.unique(res.npiv, return_counts=True))}
    assert hist == g["pivot_histogram"]
    assert W.batch_pivot_digest(res.trace, res.npiv) == g["batch_pivot_sha256"]
    assert W.batch_solution_digest(res.x[:, 0], res.x[:, 1], res.obj2) == g["batch_solution_sha256"]


@pytest.mark.parametrize("n", [10, 20])
def test_cfg5_klee_minty(cfg_digests, n):
    g = cfg_digests[f"km{n}"]
    rows, c = W.klee_minty(n)
    o = oracle.solve(rows, c, max_pivots=1 << n)
    assert o.status == 0 and o.npiv == (1 << n) - 1 == g["npiv"]
    assert o.trace[:8].tolist() == g["first8"]
    assert W.pivot_digest(o.trace) == g["pivot_sha256"]
    assert table_sha(o.table) == g["final_table_sha256"]
    assert o.rowlab.tolist() == label_codes(g["row_labels"][:-1], n)
    assert o.collab.tolist() == label_codes(g["column_labels"][:-1], n)
    assert o.x[n - 1] == float(5 ** n) and (o.x[: n - 1] == 0).all()
    assert o.objm == -float(5 ** n)


def test_cfg4_generator_digest_small_sibling(cfg_digests):
    """cfg4's 4.3 GB input is only generated on the GPU box; here: the generator's draw order
    (A, b, c) on a small sibling and the recorded golden trace shape."""
    g = cfg_digests["cfg4"]
    assert len(g["trace"]) >= 200 and g["trace"][0] == [6249, 0] and g["trace"][199] == [5220, 16]
    rows, c = W.dense_lp(8, 16, 0)
    rng = np.random.default_rng(0)
    A = -rng.uniform(0.1, 1.0, (8, 16)); b = rng.uniform(1.0, 2.0, 8) * 16; cc = -rng.uniform(0.1, 1.0, 16)
    assert np.array_equal(rows, np.hstack([A, b[:, None]])) and np.array_equal(c, cc)


# --------------------------------------------------------------------------- fresh LPs: stored record + live reference
@pytest.fixture(scope="module")
def fresh_cases():
    """tests/golden/fresh_cases.json (made by tests/golden/make_fresh_cases.py; its "provenance" says whether the
    original's simplex.py or the oracle computed it)."""
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "fresh_cases.json")) as fh:
        return json.load(fh)


def _assert_recorded(o, rec, m, what):
    assert o.status == END_TO_STATUS[rec["end"]], what
    assert o.trace.tolist() == rec["trace"], what
    assert table_sha(o.table) == rec["table_sha256"], what
    if "row_labels" in rec:
        assert oracle.label_strings(o.rowlab, o.collab, m) == (rec["row_labels"], rec["column_labels"]), what


def _assert_live(o, ref, rows, c, cap, what):
    end, trace, flat, rl, cl = drive_reference(ref, rows, c, cap)
    assert o.status == END_TO_STATUS[end], what
    assert o.trace.tolist() == trace, what
    assert np.array_equal(bits(o.table), bits(flat)), what
    assert oracle.label_strings(o.rowlab, o.collab, rows.shape[1] - 1) == (rl, cl), what


@pytest.mark.parametrize("family", ["gui2dp", "smallint", "dense"])
def test_oracle_equals_live_reference(reference_module, fresh_cases, family):
    """Fresh seeded LPs (not those of reference_cases.json): the oracle against the stored record and, where
    $SIMPLEX_REF is set, against the original's simplex.py itself."""
    recs = fresh_cases["families"][family]
    assert len(recs) == 150
    for t, (rows, c) in enumerate(fresh_lps(family)):
        o = oracle.solve(rows, c, max_pivots=60)
        _assert_recorded(o, recs[t], rows.shape[1] - 1, (family, t))
        if reference_module is not None:
            _assert_live(o, reference_module, rows, c, 60, (family, t))


def test_oracle_pick_update_equal_live_reference_medium(reference_module, fresh_cases):
    """One 60 x 90 dense LP, 25 pivots: every pick (row, column, pivot element) and the whole table after every
    pivot, against the stored record and, where $SIMPLEX_REF is set, against the original's every cell."""
    g = fresh_cases["medium"]
    rows, c = W.dense_lp(g["n"], g["m"], g["seed"])
    assert len(g["pivots"]) == 25
    sm = reference_module.SimplexMethod(rows.tolist(), c.tolist()) if reference_module is not None else None
    T = flat_of(rows, c)
    for k, (i, j, e_hex, sha) in enumerate(g["pivots"]):
        st, r, cc, ee = oracle.pick(T, 60, 90)
        assert st == oracle.PIVOT and (r, cc, float(ee).hex()) == (i, j, e_hex), k
        T = oracle.update(T, 60, 90, r, cc)
        assert table_sha(T) == sha, k
        if sm is not None:
            ok, i, j, e = sm.pick_element()
            assert ok and (i, j, e) == (r, cc, ee)
            sm.recalculate_matrix()
            got = np.asarray([v for row in sm.table for v in row])
            assert np.array_equal(bits(got), bits(T))


@pytest.mark.parametrize("n,m,cap,kind", FRESH_SHARDED_LPS)
def test_oracle_equals_live_reference_on_the_sharded_test_lps(reference_module, fresh_cases, n, m, cap, kind):
    """The LP families the sharded-flow tests use (util.make_lp: entering column on the LAST column block and
    moving between blocks; degenerate small integers), against the stored record and, where $SIMPLEX_REF is set, the
    original's simplex.py, so the oracle those tests compare against is pinned on exactly this kind of input too."""
    rec = next(r for r in fresh_cases["sharded"] if (r["n"], r["m"], r["cap"], r["kind"]) == (n, m, cap, kind))
    rows, c = make_lp(n, m, 7, kind)
    o = oracle.solve(rows, c, max_pivots=cap)
    assert len(rec["trace"]) >= 10
    _assert_recorded(o, rec, m, (n, m, kind))
    if reference_module is not None:
        _assert_live(o, reference_module, rows, c, cap, (n, m, kind))


def test_golden_file_provenance(ref_cases):
    names = [c["name"] for c in ref_cases]
    assert len(set(names)) == len(names)
    assert all(c.get("provenance") == "reference" for c in ref_cases)
    h = hashlib.sha256(repr(sorted(names)).encode()).hexdigest()
    assert len(h) == 64


# --------------------------------------------------------------------------- the idea behind the fused loop (K6)
def test_lazy_replay_of_pending_pivots_is_bit_identical():
    """csrc/spx_fused.cu prices the next F pivots from the STORED table by replaying the pending rank-1
    updates on single cells.  CPU model of that claim: any cell of the table after i pivots, evaluated
    lazily from table 0 with the reference's operation order (simplex.py:156,160,163,173-175), equals the
    materialised cell bit for bit — for pivot rows, pivot columns, pivot cells and ordinary cells alike."""
    rng = np.random.default_rng(21)
    for trial in range(12):
        n, m = int(rng.integers(2, 9)), int(rng.integers(2, 8))
        if trial % 2:
            rows = np.hstack([rng.integers(-3, 4, (n, m)).astype(float), rng.integers(0, 7, (n, 1)).astype(float)])
            c = rng.integers(-3, 1, m).astype(float)
        else:
            rows, c = W.dense_lp(n, m, seed=trial)
        T = flat_of(rows, c)
        w1 = m + 1
        levels, tables = [], [T.copy()]
        for _ in range(6):
            st, r, cc, p = oracle.pick(T, n, m)
            if st != oracle.PIVOT:
                break
            row = T[r * w1: r * w1 + m].copy()                                   # ROW_i: pivot row of table i
            col = np.array([T[i * w1 + cc] for i in range(n)] + [T[n * w1 + cc]])   # COL_i (f row last)
            levels.append((r, cc, p, row, col))
            T = oracle.update(T, n, m, r, cc)
            tables.append(T.copy())

        def lazy(t, j, upto):
            """cell (t, j) of table `upto`, from table 0 (t == n: the f row)."""
            v = tables[0][t * w1 + j] if t < n else tables[0][n * w1 + j]
            for (r, cc, p, row, col) in levels[:upto]:
                with np.errstate(all="ignore"):
                    if t == r:
                        v = np.float64(1.0) / p if j == cc else (-v) / p
                    elif j == cc:
                        v = col[t] / p
                    else:
                        v = (v * p - row[j] * col[t]) / p
            return np.float64(v)

        for upto in range(1, len(levels) + 1):
            Tm = tables[upto]
            for t in range(n + 1):
                for j in range(m):
                    want = Tm[t * w1 + j] if t < n else Tm[n * w1 + j]
                    got = lazy(t, j, upto)
                    assert bits(np.array([got]))[0] == bits(np.array([want]))[0] or (np.isnan(got) and np.isnan(want)), \
                        (trial, upto, t, j, got, want)


# --------------------------------------------------------------------------- the extension entering rule (N4)
def test_dantzig_rule_golden_cases(dantzig_cases):
    """rule="dantzig" of the oracle (most negative f cell, lowest index on ties; everything else the reference's)
    against fixtures the REFERENCE produced under that rule (make_golden.py::drive_dantzig swaps the chosen column
    into position 0, where the reference's own first-negative rule takes it)."""
    assert len(dantzig_cases) >= 150
    differs = 0
    for case in dantzig_cases:
        rows, c = case_inputs(case)
        m = rows.shape[1] - 1
        o = oracle.solve(rows, c, max_pivots=case["cap"], rule="dantzig")
        assert o.status == END_TO_STATUS[case["end"]], case["name"]
        assert o.trace.tolist() == case["trace"], case["name"]
        assert table_sha(o.table) == case["final_table_sha256"], case["name"]
        rl, cl = oracle.label_strings(o.rowlab, o.collab, m)
        assert rl == case["row_labels"] and cl == case["column_labels"], case["name"]
        differs += oracle.solve(rows, c, max_pivots=case["cap"]).trace.tolist() != case["trace"]
    assert differs >= 30                      # the rule really is a different rule on these LPs


def test_dantzig_rule_equals_reference_driven_by_column_swap(reference_module, fresh_cases):
    """Fresh LPs (not in the fixtures) under the extension rule: the oracle against the stored record and, where
    $SIMPLEX_REF is set, against the original driven by make_golden.py's column swap."""
    recs = fresh_cases["dantzig"]
    assert len(recs) == 90
    mg = None
    if reference_module is not None:
        import importlib.util
        spec = importlib.util.spec_from_file_location(
            "make_golden", os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "make_golden.py"))
        mg = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mg)
    for t, (rows, c) in enumerate(fresh_dantzig_lps()):
        o = oracle.solve(rows, c, max_pivots=150, rule="dantzig")
        _assert_recorded(o, recs[t], rows.shape[1] - 1, t)
        if mg is not None:
            sm, trace, end, _ = mg.drive_dantzig(rows.tolist(), c.tolist(), 150)
            assert o.status == END_TO_STATUS[end] and o.trace.tolist() == trace, t
            assert table_sha(o.table) == mg.table_sha(sm.table), t


# --------------------------------------------------------------------------- fixtures bench.py asserts at run time
def test_body_checksum_is_shardable_and_layout_free():
    """workloads.body_checksum_*: numpy (golden side) == torch (device side), strided views, and the column
    shards' checksums add up mod 2^64 to the whole body's."""
    import torch
    rng = np.random.default_rng(5)
    n, m = 70, 333
    big = np.zeros((n + 1, 400))
    big[:, :m] = rng.standard_normal((n + 1, m))
    body = big[:n, :m]
    whole = W.body_checksum_numpy(body)
    bits_ = np.ascontiguousarray(body).view(np.uint64)
    ref = sum(int(bits_[i, j]) * (2 * (i * m + j) + 1) for i in range(n) for j in range(m)) % (1 << 64)
    assert whole == ref
    t = torch.from_numpy(big)
    assert W.body_checksum_torch(t[:n, :m]) == whole
    parts = [W.body_checksum_torch(t[:n, a:b], m_total=m, col0=a) for a, b in ((0, 100), (100, 101), (101, 333))]
    assert sum(parts) % (1 << 64) == whole
    body2 = body.copy()
    body2[3, 7] = np.nextafter(body2[3, 7], 1.0)
    assert W.body_checksum_numpy(body2) != whole


def test_late_lp_golden_of_the_multi_gpu_preflight():
    """tests/golden/late_lp.json (asserted by bench.py at N > 1 before anything is timed) == the oracle today."""
    import json
    import os
    from util import make_lp
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "late_lp.json")) as fh:
        g = json.load(fh)
    rows, c = make_lp(g["n"], g["m"], g["seed"], "late")
    assert W.input_digest(rows, c) == g["input_sha256"]
    o = oracle.solve(rows, c, max_pivots=100000)
    n, m = g["n"], g["m"]
    body = o.table[: n * (m + 1)].reshape(n, m + 1)
    assert (o.status, o.npiv) == (g["status"], g["npiv"]) and o.trace.tolist() == g["trace"]
    assert hashlib.sha256(np.ascontiguousarray(body[:, m]).tobytes()).hexdigest() == g["b_sha256"]
    assert hashlib.sha256(o.table[n * (m + 1):].tobytes()).hexdigest() == g["f_sha256"]
    assert W.body_checksum_numpy(body[:, :m]) == g["body_checksum_u64"]
    assert min(g["owner_changes"].values()) >= 100


def test_cfg4_long_golden_extends_the_2000_pivot_golden(cfg_digests):
    """tests/golden/cfg4_long.json (every timed pivot of bench.py) starts with the round-1 golden, mark for mark."""
    import json
    import os
    here = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    with open(os.path.join(here, "cfg4_long.json")) as fh:
        gl = json.load(fh)
    tr = np.load(os.path.join(here, "cfg4_long_trace.npy"))
    old = cfg_digests["cfg4"]
    assert gl["input_sha256"] == old["input_sha256"] and gl["provenance"] == "oracle"
    assert tr[:2000].tolist() == old["trace"] and gl["npiv"] == len(tr) >= 25000
    for k, mk in old["marks"].items():
        for field in ("pivot_sha256", "b_sha256", "f_sha256"):
            assert gl["marks"][k][field] == mk[field], (k, field)
    for k, mk in gl["marks"].items():
        assert W.pivot_digest(tr[: int(k)]) == mk["pivot_sha256"], k
