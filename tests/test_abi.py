"""CPU tests of the drop-in boundary: libspx_b200.so loads without a GPU, exports every symbol
include/spx_b200.h declares, the Python mirror of spx_state matches the header, and the product
package neither imports the oracle nor falls back to a CPU path.
"""
import ctypes
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "spx_b200.h")
PKG = os.path.join(ROOT, "simplex_method_solver_b200")


def header_symbols():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(spx_[a-z0-9_]+)\s*\(", text)))


@pytest.fixture(scope="module")
def native():
    import __graft_entry__ as entry
    entry.build()
    from simplex_method_solver_b200 import _native
    return _native


def test_library_exports_every_declared_symbol(native):
    L = native.load()
    syms = header_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(L, s), f"{s} declared in include/spx_b200.h but not exported"
    # the ctypes binding covers exactly the header
    assert sorted(native.SIGNATURES) == syms


def test_dynamic_symbol_table_has_no_mangled_entry_points(native):
    out = subprocess.run(["nm", "-D", "--defined-only", native.LIB_PATH], capture_output=True, text=True).stdout
    exported = {ln.split()[-1] for ln in out.splitlines() if " T " in ln}
    for s in header_symbols():
        assert s in exported


def test_abi_constants_and_state_layout(native):
    L = native.load()
    text = open(HEADER).read()
    assert L.spx_version() == int(re.search(r"#define SPX_ABI_VERSION (\d+)", text).group(1))
    assert L.spx_state_bytes() == ctypes.sizeof(native.SpxState) == 128
    for name, val in (("SPX_PIVOT", native.PIVOT), ("SPX_OPTIMAL", native.OPTIMAL),
                      ("SPX_INCORRECT", native.INCORRECT), ("SPX_NOCONV", native.NOCONV),
                      ("SPX_CAP", native.CAP)):
        assert int(re.search(rf"#define {name}\s+(-?\d+)", text).group(1)) == val
    # pure host helpers need no device
    assert L.spx_ld(1) == 16 and L.spx_ld(16) == 16 and L.spx_ld(17) == 32 and L.spx_ld(32768) == 32768
    assert L.spx_cells(4, 2) == 14 and L.spx_cells(16384, 32768) == 536920064
    assert L.spx_colbuf_doubles(16384) >= 16385
    assert L.spx_shard_msg_doubles(16384) % 16 == 0 and L.spx_shard_msg_doubles(16384) >= 16389
    assert L.spx_batched_max_cells() >= 440
    assert L.spx_batched_fits(4, 2) == 1 and L.spx_batched_fits(72, 136) == 1 and L.spx_batched_fits(1, 4470) == 0
    assert L.spx_batched_fits(0, 2) == 0 and L.spx_batched_fits(100, 100) == 0
    smem, cluster, glob = native.ENGINE_SMEM, native.ENGINE_CLUSTER, native.ENGINE_GLOBAL
    assert L.spx_batched_route(4, 2, native.ENGINE_AUTO) == smem and L.spx_batched_route(1, 4470, 0) == cluster
    assert L.spx_batched_route(529, 800, native.ENGINE_AUTO_GLOBAL) == glob and L.spx_batched_route(4, 2, glob) == glob
    for n, m, engine in ((529, 800, 0), (0, 2, 0), (4, 2, 3), (4, 2, 6)):
        assert L.spx_batched_route(n, m, engine) == -1 and L.spx_last_error()
    assert L.spx_launch_count(1) >= 0 and L.spx_launch_count(0) == 0


def test_host_side_layout_helpers_agree_with_python(native):
    """Sizes the Python plumbing derives itself must match the library's (no device needed)."""
    L = native.load()
    for n in (9, 1000, 16384):
        msgd = L.spx_shard_msg_doubles(n)
        for world in (1, 2, 8):
            # parallel.PeerMailboxes: gathered[2][world][msg] | flags[2][world]
            flags_offset = (2 * world * msgd * 8 + 127) // 128 * 128
            assert L.spx_mailbox_bytes(n, world) == flags_offset + (2 * world * 8 + 127) // 128 * 128
            assert L.spx_fshard_xbox_bytes(n, world) > 3 * 8 * world * (n + 1) * 8      # 3 plane sets of 8 levels
        assert L.spx_mailbox_bytes(n, 17) == -1 and L.spx_fshard_xbox_bytes(n, 17) == -1
        for m in (2, 2000, 32768):
            assert L.spx_fused_workspace_bytes(n, m) >= 2 * 8 * L.spx_ld(m) * 8 + 8 * L.spx_colbuf_doubles(n) * 8
            assert L.spx_solve_workspace_bytes(n) >= 128 + (n + 1) * 8 + msgd * 8
    assert native.LOOP_MODES[None] == 0 and native.LOOP_MODES["fused"] == 4 and native.LOOP_MODES[True] == 2


def test_options_validate_ranges_and_reject_retired_keys(native):
    L = native.load()
    try:
        assert L.spx_get_option(11) == 0 and L.spx_get_option(7) == 0 and L.spx_get_option(12) == 0   # defaults
        for k in (1, 3, 4, 10, 15):                                                  # retired keys: rejected, read 0
            for v in (0, 1, 2):
                assert L.spx_set_option(k, v) != 0
            assert L.spx_get_option(k) == 0
        assert L.spx_set_option(11, 40) == 0 and L.spx_get_option(11) == 40        # rows per warp strip: multiples of 8
        assert L.spx_set_option(11, 12) != 0 and L.spx_set_option(11, 4104) != 0
        assert L.spx_set_option(12, 2) == 0 and L.spx_set_option(12, 3) != 0       # column pairs per lane: 1 or 2
        assert L.spx_set_option(6, 9) != 0 and L.spx_set_option(99, 0) != 0
    finally:
        L.spx_set_option(11, 0)
        L.spx_set_option(12, 0)


def test_argument_validation_reports_text(native):
    """Entry points reject bad arguments before touching the device (no GPU needed)."""
    L = native.load()
    rc = L.spx_pick(None, None, 4, 2, 16, 0, 0, None, None, None)
    assert rc < 0 and b"null" in L.spx_last_error()
    rc = L.spx_solve_batched(None, 1, 4, 2, 7, 10, None, None, None, None, None, None, None, None, None)
    assert rc < 0
    rc = L.spx_import_shard(None, None, None, None, 1, 1, 0, 1, 16, None)
    assert rc < 0


def test_no_cpu_fallback_without_a_device(native):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    from simplex_method_solver_b200.simplex import SimplexMethod
    from simplex_method_solver_b200.batched import solve_batched
    import numpy as np
    with pytest.raises(native.NativeUnavailable):
        SimplexMethod([[-1.0, -1.0, 10.0]], [-1.0, -5.0])
    with pytest.raises(native.NativeUnavailable):
        solve_batched(np.zeros((1, 14)), 4, 2)
    with pytest.raises(native.NativeUnavailable):
        native.lib()


def test_product_never_imports_the_oracle():
    """oracle/ is test infrastructure: nothing under the package may import, link or execute it."""
    for dirpath, _, files in os.walk(PKG):
        for f in files:
            if not f.endswith((".py", ".cu", ".cuh", ".h")):
                continue
            text = open(os.path.join(dirpath, f), errors="replace").read()
            assert not re.search(r"^\s*(import|from)\s+oracle\b", text, flags=re.M), f
            assert "liborc" not in text and "spx_oracle" not in text, f
    code = ("import sys; sys.path.insert(0, %r); import simplex_method_solver_b200.simplex, "
            "simplex_method_solver_b200.parallel, simplex_method_solver_b200.batched; "
            "assert 'oracle' not in sys.modules" % ROOT)
    subprocess.run([sys.executable, "-c", code], check=True)


def test_missing_library_fails_loudly(native, monkeypatch):
    monkeypatch.setattr(native, "_lib", None)
    monkeypatch.setattr(native, "LIB_PATH", os.path.join(PKG, "csrc", "does_not_exist.so"))
    with pytest.raises(native.NativeUnavailable):
        native.load()
