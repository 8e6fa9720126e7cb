"""The C-ABI library loads and exports exactly the symbols include/toda_b200.h declares (no GPU needed)."""
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    src = open(os.path.join(ROOT, "include", "toda_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(toda_[a-z0-9_]+)\s*\(", src)))


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as g
    g.build()
    from toda_b200 import _C
    return _C


def test_every_declared_symbol_is_exported_and_bound(built):
    syms = header_symbols()
    assert len(syms) >= 31
    out = subprocess.check_output(["nm", "-D", "--defined-only", built.LIB_PATH], text=True)
    exported = set(re.findall(r" T (toda_[a-z0-9_]+)", out))
    assert set(syms) == exported, (sorted(set(syms) - exported), sorted(exported - set(syms)))
    assert set(syms) == set(built.SIGNATURES), (sorted(set(syms) ^ set(built.SIGNATURES)))
    lib = built.lib()
    for s in syms:
        assert getattr(lib, s) is not None
    assert lib.toda_version() == 100


def test_size_queries_work_without_a_gpu(built):
    lib = built.lib()
    assert lib.toda_index_bytes(4, 41, 1440, 1440) > 4 * 41 * 1440 * 1440 // 8
    assert lib.toda_index_bytes(0, 41, 1440, 1440) == 0
    assert lib.toda_bn_workspace_bytes(128) > 0
    assert lib.toda_spconv_wgrad_workspace_bytes(100000, 100000, 27, 64, 64, 0) >= 27 * 64 * 64 * 4
    grid = built.ints([1440, 1440, 40])
    assert lib.toda_voxelize_workspace_bytes(1200000, 4, grid, 10, 120000) > 0


def test_argument_errors_of_the_entry_points_are_reported(built):
    lib = built.lib()
    rc = lib.toda_mean_vfe_fwd(None, None, 0, 10, 0, 5, None, None)
    assert rc == -1 and b"mean_vfe_fwd" in lib.toda_last_error()
    rc = lib.toda_spconv_fwd(None, None, 0, 0, None, 5, 27, None, 16, None, None, None, None, None, None, None, None, 0, 0, None,
                             None, 0, None, 0, None)
    assert rc == -1


def test_product_never_imports_the_oracle():
    """The product path must not route through oracle/ (or any CPU fallback)."""
    for dirpath, _, files in os.walk(os.path.join(ROOT, "toda_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, flags=re.M), os.path.join(dirpath, f)


def test_ops_fail_loudly_on_cpu_tensors(built):
    import torch
    from toda_b200 import ops
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.mean_vfe(torch.zeros(3, 4, 5), torch.ones(3, dtype=torch.int32))
