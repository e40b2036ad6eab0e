"""No-GPU checks of the drop-in boundary: the C-ABI library loads here and exports every symbol
``include/hrag_b200.h`` declares; the product fails loudly without a device (no CPU fallback)."""
import ctypes
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "hrag_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(hrag_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from hipporag_b200 import _lib
    lib = _lib.load()
    names = _declared_symbols()
    assert len(names) >= 15
    for n in names:
        assert hasattr(lib, n), f"libhrag_b200.so does not export {n}"
    assert sorted(_lib.SIGNATURES) == names, "ctypes SIGNATURES out of sync with include/hrag_b200.h"
    assert b"sm_100a" in lib.hrag_version()


def test_no_cpu_fallback_without_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is visible")
    from hipporag_b200 import Engine, HragError
    with pytest.raises(HragError, match="no CUDA device|CUDA"):
        Engine(0)


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "hipporag_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f"{f} imports oracle/"


def test_native_code_reads_only_the_exchange_switches():
    """Kernel variants are chosen by the code, not by environment switches: the only variables the native
    library reads are the two of the multi-GPU exchange."""
    csrc = os.path.join(ROOT, "hipporag_b200", "csrc")
    names = set()
    for f in os.listdir(csrc):
        if f.endswith((".cu", ".cuh", ".h")):
            names |= set(re.findall(r'getenv\(\s*"([^"]+)"', open(os.path.join(csrc, f)).read()))
    assert names == {"HRAG_K5_MODE", "HRAG_MIXED_PERSIST"}


def test_transition_csr_matches_oracle_restating():
    from hipporag_b200.engine import build_transition_csr
    from oracle import ppr
    rng = np.random.default_rng(0)
    n = 50
    src, dst = rng.integers(0, n - 2, 300), rng.integers(0, n - 2, 300)
    w = rng.random(300) - 0.1            # some non-positive weights
    keep = src != dst
    src, dst, w = src[keep], dst[keep], w[keep]
    row_ptr, col, val = build_transition_csr(n, src, dst, w)
    P, _ = ppr.transition_matrix(ppr.symmetric_weights(n, src, dst, w))
    P.eliminate_zeros()
    assert np.array_equal(row_ptr, P.indptr) and np.array_equal(col, P.indices)
    np.testing.assert_allclose(val, P.data, rtol=1e-7)


def test_shard_rows_partition():
    from hipporag_b200.engine import shard_rows
    for n, world in ((10, 3), (1000, 8), (7, 8), (16, 2)):
        parts = [shard_rows(n, r, world) for r in range(world)]
        assert parts[0][0] == 0 and parts[-1][1] == n
        for a, b in zip(parts, parts[1:]):
            assert a[1] == b[0]
        chunk = -(-n // world)
        assert all(hi - lo <= chunk for lo, hi in parts)
