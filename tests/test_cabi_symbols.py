"""CPU: the C-ABI library builds, loads, and exports every symbol include/treegp_b200.h declares
(no compute calls: there is no GPU here)."""
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    text = open(os.path.join(ROOT, "include", "treegp_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(tgp_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from treegp_b200 import _cabi

    lib = _cabi.load()
    names = _declared()
    assert len(names) >= 14
    for name in names:
        assert hasattr(lib, name), name
        assert name in _cabi.SIGNATURES, "binding missing for %s" % name
    assert sorted(_cabi.SIGNATURES) == names
    assert lib.tgp_abi_version() == _cabi.ABI_VERSION
    assert lib.tgp_pairbin_tile() == 32


def test_invalid_arguments_are_rejected_without_a_gpu():
    """Argument validation happens before any CUDA call."""
    import ctypes
    from treegp_b200 import _cabi

    lib = _cabi.load()
    bad = _cabi.TgpKernel(99, 2, 1.0, 1.0, 0.0, 1.0)
    rc = lib.tgp_kmat_sym(None, 10, ctypes.byref(bad), None, None, 10, 0, None)
    assert rc == -1
    assert b"kernel descriptor" in lib.tgp_last_error()
    ok = _cabi.TgpKernel(0, 2, 1.0, 1.0, 0.0, 1.0)
    assert lib.tgp_kmat_sym(None, 10, ctypes.byref(ok), None, None, 4, 0, None) == -1  # ld < N
    assert lib.tgp_potrf(ctypes.c_void_p(16), 10, 11, ctypes.c_void_p(16), None) == -1  # odd ld
    # envelope forms: one row_end entry per tgp_envelope_block() columns, no NULL envelope
    import numpy as np
    assert lib.tgp_envelope_block() == 512
    re2 = np.array([1000, 1000], dtype=np.int64)
    A16, i16 = ctypes.c_void_p(16), ctypes.c_void_p(16)
    assert lib.tgp_potrf_env(A16, 1000, 1000, None, 2, 0, i16, None) == -1
    assert b"row_end" in lib.tgp_last_error()
    assert lib.tgp_potrf_env(A16, 1000, 1000, ctypes.c_void_p(re2.ctypes.data), 3, 0, i16, None) == -1   # 2 blocks, not 3
    assert lib.tgp_potrf_env(A16, 1000, 1001, ctypes.c_void_p(re2.ctypes.data), 2, 0, i16, None) == -1   # odd ld
    assert lib.tgp_trsm_rows_env(A16, 1000, 1000, ctypes.c_void_p(re2.ctypes.data), 1, A16, 4, 1000, None) == -1
    assert lib.tgp_loglike_env(A16, A16, A16, 1000, ctypes.byref(ok), A16, 1000, A16, 0, A16, i16, None, 2, None) == -1
    assert lib.tgp_predict_var_env(A16, 4, A16, 1000, ctypes.byref(ok), A16, 1000, None, 2, A16, 128, A16, None) == -1


def test_set_option_knows_only_the_pair_count_switches():
    """The four switches of the pair counts are accepted (and set back to their defaults); any other name is an
    unknown option, including the retired Cholesky, GEMM and sweep selections."""
    from treegp_b200 import _cabi

    lib = _cabi.load()
    for name in ("potrf_fused", "potrf_lookahead", "potrf_ob", "potrf_env_lookahead", "gemm_config", "trsv_cluster",
                 "no_such_option"):
        assert lib.tgp_set_option(name.encode(), 0) == -1, name
        assert b"unknown option" in lib.tgp_last_error()
    assert lib.tgp_set_option(None, 0) == -1
    for name, default in (("pairbin_block_sums", 1), ("pairbin_fast_paths", 7), ("pairbin_record_cap", 0),
                          ("bootbin_paths", 15)):
        assert lib.tgp_set_option(name.encode(), default) == 0, name


def test_product_path_does_not_import_the_oracle():
    """The oracle is test infrastructure: nothing under treegp_b200/ may reference it."""
    pkg = os.path.join(ROOT, "treegp_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f
                assert "oracle/_build" not in src and "libpairbin_oracle" not in src, f


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    from treegp_b200 import _cabi

    monkeypatch.setattr(_cabi, "_lib", None)
    monkeypatch.setattr(_cabi, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(_cabi.TgpError):
        _cabi.load()
