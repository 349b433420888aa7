"""The C-ABI library loads and exports every symbol include/bbk.h declares (no compute calls: no GPU here)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_functions():
    text = open(os.path.join(ROOT, "include", "bbk.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    names = re.findall(r"\b(bbk_[a-z0-9_]+)\s*\(", text)
    return sorted(set(names))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__
    path = __graft_entry__.build()
    return ctypes.CDLL(path)


def test_header_declares_the_expected_entry_points():
    names = _declared_functions()
    for must in ("bbk_hist_pairs", "bbk_possible_pairs", "bbk_fit", "bbk_pvalues", "bbk_bh_qvalues", "bbk_count_band",
                 "bbk_last_error", "bbk_version"):
        assert must in names


def test_library_exports_every_declared_symbol(lib):
    for name in _declared_functions():
        assert hasattr(lib, name), "libbbk.so does not export %s" % name


def test_ctypes_signatures_and_version_match_the_header(lib):
    from blueberry_b200 import _lib
    assert sorted(_lib.SIGNATURES) == _declared_functions()
    lib.bbk_version.restype = ctypes.c_int
    assert lib.bbk_version() == 200


def test_fit_result_struct_matches_header():
    from blueberry_b200 import _lib
    text = open(os.path.join(ROOT, "include", "bbk.h")).read()
    body = text[text.index("typedef struct BbkFitResult"):text.index("} BbkFitResult;")]
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = re.findall(r"\b(?:int32_t|int64_t|double)\s+([a-z_A-Z0-9, \[\]]+);", body)
    flat = []
    for f in fields:
        for part in f.split(","):
            flat.append(re.sub(r"\[.*\]", "", part).strip())
    assert flat == [n for n, _ in _lib.FitResult._fields_]
    assert ctypes.sizeof(_lib.FitResult) == 6 * 4 + 8 + 5 * 8 + 6 * 8 + 8 * 8 + 8


def test_workspace_queries_run_without_a_gpu(lib):
    lib.bbk_fit_workspace_bytes.restype = ctypes.c_size_t
    lib.bbk_fit_workspace_bytes.argtypes = [ctypes.c_int32, ctypes.c_int32]
    assert lib.bbk_fit_workspace_bytes(512, 2001) > 0
    lib.bbk_synth_n_pairs.restype = ctypes.c_int64
    lib.bbk_synth_n_pairs.argtypes = [ctypes.c_int64, ctypes.c_int64]
    assert lib.bbk_synth_n_pairs(49851, 2000) == 97750851       # BASELINE config 2
    assert lib.bbk_synth_n_pairs(4813, 4813) == 11584891        # BASELINE config 1


def test_product_raises_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from blueberry_b200 import _lib
    from blueberry_b200.blueberry import benjamini_hochberg
    with pytest.raises(_lib.BbkError):
        benjamini_hochberg([0.1, 0.2], 2)


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "blueberry_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f
