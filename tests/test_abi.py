"""The C-ABI library builds for sm_100a, loads without a GPU and exports every symbol include/sentio_b200.h declares."""
import ctypes
import os
import re

import pytest

from conftest import ROOT


def _header_symbols():
    text = open(os.path.join(ROOT, "include", "sentio_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(sb_[a-z0-9_]+)\s*\(", text)))


def test_header_declares_the_expected_surface():
    syms = _header_symbols()
    for must in ["sb_create", "sb_destroy", "sb_last_error", "sb_dense_load", "sb_dense_topk", "sb_dense_topk_dev",
                 "sb_bm25_load", "sb_bm25_topk", "sb_bm25_topk_dev", "sb_bm25_scores", "sb_fuse", "sb_fuse_dev",
                 "sb_semantic_mmr", "sb_ce_load", "sb_ce_score", "sb_ce_score_dev", "sb_merge_shards_dev"]:
        assert must in syms


def test_library_exports_every_declared_symbol(built_lib):
    lib = ctypes.CDLL(str(built_lib))
    for name in _header_symbols():
        assert hasattr(lib, name), f"{name} declared in include/sentio_b200.h but not exported"


def test_ctypes_table_matches_header(built_lib):
    from sentio_b200._lib import SIGNATURES, load_library

    assert sorted(SIGNATURES) == _header_symbols()
    load_library()  # attaches prototypes; raises on a missing symbol


def test_argument_counts_match_header():
    from sentio_b200._lib import SIGNATURES

    text = open(os.path.join(ROOT, "include", "sentio_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    for name, (_res, args) in SIGNATURES.items():
        m = re.search(r"\b%s\s*\(([^;]*?)\)\s*;" % name, text, flags=re.S)
        assert m, name
        params = m.group(1).strip()
        n = 0 if params in ("", "void") else params.count(",") + 1
        assert n == len(args), f"{name}: header has {n} parameters, ctypes table {len(args)}"


def _gpu_visible() -> bool:
    if os.path.exists("/dev/nvidia0"):
        return True
    try:
        import torch

        return bool(torch.cuda.is_available())
    except Exception:
        return False


@pytest.mark.skipif(_gpu_visible(), reason="a GPU is visible")
def test_no_cpu_fallback_without_gpu(built_lib):
    """On a box without a GPU the product must fail loudly, not fall back."""
    from sentio_b200._lib import SentioB200Error
    from sentio_b200.engine import B200Engine

    with pytest.raises(SentioB200Error):
        B200Engine(0)


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "sentio_b200")
    for dirpath, _dirs, files in os.walk(pkg):
        for fn in files:
            if fn.endswith((".py", ".cu", ".cuh")):
                src = open(os.path.join(dirpath, fn)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f"{fn} imports oracle/"


def test_library_has_no_ab_switches():
    """Kernel A/B runs on a second build (`python -m sentio_b200.build --variant`, loaded with SENTIO_B200_LIB): the
    library's sources read no environment variable and keep no alternative code behind an SB_ macro."""
    switch = re.compile(r"^\s*#\s*(ifdef|ifndef)\s+SB_|^\s*#\s*(el)?if\b.*\bdefined\s*\(?\s*SB_", flags=re.M)
    csrc = os.path.join(ROOT, "sentio_b200", "csrc")
    for fn in sorted(os.listdir(csrc)):
        if fn.endswith((".cu", ".cuh")):
            src = open(os.path.join(csrc, fn)).read()
            assert "getenv" not in src, f"{fn} reads the environment"
            assert not switch.search(src), f"{fn} compiles code behind an SB_ macro"
