"""CPU tests of the C-ABI boundary: the library loads without a GPU, exports every symbol the header declares,
its pure-host entry points work, and compute entries fail loudly (no CPU fallback)."""
import ctypes
import importlib
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "nttt_b200.h")


@pytest.fixture(scope="module")
def lib():
    build = importlib.import_module("no-time-to-train_b200.build")
    build.build_library()
    return importlib.import_module("no-time-to-train_b200._lib")


def declared_symbols():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(nttt_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_all_exported_and_bound(lib):
    names = declared_symbols()
    assert len(names) >= 20
    cdll = lib.load()
    for name in names:
        assert hasattr(cdll, name), f"{name} declared in include/nttt_b200.h but not exported"
        assert name in lib.SIGNATURES, f"{name} has no ctypes signature in _lib.py"
    assert sorted(lib.SIGNATURES) == names


def test_version_and_error_strings(lib):
    cdll = lib.load()
    assert cdll.nttt_version() == 200 and cdll.nttt_build_is_ablation() == 0
    assert cdll.nttt_error_string(0) == b"ok"
    assert b"workspace" in cdll.nttt_error_string(-4)


def test_workspace_queries_are_pure_host(lib):
    cdll = lib.load()
    small = cdll.nttt_match_workspace_bytes(64, 256, 256, 37, 37, 384, 5, 480, 640, 64)
    big = cdll.nttt_match_workspace_bytes(1024, 256, 256, 37, 37, 1024, 80, 1024, 1024, 800)
    assert 0 < small < big
    # dominated by the packed full-res masks: 800 * 1024 * 32 words * 4 B
    assert big >= 800 * 1024 * 32 * 4
    assert cdll.nttt_match_workspace_bytes(-1, 256, 256, 37, 37, 384, 5, 480, 640, 64) == 0
    assert cdll.nttt_nms_workspace_bytes(1024) >= 1024 * 32 * 4


def test_match_args_struct_layout_with_decay_taps(lib):
    """The ctypes mirror must have the size of the C struct as compiled: the fields up to `low_latency` (at 264, padded
    to 272), then the three pointer taps of the score decay (`sel`, `ios`, `ios_inter`)."""
    assert ctypes.sizeof(lib.MatchArgs) == lib.load().nttt_sizeof_match_args() == 296
    assert lib.MatchArgs.low_latency.offset == 264
    assert [getattr(lib.MatchArgs, f).offset for f in ("sel", "ios", "ios_inter")] == [272, 280, 288]


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_cpu_fallback(lib):
    cdll = lib.load()
    out = ctypes.c_void_p()
    assert cdll.nttt_ctx_create(ctypes.byref(out), 0) == -2  # NTTT_ENODEVICE
    pkg = importlib.import_module("no-time-to-train_b200")
    with pytest.raises(RuntimeError, match="CUDA"):
        pkg.MatchingStage("cpu", pkg.StageConfig())
    with pytest.raises(ValueError, match="CUDA tensor"):
        importlib.import_module("no-time-to-train_b200.ops").threshold_pack(torch.zeros(1, 256, 256))


def test_invalid_arguments_are_rejected(lib):
    cdll = lib.load()
    assert cdll.nttt_threshold_pack(None, 4, 256, 256, 0.0, 1.0, None, None, None, None, None, None) == -1
    assert cdll.nttt_threshold_pack(None, -1, 256, 256, 0.0, 1.0, None, None, None, None, None, None) == -1
    assert cdll.nttt_match_image(None, None, None) == -1
    assert cdll.nttt_proto_prepare(None, 3, 2, 8, None, None) == -1
