"""CPU tests of the counted-stage ABI: `nttt_match_count_bind` rejects a count outside [0, capacity] and a malformed
destination with NTTT_EINVAL before any CUDA call, and `nttt_match_image_counted` needs its count, its arguments and
single-plane inputs before anything is enqueued."""
import ctypes
import importlib

import pytest

EINVAL = -1
EWORKSPACE = -4
FAKE_DEV = 0x7f0000000000  # never dereferenced: every call below is rejected on the host


@pytest.fixture(scope="module")
def lib():
    build = importlib.import_module("no-time-to-train_b200.build")
    build.build_library()
    return importlib.import_module("no-time-to-train_b200._lib")


def _capacity(lib, n):
    a = lib.MatchArgs()
    a.n = n
    return a


def _bind(lib, n, cap, dst=FAKE_DEV):
    return lib.load().nttt_match_count_bind(dst, n, ctypes.byref(cap) if cap is not None else None, None)


def test_count_bind_rejects_null_arguments(lib):
    assert _bind(lib, 5, _capacity(lib, 256), dst=None) == EINVAL
    assert _bind(lib, 5, None) == EINVAL


def test_count_bind_rejects_counts_outside_the_capacity(lib):
    cap = _capacity(lib, 256)
    for n in (-1, -(1 << 31), 257, 1 << 20):
        assert _bind(lib, n, cap) == EINVAL, n
    assert _bind(lib, 1, _capacity(lib, 0)) == EINVAL
    assert _bind(lib, 0, _capacity(lib, -1)) == EINVAL


def test_count_bind_rejects_a_misaligned_count(lib):
    for off in (1, 2, 3):
        assert _bind(lib, 5, _capacity(lib, 256), dst=FAKE_DEV + off) == EINVAL, off


def test_counted_entry_needs_its_count(lib):
    cdll = lib.load()
    a = _capacity(lib, 256)
    assert cdll.nttt_match_image_counted(FAKE_DEV, ctypes.byref(a), None, None, None, None, None) == EINVAL
    assert cdll.nttt_match_image_counted(FAKE_DEV, None, None, None, None, FAKE_DEV, None) == EINVAL
    assert cdll.nttt_match_image_counted(None, ctypes.byref(a), None, None, None, FAKE_DEV, None) == EINVAL


def test_counted_entry_rejects_multimask_inputs(lib):
    """compacted candidates are single-plane: n_multi > 1 is refused before anything is enqueued (the arguments are
    otherwise complete enough to reach the launch)"""
    cdll = lib.load()
    a = _capacity(lib, 256)
    a.lr_h = a.lr_w = 256
    a.eh = a.ew = 37
    a.c, a.n_cls, a.ori_h, a.ori_w = 384, 80, 480, 640
    a.num_out_instance, a.max_sel = 20, 160
    a.n_multi, a.multi_first = 3, 1
    a.counts = a.workspace = a.multi_ious = a.logits = a.tar_feat = a.proto = FAKE_DEV
    a.out_masks = a.out_boxes = a.out_scores = a.out_labels = a.out_index = FAKE_DEV
    a.workspace_bytes = 0  # (without the single-plane rule the call would stop at the workspace check instead)
    assert cdll.nttt_match_image(FAKE_DEV, ctypes.byref(a), None) == EWORKSPACE
    assert cdll.nttt_match_image_counted(FAKE_DEV, ctypes.byref(a), None, None, None, FAKE_DEV, None) == EINVAL
