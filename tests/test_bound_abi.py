"""CPU tests of the bound-input ABI: the ctypes mirror of `nttt_match_inputs` has the size of the C struct, and
`nttt_match_bind` rejects a binding that does not fit the stage's shapes with NTTT_EINVAL before any CUDA call."""
import ctypes
import importlib

import pytest

EINVAL = -1
FAKE_DEV = 0x7f0000000000  # never dereferenced: every call below is rejected on the host


@pytest.fixture(scope="module")
def lib():
    build = importlib.import_module("no-time-to-train_b200.build")
    build.build_library()
    return importlib.import_module("no-time-to-train_b200._lib")


def test_match_inputs_struct_layout(lib):
    """four pointers, 64 chunk bases, then (h, w)"""
    assert ctypes.sizeof(lib.MatchInputs) == lib.load().nttt_sizeof_match_inputs() == 4 * 8 + 64 * 8 + 8
    assert lib.MatchInputs.chunks.offset == 32 and lib.MatchInputs.ori_hw.offset == 544


def _shapes(lib, n, n_multi=0, n_chunks=0, chunk_prompts=0):
    a = lib.MatchArgs()
    a.n, a.n_multi, a.n_chunks, a.chunk_prompts = n, n_multi, n_chunks, chunk_prompts
    return a


def _single(lib, logits=FAKE_DEV, pred_ious=FAKE_DEV + 4096, tar_feat=FAKE_DEV + 8192):
    v = lib.MatchInputs()
    v.logits, v.pred_ious, v.tar_feat = logits, pred_ious, tar_feat
    return v


def _chunked(lib, k, multi_ious=FAKE_DEV + 4096, tar_feat=FAKE_DEV + 8192):
    v = lib.MatchInputs()
    v.multi_ious, v.tar_feat = multi_ious, tar_feat
    for i in range(k):
        v.chunks[i] = FAKE_DEV + (1 << 24) * (i + 1)
    return v


def _bind(lib, v, shapes, dst=FAKE_DEV + (1 << 32)):
    return lib.load().nttt_match_bind(dst, ctypes.byref(v), ctypes.byref(shapes), None)


def test_bind_rejects_null_pointers(lib):
    cdll = lib.load()
    sh = _shapes(lib, 128)
    assert cdll.nttt_match_bind(None, ctypes.byref(_single(lib)), ctypes.byref(sh), None) == EINVAL
    assert cdll.nttt_match_bind(FAKE_DEV, None, ctypes.byref(sh), None) == EINVAL
    assert cdll.nttt_match_bind(FAKE_DEV, ctypes.byref(_single(lib)), None, None) == EINVAL
    assert _bind(lib, _single(lib, logits=None), sh) == EINVAL
    assert _bind(lib, _single(lib, pred_ious=None), sh) == EINVAL
    assert _bind(lib, _single(lib, tar_feat=None), sh) == EINVAL
    assert _bind(lib, _single(lib), sh, dst=FAKE_DEV + 4) == EINVAL  # the struct is stored in 8-byte words
    m = _shapes(lib, 100, n_multi=4, n_chunks=4, chunk_prompts=25)
    assert _bind(lib, _chunked(lib, 4, multi_ious=None), m) == EINVAL
    v = _chunked(lib, 4)
    v.chunks[2] = None
    assert _bind(lib, v, m) == EINVAL
    one = lib.MatchInputs()  # multimask from one buffer: `logits` is needed
    one.multi_ious, one.tar_feat = FAKE_DEV, FAKE_DEV
    assert _bind(lib, one, _shapes(lib, 100, n_multi=4)) == EINVAL


def test_bind_rejects_misaligned_logits(lib):
    sh = _shapes(lib, 128)
    for off in (4, 8, 12):
        assert _bind(lib, _single(lib, logits=FAKE_DEV + off), sh) == EINVAL
    m = _shapes(lib, 100, n_multi=4, n_chunks=4, chunk_prompts=25)
    v = _chunked(lib, 4)
    v.chunks[3] += 4
    assert _bind(lib, v, m) == EINVAL
    one = lib.MatchInputs()
    one.logits, one.multi_ious, one.tar_feat = FAKE_DEV + 8, FAKE_DEV, FAKE_DEV
    assert _bind(lib, one, _shapes(lib, 100, n_multi=4)) == EINVAL


def test_bind_rejects_chunk_mismatches(lib):
    v = _chunked(lib, 64)
    assert _bind(lib, v, _shapes(lib, 100, n_multi=4, n_chunks=65, chunk_prompts=2)) == EINVAL  # > 64 chunks
    assert _bind(lib, v, _shapes(lib, 100, n_multi=4, n_chunks=4, chunk_prompts=0)) == EINVAL
    assert _bind(lib, v, _shapes(lib, 100, n_multi=4, n_chunks=4, chunk_prompts=-25)) == EINVAL
    assert _bind(lib, v, _shapes(lib, 100, n_multi=4, n_chunks=3, chunk_prompts=25)) == EINVAL  # 75 < 100 prompts
    assert _bind(lib, _chunked(lib, 3), _shapes(lib, 100, n_multi=4, n_chunks=4, chunk_prompts=25)) == EINVAL
    assert _bind(lib, _single(lib), _shapes(lib, -1)) == EINVAL


def test_bound_entry_needs_its_inputs_struct(lib):
    cdll = lib.load()
    a = _shapes(lib, 128)
    assert cdll.nttt_match_image_bound(None, ctypes.byref(a), None, FAKE_DEV, None) == EINVAL
    assert cdll.nttt_match_image_bound(FAKE_DEV, ctypes.byref(a), None, None, None) == EINVAL
