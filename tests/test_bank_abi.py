"""CPU tests of the banked-stage ABI: the ctypes mirror of `nttt_match_bank` has the size of the C struct,
`nttt_match_bank_bind` rejects a bank that does not fit the capacity with NTTT_EINVAL before any CUDA call, and
`nttt_match_image_banked` needs its bank struct."""
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


def test_match_bank_struct_layout(lib):
    """two pointers, then the live (n_cls, l_neg)"""
    assert ctypes.sizeof(lib.MatchBank) == lib.load().nttt_sizeof_match_bank() == 24
    assert lib.MatchBank.n_cls.offset == 16 and lib.MatchBank.l_neg.offset == 20


def _capacity(lib, n_cls, l_neg=0):
    a = lib.MatchArgs()
    a.n_cls, a.l_neg = n_cls, l_neg
    return a


def _bank(lib, n_cls, l_neg=0, proto=FAKE_DEV, proto_neg=None):
    return lib.MatchBank(proto, proto_neg, n_cls, l_neg)


def _bind(lib, bank, cap, dst=FAKE_DEV + (1 << 32)):
    return lib.load().nttt_match_bank_bind(dst, ctypes.byref(bank), ctypes.byref(cap), None)


def test_bank_bind_rejects_null_arguments(lib):
    cdll = lib.load()
    cap = _capacity(lib, 80)
    assert cdll.nttt_match_bank_bind(None, ctypes.byref(_bank(lib, 7)), ctypes.byref(cap), None) == EINVAL
    assert cdll.nttt_match_bank_bind(FAKE_DEV, None, ctypes.byref(cap), None) == EINVAL
    assert cdll.nttt_match_bank_bind(FAKE_DEV, ctypes.byref(_bank(lib, 7)), None, None) == EINVAL
    assert _bind(lib, _bank(lib, 7, proto=None), cap) == EINVAL
    assert _bind(lib, _bank(lib, 7, l_neg=2, proto=None, proto_neg=FAKE_DEV), _capacity(lib, 80, 3)) == EINVAL


def test_bank_bind_rejects_class_counts_outside_the_capacity(lib):
    cap = _capacity(lib, 80)
    for n_cls in (0, -1, 81, 1203):
        assert _bind(lib, _bank(lib, n_cls), cap) == EINVAL, n_cls
    assert _bind(lib, _bank(lib, 1), _capacity(lib, 0)) == EINVAL  # (no capacity admits a bank)
    neg = _capacity(lib, 80, 3)
    for n_cls in (0, 81):
        assert _bind(lib, _bank(lib, n_cls, l_neg=2, proto_neg=FAKE_DEV), neg) == EINVAL, n_cls


def test_bank_bind_rejects_the_wrong_kind_of_bank(lib):
    # a negative table for a plain capacity, and a plain bank for a negative capacity
    assert _bind(lib, _bank(lib, 7, l_neg=2, proto_neg=FAKE_DEV), _capacity(lib, 80)) == EINVAL
    assert _bind(lib, _bank(lib, 7, l_neg=2), _capacity(lib, 80, 3)) == EINVAL
    assert _bind(lib, _bank(lib, 7), _capacity(lib, 80, -1)) == EINVAL  # (a negative capacity below 0)


def test_bank_bind_rejects_negative_counts_outside_the_capacity(lib):
    cap = _capacity(lib, 80, 3)
    for l_neg in (0, -1, 4):
        assert _bind(lib, _bank(lib, 7, l_neg=l_neg, proto_neg=FAKE_DEV), cap) == EINVAL, l_neg


def test_bank_bind_rejects_a_misaligned_struct(lib):
    for off in (1, 4, 12):
        assert _bind(lib, _bank(lib, 7), _capacity(lib, 80), dst=FAKE_DEV + off) == EINVAL, off


def test_banked_entry_needs_its_bank_struct(lib):
    cdll = lib.load()
    a = _capacity(lib, 80)
    a.n = 128
    assert cdll.nttt_match_image_banked(FAKE_DEV, ctypes.byref(a), None, None, None, None) == EINVAL
    assert cdll.nttt_match_image_banked(FAKE_DEV, ctypes.byref(a), None, FAKE_DEV, None, None) == EINVAL
    assert cdll.nttt_match_image_banked(None, ctypes.byref(a), None, None, FAKE_DEV, None) == EINVAL
