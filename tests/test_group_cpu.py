"""CPU-side checks of the device-group ABI (ofdm_group_*): argument checks that need no GPU, and no group without one."""
import ctypes

import pytest


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build()
    from ofdm_b200 import _cabi
    return _cabi.load()


def _ids(*ids):
    return (ctypes.c_int32 * max(len(ids), 1))(*ids)


def test_group_argument_checks(lib):
    h = ctypes.c_void_p(1)
    assert lib.ofdm_group_create(ctypes.byref(h), _ids(0), 0, 0) == -1           # OFDM_ERR_INVALID: no members
    assert not h.value
    h = ctypes.c_void_p(1)
    assert lib.ofdm_group_create(ctypes.byref(h), None, 2, 0) == -1               # NULL device list
    assert not h.value
    lib.ofdm_group_destroy(None)                                                  # no-op
    assert lib.ofdm_group_last_error(None) == b"null group"
    assert lib.ofdm_group_size(None) == -1


def test_no_group_without_gpu(lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    h = ctypes.c_void_p(1)
    assert lib.ofdm_group_create(ctypes.byref(h), _ids(0, 0), 2, 0) == -3          # OFDM_ERR_NODEVICE: no CPU fallback
    assert not h.value
    import ofdm_b200
    with pytest.raises(ofdm_b200.OfdmError):
        ofdm_b200.Group([0])
