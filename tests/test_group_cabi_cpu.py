"""CPU-side checks of the in-process group entry points: the library exports them, and without a device they return an
error instead of crashing."""
import ctypes as C

import numpy as np
import pytest

import asgart_b200 as ab
from asgart_b200 import _lib

NEW = ["asgart_b200_ctx_copy_strand", "asgart_b200_search_group", "asgart_b200_run_files_devices"]


def test_group_symbols_exported():
    L = _lib.load()
    for s in NEW:
        assert s in _lib.SYMBOLS and hasattr(L, s), s


def test_group_entry_points_refuse_bad_arguments():
    L = _lib.load()
    assert L.asgart_b200_ctx_copy_strand(None, None) == _lib.EINVAL
    out = C.c_void_p()
    st = ab.RunSettings().to_c()
    ch = np.zeros((1, 2), dtype=np.uint64)
    assert L.asgart_b200_search_group(None, 1, ch.ctypes.data, 1, C.byref(st), ab.POST_ALL, C.byref(out)) == _lib.EINVAL
    none = (C.c_void_p * 2)(None, None)
    assert L.asgart_b200_search_group(none, 2, ch.ctypes.data, 1, C.byref(st), ab.POST_ALL, C.byref(out)) == _lib.EINVAL
    assert L.asgart_b200_search_group(none, 0, ch.ctypes.data, 1, C.byref(st), ab.POST_ALL, C.byref(out)) == _lib.EINVAL
    assert not out.value


def test_run_files_devices_argument_errors(tmp_path):
    fa = tmp_path / "a.fa"
    fa.write_text(">a\n" + "ACGT" * 100 + "\n")
    L = _lib.load()
    err = C.c_char_p()
    st = (_lib.Settings * 1)(ab.RunSettings().to_c())
    dev = (C.c_int32 * 2)(0, 0)
    assert not L.asgart_b200_run_files_devices(str(fa).encode(), st, 1, dev, 0, None, C.byref(err))
    assert b"no devices" in err.value
    trim = (_lib.Settings * 1)(ab.RunSettings(trim=(10, 100)).to_c())
    assert not L.asgart_b200_run_files_devices(str(fa).encode(), trim, 1, dev, 2, None, C.byref(err))
    assert b"--trim" in err.value


@pytest.mark.skipif(ab.device_count() > 0, reason="checks the no-device behaviour")
def test_group_run_without_device_errors(tmp_path):
    fa = tmp_path / "a.fa"
    fa.write_text(">a\n" + "ACGT" * 100 + "\n")
    with pytest.raises(ab.AsgartB200Error, match="no CPU path"):
        ab.search_duplications([str(fa)], ab.RunSettings(), devices=[0, 0])
    with pytest.raises(ab.AsgartB200Error, match="no CPU path"):
        ab.search_duplications_passes([str(fa)], [ab.RunSettings()], devices=[0])
