"""Per-PRN Doppler windows at the C ABI without a GPU: a NULL handle is an argument error, not a crash, and the
Python binding checks the window lengths before it calls the library."""
import ctypes as C

import numpy as np
import pytest

from gnssacq import api


def test_set_doppler_windows_without_a_handle_is_an_argument_error():
    lo = np.zeros(1, dtype=np.float64)
    assert api.lib.gnssacq_set_doppler_windows(None, lo.ctypes.data, lo.ctypes.data) == -1
    assert api.lib.gnssacq_set_doppler_windows(None, None, None) == -1
    assert "gnssacq_set_doppler_windows" in api.EXPORTS


def test_binding_wants_one_window_per_prn():
    s = api.Searcher.__new__(api.Searcher)          # no device needed: the length check comes first
    s.cfg = api.make_config(prns=[1, 2, 3])
    s._h = C.c_void_p()
    with pytest.raises(ValueError):
        s.set_doppler_windows([0.0, 0.0], [1.0, 1.0])
