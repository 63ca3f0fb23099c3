"""gnssacq_track_bank at the C ABI without a GPU: the symbol is exported and declared, and NULL arguments are argument
errors, not crashes."""
import ctypes as C

import numpy as np

from gnssacq import api


def test_track_bank_is_exported():
    assert "gnssacq_track_bank" in api.EXPORTS
    assert hasattr(api.lib, "gnssacq_track_bank")


def test_track_bank_null_arguments_are_argument_errors():
    ch = (api.Channel * 1)(api.Channel(prn=1, num_samples=0, sample_offset=0, carrier_hz=0.0, rem_phase=0.0,
                                       code_hz=1.023e6, rem_chip=0.0))
    loops = api.LoopParams()
    assert api.lib.gnssacq_loop_params_default(C.byref(loops)) == 0
    sp = np.zeros(3, dtype=np.float64)
    out = (api.TrackRecord * 4)()
    bi = np.zeros(12, dtype=np.float64)
    bq = np.zeros(12, dtype=np.float64)
    f = api.lib.gnssacq_track_bank
    assert f(None, 1, ch, C.byref(loops), 4, 3, sp.ctypes.data, out, bi.ctypes.data, bq.ctypes.data) == -1   # no handle
    assert f(None, 1, None, None, 4, 3, None, None, None, None) == -1
    assert f(None, 1, ch, C.byref(loops), 4, 3, None, out, bi.ctypes.data, bq.ctypes.data) == -1
    assert f(None, 1, ch, C.byref(loops), 4, 3, sp.ctypes.data, out, None, bq.ctypes.data) == -1
    assert f(None, 1, ch, C.byref(loops), 4, 3, sp.ctypes.data, out, bi.ctypes.data, None) == -1
