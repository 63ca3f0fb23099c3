"""gnssacq_track_bank: the device-side tracking loop (gnssacq_track) observed every period by a correlator bank of up
to 32 taps.  `-m gpu`.

The loop must not notice the bank (records byte-identical to gnssacq_track's), and every tap of every period must be
the correlation the oracle, and gnssacq_correlate, compute for that period's channel state."""
import ctypes as C
import functools

import numpy as np
import pytest

import gnssacq
from gnssacq import api
from oracle import tracking_ref as tr
from oracle.synth import SatSpec, SynthSpec, synth_if
from helpers import structs

pytestmark = pytest.mark.gpu

EPL = [-0.5, 0.0, 0.5]                                          # the default loop's E/P/L (spacing 0.5)
BANK25 = [round(0.6 - 0.05 * i, 2) for i in range(25)]          # trackingCT_POS_updated_multicorrelator.m:41
GRID29 = [round(0.7 - 0.05 * i, 2) for i in range(29)]          # a 29-point grid, as trackingVT_POS_updated.m:29 uses
TAPS32 = [round(-0.75 + 0.05 * i, 2) for i in range(32)]        # kTrackMaxTaps
BANKS = {"bank25": BANK25, "grid29": GRID29, "one": [0.0], "taps32": TAPS32}
# the cases of test_gpu_tracking.py::test_device_side_tracking_loop_against_the_oracle_loop
CASES = [(26e6, 0.0, 2, 1, 60), (58e6, 4.58e6, 2, 1, 25), (6e6, 1.25e6, 2, 2, 40), (6e6, 1.25e6, 1, 1, 40)]


def _cfg(fs, if_hz, data_type, precision):
    file, signal, acq = structs(fs, if_hz, data_type=data_type, data_precision=precision, datalen=2)
    return gnssacq.config_from_structs(file, signal, acq, prns=[1])


@functools.lru_cache(maxsize=None)
def _case(fs, if_hz, data_type, precision, periods):
    """That test's three-satellite signal and start states."""
    n = int(fs * 1e-3)
    truth = [(5, 1500.0, (n * 2) // 13, 5.0), (17, -2750.0, (n * 7) // 12, 4.0), (30, 420.0, 11, 6.0)]
    spec = SynthSpec(fs=fs, if_hz=if_hz, samples_per_ms=n, sigma=6.0, data_type=data_type, data_precision=precision,
                     seed=5, sats=[SatSpec(p, d, cd, a, 0.4) for p, d, cd, a in truth])
    raw = synth_if(spec, 0, periods + 3)
    start = [api.Channel(prn=p, num_samples=0, sample_offset=n - cd + 1, carrier_hz=if_hz + d + 8.0, rem_phase=0.0,
                         code_hz=1.023e6, rem_chip=0.0) for p, d, cd, a in truth]
    return raw, start, truth


def _period_channels(start, recs):
    """The gnssacq_channel of every period, rebuilt from the start state and the previous period's record."""
    out = []
    for c, ch in enumerate(recs):
        for i, r in enumerate(ch):
            prev = recs[c][i - 1] if i else None
            s = start[c]
            out.append(api.Channel(prn=s.prn, num_samples=r.num_samples,
                                   sample_offset=prev.sample_end if prev else s.sample_offset,
                                   carrier_hz=prev.carrier_hz if prev else s.carrier_hz,
                                   rem_phase=prev.rem_phase if prev else s.rem_phase,
                                   code_hz=prev.code_hz if prev else s.code_hz,
                                   rem_chip=prev.rem_chip if prev else s.rem_chip))
    return out


@pytest.mark.parametrize("bank", list(BANKS))
@pytest.mark.parametrize("fs,if_hz,data_type,precision,periods", CASES)
def test_bank_observes_the_loop(fs, if_hz, data_type, precision, periods, bank):
    """Records byte-identical to gnssacq_track's; every tap the gnssacq_correlate sum of its period's state (1e-7 of
    |P|: gnssacq_correlate takes one sincos per sample, the loop rotates a phasor), and the taps at -s, 0, +s equal to
    the record's E, P, L (1e-9); two calls byte-identical; running out of samples is GNSSACQ_ERR_SHORT_BUFFER."""
    sp = BANKS[bank]
    raw, start, truth = _case(fs, if_hz, data_type, precision, periods)
    with api.Searcher(_cfg(fs, if_hz, data_type, precision)) as s:
        s.track_load(raw)
        ref = s.track(start, periods)
        recs, bi, bq = s.track_bank(start, periods, sp)
        assert bi.shape == bq.shape == (len(start), periods, len(sp))
        assert [bytes(r) for ch in recs for r in ch] == [bytes(r) for ch in ref for r in ch]
        recs2, bi2, bq2 = s.track_bank(start, periods, sp)
        assert [bytes(r) for ch in recs2 for r in ch] == [bytes(r) for ch in recs for r in ch]
        assert bi.tobytes() == bi2.tobytes() and bq.tobytes() == bq2.tobytes()
        with pytest.raises(gnssacq.GnssAcqError) as e:                                    # trackingCT.m:107-111
            s.track_bank(start, periods + 10, sp)
        assert e.value.code == -3
        chans = _period_channels(start, recs)
        parts = [s.correlate(chans[k:k + 64], sp) for k in range(0, len(chans), 64)]       # 64 channels per call
        ci, cq = np.concatenate([a for a, _ in parts]), np.concatenate([b for _, b in parts])
    gi, gq = bi.reshape(-1, len(sp)), bq.reshape(-1, len(sp))
    flat = [r for ch in recs for r in ch]
    for k, r in enumerate(flat):
        p = max(np.hypot(r.P_i, r.P_q), 1.0)
        assert np.abs(gi[k] - ci[k]).max() <= 1e-7 * p and np.abs(gq[k] - cq[k]).max() <= 1e-7 * p, f"period {k}"
        for t, (ri, rq) in zip(EPL, ((r.E_i, r.E_q), (r.P_i, r.P_q), (r.L_i, r.L_q))):
            if t in sp:
                j = sp.index(t)
                assert abs(gi[k, j] - ri) <= 1e-9 * p and abs(gq[k, j] - rq) <= 1e-9 * p, f"period {k} tap {t}"


@pytest.mark.parametrize("bank", list(BANKS))
@pytest.mark.parametrize("fs,if_hz,data_type,precision,periods", CASES)
def test_bank_against_the_oracle_loop(fs, if_hz, data_type, precision, periods, bank):
    """The oracle runs the loop on its own correlations; in every period its bank on its own state matches the GPU
    bank to 1e-7 of max(|P|, 1), the bar of the device loop's E/P/L."""
    sp = BANKS[bank]
    raw, start, truth = _case(fs, if_hz, data_type, precision, periods)
    with api.Searcher(_cfg(fs, if_hz, data_type, precision)) as s:
        s.track_load(raw)
        recs, bi, bq = s.track_bank(start, periods, sp)
    n = int(fs * 1e-3)
    bps = data_type * precision
    for c, (p, d, cd, a) in enumerate(truth):
        st = tr.ChannelState(prn=p, carrier_basis_hz=if_hz + d + 8.0, carrier_hz=if_hz + d + 8.0, sample_pos=n - cd + 1)
        for i in range(periods):
            ns = tr.num_samples(st.code_hz, fs, st.rem_chip)
            assert recs[c][i].num_samples == ns
            x = tr.samples_of(raw[st.sample_pos * bps:(st.sample_pos + ns) * bps], data_type, precision)
            oi, oq = tr.correlate(x, fs, p, st.carrier_hz, st.rem_phase, st.code_hz, st.rem_chip, sp)
            ei, eq = tr.correlate(x, fs, p, st.carrier_hz, st.rem_phase, st.code_hz, st.rem_chip, EPL)
            scale = max(np.hypot(ei[1], eq[1]), 1.0)
            assert np.abs(bi[c, i] - oi).max() <= 1e-7 * scale, f"channel {c} period {i}: I"
            assert np.abs(bq[c, i] - oq).max() <= 1e-7 * scale, f"channel {c} period {i}: Q"
            tr.close_loops(st, ei, eq, ns, fs)


def test_track_bank_argument_errors():
    fs, if_hz, n = 6e6, 1.25e6, 6000
    start = [api.Channel(prn=1, num_samples=0, sample_offset=0, carrier_hz=if_hz, rem_phase=0.0, code_hz=1.023e6, rem_chip=0.0)]
    with api.Searcher(_cfg(fs, if_hz, 2, 1)) as s:              # (one period: a silent segment gives the loop NaNs)
        with pytest.raises(gnssacq.GnssAcqError) as e:
            s.track_bank(start, 1, EPL)                                     # nothing loaded
        assert e.value.code == -7
        s.track_load(bytes(2 * n * 4))
        s.track_bank(start, 1, EPL)
        ch = (api.Channel * 1)(*start)
        loops = api.LoopParams()
        api.lib.gnssacq_loop_params_default(C.byref(loops))
        out = (api.TrackRecord * 1)()
        bank = np.zeros(33, dtype=np.float64)
        bank2 = np.zeros(33, dtype=np.float64)
        f = lambda n_taps, sp, bi, bq: api.lib.gnssacq_track_bank(s._h, 1, ch, C.byref(loops), 1, n_taps, sp, out, bi, bq)
        sp = np.zeros(33, dtype=np.float64)
        assert f(1, sp.ctypes.data, bank.ctypes.data, bank2.ctypes.data) == 0
        assert f(0, sp.ctypes.data, bank.ctypes.data, bank2.ctypes.data) == -1
        assert f(33, sp.ctypes.data, bank.ctypes.data, bank2.ctypes.data) == -1
        for bad in (np.nan, np.inf, -np.inf):
            sp_bad = np.array([0.0, bad, 0.1])
            assert f(3, sp_bad.ctypes.data, bank.ctypes.data, bank2.ctypes.data) == -1
        assert f(3, None, bank.ctypes.data, bank2.ctypes.data) == -1
        assert f(3, sp.ctypes.data, None, bank2.ctypes.data) == -1
        assert f(3, sp.ctypes.data, bank.ctypes.data, None) == -1
        with pytest.raises(gnssacq.GnssAcqError) as e:
            s.track_bank(start, 1, [])
        assert e.value.code == -1
        s.track_bank(start, 1, EPL)                                         # the handle still works


def _bank_shape(sats, periods=70):
    """Mean |bank(tau)| / |P| over the locked periods (>= 50) of a 58 MHz channel tracking PRN 5."""
    fs, if_hz, n = 58e6, 4.58e6, 58000
    spec = SynthSpec(fs=fs, if_hz=if_hz, samples_per_ms=n, sigma=2.0, data_type=2, data_precision=1, seed=9, sats=sats)
    raw = synth_if(spec, 0, periods + 3)
    start = [api.Channel(prn=5, num_samples=0, sample_offset=n - 20000 + 1, carrier_hz=if_hz + 1508.0, rem_phase=0.0,
                         code_hz=1.023e6, rem_chip=0.0)]
    with api.Searcher(_cfg(fs, if_hz, 2, 1)) as s:
        s.track_load(raw)
        recs, bi, bq = s.track_bank(start, periods, BANK25)
    p = np.array([np.hypot(r.P_i, r.P_q) for r in recs[0]])
    return np.mean(np.hypot(bi[0, 50:], bq[0, 50:]) / p[50:, None], axis=0)


def test_bank_samples_the_correlation_function_and_shows_multipath():
    """A clean signal: the bank follows the triangle 1 - |tau|.  Add a copy of the same PRN, Doppler and phase
    delayed by 0.3 chip at half amplitude: the DLL re-centres between the two paths (0.1 chip toward the delayed
    one), and the bank is lopsided toward the direct path, which lies on the late-tap side (positive spacing) of
    the prompt: |bank(+tau)| > |bank(-tau)| for tau = 0.05 .. 0.15.  (Beyond +-0.2 chip the two-path function is
    symmetric about that lock point, so the taps there cannot tell the sides apart.)"""
    tau = np.array(BANK25)
    delay = round(0.3 * 58e6 / 1.023e6)                                    # 17 samples
    clean = _bank_shape([SatSpec(5, 1500.0, 20000, 20.0, 0.4)])
    assert np.abs(clean - (1.0 - np.abs(tau))).max() <= 0.05, clean
    two = _bank_shape([SatSpec(5, 1500.0, 20000, 20.0, 0.4), SatSpec(5, 1500.0, 20000 - delay, 10.0, 0.4)])
    for t in (0.05, 0.1, 0.15):
        i, j = BANK25.index(t), BANK25.index(-t)
        assert abs(clean[i] - clean[j]) < 0.01
        assert two[i] - two[j] > 0.02, (t, two[i], two[j])
    assert two[BANK25.index(0.1)] > 1.0                                   # the bank's peak is not the prompt
