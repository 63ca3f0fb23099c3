"""Shared helpers for the parity tests (oracle = checker, libgnssacq = thing under test)."""
from __future__ import annotations

import io
import math
from types import SimpleNamespace

import numpy as np

import oracle
from oracle.synth import SynthSpec, SatSpec, synth_if

# BASELINE.json north_star: indices / decision bit-exact unless the oracle's top two cells are
# closer than the floating-point tolerance; peak and SNR within 1e-4 relative (FP32).
TIE_TOL = 2e-5
METRIC_RTOL = 1e-4


def structs(fs, if_hz, *, data_type=2, data_precision=1, freq_min=-10000.0, freq_step=500.0,
            freq_num=None, datalen=2, skip=0):
    file = SimpleNamespace(fid=None, skip=skip, dataType=data_type, dataPrecision=data_precision)
    signal = oracle.SignalParams(IF=if_hz, Fs=fs)
    acq = oracle.AcqParams(freqStep=freq_step, freqMin=freq_min, freqNum=freq_num, datalen=datalen)
    return file, signal, acq


def small_spec(fs, if_hz, n, *, sats=None, seed=6102, data_type=2, data_precision=1, sigma=16.0):
    if sats is None:
        sats = [SatSpec(3, 990.0, 1683 % n, 1.2, 0.1), SatSpec(7, -3095.0, (n * 2) // 3, 0.9, 1.0),
                SatSpec(22, 1565.0, 17, 1.5, 2.0)]
    return SynthSpec(fs=fs, if_hz=if_hz, samples_per_ms=n, sigma=sigma, data_type=data_type,
                     data_precision=data_precision, seed=seed, sats=sats)


def oracle_rows(raw_bytes, file, signal, acq, prns, *, coh_ms=1, matlab_quirks=True):
    file = SimpleNamespace(**vars(file))
    file.fid = io.BytesIO(raw_bytes)
    file.skip = 0
    raw = oracle.read_if_block(file, signal, int(acq.datalen) * coh_ms)
    return oracle.coarse_search(raw, signal, acq, prns, coh_ms=coh_ms, matlab_quirks=matlab_quirks)


_CH = {}


def _chunk_surface(b0):
    """One block of Doppler bins of every requested PRN's surface (forked worker of oracle_rows_chunked)."""
    from oracle.acquisition_ref import carrier_table, correlation_surface, folded_blocks
    raw, signal, acq, prns, coh_ms, chunk = (_CH[k] for k in ("raw", "signal", "acq", "prns", "coh_ms", "chunk"))
    n, kk = int(signal.Sample), int(acq.datalen)
    b1 = min(int(acq.freqNum), b0 + chunk)
    sub = oracle.AcqParams(freqStep=acq.freqStep, freqMin=acq.freqMin + acq.freqStep * b0, freqNum=b1 - b0, datalen=kk)
    carrier = carrier_table(signal, sub, coh_ms)
    conj_spectra = np.conj(np.fft.fft(folded_blocks(raw, carrier, n, kk, coh_ms), axis=-1))
    return b0, b1, [correlation_surface(raw, signal, sub, p, coh_ms=coh_ms, carrier=carrier, conj_spectra=conj_spectra)
                    for p in prns]


def oracle_rows_chunked(raw_bytes, file, signal, acq, prns, *, coh_ms=1, chunk_bins=32, workers=None):
    """The same rows as :func:`oracle_rows` for grids too large to hold every forward spectrum at once
    (BASELINE configs 3 and 5: 401 / 2001 bins, 10 ms coherent).  The surface of each PRN is built from the
    oracle's own pieces (carrier_table -> folded_blocks -> correlation_surface) one block of Doppler bins at
    a time -- blocks are independent, so they run on forked workers --, then acquisition.m:62-74
    (peak_and_snr) runs on the whole surface: values and first-index tie rules are exactly coarse_search's."""
    import multiprocessing as mp
    import os
    from oracle.acquisition_ref import peak_and_snr, samples_from_bytes
    raw = samples_from_bytes(raw_bytes, file.dataType, file.dataPrecision)
    n, nb = int(signal.Sample), int(acq.freqNum)
    prns = list(prns)
    _CH.update(raw=raw, signal=signal, acq=acq, prns=prns, coh_ms=coh_ms, chunk=chunk_bins)
    surf = {p: np.empty((nb, n), dtype=np.float64) for p in prns}
    starts = list(range(0, nb, chunk_bins))
    workers = workers or max(1, min(len(starts), len(os.sched_getaffinity(0)), 16))
    if workers > 1:
        with mp.get_context("fork").Pool(workers) as pool:
            parts = pool.map(_chunk_surface, starts, chunksize=1)
    else:
        parts = [_chunk_surface(b0) for b0 in starts]
    for b0, b1, mats in parts:
        for p, m in zip(prns, mats):
            surf[p][b0:b1, :] = m
    _CH.clear()
    return [peak_and_snr(surf[p], signal, acq, p) for p in prns]


def assert_fine_frequency_matches(got, longraw, file, signal, acq, sats):
    """acquisition.m:83-127's fineFreq of every SV of `sats` (`got`, from the GPU) against the oracle on `longraw`
    ((L+1) ms as read by :89-100).  Index exact unless the oracle's two best spectral lines are within the FP32 tie
    tolerance; for I/Q data the line must also be the carrier, IF + the satellite's Doppler."""
    n, L, datalen = int(signal.Sample), int(acq.L), int(acq.datalen)
    res = signal.Fs / (L * n * datalen)
    for sat, g in zip(sats, got):
        want, idx, pk, runner = oracle.fine_frequency(longraw, file, signal, acq, sat.prn, sat.codedelay, detail=True)
        if runner >= pk * (1.0 - 1e-5):             # magnitude tie (|.|, i.e. half the relative gap of power)
            # real input: |X[k]| == |X[F-k]| exactly, so the reference's first-max over the WHOLE spectrum
            # (acquisition.m:116 searches 1:2*halffftlength) is decided by rounding; accept the mirror line too
            mirror = (L * n * datalen - idx + 2) * res if file.dataType == 1 else want
            assert min(abs(g - want), abs(g - mirror)) <= res * 1.0001, (sat.prn, g, want, mirror)
        else:
            assert g == want, (sat.prn, g, want, idx)
        # and it is the carrier: within two 5 Hz-class bins of IF + true Doppler (incl. the 1-based-index quirk)
        if file.dataType == 2:
            assert abs((g - signal.IF) - sat.doppler_hz) <= max(3 * res, 1e3 / L), (sat.prn, g)


def assert_rows_match(gpu_rows, ref_rows, *, thr=12.0, what=""):
    """BASELINE.json north_star: peak metric and SNR within 1e-4 relative for EVERY row; code phase, Doppler bin
    and the decision bit-exact unless the oracle's own top two cells are closer than TIE_TOL (then FP32 may
    legitimately name the other cell -- whose power differs from the winner's by less than TIE_TOL, so the
    metric bound still applies) or the SNR sits within 1e-4 of the threshold."""
    assert len(gpu_rows) == len(ref_rows)
    n_tie = 0
    for g, r in zip(gpu_rows, ref_rows):
        tag = f"{what} PRN {r.prn}"
        assert g.prn == r.prn, tag
        if math.isnan(r.snr_db):
            assert math.isnan(g.snr_db) and not g.acquired, tag
            continue
        tie = r.runner_up >= r.peak * (1.0 - TIE_TOL)
        assert abs(g.peak - r.peak) <= METRIC_RTOL * r.peak, f"{tag}: peak {g.peak} vs {r.peak}"
        same_cell = g.code_phase == r.code_phase and g.doppler_bin == r.doppler_bin
        if tie and not same_cell:
            # the other member of the tie: same peak to 1e-4 (checked above) but its own noise window (another
            # lag, possibly another bin's row), so its SNR is the oracle's only to the row-to-row spread
            n_tie += 1
            assert abs(g.snr_db - r.snr_db) <= 0.1, f"{tag}: snr {g.snr_db} vs {r.snr_db} (tie)"
            continue
        n_tie += int(tie)
        assert g.code_phase == r.code_phase, f"{tag}: code phase {g.code_phase} != {r.code_phase}"
        assert g.doppler_bin == r.doppler_bin, f"{tag}: bin {g.doppler_bin} != {r.doppler_bin}"
        assert g.doppler_hz == r.doppler_hz, tag
        assert abs(g.snr_db - r.snr_db) <= METRIC_RTOL * abs(r.snr_db), f"{tag}: snr {g.snr_db} vs {r.snr_db}"
        if abs(r.snr_db - thr) > METRIC_RTOL * thr:
            assert bool(g.acquired) == r.acquired, tag
    return n_tie
