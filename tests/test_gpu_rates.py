"""Front-end sample rates that are not a built transform length (`-m gpu`): each ms of N samples is zero-padded into
the smallest built transform length NF >= 2N - 1 (gnssacq_transform_size), the code spectrum is that of the code
repeated up to lag 2N - 2, and the row end reads lags < N only.  Checked against the float64 oracle, which is written
for any N: rows, every cell of the surface, padded lags that must never win, the planner's forward bases (with the
M-ms fold, bins share a base only when they are a whole number of Fs/NF AND of Fs/N apart), the features that need
no logic of their own (Doppler windows, block-granular tail, sweeps, several handles), the exchange refusal, the
Bluestein N-point DFTs of gnssacq_fft_forward and the fine-frequency stage, tracking and the acquisition() wrapper."""
import io
import math

import numpy as np
import pytest

import gnssacq
import oracle
from gnssacq import api
from oracle.acquisition_ref import carrier_table, correlation_surface, folded_blocks, peak_and_snr, samples_from_bytes
from oracle.synth import SatSpec, synth_if
from helpers import (TIE_TOL, assert_fine_frequency_matches, assert_rows_match, oracle_rows, oracle_rows_chunked,
                     small_spec, structs)
from test_gpu_parity import VARIANTS
import test_gpu_tracking

pytestmark = pytest.mark.gpu

K = 2
PRNS = [3, 22, 9]                                    # strong, weak, absent
# label -> (Fs, IF, data_type, data_precision)
RATES = {
    "2.048": (2.048e6, 0.0, 2, 1),                   # RTL-SDR, int8 I/Q
    "4.092": (4.092e6, 1.023e6, 1, 1),               # real int8, IF != 0
    "5": (5e6, 0.0, 2, 2),                           # int16 I/Q with a DC offset
    "13.000": (13e6, 0.0, 2, 1),                     # N = 13 000: NF = 26 000 (2N - 1 = 25 999)
    "13.001": (13.001e6, 0.0, 2, 1),                 # N = 13 001: NF = 58 000 (2N - 1 = 26 001)
    "16.368": (16.368e6, 4.092e6, 2, 1),
    "16.3676": (16.3676e6, 4.1304e6, 2, 1),          # off-nominal: Fs/N is not 1 kHz
    "29": (29e6, 0.0, 2, 1),
}
DC = (300, -450)


def n_of(fs):
    return int(math.ceil(fs * 1e-3))


def nf_of(n):
    return next(b for b in (6000, 26000, 58000) if b >= 2 * n - 1)


def add_dc(raw_b, dc):
    """int16 I/Q bytes with the pair dc = (I, Q) added to every sample (acquisition.m:30-32 must take it out)."""
    a = np.frombuffer(raw_b, "<i2").astype(np.int64).reshape(-1, 2) + np.asarray(dc, dtype=np.int64)
    assert np.abs(a).max() < 32768
    return a.astype("<i2").tobytes()


def block(label, n_ms, *, sats=None, seed=6102, start_ms=0):
    fs, if_hz, data_type, precision = RATES[label]
    n = n_of(fs)
    sigma = 16.0 if precision == 1 else 900.0
    c = sigma / math.sqrt(n)
    if sats is None:
        sats = [SatSpec(3, 990.0, (2 * n) // 3, 10.0 * c, 0.4), SatSpec(22, -1510.0, 17, 6.0 * c, 1.9)]
    spec = small_spec(fs, if_hz, n, sats=sats, seed=seed, data_type=data_type, data_precision=precision, sigma=sigma)
    raw_b = synth_if(spec, start_ms, n_ms)
    return add_dc(raw_b, DC) if precision == 2 else raw_b


def grid_structs(label, grid="500", datalen=K, **kw):
    fs, if_hz, data_type, precision = RATES[label]
    if grid == "500":
        step, fmin = 500.0, -2000.0
    else:                                            # the fold trap: bins exactly one transform bin Fs/NF apart
        step = fs / nf_of(n_of(fs))
        fmin = -4.0 * step
    return structs(fs, if_hz, data_type=data_type, data_precision=precision, datalen=datalen,
                   freq_min=fmin, freq_step=step, freq_num=9, **kw)


def expected_bases(signal, acq, coh_ms):
    """Forward transforms the planner needs: a bin reuses an earlier base when it is a whole number of transform bins
    (Fs/NF, |shift| < NF/2) away from it, and, with a fold of several ms, also a whole number of Fs/N."""
    fs, n = float(signal.Fs), int(signal.Sample)
    nf = nf_of(n) if n not in (6000, 26000, 58000) else n
    df, dms = fs / nf, fs / n
    bases = []
    for b in range(int(acq.freqNum)):
        f = float(signal.IF) + (float(acq.freqMin) + float(acq.freqStep) * b)
        for g in bases:
            r, q = (f - g) / df, (f - g) / dms
            if (abs(r - round(r)) * df < 1e-6 and abs(round(r)) < nf // 2 and
                    (coh_ms == 1 or nf == n or abs(q - round(q)) * dms < 1e-6)):
                break
        else:
            bases.append(f)
    return len(bases)


def cfg_from(file, signal, acq, prns, **kw):
    return gnssacq.config_from_structs(file, signal, acq, prns=prns, **kw)


def rb(rows):
    return [bytes(r) for r in rows]


def oracle_surfaces(raw_b, file, signal, acq, prns, coh_ms):
    n, kk = int(signal.Sample), int(acq.datalen)
    raw = samples_from_bytes(raw_b, file.dataType, file.dataPrecision)
    carrier = carrier_table(signal, acq, coh_ms)
    conj_spectra = np.conj(np.fft.fft(folded_blocks(raw, carrier, n, kk, coh_ms), axis=-1))
    want = [correlation_surface(raw, signal, acq, p, coh_ms=coh_ms, carrier=carrier, conj_spectra=conj_spectra)
            for p in prns]
    return want, [peak_and_snr(w, signal, acq, p) for w, p in zip(want, prns)]


def snap_doppler(rows, ref, acq):
    """The fold-trap grid's step Fs/NF is not a binary fraction, so K4's fma(step, b, freq_min) and the oracle's
    Doppler may differ in the last bits: within 1e-9 of a step they are the same bin's, and the oracle's value is
    taken so that assert_rows_match checks everything else exactly."""
    out = []
    for g, r in zip(rows, ref):
        g2 = api.Result.from_buffer_copy(g)
        if g.doppler_bin == r.doppler_bin and abs(g.doppler_hz - r.doppler_hz) <= 1e-9 * float(acq.freqStep):
            g2.doppler_hz = r.doppler_hz
        out.append(g2)
    return out


def test_planner_expectation_of_the_fold_trap():
    """The grid the cell-by-cell test uses for the fold trap: one base for a 1-ms block (every bin is a shift of the
    first), one base per bin for a 2-ms fold (Fs/NF is not a whole number of Fs/N)."""
    for label in ("2.048", "16.368", "13.001"):
        file, signal, acq = grid_structs(label, "trap")
        assert expected_bases(signal, acq, 1) == 1
        assert expected_bases(signal, acq, 2) == 9


@pytest.mark.parametrize("grid", ["500", "trap"])
@pytest.mark.parametrize("coh_ms", [1, 2])
@pytest.mark.parametrize("label", list(RATES))
def test_padded_rates_cell_by_cell_on_every_engine(label, coh_ms, grid):
    """Every cell of read_surface (a [B][N] surface: lags < N only) against acquisition.m:52-61 in float64, within
    1e-5 of the maximum, for every variant and exchange of the chosen transform; rows against :62-74; the forward
    bases the planner made; and the rows of a handle without the kept surface (the cooperative kernel's other row
    end) byte for byte."""
    file, signal, acq = grid_structs(label, grid)
    n = int(signal.Sample)
    nf = nf_of(n)
    cfg0 = cfg_from(file, signal, acq, PRNS, coh_ms=coh_ms)
    assert api.transform_size(cfg0) == nf
    raw_b = block(label, K * coh_ms)
    want, ref = oracle_surfaces(raw_b, file, signal, acq, PRNS, coh_ms)
    nb = expected_bases(signal, acq, coh_ms)
    for r, t, x in VARIANTS[nf]:
        what = f"{label} MHz N={n} NF={nf} M={coh_ms} grid={grid} R={r} T={t} X={x}"
        with api.Searcher(cfg_from(file, signal, acq, PRNS, coh_ms=coh_ms, keep_surface=True,
                                   cluster_ctas=r, threads=t, exchange=x)) as s:
            rows = s.search(raw_b)
            assert s.last_stats.n_bases == nb, what
            for i, (prn, w) in enumerate(zip(PRNS, want)):
                got = s.read_surface(i)
                assert got.shape == w.shape == (9, n)
                err = np.abs(got - w).max()
                assert err <= 1e-5 * w.max(), f"{what} PRN {prn}: {err / w.max():.3g} of the maximum"
                gi, wi = int(np.argmax(got)), int(np.argmax(w))
                if gi != wi:
                    assert w.flat[gi] >= w.flat[wi] * (1.0 - TIE_TOL), f"{what} PRN {prn}: argmax {gi} != {wi}"
        assert_rows_match(snap_doppler(rows, ref, acq), ref, what=what)
        assert all(0 <= g.code_phase < n for g in rows), what
        with api.Searcher(cfg_from(file, signal, acq, PRNS, coh_ms=coh_ms, cluster_ctas=r, threads=t, exchange=x)) as s:
            assert rb(s.search(raw_b)) == rb(rows), what


@pytest.mark.parametrize("label", ["2.048", "4.092", "13.001", "16.368", "29"])
def test_satellites_at_the_edge_lags(label):
    """Satellites at lags 0, 1, w-1, w, N-w and N-1, each on a grid bin: the row end must report them at those lags
    with the oracle's noise windows clipped to [0, N) -- the padded lags N .. NF-1 hold the wrapped-around
    correlation and must never win, enter the sum or the window."""
    fs, if_hz, data_type, precision = RATES[label]
    n = n_of(fs)
    w = int(math.ceil(fs / 1.023e6))
    lags = [0, 1, w - 1, w, n - w, n - 1]
    prns = [1, 5, 9, 13, 17, 21]
    sigma = 16.0 if precision == 1 else 900.0
    c = sigma / math.sqrt(n)
    sats = [SatSpec(p, -1500.0 + 500.0 * (i % 6), lag, 12.0 * c, 0.3 * i) for i, (p, lag) in enumerate(zip(prns, lags))]
    file, signal, acq = grid_structs(label, "500")
    raw_b = block(label, K, sats=sats)
    ref = oracle_rows(raw_b, file, signal, acq, prns)
    for r, t, x in VARIANTS[nf_of(n)]:
        with api.Searcher(cfg_from(file, signal, acq, prns, cluster_ctas=r, threads=t, exchange=x)) as s:
            rows = s.search(raw_b)
        what = f"{label} MHz R={r} T={t} X={x}"
        assert_rows_match(rows, ref, what=what)
        # the reported code phase is the oracle's, at or next to each satellite's lag (mod N)
        assert [g.code_phase for g in rows] == [o.code_phase for o in ref], what
        assert all(min((g.code_phase - lag) % n, (lag - g.code_phase) % n) <= 1 for g, lag in zip(rows, lags)), what
        assert all(g.acquired for g in rows), what


def test_full_shape_16368():
    """32 PRNs x 41 bins x 20 ms at 16.368 MHz (N = 16 368 in NF = 58 000), every row against the oracle; a 500 Hz
    grid is not a whole number of Fs/NF = 282.2 Hz, so every bin has its own forward base."""
    fs, if_hz = 16.368e6, 4.092e6
    n = n_of(fs)
    file, signal, acq = structs(fs, if_hz, datalen=20, freq_min=-10000.0, freq_step=500.0, freq_num=41)
    sats = [SatSpec(p, d, cd, a, 0.2 * p) for p, d, cd, a in
            [(2, 3210.0, 5000, 2.2), (7, -4470.0, 123, 1.8), (11, 760.0, n - 3, 1.6), (19, -8990.0, 9001, 2.0),
             (26, 6120.0, 16, 1.3), (31, -250.0, 14000, 1.9)]]
    spec = small_spec(fs, if_hz, n, sats=sats)
    raw_b = synth_if(spec, 0, 20)
    prns = list(range(1, 33))
    with api.Searcher(cfg_from(file, signal, acq, prns)) as s:
        rows = s.search(raw_b)
        st = s.last_stats
    assert st.n_bases == 41
    assert_rows_match(rows, oracle_rows_chunked(raw_b, file, signal, acq, prns), what="16.368 MHz 32 x 41 x 20")
    got = {r.prn: r for r in rows if r.acquired}
    for sat in sats:                                 # (the oracle's code phase: at or next to the synthesised delay)
        assert sat.prn in got and abs(got[sat.prn].code_phase - sat.codedelay) <= 1, sat.prn


@pytest.mark.parametrize("label", ["4.092", "16.368"])
def test_features_are_byte_identical_at_padded_rates(label, tmp_path):
    """Doppler windows against bin-range handles, the block-granular tail against whole rows, gnssacq_sweep and
    gnssacq_sweep_file against single searches, gnssacq_search_multi against one handle: the same bytes."""
    fs, if_hz, data_type, precision = RATES[label]
    n = n_of(fs)
    file, signal, acq = grid_structs(label, "500")
    prns = [3, 22, 9, 14, 30]
    bps = data_type * precision
    blob = block(label, 40)
    raw_b = blob[:K * n * bps]
    with api.Searcher(cfg_from(file, signal, acq, prns)) as s:
        full = rb(s.search(raw_b))
        # Doppler windows: PRN i keeps bins [i, i + 3]
        lo = [-2000.0 + 500.0 * i for i in range(len(prns))]
        hi = [x + 1500.0 for x in lo]
        s.set_doppler_windows(lo, hi)
        win = rb(s.search(raw_b))
        s.clear_doppler_windows()
        assert rb(s.search(raw_b)) == full
        # sweeps
        windows = [blob[j * 7 * n * bps:(j * 7 + K) * n * bps] for j in range(4)]
        single = [rb(s.search(w)) for w in windows]
        assert [rb(r) for r in s.sweep(windows)] == single
        rec = tmp_path / "rec.bin"
        rec.write_bytes(blob)
        assert [rb(r) for r in s.sweep_file(str(rec), 0, 7, 4)] == single
    for i, p in enumerate(prns):
        cfg = cfg_from(file, signal, acq, [p])
        cfg.bin_first, cfg.bin_count = i, 4
        with api.Searcher(cfg) as b:
            assert rb(b.search(raw_b)) == [win[i]], p
    with api.Searcher(cfg_from(file, signal, acq, prns, exchange=3, work_split=1)) as a, \
            api.Searcher(cfg_from(file, signal, acq, prns, exchange=3, work_split=2)) as b:
        whole = rb(a.search(raw_b))
        split = rb(b.search(raw_b))
        assert b.last_stats.work_split == 2
    assert split == whole == full
    with api.Searcher(cfg_from(file, signal, acq, prns[:2])) as a, api.Searcher(cfg_from(file, signal, acq, prns[2:])) as b:
        assert rb(api.search_multi([a, b], raw_b)) == full


def test_exchange_refuses_a_padded_handle():
    file, signal, acq = grid_structs("16.368", "500")
    cfg = cfg_from(file, signal, acq, [3, 22, 9, 14])
    mine, sh = api.shard_plan(cfg, 0, 2)
    with api.Searcher(mine) as s:
        with pytest.raises(gnssacq.GnssAcqError) as e:
            s.xchg_root(sh)
        assert e.value.code == -7
        s.search(block("16.368", K))                 # still a working handle
    mine1, sh1 = api.shard_plan(cfg, 1, 2)
    with api.Searcher(mine1) as s1:                  # (refused before the IPC handle is opened)
        with pytest.raises(gnssacq.GnssAcqError) as e:
            s1.xchg_attach(sh1, bytes(api.IPC_BYTES))
        assert e.value.code == -7


@pytest.mark.parametrize("label", ["2.048", "4.092", "16.368"])
def test_fft_forward_is_the_n_point_dft(label):
    """gnssacq_fft_forward of a padded handle: the N-point DFT (Bluestein through the NF-point engine) against
    numpy.fft.fft in float64, within 1e-5 of max|X| (DESIGN.md records the achieved error)."""
    fs, if_hz, data_type, precision = RATES[label]
    n = n_of(fs)
    file, signal, acq = grid_structs(label, "500")
    rng = np.random.default_rng(n)
    with api.Searcher(cfg_from(file, signal, acq, [1])) as s:
        for x in (rng.standard_normal(n) + 1j * rng.standard_normal(n),
                  np.exp(2j * np.pi * 0.123 * np.arange(n)) + 0.01 * rng.standard_normal(n),
                  np.r_[1.0, np.zeros(n - 1)], np.ones(n)):
            x = x.astype(np.complex64)
            got = s.fft_forward(x)
            want = np.fft.fft(x.astype(np.complex128))
            err = np.abs(got - want).max() / np.abs(want).max()
            assert err <= 1e-5, f"{label} MHz N={n}: {err:.3g} of max|X|"


@pytest.mark.parametrize("fmt", ["iq8", "real8"])
@pytest.mark.parametrize("fs,if_hz", [(4.092e6, 1.023e6), (16.368e6, 4.092e6)])
def test_fine_frequency_at_padded_rates(fs, if_hz, fmt):
    """acquisition.m:83-127 with its K*L N-point DFTs done as Bluestein convolutions through the NF-point engine."""
    data_type = 2 if fmt == "iq8" else 1
    n = n_of(fs)
    file, signal, acq = structs(fs, if_hz, data_type=data_type, data_precision=1, datalen=K)
    L = int(acq.L)
    sats = [SatSpec(3, 1234.0, (n // 3) | 1, 2.0), SatSpec(22, -2611.0, n - 1, 1.5)]
    spec = small_spec(fs, if_hz, n, sats=sats, data_type=data_type, data_precision=1)
    raw_long = synth_if(spec, 0, L + 1)
    longraw = samples_from_bytes(raw_long, data_type, 1)
    with api.Searcher(cfg_from(file, signal, acq, [s.prn for s in sats])) as s:
        got = s.fine_frequency(raw_long, L, [s.prn for s in sats], [s.codedelay for s in sats])
        again = s.fine_frequency(raw_long, L, [s.prn for s in sats], [s.codedelay for s in sats])
    assert list(got) == list(again)
    assert_fine_frequency_matches(got, longraw, file, signal, acq, sats)


def test_tracking_at_16368():
    """gnssacq_track at 16.368 MHz against the oracle's loop (the tracking kernels never needed a built N)."""
    test_gpu_tracking.test_device_side_tracking_loop_against_the_oracle_loop(16.368e6, 4.092e6, 2, 1, 25)


def test_acquisition_wrapper_end_to_end_at_16368():
    """gnssacq.acquisition(file, signal, acq) on a synthetic 16.368 MHz recording: the oracle's sv, codedelay,
    Doppler and fineFreq."""
    fs, if_hz = 16.368e6, 4.092e6
    n = n_of(fs)
    file, signal, acq = structs(fs, if_hz, datalen=4, freq_min=-5000.0, freq_step=500.0, freq_num=21)
    sats = [SatSpec(4, 1500.0, 7000, 1.6), SatSpec(12, -3000.0, 300, 1.4), SatSpec(27, 2500.0, n - 5, 1.5)]
    spec = small_spec(fs, if_hz, n, sats=sats)
    blob = synth_if(spec, 0, 16)
    file.fid, file.skip = io.BytesIO(blob), 1
    got = gnssacq.acquisition(file, signal, acq, verbose=False)
    file.fid = io.BytesIO(blob)
    want = oracle.acquisition(file, signal, acq)
    gnssacq.release_all()
    assert list(got["sv"]) == list(want["sv"]) and {s.prn for s in sats} <= {int(v) for v in got["sv"]}
    assert list(got["codedelay"]) == list(want["codedelay"])
    assert list(got["Doppler"]) == list(want["Doppler"])
    res = fs / (int(acq.L) * n * int(acq.datalen))
    assert np.abs(got["fineFreq"] - want["fineFreq"]).max() <= res * 1.0001
