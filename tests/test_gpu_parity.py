"""Parity of the CUDA path (through the C ABI) against the oracle.  `-m gpu`: runs on the B200 box.

Bar (BASELINE.json north_star): code-phase index, Doppler bin and acquired flag bit-exact unless the
oracle's two best cells differ by < 2e-5 relative; peak and SNR within 1e-4 relative (FP32)."""
import io
import math
from types import SimpleNamespace

import numpy as np
import pytest

import oracle
from oracle.acquisition_ref import correlation_surface
from oracle.synth import SatSpec, VirtualFile, synth_if, urban_spec, opensky_spec
import gnssacq
from gnssacq import api
from helpers import structs, small_spec, oracle_rows, assert_rows_match, assert_fine_frequency_matches, METRIC_RTOL

pytestmark = pytest.mark.gpu
import ctypes as _C
C_RESULT = _C.sizeof(api.Result)

# (cluster CTAs, threads, exchange: 1 = DSMEM, 2 = L2-resident buffer)
# exchange: 1 = DSMEM clusters, 2 = L2 buffer + persistent clusters, 3 = L2 buffer + cooperative CTA groups
VARIANTS = {6000: [(2, 128, 1), (1, 256, 1), (2, 128, 2), (1, 256, 2), (2, 128, 3), (1, 256, 3)],
            26000: [(2, 512, 1), (4, 256, 1), (4, 512, 1), (2, 512, 2), (4, 256, 2), (2, 512, 3), (4, 256, 3), (8, 128, 3)],
            58000: [(4, 512, 1), (8, 256, 1), (4, 512, 2), (4, 512, 3), (8, 256, 3), (16, 128, 3)]}


def cfg_from(file, signal, acq, prns, **kw):
    return gnssacq.config_from_structs(file, signal, acq, prns=prns, **kw)


@pytest.mark.parametrize("n", [6000, 26000, 58000])
def test_fft_engine_against_numpy(n):
    rng = np.random.default_rng(n)
    x = (rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64)
    want = np.fft.fft(x.astype(np.complex128))
    for r, t, _ in VARIANTS[n][:3]:
        cfg = gnssacq.make_config(fs_hz=n * 1e3, if_hz=0.0, samples_per_ms=n, prns=[1], freq_num=1,
                                  noncoh_blocks=1, cluster_ctas=r, threads=t)
        with api.Searcher(cfg) as s:
            got = s.fft_forward(x)
        err = np.abs(got - want).max() / np.abs(want).max()
        assert err < 2e-6, (n, r, t, err)


@pytest.mark.parametrize("fs,if_hz", [(6e6, 1.25e6), (26e6, 0.0), (58e6, 4.58e6)])
def test_power_surface_cellwise(fs, if_hz):
    """Every cell of acquisition.m:59's surface, not just the winner."""
    file, signal, acq = structs(fs, if_hz, datalen=2, freq_min=-1000.0, freq_step=500.0, freq_num=5)
    n = int(signal.Sample)
    prns = [3, 9, 22]
    raw_b = synth_if(small_spec(fs, if_hz, n), 0, 2)
    file.fid = io.BytesIO(raw_b)
    raw = oracle.read_if_block(file, signal, 2)
    for r, t, x in VARIANTS[n]:
        cfg = cfg_from(file, signal, acq, prns, keep_surface=True, cluster_ctas=r, threads=t, exchange=x)
        with api.Searcher(cfg) as s:
            rows = s.search(raw_b)
            for i, prn in enumerate(prns):
                want = correlation_surface(raw, signal, acq, prn)
                got = s.read_surface(i)
                assert np.abs(got - want).max() <= 1e-5 * want.max(), (n, r, t, x, prn)
                assert int(np.argmax(got)) == int(np.argmax(want))
        assert_rows_match(rows, oracle_rows(raw_b, file, signal, acq, prns), what=f"N={n} R={r} T={t} X={x}")


def test_urban_shaped_32prn_default_grid():
    """BASELINE config 2 shape (26 MHz, IF 0, 41 bins, 32 PRNs), K = 4 to keep the oracle in seconds."""
    file, signal, acq = structs(26e6, 0.0, datalen=4)
    raw_b = synth_if(urban_spec(), 0, 4)
    prns = list(range(1, 33))
    ref = oracle_rows(raw_b, file, signal, acq, prns)
    for r, t, x in VARIANTS[26000]:
        with api.Searcher(cfg_from(file, signal, acq, prns, cluster_ctas=r, threads=t, exchange=x)) as s:
            rows = s.search(raw_b)
            assert s.last_stats.exchange == x
        ties = assert_rows_match(rows, ref, what=f"urban R={r} T={t} X={x}")
        assert ties <= 2
    got = {r.prn for r in rows if r.acquired}
    assert {1, 3, 11} <= got


def test_opensky_shaped_32prn_default_grid():
    """BASELINE config 1 shape (58 MHz, IF 4.58 MHz, 41 bins, 32 PRNs), K = 2."""
    file, signal, acq = structs(58e6, 4.58e6, datalen=2)
    raw_b = synth_if(opensky_spec(), 0, 2)
    prns = list(range(1, 33))
    ref = oracle_rows(raw_b, file, signal, acq, prns)
    for r, t, x in VARIANTS[58000]:
        with api.Searcher(cfg_from(file, signal, acq, prns, cluster_ctas=r, threads=t, exchange=x)) as s:
            rows = s.search(raw_b)
        assert_rows_match(rows, ref, what=f"opensky R={r} T={t} X={x}")


def test_full_k20_urban_truth_recovery_and_wrapper():
    """Full-size config 2 through the MATLAB-mirroring wrapper: size-independent property = truth table."""
    spec = urban_spec()
    file, signal, acq = gnssacq.initParameters(shape="urban")
    file.fid = VirtualFile(spec)
    file.skip = 40
    out, rows = gnssacq.acquisition(file, signal, acq, verbose=False, return_rows=True, fine=False)
    assert set(out) == {"sv", "SNR", "Doppler", "codedelay", "fineFreq"}
    for k in out:
        assert out[k].dtype == np.float64 and out[k].ndim == 1
    got = {int(p): (int(c), float(d)) for p, c, d in zip(out["sv"], out["codedelay"], out["Doppler"])}
    for s in spec.sats:
        assert s.prn in got, s.prn
        assert got[s.prn][0] == s.codedelay
        assert abs(got[s.prn][1] - s.doppler_hz) <= 250.0
    assert list(out["sv"]) == sorted(out["sv"]) and len(rows) == 32
    # same block via the raw API: bytes in, identical rows out (idempotence)
    file.fid.seek(40 * 26000 * 2)
    raw = file.fid.read(26000 * 2 * 20)
    rows2 = gnssacq.get_searcher(gnssacq.config_from_structs(file, signal, acq)).search(raw)
    assert [(r.code_phase, r.doppler_bin, r.peak) for r in rows] == [(r.code_phase, r.doppler_bin, r.peak) for r in rows2]
    gnssacq.release_all()


@pytest.mark.parametrize("data_type,precision", [(1, 1), (2, 2)])
def test_real_and_int16_formats(data_type, precision):
    """acquisition.m:28-38: int8 real stays real; int16 is I/Q with per-component mean removed."""
    fs, if_hz = 6e6, 1.25e6
    file, signal, acq = structs(fs, if_hz, data_type=data_type, data_precision=precision, datalen=3)
    n = int(signal.Sample)
    spec = small_spec(fs, if_hz, n, data_type=data_type, data_precision=precision,
                      sigma=16.0 if precision == 1 else 900.0,
                      sats=[SatSpec(3, 990.0, 1683, 1.2 if precision == 1 else 70.0), SatSpec(22, 1565.0, 17, 1.5 if precision == 1 else 90.0)])
    raw_b = synth_if(spec, 0, 3)
    if precision == 2:   # add a DC offset the mean removal must take out
        a = np.frombuffer(raw_b, "<i2").copy()
        a[0::2] += 300
        a[1::2] -= 450
        raw_b = a.tobytes()
    prns = [1, 3, 22, 30]
    ref = oracle_rows(raw_b, file, signal, acq, prns)
    with api.Searcher(cfg_from(file, signal, acq, prns)) as s:
        rows = s.search(raw_b)
    assert_rows_match(rows, ref, what=f"type={data_type} prec={precision}")


@pytest.mark.parametrize("coh_ms,step,num", [(2, 250.0, 9), (5, 100.0, 21)])
def test_coherent_fold_and_fine_grid(coh_ms, step, num):
    """SURVEY A.8 extension (BASELINE configs 3 and 5): M-ms coherent fold, sub-kHz Doppler step."""
    fs, if_hz = 6e6, 1.25e6
    file, signal, acq = structs(fs, if_hz, datalen=2, freq_min=-1000.0, freq_step=step, freq_num=num)
    n = int(signal.Sample)
    spec = small_spec(fs, if_hz, n, sats=[SatSpec(3, 240.0, 1683, 0.5), SatSpec(22, -610.0, 17, 0.6)])
    raw_b = synth_if(spec, 0, 2 * coh_ms)
    prns = [3, 8, 22]
    ref = oracle_rows(raw_b, file, signal, acq, prns, coh_ms=coh_ms)
    with api.Searcher(cfg_from(file, signal, acq, prns, coh_ms=coh_ms)) as s:
        rows = s.search(raw_b)
        assert s.last_stats.n_bases == min(num, int(round(1000.0 / step)))
    assert_rows_match(rows, ref, what=f"M={coh_ms}")


def test_edge_cases():
    fs, if_hz = 6e6, 1.25e6
    file, signal, acq = structs(fs, if_hz, datalen=2)
    n = int(signal.Sample)
    prns = [1, 2]
    cfg = cfg_from(file, signal, acq, prns)
    with api.Searcher(cfg) as s:
        # all-zero input: 0/0 -> NaN SNR, nothing acquired, indices = first cell (acquisition.m:62-70)
        rows = s.search(bytes(s.if_bytes))
        for r in rows:
            assert not r.acquired and math.isnan(r.snr_db) and (r.code_phase, r.doppler_bin, r.peak) == (0, 0, 0.0)
        # short buffer -> error code, no crash
        with pytest.raises(gnssacq.GnssAcqError) as e:
            s.search(bytes(s.if_bytes - 2))
        assert e.value.code == -3
        # longer buffer than needed is fine (only the first datalen ms are used)
        raw_b = synth_if(small_spec(fs, if_hz, n), 0, 3)
        a = s.search(raw_b)
        b = s.search(raw_b[: s.if_bytes])
        assert [(r.code_phase, r.peak) for r in a] == [(r.code_phase, r.peak) for r in b]
    # peak in the first / last lags: the +-(w-1) exclusion window is clipped, not wrapped (acquisition.m:67)
    for cd in (0, 2, n - 1):
        spec = small_spec(fs, if_hz, n, sats=[SatSpec(5, 0.0, cd, 3.0)])
        raw_b = synth_if(spec, 0, 2)
        ref = oracle_rows(raw_b, file, signal, acq, [5])
        with api.Searcher(cfg_from(file, signal, acq, [5])) as s:
            rows = s.search(raw_b)
        assert rows[0].code_phase == cd
        assert_rows_match(rows, ref, what=f"edge lag {cd}")
    # single Doppler bin: the reference's max(max(.)) quirk (SURVEY A.5) is NOT replicated
    file1, signal1, acq1 = structs(fs, if_hz, datalen=2, freq_min=0.0, freq_num=1)
    raw_b = synth_if(small_spec(fs, if_hz, n), 0, 2)
    ref = oracle_rows(raw_b, file1, signal1, acq1, [3], matlab_quirks=False)
    with api.Searcher(cfg_from(file1, signal1, acq1, [3])) as s:
        rows = s.search(raw_b)
    assert_rows_match(rows, ref, what="single bin")


def test_prn_shards_concatenate_to_the_full_table():
    """Multi-GPU sharding is PRN-major: the union of shard tables is byte-identical to the 1-GPU table."""
    fs, if_hz = 6e6, 1.25e6
    file, signal, acq = structs(fs, if_hz, datalen=2)
    raw_b = synth_if(small_spec(fs, if_hz, int(signal.Sample)), 0, 2)
    prns = list(range(1, 33))
    with api.Searcher(cfg_from(file, signal, acq, prns)) as s:
        full = [bytes(r) for r in s.search(raw_b)]
    for world in (2, 4, 8):
        parts = []
        for rank in range(world):
            shard = prns[rank * 32 // world:(rank + 1) * 32 // world]
            with api.Searcher(cfg_from(file, signal, acq, shard)) as s:
                parts += [bytes(r) for r in s.search(raw_b)]
        assert parts == full


@pytest.mark.parametrize("fs,if_hz,data_type,precision,datalen", [
    (6e6, 1.25e6, 2, 1, 4), (6e6, 1.25e6, 1, 1, 3), (6e6, 1.25e6, 2, 2, 2), (26e6, 0.0, 2, 1, 20), (58e6, 4.58e6, 2, 1, 20)])
def test_fine_frequency_stage(fs, if_hz, data_type, precision, datalen):
    """SURVEY 8f-1: acquisition.m:83-127 (zero-padded L*N*datalen-point spectrum peak) on the GPU vs the oracle.
    Index exact unless the oracle's two best spectral lines are within the FP32 tie tolerance."""
    file, signal, acq = structs(fs, if_hz, data_type=data_type, data_precision=precision, datalen=datalen)
    n, L = int(signal.Sample), int(acq.L)
    big = precision == 2
    sats = [SatSpec(3, 1234.0, (n // 3) | 1, 90.0 if big else 2.0), SatSpec(22, -2611.0, 17, 70.0 if big else 1.5)]
    if n > 6000:
        sats = sats[:1] + [SatSpec(22, -2611.0, n - 1, 1.5)]
    spec = small_spec(fs, if_hz, n, sats=sats, data_type=data_type, data_precision=precision, sigma=900.0 if big else 16.0)
    raw_long = synth_if(spec, 0, L + 1)
    file.fid = io.BytesIO(raw_long)
    longraw = oracle.read_if_block(file, signal, L + 1)
    prns = [s.prn for s in sats]
    cds = [s.codedelay for s in sats]
    with api.Searcher(cfg_from(file, signal, acq, prns)) as s:
        got = s.fine_frequency(raw_long, L, prns, cds)
        with pytest.raises(gnssacq.GnssAcqError) as e:
            s.fine_frequency(raw_long[:-2], L, prns, cds)
        assert e.value.code == -3
    assert_fine_frequency_matches(got, longraw, file, signal, acq, sats)


def test_wrapper_fills_fine_freq():
    spec = urban_spec()
    file, signal, acq = gnssacq.initParameters(shape="urban")
    file.fid = VirtualFile(spec)
    file.skip = 7
    out = gnssacq.acquisition(file, signal, acq, verbose=False)
    assert len(out["fineFreq"]) == len(out["sv"]) > 0
    truth = {s.prn: s.doppler_hz for s in spec.sats}
    assert set(truth) <= {int(v) for v in out["sv"]}
    for sv, ff in zip(out["sv"], out["fineFreq"]):
        assert np.isfinite(ff)
        if int(sv) in truth:                                      # (a 12 dB threshold also passes the odd noise peak)
            assert abs(ff - signal.IF - truth[int(sv)]) <= 60.0  # 5 Hz bins over a 10 ms window
    gnssacq.release_all()


@pytest.mark.parametrize("shape,prns", [("urban", [1, 2, 3, 11, 22, 30]), ("opensky", [3, 5, 16, 26, 29, 32])])
def test_full_depth_k20_subset_against_oracle(shape, prns):
    """BASELINE configs 1 and 2 at their real depth (41 bins x 20 non-coherent ms) on a PRN subset (present and
    absent satellites), row by row against the oracle; and the same rows must come out of the 32-PRN search."""
    spec = urban_spec() if shape == "urban" else opensky_spec()
    file, signal, acq = gnssacq.initParameters(shape=shape)
    raw_b = synth_if(spec, 3, int(acq.datalen))
    file.dataType, file.dataPrecision = 2, 1
    ref = oracle_rows(raw_b, file, signal, acq, prns)
    with api.Searcher(cfg_from(file, signal, acq, prns)) as s:
        rows = s.search(raw_b)
    assert_rows_match(rows, ref, what=f"{shape} K=20")
    with api.Searcher(cfg_from(file, signal, acq, list(range(1, 33)))) as s:
        full = {r.prn: r for r in s.search(raw_b)}
    for r in rows:                                   # PRN sharding never changes a row (bytes identical)
        assert bytes(full[r.prn]) == bytes(r)
    # ... and neither does the schedule: whole rows per CTA group and the block-granular tail give the same bytes
    for ws in (1, 2):
        with api.Searcher(cfg_from(file, signal, acq, prns, work_split=ws)) as s:
            assert [bytes(r) for r in s.search(raw_b)] == [bytes(r) for r in rows]
            assert s.last_stats.work_split == ws
    with api.Searcher(cfg_from(file, signal, acq, list(range(1, 33)), work_split=2)) as s:
        assert all(bytes(full[r.prn]) == bytes(r) for r in s.search(raw_b))


@pytest.mark.parametrize("n,variant,datalen,prns", [
    (6000, (2, 128, 3), 3, [7]), (6000, (1, 256, 3), 7, [1, 2, 3, 4, 5]),
    (26000, (8, 128, 3), 20, [1]), (26000, (8, 128, 3), 6, [1, 2, 3, 11]), (26000, (4, 256, 3), 7, [3, 30]),
    (26000, (8, 128, 3), 1, [1, 2, 3]),
    (58000, (16, 128, 3), 9, [16]), (58000, (16, 128, 3), 3, [3, 5, 16, 26]), (58000, (8, 256, 3), 2, [16, 32]),
])
def test_block_granular_split_of_few_rows(n, variant, datalen, prns):
    """Few rows on many resident CTA groups (one rank's shard at 8 GPUs, a single-PRN re-acquisition): the
    cooperative kernel cuts tail rows at block granularity and the finishing group adds the published power
    planes in block order.  Rows against the oracle, and byte for byte against the whole-row schedule."""
    if n == 6000:
        fs, if_hz = 6e6, 1.25e6
        file, signal, acq = structs(fs, if_hz, datalen=datalen)
        raw_b = synth_if(small_spec(fs, if_hz, n), 0, datalen)
    else:
        shape = "urban" if n == 26000 else "opensky"
        file, signal, acq = gnssacq.initParameters(shape=shape)
        acq.datalen = datalen
        raw_b = synth_if(urban_spec() if shape == "urban" else opensky_spec(), 3, datalen)
        file.dataType, file.dataPrecision = 2, 1
    ref = oracle_rows(raw_b, file, signal, acq, prns)
    kw = dict(cluster_ctas=variant[0], threads=variant[1], exchange=variant[2])
    with api.Searcher(cfg_from(file, signal, acq, prns, work_split=2, **kw)) as s:
        rows = s.search(raw_b)
        again = s.search(raw_b)
        groups = s.last_stats.resident_clusters
        assert s.last_stats.work_split == (2 if datalen > 1 else 1)
    assert [bytes(r) for r in rows] == [bytes(r) for r in again]          # deterministic
    assert_rows_match(rows, ref, what=f"N={n} {variant} K={datalen} {len(prns)} PRN on {groups} groups")
    with api.Searcher(cfg_from(file, signal, acq, prns, work_split=1, **kw)) as s:
        rows1 = s.search(raw_b)
        assert s.last_stats.work_split == 1
    assert [bytes(r) for r in rows] == [bytes(r) for r in rows1]
    with api.Searcher(cfg_from(file, signal, acq, prns, **kw)) as s:              # auto: either schedule, same bytes
        assert [bytes(r) for r in s.search(raw_b)] == [bytes(r) for r in rows1]


def test_single_process_multi_handle_search():
    """gnssacq_search_multi: PRN shards on several handles (several GPUs when visible, else the same one) in ONE
    process give the bytes of the single-handle table."""
    import torch
    fs, if_hz = 6e6, 1.25e6
    file, signal, acq = structs(fs, if_hz, datalen=2)
    raw_b = synth_if(small_spec(fs, if_hz, int(signal.Sample)), 0, 2)
    prns = list(range(1, 13))
    with api.Searcher(cfg_from(file, signal, acq, prns)) as s:
        full = [bytes(r) for r in s.search(raw_b)]
    ndev = torch.cuda.device_count()
    parts = [api.Searcher(cfg_from(file, signal, acq, prns[i * 4:(i + 1) * 4], device=i % ndev)) for i in range(3)]
    try:
        rows = api.search_multi(parts, raw_b)
    finally:
        for p in parts:
            p.close()
    assert [bytes(r) for r in rows] == full


def test_fresh_handles_agree():
    """Regression (r01): the replica table was copied with a synchronous cudaMemcpy from pageable memory, which
    returns when the data is staged, and K0 ran on the handle's non-blocking stream -- about one handle in ten
    built the last PRNs' code spectra from a half-copied table.  Every fresh handle must give the same bytes."""
    file, signal, acq = structs(26e6, 0.0, datalen=2)
    raw_b = synth_if(urban_spec(), 0, 2)
    prns = list(range(1, 33))
    for variant in [(4, 256, 1), (0, 0, 0)]:
        first = None
        for _ in range(40):
            with api.Searcher(cfg_from(file, signal, acq, prns, cluster_ctas=variant[0], threads=variant[1],
                                       exchange=variant[2])) as s:
                got = [bytes(r) for r in s.search(raw_b)]
            if first is None:
                first = got
            assert got == first


@pytest.mark.parametrize("n,datalen,n_windows", [(6000, 2, 5), (26000, 2, 4), (58000, 1, 3)])
def test_reacquisition_sweep_equals_single_searches(n, datalen, n_windows):
    """gnssacq_sweep (BASELINE config 4: a window every 100 ms, copies overlapped with the searches): every
    window's rows are the bytes gnssacq_search gives for that window, and window 0 matches the oracle."""
    if n == 6000:
        fs, if_hz = 6e6, 1.25e6
        file, signal, acq = structs(fs, if_hz, datalen=datalen)
        spec = small_spec(fs, if_hz, n)
    else:
        shape = "urban" if n == 26000 else "opensky"
        file, signal, acq = gnssacq.initParameters(shape=shape)
        acq.datalen = datalen
        spec = urban_spec() if shape == "urban" else opensky_spec()
    windows = [synth_if(spec, 100 * j, datalen) for j in range(n_windows)]
    file.dataType, file.dataPrecision = 2, 1
    prns = [1, 3, 7, 16, 22, 30]
    with api.Searcher(cfg_from(file, signal, acq, prns)) as s:
        single = [[bytes(r) for r in s.search(w)] for w in windows]
        swept = s.sweep(windows)
        assert s.last_stats.kernel_launches >= 3 * n_windows
        assert [[bytes(r) for r in rows] for rows in swept] == single
        assert s.sweep([]) == []
        again = s.sweep(windows[::-1])                                  # buffers are reused correctly
        assert [[bytes(r) for r in rows] for rows in again] == single[::-1]
        with pytest.raises(gnssacq.GnssAcqError):
            s.sweep([windows[0][:-2]])
    assert_rows_match(swept[0], oracle_rows(windows[0], file, signal, acq, prns), what=f"sweep N={n} window 0")


def test_sweep_from_a_recording_file(tmp_path):
    """gnssacq_sweep_file: the library does acquisition.m:27-34's fseek/fread itself, window j = file.skip advanced by
    epoch_ms per epoch (BASELINE config 4).  Rows per window = gnssacq_search on the bytes acquisition.m would read."""
    fs, if_hz, n = 6e6, 1.25e6, 6000
    file, signal, acq = structs(fs, if_hz, datalen=2)
    spec = small_spec(fs, if_hz, n)
    total_ms, skip, epoch, n_win = 64, 3, 10, 6
    blob = synth_if(spec, 0, total_ms)
    rec = tmp_path / "rec.bin"
    rec.write_bytes(blob)
    prns = [3, 7, 22, 30]
    ms_bytes = n * 2
    with api.Searcher(cfg_from(file, signal, acq, prns)) as s:
        want = [[bytes(r) for r in s.search(blob[(skip + epoch * j) * ms_bytes:(skip + epoch * j + 2) * ms_bytes])]
                for j in range(n_win)]
        got = s.sweep_file(str(rec), skip, epoch, n_win)
        assert [[bytes(r) for r in rows] for rows in got] == want
        assert s.sweep_file(str(rec), skip, epoch, 0) == []
        with pytest.raises(gnssacq.GnssAcqError) as e:                    # the last window would run past the end
            s.sweep_file(str(rec), skip, epoch, 8)
        assert e.value.code == -3
        with pytest.raises(gnssacq.GnssAcqError):
            s.sweep_file(str(tmp_path / "missing.bin"), 0, 10, 1)
        # ... and the handle is still usable afterwards
        assert [bytes(r) for r in s.search(blob[skip * ms_bytes:(skip + 2) * ms_bytes])] == want[0]
    file.fid, file.skip = io.BytesIO(blob), skip
    assert_rows_match(got[0], oracle.coarse_search(oracle.read_if_block(file, signal, 2), signal, acq, prns), what="sweep_file window 0")


@pytest.mark.parametrize("prns,world", [([1, 3, 7, 16, 22, 30], 2), ([1, 3, 7, 16, 22, 30], 4), ([1, 3, 7, 16, 22, 30], 8),
                                        ([7], 4), ([3, 22], 5), ([7], 48)])
def test_peer_memory_exchange_shards_give_the_single_gpu_bytes(prns, world):
    """gnssacq_xchg_* (SURVEY 8e): one acquisition dealt out to `world` shards -- whole PRNs, or Doppler-bin ranges
    when there are fewer PRNs than shards --, candidates written into the root's table, K4 on the root over the full
    grid: the rows are byte for byte the single-handle search's.  (One GPU here: the shards run one after the other;
    on a multi-GPU box they run concurrently -- bench.py --gpus N.)"""
    from gnssacq.dist import LocalMultiGpu
    fs, if_hz, n = 6e6, 1.25e6, 6000
    file, signal, acq = structs(fs, if_hz, datalen=3)
    raw_b = synth_if(small_spec(fs, if_hz, n), 0, 3)
    cfg = cfg_from(file, signal, acq, prns)
    with api.Searcher(cfg) as s:
        want = [bytes(r) for r in s.search(raw_b)]
    with LocalMultiGpu(cfg, [0] * world) as m:
        assert m.serial
        got = m.search(raw_b)
        again = m.search(raw_b)
        st = m.searchers[0].last_stats
    assert [bytes(r) for r in got] == want
    assert [bytes(r) for r in again] == want
    assert st.gather_wait_ms >= 0.0
    assert_rows_match(got, oracle_rows(raw_b, file, signal, acq, prns), what=f"xchg world={world}")


@pytest.mark.parametrize("prns,world,extra", [([1, 3, 7, 16, 22, 30], 2, 0), ([1, 3, 7, 16, 22, 30], 4, 60), ([1, 3, 7, 16, 22, 30], 8, -300),
                                              ([7], 4, 250), ([3, 22], 5, 0), ([7], 48, 0)])
def test_row_range_shards_give_the_single_gpu_bytes(prns, world, extra):
    """gnssacq_shard_plan_rows: the (PRN, bin) rows cut into `world` contiguous ranges of the kernel's own bin-major
    order, the root's share weighted -- a PRN's bins end up on several shards, the root's K4 sees the full table: the
    rows are byte for byte the single-handle search's, whatever the weight."""
    from gnssacq.dist import LocalMultiGpu
    fs, if_hz, n = 6e6, 1.25e6, 6000
    file, signal, acq = structs(fs, if_hz, datalen=3)
    raw_b = synth_if(small_spec(fs, if_hz, n), 0, 3)
    cfg = cfg_from(file, signal, acq, prns)
    with api.Searcher(cfg) as s:
        want = [bytes(r) for r in s.search(raw_b)]
    with LocalMultiGpu(cfg, [0] * world, plan="rows", root_extra_permille=extra) as m:
        assert sum(sh.n_rows for sh in m.shards) == len(prns) * cfg.freq_num
        got = m.search(raw_b)
        again = m.search(raw_b)
    assert [bytes(r) for r in got] == want
    assert [bytes(r) for r in again] == want


def test_row_range_handle_alone_and_full_size():
    """A handle with config.row_first / row_count used alone reports, per PRN, the best of the rows it owns (cells it
    never writes cannot win); and at the Urban front end's size (cooperative kernel, block-granular tail) three row
    ranges with a heavy root reproduce the single-handle bytes."""
    from gnssacq.dist import LocalMultiGpu
    fs, if_hz, n = 6e6, 1.25e6, 6000
    file, signal, acq = structs(fs, if_hz, datalen=2)
    raw_b = synth_if(small_spec(fs, if_hz, n), 0, 2)
    prns = [3, 7]
    with api.Searcher(cfg_from(file, signal, acq, prns)) as s:
        full = s.search(raw_b)
    b = full[0].doppler_bin
    cfg = cfg_from(file, signal, acq, prns)
    cfg.row_first, cfg.row_count = 2 * b, 1                           # exactly PRN 3's winning row (row = bin * n_prn + index)
    with api.Searcher(cfg) as s:
        part = s.search(raw_b)
    assert bytes(part[0]) == bytes(full[0])
    assert part[1].peak == -1.0 and not part[1].acquired            # PRN 7 owns no row here
    from gnssacq.synth import urban_recording
    raw_u = urban_recording().read(0, 4)
    ucfg = gnssacq.make_config(fs_hz=26e6, if_hz=0.0, prns=[1, 3, 11], noncoh_blocks=4)
    with api.Searcher(ucfg) as s:
        want = [bytes(r) for r in s.search(raw_u)]
    with LocalMultiGpu(ucfg, [0, 0, 0], plan="rows", root_extra_permille=400) as m:
        got = m.search(raw_u)
    assert [bytes(r) for r in got] == want


def test_bin_range_handle_alone():
    """A handle that owns bins [b0, b0+n) of the grid (config.bin_first / bin_count) reports its winner in FULL-grid
    bin indices and produces the full search's candidates for those bins (same forward bases)."""
    fs, if_hz, n = 6e6, 1.25e6, 6000
    file, signal, acq = structs(fs, if_hz, datalen=2)
    raw_b = synth_if(small_spec(fs, if_hz, n), 0, 2)
    with api.Searcher(cfg_from(file, signal, acq, [3])) as s:
        full = s.search(raw_b)[0]
    lo = max(full.doppler_bin - 3, 0)
    cfg = cfg_from(file, signal, acq, [3])
    cfg.bin_first, cfg.bin_count = lo, 7
    with api.Searcher(cfg) as s:
        part = s.search(raw_b)[0]
    assert bytes(part) == bytes(full)                                  # the winner's bin is inside the range
    cfg.bin_first, cfg.bin_count = 0, 2                               # a range without the winner: its own best row
    with api.Searcher(cfg) as s:
        other = s.search(raw_b)[0]
    assert other.doppler_bin in (0, 1) and other.peak <= full.peak
    bad = cfg_from(file, signal, acq, [3])
    bad.bin_first, bad.bin_count = 40, 2
    with pytest.raises(gnssacq.GnssAcqError):
        api.Searcher(bad)


def test_fetch_follows_the_last_search_output():
    """gnssacq_fetch_results returns the rows of the LAST enqueued search also when that search wrote them into a
    caller-owned device buffer (gnssacq_enqueue_device_out), and accepts out == NULL for timings only."""
    import torch
    fs, if_hz, n = 6e6, 1.25e6, 6000
    file, signal, acq = structs(fs, if_hz, datalen=2)
    a = synth_if(small_spec(fs, if_hz, n), 0, 2)
    b = synth_if(small_spec(fs, if_hz, n, seed=77), 5, 2)
    prns = [3, 7, 22]
    with api.Searcher(cfg_from(file, signal, acq, prns)) as s:
        with pytest.raises(gnssacq.GnssAcqError) as e:
            s.fetch()
        assert e.value.code == -7                                       # nothing enqueued yet
        rows_a = [bytes(r) for r in s.search(a)]
        rows_b = [bytes(r) for r in s.search(b)]
        assert rows_a != rows_b
        s.search(a)                                                     # the handle's own table now holds A
        d_if = torch.frombuffer(bytearray(b), dtype=torch.uint8).cuda()
        d_out = torch.zeros(len(prns) * C_RESULT, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        s.enqueue_device_out(d_if.data_ptr(), d_if.numel(), d_out.data_ptr())
        assert [bytes(r) for r in s.fetch()] == rows_b                  # not the stale rows of A
        st = s.fetch_stats()
        assert st.search_ms > 0 and st.kernel_launches >= 3


def test_plain_c_example_end_to_end(tmp_path):
    """examples/acquire.c -- the ABI from plain C, no Python in the process: acquire a synthetic Opensky-shaped
    recording from a file and print acquisition.m's lines; the numbers must be the ones the ctypes path gets."""
    import os
    import re
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    pkg = os.path.join(root, "assignment-for-aae6102_gnss-sdr_b200", "gnssacq")
    exe = str(tmp_path / "acquire")
    subprocess.check_call(["gcc", "-O1", "-I", os.path.join(root, "include"), os.path.join(root, "examples", "acquire.c"),
                           "-L", pkg, "-lgnssacq", "-o", exe])
    spec = opensky_spec()
    raw = synth_if(spec, 0, 21)
    rec = tmp_path / "Opensky_synth.bin"
    rec.write_bytes(raw)
    out = subprocess.run([exe, str(rec), "0"], capture_output=True, text=True, timeout=120,
                         env=dict(os.environ, LD_LIBRARY_PATH=pkg))
    assert out.returncode == 0, out.stderr
    got = {int(m.group(1)): (float(m.group(2)), int(m.group(3)), int(m.group(4)))
           for m in re.finditer(r"SV\[\s*(\d+)\] SNR = ([\d.]+), Code phase =\s*(\d+), Raw Doppler =\s*(-?\d+)", out.stdout)}
    fine = {int(m.group(1)): float(m.group(2)) for m in re.finditer(r"SV\[\s*(\d+)\] Fine Doppler =\s*(-?[\d.]+)", out.stdout)}
    file, signal, acq = gnssacq.initParameters(shape="opensky")
    with api.Searcher(cfg_from(file, signal, acq, list(range(1, 33)))) as s:
        rows = [r for r in s.search(raw[: s.if_bytes]) if r.acquired]
        ff = s.fine_frequency(raw, int(acq.L), [r.prn for r in rows], [r.code_phase for r in rows])
    assert sorted(got) == [r.prn for r in rows] and len(rows) >= 6
    for r, f in zip(rows, ff):
        snr, cp, dop = got[r.prn]
        assert cp == r.code_phase and dop == int(r.doppler_hz) and abs(snr - r.snr_db) < 0.006
        assert abs(fine[r.prn] - (f - signal.IF)) < 1e-3
