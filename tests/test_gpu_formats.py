"""Every input format on every engine (`-m gpu`): real int8 and int16 I/Q with DC removal (acquisition.m:28-38) at
N = 6000, 26 000 and 58 000, against the float64 oracle; Doppler grids off the 1 kHz lattice; the fine-frequency
stage, the re-acquisition sweeps and the peer-memory exchange with both formats.

The format decides which code runs: comb_kernel and wipe2_kernel branch on the bytes per sample (1 real int8, 2 int8
I/Q, 4 int16 I/Q), the comb pitch and wipe2's staging depend on them and on Q, and the one shipped shape whose
staging does not fit in shared memory (Q = 29, 4 CTAs x 512 threads, int16, 2-ms fold) runs the gather K1
(wipe_pad_kernel) instead."""
import math

import numpy as np
import pytest

import gnssacq
from gnssacq import api
from oracle.acquisition_ref import carrier_table, correlation_surface, folded_blocks, peak_and_snr, samples_from_bytes
from oracle.synth import SatSpec, synth_if
from helpers import (TIE_TOL, assert_fine_frequency_matches, assert_rows_match, oracle_rows, small_spec, structs)
from test_gpu_parity import VARIANTS

pytestmark = pytest.mark.gpu

FORMATS = {"real8": (1, 1), "iq16": (2, 2)}         # (data_type, data_precision)
PRNS = [3, 22, 9]                                    # strong, weak, absent
K = 2
DC_A, DC_B = (300, -450), (-200, 350)                # int16 DC offsets (I, Q) of two different blocks


def front_end(n, data_type):
    fs, if_hz = {6000: (6e6, 1.25e6), 26000: (26e6, 0.0), 58000: (58e6, 4.58e6)}[n]
    if data_type == 1 and if_hz == 0.0:
        if_hz = 6.5e6                                # a real signal at IF 0 would put every satellite's mirror in the grid
    return fs, if_hz


def grid(n, fmt, **kw):
    data_type, precision = FORMATS[fmt]
    fs, if_hz = front_end(n, data_type)
    return structs(fs, if_hz, data_type=data_type, data_precision=precision, datalen=K,
                   freq_min=-2000.0, freq_step=500.0, freq_num=9, **kw)


def add_dc(raw_b, n, dc):
    """int16 I/Q bytes with dc[m] = (I, Q) added to every sample of ms m (a single pair: the same for every ms)."""
    a = np.frombuffer(raw_b, "<i2").astype(np.int64).reshape(-1, n, 2)
    a = a + np.asarray(dc, dtype=np.int64).reshape(-1, 1, 2)
    assert np.abs(a).max() < 32768
    return a.astype("<i2").tobytes()


def make_block(n, fmt, n_ms, *, start_ms=0, seed=6102, dc=DC_A):
    """PRN 3 strong, PRN 22 weak, PRN 9 absent: amplitudes scaled with sigma / sqrt(N), so that every N has the same
    per-block correlation SNR.  int16 gets `dc` on top (the mean removal must take it out)."""
    data_type, precision = FORMATS[fmt]
    fs, if_hz = front_end(n, data_type)
    sigma = 16.0 if precision == 1 else 900.0
    c = sigma / math.sqrt(n)
    sats = [SatSpec(3, 990.0, (2 * n) // 3, 10.0 * c, 0.4), SatSpec(22, -1510.0, 17, 6.0 * c, 1.9)]
    spec = small_spec(fs, if_hz, n, sats=sats, seed=seed, data_type=data_type, data_precision=precision, sigma=sigma)
    raw_b = synth_if(spec, start_ms, n_ms)
    return add_dc(raw_b, n, dc) if precision == 2 else raw_b


def cfg_from(file, signal, acq, prns, **kw):
    return gnssacq.config_from_structs(file, signal, acq, prns=prns, **kw)


def row_bytes(rows):
    return [bytes(r) for r in rows]


def assert_same_argmax(got, want, what):
    """First-index argmax of the FP32 surface = the float64 one's, unless the oracle's two best cells are a tie."""
    i, j = int(np.argmax(got)), int(np.argmax(want))
    if i != j:
        assert want.flat[i] >= want.flat[j] * (1.0 - TIE_TOL), f"{what}: argmax {i} != {j}"


@pytest.mark.parametrize("coh_ms", [1, 2])
@pytest.mark.parametrize("fmt", ["real8", "iq16"])
@pytest.mark.parametrize("n", [6000, 26000, 58000])
def test_every_format_on_every_engine_cell_by_cell(n, fmt, coh_ms):
    """Every cell of every PRN's surface against acquisition.m:52-61 in float64, for every engine variant and
    exchange; the rows against :62-74.  The oracle surface is computed once and shared by the variants."""
    file, signal, acq = grid(n, fmt)
    raw_b = make_block(n, fmt, K * coh_ms)
    raw = samples_from_bytes(raw_b, file.dataType, file.dataPrecision)
    carrier = carrier_table(signal, acq, coh_ms)
    conj_spectra = np.conj(np.fft.fft(folded_blocks(raw, carrier, n, K, coh_ms), axis=-1))
    want = [correlation_surface(raw, signal, acq, p, coh_ms=coh_ms, carrier=carrier, conj_spectra=conj_spectra)
            for p in PRNS]
    ref = [peak_and_snr(w, signal, acq, p) for w, p in zip(want, PRNS)]
    launches = {}
    for r, t, x in VARIANTS[n]:
        what = f"N={n} {fmt} M={coh_ms} R={r} T={t} X={x}"
        with api.Searcher(cfg_from(file, signal, acq, PRNS, coh_ms=coh_ms, keep_surface=True,
                                   cluster_ctas=r, threads=t, exchange=x)) as s:
            rows = s.search(raw_b)
            launches[(r, t, x)] = s.last_stats.kernel_launches
            for i, (prn, w) in enumerate(zip(PRNS, want)):
                got = s.read_surface(i)
                err = np.abs(got - w).max()
                assert err <= 1e-5 * w.max(), f"{what} PRN {prn}: {err / w.max():.3g} of the maximum"
                assert_same_argmax(got, w, f"{what} PRN {prn}")
        assert_rows_match(rows, ref, what=what)
    # K1 is comb_kernel + wipe2_kernel (2 launches) wherever wipe2's staging fits in 227 KB of shared memory; the one
    # shipped shape where it does not (233 728 B) runs wipe_pad_kernel (1 launch).  The last variant of each N is a comb one.
    no_comb = (n, fmt, coh_ms) == (58000, "iq16", 2)
    comb = launches[VARIANTS[n][-1]]
    assert launches == {v: comb - int(no_comb and v[:2] == (4, 512)) for v in launches}
    if no_comb:
        assert launches[(4, 512, 1)] == launches[(8, 256, 1)] - 1


# (N, fs, IF, step, freq_min, freq_num): steps that do not divide 1 kHz, steps above it, a freq_min off the step's
# lattice, and an off-nominal fs that still rounds to N = 6000 (then fs/N != 1 kHz and no bin is a shift of another)
GRIDS = [
    (6000, 6e6, 1.25e6, 300.0, -1500.0, 11),
    (26000, 26e6, 0.0, 750.0, -3000.0, 9),
    (58000, 58e6, 4.58e6, 1500.0, -6000.0, 9),
    (6000, 6e6, 1.25e6, 2000.0, -8000.0, 9),
    (26000, 26e6, 0.0, 500.0, -2125.0, 9),
    (58000, 58e6, 4.58e6, 300.0, -2125.0, 13),
    (6000, 5.9999e6, 1.25e6, 500.0, -2000.0, 9),
]


@pytest.mark.parametrize("n,fs,if_hz,step,fmin,num", GRIDS)
def test_doppler_grid_off_the_1khz_lattice(n, fs, if_hz, step, fmin, num):
    """plan_bins: bins that are a whole number of FFT bins (fs/N) apart share one forward transform and are searched
    as circular shifts of it.  The number of bases is the number of classes of IF + freq_min + step*b modulo fs/N; a
    satellite sits on a bin that is reached through a non-zero shift."""
    file, signal, acq = structs(fs, if_hz, datalen=K, freq_min=fmin, freq_step=step, freq_num=num)
    assert int(signal.Sample) == n
    if fs / n == 1000.0:
        cls = [(if_hz + fmin + step * b) % 1000.0 for b in range(num)]     # whole Hz here: exact in float64
    else:
        cls = list(range(num))               # fs/N = 999.983 Hz: no two bins are a whole number of FFT bins apart
    shifted = [b for b in range(num) if cls.index(cls[b]) != b]
    target = shifted[-1] if shifted else num // 2
    # strong enough (per-block correlation SNR ~ 450) that a neighbour bin, 300 Hz off, cannot win on noise
    c = 16.0 / math.sqrt(n)
    sats = [SatSpec(5, fmin + step * target, (n * 3) // 5, 30.0 * c, 0.8), SatSpec(12, fmin + step, 211, 5.0 * c, 2.2)]
    raw_b = synth_if(small_spec(fs, if_hz, n, sats=sats), 0, K)
    prns = [5, 12, 30]
    with api.Searcher(cfg_from(file, signal, acq, prns)) as s:
        rows = s.search(raw_b)
        assert s.last_stats.n_bases == len(set(cls))
    assert rows[0].doppler_bin == target
    assert_rows_match(rows, oracle_rows(raw_b, file, signal, acq, prns), what=f"N={n} fs={fs} step={step} fmin={fmin}")


@pytest.mark.parametrize("fmt", ["real8", "iq16"])
@pytest.mark.parametrize("n", [26000, 58000])
def test_fine_frequency_formats(n, fmt):
    """acquisition.m:83-127 at Q = 13 and Q = 29 for real int8 and for int16 I/Q with a DC offset (:92-94 removes the
    mean of the (L+1)-ms read); K = 2 keeps the oracle's L*N*K-point spectrum small."""
    data_type, precision = FORMATS[fmt]
    fs, if_hz = front_end(n, data_type)
    file, signal, acq = structs(fs, if_hz, data_type=data_type, data_precision=precision, datalen=K)
    L = int(acq.L)
    big = precision == 2
    sats = [SatSpec(3, 1234.0, (n // 3) | 1, 90.0 if big else 2.0), SatSpec(22, -2611.0, n - 1, 70.0 if big else 1.5)]
    spec = small_spec(fs, if_hz, n, sats=sats, data_type=data_type, data_precision=precision, sigma=900.0 if big else 16.0)
    raw_long = synth_if(spec, 0, L + 1)
    if big:
        raw_long = add_dc(raw_long, n, DC_A)
    longraw = samples_from_bytes(raw_long, data_type, precision)
    with api.Searcher(cfg_from(file, signal, acq, [s.prn for s in sats])) as s:
        got = s.fine_frequency(raw_long, L, [s.prn for s in sats], [s.codedelay for s in sats])
    assert_fine_frequency_matches(got, longraw, file, signal, acq, sats)


@pytest.mark.parametrize("fmt", ["real8", "iq16"])
@pytest.mark.parametrize("n", [6000, 58000])
def test_sweeps_with_both_formats(n, fmt, tmp_path):
    """gnssacq_sweep and gnssacq_sweep_file with 1 and 4 bytes per sample: every window's rows are the bytes
    gnssacq_search gives for it, window 0 matches the oracle.  The int16 recording's DC drifts from ms to ms, so a
    mean left over from another window would change the rows; sweep_file also checks the byte offsets of a window."""
    data_type, precision = FORMATS[fmt]
    skip, epoch, n_win = 3, 5, 4
    total_ms = skip + epoch * (n_win - 1) + K
    blob = make_block(n, fmt, total_ms, dc=[(300 - 40 * m, -450 + 55 * m) for m in range(total_ms)])
    rec = tmp_path / "rec.bin"
    rec.write_bytes(blob)
    ms_bytes = n * data_type * precision
    windows = [blob[(skip + epoch * j) * ms_bytes:(skip + epoch * j + K) * ms_bytes] for j in range(n_win)]
    file, signal, acq = grid(n, fmt)
    with api.Searcher(cfg_from(file, signal, acq, PRNS)) as s:
        single = [row_bytes(s.search(w)) for w in windows]
        assert [row_bytes(rows) for rows in s.sweep(windows)] == single
        assert [row_bytes(rows) for rows in s.sweep(windows[::-1])] == single[::-1]
        swept = s.sweep_file(str(rec), skip, epoch, n_win)
        assert [row_bytes(rows) for rows in swept] == single
    assert_rows_match(swept[0], oracle_rows(windows[0], file, signal, acq, PRNS), what=f"sweep_file N={n} {fmt} window 0")


@pytest.mark.parametrize("plan,world", [("prn", 2), ("prn", 5), ("rows", 2), ("rows", 4)])
@pytest.mark.parametrize("fmt", ["real8", "iq16"])
def test_peer_exchange_with_both_formats(fmt, plan, world):
    """gnssacq_xchg_* with shards on one device (run one after the other): over two steps with different blocks the
    rows are byte for byte the single-handle search's, whole PRNs, Doppler-bin ranges (more shards than PRNs) or
    row ranges per shard."""
    from gnssacq.dist import LocalMultiGpu
    n = 26000
    file, signal, acq = grid(n, fmt)
    cfg = cfg_from(file, signal, acq, PRNS)
    a = make_block(n, fmt, K, dc=DC_A)
    b = make_block(n, fmt, K, start_ms=7, seed=77, dc=DC_B)
    with api.Searcher(cfg) as s:
        want_a, want_b = row_bytes(s.search(a)), row_bytes(s.search(b))
    assert want_a != want_b
    with LocalMultiGpu(cfg, [0] * world, plan=plan) as m:
        assert m.serial
        assert row_bytes(m.search(a)) == want_a
        assert row_bytes(m.search(b)) == want_b


def test_peer_exchange_refuses_the_shape_without_comb_rows():
    """The exchange pulls the IF block with comb_kernel, which the Q = 29 / 4 x 512 / int16 / 2-ms shape does not run:
    making such a handle a root is refused (GNSSACQ_ERR_STATE) and so is a step, before anything is launched that
    another shard could wait on.  The handle itself still searches, with wipe_pad_kernel."""
    n, fmt = 58000, "iq16"
    file, signal, acq = grid(n, fmt)
    raw_b = make_block(n, fmt, 2 * K)
    cfg = cfg_from(file, signal, acq, PRNS, coh_ms=2, cluster_ctas=4, threads=512)
    mine, sh = api.shard_plan(cfg, 0, 2)
    with api.Searcher(mine) as root:
        with pytest.raises(gnssacq.GnssAcqError) as e:
            root.xchg_root(sh)
        assert e.value.code == -7
        with pytest.raises(gnssacq.GnssAcqError) as e:
            root.xchg_enqueue(raw_b)
        assert e.value.code == -7
        rows = root.search(raw_b)
    assert_rows_match(rows, oracle_rows(raw_b, file, signal, acq, mine.prn[:mine.n_prn], coh_ms=2), what="v1 root")


def test_non_root_shard_takes_its_means_from_the_block_it_pulled():
    """int16 on two GPUs: a non-root shard reads the IF block out of the root's HBM once the root has announced it.
    Its DC means must come from that block too, not from whatever the root's buffer holds when the shard starts: the
    root is held back (a sleep ahead of its upload) while the other shard is already running, and the rows must still
    be the single-handle bytes of the new block."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs: shards that wait for one another never share a device")
    from gnssacq.dist import LocalMultiGpu
    n, fmt = 6000, "iq16"
    file, signal, acq = grid(n, fmt)
    cfg = cfg_from(file, signal, acq, PRNS)
    a = make_block(n, fmt, K, dc=DC_A)
    b = make_block(n, fmt, K, start_ms=7, seed=77, dc=DC_B)
    with api.Searcher(cfg) as s:
        want_a, want_b = row_bytes(s.search(a)), row_bytes(s.search(b))
    with LocalMultiGpu(cfg, [0, 1]) as m:
        assert not m.serial
        assert row_bytes(m.search(a)) == want_a
        root = m.searchers[0]
        held = torch.cuda.Stream(device=0)
        try:
            with torch.cuda.device(0), torch.cuda.stream(held):
                torch.cuda._sleep(100_000_000)       # tens of ms: far inside the exchange's ~4 s flag time-out
            root.set_stream(held.cuda_stream)
            got_b = row_bytes(m.search(b))           # B's upload to the root waits behind the sleep
        finally:
            root.set_stream(-1)                      # GNSSACQ_OWN_STREAM, before `held` goes away
            held.synchronize()
        assert got_b == want_b
        assert row_bytes(m.search(a)) == want_a
