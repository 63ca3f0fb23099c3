"""Per-PRN Doppler windows (gnssacq_set_doppler_windows) on device 0 (`-m gpu`).

A windowed PRN's row must be byte for byte the row of a one-PRN handle made with bin_first / bin_count over its
window, and match the float64 oracle run on the window's grid.  Windows of mixed widths (the first bin, the last bin,
a single bin, bounds between bins, the full grid, a window that holds no bin) on every engine variant and exchange,
with int8 I/Q and with int16 I/Q carrying a DC offset."""
import ctypes as C
import dataclasses
import math

import numpy as np
import pytest
import torch

import gnssacq
from gnssacq import api
from oracle.synth import SatSpec, synth_if
from helpers import assert_rows_match, oracle_rows, small_spec, structs
from test_gpu_formats import add_dc, front_end
from test_gpu_parity import VARIANTS

pytestmark = pytest.mark.gpu

FORMATS = {"iq8": (2, 1), "iq16": (2, 2)}           # (data_type, data_precision)
K = 2
FMIN, STEP, NBINS = -2000.0, 500.0, 9               # bins -2000 .. 2000 Hz
PRNS = [3, 22, 9, 7, 11, 14]
WINDOWS = [(500.0, 1500.0),                          # PRN 3: three bins around its truth
           (-2000.0, -2000.0),                       # PRN 22: the first bin only
           (2000.0, 2000.0),                         # PRN 9 (absent): the last bin only
           (-1e9, 1e9),                              # PRN 7: the full grid
           (100.0, 400.0),                           # PRN 11: no bin
           (-1600.0, 600.0)]                         # PRN 14: bounds between bins (bins -1500 .. 500)
FULL = [(-1e9, 1e9)] * len(PRNS)


def window_bins(lo, hi, fmin=FMIN, step=STEP, nbins=NBINS):
    return [b for b in range(nbins) if lo <= fmin + step * b <= hi]


def grid(n, fmt):
    data_type, precision = FORMATS[fmt]
    fs, if_hz = front_end(n, data_type)
    return structs(fs, if_hz, data_type=data_type, data_precision=precision, datalen=K,
                   freq_min=FMIN, freq_step=STEP, freq_num=NBINS)


def make_block(n, fmt, *, start_ms=0, seed=6102, dc=(300, -450)):
    data_type, precision = FORMATS[fmt]
    fs, if_hz = front_end(n, data_type)
    sigma = 16.0 if precision == 1 else 900.0
    c = sigma / math.sqrt(n)
    sats = [SatSpec(3, 990.0, (2 * n) // 3, 10.0 * c, 0.4), SatSpec(22, -1510.0, 17, 6.0 * c, 1.9),
            SatSpec(7, 1480.0, n // 5, 8.0 * c, 0.7), SatSpec(14, -470.0, n // 2, 9.0 * c, 2.5)]
    spec = small_spec(fs, if_hz, n, sats=sats, seed=seed, data_type=data_type, data_precision=precision, sigma=sigma)
    raw_b = synth_if(spec, start_ms, K)
    return add_dc(raw_b, n, dc) if precision == 2 else raw_b


def cfg_for(n, fmt, prns=PRNS, **kw):
    file, signal, acq = grid(n, fmt)
    return gnssacq.config_from_structs(file, signal, acq, prns=prns, device=0, **kw)


def set_windows(s, windows):
    s.set_doppler_windows([w[0] for w in windows], [w[1] for w in windows])


def row_bytes(rows):
    return [bytes(r) for r in rows]


def assert_not_searched(row, prn):
    assert row.prn == prn and row.acquired == 0 and math.isnan(row.snr_db) and row.peak == -1.0, prn


def single_prn_row(n, fmt, prn, bins, raw_b, **variant):
    # keep_surface as on the windowed handle: the cooperative kernel's surface path sums the squares in another order
    cfg = cfg_for(n, fmt, prns=[prn], keep_surface=True, **variant)
    cfg.bin_first, cfg.bin_count = bins[0], len(bins)
    with api.Searcher(cfg) as s:
        return bytes(s.search(raw_b)[0])


def oracle_window_row(raw_b, n, fmt, prn, bins):
    """acquisition.m with acq.freqMin at the window's first bin and acq.freqNum its bin count, doppler_bin moved onto
    the handle's full grid."""
    file, signal, _ = grid(n, fmt)
    _, _, acq = structs(signal.Fs, signal.IF, datalen=K, freq_min=FMIN + STEP * bins[0], freq_step=STEP,
                        freq_num=len(bins))
    row = oracle_rows(raw_b, file, signal, acq, [prn])[0]
    return dataclasses.replace(row, doppler_bin=row.doppler_bin + bins[0])


@pytest.mark.parametrize("fmt", ["iq8", "iq16"])
@pytest.mark.parametrize("n", [6000, 26000, 58000])
def test_windowed_rows_on_every_engine(n, fmt):
    """For every engine variant: each windowed row is byte-identical to a one-PRN bin_first / bin_count handle's,
    it matches the oracle on the window's grid, the kept surface holds the unwindowed handle's rows inside the
    windows and zeros outside, all-full-grid windows and cleared windows give the unwindowed bytes."""
    raw_b = make_block(n, fmt)
    searched = [(i, p, window_bins(*w)) for i, (p, w) in enumerate(zip(PRNS, WINDOWS)) if window_bins(*w)]
    ref = {p: oracle_window_row(raw_b, n, fmt, p, bins) for _, p, bins in searched}
    for r, t, x in VARIANTS[n]:
        variant = dict(cluster_ctas=r, threads=t, exchange=x)
        what = f"N={n} {fmt} R={r} T={t} X={x}"
        with api.Searcher(cfg_for(n, fmt, keep_surface=True, **variant)) as u, \
                api.Searcher(cfg_for(n, fmt, keep_surface=True, **variant)) as w:
            full = row_bytes(u.search(raw_b))
            full_surf = [u.read_surface(i) for i in range(len(PRNS))]
            set_windows(w, WINDOWS)
            rows = w.search(raw_b)
            for i, p, bins in searched:
                assert bytes(rows[i]) == single_prn_row(n, fmt, p, bins, raw_b, **variant), f"{what} PRN {p}"
                assert_rows_match([rows[i]], [ref[p]], what=what)
                surf = w.read_surface(i)
                inside = np.zeros(NBINS, dtype=bool)
                inside[bins] = True
                assert np.array_equal(surf[inside], full_surf[i][inside]), f"{what} PRN {p}"
                assert not surf[~inside].any(), f"{what} PRN {p}"
            assert_not_searched(rows[PRNS.index(11)], 11)
            assert not w.read_surface(PRNS.index(11)).any()
            set_windows(w, FULL)
            assert row_bytes(w.search(raw_b)) == full, what
            w.clear_doppler_windows()
            assert row_bytes(w.search(raw_b)) == full, what


@pytest.mark.parametrize("fmt", ["iq8", "iq16"])
@pytest.mark.parametrize("n", [6000, 26000, 58000])
def test_windows_changed_between_enqueues(n, fmt):
    """Windows set between two stream-ordered searches: each search's rows are its own window set's (the call waits
    for the earlier search before it rewrites the tables)."""
    raw_b = make_block(n, fmt)
    other = [(-1e9, 1e9), (-1000.0, 0.0), (-2000.0, 2000.0), (0.0, 0.0), (-2000.0, -1500.0), (1.0, 2.0)]
    with api.Searcher(cfg_for(n, fmt)) as s:
        set_windows(s, WINDOWS)
        want_a = row_bytes(s.search(raw_b))
        set_windows(s, other)
        want_b = row_bytes(s.search(raw_b))
        d_if = torch.frombuffer(bytearray(raw_b), dtype=torch.uint8).to("cuda:0")
        size = len(PRNS) * C.sizeof(api.Result)
        out = [torch.zeros(size, dtype=torch.uint8, device="cuda:0") for _ in range(2)]
        torch.cuda.synchronize(0)
        set_windows(s, WINDOWS)
        s.enqueue_device_out(d_if.data_ptr(), d_if.numel(), out[0].data_ptr())
        set_windows(s, other)
        s.enqueue_device_out(d_if.data_ptr(), d_if.numel(), out[1].data_ptr())
        s.fetch_stats()
        got = [bytes(o.cpu().numpy()) for o in out]
    assert got[0] == b"".join(want_a) and got[1] == b"".join(want_b)


@pytest.mark.parametrize("fmt", ["iq8", "iq16"])
@pytest.mark.parametrize("n", [6000, 26000, 58000])
def test_sweeps_and_multi_use_the_windows(n, fmt, tmp_path):
    """gnssacq_sweep and gnssacq_sweep_file with windows: window i's rows equal gnssacq_search of window i with the
    same windows.  gnssacq_search_multi: each handle searches with its own windows."""
    blocks = [make_block(n, fmt, start_ms=3 * i, dc=(300 - 100 * i, -450 + 80 * i)) for i in range(3)]
    rec = tmp_path / "rec.bin"
    rec.write_bytes(b"".join(blocks))
    with api.Searcher(cfg_for(n, fmt)) as s:
        set_windows(s, WINDOWS)
        want = [row_bytes(s.search(b)) for b in blocks]
        assert [row_bytes(r) for r in s.sweep(blocks)] == want
        assert [row_bytes(r) for r in s.sweep_file(str(rec), 0, K, 3)] == want
    half = len(PRNS) // 2
    with api.Searcher(cfg_for(n, fmt, prns=PRNS[:half])) as a, api.Searcher(cfg_for(n, fmt, prns=PRNS[half:])) as b:
        set_windows(a, WINDOWS[:half])
        set_windows(b, WINDOWS[half:])
        assert row_bytes(api.search_multi([a, b], blocks[0])) == want[0]


def test_block_tail_for_a_small_window_set():
    """32 PRNs on the 41-bin grid at N = 58 000 deal out whole rows; one bin per PRN (32 rows on the resident
    groups) switches the cooperative kernel to the block-granular tail with the same rows, and work_split = 1 in the
    config keeps whole rows."""
    n = 58000
    file, signal, acq = structs(58e6, 4.58e6, datalen=K)
    prns = list(range(1, 33))
    sats = [SatSpec(p, -3000.0 + 250.0 * p, (997 * p) % n, 1.0, 0.3 * p) for p in (2, 5, 13, 21, 30)]
    raw_b = synth_if(small_spec(58e6, 4.58e6, n, sats=sats), 0, K)
    lo = [-10000.0 + 500.0 * ((7 * i) % 41) for i in range(32)]
    with api.Searcher(gnssacq.config_from_structs(file, signal, acq, prns=prns, device=0, exchange=3)) as s, \
            api.Searcher(gnssacq.config_from_structs(file, signal, acq, prns=prns, device=0, exchange=3,
                                                     work_split=1)) as whole:
        full = s.search(raw_b)
        assert s.last_stats.work_split == 1
        s.set_doppler_windows(lo, lo)
        rows = row_bytes(s.search(raw_b))
        assert s.last_stats.work_split == 2
        whole.set_doppler_windows(lo, lo)
        assert row_bytes(whole.search(raw_b)) == rows
        assert whole.last_stats.work_split == 1
        for i in range(32):
            if full[i].doppler_hz == lo[i]:          # the full grid's winner lies inside the window
                assert rows[i] == bytes(full[i]), prns[i]
        s.clear_doppler_windows()
        assert row_bytes(s.search(raw_b)) == row_bytes(full) and s.last_stats.work_split == 1


def test_refusals():
    """Malformed windows are GNSSACQ_ERR_INVALID_ARG; bin- or row-range handles and the exchange are
    GNSSACQ_ERR_STATE, both ways round."""
    n, fmt = 26000, "iq8"
    cfg = cfg_for(n, fmt)
    P = len(PRNS)
    lo = np.zeros(P)
    hi = np.full(P, 500.0)
    with api.Searcher(cfg) as s:
        h = s._h
        lib = api.lib
        assert lib.gnssacq_set_doppler_windows(h, lo.ctypes.data, None) == -1
        assert lib.gnssacq_set_doppler_windows(h, None, hi.ctypes.data) == -1
        assert lib.gnssacq_set_doppler_windows(h, hi.ctypes.data, lo.ctypes.data) == -1          # lo > hi
        nan = lo.copy()
        nan[2] = np.nan
        assert lib.gnssacq_set_doppler_windows(h, nan.ctypes.data, hi.ctypes.data) == -1
        assert lib.gnssacq_set_doppler_windows(h, lo.ctypes.data, nan.ctypes.data) == -1
        assert lib.gnssacq_set_doppler_windows(h, lo.ctypes.data, hi.ctypes.data) == 0
        mine0, sh0 = api.shard_plan(cfg, 0, 2)
        mine1, sh1 = api.shard_plan(cfg, 1, 2)
        with api.Searcher(mine0) as root, api.Searcher(mine1) as other:
            root.xchg_root(sh0)
            for call in (lambda: s.xchg_root(sh0), lambda: s.xchg_attach(sh1, b"\0" * api.IPC_BYTES),
                         lambda: s.xchg_attach_local(sh1, root)):
                with pytest.raises(gnssacq.GnssAcqError) as e:
                    call()
                assert e.value.code == -7
            other.xchg_attach_local(sh1, root)
            for shard in (root, other):
                with pytest.raises(gnssacq.GnssAcqError) as e:
                    shard.set_doppler_windows(np.zeros(shard.cfg.n_prn), np.zeros(shard.cfg.n_prn))
                assert e.value.code == -7
    ranged = cfg_for(n, fmt)
    ranged.bin_first, ranged.bin_count = 2, 3
    rows = cfg_for(n, fmt)
    rows.row_first, rows.row_count = 5, 20
    for c in (ranged, rows):
        with api.Searcher(c) as s:
            with pytest.raises(gnssacq.GnssAcqError) as e:
                set_windows(s, WINDOWS)
            assert e.value.code == -7
    with api.Searcher(cfg) as s:                     # cleared windows: the handle may become a root again
        set_windows(s, WINDOWS)
        s.clear_doppler_windows()
        s.xchg_root(api.shard_plan(cfg, 0, 1)[1])


def test_windows_without_a_bin_skip_the_search_kernel():
    """No PRN has a bin: K1 and K4 still run, K2 is not launched, and every row reads as not searched."""
    n, fmt = 26000, "iq16"
    raw_b = make_block(n, fmt)
    with api.Searcher(cfg_for(n, fmt)) as s:
        set_windows(s, WINDOWS)
        s.search(raw_b)
        launches = s.last_stats.kernel_launches
        set_windows(s, [(1.0, 2.0)] * len(PRNS))
        rows = s.search(raw_b)
        assert s.last_stats.kernel_launches == launches - 1
        for p, r in zip(PRNS, rows):
            assert_not_searched(r, p)


def test_closing_windowed_handles_returns_all_device_memory(tmp_path):
    """Three cycles of handles that set windows (growing the schedule into the block-granular tail, with a kept
    surface), search, sweep and clear them, then close.  Free device memory after cycles 2 and 3 is what it was after
    cycle 1."""
    torch.cuda.init()
    n, fmt = 26000, "iq16"
    blocks = [make_block(n, fmt, start_ms=3 * i) for i in range(2)]
    free = []
    for _ in range(3):
        for x in (1, 2, 3):
            with api.Searcher(cfg_for(n, fmt, keep_surface=True, exchange=x)) as s:
                s.search(blocks[0])
                set_windows(s, WINDOWS)
                s.search(blocks[0])
                s.sweep(blocks)
                set_windows(s, [(0.0, 0.0)] + [(1.0, 2.0)] * (len(PRNS) - 1))
                s.search(blocks[1])
                s.clear_doppler_windows()
                s.search(blocks[1])
        torch.cuda.synchronize(0)
        free.append(torch.cuda.mem_get_info(0)[0])
    assert abs(free[1] - free[0]) <= 2 << 20 and abs(free[2] - free[0]) <= 2 << 20, free
