"""The row end of the search (K3) on every engine (`-m gpu`; the geometry port runs on the CPU).

K3 runs in search_kernel (exchange 1), search_kernel_l2x (2) and search_kernel_coop (3).  All three call one peak scan
over their CTA's column slice (row_scan) and one +-(w-1) window sum clipped at lags 0 and N-1 (window_sum), each over
its accumulator layout: columns of Geo / Split for exchanges 1 and 2, of GeoX / SplitX for exchange 3.  Exchanges 1 and
2 share their cross-CTA reduction (cluster_row_end); exchange 3 has its own.  The cooperative kernel has two scans:
the debug scan (keep_surface: row_scan, cell by cell, GeoX::valid) and the product scan (float4 loads, `vm >= bv`
pruning, padding columns read as exact zeros).  This file checks:

- a NumPy port of Geo / GeoX / Split / SplitX (csrc/gnss_engine.h), on the CPU against the header itself, built with
  g++.  The GPU tests take their lags from the port;
- strong satellites on lags 0, 1, w-1, w, N-w, N-1 and on the first and last valid column of every rank's slice, on
  every variant, through the product scan;
- every (PRN, bin) row's candidate, not only the winner's: one-bin Doppler windows make each row the reported one;
- shifts beyond +-Q FFT bins, cell by cell: 101 bins at 1 kHz from -50 kHz (one forward base, shifts 0..+100), the
  same bins listed from the top (shifts 0..-100), and 101 bins at 250 Hz (four bases);
- the product scan against the debug scan (keep_surface 0 / 1);
- a strong block, an all-zero block and the strong block again on one handle: nothing survives a search.

plan_bins makes the first bin a grid's base, so an ascending grid has shifts >= 0 only; the descending grid
(freq_step < 0) is what reaches the negative branch of Geo::shift_coords.

Bounds are the other GPU tests': cells within 1e-5 of the surface maximum, the same first argmax unless the oracle's
top two cells are a TIE_TOL tie, rows through assert_rows_match.  Two bounds are new:
- noise_meansq within METRIC_RTOL (1e-4) of the oracle's wherever the row names the oracle's cell.  It is the mean of
  the same FP32 cells that the SNR is built from, and the SNR already has to meet 1e-4.
- product scan against debug scan: every field but the two double sums must be bit-identical, because both scans pick
  one cell of one accumulator.  noise_meansq and snr_db may differ by 1e-12 relative, because the scans add the same
  squares in another order (exchanges 1 and 2 have one scan only, so there the rows are byte-identical)."""
import dataclasses
import math
import os
import subprocess
from functools import lru_cache

import numpy as np
import pytest

import gnssacq
from gnssacq import api
from oracle.acquisition_ref import carrier_table, correlation_surface, folded_blocks, peak_and_snr, samples_from_bytes
from oracle.synth import SatSpec, synth_if
from helpers import METRIC_RTOL, assert_rows_match, oracle_rows, small_spec, structs
from test_gpu_formats import assert_same_argmax, front_end
from test_gpu_parity import VARIANTS

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "assignment-for-aae6102_gnss-sdr_b200",
                    "csrc")
SCAN_RTOL = 1e-12                                    # product vs debug scan: the two double sums only
K = 2
FMIN, STEP, NBINS = -2000.0, 500.0, 9                # bins -2000 .. 2000 Hz
SIGMA = 16.0                                         # int8 I/Q noise per component


# ------------------------------------------------------------------ geometry port (csrc/gnss_engine.h)
class Geo:
    """Geo<Q>, GeoX<Q>, Split<Q, R> and SplitX<Q, R> in NumPy (every function takes arrays)."""

    def __init__(self, q):
        self.q, self.n, self.row = q, 2000 * q, 125 * q
        m1, m2, m3 = 125 * q, 16 * q, 2000
        self.m = (m1, m2, m3)
        self.inv = (pow(m1 % 16, -1, 16), pow(m2 % 125, -1, 125), pow(m3 % q, -1, q))
        self.e = (m1 * self.inv[0], m2 * self.inv[1], m3 * self.inv[2])         # CRT idempotents
        self.nt = 5 * q
        self.ntp = self.nt + (self.nt & 1)
        self.rsx = 25 * self.ntp

    def crt(self, a, b, c):
        return (a * self.e[0] + b * self.e[1] + c * self.e[2]) % self.n

    def good(self, a, b, c):
        return (a * self.m[0] + b * self.m[1] + c * self.m[2]) % self.n

    # Geo<Q>: column (c', pos) of an a-row, pos = 25 k1 + k2 holds b' = k1 + 5 k2
    def lag_of(self, ap, col):
        cp, pos = col // 125, col % 125
        return self.crt(ap, pos // 25 + 5 * (pos % 25), cp)

    def cell_of_lag(self, m):
        bp = m % 125
        return m & 15, (m % self.q) * 125 + 25 * (bp % 5) + bp // 5

    def shift_coords(self, s):
        sm = s % self.n                              # NumPy's modulo is already in [0, N)
        return sm * self.inv[0] % 16, sm * self.inv[1] % 125, sm * self.inv[2] % self.q

    # GeoX<Q>: [16 a'][25 k2][NTP], t = c'*5 + k1 fastest; t = 5Q is padding when 5Q is odd
    def x_valid(self, e):
        return (e < self.rsx) & (e % self.ntp < self.nt)

    def x_lag_of(self, ap, e):
        k2, t = e // self.ntp, e % self.ntp
        return self.crt(ap, t % 5 + 5 * k2, t // 5)

    def x_cell_of_lag(self, m):
        bp = m % 125
        return m & 15, (bp // 5) * self.ntp + (m % self.q) * 5 + bp % 5

    def ch(self, r):                                 # Split<Q, R>::CH
        return 2 * ((self.row + 2 * r - 1) // (2 * r))

    def chx(self, r):                                # SplitX<Q, R>::CHX
        return 2 * ((self.rsx + 2 * r - 1) // (2 * r))

    def rank_columns(self, r, exchange):
        """The valid columns of every rank's K3 slice: [rank*CH, +CH) of the ROW columns (exchanges 1 and 2), or
        [rank*CHX, +CHX) of the exchange layout (exchange 3).  The last rank's slice may be partial."""
        if exchange == 3:
            w = self.chx(r)
            return [c[self.x_valid(c)] for c in (np.arange(k * w, (k + 1) * w) for k in range(r))]
        w = self.ch(r)
        return [c[c < self.row] for c in (np.arange(k * w, (k + 1) * w) for k in range(r))]

    def lag_in_layout(self, ap, col, exchange):
        return self.x_lag_of(ap, col) if exchange == 3 else self.lag_of(ap, col)


def slice_edge_lags(geo, r, exchange):
    """The lags of the first and the last valid column of every rank's slice, on a-rows that differ from rank to rank."""
    out = []
    for k, cols in enumerate(geo.rank_columns(r, exchange)):
        out.append(int(geo.lag_in_layout((5 * k + 3) % 16, cols[0], exchange)))
        out.append(int(geo.lag_in_layout((5 * k + 11) % 16, cols[-1], exchange)))
    return out


def window_edge_lags(n):
    w = math.ceil(front_end(n, 2)[0] / 1.023e6)      # acquisition.m:66
    return [0, 1, w - 1, w, n - w, n - 1]


_DUMP = r"""
#include <cstdio>
#include "gnss_engine.h"
using namespace gnss;
static void put(FILE* f, int v) { std::fwrite(&v, sizeof v, 1, f); }
template <int Q> static void dump(FILE* f) {
    using G = Geo<Q>;
    using X = GeoX<Q>;
    for (int ap = 0; ap < 16; ++ap) for (int c = 0; c < G::ROW; ++c) put(f, G::lag_of(ap, c));
    for (int ap = 0; ap < 16; ++ap) for (int e = 0; e < X::RSX; ++e) put(f, X::valid(e) ? X::lag_of(ap, e) : -1);
    for (int m = 0; m < G::N; ++m) { int ap, c; G::cell_of_lag(m, ap, c); put(f, ap); put(f, c); }
    for (int m = 0; m < G::N; ++m) { int ap, e; X::cell_of_lag(m, ap, e); put(f, ap); put(f, e); }
    for (int s = -G::N / 2; s <= G::N / 2; ++s) { int a, b, c; G::shift_coords(s, a, b, c); put(f, a); put(f, b); put(f, c); }
    put(f, X::RSX);
    put(f, Split<Q, 1>::CH); put(f, Split<Q, 2>::CH); put(f, Split<Q, 4>::CH); put(f, Split<Q, 8>::CH); put(f, Split<Q, 16>::CH);
    put(f, SplitX<Q, 1>::CHX); put(f, SplitX<Q, 2>::CHX); put(f, SplitX<Q, 4>::CHX); put(f, SplitX<Q, 8>::CHX);
    put(f, SplitX<Q, 16>::CHX);
}
int main(int, char** argv) {
    FILE* f = std::fopen(argv[1], "wb");
    if (!f) return 1;
    dump<3>(f); dump<13>(f); dump<29>(f);
    return std::fclose(f) == 0 ? 0 : 1;
}
"""


@pytest.fixture(scope="module")
def header_maps(tmp_path_factory):
    """The index maps as csrc/gnss_engine.h computes them (host build with g++), per Q."""
    d = tmp_path_factory.mktemp("geo")
    src, exe, out = d / "dump.cpp", d / "dump", d / "maps.bin"
    src.write_text(_DUMP)
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-I", CSRC, str(src), "-o", str(exe)])
    subprocess.check_call([str(exe), str(out)])
    raw = np.fromfile(out, dtype=np.int32)
    maps, at = {}, 0

    def take(k):
        nonlocal at
        at += k
        return raw[at - k:at]
    for q in (3, 13, 29):
        g = Geo(q)
        maps[q] = dict(lag=take(16 * g.row).reshape(16, g.row), xlag=take(16 * g.rsx).reshape(16, g.rsx),
                       cell=take(2 * g.n).reshape(g.n, 2), xcell=take(2 * g.n).reshape(g.n, 2),
                       shift=take(3 * (g.n + 1)).reshape(g.n + 1, 3), rsx=int(take(1)[0]),
                       ch=take(5).tolist(), chx=take(5).tolist())
    assert at == raw.size
    return maps


@pytest.mark.parametrize("q", [3, 13, 29])
def test_geometry_port(q, header_maps):
    """The port is the header: cell_of_lag(lag_of(.)) and lag_of(cell_of_lag(.)) are identities over every lag, in both
    layouts; every map equals the header's; a lag's CRT residues are its cell's coordinates; the Good map of
    shift_coords(s) is s mod N; the rank slices of every R partition the valid columns."""
    g, h = Geo(q), header_maps[q]
    m = np.arange(g.n)
    ap, col = g.cell_of_lag(m)
    assert np.array_equal(g.lag_of(ap, col), m)
    xap, e = g.x_cell_of_lag(m)
    assert g.x_valid(e).all() and np.array_equal(g.x_lag_of(xap, e), m)
    aa, cc = np.meshgrid(np.arange(16), np.arange(g.row), indexing="ij")
    lag = g.lag_of(aa, cc)
    assert np.array_equal(np.sort(lag.ravel()), m)                         # 16 x ROW cells: every lag once
    assert np.array_equal(g.cell_of_lag(lag)[1], cc)
    assert np.array_equal(lag % 16, aa) and np.array_equal(lag % q, cc // 125)
    assert np.array_equal(lag % 125, (cc % 125) // 25 + 5 * (cc % 25))
    aa, ee = np.meshgrid(np.arange(16), np.arange(g.rsx), indexing="ij")
    ok = g.x_valid(ee)
    xlag = np.where(ok, g.x_lag_of(aa, ee), -1)
    assert np.array_equal(np.sort(xlag[ok]), m)
    assert np.array_equal(g.x_cell_of_lag(xlag[ok])[1], ee[ok])
    assert np.array_equal(h["lag"], lag) and np.array_equal(h["xlag"], xlag)
    assert np.array_equal(h["cell"], np.stack([ap, col], 1)) and np.array_equal(h["xcell"], np.stack([xap, e], 1))
    s = np.arange(-(g.n // 2), g.n // 2 + 1)
    sa, sb, sc = g.shift_coords(s)
    assert np.array_equal(h["shift"], np.stack([sa, sb, sc], 1))
    assert np.array_equal(g.good(sa, sb, sc), s % g.n)
    assert h["rsx"] == g.rsx
    rs = [1, 2, 4, 8, 16]
    assert h["ch"] == [g.ch(r) for r in rs] and h["chx"] == [g.chx(r) for r in rs]
    for r in rs:
        for x, width, valid in ((1, g.row, np.arange(g.row)), (3, g.rsx, np.flatnonzero(g.x_valid(np.arange(g.rsx))))):
            cols = g.rank_columns(r, x)
            assert all(c.size for c in cols) and np.array_equal(np.concatenate(cols), valid), (r, x)
            lags = slice_edge_lags(g, r, x)
            assert len(set(lags)) == len(lags) == 2 * r and all(0 <= v < g.n for v in lags)
    # the last rank's slice is partial (CHX * R > RSX) on shipped cooperative variants of Q = 13 and 29, so the GPU
    # tests aim at a last valid column that is not the slice's last column
    if q > 3:
        assert any(r * g.chx(r) > g.rsx for r, _, x in VARIANTS[g.n] if x == 3)


# ------------------------------------------------------------------ shared GPU fixtures
def grid(n, *, fmin=FMIN, step=STEP, num=NBINS, k=K):
    fs, if_hz = front_end(n, 2)
    return structs(fs, if_hz, datalen=k, freq_min=fmin, freq_step=step, freq_num=num)


def cfg_for(n, prns, *, coh_ms=1, **kw):
    file, signal, acq = grid(n, **{k: kw.pop(k) for k in ("fmin", "step", "num") if k in kw})
    return gnssacq.config_from_structs(file, signal, acq, prns=prns, coh_ms=coh_ms, device=0, **kw)


def block(n, sats, n_ms, seed=6102):
    fs, if_hz = front_end(n, 2)
    return synth_if(small_spec(fs, if_hz, n, sats=sats, seed=seed, sigma=SIGMA), 0, n_ms)


def amp(n, a):
    """Amplitude whose per-block correlation amplitude is `a` times the noise's, at every N."""
    return a * SIGMA / math.sqrt(n)


def row_bytes(rows):
    return [bytes(r) for r in rows]


def set_windows(s, windows):
    s.set_doppler_windows([w[0] for w in windows], [w[1] for w in windows])


def variant_kw(r, t, x, ws=0):
    return dict(cluster_ctas=r, threads=t, exchange=x, work_split=ws)


def splits(x):
    return (1, 2) if x == 3 else (0,)


def assert_rows_and_noise(gpu_rows, ref_rows, what):
    """assert_rows_match, and noise_meansq within METRIC_RTOL of the oracle's where the row names the oracle's cell."""
    assert_rows_match(gpu_rows, ref_rows, what=what)
    for g, r in zip(gpu_rows, ref_rows):
        if (g.code_phase, g.doppler_bin) == (r.code_phase, r.doppler_bin):
            assert abs(g.noise_meansq - r.noise_meansq) <= METRIC_RTOL * r.noise_meansq, \
                f"{what} PRN {r.prn}: noise {g.noise_meansq} vs {r.noise_meansq}"


def assert_same_scan(prod, dbg, exchange, what):
    """Product scan (keep_surface 0) against debug scan (keep_surface 1)."""
    if exchange != 3:
        assert row_bytes(prod) == row_bytes(dbg), what
        return
    for a, b in zip(prod, dbg):
        for f in ("prn", "acquired", "code_phase", "doppler_bin", "doppler_hz", "peak"):
            assert getattr(a, f) == getattr(b, f), f"{what} PRN {a.prn}: {f} {getattr(a, f)} vs {getattr(b, f)}"
        for f in ("noise_meansq", "snr_db"):
            u, v = getattr(a, f), getattr(b, f)
            assert (math.isnan(u) and math.isnan(v)) or abs(u - v) <= SCAN_RTOL * abs(v), f"{what} PRN {a.prn}: {f} {u} vs {v}"


# ------------------------------------------------------------------ peaks on the edges of the row end
EDGE_PRNS = [2, 5, 8, 11, 14, 17, 20, 23, 26, 29]    # one satellite each per block
EDGE_AMP = 40.0
# (40x the noise's correlation amplitude: at N = 58 000, 57 samples per chip, the lag next to the peak is only 1.8 %
# weaker, and the peak has to land on the aimed lag, not beside it)


@lru_cache(maxsize=None)
def edge_blocks(n):
    """Blocks of len(EDGE_PRNS) strong satellites on the union of the edge lags of every variant of N (the last block is
    filled up from the first lags), each with its lags, bins and oracle rows."""
    geo = Geo(n // 2000)
    lags = set(window_edge_lags(n))
    for r, _, x in VARIANTS[n]:
        lags.update(slice_edge_lags(geo, r, x))
    lags = sorted(lags)
    per = len(EDGE_PRNS)
    lags += lags[:(-len(lags)) % per]
    file, signal, acq = grid(n)
    out = []
    for j in range(0, len(lags), per):
        part = lags[j:j + per]
        bins = [(2 * i + j // per) % NBINS for i in range(per)]
        sats = [SatSpec(p, FMIN + STEP * b, lag, amp(n, EDGE_AMP), 0.37 * i)
                for i, (p, lag, b) in enumerate(zip(EDGE_PRNS, part, bins))]
        raw_b = block(n, sats, K, seed=6102 + j)
        out.append((raw_b, part, bins, oracle_rows(raw_b, file, signal, acq, EDGE_PRNS)))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("n", [6000, 26000, 58000])
def test_peaks_on_the_edges_of_the_row_end(n):
    """Every variant (exchange 3 with whole rows and with the block-granular tail), product scan: satellites on lags 0, 1,
    w-1, w, N-w, N-1 and on the first / last valid column of every rank's slice of every variant of N.  Code phase and
    bin are the aimed ones, rows and noise_meansq match the oracle, the debug scan gives the same rows."""
    blocks = edge_blocks(n)
    for r, t, x in VARIANTS[n]:
        for ws in splits(x):
            what = f"N={n} R={r} T={t} X={x} split={ws}"
            with api.Searcher(cfg_for(n, EDGE_PRNS, **variant_kw(r, t, x, ws))) as prod, \
                    api.Searcher(cfg_for(n, EDGE_PRNS, keep_surface=True, **variant_kw(r, t, x, ws))) as dbg:
                for j, (raw_b, lags, bins, ref) in enumerate(blocks):
                    rows = prod.search(raw_b)
                    st = prod.last_stats
                    assert st.exchange == x and (x != 3 or st.work_split == ws), what
                    assert [g.code_phase for g in rows] == lags, f"{what} block {j}"
                    assert [g.doppler_bin for g in rows] == bins, f"{what} block {j}"
                    assert_rows_and_noise(rows, ref, f"{what} block {j}")
                    assert_same_scan(rows, dbg.search(raw_b), x, f"{what} block {j}")


# ------------------------------------------------------------------ every row's candidate
CAND_PRNS = [3, 22, 7, 9, 14]                        # PRN 9 is absent: its rows are pure noise


def candidate_block(n, coh_ms):
    w = window_edge_lags(n)[3]
    sats = [SatSpec(3, 990.0, 0, amp(n, 10.0), 0.4), SatSpec(22, -1510.0, n - 1, amp(n, 6.0), 1.9),
            SatSpec(7, 1480.0, w, amp(n, 8.0), 0.7), SatSpec(14, -470.0, (2 * n) // 3, amp(n, 3.0), 2.5)]
    return block(n, sats, K * coh_ms)


def oracle_surfaces(raw_b, signal, acq, prns, coh_ms):
    """acquisition.m:52-61 for every PRN of `prns`, sharing the forward spectra."""
    n = int(signal.Sample)
    raw = samples_from_bytes(raw_b, 2, 1)
    carrier = carrier_table(signal, acq, coh_ms)
    conj_spectra = np.conj(np.fft.fft(folded_blocks(raw, carrier, n, int(acq.datalen), coh_ms), axis=-1))
    return [correlation_surface(raw, signal, acq, p, coh_ms=coh_ms, carrier=carrier, conj_spectra=conj_spectra)
            for p in prns]


@pytest.mark.gpu
@pytest.mark.parametrize("coh_ms", [1, 3])
@pytest.mark.parametrize("n", [6000, 26000, 58000])
def test_every_rows_candidate_through_one_bin_windows(n, coh_ms):
    """Windows lo = hi = f_b for every PRN make row (p, b) the reported one.  Each is checked against acquisition.m:62-74
    on that one row of the oracle surface (no max(max(.)) quirk), bin moved back onto the full grid; product and debug
    scan agree.  Every variant at N = 6000 and 26 000, the automatic one and (8, 256, 3) at 58 000."""
    file, signal, acq = grid(n)
    raw_b = candidate_block(n, coh_ms)
    surf = oracle_surfaces(raw_b, signal, acq, CAND_PRNS, coh_ms)
    want = []
    for b in range(NBINS):
        acq_b = grid(n, fmin=FMIN + STEP * b, num=1)[2]
        want.append([dataclasses.replace(peak_and_snr(s[b:b + 1], signal, acq_b, p, matlab_quirks=False), doppler_bin=b)
                     for s, p in zip(surf, CAND_PRNS)])
    variants = VARIANTS[n] if n != 58000 else [(0, 0, 0), (8, 256, 3)]
    for r, t, x in variants:
        what = f"N={n} M={coh_ms} R={r} T={t} X={x}"
        with api.Searcher(cfg_for(n, CAND_PRNS, coh_ms=coh_ms, **variant_kw(r, t, x))) as prod, \
                api.Searcher(cfg_for(n, CAND_PRNS, coh_ms=coh_ms, keep_surface=True, **variant_kw(r, t, x))) as dbg:
            for b in range(NBINS):
                f = FMIN + STEP * b
                for s in (prod, dbg):
                    set_windows(s, [(f, f)] * len(CAND_PRNS))
                rows = prod.search(raw_b)
                assert all(g.doppler_bin == b for g in rows), f"{what} bin {b}"
                assert_rows_and_noise(rows, want[b], f"{what} bin {b}")
                assert_same_scan(rows, dbg.search(raw_b), prod.last_stats.exchange, f"{what} bin {b}")


# ------------------------------------------------------------------ large and wrapping shifts, cell by cell
# name: (freq_min, freq_step, forward bases); 101 bins each
SHIFT_GRIDS = {"1k_up": (-50000.0, 1000.0, 1), "1k_down": (50000.0, -1000.0, 1), "250_up": (-12500.0, 250.0, 4)}
SHIFT_PRNS = [5, 12, 27, 31]                         # PRN 31 is absent


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SHIFT_GRIDS))
@pytest.mark.parametrize("n", [6000, 26000, 58000])
def test_large_and_wrapping_shifts_cell_by_cell(n, name):
    """101 bins whose shifts reach 100 FFT bins, |s| > Q for every Q, both signs (1 kHz steps: one forward base), and a
    250 Hz grid (four bases, shifts to 25).  Satellites at -47 / +47 kHz and on a bin of the 250 Hz grid reached through
    a shift of 19.  Every variant, every cell against the float64 surface, every row against the oracle."""
    fmin, step, bases = SHIFT_GRIDS[name]
    num = 101
    file, signal, acq = grid(n, fmin=fmin, step=step, num=num)
    sats = [SatSpec(5, 47000.0, 1, amp(n, 12.0), 0.3), SatSpec(12, -47000.0, n - 2, amp(n, 12.0), 1.1),
            SatSpec(27, -12500.0 + 250.0 * 77, n // 3, amp(n, 12.0), 2.0)]       # bin 77 = base 1 shifted by 19
    raw_b = block(n, sats, K)
    want = oracle_surfaces(raw_b, signal, acq, SHIFT_PRNS, 1)
    ref = [peak_and_snr(w, signal, acq, p) for w, p in zip(want, SHIFT_PRNS)]
    for r, t, x in VARIANTS[n]:
        what = f"N={n} {name} R={r} T={t} X={x}"
        with api.Searcher(cfg_for(n, SHIFT_PRNS, fmin=fmin, step=step, num=num, keep_surface=True,
                                  **variant_kw(r, t, x))) as s:
            rows = s.search(raw_b)
            assert s.last_stats.n_bases == bases, what
            for i, (prn, w) in enumerate(zip(SHIFT_PRNS, want)):
                got = s.read_surface(i)
                err = np.abs(got - w).max()
                assert err <= 1e-5 * w.max(), f"{what} PRN {prn}: {err / w.max():.3g} of the maximum"
                assert_same_argmax(got, w, f"{what} PRN {prn}")
        assert_rows_and_noise(rows, ref, what)


# ------------------------------------------------------------------ no state survives a search
def assert_zero_rows(rows, first_bins, what):
    """All-zero input: 0/0 SNR, nothing acquired, the first lag of the first bin each row searched."""
    for g, b in zip(rows, first_bins):
        assert (g.code_phase, g.peak, g.acquired, g.doppler_bin, g.noise_meansq) == (0, 0.0, 0, b, 0.0), f"{what} PRN {g.prn}"
        assert g.doppler_hz == FMIN + STEP * b and math.isnan(g.snr_db), f"{what} PRN {g.prn}"


@pytest.mark.gpu
@pytest.mark.parametrize("n", [6000, 26000, 58000])
def test_no_state_survives_a_search(n):
    """On one handle: strong block A, an all-zero block, A again -- without windows, with windows (every PRN's window
    holds a bin, their first bins differ), and through gnssacq_sweep with the windows over [A, 0, A, 0].  The zero
    rows are exactly the all-zero row and the second A is byte for byte the first.  Every variant, exchange 3 with
    whole rows and with the block-granular tail."""
    a = edge_blocks(n)[0][0]
    zero = bytes(len(a))
    P = len(EDGE_PRNS)
    windows = [(FMIN + STEP * (i % 5), FMIN + STEP * (i % 5 + 3)) for i in range(P - 1)] + [(-1e9, 1e9)]
    firsts = [i % 5 for i in range(P - 1)] + [0]
    for r, t, x in VARIANTS[n]:
        for ws in splits(x):
            what = f"N={n} R={r} T={t} X={x} split={ws}"
            with api.Searcher(cfg_for(n, EDGE_PRNS, **variant_kw(r, t, x, ws))) as s:
                first = row_bytes(s.search(a))
                assert_zero_rows(s.search(zero), [0] * P, what)
                assert row_bytes(s.search(a)) == first, what
                set_windows(s, windows)
                win = row_bytes(s.search(a))
                assert_zero_rows(s.search(zero), firsts, f"{what} windows")
                assert row_bytes(s.search(a)) == win, f"{what} windows"
                swept = s.sweep([a, zero, a, zero])
                assert row_bytes(swept[0]) == win and row_bytes(swept[2]) == win, f"{what} sweep"
                assert_zero_rows(swept[1], firsts, f"{what} sweep")
                assert_zero_rows(swept[3], firsts, f"{what} sweep")
