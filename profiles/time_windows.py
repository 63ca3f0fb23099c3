"""Assisted re-acquisition: the full Doppler grid against per-PRN windows (gnssacq_set_doppler_windows).

BASELINE config-1 (Opensky, N = 58 000) and config-2 (Urban, N = 26 000) shapes, 32 PRNs, 41 bins of 500 Hz, K = 20,
on the seeded recordings of gnssacq/synth.py.  Each shape is searched over the full grid, then with a +-1 kHz window
(5 bins) around each PRN's bin nearest its true Doppler (0 Hz for PRNs not in the recording).  For each: the rows
searched, K1 (wipeoff_fft_ms) and K2 (search_ms) device times, and the time of one gnssacq_search (CUDA events from the
upload to the copy of the rows, and the host clock around the call), medians over the repeats after a warm-up.  The
same run checks that every PRN whose full-grid winner lies inside its window gets the full-grid row byte for byte.

    python profiles/time_windows.py [--reps 50] [--warmup 5] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "assignment-for-aae6102_gnss-sdr_b200"))

import numpy as np

import gnssacq
from gnssacq import api
from gnssacq.synth import opensky_recording, urban_recording

SHAPES = {
    "config1_opensky": dict(rec=lambda: opensky_recording(seed=6103), fs=58e6, if_hz=4.58e6, n=58000),
    "config2_urban": dict(rec=lambda: urban_recording(seed=6104), fs=26e6, if_hz=0.0, n=26000),
}
FMIN, STEP, BINS, K = -10000.0, 500.0, 41, 20
PRNS = list(range(1, 33))
HALF_WIDTH = 1000.0


def device_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        power = q.stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        power = "unavailable"
    return name, power


def timed(s, raw, reps, warmup):
    for _ in range(warmup):
        s.search(raw)
    search, k1, total, wall = [], [], [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        rows = s.search(raw)
        wall.append((time.perf_counter() - t0) * 1e3)
        st = s.last_stats
        search.append(st.search_ms)
        k1.append(st.wipeoff_fft_ms)
        total.append(st.total_ms)
    med = lambda v: float(np.median(v))
    return rows, dict(search_ms=med(search), wipeoff_fft_ms=med(k1), search_call_events_ms=med(total),
                      search_call_wall_ms=med(wall), search_ms_min=float(min(search)), work_split=st.work_split,
                      resident_groups=st.resident_clusters)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if a.reps < 20:
        ap.error("--reps must be at least 20")
    name, power = device_info()
    report = dict(device=name, power_limit_and_max_sm_clock=power, reps=a.reps, warmup=a.warmup, shapes={})
    for label, sh in SHAPES.items():
        rec = sh["rec"]()
        raw = rec.read(0, K)
        truth = {s.prn: s.doppler_hz for s in rec.sats}
        centre = [FMIN + STEP * min(BINS - 1, max(0, round((truth.get(p, 0.0) - FMIN) / STEP))) for p in PRNS]
        lo = [c - HALF_WIDTH for c in centre]
        hi = [c + HALF_WIDTH for c in centre]
        cfg = gnssacq.make_config(fs_hz=sh["fs"], if_hz=sh["if_hz"], samples_per_ms=sh["n"], freq_min_hz=FMIN,
                                  freq_step_hz=STEP, freq_num=BINS, noncoh_blocks=K, prns=PRNS, device=0)
        with api.Searcher(cfg) as s:
            full_rows, full = timed(s, raw, a.reps, a.warmup)
            s.set_doppler_windows(lo, hi)
            win_rows, win = timed(s, raw, a.reps, a.warmup)
        bins = [[b for b in range(BINS) if l <= FMIN + STEP * b <= h] for l, h in zip(lo, hi)]
        full["rows"] = len(PRNS) * BINS
        win["rows"] = sum(len(b) for b in bins)
        inside = [i for i, r in enumerate(full_rows) if r.doppler_bin in bins[i]]
        same = [i for i in inside if bytes(win_rows[i]) == bytes(full_rows[i])]
        for d in (full, win):
            d["k1_share_of_events"] = d["wipeoff_fft_ms"] / d["search_call_events_ms"]
        report["shapes"][label] = dict(
            full=full, windowed=win, search_ms_ratio=win["search_ms"] / full["search_ms"],
            call_ratio=win["search_call_events_ms"] / full["search_call_events_ms"],
            prns_with_winner_in_window=len(inside), identical_rows=len(same),
            acquired_full=[r.prn for r in full_rows if r.acquired],
            acquired_windowed=[r.prn for r in win_rows if r.acquired])
        if len(same) != len(inside):
            raise SystemExit(f"{label}: {len(inside) - len(same)} windowed rows differ from the full grid's")
    text = json.dumps(report, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
