"""Acquisition at front-end rates that are zero-padded into a built transform length (gnssacq_transform_size).

32 PRNs x 41 bins of 500 Hz x 20 ms through gnssacq_search at 16.368 MHz (N = 16 368 in NF = 58 000), 4.092 MHz
(N = 4 092 in NF = 26 000) and 2.048 MHz (N = 2 048 in NF = 6 000), int8 I/Q with six seeded satellites.  Per rate:
search_ms (K2 + K3) and wipeoff_fft_ms (K1) device times, the forward bases K1 makes (n_bases), the host clock around
one gnssacq_search, cells/s counted on the N useful lags (32 * 41 * N / search time), and the fine-frequency stage's
wall time for 8 SVs (L = 10).  Medians over the repeats after a warm-up.  The card's name and power limit are read in
the same run.

    python profiles/time_rates.py [--reps 30] [--warmup 5] [--out FILE]
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
sys.path.insert(0, ROOT)

import numpy as np

import gnssacq
from gnssacq import api
from oracle.synth import SatSpec, SynthSpec, synth_if

RATES = [("16.368MHz", 16.368e6, 4.092e6), ("4.092MHz", 4.092e6, 1.023e6), ("2.048MHz", 2.048e6, 0.0)]
FMIN, STEP, BINS, K, L = -10000.0, 500.0, 41, 20, 10
PRNS = list(range(1, 33))


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


def recording(fs, if_hz, n, n_ms):
    sats = [SatSpec(p, d, cd % n, a, 0.3 * p) for p, d, cd, a in
            [(2, 3210.0, 5000, 2.2), (7, -4470.0, 123, 1.8), (11, 760.0, n - 3, 1.6), (19, -8990.0, 9001, 2.0),
             (26, 6120.0, 16, 1.3), (31, -250.0, 14000, 1.9)]]
    spec = SynthSpec(fs=fs, if_hz=if_hz, samples_per_ms=n, sigma=16.0, data_type=2, data_precision=1, seed=6102,
                     sats=sats)
    return synth_if(spec, 0, n_ms)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    name, power = device_info()
    out = {"device": name, "power_limit_max_sm_clock": power, "prns": len(PRNS), "bins": BINS, "noncoh_ms": K,
           "reps": args.reps, "rates": {}}
    for label, fs, if_hz in RATES:
        cfg = gnssacq.make_config(fs_hz=fs, if_hz=if_hz, freq_min_hz=FMIN, freq_step_hz=STEP, freq_num=BINS,
                                  noncoh_blocks=K, prns=PRNS)
        n, nf = cfg.samples_per_ms, api.transform_size(cfg)
        blob = recording(fs, if_hz, n, K + L + 1)
        raw = blob[:K * n * 2]
        with api.Searcher(cfg) as s:
            for _ in range(args.warmup):
                s.search(raw)
            search, k1, wall = [], [], []
            for _ in range(args.reps):
                t0 = time.perf_counter()
                rows = s.search(raw)
                wall.append((time.perf_counter() - t0) * 1e3)
                search.append(s.last_stats.search_ms)
                k1.append(s.last_stats.wipeoff_fft_ms)
            st = s.last_stats
            acquired = sorted(r.prn for r in rows if r.acquired)
            svs = [r for r in sorted(rows, key=lambda r: -r.snr_db)][:8]
            long_raw = blob[:(L + 1) * n * 2]
            s.fine_frequency(long_raw, L, [r.prn for r in svs], [r.code_phase for r in svs])     # warm-up (scratch)
            fine = []
            for _ in range(max(3, args.reps // 5)):
                t0 = time.perf_counter()
                s.fine_frequency(long_raw, L, [r.prn for r in svs], [r.code_phase for r in svs])
                fine.append((time.perf_counter() - t0) * 1e3)
        med = float(np.median(search))
        out["rates"][label] = {
            "fs_hz": fs, "samples_per_ms": n, "transform_length": nf, "n_bases": st.n_bases,
            "exchange": st.exchange, "cluster_ctas": st.cluster_ctas, "threads": st.threads,
            "search_ms": med, "search_ms_min": float(np.min(search)), "search_ms_max": float(np.max(search)),
            "wipeoff_fft_ms": float(np.median(k1)), "gnssacq_search_wall_ms": float(np.median(wall)),
            "cells_per_s_useful_lags": len(PRNS) * BINS * n / (med * 1e-3),
            "fine_8sv_wall_ms": float(np.median(fine)), "acquired": acquired,
        }
        print(label, json.dumps(out["rates"][label]), flush=True)
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
