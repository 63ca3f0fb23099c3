#!/usr/bin/env python
"""bench.py -- search cells/s of the 32-PRN parallel code-phase acquisition (BASELINE.json metric).

A *step* is one complete coarse acquisition (acquisition.m:27-80 minus file I/O) of one synthetic IF
block of the chosen BASELINE config: K1a/K1b (re-order, wipe-off, forward FFT of every (base, block)), the
(PRN x Doppler bin x block) correlation search with on-chip non-coherent accumulation, row peaks and
the per-PRN decision.  cells = PRNs x Doppler bins x code phases (independent of K, SURVEY.md 8d).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config 1|2|3|4|5] [--impl reference] [--dump-outputs DIR]

Default workload: config 1, the Opensky-shaped block of BASELINE.json's north_star target.  The line carries
`value` (device-resident input, CUDA events), `e2e` (N = 1: through gnssacq_search with a pageable host buffer,
the call the MEX gateway makes; config 4: one gnssacq_sweep_file over `steps` epochs of a recording file),
`roofline`, `cpu_baseline`, `clocks` and `parity_checked` (the rows just timed, against the oracle on a PRN subset).
N > 1: launched by torchrun, one rank per GPU; ONE acquisition is sharded over the ranks (whole PRNs, or Doppler
bins when there are fewer PRNs than GPUs) and exchanged through peer memory inside every step -- the IF block is
pulled from rank 0 over NVLink by K1a, the candidates are stored into rank 0's table by K2, K4 runs on rank 0
(strong scaling of one acquisition; `--xchg nccl` = the r01 NCCL broadcast + all-gather instead).
`--impl reference` times the CPU restatement of acquisition.m (oracle/, NumPy float64, literal 3-FFT
loop) on all host cores, a FULL acquisition per step for configs 1 and 2: MATLAB/Octave do not exist in this
image, so the oracle port is the reference arm (cpu_baseline.kind = "port").
`--dump-outputs DIR` writes the result rows of the last timed step as DIR/<field>.npy (float64, one entry per PRN; the
reference arm: prn and peak): the inputs are seeded, so two builds run with the same arguments can be compared output
for output.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "assignment-for-aae6102_gnss-sdr_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree it runs from (which may be read-only)

METRIC = "search cells/s (PRN x Doppler x code-phase), 32-PRN acquisition"
UNIT = "cells/s"

# BASELINE.json configs restated as concrete shapes (SURVEY.md 8d table).
CONFIGS = {
    1: dict(name="config1_opensky_default", shape="opensky", fs=58e6, if_hz=4.58e6, n=58000,
            fmin=-10000.0, fstep=500.0, bins=41, k=20, m=1),
    2: dict(name="config2_urban_default", shape="urban", fs=26e6, if_hz=0.0, n=26000,
            fmin=-10000.0, fstep=500.0, bins=41, k=20, m=1),
    3: dict(name="config3_weak_signal_10msx20_50Hz", shape="opensky", fs=58e6, if_hz=4.58e6, n=58000,
            fmin=-10000.0, fstep=50.0, bins=401, k=20, m=10),
    # periodic re-acquisition over one long recording: every step searches the NEXT 20 ms window (one every
    # 100 ms, 8 distinct windows cycled); the e2e leg goes through gnssacq_sweep (copies overlap the searches)
    4: dict(name="config4_reacq_sweep_100ms", shape="opensky", fs=58e6, if_hz=4.58e6, n=58000,
            fmin=-10000.0, fstep=500.0, bins=41, k=20, m=1, sweep_windows=8, epoch_ms=100),
    5: dict(name="config5_high_dynamics_50kHz_10msx2", shape="opensky", fs=58e6, if_hz=4.58e6, n=58000,
            fmin=-50000.0, fstep=50.0, bins=2001, k=2, m=10),
}
PRNS = list(range(1, 33))


def w_unit(n: int) -> float:
    """Algorithmic FP32 flops of one (PRN, bin, block) unit (SURVEY.md 8d): one N-point transform by the
    5 N log2 N convention + 12 N (spectrum multiply 6N, |.|^2 3N, accumulate N, max / sum-of-squares 2N)."""
    return 5.0 * n * math.log2(n) + 12.0 * n


def w_fwd(n: int, m: int) -> float:
    return 5.0 * n * math.log2(n) + 8.0 * n * m


def synth_bytes(cfg) -> bytes:
    """Synthetic IF block of the config (product-side generator: the GPU arm never touches oracle/)."""
    from gnssacq.synth import opensky_recording, urban_recording
    rec = opensky_recording(seed=6102 + 1) if cfg["shape"] == "opensky" else urban_recording(seed=6102 + 2)
    return rec.read(0, cfg["k"] * cfg["m"])


def sparse_recording(cfg, raws, n_epochs, path):
    """A recording file for the config-4 sweep: `n_epochs` epochs of `epoch_ms`, the first K*M ms of each holding
    one of the synthetic windows (cycled); the rest of each epoch is a hole (never read by the sweep).  90 s at
    58 MHz int8 I/Q is 10.44 GB of file offsets but only n_epochs x 2.32 MB of data."""
    ms_bytes = cfg["n"] * 2
    with open(path, "wb") as f:
        for j in range(n_epochs):
            f.seek(j * cfg["epoch_ms"] * ms_bytes)
            f.write(raws[j % len(raws)])
        f.truncate(max(f.tell(), (n_epochs - 1) * cfg["epoch_ms"] * ms_bytes + len(raws[0])))
    return path


def synth_windows(cfg) -> list:
    """The first few windows of a re-acquisition sweep (config 4): window j starts at ms epoch_ms * j."""
    from gnssacq.synth import opensky_recording, urban_recording
    rec = opensky_recording(seed=6102 + 1) if cfg["shape"] == "opensky" else urban_recording(seed=6102 + 2)
    return [rec.read(cfg["epoch_ms"] * j, cfg["k"] * cfg["m"]) for j in range(cfg["sweep_windows"])]


# fields of gnssacq_result that the coarse search fills; fine_freq_hz stays NaN there (gnssacq_fine_frequency fills it)
DUMP_FIELDS = ("prn", "acquired", "code_phase", "doppler_bin", "doppler_hz", "peak", "noise_meansq", "snr_db")


def dump_outputs(directory, columns):
    """--dump-outputs: one float64 array per output field (rows in PRN order) as <directory>/<field>.npy."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, values in columns.items():
        np.save(os.path.join(directory, name + ".npy"), np.asarray(values, dtype=np.float64))


def dump_rows(directory, rows):
    dump_outputs(directory, {f: [getattr(r, f) for r in rows] for f in DUMP_FIELDS})


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi-equivalent sampling (NVML) of SM clock and throttle reasons DURING the timed region."""

    def __init__(self, index: int, period_s: float = 0.02):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        self.period = period_s
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def __enter__(self):
        if self.nv:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._thread:
            self._thread.join()

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


# ----------------------------------------------------------------------------- CPU reference
_W = {}


def _ref_worker(args):
    """Literal acquisition.m:53-61 loop body for one PRN over all bins and `kb` blocks."""
    prn, kb = args
    import numpy as np
    from oracle.acquisition_ref import correlation_surface
    acq = _W["acq_kb"]
    corr = correlation_surface(_W["raw"], _W["signal"], acq, prn, carrier=_W["carrier"], literal=True)
    return float(corr.max())


def _ref_setup(cfg, kb):
    import io
    import numpy as np
    import oracle
    from oracle.acquisition_ref import carrier_table, samples_from_bytes
    signal = oracle.SignalParams(IF=cfg["if_hz"], Fs=cfg["fs"])
    acq = oracle.AcqParams(freqStep=cfg["fstep"], freqMin=cfg["fmin"], freqNum=cfg["bins"], datalen=kb)
    # the CPU arm builds its input with the oracle's own generator (byte-identical to the product's, see
    # tests/test_cabi.py::test_product_and_oracle_generators_agree): nothing of libgnssacq on this path
    from oracle.synth import opensky_spec, urban_spec, synth_if
    spec = opensky_spec(seed=6102 + 1) if cfg["shape"] == "opensky" else urban_spec(seed=6102 + 2)
    raw = samples_from_bytes(synth_if(spec, 0, kb * cfg["m"]), 2, 1)
    _W.update(signal=signal, acq_kb=acq, raw=raw, carrier=carrier_table(signal, acq, 1))


def cpu_single_thread_baseline(cfg, budget_s=12.0):
    """cpu_baseline of the default run: the oracle port, ONE thread, bounded sample, linear extrapolation."""
    import numpy as np
    kb = cfg["k"] if cfg["m"] == 1 else 1
    _ref_setup(cfg, kb)
    t0 = time.perf_counter()
    done = 0
    for prn in PRNS:
        _ref_worker((prn, kb))
        done += 1
        if time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    cells = done * cfg["bins"] * cfg["n"] * (kb / cfg["k"])
    return {"value": cells / dt, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": f"{done} PRN x {cfg['bins']} bins x {kb} of {cfg['k']} blocks (coh {1} ms), literal 3-FFT loop "
                      f"of acquisition.m:53-61 in NumPy float64, {dt:.1f} s, scaled by blocks",
            "numpy": np.__version__}


def config_dict(cfg):
    """The `config` object both arms print (the driver compares them)."""
    cells = len(PRNS) * cfg["bins"] * cfg["n"]
    return {"workload": cfg["name"], "n": cfg["n"], "bins": cfg["bins"], "noncoh_blocks": cfg["k"],
            "coh_ms": cfg["m"], "prns": 32, "cells": cells, "cell_blocks": cells * cfg["k"],
            "l2": "GPU arm: L2 flushed between timed steps (256 MiB device memset outside the per-step event pair)"}


REFERENCE_BUDGET_S = 420.0


def run_reference(args, cfg):
    """The reference's own CPU implementation of the path (oracle port of acquisition.m:53-61, literal loop:
    three FFTs per (PRN, bin, block) unit, NumPy float64) on all host cores, one PRN per task.  Configs 1 and 2:
    every step is ONE FULL acquisition (32 PRNs x all bins x all K blocks), nothing scaled, as long as
    (steps + warmup) of them fit REFERENCE_BUDGET_S on this box; otherwise, and for configs 3-5 (hours of CPU
    work), a step is a bounded sample (all 32 PRNs x all bins x the first kb of K blocks, coherent length 1 ms)
    scaled by kb/K, and the line says so."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    cores = len(os.sched_getaffinity(0))
    n_steps, n_warm = args.steps, args.warmup
    # cost of one (PRN, all bins, one block) task on one core
    _ref_setup(cfg, 1)
    t0 = time.perf_counter()
    _ref_worker((1, 1))
    t_blk = time.perf_counter() - t0
    rounds = math.ceil(len(PRNS) / cores)
    full_ok = cfg["m"] == 1 and t_blk * cfg["k"] * rounds * (n_steps + n_warm) * 1.15 <= REFERENCE_BUDGET_S
    if full_ok:
        kb = cfg["k"]
    else:
        kb = max(1, min(cfg["k"], int(REFERENCE_BUDGET_S / (t_blk * rounds * (n_steps + n_warm) * 1.15))))
    _ref_setup(cfg, kb)
    pool = mp.get_context("fork").Pool(min(cores, len(PRNS)))
    tasks = [(p, kb) for p in PRNS]
    for _ in range(n_warm):
        pool.map(_ref_worker, tasks, chunksize=1)
    t0 = time.perf_counter()
    for _ in range(n_steps):
        peaks = pool.map(_ref_worker, tasks, chunksize=1)
    dt = time.perf_counter() - t0
    pool.close()
    if args.dump_outputs:
        # the per-PRN maximum of the surface over the first kb blocks (all of them when full_step is true)
        dump_outputs(args.dump_outputs, {"prn": PRNS, "peak": peaks})
    scale = kb / cfg["k"]
    cells_per_step = len(PRNS) * cfg["bins"] * cfg["n"] * scale
    value = cells_per_step * n_steps / dt
    if full_ok:
        sample = (f"per step: one full acquisition, 32 PRNs x {cfg['bins']} bins x {cfg['k']} blocks, literal "
                  f"acquisition.m:53-61 loop (3 FFTs per unit) in NumPy float64, one PRN per task on {cores} cores; nothing scaled")
    else:
        sample = (f"per step: 32 PRNs x {cfg['bins']} bins x {kb} of {cfg['k']} blocks at 1 ms coherent, literal "
                  f"acquisition.m:53-61 loop in NumPy float64 on {cores} cores; cells scaled by {kb}/{cfg['k']} "
                  f"(a full step would not fit the {REFERENCE_BUDGET_S:.0f} s budget of this arm)")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": n_steps, "warmup": n_warm, "ms_per_step": dt / n_steps * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_dict(cfg),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                         "full_step": bool(full_ok)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def parity_check(cfg, raw, rows, prns):
    """Checker for the timed result (VERDICT r01): the rows the bench just produced against the oracle on a PRN
    subset, same bytes, tolerances of tests/helpers.py (indices / decision exact unless the oracle's top two cells
    are within 2e-5, peak and SNR within 1e-4).  The oracle is only ever the checker here."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from helpers import assert_rows_match, oracle_rows_chunked, structs
    file, signal, acq = structs(cfg["fs"], cfg["if_hz"], datalen=cfg["k"], freq_min=cfg["fmin"],
                                freq_step=cfg["fstep"], freq_num=cfg["bins"])
    t0 = time.perf_counter()
    ref = oracle_rows_chunked(raw, file, signal, acq, prns, coh_ms=cfg["m"],
                              chunk_bins=max(1, min(20, cfg["bins"] // 12)) if cfg["m"] == 1 else (20 if cfg["bins"] < 1000 else 100))
    by = {r.prn: r for r in rows}
    out = {"prns": list(prns), "oracle": "oracle/acquisition_ref.py (NumPy float64 restatement of acquisition.m:41-80)",
           "oracle_s": None, "tolerance": "code phase / Doppler bin / decision exact unless oracle top-2 gap < 2e-5; peak, SNR 1e-4 rel"}
    try:
        ties = assert_rows_match([by[p] for p in prns], ref, what="bench parity")
        out.update(ok=True, ties=ties)
    except AssertionError as e:
        out.update(ok=False, error=str(e)[:300])
    out["oracle_s"] = round(time.perf_counter() - t0, 1)
    return out


# ----------------------------------------------------------------------------- GPU arm
def run_gpu(args, cfg):
    import torch
    import torch.distributed as dist
    import gnssacq
    from gnssacq import api
    from gnssacq.dist import CudaShard, PeerShard, ROW_BYTES

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torchrun --nproc-per-node {args.gpus}")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def factory(prns, device):
        return gnssacq.make_config(fs_hz=cfg["fs"], if_hz=cfg["if_hz"], samples_per_ms=cfg["n"],
                                   freq_min_hz=cfg["fmin"], freq_step_hz=cfg["fstep"], freq_num=cfg["bins"],
                                   noncoh_blocks=cfg["k"], coh_ms=cfg["m"], prns=prns, device=device,
                                   cluster_ctas=args.cluster_ctas, threads=args.threads, exchange=args.exchange)

    sweep = "sweep_windows" in cfg
    raws = synth_windows(cfg) if sweep else [synth_bytes(cfg)]
    raw = raws[0]
    h_ifs = [torch.frombuffer(bytearray(r), dtype=torch.uint8).pin_memory() for r in raws]
    d_ifs = [h.cuda() for h in h_ifs] if sweep else []
    h_if = h_ifs[0]
    peer = args.xchg == "peer"
    if peer:
        # exchange through peer memory (gnssacq_xchg_*): no NCCL inside a step.  Same call shape as CudaShard below.
        # plan "rows" (default when there is more than one GPU): contiguous row ranges, the root's share weighted so
        # that all shards FINISH together (the others start later by the IF pull) -- calibrated once after the warm-up
        plan = args.plan if args.plan != "auto" else ("rows" if world > 1 else "prn")
        ps = PeerShard(factory(PRNS, local), rank, world, local, dist if world > 1 else None, plan=plan,
                       root_extra_permille=args.root_extra if args.root_extra is not None else 0)

        class _Shard:
            searcher, n_local, max_rows = ps.searcher, ps.shard.prn_count, (len(PRNS) + world - 1) // world
            rows_local = ps.rows_local

            @staticmethod
            def enqueue(_d, h_if=None):
                ps.enqueue(h_if.numpy() if (h_if is not None and rank == 0) else None)

            fetch = staticmethod(ps.fetch)
            close = staticmethod(ps.close)

            @staticmethod
            def load(t):
                ps.upload(t)
        shard = _Shard
        shard.load(h_if)
    else:
        plan = "prn"
        shard = CudaShard(factory, PRNS, rank, world, local)
        shard.rows_local = shard.n_local * cfg["bins"]
        shard.bind_stream()
        shard.d_if.copy_(h_if)
        shard.load = lambda t: shard.d_if.copy_(t)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")     # > 126 MB L2
    d = dist if world > 1 else None

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        shard.enqueue(d)
    rows = shard.fetch()
    root_extra = None
    if peer and plan == "rows" and world > 1:
        if args.root_extra is None:
            ps.rebalance()                                  # set-up: weighs the root's share from the measured waits
            shard.searcher, shard.rows_local = ps.searcher, ps.rows_local
            for _ in range(3):
                shard.enqueue(d)
            rows = shard.fetch()
        root_extra = ps.root_extra_permille

    # ---- timed region 1: device-resident input, per-step CUDA events, L2 flushed between steps ----
    ev0 = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    ev1 = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    barrier()
    with ClockSampler(local) as clk:
        t_wall0 = time.perf_counter()
        sync_t = torch.zeros(1, device="cuda")
        for i in range(args.steps):
            flush.zero_()
            if world > 1:
                # align the ranks AFTER the flush and BEFORE the timed pair: otherwise another rank's flush
                # leaks into this rank's step through the broadcast inside it
                dist.all_reduce(sync_t)
            if sweep:
                shard.load(d_ifs[i % len(d_ifs)])           # this step's window: resident in HBM, outside the timed pair
            ev0[i].record()
            shard.enqueue(d)
            ev1[i].record()
        barrier()
        t_wall = time.perf_counter() - t_wall0
    if args.dump_outputs:
        timed_rows = shard.fetch()                          # the rows of the last timed step (rank 0 holds them)
        if rank == 0:
            dump_rows(args.dump_outputs, timed_rows)
    step_ms = [a.elapsed_time(b) for a, b in zip(ev0, ev1)]
    total_ms = torch.tensor([sum(step_ms)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_ms = float(total_ms.item())

    # ---- roofline pass: dominant kernel (search_kernel) duration from the library's own events ----
    k2_ms, k1_ms, launches, pull_ms, wait_ms = [], [], 0, [], []
    for i in range(min(args.steps, 20)):
        flush.zero_()
        if world > 1:
            dist.all_reduce(sync_t)
        shard.enqueue(d)
        if shard.searcher:
            if peer:
                shard.fetch()
                st = shard.searcher.last_stats
            else:
                st = shard.searcher.fetch_stats()
            k2_ms.append(st.search_ms)
            k1_ms.append(st.wipeoff_fft_ms)
            pull_ms.append(st.if_pull_ms)
            wait_ms.append(st.gather_wait_ms)
            launches = st.kernel_launches
    torch.cuda.synchronize()
    variant = (st.cluster_ctas, st.threads) if shard.searcher else (0, 0)

    # ---- timed region 2: end to end through the public API, host buffers, H2D + D2H inside ----
    barrier()
    t0 = time.perf_counter()
    e2e_api = "CudaShard.enqueue(h_if) + fetch: pinned H2D on rank 0, IF exchange, shard search, row exchange, D2H"
    if sweep and world == 1:
        # the public call for this workload: ONE gnssacq_sweep_file over `steps` epochs of a recording on disk --
        # the library does acquisition.m:27-34's fseek/fread itself, straight into pinned staging, overlapped
        import tempfile
        tmpdir = tempfile.mkdtemp(prefix="gnssacq_rec_")
        rec = sparse_recording(cfg, raws, args.steps, os.path.join(tmpdir, "Opensky_synth_90s.bin"))
        barrier()
        t0 = time.perf_counter()
        swept = shard.searcher.sweep_file(rec, 0, cfg["epoch_ms"], args.steps)
        rows = swept[-1]
        os.remove(rec)
        os.rmdir(tmpdir)
        e2e_api = (f"gnssacq_sweep_file (Searcher.sweep_file): {args.steps} epochs, one every {cfg['epoch_ms']} ms, read by the library "
                   "from a recording file (fseek + fread into pinned staging) -> H2D -> K1/K2/K4 -> one D2H of all rows")
    elif world == 1:
        # the call the MEX gateway makes (matlab/gnssacq_mex.c -> gnssacq_search): caller-owned pageable host
        # buffer in, result rows out; staging copy, H2D, kernels, D2H and the host sync are all inside
        import numpy as np
        host = [np.frombuffer(r, dtype=np.uint8).copy() for r in raws]
        for i in range(args.steps):
            rows = shard.searcher.search(host[i % len(host)])
        e2e_api = "gnssacq_search (Searcher.search): pageable host buffer -> library pinned staging -> H2D -> K1/K2/K4 -> D2H"
    else:
        for i in range(args.steps):
            shard.enqueue(d, h_if=h_ifs[i % len(h_ifs)])
            rows = shard.fetch()
    barrier()
    e2e_s = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_s = float(e2e_s.item())

    cells = len(PRNS) * cfg["bins"] * cfg["n"]
    # per-phase times of the exchange (SURVEY 5 metrics row): slowest non-root IF pull, the root's wait for candidates
    phase = torch.tensor([max(pull_ms) if pull_ms and rank else 0.0, sum(k2_ms) / max(len(k2_ms), 1)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(phase, op=dist.ReduceOp.MAX)
    if rank == 0:
        n_local = shard.n_local
        nb = st.n_bases
        w_search = shard.rows_local * cfg["k"] * w_unit(cfg["n"])               # flops of ONE search_kernel launch (rank 0's rows)
        k2 = sum(k2_ms) / len(k2_ms)
        try:
            fp32_peak = api.fp32_peak_tflops(local)
            peak_src = "measured: FFMA microbenchmark in this run (gnssacq_fp32_peak_tflops), 2 flop/FFMA"
        except Exception:
            fp32_peak, peak_src = 74.4, "fallback nominal 148 SM x 128 lane x 2 x 1.965 GHz"
        achieved = w_search / (k2 * 1e-3) * 1e-12
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        traffic = None
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json"))).get(cfg["name"])
        except Exception:
            pass
        line = {
            "metric": METRIC, "value": cells * args.steps / (total_ms * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": total_ms / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": config_dict(cfg),
            "run": {   "forward_bases": nb, "engine": {"cluster_ctas": variant[0], "threads": variant[1], "exchange": {1: "dsmem", 2: "l2+clusters", 3: "l2+coop-groups"}.get(st.exchange),
                                  "resident_clusters": st.resident_clusters,
                                  "work_split": {1: "whole rows", 2: "block-granular tail"}.get(st.work_split)},
                       "sharding": (f"PRN-major, {n_local} PRNs on rank 0" if plan == "prn" else
                                    f"row ranges (gnssacq_shard_plan_rows), {shard.rows_local} of {len(PRNS) * cfg['bins']} rows on rank 0, "
                                    f"root weight 1 + {root_extra}/1000 " + ("calibrated by PeerShard.rebalance() after the warm-up" if args.root_extra is None else "as given")),
                       "exchange_between_gpus": ("peer memory (CUDA IPC over NVLink): K1a pulls the IF block from rank 0, K2 stores its "
                                                 "candidates into rank 0's table, K4 on rank 0; no NCCL call inside a step" if peer else
                                                 "NCCL broadcast of the IF block + all_gather of the result rows") if world > 1 else "none (one GPU)",
                       "exchange_phases_ms": {"if_pull_max_over_ranks": float(phase[0].item()), "gather_wait_rank0": (sum(wait_ms) / len(wait_ms)) if wait_ms else 0.0,
                                              "search_kernel_max_over_ranks": float(phase[1].item())},
                       "latency_ms_32prn": e2e_s / args.steps * 1e3,
                       **({"sweep": f"{len(raws)} distinct windows, one every {cfg['epoch_ms']} ms, cycled; e2e = one gnssacq_sweep call over {args.steps} host windows"
                           if world == 1 else f"{len(raws)} distinct windows cycled, one host window per step"} if sweep else {})},
            "roofline": {"bound": "fp32", "kernel": "search_kernel", "achieved": achieved, "peak": fp32_peak,
                         "unit": "TFLOP/s", "frac": achieved / fp32_peak, "traffic": traffic,
                         "traffic_source": "dram__bytes_read+write of one search-kernel launch from the committed ncu --set full capture (profiles/r02/ncu_v16_search_c*.summary.txt via profiles/ncu_traffic.json); a bench run cannot sit under ncu, so this figure is not re-measured here",
                         "peak_source": peak_src, "nominal_peak": 74.4,
                         "algorithmic_flops_per_launch": w_search, "kernel_ms": k2,
                         "wipeoff_fft_kernel_ms": sum(k1_ms) / len(k1_ms),
                         "hbm_compulsory_bytes_per_step": len(raw) + 32 * cfg["n"] * 8 + 32 * ROW_BYTES,
                         "hbm_peak_gbs": peaks.get("hbm_gbs")},
            # secondary view: the same launch against the HBM roofline (compulsory bytes: IF block + cached code
            # spectra + result rows).  The path is FP32-bound, so this fraction is tiny by design (DESIGN.md section 4).
            "roofline_hbm": {"bound": "hbm", "kernel": "search_kernel",
                             "achieved": (len(raw) + 32 * cfg["n"] * 8 + 32 * ROW_BYTES) / (k2 * 1e-3) * 1e-9,
                             "peak": peaks.get("hbm_gbs", 6650.0), "unit": "GB/s",
                             "frac": (len(raw) + 32 * cfg["n"] * 8 + 32 * ROW_BYTES) / (k2 * 1e-3) * 1e-9 / peaks.get("hbm_gbs", 6650.0),
                             "traffic": traffic,
                             "peak_source": "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6.65 TB/s"},
            "e2e": {"value": cells * args.steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": len(raw),
                    "d2h_bytes_per_step": world * shard.max_rows * ROW_BYTES, "api": e2e_api},
            "gpu_launches": launches * args.steps,
            "clocks": clk.summary(),
            "wall_s_timed_region": t_wall,
            "acquired": [r.prn for r in rows if r.acquired],
        }
        if not args.no_parity:
            subset = [3, 8, 22, 30] if cfg["m"] == 1 else [3, 22]
            line["parity_checked"] = parity_check(cfg, raws[(args.steps - 1) % len(raws)], rows, subset)
        if world == 1 and not args.no_cpu:
            line["cpu_baseline"] = cpu_single_thread_baseline(cfg)
        print(json.dumps(line))
    shard.close()
    if world > 1:
        dist.destroy_process_group()


def run_gpu_epoch_sharded(args, cfg):
    """BASELINE config 4, the other way to use N GPUs (SURVEY 8e): the EPOCHS of the sweep are dealt out, rank r takes
    epochs r, r + N, ...; every rank searches all 32 PRNs of its epochs on its own GPU and nothing is exchanged
    (no collective on the data path).  A step is still one epoch; `steps` epochs in total."""
    import torch
    import torch.distributed as dist
    import gnssacq
    from gnssacq import api
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    raws = synth_windows(cfg)
    mine = list(range(rank, args.steps, world))                       # this rank's epochs
    s = api.Searcher(gnssacq.make_config(fs_hz=cfg["fs"], if_hz=cfg["if_hz"], samples_per_ms=cfg["n"], freq_min_hz=cfg["fmin"],
                                         freq_step_hz=cfg["fstep"], freq_num=cfg["bins"], noncoh_blocks=cfg["k"], coh_ms=cfg["m"],
                                         prns=PRNS, device=local))
    s.set_stream(torch.cuda.current_stream().cuda_stream)
    d_ifs = [torch.frombuffer(bytearray(r), dtype=torch.uint8).cuda() for r in raws]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()
    for i in range(max(args.warmup, 3)):
        s.enqueue_device(d_ifs[i % len(d_ifs)].data_ptr(), s.if_bytes)
    s.fetch()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in mine]
    barrier()
    with ClockSampler(local) as clk:
        for (a, b), j in zip(ev, mine):
            flush.zero_()
            a.record()
            s.enqueue_device(d_ifs[j % len(d_ifs)].data_ptr(), s.if_bytes)
            b.record()
        barrier()
    if args.dump_outputs and mine and mine[-1] == args.steps - 1:    # the rank that searched the last epoch
        dump_rows(args.dump_outputs, s.fetch())
    total_ms = torch.tensor([sum(a.elapsed_time(b) for a, b in ev)], dtype=torch.float64, device="cuda")
    # end to end: this rank's epochs straight from the recording file, one gnssacq_sweep_file call
    import tempfile
    tmpdir = tempfile.mkdtemp(prefix="gnssacq_rec_")
    rec = sparse_recording(cfg, raws, args.steps, os.path.join(tmpdir, f"rec_rank{rank}.bin"))
    barrier()
    t0 = time.perf_counter()
    swept = s.sweep_file(rec, rank * cfg["epoch_ms"], world * cfg["epoch_ms"], len(mine)) if mine else []
    barrier()
    e2e_s = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
    os.remove(rec)
    os.rmdir(tmpdir)
    st = s.last_stats
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    cells = len(PRNS) * cfg["bins"] * cfg["n"]
    if rank == 0:
        rows = swept[-1]
        line = {"metric": METRIC, "value": cells * args.steps / (float(total_ms.item()) * 1e-3), "unit": UNIT, "n_gpus": world,
                "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": float(total_ms.item()) / args.steps,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config_dict(cfg),
                "run": {"sharding": f"epoch-sharded: rank r searches epochs r, r+{world}, ... with all 32 PRNs; no exchange between GPUs",
                        "latency_ms_32prn": st.total_ms / max(len(mine), 1)},
                "e2e": {"value": cells * args.steps / float(e2e_s.item()), "unit": UNIT, "h2d_bytes_per_step": len(raws[0]),
                        "d2h_bytes_per_step": 32 * 56,
                        "api": "gnssacq_sweep_file per rank over its epochs of the recording (fseek/fread by the library)"},
                "gpu_launches": 4 * args.steps, "clocks": clk.summary(),
                "acquired": [r.prn for r in rows if r.acquired]}
        if not args.no_parity:
            line["parity_checked"] = parity_check(cfg, raws[mine[-1] % len(raws)], rows, [3, 8, 22, 30])
        print(json.dumps(line))
    s.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--config", type=int, default=1, choices=sorted(CONFIGS),
                    help="BASELINE.json config; default 1 = Opensky-shaped block, the north_star target")
    ap.add_argument("--impl", default="gpu", choices=["gpu", "reference"])
    ap.add_argument("--cluster-ctas", type=int, default=0)
    ap.add_argument("--threads", type=int, default=0)
    ap.add_argument("--exchange", type=int, default=0, help="0 auto, 1 DSMEM, 2 L2-resident exchange buffer")
    ap.add_argument("--xchg", default="peer", choices=["peer", "nccl"],
                    help="multi-GPU exchange: peer memory (gnssacq_xchg_*, default) or the r01 NCCL broadcast + all-gather")
    ap.add_argument("--plan", default="auto", choices=["auto", "prn", "rows"],
                    help="multi-GPU shards (peer exchange): whole PRNs / bin ranges (gnssacq_shard_plan) or weighted row ranges "
                         "(gnssacq_shard_plan_rows); auto = rows when there is more than one GPU")
    ap.add_argument("--root-extra", type=int, default=None,
                    help="plan rows: the root's extra share in 1/1000 of an equal share (default: calibrate after the warm-up)")
    ap.add_argument("--sweep-shard", default="grid", choices=["grid", "epochs"],
                    help="config 4 on N GPUs: shard every acquisition's PRN x Doppler grid (default, BASELINE's wording) or deal out the epochs")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle check of the timed result")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result rows of the last timed step as DIR/<field>.npy (float64, one entry per PRN)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    cfg = CONFIGS[args.config]
    if args.impl == "reference":
        run_reference(args, cfg)
    elif args.sweep_shard == "epochs" and "sweep_windows" in cfg:
        run_gpu_epoch_sharded(args, cfg)
    else:
        run_gpu(args, cfg)


if __name__ == "__main__":
    main()
