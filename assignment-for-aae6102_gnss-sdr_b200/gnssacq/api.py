"""ctypes binding of ``libgnssacq.so`` (``include/gnssacq.h``).

This is the binding that is testable in the build image (no MATLAB/Octave
here); ``matlab/gnssacq_mex.c`` binds the same entry points for MATLAB.
There is no CPU fallback: if the shared library is missing, importing this
module raises, and without a B200 ``gnssacq_create`` fails with
``GNSSACQ_ERR_NO_DEVICE``.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import List, Optional, Sequence

import numpy as np

GNSSACQ_MAX_PRN = 64
_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgnssacq.so")


class GnssAcqError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"gnssacq error {code}: {msg}")
        self.code = code


STATUS = {
    0: "GNSSACQ_OK", -1: "GNSSACQ_ERR_INVALID_ARG", -2: "GNSSACQ_ERR_UNSUPPORTED_N",
    -3: "GNSSACQ_ERR_SHORT_BUFFER", -4: "GNSSACQ_ERR_CUDA", -5: "GNSSACQ_ERR_NO_DEVICE",
    -6: "GNSSACQ_ERR_NOMEM", -7: "GNSSACQ_ERR_STATE",
}


class Config(C.Structure):
    _fields_ = [
        ("fs_hz", C.c_double), ("if_hz", C.c_double), ("code_hz", C.c_double),
        ("samples_per_ms", C.c_int32), ("data_type", C.c_int32), ("data_precision", C.c_int32),
        ("freq_min_hz", C.c_double), ("freq_step_hz", C.c_double), ("freq_num", C.c_int32),
        ("noncoh_blocks", C.c_int32), ("coh_ms", C.c_int32),
        ("n_prn", C.c_int32), ("prn", C.c_int32 * GNSSACQ_MAX_PRN),
        ("snr_threshold_db", C.c_double),
        ("device", C.c_int32), ("cluster_ctas", C.c_int32), ("threads", C.c_int32),
        ("keep_surface", C.c_int32), ("exchange", C.c_int32), ("work_split", C.c_int32),
        ("bin_first", C.c_int32), ("bin_count", C.c_int32),
        ("row_first", C.c_int32), ("row_count", C.c_int32),
    ]


class Result(C.Structure):
    _fields_ = [
        ("prn", C.c_int32), ("acquired", C.c_int32), ("code_phase", C.c_int32), ("doppler_bin", C.c_int32),
        ("doppler_hz", C.c_double), ("peak", C.c_double), ("noise_meansq", C.c_double),
        ("snr_db", C.c_double), ("fine_freq_hz", C.c_double),
    ]

    def as_dict(self) -> dict:
        return {n: getattr(self, n) for n, _ in self._fields_}


class Channel(C.Structure):
    """gnssacq_channel: the state of one tracking channel for one integration (trackingCT.m:42-58,78,96,104)."""
    _fields_ = [
        ("prn", C.c_int32), ("num_samples", C.c_int32), ("sample_offset", C.c_int64),
        ("carrier_hz", C.c_double), ("rem_phase", C.c_double), ("code_hz", C.c_double), ("rem_chip", C.c_double),
    ]


class LoopParams(C.Structure):
    """gnssacq_loop_params: track.DLL*/PLL*/CorrelatorSpacing (initParameters.m:59-65)."""
    _fields_ = [("dll_bw", C.c_double), ("dll_damp", C.c_double), ("dll_gain", C.c_double),
                ("pll_bw", C.c_double), ("pll_damp", C.c_double), ("pll_gain", C.c_double),
                ("spacing_chips", C.c_double)]


class TrackRecord(C.Structure):
    """gnssacq_track_record: the TckResultCT fields of one integration period (trackingCT.m:153-172)."""
    _fields_ = [("P_i", C.c_double), ("P_q", C.c_double), ("E_i", C.c_double), ("E_q", C.c_double),
                ("L_i", C.c_double), ("L_q", C.c_double), ("pll_discri", C.c_double), ("dll_discri", C.c_double),
                ("rem_chip", C.c_double), ("code_hz", C.c_double), ("carrier_hz", C.c_double), ("rem_phase", C.c_double),
                ("sample_end", C.c_int64), ("num_samples", C.c_int32), ("reserved", C.c_int32)]


class Stats(C.Structure):
    _fields_ = [
        ("h2d_ms", C.c_float), ("wipeoff_fft_ms", C.c_float), ("search_ms", C.c_float),
        ("finalize_ms", C.c_float), ("d2h_ms", C.c_float), ("total_ms", C.c_float),
        ("kernel_launches", C.c_int32), ("n_bases", C.c_int32), ("cluster_ctas", C.c_int32),
        ("threads", C.c_int32), ("exchange", C.c_int32), ("resident_clusters", C.c_int32),
        ("work_split", C.c_int32), ("if_pull_ms", C.c_float), ("gather_wait_ms", C.c_float),
    ]

    def as_dict(self) -> dict:
        return {n: getattr(self, n) for n, _ in self._fields_}


class Shard(C.Structure):
    """gnssacq_shard: one handle's place in a multi-GPU acquisition (gnssacq_shard_plan)."""
    _fields_ = [
        ("rank", C.c_int32), ("world", C.c_int32), ("n_prn_total", C.c_int32),
        ("prn_total", C.c_int32 * GNSSACQ_MAX_PRN), ("freq_num_total", C.c_int32),
        ("prn_first", C.c_int32), ("prn_count", C.c_int32), ("bin_first", C.c_int32), ("bin_count", C.c_int32),
        ("row_first", C.c_int32), ("row_count", C.c_int32), ("plan_rows", C.c_int32), ("root_extra_permille", C.c_int32),
    ]

    @property
    def n_rows(self) -> int:
        """(PRN, bin) rows this shard searches."""
        return self.row_count if self.plan_rows else self.prn_count * self.bin_count


EXPORTS = (
    "gnssacq_version", "gnssacq_config_default", "gnssacq_if_bytes", "gnssacq_create",
    "gnssacq_destroy", "gnssacq_last_error", "gnssacq_set_stream", "gnssacq_search",
    "gnssacq_search_device", "gnssacq_enqueue_device", "gnssacq_enqueue_device_out", "gnssacq_fetch_results",
    "gnssacq_ca_code", "gnssacq_code_replica", "gnssacq_read_surface", "gnssacq_fft_forward", "gnssacq_fp32_peak_tflops", "gnssacq_fine_frequency",
    "gnssacq_search_multi", "gnssacq_sweep", "gnssacq_sweep_file", "gnssacq_track_load", "gnssacq_correlate",
    "gnssacq_loop_params_default", "gnssacq_track", "gnssacq_track_bank",
    "gnssacq_shard_plan", "gnssacq_shard_plan_rows", "gnssacq_xchg_root", "gnssacq_xchg_attach", "gnssacq_xchg_attach_local",
    "gnssacq_xchg_if_buffer", "gnssacq_xchg_enqueue", "gnssacq_xchg_finish", "gnssacq_xchg_fetch",
    "gnssacq_set_doppler_windows", "gnssacq_transform_size",
)


def _load() -> C.CDLL:
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python __graft_entry__.py build` "
            "(nvcc, sm_100a).  gnssacq has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    lib.gnssacq_version.restype = C.c_char_p
    lib.gnssacq_config_default.argtypes = [C.POINTER(Config)]
    lib.gnssacq_if_bytes.argtypes = [C.POINTER(Config)]
    lib.gnssacq_if_bytes.restype = C.c_size_t
    lib.gnssacq_create.argtypes = [C.POINTER(Config), C.POINTER(vp)]
    lib.gnssacq_destroy.argtypes = [vp]
    lib.gnssacq_last_error.argtypes = [vp]
    lib.gnssacq_last_error.restype = C.c_char_p
    lib.gnssacq_set_stream.argtypes = [vp, vp]
    lib.gnssacq_search.argtypes = [vp, vp, C.c_size_t, C.POINTER(Result), C.POINTER(Stats)]
    lib.gnssacq_search_device.argtypes = [vp, vp, C.c_size_t, C.POINTER(Result), C.POINTER(Stats)]
    lib.gnssacq_enqueue_device.argtypes = [vp, vp, C.c_size_t]
    lib.gnssacq_enqueue_device_out.argtypes = [vp, vp, C.c_size_t, vp]
    lib.gnssacq_fetch_results.argtypes = [vp, C.POINTER(Result), C.POINTER(Stats)]
    lib.gnssacq_ca_code.argtypes = [C.c_int32, vp]
    lib.gnssacq_code_replica.argtypes = [C.POINTER(Config), C.c_int32, vp]
    lib.gnssacq_read_surface.argtypes = [vp, C.c_int32, vp]
    lib.gnssacq_fft_forward.argtypes = [vp, vp, vp]
    lib.gnssacq_fine_frequency.argtypes = [vp, vp, C.c_size_t, C.c_int32, C.c_int32, vp, vp, vp]
    lib.gnssacq_search_multi.argtypes = [C.POINTER(vp), C.c_int32, vp, C.c_size_t, C.POINTER(Result)]
    lib.gnssacq_track_load.argtypes = [vp, vp, C.c_size_t]
    lib.gnssacq_loop_params_default.argtypes = [C.POINTER(LoopParams)]
    lib.gnssacq_track.argtypes = [vp, C.c_int32, C.POINTER(Channel), C.POINTER(LoopParams), C.c_int32, C.POINTER(TrackRecord)]
    lib.gnssacq_track_bank.argtypes = [vp, C.c_int32, C.POINTER(Channel), C.POINTER(LoopParams), C.c_int32, C.c_int32, vp,
                                       C.POINTER(TrackRecord), vp, vp]
    lib.gnssacq_correlate.argtypes = [vp, C.c_int32, C.POINTER(Channel), C.c_int32, vp, vp, vp]
    lib.gnssacq_sweep.argtypes = [vp, C.POINTER(vp), C.c_int32, C.c_size_t, C.POINTER(Result), C.POINTER(Stats)]
    lib.gnssacq_sweep_file.argtypes = [vp, C.c_char_p, C.c_int64, C.c_int32, C.c_int32, C.POINTER(Result), C.POINTER(Stats)]
    lib.gnssacq_shard_plan.argtypes = [C.POINTER(Config), C.c_int32, C.c_int32, C.POINTER(Config), C.POINTER(Shard)]
    lib.gnssacq_shard_plan_rows.argtypes = [C.POINTER(Config), C.c_int32, C.c_int32, C.c_int32, C.POINTER(Config), C.POINTER(Shard)]
    lib.gnssacq_xchg_root.argtypes = [vp, C.POINTER(Shard), vp]
    lib.gnssacq_xchg_attach.argtypes = [vp, C.POINTER(Shard), vp]
    lib.gnssacq_xchg_attach_local.argtypes = [vp, C.POINTER(Shard), vp]
    lib.gnssacq_xchg_if_buffer.argtypes = [vp]
    lib.gnssacq_xchg_if_buffer.restype = vp
    lib.gnssacq_xchg_enqueue.argtypes = [vp, vp, C.c_size_t]
    lib.gnssacq_xchg_finish.argtypes = [vp]
    lib.gnssacq_xchg_fetch.argtypes = [vp, C.POINTER(Result), C.POINTER(Stats)]
    lib.gnssacq_fp32_peak_tflops.argtypes = [C.c_int32, C.POINTER(C.c_double)]
    lib.gnssacq_set_doppler_windows.argtypes = [vp, vp, vp]
    lib.gnssacq_transform_size.argtypes = [C.POINTER(Config), C.POINTER(C.c_int32)]
    return lib


lib = _load()


def version() -> str:
    return lib.gnssacq_version().decode()


def default_config() -> Config:
    cfg = Config()
    lib.gnssacq_config_default(C.byref(cfg))
    return cfg


def make_config(*, fs_hz=58e6, if_hz=4.58e6, code_hz=1.023e6, samples_per_ms: Optional[int] = None,
                data_type=2, data_precision=1, freq_min_hz=-10000.0, freq_step_hz=500.0,
                freq_num: Optional[int] = None, noncoh_blocks=20, coh_ms=1,
                prns: Sequence[int] = tuple(range(1, 33)), snr_threshold_db=12.0, device=-1,
                cluster_ctas=0, threads=0, keep_surface=False, exchange=0, work_split=0,
                bin_first=0, bin_count=0, row_first=0, row_count=0) -> Config:
    cfg = default_config()
    cfg.fs_hz, cfg.if_hz, cfg.code_hz = fs_hz, if_hz, code_hz
    cfg.samples_per_ms = int(samples_per_ms if samples_per_ms else np.ceil(fs_hz * 1e-3))
    cfg.data_type, cfg.data_precision = data_type, data_precision
    cfg.freq_min_hz, cfg.freq_step_hz = freq_min_hz, freq_step_hz
    cfg.freq_num = int(freq_num if freq_num is not None else 2 * abs(freq_min_hz) / freq_step_hz + 1)
    cfg.noncoh_blocks, cfg.coh_ms = noncoh_blocks, coh_ms
    prns = list(prns)
    if len(prns) > GNSSACQ_MAX_PRN:
        raise ValueError("too many PRNs")
    cfg.n_prn = len(prns)
    for i in range(GNSSACQ_MAX_PRN):
        cfg.prn[i] = prns[i] if i < len(prns) else 0
    cfg.snr_threshold_db = snr_threshold_db
    cfg.device, cfg.cluster_ctas, cfg.threads = device, cluster_ctas, threads
    cfg.keep_surface = int(bool(keep_surface))
    cfg.exchange = int(exchange)
    cfg.work_split = int(work_split)
    cfg.bin_first, cfg.bin_count = int(bin_first), int(bin_count)
    cfg.row_first, cfg.row_count = int(row_first), int(row_count)
    return cfg


def shard_plan(cfg: Config, rank: int, world: int):
    """gnssacq_shard_plan: (this shard's Config, its Shard).  Whole PRNs per shard when n_prn >= world, else all
    PRNs and a range of Doppler bins; a shard with ``bin_count == 0`` has no rows (more shards than bins)."""
    mine, sh = Config(), Shard()
    rc = lib.gnssacq_shard_plan(C.byref(cfg), rank, world, C.byref(mine), C.byref(sh))
    if rc:
        raise GnssAcqError(rc, (lib.gnssacq_last_error(None) or b"").decode())
    return mine, sh


def shard_plan_rows(cfg: Config, rank: int, world: int, root_extra_permille: int = 0):
    """gnssacq_shard_plan_rows: every shard keeps all PRNs and takes a contiguous range of the (bin-major) rows; the
    root's share is (1000 + root_extra_permille) / 1000 of the others'.  ``row_count == 0``: no rows, no handle."""
    mine, sh = Config(), Shard()
    rc = lib.gnssacq_shard_plan_rows(C.byref(cfg), rank, world, int(root_extra_permille), C.byref(mine), C.byref(sh))
    if rc:
        raise GnssAcqError(rc, (lib.gnssacq_last_error(None) or b"").decode())
    return mine, sh


IPC_BYTES = 64


def ca_code(prn: int) -> np.ndarray:
    out = np.zeros(1023, dtype=np.int8)
    rc = lib.gnssacq_ca_code(prn, out.ctypes.data)
    if rc:
        raise GnssAcqError(rc, STATUS.get(rc, "?"))
    return out


def code_replica(cfg: Config, prn: int) -> np.ndarray:
    out = np.zeros(cfg.samples_per_ms, dtype=np.int8)
    rc = lib.gnssacq_code_replica(C.byref(cfg), prn, out.ctypes.data)
    if rc:
        raise GnssAcqError(rc, STATUS.get(rc, "?"))
    return out


def transform_size(cfg: Config) -> int:
    """Transform length a search of ``cfg.samples_per_ms`` runs on (gnssacq_transform_size): samples_per_ms itself
    when it is built (6000, 26000, 58000), else the built length each ms is zero-padded into.  No device needed."""
    n = C.c_int32()
    rc = lib.gnssacq_transform_size(C.byref(cfg), C.byref(n))
    if rc:
        raise GnssAcqError(rc, (lib.gnssacq_last_error(None) or b"").decode())
    return n.value


def search_multi(searchers: Sequence["Searcher"], if_bytes) -> List[Result]:
    """One process, several GPUs: every Searcher owns a PRN shard on its own device (cfg.device)."""
    buf = np.frombuffer(if_bytes, dtype=np.uint8) if not isinstance(if_bytes, np.ndarray) else if_bytes
    buf = np.ascontiguousarray(buf)
    hs = (C.c_void_p * len(searchers))(*[s._h for s in searchers])
    n_rows = sum(s.cfg.n_prn for s in searchers)
    out = (Result * n_rows)()
    rc = lib.gnssacq_search_multi(hs, len(searchers), buf.ctypes.data, buf.nbytes, out)
    if rc:
        raise GnssAcqError(rc, STATUS.get(rc, "?"))
    return list(out)


def fp32_peak_tflops(device: int = -1) -> float:
    """Measured FP32 FMA throughput of the device (TFLOP/s), the FP32 roofline denominator."""
    out = C.c_double()
    rc = lib.gnssacq_fp32_peak_tflops(device, C.byref(out))
    if rc:
        raise GnssAcqError(rc, (lib.gnssacq_last_error(None) or b"").decode())
    return out.value


class Searcher:
    """Owns one ``gnssacq_handle`` (one GPU, one PRN shard)."""

    def __init__(self, cfg: Config):
        self.cfg = cfg
        self._h = C.c_void_p()
        rc = lib.gnssacq_create(C.byref(cfg), C.byref(self._h))
        if rc:
            raise GnssAcqError(rc, (lib.gnssacq_last_error(None) or b"").decode())
        self.if_bytes = int(lib.gnssacq_if_bytes(C.byref(cfg)))
        self.last_stats: Optional[Stats] = None

    def close(self) -> None:
        if self._h:
            lib.gnssacq_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _check(self, rc: int) -> None:
        if rc:
            raise GnssAcqError(rc, (lib.gnssacq_last_error(self._h) or b"").decode())

    def set_stream(self, cuda_stream: int) -> None:
        self._check(lib.gnssacq_set_stream(self._h, C.c_void_p(cuda_stream)))

    def set_doppler_windows(self, lo_hz: Sequence[float], hi_hz: Sequence[float]) -> None:
        """Search PRN i (cfg.prn order) only over the grid bins whose Doppler lies in [lo_hz[i], hi_hz[i]], for every
        later search until :meth:`clear_doppler_windows`.  A PRN whose window holds no bin is not searched."""
        lo = np.ascontiguousarray(lo_hz, dtype=np.float64)
        hi = np.ascontiguousarray(hi_hz, dtype=np.float64)
        if lo.shape != (self.cfg.n_prn,) or hi.shape != (self.cfg.n_prn,):
            raise ValueError(f"need {self.cfg.n_prn} lower and upper bounds")
        self._check(lib.gnssacq_set_doppler_windows(self._h, lo.ctypes.data, hi.ctypes.data))

    def clear_doppler_windows(self) -> None:
        """Search the full grid again."""
        self._check(lib.gnssacq_set_doppler_windows(self._h, None, None))

    def search(self, if_bytes) -> List[Result]:
        """Host buffer in (bytes / bytearray / numpy int8|int16), result rows out."""
        buf = np.frombuffer(if_bytes, dtype=np.uint8) if not isinstance(if_bytes, np.ndarray) else if_bytes
        buf = np.ascontiguousarray(buf)
        out = (Result * self.cfg.n_prn)()
        st = Stats()
        self._check(lib.gnssacq_search(self._h, buf.ctypes.data, buf.nbytes, out, C.byref(st)))
        self.last_stats = st
        return list(out)

    def sweep(self, windows) -> List[List[Result]]:
        """Re-acquisition sweep: one search per host window (bytes-like), copies overlapped with the searches."""
        bufs = [np.ascontiguousarray(np.frombuffer(w, dtype=np.uint8) if not isinstance(w, np.ndarray) else w)
                for w in windows]
        n, p = len(bufs), self.cfg.n_prn
        if n == 0:
            return []
        each = min(b.nbytes for b in bufs)
        ptrs = (C.c_void_p * n)(*[b.ctypes.data for b in bufs])
        out = (Result * (n * p))()
        st = Stats()
        self._check(lib.gnssacq_sweep(self._h, ptrs, n, each, out, C.byref(st)))
        self.last_stats = st
        return [list(out[i * p:(i + 1) * p]) for i in range(n)]

    def sweep_file(self, path: str, skip_ms: int, epoch_ms: int, n_windows: int) -> List[List[Result]]:
        """Re-acquisition sweep read by the library from a recording file: window j starts `skip_ms + j*epoch_ms`
        ms into the file (acquisition.m:27 with file.skip advanced by `epoch_ms` per epoch)."""
        p = self.cfg.n_prn
        if n_windows <= 0:
            return []
        out = (Result * (n_windows * p))()
        st = Stats()
        self._check(lib.gnssacq_sweep_file(self._h, os.fsencode(path), int(skip_ms), int(epoch_ms), int(n_windows),
                                           out, C.byref(st)))
        self.last_stats = st
        return [list(out[i * p:(i + 1) * p]) for i in range(n_windows)]

    def fetch_stats(self) -> "Stats":
        """Timings of the last enqueued search (synchronises); no rows copied."""
        st = Stats()
        self._check(lib.gnssacq_fetch_results(self._h, None, C.byref(st)))
        self.last_stats = st
        return st

    # ---- multi-GPU exchange through peer memory (include/gnssacq.h: gnssacq_xchg_*) ----
    def xchg_root(self, shard: "Shard") -> bytes:
        """Make this handle the root of a sharded acquisition; returns the IPC handle other processes attach to."""
        buf = C.create_string_buffer(IPC_BYTES)
        self._check(lib.gnssacq_xchg_root(self._h, C.byref(shard), buf))
        self.shard = shard
        return buf.raw

    def xchg_attach(self, shard: "Shard", root_ipc: bytes) -> None:
        self._check(lib.gnssacq_xchg_attach(self._h, C.byref(shard), C.c_char_p(root_ipc)))
        self.shard = shard

    def xchg_attach_local(self, shard: "Shard", root: "Searcher") -> None:
        self._check(lib.gnssacq_xchg_attach_local(self._h, C.byref(shard), root._h))
        self.shard = shard

    def xchg_if_buffer(self) -> int:
        return int(lib.gnssacq_xchg_if_buffer(self._h) or 0)

    def xchg_enqueue(self, host_if=None) -> None:
        if host_if is None:
            self._check(lib.gnssacq_xchg_enqueue(self._h, None, 0))
        else:
            buf = np.ascontiguousarray(np.frombuffer(host_if, dtype=np.uint8) if not isinstance(host_if, np.ndarray) else host_if)
            self._check(lib.gnssacq_xchg_enqueue(self._h, buf.ctypes.data, buf.nbytes))

    def xchg_finish(self) -> None:
        self._check(lib.gnssacq_xchg_finish(self._h))

    def xchg_fetch(self, rows: bool = True) -> List[Result]:
        st = Stats()
        if rows:
            out = (Result * self.shard.n_prn_total)()
            self._check(lib.gnssacq_xchg_fetch(self._h, out, C.byref(st)))
            self.last_stats = st
            return list(out)
        self._check(lib.gnssacq_xchg_fetch(self._h, None, C.byref(st)))
        self.last_stats = st
        return []

    def track_load(self, if_bytes) -> None:
        """Keep a segment of the recording resident in HBM for `correlate`."""
        buf = np.ascontiguousarray(np.frombuffer(if_bytes, dtype=np.uint8) if not isinstance(if_bytes, np.ndarray) else if_bytes)
        self._check(lib.gnssacq_track_load(self._h, buf.ctypes.data, buf.nbytes))

    def correlate(self, channels: Sequence["Channel"], spacing_chips: Sequence[float]):
        """One integration period of every channel: (I, Q), each float64 [n_channels, n_taps]."""
        n, t = len(channels), len(spacing_chips)
        ch = (Channel * n)(*channels)
        sp = np.ascontiguousarray(spacing_chips, dtype=np.float64)
        out_i = np.zeros((n, t), dtype=np.float64)
        out_q = np.zeros((n, t), dtype=np.float64)
        self._check(lib.gnssacq_correlate(self._h, n, ch, t, sp.ctypes.data, out_i.ctypes.data, out_q.ctypes.data))
        return out_i, out_q

    def track(self, start: Sequence["Channel"], n_periods: int, loops: Optional["LoopParams"] = None) -> List[List["TrackRecord"]]:
        """trackingCT.m:70-172 on the device: n_periods integration periods per channel, loops closed on the GPU."""
        if loops is None:
            loops = LoopParams()
            lib.gnssacq_loop_params_default(C.byref(loops))
        n = len(start)
        ch = (Channel * n)(*start)
        out = (TrackRecord * (n * n_periods))()
        self._check(lib.gnssacq_track(self._h, n, ch, C.byref(loops), n_periods, out))
        return [list(out[i * n_periods:(i + 1) * n_periods]) for i in range(n)]

    def track_bank(self, start: Sequence["Channel"], n_periods: int, spacing_chips: Sequence[float],
                   loops: Optional["LoopParams"] = None):
        """`track`, and every period the correlator bank at `spacing_chips` (it only observes the loop): (records,
        bank_i, bank_q), records as `track` returns them, bank_i / bank_q float64 [n_channels, n_periods, n_taps]."""
        if loops is None:
            loops = LoopParams()
            lib.gnssacq_loop_params_default(C.byref(loops))
        n = len(start)
        ch = (Channel * n)(*start)
        sp = np.ascontiguousarray(spacing_chips, dtype=np.float64)
        out = (TrackRecord * (n * n_periods))()
        bank_i = np.zeros((n, n_periods, sp.size), dtype=np.float64)
        bank_q = np.zeros((n, n_periods, sp.size), dtype=np.float64)
        self._check(lib.gnssacq_track_bank(self._h, n, ch, C.byref(loops), n_periods, sp.size, sp.ctypes.data, out,
                                           bank_i.ctypes.data, bank_q.ctypes.data))
        return [list(out[i * n_periods:(i + 1) * n_periods]) for i in range(n)], bank_i, bank_q

    def search_device(self, dev_ptr: int, nbytes: int) -> List[Result]:
        out = (Result * self.cfg.n_prn)()
        st = Stats()
        self._check(lib.gnssacq_search_device(self._h, C.c_void_p(dev_ptr), nbytes, out, C.byref(st)))
        self.last_stats = st
        return list(out)

    def enqueue_device(self, dev_ptr: int, nbytes: int) -> None:
        self._check(lib.gnssacq_enqueue_device(self._h, C.c_void_p(dev_ptr), nbytes))

    def enqueue_device_out(self, dev_ptr: int, nbytes: int, out_dev_ptr: int) -> None:
        """Stream-ordered search whose result rows land in caller-owned HBM (e.g. an NCCL send buffer)."""
        self._check(lib.gnssacq_enqueue_device_out(self._h, C.c_void_p(dev_ptr), nbytes, C.c_void_p(out_dev_ptr)))

    def fetch(self) -> List[Result]:
        out = (Result * self.cfg.n_prn)()
        st = Stats()
        self._check(lib.gnssacq_fetch_results(self._h, out, C.byref(st)))
        self.last_stats = st
        return list(out)

    def fine_frequency(self, if_long, L: int, prns: Sequence[int], code_phases: Sequence[int]) -> np.ndarray:
        """acquisition.m:89-121 on the GPU: `if_long` = (L+1) ms of raw IF bytes, one fineFreq per SV."""
        buf = np.frombuffer(if_long, dtype=np.uint8) if not isinstance(if_long, np.ndarray) else if_long
        buf = np.ascontiguousarray(buf)
        p = np.ascontiguousarray(prns, dtype=np.int32)
        cp = np.ascontiguousarray(code_phases, dtype=np.int32)
        out = np.full(p.size, np.nan, dtype=np.float64)
        if p.size:
            self._check(lib.gnssacq_fine_frequency(self._h, buf.ctypes.data, buf.nbytes, int(L), int(p.size),
                                                   p.ctypes.data, cp.ctypes.data, out.ctypes.data))
        return out

    def read_surface(self, prn_index: int) -> np.ndarray:
        out = np.empty((self.cfg.freq_num, self.cfg.samples_per_ms), dtype=np.float32)
        self._check(lib.gnssacq_read_surface(self._h, prn_index, out.ctypes.data))
        return out

    def fft_forward(self, x: np.ndarray) -> np.ndarray:
        x = np.ascontiguousarray(x, dtype=np.complex64)
        if x.size != self.cfg.samples_per_ms:
            raise ValueError("length must equal samples_per_ms")
        out = np.empty_like(x)
        self._check(lib.gnssacq_fft_forward(self._h, x.ctypes.data, out.ctypes.data))
        return out
