"""Handle lifetime on device 0 (`-m gpu`): closing a handle gives back every buffer its features made on first use, and
a set-up call the library rejects leaves the handle as it was."""
import numpy as np
import pytest
import torch

import gnssacq
from gnssacq import api
from gnssacq.dist import LocalMultiGpu
from oracle.synth import synth_if
from helpers import small_spec, structs

pytestmark = pytest.mark.gpu

N, K = 26000, 2
FS, IF = 26e6, 0.0
PRNS = [3, 7, 22, 9]
GRANULE = 2 << 20                                    # one 2 MiB allocation granule


def _cfg(**kw):
    file, signal, acq = structs(FS, IF, datalen=K, freq_min=-2000.0, freq_step=500.0, freq_num=9)
    return gnssacq.config_from_structs(file, signal, acq, prns=PRNS, device=0, **kw), acq


def _block(start_ms, n_ms):
    return synth_if(small_spec(FS, IF, N), start_ms, n_ms)


def _use_every_feature(tmp_path):
    cfg, acq = _cfg(keep_surface=True)
    with api.Searcher(cfg) as s:
        s.search(_block(0, K))
        s.sweep([_block(3 * i, K) for i in range(3)])
        rec = tmp_path / "rec.bin"
        rec.write_bytes(_block(0, 12))
        s.sweep_file(str(rec), 1, 4, 3)
        L = int(acq.L)
        for l in (L, L - 1):
            s.fine_frequency(_block(0, l + 1), l, [3, 7], [17, 1683 % N])
        s.track_load(_block(0, 6))
        ch = api.Channel(prn=3, num_samples=N, sample_offset=100, carrier_hz=990.0, rem_phase=0.0,
                         code_hz=1.023e6, rem_chip=0.0)
        s.correlate([ch], [-0.5, 0.0, 0.5])
        s.track([ch], 3)
        s.fft_forward(np.ones(N, dtype=np.complex64))
        s.read_surface(1)
    with LocalMultiGpu(_cfg()[0], [0, 0]) as m:
        m.search(_block(0, K))


def test_closing_handles_returns_all_device_memory(tmp_path):
    """Three cycles of: a handle that builds every lazily-made resource set (sweep staging, tracking tables,
    fine-frequency scratch at two L, FFT scratch, kept surface), then a two-shard exchange (root and a shard that
    borrows its block), all closed again.  Free device memory after cycles 2 and 3 is what it was after cycle 1."""
    torch.cuda.init()
    free = []
    for _ in range(3):
        _use_every_feature(tmp_path)
        torch.cuda.synchronize(0)
        free.append(torch.cuda.mem_get_info(0)[0])
    assert abs(free[1] - free[0]) <= GRANULE and abs(free[2] - free[0]) <= GRANULE, free


def test_rejected_exchange_setup_leaves_the_handle_usable():
    """gnssacq_xchg_root with shard 1's description (same shape, wrong rank) is refused with GNSSACQ_ERR_INVALID_ARG;
    the right shard then makes the handle the root, and with a second shard attached the exchange gives the
    single-handle rows byte for byte."""
    cfg, _ = _cfg()
    block = _block(0, K)
    with api.Searcher(cfg) as s:
        want = [bytes(r) for r in s.search(block)]
    mine0, sh0 = api.shard_plan(cfg, 0, 2)
    mine1, sh1 = api.shard_plan(cfg, 1, 2)
    assert (sh0.prn_count, sh0.bin_count) == (sh1.prn_count, sh1.bin_count)
    with api.Searcher(mine0) as root, api.Searcher(mine1) as other:
        with pytest.raises(gnssacq.GnssAcqError) as e:
            root.xchg_root(sh1)
        assert e.value.code == -1                    # GNSSACQ_ERR_INVALID_ARG
        root.xchg_root(sh0)
        other.xchg_attach_local(sh1, root)
        root.xchg_enqueue(block)
        root.xchg_fetch(rows=False)                  # one device: the shards run one after the other
        other.xchg_enqueue(None)
        other.xchg_fetch(rows=False)
        root.xchg_finish()
        assert [bytes(r) for r in root.xchg_fetch()] == want
