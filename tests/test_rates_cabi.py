"""Front-end sample rates that are not a built transform length, at the C ABI without a GPU: the transform rule of
gnssacq_transform_size, gnssacq_create getting past validation at those rates (to the missing device), the sampled
code replica at each new rate against the oracle's acquisition.m:50-51, and the MATLAB gateway, which passes
signal.Sample through unchanged."""
import ctypes as C
import os

import numpy as np
import pytest

import gnssacq
import oracle
from oracle.acquisition_ref import code_replica
from gnssacq import api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# (samples_per_ms, transform length): built lengths run as they are; any other N <= 29 000 is zero-padded into the
# smallest built length >= 2N - 1
RULE = [(2048, 6000), (3000, 6000), (3001, 26000), (4092, 26000), (13000, 26000), (13001, 58000), (16368, 58000),
        (29000, 58000), (6000, 6000), (26000, 26000), (58000, 58000), (1, 6000), (4000, 26000)]
UNSUPPORTED = [29001, 34000, 38192, 58001, 0, -6000]

# front ends the padded path opens up: (Fs, IF)
RATES = [(2.048e6, 0.0), (4.092e6, 1.023e6), (5e6, 0.0), (8.184e6, 2.046e6), (10e6, 0.0), (13e6, 0.0), (13.001e6, 0.0),
         (16.368e6, 4.092e6), (16.3676e6, 4.1304e6), (20e6, 0.0), (25e6, 0.0), (29e6, 0.0)]


def cfg_n(n, **kw):
    cfg = api.make_config(**kw)
    cfg.samples_per_ms = n                              # (make_config would take 0 as "from fs_hz")
    return cfg


@pytest.mark.parametrize("n,nf", RULE)
def test_transform_size_rule(n, nf):
    cfg = cfg_n(n)
    out = C.c_int32(-1)
    assert api.lib.gnssacq_transform_size(C.byref(cfg), C.byref(out)) == 0
    assert out.value == nf
    assert api.transform_size(cfg) == nf


@pytest.mark.parametrize("n", UNSUPPORTED)
def test_transform_size_unsupported(n):
    cfg = cfg_n(n)
    out = C.c_int32(-1)
    assert api.lib.gnssacq_transform_size(C.byref(cfg), C.byref(out)) == -2
    assert out.value == -1                              # left alone
    with pytest.raises(gnssacq.GnssAcqError) as e:
        api.transform_size(cfg)
    assert e.value.code == -2
    assert api.lib.gnssacq_transform_size(None, C.byref(out)) == -1
    assert api.lib.gnssacq_transform_size(C.byref(cfg), None) == -1


@pytest.mark.parametrize("n", [n for n, _ in RULE] + UNSUPPORTED)
def test_create_agrees_with_the_transform_rule(n):
    """Without a GPU, a supported N gets through validation and variant choice to GNSSACQ_ERR_NO_DEVICE; an
    unsupported one stops at GNSSACQ_ERR_UNSUPPORTED_N, as gnssacq_transform_size says."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    cfg = cfg_n(n, fs_hz=max(n, 1) * 1e3, if_hz=0.0)
    out = C.c_int32()
    want = api.lib.gnssacq_transform_size(C.byref(cfg), C.byref(out))
    h = C.c_void_p()
    rc = api.lib.gnssacq_create(C.byref(cfg), C.byref(h))
    assert rc == (-5 if want == 0 else -2), (n, rc)
    assert not h


@pytest.mark.parametrize("fs,if_hz", RATES)
def test_code_replica_matches_oracle_at_new_rates(fs, if_hz):
    """acquisition.m:51 samples the doubled code at ceil(n*fc/Fs) in double: re-checked at every new Fs."""
    signal = oracle.SignalParams(IF=if_hz, Fs=fs)
    n = int(signal.Sample)
    assert n == int(np.ceil(fs * 1e-3))
    cfg = gnssacq.make_config(fs_hz=fs, if_hz=if_hz)
    assert cfg.samples_per_ms == n
    assert api.transform_size(cfg) >= 2 * n - 1
    for prn in (1, 7, 19, 32, 37):
        assert np.array_equal(api.code_replica(cfg, prn), code_replica(signal, prn).astype(np.int8)), (fs, prn)


@pytest.mark.parametrize("fs,if_hz", RATES[:3] + RATES[7:9])
def test_wrapper_config_carries_signal_sample(fs, if_hz):
    """acquisition()'s config is built from signal.Sample with no rate logic of its own: the same N, hence the same
    transform rule, as the reference's initParameters.m:46."""
    from helpers import structs
    file, signal, acq = structs(fs, if_hz, datalen=4)
    cfg = gnssacq.config_from_structs(file, signal, acq, prns=[1, 2])
    assert cfg.samples_per_ms == int(signal.Sample) == int(np.ceil(fs * 1e-3))
    assert cfg.fs_hz == fs and cfg.if_hz == if_hz
    assert api.lib.gnssacq_if_bytes(C.byref(cfg)) == int(signal.Sample) * 2 * 4


def test_mex_gateway_passes_samples_per_ms_through():
    """matlab/gnssacq_mex.c has no rate logic: it copies samples_per_ms into the config and compiles against the
    header that documents the padded rates."""
    import subprocess
    src = os.path.join(ROOT, "assignment-for-aae6102_gnss-sdr_b200", "matlab", "gnssacq_mex.c")
    subprocess.check_call(["gcc", "-fsyntax-only", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                           "-I", os.path.join(ROOT, "tests", "stubs"), src])
    text = open(src).read()
    assert 'c.samples_per_ms = (int32_t)field(cs, "samples_per_ms", c.samples_per_ms);' in text
    assert "2000" not in text
