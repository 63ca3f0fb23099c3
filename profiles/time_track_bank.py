"""Device-side tracking loop with its correlator bank (gnssacq_track_bank) against gnssacq_track (E/P/L only) and the
host-driven 25-tap loop (gnssacq_correlate + loop filters in Python): wall time per tracked millisecond, 58 MHz int8
I/Q, Opensky-shaped synthetic recording, 1000 integration periods per channel.
Usage: python profiles/time_track_bank.py [--ab DIR]
--ab DIR: DIR holds a gnssacq package (its .py files and libgnssacq.so) built from another commit; gnssacq_track of
that build and of this one are timed in alternating child processes (same box, same run) and their records compared
byte for byte."""
import os
import subprocess
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
PKG = os.path.join(ROOT, "assignment-for-aae6102_gnss-sdr_b200")

CHILD = r'''
import hashlib, sys, time
sys.path[:0] = [sys.argv[2], sys.argv[1]]
import gnssacq
from gnssacq import api
from gnssacq.synth import opensky_recording
import time_track_bank as t
start = t._start()
raw = opensky_recording().read(0, t.PERIODS + 3)
with api.Searcher(gnssacq.make_config(fs_hz=t.FS, if_hz=t.IF_HZ, prns=[1])) as s:
    s.track_load(raw)
    s.track(start, t.PERIODS)
    best = 1e9
    for _ in range(5):
        t0 = time.perf_counter()
        recs = s.track(start, t.PERIODS)
        best = min(best, time.perf_counter() - t0)
print(best / t.PERIODS * 1e6, hashlib.sha1(b"".join(bytes(r) for ch in recs for r in ch)).hexdigest()[:12])
'''

FS, IF_HZ, N, PERIODS = 58e6, 4.58e6, 58000, 1000
BANK25 = [round(0.6 - 0.05 * i, 2) for i in range(25)]          # trackingCT_POS_updated_multicorrelator.m:41
TAPS32 = [round(-0.75 + 0.05 * i, 2) for i in range(32)]
TRUTH = list(zip((3, 4, 16, 22, 26, 27, 31, 32), (990.0, -3095.0, -305.0, 1565.0, 1835.0, -3225.0, 1045.0, 3345.0),
                 (3683, 12701, 26051, 2610, 57908, 49778, 39064, 20170)))     # gnssacq/synth.py::opensky_recording


def _start():
    from gnssacq import api
    return [api.Channel(prn=t[0], num_samples=0, sample_offset=N - t[2] + 1, carrier_hz=IF_HZ + t[1] + 5.0, rem_phase=0.0,
                        code_hz=1.023e6, rem_chip=0.0) for t in TRUTH]


def _timed(fn, reps=5):
    """Median wall time of `reps` calls after one warm-up call; each call ends in a stream synchronise."""
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        ts.append(time.perf_counter() - t0)
    return sorted(ts)[reps // 2], out


def main():
    import gnssacq
    from gnssacq import api
    from gnssacq.synth import opensky_recording
    from oracle import tracking_ref as tr

    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    print(f"# python profiles/time_track_bank.py on {gpu} (58 MHz int8 I/Q, {PERIODS} periods per channel, float64; "
          "median of 5 calls after a warm-up, each ending in a stream synchronise)", flush=True)
    raw = opensky_recording().read(0, PERIODS + 3)
    start = _start()
    with api.Searcher(gnssacq.make_config(fs_hz=FS, if_hz=IF_HZ, prns=[1])) as s:
        s.track_load(raw)
        for n_ch in (1, 8):
            dt, recs = _timed(lambda: s.track(start[:n_ch], PERIODS))
            print(f"gnssacq_track (E/P/L)         : {n_ch} channels: {dt / PERIODS * 1e6:6.1f} us per ms", flush=True)
            for name, sp in (("25-tap bank", BANK25), ("32 taps    ", TAPS32)):
                db, (recs_b, bi, bq) = _timed(lambda: s.track_bank(start[:n_ch], PERIODS, sp))
                same = [bytes(r) for ch in recs_b for r in ch] == [bytes(r) for ch in recs for r in ch]
                print(f"gnssacq_track_bank {name}: {n_ch} channels: {db / PERIODS * 1e6:6.1f} us per ms "
                      f"(records identical to gnssacq_track: {same})", flush=True)
            # host-driven: one gnssacq_correlate call per ms with the 25-tap bank, loop filters in Python on E/P/L
            sts = [tr.ChannelState(prn=c.prn, carrier_basis_hz=c.carrier_hz, carrier_hz=c.carrier_hz, sample_pos=c.sample_offset)
                   for c in start[:n_ch]]
            ep = [BANK25.index(-0.5), BANK25.index(0.0), BANK25.index(0.5)]

            def host_ms():
                ns = [tr.num_samples(st.code_hz, FS, st.rem_chip) for st in sts]
                chans = [api.Channel(prn=st.prn, num_samples=k, sample_offset=st.sample_pos, carrier_hz=st.carrier_hz,
                                     rem_phase=st.rem_phase, code_hz=st.code_hz, rem_chip=st.rem_chip) for st, k in zip(sts, ns)]
                gi, gq = s.correlate(chans, BANK25)
                for c, st in enumerate(sts):
                    tr.close_loops(st, gi[c][ep], gq[c][ep], ns[c], FS)
            host_ms()
            t0 = time.perf_counter()
            for _ in range(200):
                host_ms()
            dh = (time.perf_counter() - t0) / 200
            print(f"host-driven 25-tap loop       : {n_ch} channels: {dh * 1e6:6.1f} us per ms "
                  "(gnssacq_correlate + Python loop filters, 200 ms)", flush=True)
    if "--ab" in sys.argv:
        other = os.path.abspath(sys.argv[sys.argv.index("--ab") + 1])
        libs = [("other", other), ("this", PKG)]
        res = {name: [] for name, _ in libs}
        for _ in range(3):
            for name, path in libs:
                out = subprocess.run([sys.executable, "-c", CHILD, HERE, path], capture_output=True, text=True)
                if out.returncode:
                    sys.exit(f"{name}: {out.stderr[-2000:]}")
                us, digest = out.stdout.split()
                res[name].append((float(us), digest))
        print("gnssacq_track A/B, 8 channels, best of 5 calls per child, 3 alternating children each: " +
              "; ".join(f"{name} {[round(u, 2) for u, _ in v]} us per ms, records {v[0][1]}" for name, v in res.items()),
              flush=True)


if __name__ == "__main__":
    sys.path[:0] = [PKG, ROOT]
    main()
