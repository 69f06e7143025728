"""Scanner hop policy and recorder assignment (SURVEY.md §8(f)#3), CPU only. The product's host state machine (csrc/scan_policy.h, through
the C ABI) against (1) the reference's gtest vectors for getRangeSplitSampleRate / splitRange (tests/test_radio_utils.cpp:105-132),
(2) what the compiled reference functions returned (tests/golden/reference_outputs.npz), and (3) an independent Python restatement of
Scanner::worker (scanner.cpp:36-64) and SdrDevice::updateRecordings (sdr_device.cpp:82-144) on randomised notification sequences."""
import ctypes as C

import numpy as np

import oracle_lib as ol
from conftest import load_b2s
from test_oracle_kats import G

b2s = load_b2s()


def test_range_split_against_reference_vectors():
    for fs, want in G["range_split_sample_rate"]["cases"]:
        assert b2s.get_range_split_sample_rate(fs) == want
    for lo, hi, fs, want in G["split_range"]["cases"]:
        # splitRange with the split rate given directly: a policy whose device sample rate maps onto itself
        assert b2s.get_range_split_sample_rate(fs) == fs
        assert b2s.ScanPolicy([(lo, hi)], fs, 1).ranges() == [tuple(r) for r in want]
    want = ol.recorded("range_split")
    for fs, split, ranges in zip(SPLIT_RATES, want["rate"], ol.unpack_lists(want), strict=True):
        assert b2s.get_range_split_sample_rate(fs) == split
        assert b2s.ScanPolicy([(144_000_000, 174_000_000)], fs, 2).ranges() == ranges


SPLIT_RATES = (2_048_000, 20_480_000, 250_000, 1_920_000)


def record_range_split():
    """getRangeSplitSampleRate and splitRange(144-174 MHz) of the compiled reference."""
    R = ol.ref()
    buf = np.zeros(512, np.int32)
    rates, lists = [], []
    for fs in SPLIT_RATES:
        split = R.ref_get_range_split_sample_rate(fs)
        k = R.ref_split_range(144_000_000, 174_000_000, split, buf.ctypes.data_as(C.c_void_p), 256)
        rates.append(split)
        lists.append([(int(buf[2 * i]), int(buf[2 * i + 1])) for i in range(k)])
    return {"rate": np.array(rates, np.int64), **ol.pack_lists(lists)}


class PyScanner:
    """Restated from scanner.cpp:36-64 (hop rule) and sdr_device.cpp:82-144 (updateRecordings); recorder.cpp:54-96 for the recorder state."""

    MAXF = 2**31 - 1

    def __init__(self, n_ranges, n_recorders, scanning_time):
        self.n_ranges, self.scanning_time = n_ranges, scanning_time
        self.rec = [dict(recording=False, shift=self.MAXF, first=0, last=0) for _ in range(n_recorders)]
        self.ignored = set()
        self.current, self.start = 0, 0

    def notify(self, now, lst):
        actions = []
        waiting = lambda s: any(s == f for f, _ in lst)
        for i, r in enumerate(self.rec):  # sdr_device.cpp:102-110
            if r["recording"] and not waiting(r["shift"]):
                actions.append((b2s.REC_STOP, i, r["shift"], r["last"] - r["first"]))
                self.rec[i] = dict(recording=False, shift=self.MAXF, first=0, last=0)
        for shift, flush in lst:  # sdr_device.cpp:112-135
            hit = [i for i, r in enumerate(self.rec) if r["shift"] == shift]
            if hit:
                if flush:
                    self.rec[hit[0]]["last"] = now
                    actions.append((b2s.REC_FLUSH, hit[0], shift, 0))
                continue
            free = [i for i, r in enumerate(self.rec) if not r["recording"]]
            if free:
                self.rec[free[0]] = dict(recording=True, shift=shift, first=now, last=now)
                actions.append((b2s.REC_START, free[0], shift, 0))
            elif shift not in self.ignored:
                self.ignored.add(shift)
                actions.append((b2s.REC_NONE_FREE, -1, shift, 0))
        self.ignored = {s for s in self.ignored if waiting(s)}  # sdr_device.cpp:137-143
        hop = None
        if self.n_ranges > 1 and not (now <= self.start + self.scanning_time or len(lst) > 0):  # scanner.cpp:51-55
            self.current = (self.current + 1) % self.n_ranges
            self.start = now
            hop = self.current
        return actions, hop


def test_policy_follows_the_restated_scanner_on_random_notifications():
    rng = np.random.default_rng(5)
    for trial in range(30):
        n_rec = int(rng.integers(0, 4))
        ranges = [(100_000_000, 100_000_000 + int(rng.integers(1, 5)) * 2_000_000), (400_000_000, 402_000_000)][: int(rng.integers(1, 3))]
        pol = b2s.ScanPolicy(ranges, 2_048_000, n_rec, 500)
        split = pol.ranges()
        py = PyScanner(len(split), n_rec, 500)
        now = 1_000_000
        assert pol.begin(now) == split[0]
        py.start = now
        live, kinds = [], set()
        for step in range(400):
            now += int(rng.integers(5, 120))
            # the mailbox list evolves like real transmissions: births, deaths, flush flags, occasional reordering by power
            if rng.random() < 0.15 and len(live) < 5:
                live.append(int(rng.integers(-400, 400)) * 2500)
            if live and rng.random() < 0.12:
                live.pop(int(rng.integers(0, len(live))))
            if rng.random() < 0.2:
                rng.shuffle(live)
            lst = [(s, bool(rng.random() < 0.4)) for s in dict.fromkeys(live)]
            got_a, got_hop = pol.notify(now, lst)
            want_a, want_hop = py.notify(now, lst)
            assert got_a == want_a, (trial, step)
            assert got_hop == (split[want_hop] if want_hop is not None else None), (trial, step)
            kinds |= {a[0] for a in got_a}
        if n_rec >= 1:
            assert {b2s.REC_START, b2s.REC_STOP} <= kinds
