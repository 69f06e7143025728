"""ctypes binding of the CPU oracle (oracle/liboracle.so) and of the compiled reference objects (oracle/_ref/libref.so).
TEST INFRASTRUCTURE ONLY — nothing under rtl-sdr-scanner-cpp_b200/ imports this."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess

import numpy as np

from conftest import ROOT, load_b2s

ORACLE_DIR = os.path.join(ROOT, "oracle")
ORACLE_SO = os.path.join(ORACLE_DIR, "liboracle.so")
REF_SO = os.path.join(ORACLE_DIR, "_ref", "libref.so")
REF_OUTPUTS = os.path.join(ROOT, "tests", "golden", "reference_outputs.npz")
MAX_TX = 64

b2s = load_b2s()
BandConfig = b2s.BandConfig


class Outputs(C.Structure):
    _fields_ = [
        ("psd_db", C.c_void_p),
        ("noise_sub_db", C.c_void_p),
        ("avg_db", C.c_void_p),
        ("box_db", C.c_void_p),
        ("peak_index", C.c_void_p),
        ("tx_count", C.c_void_p),
        ("tx_freq", C.c_void_p),
        ("tx_flush", C.c_void_p),
        ("tx_key", C.c_void_p),
        ("tx_power", C.c_void_p),
    ]


_orc = None
_ref = None


def oracle():
    global _orc
    if _orc is None:
        if not os.path.exists(ORACLE_SO) or os.path.getmtime(ORACLE_SO) < os.path.getmtime(os.path.join(ORACLE_DIR, "scan_oracle.cpp")):
            subprocess.check_call(["make", "-C", ORACLE_DIR], stdout=subprocess.DEVNULL)
        L = C.CDLL(ORACLE_SO)
        L.orc_chain_create.restype = C.c_void_p
        L.orc_chain_create.argtypes = [C.POINTER(BandConfig)]
        L.orc_chain_destroy.argtypes = [C.c_void_p]
        L.orc_chain_push.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int64, C.c_double, C.POINTER(Outputs)]
        L.orc_chain_push_psd.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int64, C.c_double, C.POINTER(Outputs)]
        L.orc_chain_reset.argtypes = [C.c_void_p]
        L.orc_chain_set_center.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32]
        L.orc_chain_get_averager.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_int32)]
        L.orc_chain_get_noise.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_int32)]
        L.orc_chain_get_spectrogram.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.orc_chain_clear_spectrogram.argtypes = [C.c_void_p]
        L.orc_hamming.argtypes = [C.c_int, C.c_void_p]
        L.orc_fft_f64.argtypes = [C.c_int, C.c_void_p, C.c_void_p]
        L.orc_fft_f32.argtypes = [C.c_int, C.c_void_p, C.c_void_p]
        L.orc_psd_frame.argtypes = [C.POINTER(BandConfig), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_average.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
        L.orc_get_max_index.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int]
        L.orc_contains_with_margin.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int)]
        L.orc_most_frequent_value.argtypes = [C.c_void_p, C.c_int]
        L.orc_get_tuned_frequency.restype = C.c_int32
        for f in ("orc_spectrogram_message", "orc_transmission_message"):
            getattr(L, f).restype = C.c_size_t
            getattr(L, f).argtypes = [C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_int, C.c_void_p]
        L.orc_averager_create.restype = C.c_void_p
        L.orc_averager_create.argtypes = [C.c_int, C.c_int]
        for f in ("destroy", "reset"):
            getattr(L, "orc_averager_" + f).argtypes = [C.c_void_p]
        for f in ("push", "average", "data", "sum"):
            getattr(L, "orc_averager_" + f).argtypes = [C.c_void_p, C.c_void_p]
        L.orc_averager_frames.argtypes = [C.c_void_p]
        L.orc_bench_run.restype = C.c_double
        L.orc_bench_run.argtypes = [C.POINTER(BandConfig), C.c_void_p, C.c_size_t, C.c_double, C.c_int]
        _orc = L
    return _orc


def have_ref() -> bool:
    return os.path.exists(REF_SO)


def ref():
    """The reference's own objects (Averager, average, collection/radio utils), compiled from /root/reference."""
    global _ref
    if _ref is None:
        L = C.CDLL(REF_SO)
        L.ref_averager_create.restype = C.c_void_p
        L.ref_averager_create.argtypes = [C.c_int, C.c_int]
        L.ref_averager_destroy.argtypes = [C.c_void_p]
        L.ref_averager_reset.argtypes = [C.c_void_p]
        for f in ("push", "average", "data"):
            getattr(L, "ref_averager_" + f).argtypes = [C.c_void_p, C.c_void_p]
        L.ref_average.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
        L.ref_get_max_index.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int]
        L.ref_contains_with_margin.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int)]
        L.ref_most_frequent_value.argtypes = [C.c_void_p, C.c_int]
        L.ref_set_no_data.argtypes = [C.c_void_p, C.c_int]
        L.ref_get_tuned_frequency.restype = C.c_int32
        L.ref_split_range.argtypes = [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int]
        L.ref_get_resamplers_factors.argtypes = [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int]
        # the reference's own BLOCK objects (oracle/ref_blocks_shim.cpp): PSD, NoiseLearner, Transmission, Spectrogram, DataController
        if hasattr(L, "ref_chain_create"):
            L.ref_set_time.argtypes = [C.c_int64]
            L.ref_psd_work.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
            L.ref_chain_create.restype = C.c_void_p
            L.ref_chain_create.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_int, C.c_int64]
            L.ref_chain_destroy.argtypes = [C.c_void_p]
            L.ref_chain_reset.argtypes = [C.c_void_p]
            L.ref_chain_set_center.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int]
            L.ref_chain_push_row.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
            L.ref_published_get.argtypes = [C.c_int, C.c_char_p, C.c_int, C.c_void_p, C.c_int]
            L.ref_push_spectrogram.argtypes = [C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_int]
            L.ref_push_transmission.argtypes = [C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_int]
        _ref = L
    return _ref


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


# ---------------- what the reference's compiled objects returned, stored under tests/golden ----------------
# The tests that compare with the reference read its outputs from REF_OUTPUTS, so they run where the reference is absent.
# tests/golden/make_reference_outputs.py regenerates the file by calling every record_<name>() of those test modules with
# oracle/_ref/libref.so; record_<name>() builds exactly the inputs its test builds. Arrays too large to store are stored as
# one digest per row: the comparisons they stand for are bit for bit.
_recorded = None


def digest(a) -> int:
    """64-bit digest of an array's bytes (or of a bytes object)."""
    b = a if isinstance(a, bytes) else np.ascontiguousarray(a).tobytes()
    return int.from_bytes(hashlib.blake2b(b, digest_size=8).digest(), "little")


def digests(rows) -> np.ndarray:
    return np.array([digest(r) for r in rows], dtype=np.uint64)


def recorded(name: str) -> dict:
    """The arrays record_<name>() stored, keyed by field."""
    global _recorded
    if _recorded is None:
        with np.load(REF_OUTPUTS, allow_pickle=False) as z:
            _recorded = {k: z[k] for k in z.files}
    out = {k.split(".", 1)[1]: v for k, v in _recorded.items() if k.split(".", 1)[0] == name}
    assert out, f"{name} is not in {os.path.relpath(REF_OUTPUTS, ROOT)}: regenerate it with tests/golden/make_reference_outputs.py"
    return out


def pack_lists(lists) -> dict:
    """Per-frame [(shift_hz, flush)] lists -> count per frame + all pairs (int32)."""
    pairs = [p for lst in lists for p in lst]
    return {"count": np.array([len(lst) for lst in lists], np.int32), "pairs": np.array(pairs, np.int32).reshape(-1, 2)}


def unpack_lists(rec: dict):
    ends = np.cumsum(rec["count"])
    return [[(int(f), int(fl)) for f, fl in rec["pairs"][e - c : e]] for c, e in zip(rec["count"], ends)]


def have_ref_blocks() -> bool:
    return have_ref() and hasattr(ref(), "ref_chain_create")


class RefBlocksChain:
    """psd -> NoiseLearner -> Transmission (+ psd -> Spectrogram -> DataController) built from the REFERENCE's own compiled
    objects, wired like SdrDevice::setupChains (sdr_device.cpp:147-171) and driven one PSD row at a time with an injected clock."""

    def __init__(self, cfg: BandConfig, t0_ms: int, bandwidth_hz: int, with_spectrogram: bool = True):
        import json

        self.cfg, self.L = cfg, ref()
        ignored = [[int(cfg.ignored_lo_hz[i]), int(cfg.ignored_hi_hz[i])] for i in range(cfg.n_ignored)]
        text = json.dumps({"ignored": ignored, "bandwidth": int(bandwidth_hz), "min_time_ms": int(cfg.min_time_ms), "timeout_ms": int(cfg.timeout_ms),
                           "tuning_step": int(cfg.tuning_step_hz)})
        self.h = C.c_void_p(self.L.ref_chain_create(text.encode(), cfg.fft_size, cfg.sample_rate_hz, cfg.center_hz, cfg.range_lo_hz, cfg.range_hi_hz,
                                                    cfg.group_size_bins, cfg.start_level, cfg.stop_level, 1 if with_spectrogram else 0, t0_ms))
        self.L.ref_published_clear()

    def push_row(self, psd_row, now_ms):
        n = self.cfg.fft_size
        row = np.ascontiguousarray(psd_row, dtype=np.float32)
        q = np.empty(n, dtype=np.float32)
        cap = 1024  # the reference's list is unbounded; the oracle / engine report the first MAX_TX entries
        freq = np.zeros(cap, dtype=np.int32)
        flush = np.zeros(cap, dtype=np.int32)
        k = self.L.ref_chain_push_row(self.h, _p(row), int(now_ms), _p(q), _p(freq), _p(flush), cap)
        return q, [(int(freq[i]), int(flush[i])) for i in range(min(k, cap))]

    def reset(self):
        self.L.ref_chain_reset(self.h)

    def set_center(self, c, lo, hi):
        self.L.ref_chain_set_center(self.h, c, lo, hi)

    def published(self, clear=True):
        out = []
        for i in range(self.L.ref_published_count()):
            topic = C.create_string_buffer(128)
            buf = np.empty(1 << 16, dtype=np.uint8)
            k = self.L.ref_published_get(i, topic, 128, _p(buf), buf.size)
            out.append((topic.value.decode(), buf[:k].tobytes()))
        if clear:
            self.L.ref_published_clear()
        return out

    def __del__(self):
        try:
            self.L.ref_chain_destroy(self.h)
        except Exception:
            pass


class CpuAverager:
    """Averager through either the oracle restatement (kind='orc') or the compiled reference (kind='ref')."""

    def __init__(self, size, group, kind="orc"):
        self.size, self.group, self.kind = size, group, kind
        self.L = oracle() if kind == "orc" else ref()
        self.h = C.c_void_p(getattr(self.L, f"{kind}_averager_create")(size, group))

    def push(self, row):
        x = np.ascontiguousarray(row, dtype=np.float32)
        getattr(self.L, f"{self.kind}_averager_push")(self.h, _p(x))

    def reset(self):
        getattr(self.L, f"{self.kind}_averager_reset")(self.h)

    def average(self):
        out = np.empty(self.size, dtype=np.float32)
        getattr(self.L, f"{self.kind}_averager_average")(self.h, _p(out))
        return out

    def data(self):
        out = np.empty((self.group, self.size), dtype=np.float32)
        getattr(self.L, f"{self.kind}_averager_data")(self.h, _p(out))
        return out

    def sum(self):
        assert self.kind == "orc"
        out = np.empty(self.size, dtype=np.float32)
        self.L.orc_averager_sum(self.h, _p(out))
        return out, self.L.orc_averager_frames(self.h)

    def __del__(self):
        try:
            getattr(self.L, f"{self.kind}_averager_destroy")(self.h)
        except Exception:
            pass


def cpu_average(x, group, kind="orc"):
    x = np.ascontiguousarray(x, dtype=np.float32)
    # zeros, like Transmission::process's avgPower (transmission.cpp:60): with groupSize 1 the reference loop
    # (utils.cpp:38) never writes the last element, so it keeps this initial 0.0
    out = np.zeros_like(x)
    L = oracle() if kind == "orc" else ref()
    getattr(L, f"{kind}_average")(_p(x), _p(out), x.shape[0], group)
    return out


class ChainResult:
    pass


class OracleChain:
    """The restated decimator..transmission(+spectrogram) chain (oracle/scan_oracle.cpp)."""

    def __init__(self, cfg: BandConfig, fp32: bool = False):
        self.cfg = BandConfig.from_buffer_copy(cfg)
        if fp32:
            self.cfg.flags |= 1
        else:
            self.cfg.flags &= ~1
        self.L = oracle()
        self.h = C.c_void_p(self.L.orc_chain_create(C.byref(self.cfg)))
        assert self.h, "orc_chain_create failed"

    def push(self, iq, n_frames, t0_ms, period_ms, dense=("psd_db", "noise_sub_db", "avg_db", "box_db"), psd_rows=False):
        """iq: the frames' IQ samples — or, with psd_rows=True, their PSD rows [n_frames][N] (the chain from PSD::work's output on)."""
        n = self.cfg.fft_size
        iq = np.ascontiguousarray(iq)
        r = ChainResult()
        o = Outputs()
        for name in ("psd_db", "noise_sub_db", "avg_db", "box_db"):
            if name in dense:
                arr = np.zeros((n_frames, n), dtype=np.float32)
                setattr(o, name, arr.ctypes.data)
                setattr(r, name, arr)
            else:
                setattr(r, name, None)
        r.peak_index = np.zeros(n_frames, dtype=np.int32)
        r.tx_count = np.zeros(n_frames, dtype=np.int32)
        r.tx_freq = np.zeros((n_frames, MAX_TX), dtype=np.int32)
        r.tx_flush = np.zeros((n_frames, MAX_TX), dtype=np.int32)
        r.tx_key = np.zeros((n_frames, MAX_TX), dtype=np.int32)
        r.tx_power = np.zeros((n_frames, MAX_TX), dtype=np.float32)
        for name in ("peak_index", "tx_count", "tx_freq", "tx_flush", "tx_key", "tx_power"):
            setattr(o, name, getattr(r, name).ctypes.data)
        if psd_rows:
            rc = self.L.orc_chain_push_psd(self.h, _p(np.ascontiguousarray(iq, dtype=np.float32)), n_frames, t0_ms, period_ms, C.byref(o))
        else:
            rc = self.L.orc_chain_push(self.h, _p(iq), n_frames, t0_ms, period_ms, C.byref(o))
        assert rc == 0
        r.frame_tx = [
            [(int(r.tx_freq[k, s]), int(r.tx_flush[k, s]), int(r.tx_key[k, s]), float(r.tx_power[k, s])) for s in range(min(int(r.tx_count[k]), MAX_TX))]
            for k in range(n_frames)
        ]
        return r

    def reset(self):
        self.L.orc_chain_reset(self.h)

    def set_center(self, c, lo, hi):
        self.L.orc_chain_set_center(self.h, c, lo, hi)

    def get_averager(self):
        n, y = self.cfg.fft_size, self.cfg.grouping_y
        s = np.empty(n, dtype=np.float32)
        a = np.empty(n, dtype=np.float32)
        ring = np.empty((y, n), dtype=np.float32)
        f = C.c_int32()
        self.L.orc_chain_get_averager(self.h, _p(s), _p(a), _p(ring), C.byref(f))
        return s, a, ring, f.value

    def get_noise(self):
        thr = np.full(self.cfg.fft_size, -np.finfo(np.float32).max, dtype=np.float32)
        samples = C.c_int32()
        ready = self.L.orc_chain_get_noise(self.h, _p(thr), C.byref(samples))
        return thr, samples.value, bool(ready)

    def get_signals(self, cap=4096):
        keys, first, last, power = np.zeros(cap, np.int32), np.zeros(cap, np.int64), np.zeros(cap, np.int64), np.zeros(cap, np.float32)
        self.L.orc_chain_get_signals.argtypes = [C.c_void_p] + [C.c_void_p] * 4 + [C.c_int]
        k = min(self.L.orc_chain_get_signals(self.h, _p(keys), _p(first), _p(last), _p(power), cap), cap)
        return keys[:k], first[:k], last[:k], power[:k]

    def get_transmissions(self, cap=4096):
        """The complete sorted list after the most recent frame: [(shift_hz, flush, key, power)]."""
        f, fl, key, pw = np.zeros(cap, np.int32), np.zeros(cap, np.int32), np.zeros(cap, np.int32), np.zeros(cap, np.float32)
        self.L.orc_chain_get_transmissions.argtypes = [C.c_void_p] + [C.c_void_p] * 4 + [C.c_int]
        k = min(self.L.orc_chain_get_transmissions(self.h, _p(f), _p(fl), _p(key), _p(pw), cap), cap)
        return [(int(f[i]), int(fl[i]), int(key[i]), float(pw[i])) for i in range(k)]

    def get_spectrogram(self, cap=64):
        m = max(self.cfg.spectrogram_out_size, 1)
        times = np.zeros(cap, dtype=np.int64)
        centers = np.zeros(cap, dtype=np.int32)
        rows = np.zeros((cap, m), dtype=np.int8)
        k = self.L.orc_chain_get_spectrogram(self.h, _p(times), _p(centers), _p(rows), cap)
        self.L.orc_chain_clear_spectrogram(self.h)
        k = min(k, cap)
        return times[:k], centers[:k], rows[:k]

    def __del__(self):
        try:
            self.L.orc_chain_destroy(self.h)
        except Exception:
            pass


def oracle_psd_frame(cfg, iq_frame, window=None, want_linear=False):
    n = cfg.fft_size
    psd = np.empty(n, dtype=np.float32)
    lin = np.empty(n, dtype=np.float32) if want_linear else None
    iq_frame = np.ascontiguousarray(iq_frame)
    oracle().orc_psd_frame(C.byref(cfg), _p(window), _p(iq_frame), _p(psd), _p(lin))
    return (psd, lin) if want_linear else psd


def hamming(n):
    w = np.empty(n, dtype=np.float32)
    oracle().orc_hamming(n, _p(w))
    return w


def db_rows_stats(got_db, ref_db):
    """Parity statistics for dB rows against the oracle (DESIGN.md "Parity criterion").
    worst / pass_frac: the floored linear-power criterion |p - p_ref| <= tol * max(p_ref, median_row(p_ref));
    db_max_main: largest |dB error| over bins within 10 dB of (or above) the row median — the bins that matter to the
    detector; deep nulls far below the noise floor have unbounded dB error in ANY fp32 FFT and are covered by `worst`."""
    got = np.asarray(got_db, np.float64)
    ref = np.asarray(ref_db, np.float64)
    pg, pr = 10.0 ** (got / 10.0), 10.0 ** (ref / 10.0)
    med = np.median(pr, axis=-1, keepdims=True)
    rel = np.abs(pg - pr) / np.maximum(pr, med)
    main = ref >= (10.0 * np.log10(med) - 10.0)
    return {
        "worst": float(rel.max()),
        "pass_frac": float(np.mean(rel <= 1e-5)),
        "db_max_main": float(np.max(np.abs(got - ref)[main])),
        "db_max_all": float(np.max(np.abs(got - ref))),
    }


def worst_tolerance(n_fft):
    """Bound on the single worst floored relative power error of a row. 1e-4 up to N = 16384; above, it widens with sqrt(N / 16384):
    the worst of N samples of fp32 rounding noise grows with N and log N — the oracle's OWN fp32 FFT against its fp64 FFT gives
    3.0e-5 / 6.1e-5 / 9.1e-5 for one frame of N = 16384 / 65536 / 262144 (measured, see DESIGN.md section 4)."""
    return 1e-4 * max(1.0, n_fft / 16384.0) ** 0.5


def assert_db_rows_close(got_db, ref_db, what=""):
    st = db_rows_stats(got_db, ref_db)
    # 1e-5 relative on power == 4.3e-5 dB; the fp32 rounding of a dB value near -70 is already 3.8e-6 dB
    assert st["worst"] <= worst_tolerance(np.asarray(ref_db).shape[-1]) and st["pass_frac"] >= 0.995 and st["db_max_main"] <= 2e-3, (what, st)
    return st
