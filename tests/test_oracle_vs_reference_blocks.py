"""Pins the oracle (and the wire-format helpers) against what the REFERENCE'S OWN COMPILED BLOCKS returned.

The reference objects are sources/radio/blocks/{psd,noise_learner,transmission,spectrogram}.cpp, sources/radio/{signal,averager}.cpp,
sources/network/data_controller.cpp and sources/utils/*.cpp of the reference, compiled unmodified into oracle/_ref/libref.so by
`make -C oracle ref` (see oracle/ref_blocks_shim.cpp for the name-only stand-ins of GNU Radio / Paho / Config and for the injected
clock). What they returned for the inputs of these tests is stored in tests/golden/reference_outputs.npz: record_<name>() below
made it (tests/golden/make_reference_outputs.py runs them), so the tests need no reference code. The same PSD rows go through the
reference objects and through oracle/scan_oracle.cpp with the same frame clock; everything must agree exactly:
  * PSD::work                      bit for bit on identical spectra
  * NoiseLearner::work             every output row bit for bit, the length of the learning phase
  * Transmission::work             the FrequencyFlush list handed to TransmissionNotification, every frame
  * Spectrogram::work + DataController::pushSpectrogram   every published payload, byte for byte
The window and the FFT itself are gr::fft::fft_v (GNU Radio + FFTW, not in the reference tree): those stay unpinned."""
import ctypes as C
import struct

import numpy as np
import pytest

import oracle_lib as ol
from conftest import ROOT, load_b2s

b2s = load_b2s()
import sys  # noqa: E402

sys.path.insert(0, ROOT)
import __graft_entry__ as ge  # noqa: E402

synth = ge.load_synth()

NOISE_LEARNING_MS = 2000  # NOISE_LEARNING_TIME, sources/config.h:24 (compiled into the reference objects)
PERIOD_MS = 25.0          # frame clock of the test: 2000 ms of learning = 81 frames
T0 = 1_700_000_000_000


def _scene(n=1024, fs=2_048_000, frames=520, **kw):
    learn = b2s.lib().b2s_learn_frames_from_ms(NOISE_LEARNING_MS, PERIOD_MS)
    bw = 16 * fs // n
    cfg = b2s.make_config(n, fs, learn_frames=learn, recording_bandwidth_hz=bw, min_time_ms=200, timeout_ms=300, **kw)
    tones = synth.standard_scene(n, frames, learn)
    iq = synth.make_iq_int8(n, frames, tones, seed=synth.seed_for(7), quiet_frames=learn)
    return cfg, iq, frames, learn, bw


def _now(k):
    return T0 + int(np.floor(k * PERIOD_MS + 0.5))


def _reference_rows(ref, psd_rows, times):
    """PSD rows through the reference chain: a digest of every NoiseLearner row and the Transmission list of every frame."""
    rows, lists = [], []
    for row, now in zip(psd_rows, times):
        q, tx = ref.push_row(row, now)
        rows.append(q)
        lists.append(tx)
    return {"rows": ol.digests(rows), **ol.pack_lists(lists)}


def _assert_follows(want, r, what=""):
    """The oracle's NoiseLearner rows and lists of one push `r` against the reference's, frame by frame."""
    lists = ol.unpack_lists(want)
    assert len(lists) == len(r.frame_tx)
    for k, tx in enumerate(lists):
        assert ol.digest(r.noise_sub_db[k]) == want["rows"][k], f"NoiseLearner row {k}{what}"
        assert tx == [(f, fl) for f, fl, _, _ in r.frame_tx[k]], f"transmission list of frame {k}{what}"
    return lists


def _spectra():
    rng = np.random.default_rng(3)
    n, items, fs = 512, 5, 2_048_000
    x = (rng.standard_normal(2 * n * items) * rng.choice([1e-3, 1.0, 300.0], 2 * n * items)).astype(np.float32)
    x[:4] = 0.0  # |z| = 0 -> -inf in both
    return n, items, fs, x


def record_psd_work():
    n, items, fs, x = _spectra()
    got = np.empty(n * items, dtype=np.float32)
    ol.ref().ref_psd_work(n, fs, x.ctypes.data_as(C.c_void_p), got.ctypes.data_as(C.c_void_p), items)
    return {"rows": ol.digests(got.reshape(items, n)), "first": got[:1]}


def test_psd_work_bit_exact():
    n, items, fs, x = _spectra()
    want = ol.recorded("psd_work")
    got = np.empty(n * items, dtype=np.float32)
    ol.oracle().orc_psd_from_spectrum(n, fs, x.ctypes.data_as(C.c_void_p), got.ctypes.data_as(C.c_void_p), items)
    assert np.array_equal(ol.digests(got.reshape(items, n)), want["rows"])
    assert np.isneginf(want["first"][0]) and np.isneginf(got[0])


def record_noise_learner_and_transmission():
    cfg, iq, frames, learn, bw = _scene()
    r = ol.OracleChain(cfg).push(iq, frames, T0, PERIOD_MS, dense=("psd_db",))
    return _reference_rows(ol.RefBlocksChain(cfg, _now(0), bw, with_spectrogram=False), r.psd_db, [_now(k) for k in range(frames)])


def test_noise_learner_and_transmission_follow_the_reference_objects_frame_by_frame():
    cfg, iq, frames, learn, bw = _scene()
    r = ol.OracleChain(cfg).push(iq, frames, T0, PERIOD_MS, dense=("psd_db", "noise_sub_db"))
    lists = _assert_follows(ol.recorded("noise_learner_and_transmission"), r)
    n_tx_frames = sum(1 for tx in lists if tx)
    flushes = sum(fl for tx in lists for _, fl in tx)
    # the learning phase had the reference's own length: -100 rows, then real ones
    assert np.all(r.noise_sub_db[learn - 1] == -100.0) and not np.all(r.noise_sub_db[learn] == -100.0)
    assert n_tx_frames > 100 and flushes > 20, (n_tx_frames, flushes)  # the scene really exercises start / flush / stop / time-out


HOP_HALF = 300


def _hop_and_reset_legs():
    """The oracle before and after SdrDevice::setFrequencyRange (sdr_device.cpp:66-77): resetBuffers, new centre -> a fresh noise
    entry is learned. Returns what the reference chain needs to replay it."""
    cfg, iq, frames, learn, bw = _scene(frames=420)
    orc = ol.OracleChain(cfg)
    r1 = orc.push(iq[: HOP_HALF * cfg.fft_size * 2], HOP_HALF, T0, PERIOD_MS, dense=("psd_db", "noise_sub_db"))
    orc.reset()
    new_c = cfg.center_hz + 1_000_000
    centre = (new_c, new_c - cfg.sample_rate_hz // 2, new_c + cfg.sample_rate_hz // 2)
    orc.set_center(*centre)
    rest = frames - HOP_HALF
    t1 = _now(HOP_HALF)
    r2 = orc.push(iq[HOP_HALF * cfg.fft_size * 2 :], rest, t1, PERIOD_MS, dense=("psd_db", "noise_sub_db"))
    return cfg, bw, r1, r2, centre, [t1 + int(np.floor(k * PERIOD_MS + 0.5)) for k in range(rest)]


def record_hop_and_reset():
    cfg, bw, r1, r2, centre, times2 = _hop_and_reset_legs()
    ref = ol.RefBlocksChain(cfg, _now(0), bw, with_spectrogram=False)
    before = _reference_rows(ref, r1.psd_db, [_now(k) for k in range(HOP_HALF)])
    ref.reset()
    ref.set_center(*centre)
    after = _reference_rows(ref, r2.psd_db, times2)
    return {"before_" + k: v for k, v in before.items()} | {"after_" + k: v for k, v in after.items()}


def test_hop_and_reset_follow_the_reference_objects():
    cfg, bw, r1, r2, centre, times2 = _hop_and_reset_legs()
    want = ol.recorded("hop_and_reset")
    before = {k[len("before_"):]: v for k, v in want.items() if k.startswith("before_")}
    after = {k[len("after_"):]: v for k, v in want.items() if k.startswith("after_")}
    assert ol.unpack_lists(before) == [[(f, fl) for f, fl, _, _ in tx] for tx in r1.frame_tx]
    _assert_follows(after, r2, " after the hop")


HOP_SCHEDULE = dict(n=1024, fs=2_048_000, dwell=20, hops=14)  # 20 frames x 25 ms = 500 ms per visit


def _hop_schedule():
    """Scanner hops every 500 ms between two centres; the oracle's result of every visit (reset + retune before each)."""
    n, fs, dwell, hops = (HOP_SCHEDULE[k] for k in ("n", "fs", "dwell", "hops"))
    bw = 16 * fs // n
    cfg = b2s.make_config(n, fs, learn_frames=10_000, noise_learning_ms=NOISE_LEARNING_MS, recording_bandwidth_hz=bw, min_time_ms=200, timeout_ms=300)
    frames = dwell * hops
    tones = synth.standard_scene(n, frames, 0)
    iq = synth.make_iq_int8(n, frames, tones, seed=synth.seed_for(11), quiet_frames=0)
    centres = [cfg.center_hz, cfg.center_hz + 3_000_000]
    orc = ol.OracleChain(cfg)
    visits = []
    for h in range(hops):
        c = centres[h % 2]
        orc.reset()  # SdrDevice::setFrequencyRange: resetBuffers on every retune (sdr_device.cpp:74)
        orc.set_center(c, c - fs // 2, c + fs // 2)
        k0 = h * dwell
        r = orc.push(iq[k0 * 2 * n : (k0 + dwell) * 2 * n], dwell, _now(k0), PERIOD_MS, dense=("psd_db", "noise_sub_db"))
        visits.append((c, k0, r, [_now(k0) + int(np.floor(k * PERIOD_MS + 0.5)) for k in range(dwell)]))
    return cfg, bw, centres, visits


def record_noise_learning_clock():
    cfg, bw, centres, visits = _hop_schedule()
    fs = cfg.sample_rate_hz
    ref = ol.RefBlocksChain(cfg, _now(0), bw, with_spectrogram=False)
    out = {}
    for h, (c, k0, r, times) in enumerate(visits):
        ref.reset()
        ref.set_center(c, c - fs // 2, c + fs // 2)
        out |= {f"{h}_{k}": v for k, v in _reference_rows(ref, r.psd_db, times).items()}
    return out


def test_noise_learning_follows_the_reference_clock_under_a_hop_schedule():
    """Scanner hops every 500 ms (RANGE_SCANNING_TIME) between two centres: the reference's Noise finishes NOISE_LEARNING_TIME after the FIRST
    visit of a centre (noise_learner.cpp:11,23), the time spent on the other centre included — not after 2 s of dwell. The oracle's clock rule
    (noise_learning_ms) must give the same learning frames, rows and transmission lists as the compiled NoiseLearner / Transmission."""
    cfg, bw, centres, visits = _hop_schedule()
    want = ol.recorded("noise_learning_clock")
    learning_frames = {c: 0 for c in centres}
    first_real = {}
    for h, (c, k0, r, _) in enumerate(visits):
        _assert_follows({k: want[f"{h}_{k}"] for k in ("rows", "count", "pairs")}, r, f" of hop {h}")
        for k, q in enumerate(r.noise_sub_db):  # the reference's rows, bit for bit
            if np.all(q == -100.0):
                learning_frames[c] += 1
            else:
                first_real.setdefault(c, k0 + k)
    # centre 0: first frame at 0 ms, visits at 0, 1000, 2000 ms -> the frame stamped 2000 ms (frame 80) is its last learning frame;
    # centre 1: first frame at 500 ms -> the frame stamped 2500 ms (frame 100). 41 learning frames each instead of 81 frames of dwell.
    assert first_real == {centres[0]: 81, centres[1]: 101}, first_real
    assert learning_frames == {centres[0]: 41, centres[1]: 41}, learning_frames


SPECTROGRAM_GEOMETRIES = [(2048, 2_048_000), (8192, 2_048_000)]


def _spectrogram_scene(n, fs):
    cfg, iq, frames, learn, bw = _scene(n=n, fs=fs, frames=260)
    orc = ol.OracleChain(cfg)
    r = orc.push(iq, frames, T0, PERIOD_MS, dense=("psd_db",))
    return cfg, bw, orc, r.psd_db


def record_spectrogram_payloads():
    out = {}
    for n, fs in SPECTROGRAM_GEOMETRIES:
        cfg, bw, _, psd = _spectrogram_scene(n, fs)
        ref = ol.RefBlocksChain(cfg, _now(0), bw, with_spectrogram=True)
        for k in range(len(psd)):
            ref.push_row(psd[k], _now(k))
        pub = [p for t, p in ref.published() if t == "sdr/dev/spectrogram"]
        out[f"{n}_headers"] = np.array([struct.unpack("<QiiiI", p[:24]) for p in pub], np.int64)
        out[f"{n}_payloads"] = ol.digests(pub)
    return out


@pytest.mark.parametrize("n,fs", SPECTROGRAM_GEOMETRIES)
def test_spectrogram_payloads_byte_for_byte(n, fs):
    """Output size = min(16384, getFft(fs, 1000)) = 2048 (spectrogram.cpp:14). n = 2048: decimator factor 1; n = 8192 (the
    reference's own detection FFT at 2.048 MS/s, getFft(fs, 250)): factor 4, mean of adjacent bins (spectrogram.cpp:50-58).
    (N < 2048 is not a valid geometry for the reference at this rate: m_inputSize / m_outputSize would be 0.)"""
    cfg, bw, orc, _ = _spectrogram_scene(n, fs)
    assert cfg.spectrogram_out_size == b2s.get_fft(fs, 1000) == 2048
    want = ol.recorded("spectrogram_payloads")
    headers, payloads = want[f"{n}_headers"], want[f"{n}_payloads"]
    times, centers, rows = orc.get_spectrogram(cap=64)
    assert len(payloads) == len(times) >= 5
    m = cfg.spectrogram_out_size
    # Spectrogram::Container::m_counter is never initialised (spectrogram.cpp:9): the divisor of the FIRST row is whatever the
    # allocator left there. Every later row is well defined; compare those strictly and the first one's header only.
    for i, (t_ms, start, stop, step, size) in enumerate(headers.tolist()):
        assert (t_ms, size) == (int(times[i]), m)
        assert (start, stop, step) == (cfg.center_hz - fs // 2, cfg.center_hz + fs // 2, fs // m)
        if i >= 1:
            msg = b2s.pack_spectrogram_message(int(times[i]), int(centers[i]), fs, rows[i])
            assert msg[24:] == rows[i].tobytes() and ol.digest(msg) == payloads[i], f"spectrogram row {i}"


def _wire_cases():
    rng = np.random.default_rng(11)
    for size in (3, 1000, 16384):
        t_ms, f, fs = int(rng.integers(1, 2**41)), int(rng.integers(10**8, 10**9)), 20_000_000
        row = rng.integers(-128, 128, size).astype(np.int8)
        iq = rng.integers(-128, 128, 2 * size).astype(np.int8)
        yield size, t_ms, f, fs, row, iq


def record_wire_messages():
    R = ol.ref()
    out = {}
    for size, t_ms, f, fs, row, iq in _wire_cases():
        R.ref_published_clear()
        R.ref_push_spectrogram(t_ms, f, fs, row.ctypes.data_as(C.c_void_p), size)
        R.ref_push_transmission(t_ms, f, fs, iq.ctypes.data_as(C.c_void_p), size)
        got = {}
        for i in range(R.ref_published_count()):
            topic = C.create_string_buffer(128)
            buf = np.empty(1 << 16, dtype=np.uint8)
            k = R.ref_published_get(i, topic, 128, buf.ctypes.data_as(C.c_void_p), buf.size)
            got[topic.value.decode()] = buf[:k].tobytes()
        out[f"{size}"] = ol.digests([got["sdr/dev/spectrogram"], got["sdr/dev/transmission/uint8"]])
    return out


def test_wire_messages_against_the_reference_data_controller():
    want = ol.recorded("wire_messages")
    for size, t_ms, f, fs, row, iq in _wire_cases():
        assert ol.digest(b2s.pack_spectrogram_message(t_ms, f, fs, row)) == want[f"{size}"][0], size
        assert ol.digest(b2s.pack_transmission_message(t_ms, f, fs, iq)) == want[f"{size}"][1], size
