"""Recorder DSP chain (SURVEY.md §8(f)#1): rotate -> rational resamplers -> int8, reference sources/radio/recorder.cpp:22-40,58-73.
CPU part: the factor pairs against the reference's gtest vectors and compiled object, the tap design of the engine against the numpy
restatement. GPU part (-m gpu): the chain on the device against oracle/recorder_oracle.py (GNU Radio's resampler is out of tree:
parity unpinned, see the oracle's header), chunked pushes against one push bit for bit."""
import os
import sys

import numpy as np
import pytest

import oracle_lib as ol
from conftest import ROOT, load_b2s
from test_oracle_kats import G

sys.path.insert(0, os.path.join(ROOT, "oracle"))
import recorder_oracle as ro  # noqa: E402

b2s = load_b2s()


def test_resampler_factors_match_the_reference_vectors():
    for fs, bw, thr, expect in G["resamplers"]["cases"]:
        want = [tuple(p) for p in expect]
        assert ro.resamplers_factors(fs, bw, thr) == want, (fs, bw)
        if max(max(p) for p in want) < 100000:
            assert b2s.get_resamplers_factors(fs, bw, thr) == want, (fs, bw)
    assert b2s.get_resamplers_factors(40_000_000, 32_000) == [(1, 25), (1, 50)]  # BASELINE config 4 (SURVEY.md 8d)
    for (fs, bw), want in zip(RESAMPLER_CASES, ol.unpack_lists(ol.recorded("resamplers_factors")), strict=True):
        assert ro.resamplers_factors(fs, bw) == want == b2s.get_resamplers_factors(fs, bw)


RESAMPLER_CASES = ((40_000_000, 32_000), (20_000_000, 32_000), (2_048_000, 32_000), (1_024_000, 20_000), (2_400_000, 12_500))


def record_resamplers_factors():
    """getResamplersFactors of the compiled reference (threshold 125)."""
    import ctypes as C

    buf = np.zeros(32, np.int32)
    lists = []
    for fs, bw in RESAMPLER_CASES:
        k = ol.ref().ref_get_resamplers_factors(fs, bw, 125, buf.ctypes.data_as(C.c_void_p), 16)
        lists.append([(int(buf[2 * i]), int(buf[2 * i + 1])) for i in range(k)])
    return ol.pack_lists(lists)


def test_tap_design_known_properties():
    for interp, decim in ((1, 25), (1, 50), (5, 16), (2, 125)):
        h = ro.design_resampler_taps(interp, decim).astype(np.float64)
        assert len(h) % 2 == 1 and np.allclose(h, h[::-1])  # linear phase
        assert abs(h.sum() - interp) < 1e-4 * interp  # DC gain = interpolation
        w = np.fft.rfft(h, 1 << 16)
        f = np.arange(len(w)) / (1 << 16)  # cycles per sample at the rate I * fs_in
        rate = min(1.0, interp / decim)
        stop = np.abs(w[f >= 1.06 * 0.5 * rate / interp])  # just beyond the new Nyquist frequency (in cycles per sample at I * fs_in)
        assert 20 * np.log10(stop.max() / interp) < -60  # Kaiser beta 7: > 60 dB in the stop band
        assert abs(20 * np.log10(np.abs(w[f <= 0.35 * rate / interp]).min() / interp)) < 0.1  # flat over the fractional bandwidth
    assert len(ro.design_resampler_taps(1, 25)) == 821 and len(ro.design_resampler_taps(1, 50)) == 1641


def _stream(fs, n, tones, seed=1, sigma=6.0):
    rng = np.random.default_rng(seed)
    t = np.arange(n, dtype=np.float64)
    x = sigma * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
    for f_hz, amp in tones:
        x += amp * np.exp(2j * np.pi * (f_hz / fs) * t)
    iq = np.empty(2 * n, np.int8)
    iq[0::2] = np.clip(np.rint(x.real), -128, 127)
    iq[1::2] = np.clip(np.rint(x.imag), -128, 127)
    return iq


@pytest.mark.gpu
@pytest.mark.parametrize("fs,bw,shift,n", [(40_000_000, 32_000, 4_700_000, 1 << 21), (1_024_000, 20_000, -237_500, 1 << 18), (2_048_000, 32_000, 0, 1 << 18)])
def test_recorder_chain_matches_the_oracle(engine, fs, bw, shift, n):
    iq = _stream(fs, n, [(shift + 3_000, 50.0), (shift - 6_500, 20.0), (shift + 4 * bw, 60.0)])  # the third tone is outside the recorded band
    rec = b2s.Recorder(engine, fs, bw, max_samples_per_push=n)
    assert [(i, d) for i, d, _ in rec.stages()] == ro.resamplers_factors(fs, bw)
    for k, (i, d, nt) in enumerate(rec.stages()):
        want = ro.design_resampler_taps(i, d)
        assert nt == len(want) and np.max(np.abs(rec.taps(k) - want)) <= 2e-7 * max(1.0, float(np.max(np.abs(want))))
    rec.start(shift)
    got = rec.push(iq)
    x = (iq[0::2].astype(np.float64) + 1j * iq[1::2].astype(np.float64)) / 127.0
    want = ro.recorder_chain(x, fs, bw, shift)
    assert len(got) == len(want) == 2 * ((n * bw) // fs) or abs(len(got) - len(want)) == 0
    d = np.abs(got.astype(int) - want.astype(int))
    assert d.max() <= 1 and np.mean(d == 0) >= 0.99, (d.max(), np.mean(d == 0))
    assert np.abs(want.astype(int)).max() > 30  # the in-band tones came through; the out-of-band one did not saturate anything
    # chunked pushes (uneven pieces, some shorter than the filters' history) = one push, bit for bit
    rec.start(shift)
    parts, k = [], 0
    for m in [1, 7, 1000, 30_001, 5, 250_000, 17, 99_999] * 50:
        if k >= n:
            break
        m = min(m, n - k)
        parts.append(rec.push(iq[2 * k : 2 * (k + m)]))
        k += m
    assert np.array_equal(np.concatenate(parts), got)
    # float input (what SdrSource delivers) gives the same bytes up to the unpack rounding
    recf = b2s.Recorder(engine, fs, bw, iq_format=b2s.IQ_CF32, max_samples_per_push=n)
    recf.start(shift)
    gf = recf.push((iq.astype(np.float32) * np.float32(1 / 127.0)).astype(np.float32))
    assert np.max(np.abs(gf.astype(int) - got.astype(int))) <= 1


@pytest.mark.gpu
def test_recorder_messages_through_the_wire_format(engine):
    """Recorder::flush publishes chunks of roundUp(bandwidth * 100 ms, 4096) samples as sdr/<dev>/transmission/uint8 (recorder.cpp:35,
    data_controller.cpp:27-42): the chain's int8 output packs into exactly the bytes the reference's DataController would send."""
    fs, bw, shift, n = 2_048_000, 32_000, 250_000, 1 << 20
    iq = _stream(fs, n, [(shift + 1_000, 60.0)])
    rec = b2s.Recorder(engine, fs, bw, max_samples_per_push=n)
    rec.start(shift)
    out = rec.push(iq)
    chunk = -(-(bw * 100 // 1000) // 4096) * 4096  # roundUp(bandwidth * RECORDER_FLUSH_INTERVAL / 1000, 4096)
    assert chunk == 4096 and len(out) // 2 >= 2 * chunk
    msg = b2s.pack_transmission_message(1_700_000_000_123, 145_000_000 + shift, bw, out[: 2 * chunk])
    assert len(msg) == 20 + 2 * chunk and np.array_equal(np.frombuffer(msg[20:], np.uint8), out[: 2 * chunk].view(np.uint8) ^ 0x80)
    if ol.have_ref() and hasattr(ol.ref(), "ref_push_transmission"):
        import ctypes as C

        R = ol.ref()
        R.ref_published_clear()
        R.ref_push_transmission(1_700_000_000_123, 145_000_000 + shift, bw, out[: 2 * chunk].ctypes.data_as(C.c_void_p), chunk)
        topic = C.create_string_buffer(128)
        buf = np.empty(1 << 16, dtype=np.uint8)
        k = R.ref_published_get(0, topic, 128, buf.ctypes.data_as(C.c_void_p), buf.size)
        assert topic.value.decode() == "sdr/dev/transmission/uint8" and buf[:k].tobytes() == msg
