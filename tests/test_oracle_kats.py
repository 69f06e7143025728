"""Pins the CPU oracle (oracle/scan_oracle.cpp):
  (1) against the reference's own gtest known-answer vectors (tests/golden/reference_kats.json), and
  (2) against what the reference's own compiled objects returned for random inputs (stored in tests/golden/reference_outputs.npz),
      bit for bit — for every hot-path piece that the reference can be built for (SURVEY.md §8c).
CPU only (-m "not gpu")."""
import ctypes as C
import json
import os

import numpy as np
import pytest

import oracle_lib as ol
from conftest import ROOT

G = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_kats.json")))
needs_ref = pytest.mark.skipif(not ol.have_ref(), reason="oracle/_ref/libref.so not built (needs the reference sources)")
KINDS = ["orc"] + (["ref"] if ol.have_ref() else [])


def _lib(kind):
    return ol.oracle() if kind == "orc" else ol.ref()


@pytest.mark.parametrize("kind", KINDS)
def test_average_kat(kind):
    g = G["average"]
    out = ol.cpu_average(np.array(g["input"], np.float32), g["group"], kind)
    np.testing.assert_allclose(out, np.array(g["expect"], np.float32), rtol=4e-7)  # EXPECT_FLOAT_EQ = 4 ulp


@pytest.mark.parametrize("kind", KINDS)
def test_contains_with_margin_kat(kind):
    g = G["contains_with_margin"]
    keys = np.array(g["keys"], np.int32)
    for index, margin, expect in g["cases"]:
        found = C.c_int()
        got = getattr(_lib(kind), f"{kind}_contains_with_margin")(keys.ctypes.data_as(C.c_void_p), len(keys), index, margin, C.byref(found))
        assert bool(got) == expect, (index, margin)


@pytest.mark.parametrize("kind", KINDS)
def test_most_frequent_value_kat(kind):
    for data, expect in G["most_frequent_value"]["cases"]:
        v = np.array(data, np.int32)
        assert getattr(_lib(kind), f"{kind}_most_frequent_value")(v.ctypes.data_as(C.c_void_p), len(v)) == expect


@pytest.mark.parametrize("kind", KINDS)
def test_get_max_index_kat(kind):
    g = G["get_max_index"]
    d = np.array(g["data"], np.float32)
    for index, group, expect in g["cases"]:
        assert getattr(_lib(kind), f"{kind}_get_max_index")(d.ctypes.data_as(C.c_void_p), len(d), index, group) == expect


@pytest.mark.parametrize("kind", KINDS)
def test_get_fft_and_tuned_kat(kind):
    L = _lib(kind)
    for fs, step, expect in G["get_fft"]["cases"]:
        assert getattr(L, f"{kind}_get_fft")(fs, step) == expect
    for f, step, expect in G["get_tuned_frequency"]["cases"]:
        assert getattr(L, f"{kind}_get_tuned_frequency")(f, step) == expect


def _run_averager_script(av):
    g = G["averager"]
    size, group = g["size"], g["group"]
    for st in g["steps"]:
        if st["op"] == "push":
            av.push(np.full(size, st["v"], np.float32))
        elif st["op"] == "reset":
            av.reset()
        assert np.array_equal(av.average(), np.full(size, st["avg"], np.float32)), st
        assert np.array_equal(av.data(), np.array([[r] * size for r in st["rows"]], np.float32)), st


@pytest.mark.parametrize("kind", KINDS)
def test_averager_kat(kind):
    g = G["averager"]
    _run_averager_script(ol.CpuAverager(g["size"], g["group"], kind))


def _fixture_mean(raw, group):
    s = np.zeros(raw[0].shape, np.float32)
    for r in raw:  # same accumulation order as AveragerTest::average(), tests/test_averager.cpp:29-40
        s = (s + r).astype(np.float32)
    return (s / np.float32(group)).astype(np.float32)


def run_averager_fixture(av, size, group, rows_iter):
    """AveragerTest fixture (tests/test_averager.cpp:13-44): exact equality of average() and data() after every add."""
    raw = [np.zeros(size, np.float32) for _ in range(group)]
    pushed = 0
    for row in rows_iter:
        row = np.asarray(row, np.float32)
        av.push(row)
        raw.append(row)
        raw = raw[-group:]
        pushed += 1
        if pushed < group:
            assert np.array_equal(av.average(), np.full(size, -100, np.float32))
        else:
            assert np.array_equal(av.average(), _fixture_mean(raw, group))
        assert np.array_equal(av.data(), np.stack(raw))


@pytest.mark.parametrize("kind", KINDS)
def test_averager_fixture_kat(kind):
    g = G["averager_fixture"]
    size, group = g["size"], g["group"]
    run_averager_fixture(ol.CpuAverager(size, group, kind), size, group, g["simple"])
    rows = list(g["big"]["prefix"]) + [[i * 11 + j * 7 for j in range(size)] for i in range(*g["big"]["ramp_i"])]
    run_averager_fixture(ol.CpuAverager(size, group, kind), size, group, rows)


# ---------------- oracle == compiled reference, bit for bit, on random data ----------------
# The reference's outputs are read from tests/golden/reference_outputs.npz (oracle_lib.recorded); record_<name>() made them from
# the compiled reference on the same inputs.
AVERAGER_SHAPES = [(5, 3), (64, 21), (1000, 21), (4096, 21), (33, 1)]
AVERAGE_SHAPES = [(9, 5), (100, 21), (4096, 21), (16384, 21), (50, 1), (10, 21), (7, 4)]


def _averager_steps(av, size, group):
    """Pushes the random rows of the test; yields (average, data) after every push."""
    rng = np.random.default_rng(size * 131 + group)
    for step in range(3 * group + 7):
        if step == 2 * group + 1:
            av.reset()
        av.push((rng.standard_normal(size) * 30 - 20).astype(np.float32))
        yield av.average(), av.data()


def record_averager_bitwise():
    out = {}
    for size, group in AVERAGER_SHAPES:
        steps = list(_averager_steps(ol.CpuAverager(size, group, "ref"), size, group))
        out[f"avg_{size}_{group}"] = ol.digests(a for a, _ in steps)
        out[f"data_{size}_{group}"] = ol.digests(d for _, d in steps)
    return out


@pytest.mark.parametrize("size,group", AVERAGER_SHAPES)
def test_averager_matches_reference_bitwise(size, group):
    want = ol.recorded("averager_bitwise")
    assert len(want[f"avg_{size}_{group}"]) == 3 * group + 7
    for step, (avg, data) in enumerate(_averager_steps(ol.CpuAverager(size, group, "orc"), size, group)):
        assert ol.digest(avg) == want[f"avg_{size}_{group}"][step], step
        assert ol.digest(data) == want[f"data_{size}_{group}"][step], step


def _average_inputs(size, group):
    rng = np.random.default_rng(size + group)
    for scale in (1.0, 40.0):
        yield (rng.standard_normal(size) * scale - 7).astype(np.float32)
    yield np.full(size, -100, np.float32)


def record_average_bitwise():
    return {f"{size}_{group}": ol.digests(ol.cpu_average(x, group, "ref") for x in _average_inputs(size, group)) for size, group in AVERAGE_SHAPES}


@pytest.mark.parametrize("size,group", AVERAGE_SHAPES)
def test_average_matches_reference_bitwise(size, group):
    want = ol.recorded("average_bitwise")[f"{size}_{group}"]
    got = ol.digests(ol.cpu_average(x, group, "orc") for x in _average_inputs(size, group))
    assert np.array_equal(got, want)


def _collection_cases():
    rng = np.random.default_rng(7)
    for _ in range(300):
        n = int(rng.integers(1, 200))
        d = rng.integers(-5, 6, n).astype(np.float32)  # many ties: first-maximum rule matters
        idx, grp = int(rng.integers(0, n)), int(rng.integers(0, 64))
        v = rng.integers(0, 8, int(rng.integers(1, 30))).astype(np.int32)
        keys = np.unique(rng.integers(0, 500, int(rng.integers(0, 12)))).astype(np.int32)
        index, margin = int(rng.integers(-10, 510)), int(rng.integers(0, 140))
        yield d, idx, grp, v, keys, index, margin


def _collection_results(kind):
    """[max index, most frequent value, contains, found key (-1 when not contained)] per case."""
    L = _lib(kind)
    out = []
    for d, idx, grp, v, keys, index, margin in _collection_cases():
        found = C.c_int(-1)
        contains = getattr(L, f"{kind}_contains_with_margin")(keys.ctypes.data_as(C.c_void_p), len(keys), index, margin, C.byref(found))
        out.append((getattr(L, f"{kind}_get_max_index")(d.ctypes.data_as(C.c_void_p), len(d), idx, grp),
                    getattr(L, f"{kind}_most_frequent_value")(v.ctypes.data_as(C.c_void_p), len(v)), contains, found.value if contains else -1))
    return np.array(out, np.int64)


def record_collection_utils():
    return {"results": _collection_results("ref")}


def test_collection_utils_match_reference_random():
    got, want = _collection_results("orc"), ol.recorded("collection_utils")["results"]
    assert got.shape == want.shape
    for i in range(len(want)):
        assert tuple(got[i]) == tuple(want[i]), i


def _tuned_cases():
    rng = np.random.default_rng(11)
    return [(int(rng.integers(-2_000_000, 2_000_000)), int(rng.integers(1, 100_000))) for _ in range(2000)]


FFT_CASES = [(fs, step) for fs in (250_000, 1_024_000, 2_048_000, 2_400_000, 10_000_000, 20_000_000, 40_000_000, 61_440_000) for step in (100, 250, 625, 1000)]


def _radio_results(kind):
    L = _lib(kind)
    return {"tuned": np.array([getattr(L, f"{kind}_get_tuned_frequency")(f, step) for f, step in _tuned_cases()], np.int64),
            "fft": np.array([getattr(L, f"{kind}_get_fft")(fs, step) for fs, step in FFT_CASES], np.int64)}


def record_radio_utils():
    return _radio_results("ref")


def test_radio_utils_match_reference_random():
    got, want = _radio_results("orc"), ol.recorded("radio_utils")
    assert np.array_equal(got["tuned"], want["tuned"])
    assert np.array_equal(got["fft"], want["fft"])


@needs_ref
def test_reference_only_kats():
    """Vectors for reference helpers that sit beside the hot path (range splitting, resampler factors)."""
    R = ol.ref()
    for fs, expect in G["range_split_sample_rate"]["cases"]:
        assert R.ref_get_range_split_sample_rate(fs) == expect
    buf = np.zeros(64, np.int32)
    for lo, hi, fs, expect in G["split_range"]["cases"]:
        n = R.ref_split_range(lo, hi, fs, buf.ctypes.data_as(C.c_void_p), 32)
        assert buf[: 2 * n].reshape(-1, 2).tolist() == expect
    for fs, bw, thr, expect in G["resamplers"]["cases"]:
        n = R.ref_get_resamplers_factors(fs, bw, thr, buf.ctypes.data_as(C.c_void_p), 32)
        assert buf[: 2 * n].reshape(-1, 2).tolist() == expect
    for v, f, e in G["round"]["up"]:
        assert R.ref_round_up(v, f) == e
    for v, f, e in G["round"]["down"]:
        assert R.ref_round_down(v, f) == e
