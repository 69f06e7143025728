"""Randomised PSD scenes through the REFERENCE'S OWN compiled NoiseLearner -> Transmission objects and through the oracle
(same rows, same injected clock): NoiseLearner rows bit for bit, the FrequencyFlush list of every frame identical. Many
concurrent carriers, drifting and overlapping, near the band edges, ignored ranges, scan-range limits, odd / even group sizes.
What the reference objects returned is read from tests/golden/reference_outputs.npz (record_random_scenes made it)."""
import numpy as np
import pytest

import oracle_lib as ol
from conftest import load_b2s

b2s = load_b2s()

PERIOD_MS = 100.0  # NOISE_LEARNING_TIME = 2000 ms (config.h:24) = 21 frames of this clock
T0 = 1_700_000_000_000


def _scene(seed):
    rng = np.random.default_rng(1000 + seed)
    n = int(rng.choice([256, 512]))
    fs = 2_048_000
    frames = 240
    learn = b2s.lib().b2s_learn_frames_from_ms(2000, PERIOD_MS)
    bw = int(rng.choice([6, 9, 16, 25])) * fs // n
    center = 100_000_000
    kw = {}
    if rng.random() < 0.5:
        lo = center - fs // 2 + int(rng.integers(0, fs - 200_000))
        kw["ignored"] = [(lo, lo + int(rng.integers(20_000, 150_000)))]
    cfg = b2s.make_config(n, fs, center_hz=center, learn_frames=learn, recording_bandwidth_hz=bw, min_time_ms=int(rng.choice([0, 500, 1500])),
                          timeout_ms=int(rng.choice([300, 1000, 2500])), **kw)
    if rng.random() < 0.4:
        cfg.range_lo_hz = center - int(rng.integers(100_000, fs // 2))
        cfg.range_hi_hz = center + int(rng.integers(100_000, fs // 2))
    psd = (-60.0 + 1.5 * rng.standard_normal((frames, n))).astype(np.float32)
    bins = np.arange(n)
    for _ in range(int(rng.integers(3, 9))):
        c = float(rng.integers(0, n))
        a, b = sorted(int(x) for x in rng.integers(learn, frames, 2))
        level, width, drift = float(rng.uniform(12.0, 70.0)), float(rng.uniform(3.0, 14.0)), float(rng.uniform(-0.05, 0.05))
        for t in range(a, b):
            cc = c + drift * (t - a) + 2.0 * np.sin(0.7 * t)
            psd[t] += (level * np.exp(-0.5 * ((bins - cc) / width) ** 2)).astype(np.float32)
            if rng.random() < 0.03:
                psd[t] -= np.float32(level)
    return cfg, psd, frames, bw


SEEDS = range(16)


def record_random_scenes():
    out = {}
    for seed in SEEDS:
        cfg, psd, frames, bw = _scene(seed)
        ref = ol.RefBlocksChain(cfg, T0, bw, with_spectrogram=False)
        rows, lists = [], []
        for k in range(frames):
            q, tx = ref.push_row(psd[k], T0 + int(np.floor(k * PERIOD_MS + 0.5)))
            rows.append(q)
            lists.append(tx)
        out |= {f"{seed}_rows": ol.digests(rows)} | {f"{seed}_{k}": v for k, v in ol.pack_lists(lists).items()}
    return out


@pytest.mark.parametrize("seed", SEEDS)
def test_random_scene_against_the_reference_objects(seed):
    cfg, psd, frames, bw = _scene(seed)
    r = ol.OracleChain(cfg).push(psd, frames, T0, PERIOD_MS, dense=("noise_sub_db",), psd_rows=True)
    want = ol.recorded("random_scenes")
    lists = ol.unpack_lists({"count": want[f"{seed}_count"], "pairs": want[f"{seed}_pairs"]})
    assert len(lists) == frames
    for k, tx in enumerate(lists):
        assert ol.digest(r.noise_sub_db[k]) == want[f"{seed}_rows"][k], f"seed {seed}: NoiseLearner row {k}"
        assert _same_up_to_ties(tx, r.frame_tx[k]), f"seed {seed}: list of frame {k}: reference {tx} oracle {r.frame_tx[k]}"


def _same_up_to_ties(ref_list, oracle_list):
    """getSortedTransmissions orders by power with an UNSTABLE std::sort (transmission.cpp:169): entries of exactly equal power
    may come out in any order (the oracle and the engine define: lower key first). Equal as sequences of equal-power groups.
    The oracle reports at most MAX_TX entries of the (unbounded) reference list: a tie group cut by that cap cannot be compared."""
    capped = len(oracle_list) == ol.MAX_TX
    if (len(ref_list) != len(oracle_list)) if not capped else (len(ref_list) < ol.MAX_TX):
        return False
    i = 0
    while i < len(oracle_list):
        j = i
        while j < len(oracle_list) and oracle_list[j][3] == oracle_list[i][3]:
            j += 1
        if capped and j == len(oracle_list):
            break
        if sorted(ref_list[i:j]) != sorted((f, fl) for f, fl, _, _ in oracle_list[i:j]):
            return False
        i = j
    return True
