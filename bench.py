#!/usr/bin/env python
"""bench.py — IQ MSamples/s through the fused unpack+FFT+power+detect path (BASELINE.json metric).

Default workload (`--config 2`, BASELINE.json configs[1], SURVEY.md §8d "Config 2"): ONE 20 MS/s band, N = 16384-point FFT,
r = 1, T = 4096 frames per step = 67.1 M complex samples = 134 MB of int8 IQ (> the 126 MB L2, so every step streams its input
from HBM; no L2 flush is needed). A step is one b2s_band_push of T frames per band: K1 (unpack, window, FFT, dB), K2 (noise,
Averager, boxcar, threshold, spectrogram), the ordering of the detection entries and K4 (the signal map, on the device).
The bands run in their asynchronous result mode (B2S_FLAG_ASYNC); the timed region ends with b2s_band_sync on every band,
i.e. after ALL work of all K steps.

Other workloads (SURVEY.md §8d), selected with --config:
  1  single 2.048 MS/s band, N = 4096 (the reference's CPU-runnable case; here also through the GPU path), T = 4096
  3  8-band hop set, N = 8192, fs = 2.048 MS/s each, one stream per band, T = 1024 frames per band per step; with --hop the bands
     are retuned like Scanner does: b2s_band_reset (Transmission::resetBuffers) every 125 frames
  4  40 MS/s wideband, N = 32768, four keyed FM carriers, T = 2048 (detect part)
  5  8 bands per GPU (64 on 8 GPUs), N = 32768, fs = 20 MS/s; --frames T sweeps T in {64, 256, 1024, 4096}; --sweep runs all four

  value : steady-state throughput with the IQ already resident in HBM (B2S_FLAG_IQ_ON_DEVICE), CUDA-event timed.
  e2e   : the same call with the IQ in pinned HOST memory: the host->device copy of every step's input and the
          device->host read of its results are inside the timed region.
  roofline : dominant kernel (K1 k_spectrum3): algorithmic bytes 6 B/sample (2 B int8 IQ read + 4 B fp32 dB row written,
          SURVEY.md §8d) x samples per launch / that kernel's mean launch time (CUDA events inside the library, on the
          launching stream) vs. the measured HBM copy bandwidth in MEASURED_PEAKS.json.
  cpu_baseline : the CPU oracle port (fp32, oracle/liboracle.so; FFTW3f through dlopen when the box has it) on a bounded
          sample of the same workload, all host cores and one thread.
N > 1 GPUs (torchrun): one process per GPU, the workload's bands replicated per GPU, no data-path collective ("weak" scaling);
the time is the max over ranks (device-timed), value = N x samples / that.

`--impl reference` times the reference's CPU path instead (the oracle port; the reference's own GNU Radio/FFTW chain
cannot be built in this image — see DESIGN.md), with all host threads, on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

LEARN = 100
ALG_BYTES_PER_SAMPLE = 6.0
K2_ALG_BYTES_PER_SAMPLE = 4.0  # k_detect reads every fp32 dB row once (its outputs are sparse)
METRIC = "IQ MSamples/s through FFT+power+detect"
# dram__bytes_read.sum + dram__bytes_write.sum of ONE K1 launch of the config-2 workload from the committed `ncu --set full` capture
K1_TRAFFIC = {"bytes": None, "source": None}
_TRAFFIC_FILE = os.path.join(ROOT, "profiles", "k1_traffic.json")
if os.path.exists(_TRAFFIC_FILE):
    try:
        K1_TRAFFIC = json.load(open(_TRAFFIC_FILE))
    except Exception:
        pass

HOP_CENTRES_MHZ = [108.0, 118.0, 137.5, 144.8, 156.8, 162.4, 433.9, 440.0]  # 108/144/440-style set (reference README.md:5)

WORKLOADS = {
    1: dict(name="configs[0]: single 2.048 MS/s band, 4096-pt FFT (through the GPU path)", n=4096, fs=2_048_000, frames=4096, bands=1),
    2: dict(name="configs[1]: single 20 MS/s band, 16384-pt FFT, fused unpack+FFT+power+detect", n=16384, fs=20_000_000, frames=4096, bands=1),
    3: dict(name="configs[2]: 8-band hop set, 8192-pt FFT, per-band CUDA streams", n=8192, fs=2_048_000, frames=1024, bands=8),
    4: dict(name="configs[3]: 40 MS/s wideband, 32768-pt FFT, 4 keyed transmissions (detect part)", n=32768, fs=40_000_000, frames=2048, bands=1),
    5: dict(name="configs[4]: 8 bands per GPU (64 on 8 GPUs), 32768-pt FFT, 20 MS/s", n=32768, fs=20_000_000, frames=1024, bands=8),
}


def bench_tones(synth, n_fft, frames, learn):
    """Four keyed NFM-like carriers (SURVEY.md §8d generator): starts, stops and time-outs all occur inside a step."""
    span = frames - learn
    a = learn
    return [
        synth.Tone(0.31 * n_fft / 2 + 0.1, amplitude=40.0, fm_dev_bins=5.0, on_frames=[(a + int(0.05 * span), a + int(0.60 * span))]),
        synth.Tone(-0.62 * n_fft / 2 + 0.1, amplitude=40.0, fm_dev_bins=5.0, on_frames=[(a + int(0.20 * span), a + int(0.35 * span)), (a + int(0.55 * span), a + int(0.90 * span))]),
        synth.Tone(0.055 * n_fft / 2 + 0.1, amplitude=40.0, fm_dev_bins=5.0, on_frames=[(a + int(0.10 * span), a + int(0.45 * span))], phase=1.0),
        synth.Tone(-0.17 * n_fft / 2 + 0.1, amplitude=40.0, fm_dev_bins=5.0, on_frames=[(a + int(0.40 * span), a + int(0.95 * span))], phase=2.0),
    ]


def wideband_tones(synth, n_fft, fs, frames, learn):
    """Config 4 (SURVEY.md §8d): carriers at -12.5, -3.2, +4.7, +15.1 MHz, 12.5 kHz deviation, keyed on/off in staggered thirds."""
    span = frames - learn
    out = []
    for i, mhz in enumerate((-12.5, -3.2, 4.7, 15.1)):
        off = mhz * 1e6 / (fs / n_fft)
        a = learn + int((0.05 + 0.12 * i) * span)
        out.append(synth.Tone(round(off) + 0.1, amplitude=40.0, fm_dev_bins=12_500 / (fs / n_fft), on_frames=[(a, a + int(0.3 * span)), (a + int(0.55 * span), a + int(0.75 * span))], phase=float(i)))
    return out


def bands_for_rank(n_bands: int, rank: int, world: int):
    """SURVEY.md §8e partitioning: band b lives on GPU b mod G; frames of a band never leave their GPU."""
    return [b for b in range(n_bands) if b % world == rank]


def reduce_step_time(ms_local: float, device=None) -> float:
    """Max over ranks of the device-timed region (the slowest rank defines the step); identity for one rank."""
    import torch
    import torch.distributed as dist

    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return float(ms_local)
    t = torch.tensor([ms_local], dtype=torch.float64, device=device if device is not None else "cpu")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def aggregate_msps(samples_per_rank_step: int, steps: int, world: int, ms_max: float) -> float:
    """Whole-job throughput: all ranks' samples over the slowest rank's time."""
    return world * samples_per_rank_step * steps / (ms_max / 1000.0) / 1e6


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def cpu_sample(b2s, synth, ol, wl, iq_segment_fn, threads: int, budget_s: float, per_thread: int):
    """The oracle port (fp32 FFT) on `threads` host threads, one chain per thread, `per_thread` frames each; repeated until ~budget_s."""
    import numpy as np

    n, fs = wl["n"], wl["fs"]
    cfg = b2s.make_config(n, fs, learn_frames=LEARN)
    period = synth.frame_period_ms(n, fs)
    seg = iq_segment_fn(per_thread)
    iq = np.tile(seg, threads)
    frames = per_thread * threads
    L = ol.oracle()
    L.orc_bench_run.restype = C.c_double
    L.orc_bench_run(C.byref(cfg), iq.ctypes.data_as(C.c_void_p), frames, period, threads)  # warm-up
    runs = []
    t_all = 0.0
    while t_all < budget_s and len(runs) < 20:
        dt = L.orc_bench_run(C.byref(cfg), iq.ctypes.data_as(C.c_void_p), frames, period, threads)
        runs.append(frames * n / dt / 1e6)
        t_all += dt
    stages = (C.c_double * 3)()
    L.orc_bench_stage_seconds(stages)
    tot = sum(stages) or 1.0
    runs.sort()
    return {"value": runs[len(runs) // 2], "min": runs[0], "max": runs[-1], "reps": len(runs), "frames": frames,
            "stage_split": {"unpack_window_fft": stages[0] / tot, "psd_db": stages[1] / tot, "noise_averager_detect": stages[2] / tot}}


def bind_to_gpu_numa(index: int):
    """Run this process (and the threads the library starts) on the CPU cores of the NUMA node the GPU hangs off, BEFORE any pinned
    buffer is allocated (first touch puts the pages there): at 8 GPUs the e2e leg otherwise crosses the socket link for half the
    GPUs (round 1: 37.5 instead of 52 GB/s per GPU). Returns what was done, for the JSON line."""
    try:
        out = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=pci.bus_id", "--format=csv,noheader"], capture_output=True, text=True, timeout=20).stdout.strip()
        bus = out.lower()
        if bus.startswith("00000000:"):
            bus = bus[4:]  # sysfs uses a 4-digit domain
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read().strip())
        if node < 0:
            return {"numa_node": None, "note": "the platform reports no NUMA node for the GPU"}
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus += list(range(int(a), int(b or a) + 1))
        allowed = sorted(set(cpus) & os.sched_getaffinity(0))
        if allowed:
            os.sched_setaffinity(0, allowed)
        return {"numa_node": node, "cpus": len(allowed)}
    except Exception as e:  # not fatal: the measurement just runs unbound
        return {"numa_node": None, "note": f"not bound: {type(e).__name__}"}


def fft_backend(ol):
    try:
        L = ol.oracle()
        L.orc_fft_backend.restype = C.c_char_p
        return L.orc_fft_backend().decode()
    except Exception:
        return "in-repo fp32 radix-4 Stockham (FFTW unavailable)"


def band_outputs(bands, counts, t_last_ms):
    """What a caller of the timed path holds after its last step, per band: the counts of the last push's result, the complete
    transmission mailbox, the live signal map, the spectrogram rows completed during that step, and the Averager output and noise
    threshold the detector compared against. Integers and times as float64, dB values as float32."""
    import numpy as np

    out = []
    for band, c in zip(bands, counts):
        tx = band.get_transmissions()
        keys, first, last, power = band.get_signals(cap=4096)
        times = [np.zeros(0, np.int64)]
        rows = [np.zeros((0, max(band.cfg.spectrogram_out_size, 1)), np.int8)]
        while True:  # consume the band's row list; rows stamped before the last step belong to earlier steps
            t, _, r = band.get_spectrogram(cap=256)
            if len(t) == 0:
                break
            keep = t >= int(t_last_ms)
            times.append(t[keep])
            rows.append(r[keep])
        _, avg, _, _ = band.get_averager()
        thr, _, _ = band.get_noise()
        out.append({
            "result_counts": np.array(c, np.float64),  # n_transmissions, n_detect_entries, n_spectrogram_rows, n_transmissions_total
            "transmissions": np.array(tx, np.float64).reshape(-1, 4),  # shift_hz, flush, key, power
            "signals": np.stack([keys, first, last, power], axis=1).astype(np.float64),  # key, first_ms, last_ms, power
            "spectrogram_times_ms": np.concatenate(times).astype(np.float64),
            "spectrogram_rows": np.concatenate(rows).astype(np.float32),
            "averager_db": avg,
            "noise_threshold_db": thr,
        })
    return out


DUMP_BUDGET_BYTES = 64 << 20


def dump_outputs(directory, per_band):
    """DIR/band<b>_<name>.npy for every band; above DUMP_BUDGET_BYTES in all, a fixed seeded sample of whole bands is written."""
    import numpy as np

    sizes = [sum(a.nbytes for a in d.values()) for d in per_band]
    keep = list(range(len(per_band)))
    if sum(sizes) > DUMP_BUDGET_BYTES:
        keep, total = [], 0
        for b in np.random.default_rng(0).permutation(len(per_band)):
            if total + sizes[b] <= DUMP_BUDGET_BYTES:
                keep.append(int(b))
                total += sizes[b]
        keep.sort()
    os.makedirs(directory, exist_ok=True)
    for b in keep:
        for name, a in per_band[b].items():
            np.save(os.path.join(directory, f"band{b}_{name}.npy"), a)


def run_reference(args, rank, world):
    """Reference arm: the CPU restatement of the reference path (oracle port, fp32), all host threads."""
    if rank != 0:
        return
    import numpy as np
    import __graft_entry__ as ge
    import oracle_lib as ol

    b2s, synth = ge.load_b2s(), ge.load_synth()
    wl = WORKLOADS[args.config]
    n, fs = wl["n"], wl["fs"]
    cores = len(os.sched_getaffinity(0))
    per_thread = max(64, min(512, (1 << 23) // n))

    def segment(frames, learn=LEARN):
        return synth.make_iq_int8(n, frames, bench_tones(synth, n, frames, learn), seed=synth.seed_for(args.config), quiet_frames=learn)

    # one step = one bounded sample (cores x per_thread frames); K steps after W warm-ups, as the contract asks
    cfg = b2s.make_config(n, fs, learn_frames=LEARN)
    period = synth.frame_period_ms(n, fs)
    L = ol.oracle()
    L.orc_bench_run.restype = C.c_double
    # size the per-step sample so that the K timed steps end within about a minute (a probe step tells the box's speed); the share of
    # (cheap) learning frames per chain stays what it is at full size: LEARN of 512
    full = per_thread
    probe = np.tile(segment(per_thread), cores)
    t_probe = L.orc_bench_run(C.byref(cfg), probe.ctypes.data_as(C.c_void_p), per_thread * cores, period, cores)
    if t_probe * args.steps > 60.0:
        per_thread = max(64, int(per_thread * 60.0 / (t_probe * args.steps)))
    if per_thread != full:
        learn = max(8, per_thread * LEARN // full)
        cfg = b2s.make_config(n, fs, learn_frames=learn)
        iq = np.tile(segment(per_thread, learn), cores)
    else:
        iq = probe
    frames = per_thread * cores
    times = []
    for i in range(args.warmup + args.steps):
        dt = L.orc_bench_run(C.byref(cfg), iq.ctypes.data_as(C.c_void_p), frames, period, cores)
        if i >= args.warmup:
            times.append(dt)
    total = sum(times)
    value = frames * n * args.steps / total / 1e6
    per_step = sorted(frames * n / t / 1e6 for t in times)
    single = cpu_sample(b2s, synth, ol, wl, segment, 1, 3.0, per_thread)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "MS/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1000.0 * total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl["name"] + " (CPU arm: bounded sample)", "fft_size": n, "sample_rate_hz": fs, "frames_per_step": frames, "l2": "n/a (CPU)"},
        "cpu_baseline": {"value": value, "unit": "MS/s", "cores": cores, "kind": "port", "fft": fft_backend(ol),
                         "spread": {"min": per_step[0], "median": per_step[len(per_step) // 2], "max": per_step[-1]},
                         "single_thread": single["value"], "stage_split_single_thread": single["stage_split"],
                         "sample": f"{frames} frames ({cores} threads x {per_thread} frames, one chain per thread) of the workload per step; restated CPU path, fp32 FFT"},
        "e2e": {"value": value, "unit": "MS/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)  # 100 x 0.44 ms: a 44 ms timed region (20 steps were 9 ms: credible but fragile)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b2s", choices=["b2s", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(WORKLOADS))
    ap.add_argument("--frames", type=int, default=0, help="frames per band per step (default = the workload's)")
    ap.add_argument("--bands", type=int, default=0, help="bands per GPU (default = the workload's)")
    ap.add_argument("--hop", action="store_true", help="config 3 hop variant: b2s_band_reset every 125 frames")
    ap.add_argument("--sweep", action="store_true", help="config 5: run T in {64, 256, 1024, 4096} and report all four")
    ap.add_argument("--skip-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the bands returned for the last timed step of the device-resident run as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "b2s" else max(args.warmup, 1)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import numpy as np
    import torch
    import torch.distributed as dist

    import __graft_entry__ as ge

    b2s, synth = ge.load_b2s(), ge.load_synth()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the hot path has no CPU fallback")
    all_cpus = os.sched_getaffinity(0)
    numa = bind_to_gpu_numa(local_rank)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    wl = dict(WORKLOADS[args.config])
    if args.frames:
        wl["frames"] = args.frames
    if args.bands:
        wl["bands"] = args.bands
    n, fs, n_bands = wl["n"], wl["fs"], wl["bands"]
    period = synth.frame_period_ms(n, fs)
    eng = b2s.Engine(local_rank)
    main_stream = torch.cuda.current_stream(dev)

    def tones_for(T):
        return wideband_tones(synth, n, fs, T, LEARN) if args.config == 4 else bench_tones(synth, n, T, LEARN)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def centre(b):
        if args.config == 3:
            return int(HOP_CENTRES_MHZ[b % 8] * 1e6)
        return 150_000_000 + 1_000_000 * (rank * n_bands + b)

    def run(T, steps, warmup, on_device, hop=False, capture=False):
        """One measurement: n_bands bands, `steps` timed steps of T frames per band. Returns (ms max over ranks, summed profile, clocks, stats);
        with `capture`, stats["outputs"] holds what every band returned for the last timed step (see band_outputs)."""
        iq_dev = [synth.make_iq_int8_torch(n, T, tones_for(T), seed=synth.seed_for(args.config, rank * n_bands + b), quiet_frames=LEARN, device=dev) for b in range(n_bands)]
        hosts = None
        if not on_device:
            hosts = []
            for x in iq_dev:
                h = torch.empty(x.numel(), dtype=torch.int8, pin_memory=True)
                h.copy_(x)
                hosts.append(h)
        torch.cuda.synchronize()
        flags = b2s.FLAG_ASYNC | (b2s.FLAG_IQ_ON_DEVICE if on_device else 0)
        bands, streams = [], []
        for b in range(n_bands):
            cfg = b2s.make_config(n, fs, center_hz=centre(b), learn_frames=LEARN, max_frames_per_push=T, flags=flags)
            band = b2s.Band(eng, cfg)
            st = main_stream if n_bands == 1 else torch.cuda.Stream(dev)
            band.set_stream(st.cuda_stream)
            band.set_profiling(True)
            bands.append(band)
            streams.append(st)
        ptrs = [(x.data_ptr() if on_device else h.data_ptr()) for x, h in zip(iq_dev, hosts or iq_dev)]
        piece = 125 if hop else T  # Scanner dwell: 500 ms at 250 frames/s (scanner.cpp:46-60), then resetBuffers (sdr_device.cpp:74)
        res = b2s.Result()
        t_ms = 0.0

        def step():
            nonlocal t_ms
            for k0 in range(0, T, piece):
                m = min(piece, T - k0)
                for band, p in zip(bands, ptrs):
                    band.push_raw(p + k0 * 2 * n, m, int(t_ms + k0 * period), period)
                if hop:
                    for band in bands:
                        band.reset()
            t_ms += T * period

        for _ in range(warmup):
            step()
        for band in bands:
            band.sync(res)
            band.get_profile(reset=True)
        sampler = ClockSampler(local_rank)
        barrier()
        sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(main_stream)
        for _ in range(steps):
            step()
        n_tx, n_ent = 0, 0
        counts = []
        for band in bands:  # async result mode: every push's kernels AND bookkeeping are complete before the clock stops
            band.sync(res)
            n_tx += res.n_transmissions_total
            n_ent += res.n_detect_entries
            counts.append((res.n_transmissions, res.n_detect_entries, res.n_spectrogram_rows, res.n_transmissions_total))
        e1.record(main_stream)
        barrier()
        clocks = sampler.stop()
        ms = e0.elapsed_time(e1)
        # before the untimed profiling pushes below change the bands' state
        outputs = band_outputs(bands, counts, t_ms - T * period) if capture else None
        profs = [band.get_profile(reset=True) for band in bands]
        cta = None
        if on_device and n_bands == 1:
            # K2's per-CTA balance: three extra untimed pushes with profiling level 2 (one small device->host copy per push)
            bands[0].set_profiling(2)
            for i in range(3):
                bands[0].push_raw(ptrs[0], T, int(t_ms), period)
                t_ms += T * period
            bands[0].sync(res)
            pb = bands[0].get_profile(reset=True)
            cta = (pb.detect_cta_median_ms / max(pb.detect_launches, 1), pb.detect_cta_max_ms / max(pb.detect_launches, 1))
        for band in bands:
            band.close()
        del iq_dev, hosts
        agg = {k: sum(getattr(p, k) for p in profs) for k in ("spectral_ms", "detect_ms", "window_ms", "tracker_host_ms", "track_ms", "spectral_launches", "detect_launches",
                                                              "window_launches", "track_launches", "track_evals", "track_events", "track_best_index", "pushes", "h2d_bytes", "d2h_bytes")}
        return reduce_step_time(ms, dev), agg, clocks, {"n_tx": n_tx, "n_entries": n_ent, "cta": cta, "outputs": outputs}

    peak, peak_src = measured_peaks()

    def summarise(T, steps, ms, agg, hop=False):
        samples_step = n_bands * T * n
        k1_ms = agg["spectral_ms"] / max(agg["spectral_launches"], 1)
        k2_ms = agg["detect_ms"] / max(agg["detect_launches"], 1)
        per_launch = (125 if hop else T) * n  # samples one K1 / K2 launch processes
        return {
            "frames_per_step": T, "value": aggregate_msps(samples_step, steps, world, ms), "ms_per_step": ms / steps,
            "k1_ms": k1_ms, "k2_ms": k2_ms, "k4_ms": agg["track_ms"] / max(agg["track_launches"], 1),
            "k1_frac": ALG_BYTES_PER_SAMPLE * per_launch / (k1_ms / 1000.0) / 1e9 / peak,
            "k2_frac": K2_ALG_BYTES_PER_SAMPLE * per_launch / (k2_ms / 1000.0) / 1e9 / peak,
            # whole path: algorithmic bytes of the step over the step time (the kernels of different bands overlap)
            "path_frac": ALG_BYTES_PER_SAMPLE * samples_step / (ms / steps / 1000.0) / 1e9 / peak,
        }

    T = wl["frames"]
    # ---- device-resident run (value + roofline) ----
    ms, agg, clocks, stats = run(T, args.steps, args.warmup, True, hop=args.hop, capture=bool(args.dump_outputs))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, stats["outputs"])
    head = summarise(T, args.steps, ms, agg, hop=args.hop)
    samples_step = n_bands * T * n
    k1_ms, k2_ms = head["k1_ms"], head["k2_ms"]
    launch_samples = (125 if args.hop else T) * n
    achieved = ALG_BYTES_PER_SAMPLE * launch_samples / (k1_ms / 1000.0) / 1e9
    # kernels of this library per push: K1 (+ k_peak_unpack in the split mode), k_detect, k_entries_prefix, k_entries_sort, k_track
    launches = int(agg["spectral_launches"] * (2 if n > 16384 else 1) + 3 * agg["detect_launches"] + agg["window_launches"] + agg["track_launches"])
    sweep = None
    if args.sweep:
        sweep = []
        for Ts in (64, 256, 1024, 4096):
            ms_s, agg_s, _, _ = run(Ts, max(args.steps, 5), 3, True)
            sweep.append(summarise(Ts, max(args.steps, 5), ms_s, agg_s))

    # ---- config 4's record leg (SURVEY.md 8(f)#1): rotate + resample 40 MS/s -> 32 kS/s + int8 for the four carriers ----
    record = None
    if args.config == 4 and rank == 0:
        iq4 = synth.make_iq_int8_torch(n, T, tones_for(T), seed=synth.seed_for(4, 0), quiet_frames=LEARN, device=dev)
        shifts = [b2s.get_tuned_frequency(int(mhz * 1e6), 2500) for mhz in (-12.5, -3.2, 4.7, 15.1)]
        recs = [b2s.Recorder(eng, fs, 32_000, on_device=True, max_samples_per_push=T * n) for _ in shifts]
        for r_, sh in zip(recs, shifts):
            r_.start(sh)
            r_.push(iq4.data_ptr(), T * n)  # warm-up
        torch.cuda.synchronize()
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 3
        r0.record(main_stream)
        out_samples = 0
        for _ in range(reps):
            for r_ in recs:
                out_samples += len(r_.push(iq4.data_ptr(), T * n)) // 2
        r1.record(main_stream)
        torch.cuda.synchronize()
        ms_r = r0.elapsed_time(r1) / reps
        record = {"recorders": len(recs), "ms_per_step": ms_r, "input_msps_per_recorder": T * n / (ms_r / len(recs) / 1000.0) / 1e6,
                  "output_samples_per_step": out_samples // reps, "stages": [list(x) for x in recs[0].stages()],
                  "note": "each recorder reads the step's device-resident IQ (67.1 M samples) once; synchronous pushes, one after the other"}
        for r_ in recs:
            r_.close()
        del iq4

    # ---- end-to-end run: pinned host IQ, H2D inside the timed region ----
    e2e = None
    if not args.skip_e2e:
        steps_e = max(3, min(args.steps, 10))
        ms_e, agg_e, _, _ = run(T, steps_e, 3, False, hop=args.hop)
        e2e = {
            "value": aggregate_msps(samples_step, steps_e, world, ms_e), "unit": "MS/s",
            "h2d_bytes_per_step": int(agg_e["h2d_bytes"] // steps_e), "d2h_bytes_per_step": int(agg_e["d2h_bytes"] // steps_e),
            "steps": steps_e, "ms_per_step": ms_e / steps_e,
            "pcie_gbs_per_gpu": agg_e["h2d_bytes"] / steps_e / (ms_e / steps_e / 1000.0) / 1e9, "host_binding": numa,
        }

    # ---- cpu baseline (rank 0, N = 1 only): bounded sample of the same workload, all cores and one thread ----
    cpu = None
    if rank == 0 and world == 1 and not args.skip_cpu:
        import oracle_lib as ol

        os.sched_setaffinity(0, all_cpus)  # the CPU arm uses every host core, not just the GPU's NUMA node
        cores = len(all_cpus)
        per_thread = max(64, min(512, (1 << 23) // n))

        def segment(frames):
            return synth.make_iq_int8(n, frames, tones_for(max(frames, LEARN + 8)), seed=synth.seed_for(args.config), quiet_frames=LEARN)

        allc = cpu_sample(b2s, synth, ol, wl, segment, cores, 8.0, per_thread)
        one = cpu_sample(b2s, synth, ol, wl, segment, 1, 3.0, per_thread)
        cpu = {"value": allc["value"], "unit": "MS/s", "cores": cores, "kind": "port", "fft": fft_backend(ol),
               "spread": {"min": allc["min"], "max": allc["max"], "reps": allc["reps"]}, "single_thread": one["value"], "stage_split_single_thread": one["stage_split"],
               "sample": f"{allc['reps']} x {allc['frames']} frames ({cores} threads x {per_thread} frames, one chain per thread) of the workload; restated CPU path with fp32 FFT"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": head["value"], "unit": "MS/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["name"] + (" — hop variant: b2s_band_reset every 125 frames" if args.hop else ""), "fft_size": n, "sample_rate_hz": fs,
                       "frames_per_step": T, "bands_per_gpu": n_bands, "input": "int8 IQ (CS8)",
                       "l2": f"{samples_step * 2 / 1e6:.0f} MB of input per step and GPU " + ("> 126 MB L2 (no flush needed)" if samples_step * 2 > 126e6 else "(+ the 4 B/sample rows written: the step's working set exceeds the 126 MB L2)" if samples_step * 6 > 126e6 else "< L2: inputs may be L2-resident"),
                       "parallelism": f"bands sharded, {world} GPU(s), no data-path collective"},
            "roofline": {"bound": "hbm", "kernel": f"k_spectrum3 (N={n})", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": K1_TRAFFIC["bytes"] if (args.config == 2 and T == 4096) else None, "traffic_source": K1_TRAFFIC["source"],
                         "peak_source": peak_src, "algorithmic_bytes_per_launch": ALG_BYTES_PER_SAMPLE * launch_samples, "kernel_ms": k1_ms,
                         "other_kernels_ms": {"k_detect+list_ordering": k2_ms, "k_track (beside the next step's K1)": head["k4_ms"],
                                              "k_window_query_total": agg["window_ms"] / args.steps, "host_per_step": agg["tracker_host_ms"] / args.steps},
                         "k_detect": {"achieved": K2_ALG_BYTES_PER_SAMPLE * launch_samples / (k2_ms / 1000.0) / 1e9, "unit": "GB/s", "frac": head["k2_frac"],
                                      "cta_median_ms": stats["cta"][0] if stats["cta"] else None, "cta_max_ms": stats["cta"][1] if stats["cta"] else None},
                         "path": {"achieved": ALG_BYTES_PER_SAMPLE * samples_step / (ms / args.steps / 1000.0) / 1e9, "frac": head["path_frac"],
                                  "note": "6 B/sample x samples per step / step time (all kernels, all bands)"}},
            "cpu_baseline": cpu,
            "e2e": e2e,
            "gpu_launches": launches,
            "clocks": clocks,
            "detections": {"transmissions_after_last_step": stats["n_tx"], "detect_entries_last_step": stats["n_entries"],
                           "k4_per_push": {k: agg[k] / max(agg["track_launches"], 1) for k in ("track_evals", "track_events", "track_best_index")}},
        }
        if sweep is not None:
            line["sweep"] = sweep
        if record is not None:
            line["record_leg"] = record
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
