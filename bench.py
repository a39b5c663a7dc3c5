#!/usr/bin/env python
"""bench.py — headline benchmark of the B200-native OpenWebRX+ DSP hot path.

Metric (BASELINE.json): channel-MS/s = wideband input MS/s x concurrent client channels (+ waterfall lines/s).

  python bench.py --gpus 1 --steps K --warmup W     BASELINE config 2 on one GPU: "Selector DDC + NFM/AM/USB demod, 10 MS/s
                                                     wideband, 64 concurrent 12 kHz client channels on 1xB200".  The line also
                                                     carries `configs`: C1 ... C5 each measured on this GPU with its own SURVEY 8(d)
                                                     roofline and a CPU-port figure.
  torchrun ... bench.py --gpus N (N > 1)            BASELINE config 3: 61.44 MS/s wideband, 1024 client channels sharded N ways
                                                     (STRONG scaling: the total is fixed), the IQ block crossing NVLink every step,
                                                     plus the north-star load paced at real time as a sub-object.
  python bench.py --impl reference ...              the CPU chain (oracle port; pycsdr cannot be built here) on the host cores
  python bench.py --gpus 1 ... --dump-outputs DIR   also writes DIR/audio.npy: the float32 audio [channels, samples] of the last
                                                     timed step, as a caller of the device path receives it; the input is seeded,
                                                     so two builds run with the same arguments can be compared output for output

A step = one pass of the hot path (Shift -> FirDecimate -> [FractionalDecimator] -> Bandpass -> Squelch -> demodulator -> Agc for
every channel) over one synthetic IQ block.  Prints ONE JSON line (rank 0): `value` = device-resident throughput (CUDA events,
max over ranks); `e2e` = the same through the public host API from pinned host memory with the audio read back; `roofline` =
SURVEY 8(d)'s algorithmic bytes of a step over the measured step time (the kernels' own operand traffic is in
`roofline_kernel` / `dram_bytes_per_step`); `cpu_baseline` = the oracle port on the host cores."""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "channel-MS/s (input MS/s x clients) + waterfall FFT frames/s"
BLOCK = 1 << 24           # samples per selector step: 134 MB of complex64 > the 126 MB L2
OUT_RATE = 12000

# BASELINE.json configs (SURVEY 8d)
C2 = dict(name="C2", fs=10_000_000, out_rate=12000, channels=64, block=BLOCK,
          workload="C2: Selector DDC + NFM/AM/USB demod, 10 MS/s wideband, 64 x 12 kHz channels per GPU")
# (C3 steps are 2^25 samples = 0.55 s of signal: with D = 5120 the per-channel fast-convolution table is 10.5 MB, and a pass has to
# hold >= 30 overlap-save blocks before the tensor-core contraction amortises reading it — VERDICT r1 task 4d)
C3 = dict(name="C3", fs=61_440_000, out_rate=12000, channels=1024, block=1 << 25,
          workload="C3: 61.44 MS/s wideband, 1024 x 12 kHz client channels (NFM/AM/USB) in total, sharded across the GPUs (strong scaling), "
                   "IQ block over NVLink every step")
C5 = dict(name="C5", fs=20_000_000, out_rate=250000, channels=128, block=1 << 23, wfm=True, audio_rate=48000,
          workload="C5: WFM broadcast front end, 20 MS/s wideband, 128 channels -> 250 kHz IF -> 48 kHz audio, de-emphasis 50 us")
C1 = dict(name="C1", fs=2_400_000, n=4096, fps=9, ov=0.3, lines=592,
          workload="C1: FftChain 2.4 MS/s, 4096-pt, 9 fps, overlap 0.3 (avg 93, hop 2867), LogAveragePower + ADPCM")
C4 = dict(name="C4", fs=61_440_000, n=65536, fps=30, ov=0.3, lines=512, noise_filter=True,
          workload="C4: 65536-pt waterfall at 30 fps on 61.44 MS/s (avg 45, hop 45511), spectral-subtraction noise filter + ADPCM")


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), float(d.get("sm_max_mhz", 1965.0)), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, 1965.0, "fallback (B200_PROFILING.md)"


def load_traffic():
    """DRAM bytes of ONE step per config (sum of dram__bytes_read + dram__bytes_write over every kernel of the step), from the
    committed ncu run profiles/r2_step_traffic.json (tools/step_traffic.py); {} when absent"""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "r2_step_traffic.json")))
    except Exception:
        return {}


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region (B200_PROFILING.md): NVML polled every few ms from a
    thread (the main thread sits in cudaStreamSynchronize with the GIL released); nvidia-smi -lms as fallback."""
    REASONS = (("hw_slowdown", 0x8), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40), ("sw_power_cap", 0x4))

    def __init__(self, index):
        self.index = index
        self.samples = []          # (sm_mhz, max_mhz, reason_mask, t)
        self.stop_flag = False
        self.thread = None
        self.proc = None
        self.lines = []

    def _nvml_loop(self):
        import pynvml
        h, mx = self.handle, self.max_mhz
        while not self.stop_flag:
            try:
                sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
                try:
                    mask = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    mask = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.samples.append((float(sm), float(mx), int(mask), time.perf_counter()))
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()                 # the slow part, done before any timed work
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
            pynvml.nvmlDeviceGetClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
            self.thread = threading.Thread(target=self._nvml_loop, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.thread = None
        try:
            q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits",
                                          "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def mark(self):
        """start of the timed regions: the sampler has been running since before the warm-up (NVML start-up is slow)"""
        self.t_mark = time.perf_counter()

    def stop(self):
        reasons = set()
        window = "timed regions"
        if self.thread is not None:
            t_end = time.perf_counter()
            self.stop_flag = True
            self.thread.join(1.0)
            t0 = getattr(self, "t_mark", 0.0)
            inside = [x for x in self.samples if t0 <= x[3] <= t_end]
            if len(inside) < 3:
                inside, window = list(self.samples), "warm-up + timed regions"
            for _, _, mask, _ in inside:
                for name, bit in self.REASONS:
                    if mask & bit:
                        reasons.add(name)
            sm = [x[0] for x in inside]
            mx = [x[1] for x in inside]
        elif self.proc is not None:
            time.sleep(0.05)
            self.proc.terminate()
            sm, mx = [], []
            for l in self.lines:
                f = [x.strip() for x in l.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1])); mx.append(float(f[2]))
                except ValueError:
                    continue
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
        else:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no clock source"], "samples": 0}
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm), "window": window}


# ------------------------------------------------------------------------------------------------ synthetic input
def channel_plan(rank, n_ch, fs=C2["fs"], wfm=False):
    from openwebrx_b200.synth import carrier_plan
    if wfm:
        return carrier_plan(n_ch, fs, seed=20260101 + rank, wfm=True, span=0.4)
    return carrier_plan(64, fs, seed=20260101 + rank)[:n_ch] if n_ch <= 64 else carrier_plan(n_ch, fs, seed=20260101 + rank)


def synth_iq_torch(n, fs, carriers, device, seed=20260101):
    """Same signal model as openwebrx_b200.synth.make_iq, generated on the GPU (plumbing, untimed)."""
    import torch
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    x = torch.empty(n, 2, device=device, dtype=torch.float32)
    chunk = 1 << 21
    for s in range(0, n, chunk):
        e = min(n, s + chunk)
        t = (torch.arange(s, e, device=device, dtype=torch.float64)) / fs
        re = 1e-3 * torch.randn(e - s, device=device, generator=g, dtype=torch.float32)
        im = 1e-3 * torch.randn(e - s, device=device, generator=g, dtype=torch.float32)
        for c in carriers:
            f, a, kind = c["offset"], c["amp"], c["kind"]
            if kind == "am":
                env = a * (1.0 + 0.5 * torch.cos(2 * np.pi * 1000.0 * t)) / 1.5
                ph = 2 * np.pi * ((f * t) % 1.0)
                re += (env * torch.cos(ph)).float(); im += (env * torch.sin(ph)).float()
            elif kind in ("nfm", "wfm"):
                ph = 2 * np.pi * ((f * t) % 1.0) + (2.5 if kind == "nfm" else 75.0) * torch.sin(2 * np.pi * 1000.0 * t)
                re += (a * torch.cos(ph)).float(); im += (a * torch.sin(ph)).float()
            else:
                for df in (700.0, 1900.0):
                    ph = 2 * np.pi * (((f + df) * t) % 1.0)
                    re += (0.5 * a * torch.cos(ph)).float(); im += (0.5 * a * torch.sin(ph)).float()
        x[s:e, 0] = re; x[s:e, 1] = im
    return x


def quick_iq_torch(n, device, seed):
    """noise floor + one strong tone: the kernels' time does not depend on the content; used where the full carrier model (one
    oscillator per channel: 1024 for C3) would only cost set-up time"""
    import torch
    g = torch.Generator(device=device); g.manual_seed(seed)
    x = 1e-3 * torch.randn(n, 2, device=device, generator=g, dtype=torch.float32)
    tt = torch.arange(n, device=device, dtype=torch.float32)
    x[:, 0] += 0.3 * torch.cos(0.7 * tt); x[:, 1] += 0.3 * torch.sin(0.7 * tt)
    return x


# ------------------------------------------------------------------------------------------------ SURVEY 8(d) models
def selector_model(cfg, n_ch, block=None):
    """SURVEY 8(d), per IQ block of Nin samples with C channels resident on one GPU:
         bytes = 8 Nin (IQ read once per GPU) + 4 C Nin / Dtot (float audio out)
         FLOPs(direct form) = C Nin (8 + 4 T / D) + C (Nin / Dtot) (8 Tbp + 30)"""
    from openwebrx_b200.params import decimator_params, filter_length
    fs, out = cfg["fs"], cfg["out_rate"]
    block = block or cfg["block"]
    D, frac, transition, _ = decimator_params(fs, out)
    T = filter_length(transition)
    n_k = (block - T) // D + 1
    consumed = n_k * D
    audio_rate = cfg.get("audio_rate", out)
    dtot = fs / audio_rate
    tbp = filter_length(320.0 / out)
    return dict(D=D, T=T, fraction=frac, n_k=n_k, consumed=consumed,
                bytes=8.0 * block + 4.0 * n_ch * block / dtot,
                flops=n_ch * float(block) * (8.0 + 4.0 * T / D) + n_ch * (block / (fs / out)) * (8.0 * tbp + 30.0))


def waterfall_model(cfg):
    """SURVEY 8(d), per output line: bytes = 8 U + out (U = unique input samples), FLOPs = avg (5 N log2 N + 5 N) + 4 N"""
    from openwebrx_b200.params import fftchain_params
    n = cfg["n"]
    avg, every_n = fftchain_params(cfg["fs"], n, cfg["ov"], cfg["fps"])
    unique = (avg - 1) * every_n + n if every_n < n else avg * n
    return dict(avg=avg, every_n=every_n, bytes=8.0 * unique + (n + 10) // 2, flops=avg * (5.0 * n * np.log2(n) + 5.0 * n) + 4.0 * n)


def roofline(bytes_per_step, flops_per_step, ms, hbm_peak, peak_src, f_mhz, note):
    s = ms * 1e-3
    ach = bytes_per_step / s / 1e9
    fp32_peak = 148 * 128 * 2 * f_mhz * 1e6 / 1e12
    return {"bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak, "peak_source": peak_src,
            "algorithmic_bytes": bytes_per_step, "fp32_tflops_direct_form": flops_per_step / s / 1e12,
            "fp32_frac_direct_form": flops_per_step / s / 1e12 / fp32_peak,
            "fp32_peak_def": "148 SM x 128 lanes x 2 x %.0f MHz (observed)" % f_mhz, "note": note}


# ------------------------------------------------------------------------------------------------ CPU baselines (oracle port)
def cpu_chain_rate(cfg, carriers, seconds_budget, n_samples, threads):
    """Times the oracle port of the per-client chain (one chain per client, one pass per stage — the reference's structure) on
    `threads` host threads.  Returns (channel-MS/s, chains run, wall s)."""
    import oracle
    from openwebrx_b200.synth import BANDPASS, make_iq
    kind = {"nfm": oracle.DEMOD_NFM, "am": oracle.DEMOD_AM, "usb": oracle.DEMOD_SSB, "wfm": oracle.DEMOD_WFM}
    fs, out = cfg["fs"], cfg["out_rate"]
    iq = make_iq(n_samples, fs, carriers[:4], seed=1)
    oracle.lib()

    def one(c):
        oracle.client_chain_run(iq, fs, out, c["offset"], BANDPASS[c["kind"]], kind[c["kind"]], audio_rate=float(cfg.get("audio_rate", 48000)),
                                fast_shift=True)

    t0 = time.perf_counter(); one(carriers[0]); t1 = time.perf_counter() - t0
    per_thread = max(1, int(seconds_budget / max(t1, 1e-3)))
    done = [0] * threads

    def worker(i):
        for k in range(per_thread):
            one(carriers[(i + k) % len(carriers)])
            done[i] += 1

    ths = [threading.Thread(target=worker, args=(i,)) for i in range(threads)]
    t0 = time.perf_counter()
    for t in ths: t.start()
    for t in ths: t.join()
    wall = time.perf_counter() - t0
    total = sum(done)
    return total * n_samples / wall / 1e6, total, wall


def cpu_waterfall_rate(cfg, lines):
    """the oracle's FftChain (one stream: single-threaded, like the reference's one chain per source) over `lines` lines"""
    import oracle
    m = waterfall_model(cfg)
    n = cfg["n"]
    rng = np.random.default_rng(3)
    ns = m["every_n"] * m["avg"] * lines + n
    x = (1e-3 * (rng.standard_normal(ns) + 1j * rng.standard_normal(ns))).astype(np.complex64)
    t0 = time.perf_counter()
    r = oracle.fftchain_run(x, n, m["every_n"], m["avg"])
    wall = time.perf_counter() - t0
    assert len(r["lines"]) == lines
    return lines / wall, wall


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path.  pycsdr/libcsdr are not in the reference tree and
    cannot be built (SURVEY F2-F4), so this times the oracle port (cpu_baseline.kind "port") with all host threads, on the same
    config / metric as our arm: C2 at --gpus 1, C3 at --gpus N > 1."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    cfg = C2 if args.gpus <= 1 else C3
    carriers = channel_plan(0, 64, cfg["fs"])
    n_samples = 1 << 20
    vals, ms = [], []
    for step in range(args.warmup + args.steps):
        v, total, wall = cpu_chain_rate(cfg, carriers, 1.0, n_samples, threads)
        if step >= args.warmup:
            vals.append(v); ms.append(wall * 1e3)
    value = float(np.mean(vals)) if vals else 0.0
    sample = "%d threads x oracle client chains (%.2f MS/s -> 12 kHz NFM/AM/USB) over %d-sample records, ~1 s per step" % (
        threads, cfg["fs"] / 1e6, n_samples)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "channel-MS/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": float(np.mean(ms)) if ms else None, "higher_is_better": True,
            "scaling": "weak" if args.gpus <= 1 else "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": cfg["workload"]},
            "cpu_baseline": {"value": value, "unit": "channel-MS/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "channel-MS/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ device-resident measurements
def make_bank(cfg, carriers, local, rank_offset=0):
    from openwebrx_b200 import ChannelBank
    from openwebrx_b200.synth import BANDPASS
    bank = ChannelBank(cfg["fs"], device=local)
    kw = dict(audio_rate=float(cfg["audio_rate"]), tau=50e-6) if cfg.get("wfm") else {}
    chans = [bank.add_channel(cfg["out_rate"], demod=c["kind"], offset=c["offset"] + rank_offset, bandpass=BANDPASS[c["kind"]], **kw)
             for c in carriers]
    return bank, chans


def time_bank_device(torch, bank, blocks, n, stream, steps, warmup):
    """`steps` pipelined device-resident passes over alternating resident blocks (2 x 134 MB between two reads of the same bytes:
    beyond the 126 MB L2); CUDA events on the launching stream; returns (ms per step, per-stage ms, kernel launches per step)"""
    from openwebrx_b200 import _native as N
    sp = stream.cuda_stream
    bank.set_pipelined(True)
    for i in range(warmup):
        bank.process_device(blocks[i & 1], n, stream=sp)
    bank.join(sp); stream.synchronize()
    if steps <= 0:
        return None, {}, 0
    bank.profile(True); bank.profile_read(reset=True)
    l0 = N.lib.owrx_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for i in range(steps):
        bank.process_device(blocks[i & 1], n, stream=sp)
    bank.join(sp)
    e1.record(stream); stream.synchronize()
    ms = e0.elapsed_time(e1) / steps
    prof = bank.profile_read_ex(reset=True)
    bank.profile(False)
    stages = {k: v[0] / steps for k, v in prof.items() if v[1]}          # device time per step (a stage may be several brackets)
    return ms, stages, (N.lib.owrx_launch_count() - l0) / steps


def dump_audio(path, bank, chans):
    """the outputs of the last process_device step: owrx_bank_drain moves them to the host queues, one read pops every channel's
    audio; written as float32 [channels, samples] (every channel of the workload has the same output rate)"""
    bank.drain()
    buf = np.empty((len(chans), 1 << 15), np.float32)
    counts = bank.read_audio_all(chans, buf)
    assert len(set(counts)) == 1 and counts[0] > 0, counts
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "audio.npy"), buf[:, :counts[0]])


def bench_selector_config(torch, dev, cfg, n_ch, hbm_peak, peak_src, f_mhz, steps=5, warmup=3, cpu_seconds=1.5):
    """one selector config on this GPU, device-resident, with its SURVEY 8(d) roofline and the CPU port beside it"""
    m = selector_model(cfg, n_ch)
    carriers = channel_plan(0, n_ch, cfg["fs"], wfm=bool(cfg.get("wfm")))
    bank, _ = make_bank(cfg, carriers, dev.index or 0)
    blocks = [quick_iq_torch(cfg["block"], dev, 11), quick_iq_torch(cfg["block"], dev, 12)]
    stream = torch.cuda.current_stream()
    ms, stages, launches = time_bank_device(torch, bank, blocks, cfg["block"], stream, steps, warmup)
    form = bank.fir_form()
    bank.close()
    del blocks
    torch.cuda.empty_cache()
    threads = os.cpu_count() or 1
    v, total, wall = cpu_chain_rate(cfg, carriers[:64], cpu_seconds, 1 << 20, threads)
    wl = cfg["workload"] if cfg is not C3 else ("C3 on ONE GPU (the N = 1 point of the strong-scaling curve): 61.44 MS/s wideband, "
                                                "1024 x 12 kHz channels")
    return {"workload": wl, "channels": n_ch, "block_samples": cfg["block"], "decimation": m["D"], "fir_taps": m["T"],
            "value": n_ch * m["consumed"] / (ms * 1e-3) / 1e6, "unit": "channel-MS/s", "ms_per_step": ms, "steps": steps,
            "realtime_factor": m["consumed"] / cfg["fs"] / (ms * 1e-3), "fir_form": form, "stages_ms": stages, "gpu_launches_per_step": launches,
            "roofline": roofline(m["bytes"], m["flops"], ms, hbm_peak, peak_src, f_mhz,
                                 "SURVEY 8(d): 8 Nin + 4 C Nin / Dtot bytes per step over the step time; the fast-convolution form trades "
                                 "the direct form's FLOPs for operand traffic, so neither 8(d) roof binds the step"),
            "cpu_baseline": {"value": v, "unit": "channel-MS/s", "cores": threads, "kind": "port",
                             "sample": "%d oracle client chains over 2^20-sample records on %d threads, %.1f s wall" % (total, threads, wall)},
            "data": "synthetic: noise floor + one tone (kernel time does not depend on the content)"}


def bench_waterfall(torch, dev, cfg, hbm_peak, peak_src, f_mhz, steps=5, cpu_lines=None):
    """one FftChain config on this GPU: `lines` lines per batch, device-resident, pipelined side-stream ADPCM encoder"""
    from openwebrx_b200 import Waterfall
    m = waterfall_model(cfg)
    n, lines = cfg["n"], cfg["lines"]
    ns = m["every_n"] * m["avg"] * lines + n
    iq = quick_iq_torch(ns, dev, 7)                       # C1: 1.27 GB, C4: 8.4 GB of IQ — far beyond L2
    wf = Waterfall(cfg["fs"], n, cfg["ov"], cfg["fps"], "adpcm", device=dev.index or 0)
    if cfg.get("noise_filter"):
        wf.set_noise_filter(True)
    out = torch.empty(lines * wf.line_bytes, dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream()
    assert st.cuda_stream != 0
    torch.cuda.synchronize()
    wf.set_pipelined(True)        # ADPCM of batch i on the side stream beside the FFT pass of batch i+1
    for _ in range(3):
        wf.process_device(iq, ns, out, out.numel(), stream=st.cuda_stream)
    wf.join(st.cuda_stream)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for _ in range(steps):
        got = wf.process_device(iq, ns, out, out.numel(), stream=st.cuda_stream)
    wf.join(st.cuda_stream)
    e1.record(st)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    wf.close()
    del iq, out
    torch.cuda.empty_cache()
    cpu_lines = cpu_lines or (40 if n <= 4096 else 4)
    cl, cwall = cpu_waterfall_rate(cfg, cpu_lines)
    return {"workload": cfg["workload"], "lines_per_batch": int(got), "value": got / (ms * 1e-3), "unit": "lines/s",
            "ffts_per_s": got * m["avg"] / (ms * 1e-3), "ms_per_step": ms, "steps": steps, "realtime_factor": got / (ms * 1e-3) / cfg["fps"],
            "roofline": roofline(m["bytes"] * got, m["flops"] * got, ms, hbm_peak, peak_src, f_mhz,
                                 "SURVEY 8(d): (8 U + out) bytes per line over the whole FftChain batch (FFT + finalize + ADPCM launches)"),
            "cpu_baseline": {"value": cl, "unit": "lines/s", "cores": 1, "kind": "port",
                             "sample": "%d lines through the oracle's FftChain, single thread (one stream), %.2f s wall" % (cpu_lines, cwall)},
            "data": "synthetic: noise floor + one tone"}


# ------------------------------------------------------------------------------------------------ our arm
def run_ours(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # the hop runs beside the DSP kernels: NCCL's copy CTAs take SMs from the latency-bound low-rate stages; 16 channels
        # carry the block with half the CTAs of the default (measured on 2 B200, tools/nccl_channels_sweep.sh)
        os.environ.setdefault("NCCL_MAX_NCHANNELS", "16")
        dist.init_process_group("nccl", device_id=dev)
        return run_sharded(args, torch, dist, world, rank, local, dev)
    return run_single(args, torch, local, dev)


def run_single(args, torch, local, dev):
    from openwebrx_b200 import ChannelBank
    from openwebrx_b200.synth import BANDPASS
    hbm_peak, sm_max, peak_src = load_peaks()
    cfg = C2
    n_ch = cfg["channels"]
    m = selector_model(cfg, n_ch)
    D, T, consumed = m["D"], m["T"], m["consumed"]

    carriers = channel_plan(0, n_ch)
    bank, chans = make_bank(cfg, carriers, local)
    iq = synth_iq_torch(BLOCK, cfg["fs"], carriers, dev)
    blocks = [iq, iq.clone()]
    stream = torch.cuda.Stream(device=dev)          # a created (non-default) stream: the C ABI treats NULL as "the object's own"
    torch.cuda.synchronize()
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0

    clocks = ClockSampler(local)
    clocks.start()                                  # NVML start-up takes longer than a short timed region: poll from the warm-up on
    time_bank_device(torch, bank, blocks, BLOCK, stream, 0, args.warmup)
    clocks.mark()
    ms_step, stages, launches = time_bank_device(torch, bank, blocks, BLOCK, stream, args.steps, 0)
    fir_form = bank.fir_form()
    value = n_ch * consumed / (ms_step * 1e-3) / 1e6
    if args.dump_outputs:
        dump_audio(args.dump_outputs, bank, chans)

    # ---- e2e: public host API, pinned host input, H2D + audio D2H inside the timed region
    h_iq = torch.empty(BLOCK, 2, dtype=torch.float32).pin_memory()
    h_iq.copy_(iq)
    audio_buf = np.empty((n_ch, 1 << 15), np.float32)      # ~20 160 samples per channel and block

    def new_bank():
        b = ChannelBank(cfg["fs"], device=local)
        return b, [b.add_channel(OUT_RATE, demod=c["kind"], offset=c["offset"], bandpass=BANDPASS[c["kind"]]) for c in carriers]

    def e2e_loop(b, chs, steps, ptr, **kw):
        got = 0
        for i in range(steps):
            b.feed_ptr(ptr, BLOCK, **kw)
            got += sum(b.read_audio_all(chs, audio_buf))
        b.flush()                                     # streaming mode: the last block's final outputs
        got += sum(b.read_audio_all(chs, audio_buf))
        return got

    # the host API in its streaming mode (owrx_bank_set_deferred_drain): a feed only enqueues and returns, the kernel tail, D2H
    # and queue hand-over of block i run under the upload of block i+1; every block is uploaded from pinned host memory and
    # every block's audio is read back inside the timed region (the last one after a flush)
    bank2, ch2 = new_bank()
    bank2.set_deferred_drain(True)
    e2e_loop(bank2, ch2, 3, h_iq.data_ptr())
    torch.cuda.synchronize()
    e2e_steps = max(1, min(args.steps, 10))
    t0 = time.perf_counter()
    n_audio = e2e_loop(bank2, ch2, e2e_steps, h_iq.data_ptr())
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
    bank2.set_deferred_drain(False)
    e2e_loop(bank2, ch2, 1, h_iq.data_ptr())
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        bank2.feed_ptr(h_iq.data_ptr(), BLOCK)
        bank2.read_audio_all(ch2, audio_buf)
    torch.cuda.synchronize()
    ms_sync = (time.perf_counter() - t0) * 1e3 / e2e_steps
    e2e_consumed = (BLOCK // D) * D                   # the streaming path carries the FIR tail between blocks
    e2e_sync = {"value": n_ch * e2e_consumed / (ms_sync * 1e-3) / 1e6, "unit": "channel-MS/s", "ms_per_step": ms_sync,
                "note": "owrx_bank_feed in its default synchronous mode"}
    e2e_value = n_ch * e2e_consumed / (e2e_ms * 1e-3) / 1e6
    d2h = (n_audio // (e2e_steps + 1)) * 4
    bank2.close()

    # ---- the same end-to-end step for a source that delivers complex int16 (SURVEY 8f-4): half the PCIe bytes, Convert on the GPU
    h16 = torch.empty(BLOCK, 2, dtype=torch.int16).pin_memory()
    h16.copy_((iq.clamp(-1, 1) * 32767.0).to(torch.int16))
    bank3, ch3 = new_bank()
    bank3.set_deferred_drain(True)
    e2e_loop(bank3, ch3, 3, h16.data_ptr(), fmt="cs16")
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    e2e_loop(bank3, ch3, e2e_steps, h16.data_ptr(), fmt="cs16")
    torch.cuda.synchronize()
    ms16 = (time.perf_counter() - t0) * 1e3 / e2e_steps
    e2e_cs16 = {"value": n_ch * e2e_consumed / (ms16 * 1e-3) / 1e6, "unit": "channel-MS/s", "h2d_bytes_per_step": BLOCK * 4,
                "d2h_bytes_per_step": int(d2h), "ms_per_step": ms16,
                "note": "same step fed with complex int16 host samples (owrx_bank_feed_fmt): Convert runs on the GPU"}
    bank3.close()
    bank.close()
    del blocks, iq, h16, h_iq
    torch.cuda.empty_cache()

    f_mhz = (clocks.samples[-1][0] if clocks.samples else sm_max) or sm_max
    # ---- every BASELINE config on this GPU, each with its 8(d) roofline and the CPU port
    subs = {}
    if not args.headline_only:
        # (25 / 12 batches per timed run: the side-stream encoder of the LAST batch is exposed once — 0.25 ms at C1, 3.8 ms at C4 —
        # and a five-batch run charged a fifth of it to every batch)
        subs["C1"] = bench_waterfall(torch, dev, C1, hbm_peak, peak_src, f_mhz, steps=25)
        subs["C3"] = bench_selector_config(torch, dev, C3, 1024, hbm_peak, peak_src, f_mhz, steps=3, warmup=3)
        subs["C4"] = bench_waterfall(torch, dev, C4, hbm_peak, peak_src, f_mhz, steps=12)
        subs["C5"] = bench_selector_config(torch, dev, C5, 128, hbm_peak, peak_src, f_mhz)
    clk = clocks.stop()
    f_obs = (clk or {}).get("sm_mhz") or sm_max

    # ---- CPU baseline beside the headline (bounded sample)
    cpu = None
    if not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        v, total, wall = cpu_chain_rate(cfg, carriers, 2.0, 1 << 20, threads)
        cpu = {"value": v, "unit": "channel-MS/s", "cores": threads, "kind": "port",
               "sample": "%d oracle client chains (C2 shape) over 2^20-sample records on %d threads, %.1f s wall" % (total, threads, wall)}

    # ---- rooflines.  Headline: SURVEY 8(d)'s algorithmic bytes of the step over the measured step time.
    traffic = load_traffic()
    t_c2 = traffic.get("C2", {})
    dram_step = t_c2.get("dram_bytes_per_step")
    dominant = max(stages, key=stages.get) if stages else None
    rl = roofline(m["bytes"], m["flops"], ms_step, hbm_peak, peak_src, f_obs,
                  "SURVEY 8(d): (8 Nin + 4 C Nin / Dtot) = %.1f MB per step over the measured step time.  The step is a pipeline of "
                  "kernels (stages_ms); the fast-convolution channeliser replaces the direct form's 53 FMA per sample and channel by "
                  "~4.5 and pays with operand traffic (dram_bytes_per_step), so neither 8(d) roof binds it" % (m["bytes"] / 1e6))
    rl["kernel"] = ("whole C2 step (dominant stage by in-pipeline time: %s, %.3f ms)" % (dominant, stages[dominant])) if dominant else "whole C2 step"
    rl["traffic"] = dram_step
    rl["traffic_over_algorithmic"] = (dram_step / m["bytes"]) if dram_step else None
    c2cfg = {"workload": cfg["workload"], "channels": n_ch, "value": value, "unit": "channel-MS/s", "ms_per_step": ms_step, "roofline": rl,
             "cpu_baseline": cpu, "stages_ms": stages, "fir_form": fir_form}
    configs = {"C1": subs.get("C1"), "C2": c2cfg, "C3": subs.get("C3"), "C4": subs.get("C4"), "C5": subs.get("C5")}
    for k, v in configs.items():
        tk = traffic.get(k, {}).get("dram_bytes_per_step")
        if v is not None and k != "C2" and tk:
            v["roofline"]["traffic"] = tk
            v["roofline"]["traffic_over_algorithmic"] = tk / v["roofline"]["algorithmic_bytes"]

    # the contraction kernel's own operand roofline (what the round-1 line reported as `roofline`)
    rk = None
    if fir_form == "fastconv_tc" and "fc_contract" in stages:
        M, P = 256, -(-T // D)
        Kb, Dp = M - P + 1, -(-D // 32) * 32
        B = -(-m["n_k"] // Kb)
        fmt_env = os.environ.get("OWRX_FC_TC_FMT")                             # operand split (fc_pick_tc_levels): fp16 x 2 for D >= 2048
        lv = 3 if fmt_env == "bf16x3" else 2 if fmt_env == "f16x2" else (2 if D >= 2048 else 3)
        eb = 4.0 * lv                                                          # bytes per complex operand entry
        op_bytes = eb * M * B * Dp + eb * M * Dp * n_ch + 8.0 * M * B * n_ch
        ks = stages["fc_contract"] * 1e-3
        fmt = "fp16x2, block-scaled" if lv == 2 else "bf16x3"
        rk = {"kernel": "fc_contract_tc_kernel (tcgen05 %s -> FP32 in TMEM; %d blocks x %d branches x %d ch)" % (fmt, B, D, n_ch),
              "bound": "hbm", "achieved": op_bytes / ks / 1e9, "peak": hbm_peak, "unit": "GB/s", "frac": op_bytes / ks / 1e9 / hbm_peak,
              "operand_bytes": op_bytes, "kernel_ms": stages["fc_contract"], "kernel_share_of_step": stages["fc_contract"] / ms_step,
              "note": "the kernel's OWN operand bytes (%s spectra + table + Z), not SURVEY 8(d)'s algorithmic bytes" % fmt}

    line = {
        "metric": METRIC, "value": value, "unit": "channel-MS/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": cfg["workload"], "channels_total": n_ch, "block_samples": BLOCK, "decimation": D, "fir_taps": T,
                   "l2": "two resident 134 MB input blocks alternate (268 MB between re-reads > 126 MB L2); no flush needed",
                   "parallelism": "1 GPU", "realtime_factor": value / (cfg["fs"] / 1e6 * n_ch)},
        "e2e": {"value": e2e_value, "unit": "channel-MS/s", "h2d_bytes_per_step": BLOCK * 8, "d2h_bytes_per_step": int(d2h), "ms_per_step": e2e_ms,
                "mode": "streaming (owrx_bank_set_deferred_drain): block i's outputs are drained under block i+1's upload; all blocks' audio "
                        "read inside the timed region (last block after owrx_bank_flush)"},
        "e2e_sync": e2e_sync, "e2e_cs16": e2e_cs16,
        "gpu_launches": int(round(launches * args.steps)),
        "clocks": clk,
        "roofline": rl, "roofline_kernel": rk,
        "dram_bytes_per_step": dram_step, "dram_source": t_c2.get("source"),
        "fir_form": fir_form, "stages_ms": stages, "dominant_stage": dominant,
        "configs": configs,
        "waterfall": configs.get("C1"),
        "cpu_baseline": cpu,
    }
    print(json.dumps(line))


def run_sharded(args, torch, dist, world, rank, local, dev):
    """N > 1: BASELINE config 3, strong scaling.  The 1024 channels are partitioned across the ranks (SURVEY 8e); the wideband
    block lives SHARDED, 1/N per GPU — the layout of a sharded ingest, every rank uploading its slice over its own PCIe link —
    and is all-gathered over NVLink every step, one block ahead of the DSP pass."""
    from openwebrx_b200 import _native as N
    from openwebrx_b200.sharding import make_hop, shard_channels
    from openwebrx_b200.synth import carrier_plan
    hbm_peak, sm_max, peak_src = load_peaks()
    cfg = C3
    BLOCK = cfg["block"]
    total = cfg["channels"]
    mine = list(shard_channels(total, world, rank))
    cars = carrier_plan(total, cfg["fs"], seed=20260101)
    m = selector_model(cfg, len(mine))
    consumed = m["consumed"]
    bank, chans = make_bank(cfg, [cars[c] for c in mine], local)
    assert BLOCK % world == 0
    shard = BLOCK // world

    # every rank's resident slice of two alternating blocks (same generator on every rank: slices of one signal)
    slices = []
    for seed in (21, 22):
        full = quick_iq_torch(BLOCK, dev, seed)
        slices.append(full[rank * shard:(rank + 1) * shard].clone())
        del full
    torch.cuda.empty_cache()
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.synchronize()
    torch.cuda.set_stream(stream)
    sp = stream.cuda_stream
    hop = make_hop(os.environ.get("OWRX_HOP", "auto"), BLOCK, world, rank, dev)

    def barrier():
        dist.barrier()
        torch.cuda.synchronize()

    sent = [0]

    def step(i):
        # block i + 1 crosses NVLink on the hop's stream while block i is processed; buffers alternate
        while sent[0] <= i + 1:
            hop.gather(sent[0], slices[sent[0] & 1])
            sent[0] += 1
        buf = hop.recv(i, stream)
        bank.process_device(buf, BLOCK, stream=sp)
        hop.release(i, stream)

    bank.set_pipelined(True)
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    for i in range(args.warmup):
        step(i)
    bank.join(sp)
    barrier()
    # the hop delivers every rank's slice bit for bit: a checksum of the gathered block against the slices' own
    chk = hop.recv(args.warmup - 1, stream).double().sum().reshape(1)
    want = slices[(args.warmup - 1) & 1].double().sum().reshape(1)
    dist.all_reduce(want)
    assert abs(float(chk.item()) - float(want.item())) <= 1e-6 * max(1.0, abs(float(want.item()))), "the hop delivered a different block"
    bank.profile(True); bank.profile_read(reset=True)
    l0 = N.lib.owrx_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    clocks.mark()
    ev0.record(stream)
    for i in range(args.steps):
        step(args.warmup + i)
    bank.join(sp)
    ev1.record(stream)
    barrier()
    ms_total = ev0.elapsed_time(ev1)
    launches = N.lib.owrx_launch_count() - l0
    prof = bank.profile_read_ex(reset=True)
    bank.profile(False)
    stages = {k: v[0] / args.steps for k, v in prof.items() if v[1]}     # device time per step (a stage may be several brackets)
    hop_ms = hop.mean_ms()
    t = torch.tensor([ms_total, hop_ms or 0.0], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t[0].item()) / args.steps
    hop_ms = float(t[1].item())
    value = total * consumed / (ms_step * 1e-3) / 1e6
    clk = clocks.stop() if rank == 0 else None

    # ---- e2e: sharded ingest.  Every rank uploads ITS slice of the block from pinned host memory over its own PCIe link, the
    # slices are all-gathered over NVLink, every rank runs its channels and returns their audio to the host.
    h_slice = torch.empty(shard, 2, dtype=torch.float32).pin_memory()
    h_slice.copy_(slices[0])
    up = [torch.empty_like(slices[0]), torch.empty_like(slices[0])]
    audio_buf = np.empty((len(chans), 1 << 15), np.float32)
    cnt = [sent[0]]

    up_stream = torch.cuda.Stream(device=dev)
    ev_up = [torch.cuda.Event(), torch.cuda.Event()]
    ev_read = [torch.cuda.Event(), torch.cuda.Event()]

    def ingest(j):
        # H2D of this rank's 1/N of the block on its own stream: the upload of block j + 1 runs beside the all-gather of block j
        # instead of behind it (events: the gather of block j - 1 has read this upload buffer; the gather waits for the upload)
        b = j & 1
        up_stream.wait_event(ev_read[b])
        with torch.cuda.stream(up_stream):
            up[b].copy_(h_slice, non_blocking=True)
            ev_up[b].record(up_stream)
        hop.stream.wait_event(ev_up[b])
        hop.gather(j, up[b])
        ev_read[b].record(hop.stream)

    def e2e_step():
        # one block ahead on the way in (block j + 1 is uploaded and all-gathered under block j's DSP pass) and one block behind
        # on the way out (split-phase drain: block j - 1's audio crosses PCIe and is read on the host while block j is processed)
        j = cnt[0]
        cnt[0] += 1
        ingest(j + 1)
        buf = hop.recv(j, stream)
        bank.process_device(buf, BLOCK, stream=sp)
        hop.release(j, stream)
        bank.drain_end()                                             # block j - 1 (no-op for the first block)
        got = sum(bank.read_audio_all(chans, audio_buf))
        bank.drain_begin()                                           # block j: copied behind its kernels
        return got

    ingest(cnt[0])
    for _ in range(3):
        e2e_step()
    bank.drain_end()                                                 # the warm-up's last block: outside the timed region
    bank.read_audio_all(chans, audio_buf)
    barrier()
    e2e_steps = max(1, min(args.steps, 10))
    t0 = time.perf_counter()
    n_audio = 0
    for _ in range(e2e_steps):
        n_audio += e2e_step()
    bank.drain_end()                                                 # the last block's audio, inside the timed region
    n_audio += sum(bank.read_audio_all(chans, audio_buf))
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
    t = torch.tensor([e2e_ms, float(n_audio)], device=dev, dtype=torch.float64)
    t2 = t.clone()
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dist.all_reduce(t2, op=dist.ReduceOp.SUM)
    e2e_ms = float(t[0].item())
    d2h = float(t2[1].item()) / e2e_steps * 4
    e2e_value = total * consumed / (e2e_ms * 1e-3) / 1e6
    fir_form = bank.fir_form()
    bank.close()
    del slices, up
    torch.cuda.empty_cache()

    ns = None
    if not args.headline_only:
        ns = paced_north_star(torch, dist, world, rank, local, dev, seconds=float(os.environ.get("OWRX_NORTH_STAR_SECONDS", "3")))
    if rank != 0:
        dist.destroy_process_group()
        return
    f_obs = (clk or {}).get("sm_mhz") or sm_max
    m_all = selector_model(cfg, total)
    rl = roofline(m["bytes"], m["flops"], ms_step, hbm_peak, peak_src, f_obs,
                  "per GPU, SURVEY 8(d): 8 Nin + 4 (C / N) Nin / Dtot bytes per step (every GPU reads the whole block and writes its share "
                  "of the audio) over the step time, max over ranks")
    rl["kernel"] = "whole C3 step on one rank (%d of the 1024 channels)" % len(mine)
    rl["traffic"] = None
    dominant = max(stages, key=stages.get) if stages else None
    nvlink_bytes = BLOCK * 8.0 * (world - 1) / world          # into every GPU per step
    line = {
        "metric": METRIC, "value": value, "unit": "channel-MS/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": cfg["workload"], "channels_total": total, "channels_per_gpu": len(mine), "block_samples": BLOCK,
                   "decimation": m["D"], "fir_taps": m["T"],
                   "l2": "two 134 MB blocks alternate (268 MB between re-reads > 126 MB L2); no flush needed",
                   "parallelism": "channels sharded x%d; IQ block resident sharded 1/N per GPU, all-gathered every step: %s" % (world, hop.kind),
                   "realtime_factor": value / (cfg["fs"] / 1e6 * total)},
        "e2e": {"value": e2e_value, "unit": "channel-MS/s", "h2d_bytes_per_step": BLOCK * 8, "d2h_bytes_per_step": int(d2h), "ms_per_step": e2e_ms,
                "mode": "sharded ingest: every rank uploads 1/N of the block from pinned host memory over its own PCIe link (%d bytes per rank "
                        "and step), all-gather over NVLink, owrx_bank_process_device + owrx_bank_drain + the audio of every channel read on "
                        "the host, on every rank; block j + 1's upload and all-gather run under block j's DSP pass, block j - 1's audio is "
                        "drained (owrx_bank_drain_begin / _end) and read under it too" % (shard * 8)},
        "gpu_launches": int(launches),
        "clocks": clk,
        "roofline": rl,
        "hop": {"kind": hop.kind, "ms_per_block": hop_ms, "nvlink_bytes_in_per_gpu": nvlink_bytes,
                "nvlink_GBps_in_per_gpu": (nvlink_bytes / (hop_ms * 1e-3) / 1e9) if hop_ms else None,
                "note": "device time of one all-gather on the hop's stream (max over ranks); it runs one block ahead, under the DSP pass"},
        "fir_form": fir_form, "stages_ms": stages, "dominant_stage": dominant,
        "all_gpus_algorithmic_GBps": m_all["bytes"] / (ms_step * 1e-3) / 1e9,
        "north_star": ns,
        "cpu_baseline": None,
    }
    print(json.dumps(line))
    dist.destroy_process_group()


def paced_north_star(torch, dist, world, rank, local, dev, seconds=3.0, fps=30):
    """BASELINE north_star, paced at REAL TIME: 61.44 MS/s arrive in 1/30 s blocks; every rank uploads its 1/N of each block
    (sharded ingest), the block is all-gathered, every rank runs its share of the 1024 x 12 kHz channels through the device
    path and pops their audio on the host; rank 0 also runs the 65536-point 30 fps waterfall (with the noise filter of config 4)
    through the host API.  Reports how long a block keeps the slowest rank busy against the 33.3 ms budget."""
    from openwebrx_b200 import Waterfall
    from openwebrx_b200.sharding import make_hop, shard_channels
    from openwebrx_b200.synth import carrier_plan
    fs = C3["fs"]
    block = int(fs / fps)
    block -= block % (8 * world)
    shard = block // world
    n_blocks = int(seconds * fps)
    mine = list(shard_channels(1024, world, rank))
    cars = carrier_plan(1024, fs, seed=7)
    bank, chans = make_bank(C3, [cars[c] for c in mine], local)
    audio = np.empty((len(chans), 1 << 12), np.float32)
    win = torch.empty(block + (1 << 18), 2, device=dev)          # [carry | new]: owrx_bank_process_device keeps no wideband history
    carry = [0]
    g = torch.Generator(); g.manual_seed(1 + rank)
    ring = [(1e-3 * torch.randn(shard, 2, generator=g)).pin_memory() for _ in range(4)]
    full_ring, wf = None, None
    if rank == 0:
        full_ring = [(1e-3 * torch.randn(block, 2, generator=g)).pin_memory() for _ in range(2)]
        wf = Waterfall(fs, 65536, 0.3, fps, "adpcm", device=local)
        wf.set_noise_filter(True)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    hop = make_hop(os.environ.get("OWRX_HOP", "auto"), block, world, rank, dev)
    up = [torch.empty(shard, 2, device=dev), torch.empty(shard, 2, device=dev)]
    cnt = [0]

    def one(k):
        j = cnt[0]
        cnt[0] += 1
        hop.stream.wait_stream(stream)
        with torch.cuda.stream(hop.stream):
            up[j & 1].copy_(ring[k % len(ring)], non_blocking=True)
        hop.gather(j, up[j & 1])
        buf = hop.recv(j, stream)
        win[carry[0]:carry[0] + block].copy_(buf, non_blocking=True)
        hop.release(j, stream)
        n = carry[0] + block
        bank.process_device(win, n, stream=stream.cuda_stream)
        used = bank.last_consumed()
        carry[0] = n - used
        assert 0 <= carry[0] <= (1 << 18)
        tail = win[used:n].clone()
        win[:carry[0]].copy_(tail, non_blocking=True)
        bank.drain()
        got = sum(bank.read_audio_all(chans, audio))
        lines = len(wf.feed(full_ring[k & 1].numpy().view(np.complex64).reshape(-1))) if rank == 0 else 0
        return got, lines

    for k in range(4):
        one(k)
    torch.cuda.synchronize()
    dist.barrier()
    busy, n_audio, n_lines, late = [], 0, 0, 0
    period = 1.0 / fps
    t0 = time.perf_counter()
    for k in range(n_blocks):
        s = time.perf_counter()
        deadline = t0 + k * period
        if s < deadline:
            time.sleep(deadline - s)
        elif s - deadline > period:
            late += 1
        s = time.perf_counter()
        a, l = one(k)
        busy.append(time.perf_counter() - s)
        n_audio += a; n_lines += l
    wall = time.perf_counter() - t0
    busy = np.asarray(busy) * 1e3
    stats = torch.tensor([busy.mean(), np.percentile(busy, 99), busy.max(), float(late), n_audio / max(len(chans), 1) / wall], device=dev, dtype=torch.float64)
    allst = [torch.zeros_like(stats) for _ in range(world)]
    dist.all_gather(allst, stats)
    allst = torch.stack(allst).cpu().numpy()
    bank.close()
    if wf is not None:
        wf.close()
    return {"workload": "1024 x 12 kHz channels on %d GPUs (%d each) + 65536-pt %d fps waterfall with noise filter on rank 0, from 61.44 MS/s in %d "
                        "blocks of 1/%d s paced at the true rate; sharded ingest (each rank uploads 1/N), all-gather (%s), audio of every "
                        "channel read on the host" % (world, len(mine), fps, n_blocks, fps, hop.kind),
            "budget_ms_per_block": period * 1e3, "block_ms_mean_max_over_ranks": float(allst[:, 0].max()),
            "block_ms_p99_max_over_ranks": float(allst[:, 1].max()), "block_ms_max_over_ranks": float(allst[:, 2].max()),
            "headroom_x": float(period * 1e3 / allst[:, 0].max()), "late_blocks": int(allst[:, 3].max()),
            "audio_samples_per_channel_per_s_min_over_ranks": float(allst[:, 4].min()), "waterfall_lines_per_s": n_lines / wall, "wall_s": wall}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--headline-only", action="store_true", help="skip the per-config sub-benchmarks (C1, C3, C4, C5 / the paced north-star run)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the audio of the last timed step to DIR/audio.npy (--gpus 1)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.gpus != 1):
        ap.error("--dump-outputs covers the one-GPU workload of --impl ours (--gpus 1)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    # stdout carries exactly ONE JSON line: anything a library prints on fd 1 meanwhile (NCCL's version banner under
    # NCCL_DEBUG=VERSION, ...) is sent to stderr, and the line is written to the real stdout at the end
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    out = io.StringIO()
    with contextlib.redirect_stdout(out):
        if args.impl == "reference":
            run_reference(args)
        else:
            run_ours(args)
    sys.stdout.flush()
    os.dup2(real_stdout, 1)
    os.close(real_stdout)
    sys.stdout.write(out.getvalue())
    sys.stdout.flush()


if __name__ == "__main__":
    main()
