#!/usr/bin/env python
"""Cost of the demodulated-audio tap at the C2 step: 10 MS/s -> 12 kHz, 64 channels in one group, 2^24-sample device blocks,
every channel's client audio as ADPCM (AdpcmEncoder(sync=True)), with 0, 8 and 64 channels tapped as S16 (what a WSJT-style
decoder reads).  Every step is process_device (pipelined) followed by the split-phase drain, as a streaming host runs it; the
cases run twice in mirrored order to show the spread.  One JSON line per run: wall ms per step (host clock around steps that
end in a synchronise), the gather kernel's device ms per step (CUDA events around its launches, in a separate profiled run),
kernel launches per step, the tap's D2H bytes per step (the S16 samples delivered), and the card's name and power limit.

usage: tools/audio_tap_probe.py [out.jsonl]   (default profiles/r3_audio_tap_probe.jsonl)"""
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench                                                             # noqa: E402
from openwebrx_b200 import _native as N                                 # noqa: E402


def run(blocks, cars, n_tap, steps, profile, warmup=4):
    bank, chans = bench.make_bank(bench.C2, cars, 0)
    bank.set_outputs(N.OUT_AUDIO)
    for i, ch in enumerate(chans):
        ch.setAudioFormat("adpcm")
        if i < n_tap:
            ch.set_audio_tap("s16")
    st = torch.cuda.Stream()
    sp = st.cuda_stream
    bank.set_pipelined(True)
    n = bench.C2["block"]

    def step(i):
        bank.process_device(blocks[i & 1], n, stream=sp)
        bank.drain_begin()
        bank.drain_end()
    for i in range(warmup):
        step(i)
    bank.join(sp); st.synchronize()
    for ch in chans:
        ch.read_bytes(); ch.read_audio_tap()
    bank.profile(profile)
    bank.profile_read_ex(reset=True)
    l0 = N.lib.owrx_launch_count()
    t0 = time.perf_counter()
    for i in range(steps):
        step(i)
    bank.join(sp); st.synchronize()
    wall = (time.perf_counter() - t0) * 1e3 / steps
    launches = (N.lib.owrx_launch_count() - l0) / steps
    prof = bank.profile_read_ex(reset=True)
    tap_bytes = sum(2 * len(ch.read_audio_tap()) for ch in chans) / steps
    bank.close()
    r = dict(tapped_s16=n_tap, steps=steps, profiled=profile, launches_per_step=launches, tap_d2h_bytes_per_step=int(tap_bytes))
    if profile:
        r["gather_kernel_ms_per_step"] = round(prof["tap"][0] / steps, 4)
        r["gather_launches_per_step"] = prof["tap"][1] / steps
    else:
        r["wall_ms_per_step"] = round(wall, 3)
    return r


if __name__ == "__main__":
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r3_audio_tap_probe.jsonl")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    steps = int(os.environ.get("PROBE_STEPS", "20"))
    cars = bench.channel_plan(0, 64)
    iq = bench.synth_iq_torch(bench.C2["block"], bench.C2["fs"], cars, dev)
    blocks = [iq, iq.clone()]
    try:
        gpu = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        gpu = torch.cuda.get_device_name(0)
    cases = [0, 8, 64]
    with open(out, "w") as f:
        for k, prof in [(k, False) for k in cases + cases[::-1]] + [(k, True) for k in cases[1:]]:
            r = run(blocks, cars, k, steps, profile=prof)
            r["gpu"] = gpu
            line = json.dumps(r)
            print(line, flush=True)
            f.write(line + "\n")
