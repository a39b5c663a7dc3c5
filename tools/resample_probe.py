#!/usr/bin/env python
"""Cost of the client-audio resampler at the C2 shape: 10 MS/s -> 12 kHz, 64 channels in one group, 2^24-sample device blocks,
every channel's audio as ADPCM (AdpcmEncoder(sync=True)), with 0, 21 and 64 channels at 12000 -> 11025 (a 44.1 kHz sound card)
and 16 channels at 12000 -> 48000 (HD audio).  Every step is process_device (pipelined) followed by the split-phase drain, as a
streaming host runs it; the cases run twice in mirrored order to show the spread.  One JSON line per run: wall ms per step (host
clock around steps that end in a synchronise), the resample kernel's device ms per step (CUDA events around its launches, in a
separate profiled run), kernel launches per step, and the card's name and power limit."""
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench                                                             # noqa: E402
from openwebrx_b200 import _native as N                                 # noqa: E402


def run(blocks, cars, n_rs, ratio, steps, profile, warmup=4):
    bank, chans = bench.make_bank(bench.C2, cars, 0)
    bank.set_outputs(N.OUT_AUDIO)
    for i, ch in enumerate(chans):
        ch.setAudioFormat("adpcm")
        if i < n_rs:
            ch.set_audio_resampler(*ratio)
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
        ch.read_bytes()
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
    out_bytes = sum(len(ch.read_bytes()) for ch in chans) / steps
    bank.close()
    r = dict(resampled=n_rs, ratio="%d->%d" % ratio if n_rs else None, steps=steps, profiled=profile,
             launches_per_step=launches, client_bytes_per_step=int(out_bytes))
    if profile:
        r["resample_kernel_ms_per_step"] = round(prof["resample"][0] / steps, 4)
        r["resample_launches_per_step"] = prof["resample"][1] / steps
    else:
        r["wall_ms_per_step"] = round(wall, 3)
    return r


if __name__ == "__main__":
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
    cases = [(0, (12000, 11025)), (21, (12000, 11025)), (64, (12000, 11025)), (16, (12000, 48000))]
    for k, ratio in cases + cases[::-1]:
        r = run(blocks, cars, k, ratio, steps, profile=False)
        r["gpu"] = gpu
        print(json.dumps(r), flush=True)
    for k, ratio in cases[1:]:
        r = run(blocks, cars, k, ratio, steps, profile=True)
        r["gpu"] = gpu
        print(json.dumps(r), flush=True)
