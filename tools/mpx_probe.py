#!/usr/bin/env python
"""Cost of the WFM multiplex tap at the C5 shape: 20 MS/s -> 250 kHz IF, 128 WFM channels in one group, 2^23-sample device
blocks, with 0, 8 and 128 channels tapped (S16, what the RDS path reads).  Every step is process_device (pipelined) followed by
the split-phase drain, as a streaming host runs it; the cases run twice in mirrored order to show the spread.  One JSON line per
run: wall ms per step (host clock around steps that end in a synchronise), tap D2H bytes per step, kernel launches per step."""
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench                                                             # noqa: E402
from openwebrx_b200 import _native as N                                 # noqa: E402


def run(blocks, cars, tapped, steps, warmup=4):
    bank, chans = bench.make_bank(bench.C5, cars, 0)
    bank.set_outputs(N.OUT_AUDIO)
    for ch in chans[:tapped]:
        ch.set_mpx("s16")
    st = torch.cuda.Stream()
    sp = st.cuda_stream
    bank.set_pipelined(True)
    n = bench.C5["block"]

    def step(i):
        bank.process_device(blocks[i & 1], n, stream=sp)
        bank.drain_begin()
        bank.drain_end()
    for i in range(warmup):
        step(i)
    bank.join(sp); st.synchronize()
    for ch in chans[:tapped]:
        ch.read_mpx()
    l0 = N.lib.owrx_launch_count()
    t0 = time.perf_counter()
    for i in range(steps):
        step(i)
    bank.join(sp); st.synchronize()
    wall = (time.perf_counter() - t0) * 1e3 / steps
    launches = (N.lib.owrx_launch_count() - l0) / steps
    tap_bytes = sum(ch.read_mpx().nbytes for ch in chans[:tapped]) / steps
    bank.close()
    return dict(tapped=tapped, format="s16", steps=steps, wall_ms_per_step=round(wall, 3), tap_d2h_bytes_per_step=int(tap_bytes),
                launches_per_step=launches)


if __name__ == "__main__":
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    steps = int(os.environ.get("PROBE_STEPS", "20"))
    cars = bench.channel_plan(0, 128, fs=bench.C5["fs"], wfm=True)
    iq = bench.synth_iq_torch(bench.C5["block"], bench.C5["fs"], cars, dev)
    blocks = [iq, iq.clone()]
    try:
        gpu = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        gpu = torch.cuda.get_device_name(0)
    for k in (0, 8, 128, 128, 8, 0):
        r = run(blocks, cars, k, steps)
        r["gpu"] = gpu
        print(json.dumps(r), flush=True)
