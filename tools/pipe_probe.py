#!/usr/bin/env python
"""Stage times of the C2 device path with the three-stream pipeline on and off (each stage's own CUDA-event bracket):
off = every stage alone on the GPU, on = what the stages cost while they overlap.  One JSON line per run; the environment
selects the kernel variants (OWRX_TAIL_FUSED, OWRX_AGC_PAD_KB, ...), so A/B runs are separate invocations."""
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench                                                             # noqa: E402


def run(pipelined, blocks, cars, steps=30):
    bank, _ = bench.make_bank(bench.C2, cars, 0)
    st = torch.cuda.Stream(priority=int(os.environ.get("PROBE_STREAM_PRIORITY", "0")))
    torch.cuda.set_stream(st)
    bank.set_pipelined(pipelined)
    for i in range(3):
        bank.process_device(blocks[i & 1], bench.BLOCK, stream=st.cuda_stream)
    bank.join(st.cuda_stream); st.synchronize()
    bank.profile(True); bank.profile_read_ex(reset=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for i in range(steps):
        bank.process_device(blocks[i & 1], bench.BLOCK, stream=st.cuda_stream)
    bank.join(st.cuda_stream)
    e1.record(st); st.synchronize()
    prof = {k: round(v[0] / max(v[1], 1), 4) for k, v in bank.profile_read_ex().items() if v[1]}
    bank.profile(False)
    bank.close()
    return dict(pipelined=pipelined, ms_per_block=round(e0.elapsed_time(e1) / steps, 4), stages_ms=prof)


if __name__ == "__main__":
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    cars = bench.channel_plan(0, 64)
    iq = bench.synth_iq_torch(bench.BLOCK, bench.C2["fs"], cars, dev)
    blocks = [iq, iq.clone()]
    env = {k: v for k, v in os.environ.items() if k.startswith("OWRX_") or k.startswith("PROBE_")}
    print(json.dumps({"env": env, "alone": run(False, blocks, cars), "pipelined": run(True, blocks, cars)}))
