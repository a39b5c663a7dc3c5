#!/usr/bin/env python
"""Times the waterfall FftChain on one GPU, device-resident (CUDA events, inputs far beyond L2):
  wf_probe.py c1 [lines]     2.4 MS/s, 4096-pt, 9 fps   (avg 93, hop 2867)        default 592 lines
  wf_probe.py c4 [lines]     61.44 MS/s, 65536-pt, 30 fps (avg 45, hop 45511)      default 128 lines
Reports the whole chain with ADPCM (pipelined side-stream encoder) and with compression "none" (FFT + finalize only),
each as ms per batch, lines/s and the fraction of the measured HBM peak on SURVEY 8(d)'s algorithmic bytes (8 U + out per line)."""
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench                                                             # noqa: E402
from openwebrx_b200 import Waterfall, fftchain_params                   # noqa: E402

SHAPES = {"c1": (2.4e6, 4096, 9, 0.3, 592), "c4": (61.44e6, 65536, 30, 0.3, 128)}


def run(which, lines, steps=5):
    fs, n, fps, ov, _ = SHAPES[which]
    dev = torch.device("cuda", 0)
    hbm, _, _ = bench.load_peaks()
    avg, every_n = fftchain_params(fs, n, ov, fps)
    ns = every_n * avg * lines + n
    g = torch.Generator(device=dev); g.manual_seed(7)
    iq = 1e-3 * torch.randn(ns, 2, device=dev, generator=g, dtype=torch.float32)
    tt = torch.arange(ns, device=dev, dtype=torch.float32)
    iq[:, 0] += 0.3 * torch.cos(0.7 * tt); iq[:, 1] += 0.3 * torch.sin(0.7 * tt)
    del tt
    st = torch.cuda.Stream(device=dev)
    out = {"shape": which, "lines": lines, "avg": avg, "every_n": every_n, "input_GB": ns * 8 / 1e9}
    for comp in ("adpcm", "none"):
        wf = Waterfall(fs, n, ov, fps, comp, device=0)
        buf = torch.empty(lines * wf.line_bytes, dtype=torch.uint8, device=dev)
        wf.set_pipelined(comp == "adpcm")
        torch.cuda.synchronize()
        for _ in range(3):
            wf.process_device(iq, ns, buf, buf.numel(), stream=st.cuda_stream)
        wf.join(st.cuda_stream); st.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        for _ in range(steps):
            got = wf.process_device(iq, ns, buf, buf.numel(), stream=st.cuda_stream)
        wf.join(st.cuda_stream)
        e1.record(st); st.synchronize()
        ms = e0.elapsed_time(e1) / steps
        unique = 8.0 * ((avg - 1) * every_n + n) + wf.line_bytes
        gbs = unique * got / (ms * 1e-3) / 1e9
        out[comp] = {"ms_per_batch": ms, "lines_per_s": got / (ms * 1e-3), "hbm_GBps": gbs, "hbm_frac": gbs / hbm,
                     "ns_per_fft_4096": ms * 1e6 / (got * avg * max(1, n // 4096))}
        wf.close()
    return out


if __name__ == "__main__":
    which = sys.argv[1] if len(sys.argv) > 1 else "c1"
    lines = int(sys.argv[2]) if len(sys.argv) > 2 else SHAPES[which][4]
    print(json.dumps(run(which, lines)))
