#!/usr/bin/env python
"""Generates the committed golden fixtures.  Needs an OpenWebRX source tree: OWRX_REFERENCE=<path>.

1. params_reference.json — the exact constructor / setter arguments the reference's UNMODIFIED
   csdr.chain classes (FftChain, Selector, Decimator, NFm/Am/Ssb/WFm) hand to pycsdr, captured with a
   recording stub of `pycsdr` (the real extension is not installable here).  This pins the host-side
   parameter math of openwebrx_b200.params / the C ABI to the reference itself.
2. oracle_vectors.npz — small seeded inputs and the CPU oracle's outputs (the oracle is the only
   executable statement of the arithmetic available; see oracle/csdr_oracle.h "PARITY UNPINNED").
"""
import json
import os
import sys
import types
from enum import Enum

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.environ["OWRX_REFERENCE"]        # an OpenWebRX source tree

LOG = []


def _install_recording_stub():
    class Format(Enum):
        CHAR = "char"; SHORT = "short"; FLOAT = "float"; COMPLEX_FLOAT = "complex_float"; COMPLEX_SHORT = "complex_short"

    class AgcProfile(Enum):
        SLOW = "Slow"; FAST = "Fast"

    def enc(v):
        if isinstance(v, Enum):
            return "%s.%s" % (type(v).__name__, v.name)
        if isinstance(v, (int, float, str, bool)) or v is None:
            return v
        return type(v).__name__

    class Base:
        _in = Format.COMPLEX_FLOAT; _out = Format.COMPLEX_FLOAT

        def __init__(self, *a, **k):
            if type(self).__module__ == "pycsdr.modules":
                LOG.append(["ctor", type(self).__name__, [enc(x) for x in a], {kk: enc(v) for kk, v in k.items()}])

        def setReader(self, r): pass
        def setWriter(self, w): pass
        def stop(self): pass
        def getInputFormat(self): return self._in
        def getOutputFormat(self): return self._out

        def __getattr__(self, name):
            if name.startswith("set"):
                def rec(*a, **k):
                    LOG.append(["call", type(self).__name__ + "." + name, [enc(x) for x in a], {kk: enc(v) for kk, v in k.items()}])
                return rec
            raise AttributeError(name)

    class Buffer(Base):
        def __init__(self, fmt=None):
            self.fmt = fmt
        def getReader(self): return Base()
        def getFormat(self): return self.fmt

    mods = types.ModuleType("pycsdr.modules")
    typs = types.ModuleType("pycsdr.types")
    pkg = types.ModuleType("pycsdr")
    typs.Format = Format; typs.AgcProfile = AgcProfile
    F = Format
    fmts = dict(Fft=(F.COMPLEX_FLOAT, F.COMPLEX_FLOAT), LogPower=(F.COMPLEX_FLOAT, F.FLOAT), LogAveragePower=(F.COMPLEX_FLOAT, F.FLOAT),
                FftSwap=(F.FLOAT, F.FLOAT), FftAdpcm=(F.FLOAT, F.CHAR), AmDemod=(F.COMPLEX_FLOAT, F.FLOAT), FmDemod=(F.COMPLEX_FLOAT, F.FLOAT),
                RealPart=(F.COMPLEX_FLOAT, F.FLOAT), DcBlock=(F.FLOAT, F.FLOAT), Limit=(F.FLOAT, F.FLOAT), NfmDeemphasis=(F.FLOAT, F.FLOAT),
                WfmDeemphasis=(F.FLOAT, F.FLOAT), Agc=(F.FLOAT, F.FLOAT))
    names = ["Module", "Reader", "Writer", "TcpSource", "Fft", "LogPower", "LogAveragePower", "FftSwap", "FftAdpcm", "Shift",
             "FirDecimate", "FractionalDecimator", "Bandpass", "Squelch", "AmDemod", "DcBlock", "FmDemod", "Limit",
             "NfmDeemphasis", "WfmDeemphasis", "Agc", "Afc", "RealPart", "Gain", "Convert", "AdpcmEncoder", "AudioResampler",
             "NoiseFilter", "Lowpass", "Downmix", "Throttle", "ExecModule", "SnrSquelch", "TimingRecovery", "DBPskDecoder",
             "VaricodeDecoder", "RttyDecoder", "BaudotDecoder", "MFRttyDecoder", "CwDecoder", "SstvDecoder", "FaxDecoder",
             "SitorBDecoder", "Ccir476Decoder", "DscDecoder", "Ccir493Decoder", "NavtexDecoder", "SmartSquelch"]
    for n in names:
        i, o = fmts.get(n, (F.COMPLEX_FLOAT, F.COMPLEX_FLOAT))
        setattr(mods, n, type(n, (Base,), {"__module__": "pycsdr.modules", "_in": i, "_out": o}))
    mods.Buffer = Buffer
    mods.version = "0.18.36"; mods.csdr_version = "0.18.36"
    pkg.modules = mods; pkg.types = typs
    sys.modules["pycsdr"] = pkg; sys.modules["pycsdr.modules"] = mods; sys.modules["pycsdr.types"] = typs
    return Format, AgcProfile


def capture(fn):
    del LOG[:]
    fn()
    return [list(x) for x in LOG]


def make_params():
    Format, AgcProfile = _install_recording_stub()
    sys.path.insert(0, REF)
    from csdr.chain.fft import FftChain
    from csdr.chain.selector import Selector, Decimator
    out = {"reference": "tildearrow/openwebrx 1.2.97 (owrx/version.py:3)", "fftchain": [], "selector": [], "decimator": []}
    for fs, n, ov, fps in [(2400000, 4096, 0.3, 9), (10000000, 4096, 0.3, 9), (61440000, 65536, 0.3, 30), (12000, 2048, 0.3, 9),
                           (2400000, 4096, 0.0, 9), (2048000, 16384, 0.5, 25), (250000, 256, 0.9, 60)]:
        log = capture(lambda: FftChain(fs, n, ov, fps, "adpcm"))
        avg = [c for c in log if c[0] == "ctor" and c[1] in ("LogAveragePower", "LogPower")][-1]
        every = [c for c in log if c[1] == "Fft.setEveryNSamples"]
        out["fftchain"].append(dict(args=[fs, n, ov, fps], averager=avg[1], avg_number=avg[3].get("avg_number", 0),
                                    every_n_samples=every[-1][2][0] if every else 0, log=log))
    for fs, orate in [(2400000, 12000), (10000000, 12000), (61440000, 12000), (20000000, 250000), (20000000, 12000),
                      (61440000, 250000), (10000000, 48000), (2400000, 11025), (2048000, 44100), (12000, 12000)]:
        log = capture(lambda: Decimator(fs, orate))
        fd = [c for c in log if c[0] == "ctor" and c[1] == "FirDecimate"][-1]
        fr = [c for c in log if c[0] == "ctor" and c[1] == "FractionalDecimator"]
        out["decimator"].append(dict(args=[fs, orate], decimation=fd[2][0], transition=fd[2][1], cutoff=fd[2][2],
                                     fraction=fr[-1][2][1] if fr else 1.0))

    def sel():
        s = Selector(10000000, 12000)
        s.setFrequencyOffset(1234567)
        s.setBandpass(-5999, 5999)
        s.setSquelchLevel(-60)
        s.setBandpass(150, 3000)
        s.setOutputRate(250000)
    out["selector"] = capture(sel)
    with open(os.path.join(HERE, "params_reference.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
    for k in ("pycsdr", "pycsdr.modules", "pycsdr.types"):
        sys.modules.pop(k, None)


def make_vectors():
    sys.path.insert(0, ROOT)
    import oracle
    from openwebrx_b200.synth import carrier_plan, make_iq, BANDPASS
    v = {}
    # waterfall: 1024-pt, avg 4, hop 700 (overlapped), two lines, adpcm + raw dB
    fs = 2.4e6
    cars = carrier_plan(5, fs, seed=101)
    iq = make_iq(700 * 8 + 1024, fs, cars, seed=101)
    r = oracle.fftchain_run(iq, 1024, 700, 4)
    v["wf_iq"] = iq; v["wf_db"] = r["db"]; v["wf_s16"] = r["s16"]; v["wf_adpcm"] = r["lines"]
    # selector: 240 kS/s -> 12 kHz (D = 20, T = 533), NFM / AM / USB, one squelch block + a bit
    fs2 = 240000.0
    cars2 = carrier_plan(3, fs2, seed=102, span=0.35)
    iq2 = make_iq(533 + 20 * (750 * 2 + 30), fs2, cars2, seed=102)
    v["sel_iq"] = iq2
    v["sel_offsets"] = np.array([c["offset"] for c in cars2]); v["sel_kinds"] = np.array([c["kind"] for c in cars2])
    kind = {"nfm": 0, "am": 1, "usb": 2}
    for i, c in enumerate(cars2):
        o = oracle.client_chain_run(iq2, fs2, 12000, c["offset"], BANDPASS[c["kind"]], kind[c["kind"]])
        v["sel_if_%d" % i] = o["if_"]; v["sel_demod_%d" % i] = o["demod"]; v["sel_audio_%d" % i] = o["audio"]
    # audio ADPCM with SYNC framing
    rng = np.random.default_rng(103)
    s16 = (8000 * np.sin(np.arange(5000) * 0.05) + 300 * rng.standard_normal(5000)).astype(np.int16)
    v["au_s16"] = s16; v["au_adpcm"] = oracle.adpcm_sync_encode(s16)
    # spec-defined waterfall noise filter (BASELINE config 4) on the same IQ: three lines so that the floor recurrence runs
    iq3 = make_iq(700 * 12 + 1024, fs, cars, seed=104)
    v["wfnf_iq"] = iq3
    v["wfnf_db"] = oracle.fftchain_run(iq3, 1024, 700, 4, compression="none", noise_filter=(0.9, 0.05, 0.02))["db"]
    # source-side Convert(COMPLEX_SHORT, COMPLEX_FLOAT) + Gain(5.0) (owrx/source/fifi_sdr.py:27-28) and the uint8 form
    raw16 = rng.integers(-32768, 32768, 512, dtype=np.int16)
    raw8 = rng.integers(0, 256, 512, dtype=np.uint8)
    v["raw_cs16"] = raw16; v["raw_cs16_cf"] = oracle.convert_raw_iq(raw16, "cs16", 5.0)
    v["raw_cu8"] = raw8; v["raw_cu8_cf"] = oracle.convert_raw_iq(raw8, "cu8", 1.0)
    np.savez_compressed(os.path.join(HERE, "oracle_vectors.npz"), **v)


if __name__ == "__main__":
    make_params()
    make_vectors()
    print("wrote", os.listdir(HERE))
