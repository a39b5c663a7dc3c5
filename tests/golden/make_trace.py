#!/usr/bin/env python
"""Records the pycsdr call sequences of the reference's own, UNMODIFIED callers of the hot path and commits them as
fixtures (tests/golden/trace_*.json).  Needs an OpenWebRX source tree: OWRX_REFERENCE=<path>.  A GPU run replays the
fixtures (tests/test_gpu_trace_replay.py) with IQ flowing between the recorded steps.

  trace_spectrum.json  owrx/fft.py:13-109     SpectrumThread(sdrSource).start(), then the on-the-fly property changes
                                             (fft_fps, fft_compression) it wires to FftChain (csdr/chain/fft.py:25-96)
  trace_client.json    owrx/dsp.py:437-937    DspManager(handler, sdrSource) — which builds ClientDemodulatorChain
                                             (owrx/dsp.py:39-94) — .start(), then the property updates a browser sends:
                                             offset_freq, low_cut/high_cut, squelch_level, mod = am / usb / wfm / nfm
                                             (stopDemodulator + setDemodulator, :96-148), the secondary FFT on selectorBuffer
                                             (:220-225) and a SecondarySelector on the same buffer (:188-207,
                                             csdr/chain/selector.py:217-244)

How: the repo's `pycsdr` shim IS the pycsdr the reference imports; every constructor and every wiring / control method of
its classes is wrapped by a logger that names objects in creation order.  Data-path calls (read / write) are not logged.
What the reference does next can depend on what pycsdr answers (ValueError on a format mismatch, owrx/fft.py:61-68): the
answers here are the shim's own, the same ones the replay gets."""
import json
import os
import sys
import tempfile
import threading
from enum import Enum

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.environ["OWRX_REFERENCE"]        # an OpenWebRX source tree
sys.path.insert(0, ROOT)
sys.path.insert(0, REF)

import pycsdr.modules as M                      # noqa: E402
from pycsdr.types import AgcProfile, Format     # noqa: E402

LOG = []
IDS = {}
COUNT = {"b": 0, "r": 0, "m": 0}
MAIN = threading.get_ident()
WRAPPED = ("setReader", "setWriter", "stop", "resume", "getReader")


def _oid(obj, create=False):
    k = id(obj)
    if k not in IDS:
        if not create:
            return None
        p = "b" if isinstance(obj, M.Buffer) else ("r" if isinstance(obj, M.Reader) else "m")
        IDS[k] = "%s%d" % (p, COUNT[p])
        COUNT[p] += 1
        _KEEP.append(obj)                        # ids are object addresses: keep every named object alive
    return IDS[k]


_KEEP = []


def _enc(v):
    if isinstance(v, Format):
        return {"format": v.name}
    if isinstance(v, AgcProfile):
        return {"agc": v.name}
    if isinstance(v, Enum):
        return {"enum": "%s.%s" % (type(v).__name__, v.name)}
    if isinstance(v, (bool, int, float, str)) or v is None:
        return v
    oid = _oid(v)
    if oid is not None:
        return {"ref": oid}
    return {"foreign": type(v).__name__}


_DEPTH = threading.local()


def _enter():
    d = getattr(_DEPTH, "d", 0)
    _DEPTH.d = d + 1
    return d


def _leave():
    _DEPTH.d -= 1


def _wrap_class(cls):
    """log constructors and wiring / control methods, but only the OUTERMOST call on the main thread: what the reference
    itself calls, not what the shim calls internally while serving it (super().__init__, the runner's own getReader...)"""
    if "__init__" in vars(cls):
        orig_init = cls.__init__

        def init(self, *a, __orig=orig_init, **k):
            depth = _enter()
            try:
                __orig(self, *a, **k)
            finally:
                _leave()
            # only pycsdr's own classes are pycsdr objects: the reference subclasses Module for its Python chains
            if depth == 0 and type(self).__module__ == "pycsdr.modules" and threading.get_ident() == MAIN and _oid(self) is None \
                    and not isinstance(self, M.Reader):          # a Reader is named by the getReader() call that made it
                LOG.append({"op": "new", "id": _oid(self, True), "cls": type(self).__name__, "args": [_enc(x) for x in a],
                            "kwargs": {kk: _enc(v) for kk, v in k.items()}})
        cls.__init__ = init
    for name, fn in list(vars(cls).items()):
        if not callable(fn) or not (name in WRAPPED or (name.startswith("set") and name[3:4].isupper())):
            continue

        def method(self, *a, __orig=fn, __name=name, **k):
            depth = _enter()
            ent = None
            if depth == 0 and type(self).__module__ == "pycsdr.modules" and threading.get_ident() == MAIN and _oid(self) is not None:
                ent = {"op": "call", "id": _oid(self), "method": __name, "args": [_enc(x) for x in a],
                       "kwargs": {kk: _enc(v) for kk, v in k.items()}}
                LOG.append(ent)
            try:
                ret = __orig(self, *a, **k)
            except Exception as e:
                if ent is not None:
                    ent["raises"] = type(e).__name__
                raise
            finally:
                _leave()
            if ent is not None and isinstance(ret, M.Reader):
                ent["ret"] = _oid(ret, True)
            return ret
        setattr(cls, name, method)


def install():
    seen = set()
    for name, obj in list(vars(M).items()):
        if isinstance(obj, type) and obj.__module__ == "pycsdr.modules" and obj not in seen and not name.startswith("_"):
            seen.add(obj)
            _wrap_class(obj)
    _wrap_class(M._Stage)
    _wrap_class(M._Unfused)


def mark(name, **info):
    LOG.append({"op": "mark", "name": name, **info})


def take():
    out = list(LOG)
    del LOG[:]
    return out


# ---------------------------------------------------------------- the reference's environment, faked at its own interfaces
def _reference_config():
    from pathlib import Path
    d = tempfile.mkdtemp(prefix="owrx_trace_")
    conf = os.path.join(d, "openwebrx.conf")
    with open(conf, "w") as f:
        f.write("[core]\ndata_directory = %s\ntemporary_directory = %s\n" % (d, d))
    from owrx.config.core import CoreConfig
    CoreConfig.load(Path(conf))
    from owrx.config import Config
    return Config.get()


class FakeSdrSource:
    """what SpectrumThread / DspManager touch of owrx.source.SdrSource (owrx/source/__init__.py:301-330,462,510-527,564)"""

    def __init__(self, props, buffer):
        self.props = props
        self.buffer = buffer
        self.spectrum = []
        self.clients = []

    def getProps(self):
        return self.props

    def addClient(self, c):
        self.clients.append(c)

    def removeClient(self, c):
        if c in self.clients:
            self.clients.remove(c)

    def isAvailable(self):
        return True

    def getBuffer(self):
        return self.buffer

    def writeSpectrumData(self, data):
        self.spectrum.append(bytes(data))


class FakeHandler:
    """the websocket connection's writer methods (owrx/connection.py:473-489)"""

    def __getattr__(self, name):
        if name.startswith("write_"):
            return lambda *a, **k: None
        raise AttributeError(name)


def record_spectrum():
    from owrx.property import PropertyLayer
    from owrx.fft import SpectrumThread
    src = M.Buffer(Format.COMPLEX_FLOAT)
    take()
    props = PropertyLayer(samp_rate=2400000, fft_size=4096, fft_fps=9, fft_voverlap_factor=0.3, fft_compression="adpcm")
    sdr = FakeSdrSource(props, src)
    st = SpectrumThread(sdr)
    st.start()
    mark("start", source=_oid(src), output=_oid(st.reader), fs=2400000, n=4096, avg=93, every_n=2867, compression="adpcm")
    props["fft_fps"] = 30
    mark("fps30", source=_oid(src), output=_oid(st.reader), fs=2400000, n=4096, avg=28, every_n=2857, compression="adpcm")
    props["fft_compression"] = "none"
    mark("uncompressed", source=_oid(src), output=_oid(st.reader), fs=2400000, n=4096, avg=28, every_n=2857, compression="none")
    props["fft_size"] = 1024                    # restart(): stop() + start() with a new FftChain (owrx/fft.py:52,90-92)
    avg = int(round(2400000 / 1024 / 30 / (1.0 - 0.3)))
    mark("size1024", source=_oid(src), output=_oid(st.reader), fs=2400000, n=1024, avg=avg, every_n=int(2400000 / 30 / avg),
         compression="none")
    st.stop()
    mark("stopped")
    return {"source": _oid(src), "events": take(),
            "recorded_from": "owrx/fft.py:13-109 SpectrumThread on a fake SdrSource (samp_rate 2.4 MS/s, fft_size 4096, fft_fps 9, "
                             "fft_voverlap_factor 0.3, fft_compression adpcm)"}


def record_client():
    from owrx.property import PropertyLayer, PropertyStack
    from owrx.dsp import DspManager
    from csdr.chain.selector import SecondarySelector
    from owrx.config import Config
    cfg = Config.get()
    fs = 2400000
    src = M.Buffer(Format.COMPLEX_FLOAT)
    take()
    stack = PropertyStack()
    stack.addLayer(0, PropertyLayer(samp_rate=fs, center_freq=145000000, start_mod="nfm", start_freq=145000000 + 250000))
    stack.addLayer(1, cfg)
    sdr = FakeSdrSource(stack, src)
    dsp = DspManager(FakeHandler(), sdr)
    dsp.start()

    def state(name, **kw):
        tags = {t: _oid(r) for t, r in dsp.readers.items()}
        mark(name, source=_oid(src), readers=tags, fs=fs, **kw)

    state("nfm_start", demod="nfm", out_rate=12000, offset=250000, bandpass=[-5999, 5999], squelch_db=-150, audio="adpcm")
    dsp.setProperties({"offset_freq": -321000, "low_cut": -5999, "high_cut": 5999})
    state("nfm_retuned", demod="nfm", out_rate=12000, offset=-321000, bandpass=[-5999, 5999], squelch_db=-150, audio="adpcm")
    dsp.setProperties({"squelch_level": -20})
    state("nfm_squelched", demod="nfm", out_rate=12000, offset=-321000, bandpass=[-5999, 5999], squelch_db=-20, audio="adpcm")
    dsp.setProperties({"squelch_level": -150, "mod": "am", "low_cut": -4700, "high_cut": 4700})
    state("am", demod="am", out_rate=12000, offset=-321000, bandpass=[-4700, 4700], squelch_db=-150, audio="adpcm")
    dsp.setProperties({"mod": "usb", "low_cut": 150, "high_cut": 3000, "offset_freq": 600000})
    state("usb", demod="usb", out_rate=12000, offset=600000, bandpass=[150, 3000], squelch_db=-150, audio="adpcm", agc="fast")
    # secondary FFT on the shared selectorBuffer: what setSecondaryDemodulator does for modes with isSecondaryFftShown()
    # (owrx/dsp.py:215-225) — the digital decoders behind those modes are outside the hot path, the FFT chain is not
    dsp.chain._createSecondaryFftChain()
    dsp.chain.secondaryFftChain.setSampleRate(dsp.chain._getSelectorOutputRate())
    # and a SecondarySelector on the same buffer, wired as owrx/dsp.py:188-207 does
    sec = SecondarySelector(12000, 500)
    sec.setReader(dsp.chain.selectorBuffer.getReader())
    sec.setFrequencyOffset(1000)
    sec_out = M.Buffer(Format.COMPLEX_FLOAT)
    sec.setWriter(sec_out)
    sec_reader = sec_out.getReader()
    state("usb_secondary", demod="usb", out_rate=12000, offset=600000, bandpass=[150, 3000], squelch_db=-150, audio="adpcm", agc="fast",
          secondary_fft=dict(n=2048, avg=1, every_n=1333, compression="adpcm"),
          secondary_selector=dict(offset=1000, bandwidth=500, output=_oid(sec_reader)))
    sec.stop()
    dsp.chain.secondaryFftChain.stop()
    dsp.chain.secondaryFftChain = None
    dsp.setProperties({"mod": "wfm", "low_cut": -75000, "high_cut": 75000, "offset_freq": 100000})
    state("wfm", demod="wfm", out_rate=250000, offset=100000, bandpass=[-75000, 75000], squelch_db=-150, audio="adpcm", hd=True,
          audio_rate=48000, tau=50e-6)
    dsp.setProperties({"mod": "nfm", "low_cut": -4000, "high_cut": 4000})
    state("nfm_again", demod="nfm", out_rate=12000, offset=100000, bandpass=[-4000, 4000], squelch_db=-150, audio="adpcm")
    dsp.stop()
    mark("stopped")
    return {"source": _oid(src), "events": take(),
            "recorded_from": "owrx/dsp.py:437-937 DspManager (-> ClientDemodulatorChain :39-425) on a fake SdrSource / connection handler "
                             "(samp_rate 2.4 MS/s, start_mod nfm, default config), driven through setProperties like owrx/connection.py:438"}


def main():
    install()
    _reference_config()
    for name, fn in (("trace_spectrum.json", record_spectrum), ("trace_client.json", record_client)):
        tr = fn()
        tr["reference"] = "tildearrow/openwebrx 1.2.97"
        with open(os.path.join(HERE, name), "w") as f:
            json.dump(tr, f, indent=0)
        ops = [e for e in tr["events"] if e["op"] != "mark"]
        print(name, len(tr["events"]), "events,", len(ops), "pycsdr calls,", [e["name"] for e in tr["events"] if e["op"] == "mark"])
    os._exit(0)                                  # pump threads of the reference block in read(); nothing to wait for


if __name__ == "__main__":
    main()
