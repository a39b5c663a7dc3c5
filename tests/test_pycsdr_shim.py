"""CPU tests of the drop-in `pycsdr` package: Buffer/Reader semantics, the module API surface the
reference uses (SURVEY 8b, Appendix C/D), and chain discovery on chains built by the reference's own
UNMODIFIED classes when the environment variable OWRX_REFERENCE names an OpenWebRX source tree."""
import os
import sys
import threading
import time
from abc import ABCMeta

import numpy as np
import pytest

import pycsdr.modules as M
from pycsdr.types import AgcProfile, Format

REF = os.environ.get("OWRX_REFERENCE", "")
HAVE_REF = bool(REF) and os.path.isdir(os.path.join(REF, "csdr", "chain"))
NO_REF = "needs an OpenWebRX source tree named by OWRX_REFERENCE"


def test_buffer_multi_reader_and_stop():
    b = M.Buffer(Format.FLOAT)
    r1, r2 = b.getReader(), b.getReader()
    b.write(b"\x01\x02\x03\x04")
    b.write(bytearray(b"\x05\x06\x07\x08"))
    d1 = r1._read(True)                                 # internal: everything that has arrived
    assert bytes(d1) == b"\x01\x02\x03\x04\x05\x06\x07\x08" and len(d1) == 8
    assert b"\x02" + d1 == b"\x02" + bytes(d1) and d1.tobytes()[:2] == b"\x01\x02"       # owrx/connection.py:475 usage
    assert bytes(r2.read()) == b"\x01\x02\x03\x04"    # independent cursor; public read() = one write unit
    assert bytes(r2.read()) == b"\x05\x06\x07\x08"
    r3 = b.getReader()                                  # late reader only sees new data
    got = []
    t = threading.Thread(target=lambda: got.append(r3.read()))
    t.start()
    time.sleep(0.05)
    assert t.is_alive()                                 # blocked
    r3.stop()                                           # stop() wakes a blocked read(), which returns None
    t.join(2)
    assert not t.is_alive() and got == [None]
    r3.resume()
    b.write(b"abcd")
    assert bytes(r3.read()) == b"abcd"
    assert b.getFormat() is Format.FLOAT and isinstance(b, M.Writer)
    with pytest.raises(ValueError):
        M.Buffer("float")


def test_module_base_is_subclassable_like_the_reference_does():
    class Mod(M.Module, metaclass=ABCMeta):             # csdr/module/__init__.py:16-20
        def __init__(self):
            self.reader = None
            super().__init__()

    class ThreadMod(Mod, threading.Thread):             # csdr/module/__init__.py:74-78
        def __init__(self):
            super().__init__()

    m = Mod()
    m.stop()                                            # inherited no-op stop (owrx/dsp.py:143)
    ThreadMod()


def test_constructor_signatures_recorded_in_survey_appendix_d():
    f = M.Fft(size=4096, every_n_samples=0); f.setEveryNSamples(2867)
    M.LogPower(add_db=-70); M.LogAveragePower(add_db=-70, fft_size=4096, avg_number=93)
    M.FftSwap(fft_size=4096); M.FftAdpcm(fft_size=4096); M.FftAdpcm(4096)
    s = M.Shift(0.0); s.setRate(-0.1234567)
    M.FirDecimate(833, 0.00017999999999999998, 0.49979999999999997)
    M.FractionalDecimator(Format.COMPLEX_FLOAT, 1.0004001600640255)
    M.FractionalDecimator(Format.FLOAT, 5.208333333333333, prefilter=True)
    bp = M.Bandpass(transition=0.02666666666666667, use_fft=True); bp.setBandpass(-0.49, 0.49)
    bp2 = M.Bandpass(-0.1, 0.1, 0.1, use_fft=True)
    assert (bp2.low, bp2.high, bp2.transition) == (-0.1, 0.1, 0.1)
    sq = M.Squelch(Format.COMPLEX_FLOAT, length=750, decimation=5, hangLength=1500, flushLength=3750, reportInterval=4)
    assert sq.level == 0.0                               # default must be "open" (SURVEY 8b item 6)
    sq.setSquelchLevel(1e-6); sq.setPowerWriter(M.Buffer(Format.FLOAT))
    a = M.Agc(Format.FLOAT); a.setProfile(AgcProfile.SLOW); a.setInitialGain(200); a.setMaxGain(3)
    assert AgcProfile("Fast") is AgcProfile.FAST         # owrx/dsp.py:619
    M.AmDemod(); M.DcBlock(); M.FmDemod(); M.Limit(); M.NfmDeemphasis(12000); M.WfmDeemphasis(48000, 5e-05); M.RealPart()
    M.Convert(Format.FLOAT, Format.SHORT); M.AdpcmEncoder(sync=True); M.AudioResampler(48000, 12000); M.Gain(Format.FLOAT, 100.0)
    assert M.version >= "0.18.0" and M.csdr_version >= "0.18.0"
    for name in ("Afc", "NoiseFilter", "Lowpass", "Downmix", "Throttle", "ExecModule", "SnrSquelch", "TimingRecovery",
                 "DBPskDecoder", "VaricodeDecoder", "RttyDecoder", "BaudotDecoder", "MFRttyDecoder", "CwDecoder", "SstvDecoder",
                 "FaxDecoder", "SitorBDecoder", "Ccir476Decoder", "DscDecoder", "Ccir493Decoder", "NavtexDecoder", "TcpSource",
                 "Reader", "Writer", "Buffer", "Module"):
        assert hasattr(M, name), name
    with pytest.raises(NotImplementedError):
        M.CwDecoder(12000)


def test_format_mismatch_raises_valueerror():
    swap = M.FftSwap(fft_size=1024)
    with pytest.raises(ValueError):
        swap.setWriter(M.Buffer(Format.CHAR))           # owrx/fft.py:64-71 relies on this
    with pytest.raises(ValueError):
        swap.setReader(M.Buffer(Format.COMPLEX_FLOAT).getReader())
    swap.setWriter(M.Buffer(Format.FLOAT))


def _connect(workers):
    """the reference's Chain._connect pattern (csdr/chain/__init__.py:21-25), restated locally"""
    for a, b in zip(workers[:-1], workers[1:]):
        buf = M.Buffer(a.getOutputFormat())
        a.setWriter(buf)
        b.setReader(buf.getReader())


def test_chain_discovery_without_gpu():
    agc = M.Agc(Format.FLOAT); agc.setProfile(AgcProfile.SLOW); agc.setMaxGain(3)
    ws = [M.Shift(0.0), M.FirDecimate(200, 0.00075, 0.5), M.Bandpass(transition=320.0 / 12000, use_fft=True),
          M.Squelch(Format.COMPLEX_FLOAT, length=750, decimation=5, hangLength=1500, flushLength=3750, reportInterval=4),
          M.FmDemod(), M.Limit(), M.NfmDeemphasis(12000), agc, M.Convert(Format.FLOAT, Format.SHORT), M.AdpcmEncoder(sync=True)]
    _connect(ws)
    ws[-1].setWriter(M.Buffer(Format.CHAR))
    chain, links = M._walk(ws[0])
    assert chain == ws and len(links) == len(ws) - 1
    d = M._ChannelPlan.match(chain)
    assert d and d["demod"] == "nfm" and d["audio_fmt"] == "adpcm" and d["tail"] is ws[-1] and d["squelch"] is ws[3]
    ws[5].stop()                                         # a stopped stage breaks the chain (Chain.replace stops old workers)
    chain2, _ = M._walk(ws[0])
    assert len(chain2) == 5 and M._ChannelPlan.match(chain2) is None
    wf = [M.Fft(size=1024, every_n_samples=700), M.LogAveragePower(add_db=-70, fft_size=1024, avg_number=4), M.FftSwap(fft_size=1024)]
    _connect(wf)
    assert M._WaterfallPlan.match(M._walk(wf[0])[0]) is None          # no writer yet: incomplete, not an error
    wf[-1].setWriter(M.Buffer(Format.FLOAT))
    assert len(M._WaterfallPlan.match(M._walk(wf[0])[0])) == 3


@pytest.mark.skipif(not HAVE_REF, reason=NO_REF)
def test_reference_classes_run_unmodified_on_the_shim():
    sys.path.insert(0, REF)
    try:
        from csdr.chain.fft import FftChain
        from csdr.chain.selector import Selector
        from csdr.chain.analog import Am, NFm, Ssb, WFm
        from csdr.chain.clientaudio import ClientAudioChain
        from csdr.chain import Chain
        fc = FftChain(2400000, 4096, 0.3, 9, "adpcm")
        src = M.Buffer(Format.COMPLEX_FLOAT)
        fc.setReader(src.getReader())
        out = M.Buffer(Format.CHAR)
        fc.setWriter(out)
        m = M._WaterfallPlan.match(M._walk(fc.fft)[0])
        assert m and len(m) == 4 and m[0].every_n_samples == 2867 and m[1].avg_number == 93
        fc.setFps(30)                                     # replaces the averager, re-attaches the same Reader object
        m = M._WaterfallPlan.match(M._walk(fc.fft)[0])
        assert m and m[1].avg_number == 28 and m[0].every_n_samples == 2857
        with pytest.raises(ValueError):                   # owrx/fft.py:61-68 expects and swallows this
            fc.setCompression("none")
        out2 = M.Buffer(fc.getOutputFormat())
        fc.setWriter(out2)
        assert len(M._WaterfallPlan.match(M._walk(fc.fft)[0])) == 3
        # a whole client chain as owrx/dsp.py:39-72 builds it
        for demod, name, fmt in ((NFm(12000), "nfm", "adpcm"), (Am(), "am", "adpcm"), (Ssb(AgcProfile("Fast")), "ssb", "adpcm")):
            sel = Selector(10000000, 12000)
            audio = ClientAudioChain(demod.getOutputFormat(), 12000, 12000, "adpcm", False, 0)
            chain = Chain([sel, demod, audio])
            sel.setBandpass(-5999, 5999)
            sel.setFrequencyOffset(1234567)
            chain.setReader(src.getReader())
            chain.setWriter(M.Buffer(Format.CHAR))
            d = M._ChannelPlan.match(M._walk(sel.shift)[0])
            assert d and d["demod"] == name and d["audio_fmt"] == fmt and d["frac"] is not None and d["bandpass"].low == -5999 / 12000
            assert d["shift"].rate == -0.1234567 and d["fir"].decimation == 833
            chain.stop()
        sel = Selector(20000000, 250000)
        w = WFm(48000, 50e-6, False)
        chain = Chain([sel, w])
        chain.setReader(src.getReader()); chain.setWriter(M.Buffer(Format.FLOAT))
        d = M._ChannelPlan.match(M._walk(sel.shift)[0])
        assert d and d["demod"] == "wfm" and d["wfm_frac"].rate == 250000.0 / 48000 and d["fir"].decimation == 80
        chain.stop()
    finally:
        sys.path.remove(REF)
        for k in [k for k in sys.modules if k == "csdr" or k.startswith("csdr.") or k == "owrx" or k.startswith("owrx.")]:
            sys.modules.pop(k)


def test_source_side_convert_gain_forwards_raw_samples_tagged():
    """owrx/source/fifi_sdr.py:27-28 + owrx/source/direct.py:59-71: Buffer(COMPLEX_SHORT) -> Chain([Convert(COMPLEX_SHORT,
    COMPLEX_FLOAT), Gain(COMPLEX_FLOAT, 5.0)]) -> Buffer(COMPLEX_FLOAT).  The shim never converts on the host: the raw
    samples arrive in the float buffer tagged ("cs16", 5.0) for owrx_*_feed_fmt (SURVEY 8f-4)."""
    import time
    raw_buf = M.Buffer(Format.COMPLEX_SHORT)
    conv, gain = M.Convert(Format.COMPLEX_SHORT, Format.COMPLEX_FLOAT), M.Gain(Format.COMPLEX_FLOAT, 5.0)
    mid, out = M.Buffer(Format.COMPLEX_FLOAT), M.Buffer(Format.COMPLEX_FLOAT)
    # the order csdr.chain.Chain wires its workers in: internal buffers first, then reader and writer
    conv.setWriter(mid); gain.setReader(mid.getReader())
    conv.setReader(raw_buf.getReader()); gain.setWriter(out)
    rd = out.getReader()
    payload = np.arange(-8, 8, dtype=np.int16).tobytes()
    raw_buf.write(payload)
    got = rd.read()
    assert bytes(got) == payload and out._raw == ("cs16", 5.0)
    with pytest.raises(ValueError):
        conv.setReader(M.Buffer(Format.COMPLEX_FLOAT).getReader())        # wrong input format
    # the client-audio Convert(FLOAT, SHORT) is no ingress stage: no pump
    c2 = M.Convert(Format.FLOAT, Format.SHORT)
    c2.setReader(M.Buffer(Format.FLOAT).getReader())
    assert c2._pump is None
    raw_buf.getReader  # keep alive
    conv.stop(); gain.stop()


@pytest.mark.skipif(not HAVE_REF, reason=NO_REF)
def test_reference_fifi_sdr_format_conversion_runs_on_the_shim():
    """the reference's UNMODIFIED FifiSdrSource.getFormatConversion() (owrx/source/fifi_sdr.py:27-28), wired the way
    DirectSource.getBuffer does (owrx/source/direct.py:59-71), hands raw int16 samples on with gain 5.0"""
    if REF not in sys.path:
        sys.path.insert(0, REF)
    from owrx.source.fifi_sdr import FifiSdrSource
    conversion = FifiSdrSource.getFormatConversion(None)
    assert conversion.getInputFormat() is Format.COMPLEX_SHORT and conversion.getOutputFormat() is Format.COMPLEX_FLOAT
    src = M.Buffer(Format.COMPLEX_SHORT)
    conversion.setReader(src.getReader())
    out = M.Buffer(Format.COMPLEX_FLOAT)
    conversion.setWriter(out)
    rd = out.getReader()
    payload = np.arange(100, dtype=np.int16).tobytes()
    src.write(payload)
    assert bytes(rd.read()) == payload and out._raw == ("cs16", 5.0)
    conversion.stop()


def test_fused_stage_readers_do_not_pin_the_source_buffer():
    """ADVICE r1: head stages get a Reader through Chain.setReader that nobody ever reads (the runner reads the Buffer through
    its own cursor): such wiring tokens must not make Buffer._trim keep every chunk"""
    src = M.Buffer(Format.COMPLEX_FLOAT)
    fft = M.Fft(size=1024, every_n_samples=700)
    fft.setReader(src.getReader())                      # attaches a runner with its own reader; this one is only a token
    assert fft._reader._virtual
    runner = src._runner
    assert runner is not None
    chunk = bytes(8 * 1000)
    for _ in range(200):
        src.write(chunk)
    deadline = time.time() + 10
    while time.time() < deadline and runner.processed < src._end:
        time.sleep(0.01)
    src.write(chunk)                                    # a write trims what every live cursor has passed
    time.sleep(0.2)
    assert len(src._chunks) <= 4, len(src._chunks)
    # a cursor somebody really reads counts again, from the moment it is read
    r = src.getReader()
    src.write(b"\x01" * 8)
    assert bytes(r.read()) == b"\x01" * 8
    fft.stop()


class _FakeRing:
    """stands in for the cudaHostAlloc'd arena (no CUDA device in the build container): same fields as pycsdr.modules._PinnedRing"""

    def __init__(self, nbytes):
        self.store = bytearray(nbytes)
        self.view = memoryview(self.store)
        self.size, self.head, self.ptr = nbytes, 0, 1


def test_ring_backed_source_buffer_logic():
    """SURVEY 8f-4: the page-locked ingress ring's bookkeeping (chunks never split across the wrap, adjacent chunks merge into one
    feed, a Python reader gets copies, regions being fed are not overwritten, unread data in the way is dropped oldest-first)"""
    import threading
    import time
    import pycsdr.modules as M
    from pycsdr.types import Format
    buf = M.Buffer(Format.COMPLEX_FLOAT)
    buf._ring = _FakeRing(1024)
    runner_rd, py_rd = buf.getReader(), buf.getReader()
    a, b = bytes(range(200)), bytes(range(50, 250))
    buf.write(a); buf.write(b)
    views = runner_rd._read_views()
    assert len(views) == 1 and bytes(views[0]) == a + b            # adjacent ring chunks merge into ONE view (one feed, zero copy)
    assert views[0].obj is buf._ring.store                          # ... into the ring itself
    assert buf._inflight == [(0, 400)]
    got = py_rd.read()
    assert isinstance(got.obj, bytes) and bytes(got) == a           # a Python pump gets its own copy, one write = one read
    assert bytes(py_rd.read()) == b
    # the next 400 bytes fit behind (400..800); the one after would wrap onto the region the runner is still feeding from
    buf.write(bytes(400))
    done = []
    th = threading.Thread(target=lambda: (buf.write(b"\x07" * 300), done.append(1)), daemon=True)
    th.start()
    time.sleep(0.3)
    assert not done, "the writer overwrote a region the runner is feeding from"
    assert bytes(views[0]) == a + b
    runner_rd._release()
    th.join(5)
    assert done and buf._ring.head == 300                          # wrapped to offset 0, never split
    # unread chunks in the way are dropped oldest-first (ring semantics), whole chunks only
    v2 = runner_rd._read_views()
    assert [len(v) for v in v2] == [400, 300]                       # not adjacent across the wrap: two feeds
    runner_rd._release()
    big = M.Buffer(Format.CHAR); big._ring = _FakeRing(1024)
    rd = big.getReader()
    for k in range(6):
        big.write(bytes([k]) * 256)                                 # 6 x 256 through 1024 bytes with nobody reading
    vs = rd._read_views()
    assert b"".join(bytes(v) for v in vs) == b"".join(bytes([k]) * 256 for k in (2, 3, 4, 5))
    rd._release()
