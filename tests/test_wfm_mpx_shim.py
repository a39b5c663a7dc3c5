"""CPU tests of the pycsdr shim's WFM multiplex tap: which tap a WFm chain's consumers ask for (_ChannelPlan.match), and the
host ExecModule that the reference's RDS decoder module (redsea) builds on."""
import sys
import time

import pycsdr.modules as M
from pycsdr.types import Format

COPY = "import sys\nwhile True:\n    d = sys.stdin.buffer.read1(65536)\n    if not d:\n        break\n    sys.stdout.buffer.write(d)\n    sys.stdout.buffer.flush()\n"


def _wfm_chain():
    """Shift -> FirDecimate -> FmDemod -> Limit -> FractionalDecimator(FLOAT) -> WfmDeemphasis, joined with Buffers the way
    csdr.chain.Chain does; the head gets no reader, so no source runner starts"""
    lim = M.Limit()
    ws = [M.Shift(0.1), M.FirDecimate(80, 0.15 * 250000 / 20e6, 0.5), M.FmDemod(), lim,
          M.FractionalDecimator(Format.FLOAT, 250000.0 / 48000, prefilter=True), M.WfmDeemphasis(48000, 50e-6)]
    for a, b in zip(ws[:-1], ws[1:]):
        buf = M.Buffer(a.getOutputFormat())
        a.setWriter(buf)
        b.setReader(buf.getReader())
    ws[-1].setWriter(M.Buffer(Format.FLOAT))
    return ws, lim._writer


def _match(ws):
    d = M._ChannelPlan.match(M._walk(ws[0])[0])
    assert d and d["demod"] == "wfm" and d["wfm_frac"] is ws[4]
    return d


def test_match_records_no_tap_without_a_consumer():
    ws, _ = _wfm_chain()
    d = _match(ws)
    assert d["mpx"] is None and d["mpx_writer"] is None


def test_match_fuses_convert_float_short_as_the_s16_tap():
    ws, tap = _wfm_chain()
    conv = M.Convert(Format.FLOAT, Format.SHORT)                # the reference's RDS path (csdr/chain/analog.py:73-76)
    conv.setReader(tap.getReader())
    out = M.Buffer(Format.SHORT)
    conv.setWriter(out)
    d = _match(ws)                                               # the chain still continues through the FractionalDecimator
    assert d["mpx"] == "s16" and d["mpx_writer"] is out
    conv.stop()
    assert _match(ws)["mpx"] is None


def test_match_reports_a_float_reader_it_cannot_serve_beside_the_convert(caplog):
    ws, tap = _wfm_chain()
    conv = M.Convert(Format.FLOAT, Format.SHORT)
    conv.setReader(tap.getReader())
    conv.setWriter(M.Buffer(Format.SHORT))
    r = tap.getReader()
    with caplog.at_level("WARNING", logger="pycsdr.modules"):
        assert _match(ws)["mpx"] == "s16"
    assert any("float reader receives nothing" in m for m in caplog.messages)
    r.stop()
    conv.stop()


def test_match_gives_any_other_reader_the_f32_tap():
    ws, tap = _wfm_chain()
    r = tap.getReader()                                          # e.g. a Python module reading metaTapBuffer itself
    d = _match(ws)
    assert d["mpx"] == "f32" and d["mpx_writer"] is tap
    r.stop()
    assert _match(ws)["mpx"] is None


def test_exec_module_round_trips_bytes_and_reaps_its_child():
    inb, outb = M.Buffer(Format.SHORT), M.Buffer(Format.CHAR)
    em = M.ExecModule(Format.SHORT, Format.CHAR, [sys.executable, "-c", COPY])
    assert em.getInputFormat() is Format.SHORT and em.getOutputFormat() is Format.CHAR
    em.setReader(inb.getReader())
    em.setWriter(outb)
    rd = outb.getReader()
    payload = bytes(range(256)) * 300
    for o in range(0, len(payload), 7000):
        inb.write(payload[o:o + 7000])
    got = b""
    t0 = time.time()
    while len(got) < len(payload) and time.time() - t0 < 30:
        got += bytes(rd._read(True))
    assert got == payload
    # a new reader while the stdin pump waits on the old one: the old cursor is stopped, the pump moves over
    inb2 = M.Buffer(Format.SHORT)
    old = em._reader
    em.setReader(inb2.getReader())
    assert old._stopped
    inb2.write(b"moved")
    got = b""
    t0 = time.time()
    while len(got) < 5 and time.time() - t0 < 30:
        got += bytes(rd._read(True))
    assert got == b"moved"
    em.stop()
    assert em._proc.returncode is not None
    assert all(not t.is_alive() for t in em._threads)
    em.stop()                                                    # idempotent
