"""CPU tests of the pycsdr shim's demodulated-audio tap: a secondary demodulator (Convert(FLOAT, SHORT) -> decoder) reading the
demodulator's audio Buffer beside the client-audio Converter.  Which stage continues the chain (_walk) and which tap the
second reader asks for (_ChannelPlan.match)."""
import pycsdr.modules as M
from pycsdr.types import Format


def _join(ws):
    for a, b in zip(ws[:-1], ws[1:]):
        buf = M.Buffer(a.getOutputFormat())
        a.setWriter(buf)
        b.setReader(buf.getReader())
    ws[-1].setWriter(M.Buffer(ws[-1].getOutputFormat()))


def _decoder(audio):
    """a WSJT-style secondary demodulator's front: Convert(FLOAT, SHORT) on the audio Buffer, into a Buffer of its own"""
    conv = M.Convert(Format.FLOAT, Format.SHORT)
    conv.setReader(audio.getReader())
    conv.setWriter(M.Buffer(Format.SHORT))
    return conv


def _usb(decoder_first, converter="adpcm"):
    """Shift -> FirDecimate -> RealPart -> Agc -> client audio, plus a decoder on the Agc's Buffer, constructed either before
    or after the client audio chain; the head gets no reader, so no runner starts.  Returns (stages, client Convert, decoder)"""
    demod = [M.Shift(0.1), M.FirDecimate(200, 0.15 * 12000 / 2.4e6, 0.5), M.RealPart(), M.Agc(Format.FLOAT)]
    _join(demod)
    audio = demod[-1]._writer
    dec = _decoder(audio) if decoder_first else None
    if converter == "adpcm":
        client = [M.Convert(Format.FLOAT, Format.SHORT), M.AdpcmEncoder(sync=True)]
    elif converter == "resampler":
        client = [M.AudioResampler(12000, 48000), M.Limit(), M.Convert(Format.FLOAT, Format.SHORT), M.AdpcmEncoder(sync=True)]
    else:
        client = [M.Convert(Format.FLOAT, Format.SHORT)]
    _join(client)
    client[0].setReader(audio.getReader())
    if not decoder_first:
        dec = _decoder(audio)
    return demod + client, dec


def _stop(*groups):
    for g in groups:
        for m in (g if isinstance(g, list) else [g]):
            m.stop()


def test_walk_takes_the_client_audio_chain_whatever_the_construction_order():
    for _ in range(6):
        for first in (True, False):
            for conv in ("adpcm", "resampler"):
                ws, dec = _usb(first, conv)
                chain = M._walk(ws[0])[0]
                assert chain == ws, (first, conv, [type(m).__name__ for m in chain])
                assert dec not in chain
                _stop(ws, dec)


def test_walk_between_two_bare_converts_is_stable():
    """two bare Convert(FLOAT, SHORT) readers give the same bytes: either may continue the chain, but always the same one"""
    for first in (True, False):
        ws, dec = _usb(first, "s16")
        picks = {M._walk(ws[0])[0][-1] for _ in range(5)}
        assert len(picks) == 1 and picks <= {ws[-1], dec}
        _stop(ws, dec)


def test_match_records_the_s16_tap_for_a_decoder():
    for first in (True, False):
        ws, dec = _usb(first)
        d = M._ChannelPlan.match(M._walk(ws[0])[0])
        assert d["demod"] == "ssb" and d["audio_fmt"] == "adpcm" and d["tail"] is ws[-1]
        assert d["atap"] == "s16" and d["atap_writer"] is dec._writer
        dec.stop()
        d = M._ChannelPlan.match(M._walk(ws[0])[0])
        assert d["atap"] is None and d["atap_writer"] is None
        _stop(ws)


def test_match_records_the_tap_behind_a_resampler_and_after_nfm():
    ws, dec = _usb(False, "resampler")
    d = M._ChannelPlan.match(M._walk(ws[0])[0])
    assert d["resampler"] == (12000, 48000) and d["atap"] == "s16" and d["atap_writer"] is dec._writer
    _stop(ws, dec)
    nfm = [M.Shift(0.1), M.FirDecimate(200, 0.15 * 12000 / 2.4e6, 0.5), M.FmDemod(), M.Limit(), M.NfmDeemphasis(12000),
           M.Agc(Format.FLOAT), M.Convert(Format.FLOAT, Format.SHORT)]
    _join(nfm)
    dec = _decoder(nfm[5]._writer)
    d = M._ChannelPlan.match(M._walk(nfm[0])[0])
    assert d["demod"] == "nfm" and d["atap"] == "s16"
    _stop(nfm, dec)


def test_match_gives_any_other_reader_the_f32_tap():
    ws, dec = _usb(True)
    dec.stop()
    audio = ws[3]._writer
    r = audio.getReader()                                        # e.g. a Python decoder reading the float audio itself
    d = M._ChannelPlan.match(M._walk(ws[0])[0])
    assert d["atap"] == "f32" and d["atap_writer"] is audio
    r.stop()
    assert M._ChannelPlan.match(M._walk(ws[0])[0])["atap"] is None
    _stop(ws)


def test_match_records_no_tap_with_float_client_audio():
    demod = [M.Shift(0.1), M.FirDecimate(200, 0.15 * 12000 / 2.4e6, 0.5), M.RealPart(), M.Agc(Format.FLOAT)]
    _join(demod)
    r = demod[-1]._writer.getReader()                             # the client reads float audio: the Buffer is materialised
    d = M._ChannelPlan.match(M._walk(demod[0])[0])
    assert d["audio_fmt"] == "f32" and d["atap"] is None and d["atap_writer"] is None
    r.stop()
    _stop(demod)


def test_match_reports_a_float_reader_it_cannot_serve_beside_the_decoder(caplog):
    ws, dec = _usb(True)
    r = ws[3]._writer.getReader()
    with caplog.at_level("WARNING", logger="pycsdr.modules"):
        for _ in range(3):
            assert M._ChannelPlan.match(M._walk(ws[0])[0])["atap"] == "s16"
    hits = [m for m in caplog.messages if "audio buffer" in m and "float reader receives nothing" in m]
    assert len(hits) == 1
    r.stop()
    _stop(ws, dec)
