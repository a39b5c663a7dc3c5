"""CPU tests of the client-audio resampler (AudioResampler -> Limit, csdr/chain/clientaudio.py:6-19): the spec-defined reference's
design and streaming arithmetic (tests/audio_resampler_ref.py) against scipy, and the chains the pycsdr shim fuses (_ChannelPlan.match), including the two
Converter shapes recorded from the unmodified reference (tests/golden/trace_client.json)."""
import numpy as np
import pytest
from scipy import signal

import audio_resampler_ref as ref
import pycsdr.modules as M
from pycsdr.types import Format

# (in, out, L, M, K): the ratios the browser's rates give (SURVEY.md:316) and the two recorded ones
RATIOS = [(12000, 11025, 147, 160, 67), (48000, 44100, 147, 160, 67), (48000, 12000, 1, 4, 247), (12000, 48000, 4, 1, 62),
          (22050, 12000, 80, 147, 113)]


@pytest.mark.parametrize("fin,fout,L,Mr,K", RATIOS)
def test_reference_taps_are_the_kaiser_firwin_design(fin, fout, L, Mr, K):
    h, l, m, k = ref.design(fin, fout)
    assert (l, m, k) == (L, Mr, K) and len(h) == L * K
    beta = 0.1102 * (96.0 - 8.7)
    want = signal.firwin(L * K, 0.45 * min(fin, fout), window=("kaiser", beta), fs=L * fin) * L
    assert np.max(np.abs(h - want)) <= 1e-12 * np.max(np.abs(want))
    assert abs(h.sum() - L) <= 1e-9 * L


def _upfirdn(x, fin, fout):
    h, L, Mr, _ = ref.design(fin, fout)
    n = -(-len(x) * L // Mr)                                    # ceil(n_in * L / M) outputs exist after n_in inputs
    return np.clip(signal.upfirdn(h, x.astype(np.float64), L, Mr)[:n], -1.0, 1.0)


@pytest.mark.parametrize("fin,fout,L,Mr,K", RATIOS)
def test_reference_resample_equals_float64_upfirdn_whatever_the_partition(fin, fout, L, Mr, K):
    rng = np.random.default_rng(fin + fout)
    t = np.arange(20000) / fin
    x = (0.6 * np.sin(2 * np.pi * 440.0 * t) + 0.3 * rng.standard_normal(len(t))).astype(np.float32)
    x[5000:5200] *= 4.0                                         # some samples past full scale: Limit clamps them
    want = _upfirdn(x, fin, fout)
    ragged = rng.integers(1, 700, 60)
    for parts in (None, ragged, [1] * 50 + [3, 7, 2]):
        got = ref.resample(x, fin, fout, parts)
        assert len(got) == len(want)
        assert np.sqrt(np.mean((got - want) ** 2) / np.mean(want ** 2)) <= 1e-6
        assert np.abs(got).max() <= 1.0


def test_reference_rejects_ratios_beyond_65536_taps():
    assert ref.design(1, 48000) is None
    assert ref.design(48000, 1) is None
    with pytest.raises(ValueError):
        ref.resample(np.zeros(10, np.float32), 48000, 1)


def _join(ws):
    for a, b in zip(ws[:-1], ws[1:]):
        buf = M.Buffer(a.getOutputFormat())
        a.setWriter(buf)
        b.setReader(buf.getReader())
    ws[-1].setWriter(M.Buffer(ws[-1].getOutputFormat()))


def _ssb_chain(converter, adpcm=True):
    """Shift -> FirDecimate -> RealPart -> Agc, then the client audio chain; the head gets no reader, so no runner starts"""
    ws = [M.Shift(0.1), M.FirDecimate(200, 0.15 * 12000 / 2.4e6, 0.5), M.RealPart(), M.Agc(Format.FLOAT)] + converter
    if adpcm:
        ws.append(M.AdpcmEncoder(sync=True))
    _join(ws)
    return ws


def _stop(ws):
    for m in ws:
        m.stop()


@pytest.mark.parametrize("adpcm", [True, False])
@pytest.mark.parametrize("fin,fout", [(48000, 12000), (12000, 48000), (12000, 11025)])
def test_match_fuses_the_recorded_converter(fin, fout, adpcm):
    conv = [M.AudioResampler(fin, fout), M.Limit(), M.Convert(Format.FLOAT, Format.SHORT)]
    ws = _ssb_chain(conv, adpcm)
    d = M._ChannelPlan.match(M._walk(ws[0])[0])
    assert d is not None and d["demod"] == "ssb"
    assert d["resampler"] == (fin, fout)
    assert d["audio_fmt"] == ("adpcm" if adpcm else "s16")
    assert d["tail"] is ws[-1] and d["stages"] == ws
    _stop(ws)


def test_match_without_a_resampler_is_unchanged():
    ws = _ssb_chain([M.Convert(Format.FLOAT, Format.SHORT)])
    d = M._ChannelPlan.match(M._walk(ws[0])[0])
    assert d is not None and d["resampler"] is None and d["audio_fmt"] == "adpcm"
    _stop(ws)


def test_match_after_nfm_and_wfm():
    lim = M.Limit()
    nfm = [M.Shift(0.1), M.FirDecimate(200, 0.15 * 12000 / 2.4e6, 0.5), M.FmDemod(), lim, M.NfmDeemphasis(12000),
           M.Agc(Format.FLOAT), M.AudioResampler(12000, 11025), M.Limit(), M.Convert(Format.FLOAT, Format.SHORT)]
    _join(nfm)
    d = M._ChannelPlan.match(M._walk(nfm[0])[0])
    assert d["demod"] == "nfm" and d["resampler"] == (12000, 11025) and d["audio_fmt"] == "s16"
    _stop(nfm)
    wfm = [M.Shift(0.1), M.FirDecimate(8, 0.15 * 250000 / 2e6, 0.5), M.FmDemod(), M.Limit(),
           M.FractionalDecimator(Format.FLOAT, 250000.0 / 48000, prefilter=True), M.WfmDeemphasis(48000, 50e-6),
           M.AudioResampler(48000, 44100), M.Limit(), M.Convert(Format.FLOAT, Format.SHORT), M.AdpcmEncoder(sync=True)]
    _join(wfm)
    d = M._ChannelPlan.match(M._walk(wfm[0])[0])
    assert d["demod"] == "wfm" and d["resampler"] == (48000, 44100) and d["audio_fmt"] == "adpcm"
    _stop(wfm)


@pytest.mark.parametrize("conv", [
    lambda: [M.AudioResampler(12000, 11025), M.Convert(Format.FLOAT, Format.SHORT)],            # no Limit
    lambda: [M.AudioResampler(12000, 11025), M.Limit()],                                       # no Convert
    lambda: [M.AudioResampler(48000, 1), M.Limit(), M.Convert(Format.FLOAT, Format.SHORT)],    # > 65536 taps
    lambda: [M.AudioResampler(0, 12000), M.Limit(), M.Convert(Format.FLOAT, Format.SHORT)],    # not a rate
])
def test_match_refuses_other_tails(conv):
    ws = _ssb_chain(conv(), adpcm=False)
    assert M._ChannelPlan.match(M._walk(ws[0])[0]) is None
    _stop(ws)


def test_resampler_stages_do_not_key_the_channel():
    """a replaced AudioResampler (or its Limit) reaches the bank through the setter, not as a new channel"""
    ws = _ssb_chain([M.AudioResampler(12000, 11025), M.Limit(), M.Convert(Format.FLOAT, Format.SHORT)])
    d = M._ChannelPlan.match(M._walk(ws[0])[0])
    assert set(d["resampler_stages"]) == {ws[4], ws[5]}
    _stop(ws)


def test_audio_resampler_is_fused_and_constructible_as_recorded():
    rs = M.AudioResampler(48000, 12000)                          # the transient of the WFM switch (SURVEY D.3)
    assert not isinstance(rs, M._Unfused)
    assert (rs.inputRate, rs.outputRate) == (48000, 12000)
    assert rs.getInputFormat() is Format.FLOAT and rs.getOutputFormat() is Format.FLOAT
    rs.stop()
