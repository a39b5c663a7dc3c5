"""GPU tests of the drop-in boundary: pycsdr module objects wired with the reference's Chain._connect
pattern (csdr/chain/__init__.py:21-25, restated locally: the reference's own classes are not part of this
repository)."""
import sys
import threading
import time

import numpy as np
import pytest

import oracle
import pycsdr.modules as M
from openwebrx_b200 import ChannelBank, _native as N
from openwebrx_b200.synth import BANDPASS, carrier_plan, make_iq
from pycsdr.types import AgcProfile, Format
from test_oracle import JsImaAdpcmCodec, browser_fft_decode

pytestmark = pytest.mark.gpu


def _connect(workers):
    for a, b in zip(workers[:-1], workers[1:]):
        buf = M.Buffer(a.getOutputFormat())
        a.setWriter(buf)
        b.setReader(buf.getReader())


def _collect(reader, want, timeout=30.0):
    """pump like csdr/module/__init__.py:36-53: one read() result = one message"""
    msgs, n = [], 0
    t0 = time.time()
    box = []

    def pump():
        while True:
            d = reader.read()
            if d is None:
                break
            box.append(bytes(d))
    th = threading.Thread(target=pump, daemon=True)
    th.start()
    while time.time() - t0 < timeout:
        n = sum(len(b) for b in box)
        if n >= want:
            break
        time.sleep(0.02)
    reader.stop()
    th.join(2)
    return list(box)


def test_fft_chain_through_module_api(gpu):
    fs, n, every_n, avg = 2.4e6, 1024, 700, 4
    iq = make_iq(every_n * avg * 6 + n, fs, carrier_plan(5, fs, seed=31), seed=31)
    ws = [M.Fft(size=n, every_n_samples=0), M.LogAveragePower(add_db=-70, fft_size=n, avg_number=avg), M.FftSwap(fft_size=n),
          M.FftAdpcm(fft_size=n)]
    ws[0].setEveryNSamples(every_n)
    _connect(ws)
    src = M.Buffer(Format.COMPLEX_FLOAT)
    out = M.Buffer(Format.CHAR)
    ws[-1].setWriter(out)
    rd = out.getReader()
    ws[0].setReader(src.getReader())
    raw = iq.tobytes()
    for o in range(0, len(raw), 8 * 1000):                 # ragged delivery like a TCP source
        src.write(raw[o:o + 8 * 1000])
    lb = (n + 10) // 2
    msgs = _collect(rd, 6 * lb)
    ref = oracle.fftchain_run(iq, n, every_n, avg)
    assert len(msgs) == 6 and all(len(m) == lb for m in msgs)       # one message per line (htdocs/openwebrx.js:1124-1131)
    for m, db in zip(msgs, ref["db"]):
        shown = browser_fft_decode(np.frombuffer(m, np.uint8))      # what the browser would display
        assert np.median(np.abs(shown - db)) < 0.6
    same = sum(m == l.tobytes() for m, l in zip(msgs, ref["lines"]))
    assert same >= 4                                                 # byte-identical unless an int16 sits on a rounding edge
    # the same chain without FftAdpcm (compression "none", csdr/chain/fft.py:87-96): the float32 dB lines themselves, held to the
    # north-star tolerance through the module API
    ws = [M.Fft(size=n, every_n_samples=0), M.LogAveragePower(add_db=-70, fft_size=n, avg_number=avg), M.FftSwap(fft_size=n)]
    ws[0].setEveryNSamples(every_n)
    _connect(ws)
    src, out = M.Buffer(Format.COMPLEX_FLOAT), M.Buffer(Format.FLOAT)
    ws[-1].setWriter(out)
    rd = out.getReader()
    ws[0].setReader(src.getReader())
    for o in range(0, len(raw), 8 * 1000):
        src.write(raw[o:o + 8 * 1000])
    msgs = _collect(rd, 6 * 4 * n)
    assert len(msgs) == 6 and all(len(m) == 4 * n for m in msgs)
    from test_gpu_waterfall import _assert_db_parity, _truth_db
    got = np.stack([np.frombuffer(m, np.float32) for m in msgs])
    _assert_db_parity(got, ref["db"], _truth_db(iq, n, every_n, avg))   # 0.01 dB, as in test_gpu_waterfall


def test_two_clients_share_one_source_buffer(gpu):
    fs, out_rate = 2.4e6, 12000
    cars = carrier_plan(2, fs, seed=32)
    cars[0]["kind"], cars[1]["kind"] = "nfm", "am"
    iq = make_iq(5333 + 200 * (750 * 2 + 20), fs, cars, seed=32)
    src = M.Buffer(Format.COMPLEX_FLOAT)
    readers, tails = [], []
    for c in cars:
        agc = M.Agc(Format.FLOAT); agc.setProfile(AgcProfile.SLOW)
        if c["kind"] == "nfm":
            agc.setMaxGain(3)
            demod = [M.FmDemod(), M.Limit(), M.NfmDeemphasis(12000), agc]
        else:
            agc.setInitialGain(200)
            demod = [M.AmDemod(), M.DcBlock(), agc]
        bp = M.Bandpass(transition=320.0 / out_rate, use_fft=True)
        lo, hi = BANDPASS[c["kind"]]
        bp.setBandpass(lo / out_rate, hi / out_rate)
        sh = M.Shift(0.0); sh.setRate(-c["offset"] / fs)
        ws = [sh, M.FirDecimate(200, 0.15 * out_rate / fs, 0.5), bp,
              M.Squelch(Format.COMPLEX_FLOAT, length=750, decimation=5, hangLength=1500, flushLength=3750, reportInterval=4)] + demod
        _connect(ws)
        ob = M.Buffer(Format.FLOAT)
        ws[-1].setWriter(ob)
        readers.append(ob.getReader())
        ws[0].setReader(src.getReader())
        tails.append(ws)
    raw = iq.tobytes()
    step = 8 * 100000
    for o in range(0, len(raw), step):
        src.write(raw[o:o + step])
    kind = {"nfm": oracle.DEMOD_NFM, "am": oracle.DEMOD_AM}
    for rd, c in zip(readers, cars):
        ref = oracle.client_chain_run(iq, fs, out_rate, c["offset"], BANDPASS[c["kind"]], kind[c["kind"]])
        got = np.frombuffer(b"".join(_collect(rd, 4 * len(ref["audio"]))), np.float32)
        assert len(got) == len(ref["audio"]) == 1500
        err = np.sqrt(np.mean((got - ref["audio"]) ** 2)) / np.sqrt(np.mean(ref["audio"] ** 2))
        assert err < 1e-2                                   # post-AGC (spec-defined); pre-AGC parity is in test_gpu_selector
    assert src._runner is not None and len(src._runner.channels) == 2      # both clients ride one bank / one feed per block


def test_audio_tail_convert_and_adpcm_bit_exact(gpu):
    # SURVEY 8f-1: Convert(FLOAT,SHORT) + AdpcmEncoder(sync=True) on the GPU; integer path => bit-exact
    fs, out_rate = 2.4e6, 12000
    cars = carrier_plan(3, fs, seed=33)
    iq = make_iq(5333 + 200 * (750 * 6 + 5), fs, cars, seed=33)
    bank = ChannelBank(fs)
    trip = []
    for c in cars:
        chs = []
        for fmt in ("f32", "s16", "adpcm"):
            ch = bank.add_channel(out_rate, demod=c["kind"], offset=c["offset"], bandpass=BANDPASS[c["kind"]])
            ch.setAudioFormat(fmt)
            chs.append(ch)
        trip.append(chs)
    for o in range(0, len(iq), 333333):                     # state (predictor, step, sync counter, odd nibble) carries across feeds
        bank.feed(iq[o:o + 333333])
    for f32, s16, adp in trip:
        audio = f32.read_audio()
        assert len(audio) == 4500
        want16 = oracle.convert_f_s16(audio)
        assert np.array_equal(s16.read_bytes().view(np.int16), want16)
        want = oracle.adpcm_sync_encode(want16)
        got = adp.read_bytes()
        assert np.array_equal(got, want)
        dec = JsImaAdpcmCodec().decodeWithSync(bytes(got))  # and the browser's decoder accepts it
        assert len(dec) == 4500


# (The reference's own FftChain / SpectrumThread / DspManager classes are not part of this repository.  Their recorded call
# traces are replayed with data in tests/test_gpu_trace_replay.py; the classes themselves run unmodified on the shim, without a
# device, in tests/test_pycsdr_shim.py when OWRX_REFERENCE names an OpenWebRX source tree.)


def test_raw_ingress_formats_equal_cpu_side_convert(gpu):
    """SURVEY 8f-4: int16 / uint8 source samples converted on the GPU (owrx_*_feed_fmt) give exactly what the reference's
    CPU-side Convert (+ Gain) followed by the float path gives (owrx/source/fifi_sdr.py:27-28, owrx/source/direct.py:59-71)"""
    import oracle
    from openwebrx_b200 import ChannelBank, Waterfall, _native as N
    from openwebrx_b200.synth import BANDPASS, carrier_plan, make_iq
    fs = 2.4e6
    cars = carrier_plan(3, fs, seed=51)
    iq = make_iq(5333 + 200 * 1500 + 4099, fs, cars, seed=51)
    for fmt, gain in (("cs16", 5.0), ("cu8", 1.0)):
        f = iq.view(np.float32)
        raw = (np.clip(f, -1, 1) * 30000).astype(np.int16) if fmt == "cs16" else (np.clip(f, -1, 1) * 120 + 127.5).astype(np.uint8)
        as_float = oracle.convert_raw_iq(raw, fmt, gain)
        outs = []
        for use_raw in (True, False):
            bank = ChannelBank(fs, outputs=N.OUT_IF | N.OUT_DEMOD)
            chans = [bank.add_channel(12000, demod=c["kind"], offset=c["offset"], bandpass=BANDPASS[c["kind"]]) for c in cars]
            cut = 2 * 123457                                   # ragged two-part feed (chunk boundaries inside the raw stream)
            if use_raw:
                bank.feed_raw(raw[:cut], fmt, gain); bank.feed_raw(raw[cut:], fmt, gain)
            else:
                bank.feed(as_float[:cut // 2]); bank.feed(as_float[cut // 2:])
            outs.append([(c.read_if(), c.read_demod()) for c in chans])
            bank.close()
        for (a_if, a_dm), (b_if, b_dm) in zip(*outs):
            assert len(a_if) == len(b_if) > 1000 and np.array_equal(a_if, b_if) and np.array_equal(a_dm, b_dm)
        wf_a, wf_b = Waterfall(fs, 1024, 0.3, 60, "adpcm"), Waterfall(fs, 1024, 0.3, 60, "adpcm")
        la, lb = wf_a.feed_raw(raw, fmt, gain), wf_b.feed(as_float)
        assert len(la) == len(lb) >= 4 and all(x == y for x, y in zip(la, lb))
    with pytest.raises(ValueError):
        N.check(N.lib.owrx_bank_feed_fmt(ChannelBank(fs)._h, raw.ctypes.data, 10, 7, 1.0))


def test_f3_resampler_and_secondary_fft_shapes(gpu):
    """SURVEY 8f-3: the same kernels at the reference's secondary shapes.
    (a) Resampler for background services (owrx/source/resampler.py:11-24): Chain([Shift(shift), FirDecimate(decimation,
        0.15 * if_rate / samp_rate)]) producing COMPLEX_FLOAT at the service rate — here 2.4 MS/s -> 48 kHz (D = 50), checked
        stage by stage against the oracle's Shift and FirDecimate;
    (b) secondary FFT on the selector output (owrx/dsp.py:220-225): 2048 points at 12 kHz, 9 fps -> LogAveragePower with avg 1."""
    import oracle
    from openwebrx_b200 import ChannelBank, Waterfall, _native as N, fftchain_params
    from openwebrx_b200.synth import carrier_plan, make_iq
    fs, rate = 2.4e6, 48000.0
    cars = carrier_plan(3, fs, seed=71)
    D = int(fs / rate)
    tr = 0.15 * (fs / D) / fs
    taps = oracle.firdes_lowpass(oracle.filter_len(tr), 0.5 / D)
    iq = make_iq(len(taps) + D * 3000, fs, cars, seed=71)
    bank = ChannelBank(fs, outputs=N.OUT_IF)
    chans = [bank.add_channel(rate, demod="none", offset=c["offset"]) for c in cars]      # no Bandpass, Squelch open
    bank.feed(iq)
    for ch, c in zip(chans, cars):
        want = oracle.fir_decimate(oracle.shift(iq, -c["offset"] / fs), taps, D)
        got = ch.read_if()
        assert len(got) == len(want) == 3001
        err = np.sqrt(np.mean(np.abs(got - want) ** 2)) / np.sqrt(np.mean(np.abs(want) ** 2))
        assert err <= 1e-4, err
    bank.close()
    # (b) the selector output of a 12 kHz client feeds a 2048-point FftChain
    avg, every_n = fftchain_params(12000, 2048, 0.3, 9)
    assert (avg, every_n) == (1, 1333)
    rng = np.random.default_rng(72)
    x = (rng.standard_normal(every_n * 6 + 2048) + 1j * rng.standard_normal(every_n * 6 + 2048)).astype(np.complex64) * 0.05
    x += (0.3 * np.exp(2j * np.pi * 0.11 * np.arange(len(x)))).astype(np.complex64)
    ref = oracle.fftchain_run(x, 2048, every_n, avg)
    wf = Waterfall(12000, 2048, 0.3, 9, "adpcm")
    lines = wf.feed(x)
    assert len(lines) == len(ref["lines"]) == 7
    for l, want in zip(lines, ref["lines"]):
        got_db = oracle.ima_adpcm_decode(np.frombuffer(l, np.uint8))[10:].astype(np.int32)
        want_db = oracle.ima_adpcm_decode(np.ascontiguousarray(want))[10:].astype(np.int32)
        assert np.abs(got_db - want_db).max() <= 300        # 1/100 dB units through the lossy codec: a few quantiser steps


def test_f2_websocket_message_framing(gpu):
    """SURVEY 8f-2: outputs leave as websocket messages — a 1-byte type prefix + payload (owrx/connection.py:473-481)"""
    from openwebrx_b200 import ChannelBank, Waterfall
    from openwebrx_b200.synth import BANDPASS, carrier_plan, make_iq
    fs = 2.4e6
    cars = carrier_plan(2, fs, seed=81)
    iq = make_iq(5333 + 200 * 3000 + 5000, fs, cars, seed=81)
    wf_a, wf_b = Waterfall(fs, 1024, 0.3, 60, "adpcm"), Waterfall(fs, 1024, 0.3, 60, "adpcm")
    plain = wf_a.feed(iq)
    N.check(N.lib.owrx_wf_feed(wf_b._h, iq.ctypes.data, iq.size))
    msgs = wf_b.read_messages()
    assert len(msgs) == len(plain) >= 4 and all(m == b"\x01" + l for m, l in zip(msgs, plain))
    out = {}
    for framed in (False, True):
        bank = ChannelBank(fs)
        ch = bank.add_channel(12000, demod="nfm", offset=cars[0]["offset"], bandpass=BANDPASS["nfm"])
        ch.setAudioFormat("adpcm")
        bank.feed(iq)
        if framed:
            m = ch.read_message(cap=1 << 20)
            assert m[:1] == b"\x02" and ch.read_message() is None
            out[framed] = m[1:]
        else:
            out[framed] = bytes(ch.read_bytes())
        bank.close()
    assert out[True] == out[False] and out[True][:4] == b"SYNC"
    with pytest.raises(ValueError):
        N.check(N.lib.owrx_chan_read_message(ChannelBank(fs)._h, 0, 3, iq.ctypes.data, 10, None))


def test_f4_source_side_convert_chain_through_the_shim(gpu):
    """the reference's source-side conversion chain (owrx/source/fifi_sdr.py:27-28) in front of a waterfall chain and a
    client chain, all through the pycsdr shim: raw int16 samples go to the GPU as they are; results equal the library fed
    with the oracle's Convert + Gain output"""
    from openwebrx_b200 import ChannelBank, Waterfall
    fs = 2.4e6
    cars = carrier_plan(2, fs, seed=91)
    iq = make_iq(5333 + 200 * 2250 + 4099, fs, cars, seed=91)
    raw = (np.clip(iq.view(np.float32), -1, 1) * 6000).astype(np.int16)         # x 5.0 stays within +-1
    as_float = oracle.convert_raw_iq(raw, "cs16", 5.0)
    # ---- the shim topology: Buffer(CS16) -> Convert -> Gain(5) -> Buffer(CF32) -> {FftChain modules, Selector-like chain}
    src = M.Buffer(Format.COMPLEX_SHORT)
    conv, gain = M.Convert(Format.COMPLEX_SHORT, Format.COMPLEX_FLOAT), M.Gain(Format.COMPLEX_FLOAT, 5.0)
    mid, fbuf = M.Buffer(Format.COMPLEX_FLOAT), M.Buffer(Format.COMPLEX_FLOAT)
    conv.setWriter(mid); gain.setReader(mid.getReader()); conv.setReader(src.getReader()); gain.setWriter(fbuf)
    avg, every_n = 4, 700
    fft, lap, swap, ad = M.Fft(size=1024, every_n_samples=every_n), M.LogAveragePower(add_db=-70.0, fft_size=1024, avg_number=avg), \
        M.FftSwap(fft_size=1024), M.FftAdpcm(fft_size=1024)
    b1, b2, b3, out = M.Buffer(Format.COMPLEX_FLOAT), M.Buffer(Format.FLOAT), M.Buffer(Format.FLOAT), M.Buffer(Format.CHAR)
    fft.setWriter(b1); lap.setReader(b1.getReader()); lap.setWriter(b2); swap.setReader(b2.getReader()); swap.setWriter(b3)
    ad.setReader(b3.getReader()); ad.setWriter(out)
    rd = out.getReader()
    fft.setReader(fbuf.getReader())
    time.sleep(0.3)
    n_lines = ((len(iq) - 1024) // every_n + 1) // avg
    src.write(raw.tobytes())
    lines = []
    deadline = time.time() + 20
    while len(lines) < n_lines and time.time() < deadline:
        d = rd.read()
        if d is None:
            break
        lines.append(bytes(d))
    want = oracle.fftchain_run(as_float, 1024, every_n, avg)
    assert len(lines) == n_lines == len(want["lines"])
    wf = Waterfall(fs, 1024, 0.0, 1, "adpcm")
    N.check(N.lib.owrx_wf_set_every_n_samples(wf._h, every_n)); N.check(N.lib.owrx_wf_set_avg_number(wf._h, avg))
    direct = wf.feed(as_float)
    assert lines == direct                                                    # same bytes as the library fed with floats
    for m in (fft, lap, swap, ad, conv, gain):
        m.stop()
    rd.stop()
