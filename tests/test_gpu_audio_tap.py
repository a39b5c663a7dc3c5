"""GPU tests of the demodulated-audio tap (owrx_chan_set_audio_tap): the Buffer the primary demodulator's last stage writes (Agc,
or WfmDeemphasis for WFM), which the reference's secondary demodulators read beside the client-audio Converter, gathered from
the channel bank per tapped channel at the demodulator rate.

The reference's secondary-demodulator wiring (owrx/dsp.py, csdr/chain/digimodes.py) is not in this tree and has not been
checked line by line: these tests build that wiring by hand, as a second reader of the demodulator's audio Buffer."""
import threading
import time

import numpy as np
import pytest

import oracle
import pycsdr.modules as M
from openwebrx_b200 import ChannelBank, _native as N
from openwebrx_b200.synth import BANDPASS, carrier_plan, make_iq
from pycsdr.types import AgcProfile, Format

pytestmark = pytest.mark.gpu

BLOCK = 750                  # squelch block of a 12 kHz channel (Selector: outputRate / 16): audio advances in whole blocks


def _gpu_iq(n, fs, cars, seed):
    import torch
    import bench
    return bench.synth_iq_torch(n, fs, cars, torch.device("cuda", 0), seed=seed).cpu().numpy().view(np.complex64).reshape(-1)


def _small(seed, k=3, blocks=8):
    fs = 2.4e6
    cars = carrier_plan(k, fs, seed=seed)
    return fs, cars, make_iq(5333 + 200 * (BLOCK * blocks + 5), fs, cars, seed=seed)


def _device_run(bank, iq, split=False):
    import torch
    d_iq = torch.from_numpy(iq.view(np.float32)).cuda()
    st = torch.cuda.Stream()
    torch.cuda.synchronize()
    bank.process_device(d_iq, len(iq), stream=st.cuda_stream)
    if split:
        bank.drain_begin()
        bank.drain_end()
    else:
        bank.drain()
    st.synchronize()


def _bank(fs, cars, setup, outputs=N.OUT_AUDIO, mode="direct"):
    """one 12 kHz channel per carrier; setup[i] = (audio tap, client-audio format, resampler or None)"""
    bank = ChannelBank(fs, outputs=outputs)
    bank.set_fir_mode(mode)
    chans = []
    for c, (tap, fmt, rs) in zip(cars, setup):
        ch = bank.add_channel(12000, demod=c["kind"], offset=c["offset"], bandpass=BANDPASS[c["kind"]])
        ch.setAudioFormat(fmt)
        if rs:
            ch.set_audio_resampler(*rs)
        if tap != "off":
            ch.set_audio_tap(tap)
        chans.append(ch)
    return bank, chans


def test_c2_tap_is_the_audio_at_the_demodulator_rate(gpu):
    """C2 shape (10 MS/s -> 12 kHz, NFM / AM / USB side by side in one group): the F32 tap equals owrx_chan_read_audio bit for
    bit, whatever the client-audio format and resampler (12000 -> 48000, 12000 -> 11025: the tap stays at 12 kHz with the
    audio's sample count); an S16 twin equals the oracle's Convert(FLOAT, SHORT) of it; untapped channels get nothing"""
    fs = 10e6
    cars = carrier_plan(24, fs, seed=71)
    iq = _gpu_iq(1 << 22, fs, cars, seed=71)
    client = [("f32", None), ("s16", (12000, 48000)), ("adpcm", (12000, 11025)), ("adpcm", None)]
    setup = [("f32" if i % 4 != 3 else "off",) + client[i % 4] for i in range(len(cars))]
    setup += [("s16", "adpcm", None)] * 3                         # S16 twins of the first three (NFM / AM / USB) channels
    bank, chans = _bank(fs, cars + cars[:3], setup, mode="auto")
    _device_run(bank, iq)
    audio = [ch.read_audio() for ch in chans]
    taps = [ch.read_audio_tap() for ch in chans]
    for i, (ch, a, got) in enumerate(zip(chans, audio, taps)):
        if setup[i][0] == "off":
            assert len(got) == 0, i
            continue
        assert len(a) >= 6 * BLOCK, i
        if setup[i][0] == "f32":
            assert got.dtype == np.float32 and np.array_equal(got, a), (i, cars[i]["kind"])
        else:
            assert got.dtype == np.int16 and np.array_equal(got, oracle.convert_f_s16(taps[i - len(cars)])), i
        b = ch.read_bytes()
        rs = setup[i][2]
        if rs == (12000, 48000):
            assert len(b) == 2 * 4 * len(a)                       # the client's S16 is at 48 kHz, the tap at 12 kHz
        elif rs == (12000, 11025):
            assert len(b) > 0
    print("[audio tap C2] %s: %d tapped channels" % (bank.fir_form(), sum(1 for s in setup if s[0] != "off")))
    bank.close()


def test_s16_tap_is_convert_of_the_f32_tap(gpu):
    fs, cars, iq = _small(72, k=3)
    bank, chans = _bank(fs, cars + cars, [("f32", "adpcm", None)] * 3 + [("s16", "adpcm", None)] * 3)
    bank.feed(iq)
    taps = [ch.read_audio_tap() for ch in chans]
    for f, s in zip(taps[:3], taps[3:]):
        assert f.dtype == np.float32 and s.dtype == np.int16 and len(f) == len(s) == 8 * BLOCK
        assert np.array_equal(s, oracle.convert_f_s16(f))


def test_wfm_c5_audio_tap_beside_the_multiplex_tap(gpu):
    """C5 shape (20 MS/s -> 250 kHz WFM, 48 kHz audio): the audio tap equals the audio; the multiplex tap, the audio and the
    client bytes are bit-identical with the audio tap on and off, also where both taps are on one channel"""
    fs = 20e6
    cars = carrier_plan(8, fs, seed=73, wfm=True, span=0.4)
    iq = _gpu_iq(1 << 22, fs, cars, seed=73)
    banks = []
    for tapped in (False, True):
        bank = ChannelBank(fs, outputs=N.OUT_AUDIO)
        chans = []
        for i, c in enumerate(cars):
            ch = bank.add_channel(250000, demod="wfm", offset=c["offset"], bandpass=BANDPASS["wfm"], audio_rate=48000.0, tau=50e-6)
            ch.setAudioFormat("adpcm")
            ch.set_mpx("f32" if i % 2 == 0 else "s16")
            if tapped and i % 4 != 3:
                ch.set_audio_tap("f32" if i % 4 != 2 else "s16")
            chans.append(ch)
        _device_run(bank, iq)
        banks.append((bank, chans))
    (_, plain), (_, tapped) = banks
    for i, (a, b) in enumerate(zip(plain, tapped)):
        audio = a.read_audio()
        assert len(audio) > 5000 and np.array_equal(audio, b.read_audio())
        assert np.array_equal(a.read_mpx(), b.read_mpx())
        assert np.array_equal(a.read_bytes(), b.read_bytes())
        got = b.read_audio_tap()
        if i % 4 == 3:
            assert len(got) == 0
        elif i % 4 == 2:
            assert np.array_equal(got, oracle.convert_f_s16(audio))
        else:
            assert got.dtype == np.float32 and np.array_equal(got, audio)
        assert len(a.read_audio_tap()) == 0
    for bank, _ in banks:
        bank.close()


def test_tap_changes_no_other_output_and_adds_one_launch_per_tapped_group(gpu):
    fs, cars, iq = _small(74, k=3)
    outs = N.OUT_AUDIO | N.OUT_IF | N.OUT_POWER
    client = [("s16", None), ("adpcm", None), ("adpcm", (12000, 11025))]

    def make(taps):
        bank, chans = _bank(fs, cars, [(t,) + c for t, c in zip(taps, client)], outputs=outs)
        # a second group (another output rate) that nobody taps
        other = bank.add_channel(48000, demod="nfm", offset=cars[0]["offset"], bandpass=BANDPASS["nfm"])
        other.setAudioFormat("adpcm")
        return bank, chans + [other]
    plain, pc = make(["off"] * 3)
    tapped, tc = make(["f32", "off", "s16"])
    for bank in (plain, tapped):
        bank.feed(iq)
    for a, b in zip(pc, tc):
        assert np.array_equal(a.read_audio(), b.read_audio())
        assert np.array_equal(a.read_if(), b.read_if())
        assert np.array_equal(a.read_power(), b.read_power())
        assert np.array_equal(a.read_bytes(), b.read_bytes())
    assert len(tc[0].read_audio_tap()) == 8 * BLOCK and len(tc[2].read_audio_tap()) == 8 * BLOCK
    assert len(tc[1].read_audio_tap()) == 0 and len(tc[3].read_audio_tap()) == 0

    def launches(bank):
        n0 = N.lib.owrx_launch_count()
        _device_run(bank, iq)
        return N.lib.owrx_launch_count() - n0
    for bank in (plain, tapped):
        launches(bank)                                # first device block: table builds
    n_plain, n_tapped = launches(plain), launches(tapped)
    assert n_tapped == n_plain + 1                    # one gather per tail pass of the tapped group, none in the other
    for ch in tc[:3]:
        ch.set_audio_tap("off")
    launches(tapped)
    assert launches(tapped) == launches(plain)


def test_every_delivery_mode_gives_the_same_tap(gpu):
    fs, cars, iq = _small(75, k=2)
    setup = [("f32", "adpcm", None), ("s16", "s16", (12000, 48000))]
    got = {}
    bank, chans = _bank(fs, cars, setup)
    bank.feed(iq)
    got["feed"] = [ch.read_audio_tap() for ch in chans]
    bank, chans = _bank(fs, cars, setup)
    bank.set_deferred_drain(True)
    bank.feed(iq)
    assert all(len(ch.read_audio_tap()) == 0 for ch in chans)    # still in flight
    bank.flush()
    got["deferred"] = [ch.read_audio_tap() for ch in chans]
    bank, chans = _bank(fs, cars, setup)
    _device_run(bank, iq)
    got["drain"] = [ch.read_audio_tap() for ch in chans]
    bank, chans = _bank(fs, cars, setup, outputs=N.OUT_IF)       # no client bytes: _begin really splits
    for ch in chans:
        ch.setAudioFormat("f32")
    _device_run(bank, iq, split=True)
    got["split"] = [ch.read_audio_tap() for ch in chans]
    for k, v in got.items():
        assert [len(x) for x in v] == [8 * BLOCK] * 2, k
        for x, y in zip(v, got["feed"]):
            assert x.dtype == y.dtype and np.array_equal(x, y), k
    # the pipelined device path: the split-phase drain gives what the synchronous drain gives, and the audio itself
    piped = {}
    for split in (False, True):
        bank, chans = _bank(fs, cars, setup, outputs=N.OUT_AUDIO)
        for ch in chans:
            ch.setAudioFormat("f32")
        bank.set_pipelined(True)
        _device_run(bank, iq, split=split)
        piped[split] = [(ch.read_audio_tap(), ch.read_audio()) for ch in chans]
    for (x, ax), (y, ay) in zip(piped[True], piped[False]):
        assert len(x) == 8 * BLOCK and np.array_equal(x, y) and np.array_equal(ax, ay)
    assert np.array_equal(piped[True][0][0], piped[True][0][1])
    # a ragged multi-part feed against the one-shot feed
    one, oc = _bank(fs, cars, [("f32", "adpcm", None)] * 2)
    one.feed(iq)
    rag, rc = _bank(fs, cars, [("f32", "adpcm", None)] * 2)
    rng = np.random.default_rng(7)
    pos = 0
    while pos < len(iq):
        step = int(rng.integers(1, 120000))
        rag.feed(iq[pos:pos + step])
        pos += step
    for a, b in zip(oc, rc):
        x, y = a.read_audio_tap(), b.read_audio_tap()
        assert len(x) == len(y) == 8 * BLOCK
        assert np.abs(x.astype(np.float64) - y).max() <= 1e-6


def test_tap_control_path(gpu):
    fs, cars, iq = _small(76, k=3, blocks=12)
    c = [x for x in cars if x["kind"] == "nfm"][0]
    third = len(iq) // 3
    # enabled mid-stream: starts at the next block boundary, equal to the audio from there on
    bank, (twin, late) = _bank(fs, [c, c], [("f32", "adpcm", None), ("off", "adpcm", None)])
    bank.feed(iq[:third])
    assert len(twin.read_audio_tap()) > 0 and len(late.read_audio_tap()) == 0
    late.set_audio_tap("f32")
    late.read_audio()
    bank.feed(iq[third:2 * third])
    tail, rest = late.read_audio_tap(), twin.read_audio_tap()
    assert len(tail) > 0 and np.array_equal(tail, rest) and np.array_equal(tail, late.read_audio())
    # a format change drops what is queued
    bank.feed(iq[2 * third:])
    late.set_audio_tap("s16")
    assert len(late.read_audio_tap()) == 0
    twin.read_audio_tap()
    late.read_audio()
    # the tap survives a re-mode between demodulators (NFM -> USB), and is off after a re-mode to none
    late.setDemodulator("usb")
    iq2 = make_iq(200 * BLOCK * 4, fs, cars, seed=77, t0=len(iq))
    bank.feed(iq2)
    a = late.read_audio()
    assert len(a) > 0 and np.array_equal(late.read_audio_tap(), oracle.convert_f_s16(a))
    late.setDemodulator("none")
    assert late._atap == "off"
    bank.feed(iq2)
    assert len(late.read_audio_tap()) == 0
    with pytest.raises(ValueError):
        late.set_audio_tap("f32")                                # no demodulator: no audio to tap
    late.set_audio_tap("off")
    with pytest.raises(ValueError):
        twin.set_audio_tap("adpcm")
    with pytest.raises(ValueError):
        N.check(N.lib.owrx_chan_set_audio_tap(bank._h, twin.id, 3))
    # a tapped client leaves while a split-phase drain is pending; its id goes to a new tapped client before _end
    import torch
    bank, (keep, gone) = _bank(fs, [c, c], [("f32", "f32", None)] * 2)
    d_iq = torch.from_numpy(iq.view(np.float32)).cuda()
    torch.cuda.synchronize()
    bank.process_device(d_iq, len(iq))
    bank.drain_begin()
    old_id = gone.id
    gone.remove()
    new = bank.add_channel(12000, demod=c["kind"], offset=c["offset"], bandpass=BANDPASS[c["kind"]])
    assert new.id == old_id
    new.set_audio_tap("f32")
    bank.drain_end()
    assert len(keep.read_audio_tap()) == 12 * BLOCK               # the drain did deliver
    assert len(new.read_audio_tap()) == 0                        # but none of the departed client's audio


# ---------------------------------------------------------------- the pycsdr shim, with a secondary demodulator
def _shim_run(c, fs, iq, client, decoder, order, timeout=60.0):
    """Ssb as OpenWebRX builds it on the shim, the client audio chain `client` ("s16" | "adpcm" | "resampler") after the Agc,
    and (decoder=True) a WSJT-style secondary demodulator's Convert(FLOAT, SHORT) -> Buffer on the Agc's Buffer, read by a
    Python thread; constructed before ("first") or after ("last") the client audio chain.  Returns (client bytes, decoder bytes)."""
    out_rate = 12000
    agc = M.Agc(Format.FLOAT)
    agc.setProfile(AgcProfile.FAST)
    bp = M.Bandpass(transition=320.0 / out_rate, use_fft=True)
    bp.setBandpass(BANDPASS["usb"][0] / out_rate, BANDPASS["usb"][1] / out_rate)
    sh = M.Shift(0.0)
    sh.setRate(-c["offset"] / fs)
    ws = [sh, M.FirDecimate(200, 0.15 * out_rate / fs, 0.5), bp,
          M.Squelch(Format.COMPLEX_FLOAT, length=750, decimation=5, hangLength=1500, flushLength=3750, reportInterval=4),
          M.RealPart(), agc]
    for a, b in zip(ws[:-1], ws[1:]):
        buf = M.Buffer(a.getOutputFormat())
        a.setWriter(buf)
        b.setReader(buf.getReader())
    audio = M.Buffer(Format.FLOAT)
    agc.setWriter(audio)

    def add_decoder():
        conv = M.Convert(Format.FLOAT, Format.SHORT)
        conv.setReader(audio.getReader())
        out = M.Buffer(Format.SHORT)
        conv.setWriter(out)
        return conv, out
    dec = add_decoder() if decoder and order == "first" else None
    cl = {"s16": [M.Convert(Format.FLOAT, Format.SHORT)],
          "adpcm": [M.Convert(Format.FLOAT, Format.SHORT), M.AdpcmEncoder(sync=True)],
          "resampler": [M.AudioResampler(12000, 48000), M.Limit(), M.Convert(Format.FLOAT, Format.SHORT),
                        M.AdpcmEncoder(sync=True)]}[client]
    for a, b in zip(cl[:-1], cl[1:]):
        buf = M.Buffer(a.getOutputFormat())
        a.setWriter(buf)
        b.setReader(buf.getReader())
    cl_out = M.Buffer(cl[-1].getOutputFormat())
    cl[-1].setWriter(cl_out)
    cl[0].setReader(audio.getReader())
    if decoder and order == "last":
        dec = add_decoder()
    readers = [cl_out.getReader()] + ([dec[1].getReader()] if dec else [])
    boxes = [[] for _ in readers]

    def pump(rd, box):
        while True:
            d = rd.read()
            if d is None:
                break
            box.append(bytes(d))
    ths = [threading.Thread(target=pump, args=(rd, box), daemon=True) for rd, box in zip(readers, boxes)]
    for th in ths:
        th.start()
    src = M.Buffer(Format.COMPLEX_FLOAT)
    sh.setReader(src.getReader())
    src.write(iq.tobytes())                                      # one block: one feed of the bank
    # 6 squelch blocks of 12 kHz audio: 4500 samples (x4 behind the 12000 -> 48000 resampler); ADPCM: half a byte per sample
    # plus an 8-byte SYNC block per 1001 bytes
    n = 4500 * (4 if client == "resampler" else 1)
    want = [2 * n if client == "s16" else n // 2 + 8 * ((n // 2 + 1000) // 1001)] + ([2 * 4500] if dec else [])
    t0 = time.time()
    while any(sum(len(x) for x in box) < w for box, w in zip(boxes, want)) and time.time() - t0 < timeout:
        time.sleep(0.02)
    time.sleep(0.2)                                              # nothing beyond the block may arrive
    for rd in readers:
        rd.stop()
    for th in ths:
        th.join(5)
    for m in ws + cl + ([dec[0]] if dec else []):
        m.stop()
    got = [b"".join(box) for box in boxes]
    assert [len(g) for g in got] == want, (client, decoder, order, [len(g) for g in got], want)
    return got[0], (got[1] if dec else None)


def test_shim_secondary_demodulator_beside_the_client_audio(gpu):
    """a USB client whose browser audio is Convert -> AdpcmEncoder (directly, or behind AudioResampler(12000, 48000) -> Limit),
    plus a digital-mode decoder's Convert(FLOAT, SHORT) -> Buffer on the Agc's Buffer, in both construction orders: the
    browser's bytes are those of the same chain without the decoder, and the decoder's S16 are the client S16 bytes of an
    otherwise identical chain, bit for bit"""
    fs = 2.4e6
    cars = carrier_plan(3, fs, seed=78)
    c = [x for x in cars if x["kind"] == "usb"][0]
    iq = make_iq(5333 + 200 * (BLOCK * 6 + 5), fs, [c], seed=78)
    s16_ref, _ = _shim_run(c, fs, iq, "s16", False, None)
    for client in ("adpcm", "resampler"):
        ref, _ = _shim_run(c, fs, iq, client, False, None)
        for order in ("first", "last"):
            got, dec = _shim_run(c, fs, iq, client, True, order)
            assert got == ref, (client, order)
            assert dec == s16_ref, (client, order)
