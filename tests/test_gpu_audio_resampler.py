"""GPU tests of the client-audio resampler (owrx_chan_set_audio_resampler): AudioResampler(in, out) -> Limit in front of the
Convert(FLOAT, SHORT) [+ AdpcmEncoder(sync=True)] tail, as the reference's Converter builds it when the client's audio rate
differs from the demodulator's (csdr/chain/clientaudio.py:6-19,34).  The resampler is spec-defined (tests/audio_resampler_ref.py): it is
held to float64 upfirdn of the channel's own float audio, not to libsamplerate."""
import numpy as np
import pytest
from scipy import signal

import audio_resampler_ref
import oracle
import pycsdr.modules as M
from openwebrx_b200 import ChannelBank, _native as N
from openwebrx_b200.synth import BANDPASS, carrier_plan, make_iq
from pycsdr.types import AgcProfile, Format
from test_oracle import JsImaAdpcmCodec

pytestmark = pytest.mark.gpu

C2_RATIOS = [(12000, 11025), (12000, 48000), (48000, 12000)]


def _want_s16(audio, fin, fout):
    """Limit(upfirdn(h, audio)) * 32767 truncated, in float64: what the channel's S16 bytes must be (within 1 LSB)"""
    h, L, Mr, _ = audio_resampler_ref.design(fin, fout)
    n = -(-len(audio) * L // Mr)
    y = np.clip(signal.upfirdn(h, audio.astype(np.float64), L, Mr)[:n], -1.0, 1.0)
    return np.trunc(y * 32767.0)


def _check_s16(got, audio, fin, fout, what):
    want = _want_s16(audio, fin, fout)
    assert len(got) == len(want) > 0, (what, len(got), len(want))
    err = np.abs(got.astype(np.float64) - want)
    rel = float(np.sqrt(np.mean(err ** 2) / max(np.mean(want ** 2), 1.0)))
    assert err.max() <= 1.0 and rel <= 1e-4, (what, float(err.max()), rel)
    return rel


def _gpu_iq(n, fs, cars, seed):
    import torch
    import bench
    return bench.synth_iq_torch(n, fs, cars, torch.device("cuda", 0), seed=seed).cpu().numpy().view(np.complex64).reshape(-1)


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


@pytest.mark.parametrize("mode", ["auto", "direct"])
def test_own_input_exactness_c2_mixed_ratios(gpu, mode):
    """C2 shape (10 MS/s -> 12 kHz, 64 channels in one group): every third channel at each of 12000->11025, 12000->48000 and
    48000->12000 (the ratios are per slot), S16 bytes against the channel's own float audio; the ADPCM bytes of a twin channel
    against the oracle's AdpcmEncoder(sync) of the S16 stream, bit for bit"""
    fs = 10e6
    cars = carrier_plan(62, fs, seed=61)
    iq = _gpu_iq(1 << 23, fs, cars, seed=61)
    bank = ChannelBank(fs, outputs=N.OUT_AUDIO)
    bank.set_fir_mode(mode)
    chans = []
    for i, c in enumerate(cars):
        ch = bank.add_channel(12000, demod=c["kind"], offset=c["offset"], bandpass=BANDPASS[c["kind"]])
        ch.setAudioFormat("s16")
        ch.set_audio_resampler(*C2_RATIOS[i % 3])
        chans.append(ch)
    twins = []
    for c, r in zip(cars[:2], C2_RATIOS):
        t = bank.add_channel(12000, demod=c["kind"], offset=c["offset"], bandpass=BANDPASS[c["kind"]])
        t.setAudioFormat("adpcm")
        t.set_audio_resampler(*r)
        twins.append(t)
    _device_run(bank, iq)
    worst = 0.0
    s16 = []
    for i, ch in enumerate(chans):
        audio = ch.read_audio()
        got = ch.read_bytes().view(np.int16)
        s16.append(got)
        assert len(audio) > 9000
        worst = max(worst, _check_s16(got, audio, *C2_RATIOS[i % 3], what=(mode, i)))
    for i, t in enumerate(twins):
        assert np.array_equal(t.read_bytes(), oracle.adpcm_sync_encode(s16[i]))
    print("[resampler C2] %s->%s: worst rel RMS %.3e" % (mode, bank.fir_form(), worst))
    bank.close()


@pytest.mark.parametrize("mode", ["auto", "direct"])
def test_own_input_exactness_wfm_48000_to_44100(gpu, mode):
    """C5 shape (20 MS/s -> 250 kHz WFM, 8 channels, 48 kHz audio) at 48000 -> 44100"""
    fs = 20e6
    cars = carrier_plan(8, fs, seed=62, wfm=True, span=0.4)
    iq = _gpu_iq(1 << 22, fs, cars, seed=62)
    bank = ChannelBank(fs, outputs=N.OUT_AUDIO)
    bank.set_fir_mode(mode)
    chans = []
    for c in cars:
        ch = bank.add_channel(250000, demod="wfm", offset=c["offset"], bandpass=BANDPASS["wfm"], audio_rate=48000.0, tau=50e-6)
        ch.setAudioFormat("s16")
        ch.set_audio_resampler(48000, 44100)
        chans.append(ch)
    _device_run(bank, iq)
    for i, ch in enumerate(chans):
        _check_s16(ch.read_bytes().view(np.int16), ch.read_audio(), 48000, 44100, what=(mode, i))
    bank.close()


def _small(seed, k=3, blocks=8):
    fs = 2.4e6
    cars = carrier_plan(k, fs, seed=seed)
    return fs, cars, make_iq(5333 + 200 * (750 * blocks + 5), fs, cars, seed=seed)


def _bank(fs, cars, setup, outputs=N.OUT_AUDIO, mode="direct"):
    """one channel per carrier; setup[i] = (format, ratio or None)"""
    bank = ChannelBank(fs, outputs=outputs)
    bank.set_fir_mode(mode)
    chans = []
    for c, (fmt, r) in zip(cars, setup):
        ch = bank.add_channel(12000, demod=c["kind"], offset=c["offset"], bandpass=BANDPASS[c["kind"]])
        ch.setAudioFormat(fmt)
        if r:
            ch.set_audio_resampler(*r)
        chans.append(ch)
    return bank, chans


def test_no_change_for_other_channels_and_one_launch_per_pass(gpu):
    fs, cars, iq = _small(63, k=4)
    outs = N.OUT_AUDIO | N.OUT_IF | N.OUT_POWER
    plain, pc = _bank(fs, cars, [("s16", None), ("adpcm", None), ("f32", None), ("s16", None)], outputs=outs)
    mixed, mc = _bank(fs, cars, [("s16", None), ("adpcm", None), ("f32", None), ("adpcm", (12000, 11025))], outputs=outs)
    for bank in (plain, mixed):
        bank.feed(iq)
    for a, b in zip(pc[:3], mc[:3]):
        assert np.array_equal(a.read_audio(), b.read_audio())
        assert np.array_equal(a.read_if(), b.read_if())
        assert np.array_equal(a.read_power(), b.read_power())
        assert np.array_equal(a.read_bytes(), b.read_bytes())
    assert len(mc[3].read_bytes()) > 0

    def launches(bank):
        n0 = N.lib.owrx_launch_count()
        _device_run(bank, iq)
        return N.lib.owrx_launch_count() - n0
    for bank in (plain, mixed):
        launches(bank)
    n_plain, n_mixed = launches(plain), launches(mixed)
    assert n_mixed == n_plain + 1                           # one resampler launch per tail pass, nothing else
    mc[3].set_audio_resampler(None)
    launches(mixed)
    assert launches(mixed) == launches(plain)


def test_every_delivery_mode_gives_the_same_bytes(gpu):
    fs, cars, iq = _small(64, k=3)
    setup = [("s16", (12000, 11025)), ("adpcm", (12000, 48000)), ("s16", (48000, 12000))]
    got = {}
    bank, chans = _bank(fs, cars, setup)
    bank.feed(iq)
    got["feed"] = [ch.read_bytes() for ch in chans]
    bank, chans = _bank(fs, cars, setup)
    bank.set_deferred_drain(True)
    bank.feed(iq)
    bank.flush()
    got["deferred"] = [ch.read_bytes() for ch in chans]
    bank, chans = _bank(fs, cars, setup)
    _device_run(bank, iq)
    got["drain"] = [ch.read_bytes() for ch in chans]
    bank, chans = _bank(fs, cars, setup)
    _device_run(bank, iq, split=True)
    got["split"] = [ch.read_bytes() for ch in chans]
    for k, v in got.items():
        assert all(len(x) > 0 for x in v), k
        for x, y in zip(v, got["feed"]):
            assert np.array_equal(x, y), k
    # the pipelined device path (whose float audio may differ from the single-stream path in the last bit, resampler or not):
    # the split-phase drain gives what the synchronous drain gives
    piped = {}
    for split in (False, True):
        bank, chans = _bank(fs, cars, setup)
        bank.set_pipelined(True)
        _device_run(bank, iq, split=split)
        piped[split] = [ch.read_bytes() for ch in chans]
    for x, y in zip(piped[True], piped[False]):
        assert len(x) > 0 and np.array_equal(x, y)
    # a ragged feed: the resampler's output does not depend on how its input arrives
    rag, rc = _bank(fs, cars, setup)
    rng = np.random.default_rng(5)
    pos = 0
    while pos < len(iq):
        step = int(rng.integers(1, 150000))
        rag.feed(iq[pos:pos + step])
        pos += step
    for i, (ch, (fmt, r)) in enumerate(zip(rc, setup)):
        audio, b = ch.read_audio(), ch.read_bytes()
        if fmt == "s16":
            _check_s16(b.view(np.int16), audio, *r, what=("ragged", i))
            assert len(b) == len(got["feed"][i])
            one = got["feed"][i].view(np.int16).astype(np.int64)
            assert np.abs(b.view(np.int16).astype(np.int64) - one).max() <= 1


def test_control_path(gpu):
    fs, cars, iq = _small(65, k=1, blocks=12)
    c = cars[0]
    third = len(iq) // 3
    bank, (ch,) = _bank(fs, [c], [("s16", None)])
    bank.feed(iq[:third])
    assert len(ch.read_bytes()) == 2 * len(ch.read_audio())
    # set mid-stream: starts from empty history at the next block
    ch.set_audio_resampler(12000, 11025)
    bank.feed(iq[third:2 * third])
    _check_s16(ch.read_bytes().view(np.int16), ch.read_audio(), 12000, 11025, what="set mid-stream")
    # a new ratio mid-stream starts over as well
    ch.set_audio_resampler(12000, 48000)
    bank.feed(iq[2 * third:])
    _check_s16(ch.read_bytes().view(np.int16), ch.read_audio(), 12000, 48000, what="changed mid-stream")
    # a resampled client leaves while a split-phase drain is pending; its id goes to a new resampled client before _end
    import torch
    bank, (keep, gone) = _bank(fs, [c, c], [("s16", (12000, 11025))] * 2)
    d_iq = torch.from_numpy(iq.view(np.float32)).cuda()
    torch.cuda.synchronize()
    bank.process_device(d_iq, len(iq))
    bank.drain_begin()
    old_id = gone.id
    gone.remove()
    new = bank.add_channel(12000, demod=c["kind"], offset=c["offset"], bandpass=BANDPASS[c["kind"]])
    assert new.id == old_id
    new.setAudioFormat("s16")
    new.set_audio_resampler(12000, 11025)
    bank.drain_end()
    assert len(keep.read_bytes()) > 0
    assert len(new.read_bytes()) == 0
    # rejected: a channel without a demodulator, and a ratio beyond 65536 taps
    nb = ChannelBank(fs)
    none = nb.add_channel(12000, demod="none")
    with pytest.raises(ValueError):
        none.set_audio_resampler(12000, 11025)
    none.set_audio_resampler(None)
    ok = nb.add_channel(12000, demod="nfm")
    with pytest.raises(ValueError):
        ok.set_audio_resampler(48000, 1)
    with pytest.raises(ValueError):
        ok.set_audio_resampler(-1, 12000)


def test_shim_ssb_chain_with_the_client_converter(gpu):
    """Ssb as OpenWebRX builds it, with the Converter for a 44.1 kHz sound card's 11025 Hz client rate:
    ... -> RealPart -> Agc -> AudioResampler(12000, 11025) -> Limit -> Convert(FLOAT, SHORT) -> AdpcmEncoder(sync=True)"""
    fs, out_rate = 2.4e6, 12000
    cars = carrier_plan(3, fs, seed=66)
    c = [x for x in cars if x["kind"] == "usb"][0]
    iq = make_iq(5333 + 200 * (750 * 6 + 5), fs, [c], seed=66)
    agc = M.Agc(Format.FLOAT)
    agc.setProfile(AgcProfile.FAST)
    bp = M.Bandpass(transition=320.0 / out_rate, use_fft=True)
    bp.setBandpass(BANDPASS["usb"][0] / out_rate, BANDPASS["usb"][1] / out_rate)
    sh = M.Shift(0.0)
    sh.setRate(-c["offset"] / fs)
    ws = [sh, M.FirDecimate(200, 0.15 * out_rate / fs, 0.5), bp,
          M.Squelch(Format.COMPLEX_FLOAT, length=750, decimation=5, hangLength=1500, flushLength=3750, reportInterval=4),
          M.RealPart(), agc, M.AudioResampler(12000, 11025), M.Limit(), M.Convert(Format.FLOAT, Format.SHORT),
          M.AdpcmEncoder(sync=True)]
    for a, b in zip(ws[:-1], ws[1:]):
        buf = M.Buffer(a.getOutputFormat())
        a.setWriter(buf)
        b.setReader(buf.getReader())
    out = M.Buffer(Format.CHAR)
    ws[-1].setWriter(out)
    rd = out.getReader()
    src = M.Buffer(Format.COMPLEX_FLOAT)
    sh.setReader(src.getReader())
    raw = iq.tobytes()
    for o in range(0, len(raw), 8 * 100000):
        src.write(raw[o:o + 8 * 100000])
    from test_gpu_pycsdr import _collect
    n_out = -(-4500 * 147 // 160)                                # ceil(4500 * L / M) samples at 11025 Hz
    data = n_out // 2                                            # whole ADPCM bytes; SYNC blocks every 1001 of them
    got = np.asarray(JsImaAdpcmCodec().decodeWithSync(b"".join(_collect(rd, data + 8 * ((data + 1000) // 1001)))), np.float64)
    # the same chain as a bank channel: its S16 bytes are held to its own float audio, and their ADPCM stream decoded is
    # what the shim's client hears (the shim's runner feeds the source in other pieces: within the codec's noise)
    bank = ChannelBank(fs, outputs=N.OUT_AUDIO)
    ch = bank.add_channel(out_rate, demod="usb", offset=c["offset"], bandpass=BANDPASS["usb"], agc_profile="fast")
    ch.setAudioFormat("s16")
    ch.set_audio_resampler(12000, 11025)
    bank.feed(iq)
    s16, audio = ch.read_bytes().view(np.int16), ch.read_audio()
    _check_s16(s16, audio, 12000, 11025, what="shim twin")
    ref = np.asarray(JsImaAdpcmCodec().decodeWithSync(oracle.adpcm_sync_encode(s16).tobytes()), np.float64)
    assert len(got) == len(ref) == 2 * data
    rel = float(np.sqrt(np.mean((got - ref) ** 2) / np.mean(ref ** 2)))
    print("[resampler shim] %d samples, rel RMS against the bank twin %.3e" % (len(got), rel))
    assert rel <= 0.02, rel
    for m in ws:
        m.stop()
