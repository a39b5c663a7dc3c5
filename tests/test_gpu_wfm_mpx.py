"""GPU tests of the WFM multiplex tap (owrx_chan_set_mpx): the WFm chain's Limit output that the reference writes into its
metaTapBuffer for the RDS path (csdr/chain/analog.py:62,73-76), gathered from the channel bank per tapped channel."""
import os
import sys
import threading
import time

import numpy as np
import pytest

import oracle
import pycsdr.modules as M
from openwebrx_b200 import ChannelBank, _native as N
from openwebrx_b200.synth import BANDPASS, carrier_plan, make_iq
from pycsdr.types import Format

pytestmark = pytest.mark.gpu

TOL = 1e-4
SQ = 15625                   # squelch block of a 250 kHz IF (Selector: outputRate / 16): the tap advances in whole blocks


def rel_rms(a, b):
    n = min(len(a), len(b))
    a, b = np.asarray(a[:n], np.float64), np.asarray(b[:n], np.float64)
    den = np.sqrt(np.mean(b ** 2))
    return float(np.sqrt(np.mean((a - b) ** 2)) / den)


def _input(fs, k, seed, blocks=3):
    """k WFM carriers, enough IQ for `blocks` squelch blocks of IF (plus the FirDecimate / FractionalDecimator lead)"""
    cars = carrier_plan(k, fs, seed=seed, wfm=True, span=0.3 if fs < 1e7 else 0.4)
    D = int(fs / 250000)
    n = int(round(fs / 250000 * (SQ * blocks + 100))) + int(4 / (0.15 * 250000 / fs)) + D
    return cars, make_iq(n, fs, cars, seed=seed)


def _bank(fs, cars, mpx, outputs=N.OUT_IF, mode="auto"):
    bank = ChannelBank(fs, outputs=outputs)
    bank.set_fir_mode(mode)
    chans = []
    for c, f in zip(cars, mpx):
        ch = bank.add_channel(250000, demod="wfm", offset=c["offset"], bandpass=BANDPASS["wfm"], audio_rate=48000.0, tau=50e-6)
        if f != "off":
            ch.set_mpx(f)
        chans.append(ch)
    return bank, chans


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


@pytest.mark.parametrize("fs", [20e6, 2.4e6])
def test_tap_equals_limit_of_fm_demod_of_the_oracle_if(gpu, fs):
    """C5 shape (20 MS/s -> 250 kHz, D = 80, 3125-tap band-pass, 8 channels) and 2.4 MS/s -> 250 kHz (D = 9 + a fractional
    stage): the F32 tap against Limit(FmDemod(IF)) of the oracle chain, through the form AUTO picks and the direct form"""
    cars, iq = _input(fs, 8 if fs > 1e7 else 3, seed=41)
    refs = [oracle.client_chain_run(iq, fs, 250000, c["offset"], BANDPASS["wfm"], oracle.DEMOD_WFM, audio_rate=48000.0,
                                    wfm_tau=50e-6) for c in cars]
    want = [oracle.limit(oracle.fm_demod(r["if_"])) for r in refs]
    for mode in ("auto", "direct"):
        bank, chans = _bank(fs, cars, ["f32"] * len(cars), mode=mode)
        _device_run(bank, iq)
        worst = 0.0
        for ch, w in zip(chans, want):
            got = ch.read_mpx()
            assert got.dtype == np.float32 and len(got) == 3 * SQ <= len(w)
            worst = max(worst, rel_rms(got, w))
        print("[mpx parity] fs=%g %s->%s: worst rel RMS %.3e (tolerance %g)" % (fs, mode, bank.fir_form(), worst, TOL))
        assert worst <= TOL, (fs, mode, worst)
        bank.close()


def test_s16_tap_is_convert_of_the_f32_tap(gpu):
    fs = 2.4e6
    cars, iq = _input(fs, 1, seed=42)
    bank, (a, b) = _bank(fs, [cars[0], cars[0]], ["f32", "s16"])
    bank.feed(iq)
    f, s = a.read_mpx(), b.read_mpx()
    assert s.dtype == np.int16 and len(f) == len(s) == 3 * SQ
    assert np.array_equal(s, oracle.convert_f_s16(f))


def test_tap_changes_no_other_output_and_no_launch_without_it(gpu):
    fs = 2.4e6
    cars, iq = _input(fs, 3, seed=43)
    outs = N.OUT_AUDIO | N.OUT_IF | N.OUT_POWER
    plain, pc = _bank(fs, cars, ["off"] * 3, outputs=outs)
    tapped, tc = _bank(fs, cars, ["f32", "off", "s16"], outputs=outs)
    for bank in (plain, tapped):
        bank.feed(iq)
    for a, b in zip(pc, tc):
        assert np.array_equal(a.read_audio(), b.read_audio())
        assert np.array_equal(a.read_if(), b.read_if())
        assert np.array_equal(a.read_power(), b.read_power())
    assert len(tc[0].read_mpx()) == 3 * SQ and len(tc[1].read_mpx()) == 0

    def launches(bank):
        n0 = N.lib.owrx_launch_count()
        _device_run(bank, iq)
        return N.lib.owrx_launch_count() - n0
    for bank in (plain, tapped):
        launches(bank)                                # first device block: table builds
    n_plain, n_tapped = launches(plain), launches(tapped)
    assert n_tapped == n_plain + 1                    # one gather per tail pass, nothing else
    for ch in tc:
        ch.set_mpx("off")
    launches(tapped)
    assert launches(tapped) == launches(plain)


def test_every_delivery_mode_gives_the_same_tap(gpu):
    fs = 2.4e6
    cars, iq = _input(fs, 2, seed=44)
    fmts = ["f32", "s16"]
    got = {}
    bank, chans = _bank(fs, cars, fmts)
    bank.feed(iq)
    got["feed"] = [ch.read_mpx() for ch in chans]
    bank, chans = _bank(fs, cars, fmts)
    bank.set_deferred_drain(True)
    bank.feed(iq)
    assert all(len(ch.read_mpx()) == 0 for ch in chans)          # still in flight
    bank.flush()
    got["deferred"] = [ch.read_mpx() for ch in chans]
    bank, chans = _bank(fs, cars, fmts)
    _device_run(bank, iq)
    got["drain"] = [ch.read_mpx() for ch in chans]
    bank, chans = _bank(fs, cars, fmts)
    bank.set_pipelined(True)
    _device_run(bank, iq, split=True)
    got["split"] = [ch.read_mpx() for ch in chans]
    for k, v in got.items():
        assert [len(x) for x in v] == [3 * SQ] * 2, k
        for x, y in zip(v, got["feed"]):
            assert x.dtype == y.dtype and np.array_equal(x, y), k
    # a ragged multi-part feed against the one-shot feed (direct form for both: the per-feed form choice stays out of it)
    one, oc = _bank(fs, cars, ["f32", "f32"], mode="direct")
    one.feed(iq)
    rag, rc = _bank(fs, cars, ["f32", "f32"], mode="direct")
    rng = np.random.default_rng(3)
    pos = 0
    while pos < len(iq):
        step = int(rng.integers(1, 120000))
        rag.feed(iq[pos:pos + step])
        pos += step
    for a, b in zip(oc, rc):
        x, y = a.read_mpx(), b.read_mpx()
        assert len(x) == len(y) == 3 * SQ
        assert rel_rms(y, x) <= 1e-6


def test_tap_control_path(gpu):
    fs = 2.4e6
    cars, iq = _input(fs, 1, seed=45, blocks=6)
    half = len(iq) // 2
    # enabled mid-stream: starts at the next block boundary, equal to the tail of an always-on twin
    bank, (twin, late) = _bank(fs, [cars[0], cars[0]], ["f32", "off"])
    bank.feed(iq[:half])
    first = twin.read_mpx()
    late.set_mpx("f32")
    bank.feed(iq[half:])
    rest, tail = twin.read_mpx(), late.read_mpx()
    assert len(first) > 0 and len(tail) == len(rest) > 0
    assert np.array_equal(tail, rest)
    # a tapped client leaves while a split-phase drain is pending; its id goes to a new tapped client before _end
    import torch
    bank, (keep, gone) = _bank(fs, [cars[0], cars[0]], ["f32", "f32"])
    d_iq = torch.from_numpy(iq.view(np.float32)).cuda()
    torch.cuda.synchronize()
    bank.process_device(d_iq, len(iq))
    bank.drain_begin()
    old_id = gone.id
    gone.remove()
    new = bank.add_channel(250000, demod="wfm", offset=cars[0]["offset"], bandpass=BANDPASS["wfm"], audio_rate=48000.0, tau=50e-6)
    assert new.id == old_id
    new.set_mpx("f32")
    bank.drain_end()
    assert len(keep.read_mpx()) == 6 * SQ                         # the drain did deliver
    assert len(new.read_mpx()) == 0                              # but none of the departed client's multiplex
    # an NFM channel has no multiplex tap
    nb = ChannelBank(fs)
    nfm = nb.add_channel(12000, demod="nfm")
    with pytest.raises(ValueError):
        nfm.set_mpx("f32")
    nfm.set_mpx("off")
    with pytest.raises(ValueError):
        late.set_mpx("mpx")


# ---------------------------------------------------------------- the pycsdr shim, with the reference's meta chain
COPY = "import sys\nwhile True:\n    d = sys.stdin.buffer.read1(65536)\n    if not d:\n        break\n    sys.stdout.buffer.write(d)\n    sys.stdout.buffer.flush()\n"


def _children():
    me, out = os.getpid(), []
    for p in os.listdir("/proc"):
        if p.isdigit():
            try:
                with open("/proc/%s/stat" % p) as f:
                    st = f.read().rsplit(")", 1)[1].split()
            except OSError:
                continue
            if int(st[1]) == me and st[0] != "Z":
                out.append(int(p))
    return out


def test_shim_rds_path_through_exec_module(gpu):
    """WFm as OpenWebRX builds it on the shim, plus its meta chain: Convert(FLOAT, SHORT) on the Limit's buffer, then an
    ExecModule in place of redsea (here a stdin -> stdout copy): the bytes out of it are the bank's own S16 tap"""
    fs, out = 2.4e6, 250000
    cars, iq = _input(fs, 1, seed=46)
    c = cars[0]
    D = int(fs / out)
    sh = M.Shift(0.0)
    sh.setRate(-c["offset"] / fs)
    bp = M.Bandpass(transition=320.0 / out, use_fft=True)
    bp.setBandpass(BANDPASS["wfm"][0] / out, BANDPASS["wfm"][1] / out)
    lim = M.Limit()
    ws = [sh, M.FirDecimate(D, 0.15 * out / fs, 0.5 * D / (fs / out)), M.FractionalDecimator(Format.COMPLEX_FLOAT, (fs / D) / out),
          bp, M.Squelch(Format.COMPLEX_FLOAT, length=out // 16, decimation=5, hangLength=2 * (out // 16)), M.FmDemod(), lim,
          M.FractionalDecimator(Format.FLOAT, 250000.0 / 48000, prefilter=True), M.WfmDeemphasis(48000, 50e-6)]
    for a, b in zip(ws[:-1], ws[1:]):
        buf = M.Buffer(a.getOutputFormat())
        a.setWriter(buf)
        b.setReader(buf.getReader())
    ws[-1].setWriter(M.Buffer(Format.FLOAT))
    conv = M.Convert(Format.FLOAT, Format.SHORT)
    exe = M.ExecModule(Format.SHORT, Format.CHAR, [sys.executable, "-c", COPY])
    conv.setReader(lim._writer.getReader())
    mid, rds = M.Buffer(Format.SHORT), M.Buffer(Format.CHAR)
    conv.setWriter(mid)
    exe.setReader(mid.getReader())
    exe.setWriter(rds)
    rd = rds.getReader()
    src = M.Buffer(Format.COMPLEX_FLOAT)
    sh.setReader(src.getReader())
    src.write(iq.tobytes())                                       # one block: the same FirDecimate pass as bank.feed below
    want_n = 2 * 3 * SQ
    box = []

    def pump():
        while True:
            d = rd.read()
            if d is None:
                break
            box.append(bytes(d))
    th = threading.Thread(target=pump, daemon=True)
    th.start()
    t0 = time.time()
    while sum(len(b) for b in box) < want_n and time.time() - t0 < 60:
        time.sleep(0.02)
    rd.stop()
    th.join(5)
    got = np.frombuffer(b"".join(box), np.int16)
    bank, (ch,) = _bank(fs, [c], ["s16"])
    bank.feed(iq)
    ref = ch.read_mpx()
    assert len(ref) == 3 * SQ and np.array_equal(got, ref)
    pid = exe._proc.pid
    exe.stop()
    conv.stop()
    for m in ws:
        m.stop()
    assert exe._proc.returncode is not None and pid not in _children()
