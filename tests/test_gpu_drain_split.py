"""Split-phase drain of the device path (owrx_bank_drain_begin / _end): block i's outputs are copied to the host while block
i + 1 is already being processed; queues must receive exactly what the synchronous owrx_bank_drain delivers."""
import numpy as np
import pytest

from openwebrx_b200 import ChannelBank
from openwebrx_b200 import _native as N
from openwebrx_b200.synth import BANDPASS, carrier_plan, make_iq

pytestmark = pytest.mark.gpu


def _blocks(fs, cars, n_blocks, n):
    # one continuous stream cut into [carry | new] blocks the way a streaming host presents them
    return make_iq(n * n_blocks + 4096, fs, cars, seed=11)


def _dev(x):
    import torch
    return torch.from_numpy(np.ascontiguousarray(x).view(np.float32)).cuda()


# fallback: S-meter power reports and two client-audio formats, with which drain_begin completes the drain at once
@pytest.mark.parametrize("pipelined, fallback", [(False, False), (True, False), (False, True), (True, True)],
                         ids=["False", "True", "fallback-False", "fallback-True"])
def test_split_phase_drain_equals_synchronous_drain(gpu, pipelined, fallback):
    import torch
    fs, out, n, n_blocks = 2.4e6, 12000, 1 << 19, 5
    cars = carrier_plan(6, fs, seed=9)
    iq = _blocks(fs, cars, n_blocks, n)

    def run(split):
        bank = ChannelBank(fs, outputs=N.OUT_AUDIO | N.OUT_DEMOD | N.OUT_IF | (N.OUT_POWER if fallback else 0))
        chans = [bank.add_channel(out, demod=c["kind"], offset=c["offset"], bandpass=BANDPASS[c["kind"]]) for c in cars]
        if fallback:
            chans[1].setAudioFormat("s16")
            chans[2].setAudioFormat("adpcm")
        bank.set_pipelined(pipelined)
        st = torch.cuda.Stream()
        got = [[[], [], [], [], [], []] for _ in chans]

        def pop():
            for i, ch in enumerate(chans):
                for q, x in zip(got[i], (ch.read_audio(), ch.read_demod(), ch.read_if(), ch.read_power(), ch.read_bytes(),
                                         ch.read_mpx())):
                    q.append(x)

        pos = 0
        keep = []                                   # device blocks stay alive until everything issued on `st` has run
        for b in range(n_blocks):
            blk = torch.from_numpy(iq[pos:pos + n].view(np.float32)).cuda()
            keep.append(blk)
            bank.process_device(blk, n, stream=st.cuda_stream)
            pos += bank.last_consumed()
            if split:
                bank.drain_end()                    # the previous block (no-op for the first)
                if b:
                    pop()
                bank.drain_begin()                  # this block: copied while the next one is processed
            else:
                bank.drain()
                pop()
        if split:
            bank.drain_end()
            pop()
        st.synchronize()
        bank.close()
        return [[np.concatenate(x) for x in ch] for ch in got]

    want, have = run(False), run(True)
    for i, (w, h) in enumerate(zip(want, have)):
        # audio, demod, IF; power; client-audio bytes (S16 and ADPCM channels); the multiplex tap (no WFM channel: none)
        filled = [True] * 3 + [fallback, fallback and i in (1, 2), False]
        for a, b, full in zip(w, h, filled):
            assert len(a) == len(b) and (len(a) > 0) == full
            assert np.array_equal(a, b)


def test_drain_begin_twice_is_refused(gpu):
    import torch
    fs = 2.4e6
    cars = carrier_plan(2, fs, seed=9)
    bank = ChannelBank(fs, outputs=N.OUT_AUDIO)
    for c in cars:
        bank.add_channel(12000, demod=c["kind"], offset=c["offset"], bandpass=BANDPASS[c["kind"]])
    iq = torch.from_numpy(make_iq(1 << 18, fs, cars, seed=3).view(np.float32)).cuda()
    bank.process_device(iq, 1 << 18)
    bank.drain_begin()
    with pytest.raises(Exception):
        bank.drain_begin()
    bank.drain_end()
    bank.drain_end()                                # no-op
    bank.close()


def test_reused_id_gets_nothing_of_a_split_phase_drain(gpu):
    # a client leaves between drain_begin and drain_end and a new client takes its id: the new client's queues stay empty
    fs = 2.4e6
    cars = carrier_plan(2, fs, seed=13)
    bank = ChannelBank(fs, outputs=N.OUT_AUDIO | N.OUT_DEMOD | N.OUT_IF)
    keep, gone = [bank.add_channel(12000, demod=c["kind"], offset=c["offset"], bandpass=BANDPASS[c["kind"]]) for c in cars]
    iq = _dev(make_iq(1 << 19, fs, cars, seed=13))
    bank.process_device(iq, 1 << 19)
    bank.drain_begin()
    old_id = gone.id
    gone.remove()
    new = bank.add_channel(12000, demod=cars[1]["kind"], offset=cars[1]["offset"], bandpass=BANDPASS[cars[1]["kind"]])
    assert new.id == old_id
    bank.drain_end()
    assert len(keep.read_audio()) > 0 and len(keep.read_demod()) > 0 and len(keep.read_if()) > 0
    assert len(new.read_audio()) == 0 and len(new.read_demod()) == 0 and len(new.read_if()) == 0
    bank.close()


def test_power_reports_keep_their_phase_across_device_blocks(gpu):
    # S-meter power is reported for every 4th squelch block of the stream; a device block holds about 1.75 squelch blocks, so
    # the report phase moves from block to block.  Whatever the drain, the reports equal the oracle's over the concatenated IF.
    import oracle
    fs, n = 2.4e6, 1 << 18
    cars = [dict(offset=100000, amp=0.2, kind="nfm")]
    iq = make_iq(5333 + 200 * (750 * 24), fs, cars, seed=27)
    bank = ChannelBank(fs, outputs=N.OUT_IF | N.OUT_POWER)
    ch = bank.add_channel(12000, demod="nfm", offset=100000, bandpass=BANDPASS["nfm"])
    if_, power = [], []
    pos, b = 0, 0
    while pos + n <= len(iq):
        blk = _dev(iq[pos:pos + n])
        bank.process_device(blk, n)                 # (both drains below wait for the block: power reports are on)
        pos += bank.last_consumed()
        if b % 2:
            bank.drain_begin()
            bank.drain_end()
        else:
            bank.drain()
        if_.append(ch.read_if()); power.append(ch.read_power())
        b += 1
    bank.close()
    if_, power = np.concatenate(if_), np.concatenate(power)
    _, pw = oracle.squelch(if_, 750, 5, 1500, 10 ** (-30 / 10), 4)
    assert b >= 10 and len(power) == len(pw) >= 4 and np.allclose(power, pw, rtol=1e-5)


def test_chunked_host_feed_synchronous_equals_deferred(gpu):
    # a feed of more than one 2^21-sample upload chunk drains chunk c - 1 while chunk c is processed; with every output on,
    # that gives byte for byte what the deferred drain delivers after flush()
    fs, n = 2.4e6, 3 << 20
    cars = carrier_plan(3, fs, seed=17)
    wfm = carrier_plan(1, fs, seed=18, wfm=True, span=0.3)
    iq = make_iq(n, fs, cars + wfm, seed=17)
    got = {}
    for deferred in (False, True):
        bank = ChannelBank(fs, outputs=N.OUT_AUDIO | N.OUT_DEMOD | N.OUT_IF | N.OUT_POWER)
        chans = [bank.add_channel(12000, demod=c["kind"], offset=c["offset"], bandpass=BANDPASS[c["kind"]]) for c in cars]
        chans[1].setAudioFormat("s16")
        chans[2].setAudioFormat("adpcm")
        w = bank.add_channel(250000, demod="wfm", offset=wfm[0]["offset"], bandpass=BANDPASS["wfm"], audio_rate=48000.0, tau=50e-6)
        w.set_mpx("f32")
        chans.append(w)
        bank.set_deferred_drain(deferred)
        bank.feed(iq)
        bank.flush()
        got[deferred] = [(ch.read_audio(), ch.read_demod(), ch.read_if(), ch.read_power(), ch.read_bytes(), ch.read_mpx())
                         for ch in chans]
        bank.close()
    for i, (a, b) in enumerate(zip(got[False], got[True])):
        for k, (x, y) in enumerate(zip(a, b)):
            assert len(x) == len(y) and np.array_equal(x, y), (i, k)
            assert len(x) > 0 or (k == 4 and i in (0, 3)) or (k == 5 and i < 3), (i, k)
