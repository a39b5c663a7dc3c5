"""GPU parity: batched Selector + demodulators (K3/K4/K5) against the CPU oracle, through the C ABI."""
import numpy as np
import pytest

import oracle
from openwebrx_b200 import ChannelBank
from openwebrx_b200 import _native as N
from openwebrx_b200.synth import BANDPASS, carrier_plan, make_iq

pytestmark = pytest.mark.gpu


_FORMS = {
    # name: (OWRX_FIR_MODE, OWRX_FC_TC_FORM, OWRX_FC_M, OWRX_FC_TC_FMT)
    "direct": ("direct", "0", "256", "f16x2"),
    "fastconv": ("fastconv", "0", "256", "f16x2"),
    "fastconv_tc": ("fastconv_tc", "0", "256", "f16x2"),
    "fastconv_tct": ("fastconv_tc", "1", "256", "f16x2"),
    "fastconv_m64": ("fastconv", "0", "64", "f16x2"),
    "fastconv_tct_m64": ("fastconv_tc", "1", "64", "f16x2"),
    "fastconv_tc_bf16x3": ("fastconv_tc", "0", "256", "bf16x3"),
    "fastconv_tct_m64_bf16x3": ("fastconv_tc", "1", "64", "bf16x3"),
}


@pytest.fixture(autouse=True, params=list(_FORMS))
def fir_mode(request, monkeypatch):
    """every parity case runs through all evaluations of Shift + FirDecimate: the direct-form K3 kernel, the polyphase
    fast-convolution path K3F with its contraction on the FP32 pipe, and K3F with the contraction on the tensor cores
    (tcgen05) in both operand arrangements — overlap-save blocks in the MMA's M (fc_contract_tc_kernel) and channel slots in
    M (fc_contract_tct_kernel: what the cost model picks for groups of >= 128 slots and short passes) — with both branch FFT
    sizes (256 points; 64 points: the default of groups with D >= 2048) and both operand splits (block-scaled fp16 x 2: the
    default; bf16 x 3)
    (owrx_bank_create reads every one of these variables: a bank keeps the forms of the environment it was created in)"""
    mode, form, m, fmt = _FORMS[request.param]
    monkeypatch.setenv("OWRX_FIR_MODE", str(N.FIR_MODES[mode]))
    monkeypatch.setenv("OWRX_FC_TC_FORM", form)
    monkeypatch.setenv("OWRX_FC_M", m)
    monkeypatch.setenv("OWRX_FC_TC_FMT", fmt)
    return request.param

AUDIO_TOL = 1e-4       # north_star: demodulated audio within 1e-4 relative RMS (float32), pre-AGC
KIND = {"nfm": oracle.DEMOD_NFM, "am": oracle.DEMOD_AM, "usb": oracle.DEMOD_SSB, "wfm": oracle.DEMOD_WFM}


def rel_rms(a, b):
    n = min(len(a), len(b))
    a = np.asarray(a[:n], np.complex128 if np.iscomplexobj(a) else np.float64)
    b = np.asarray(b[:n], a.dtype)
    den = np.sqrt(np.mean(np.abs(b) ** 2))
    return float(np.sqrt(np.mean(np.abs(a - b) ** 2)) / den) if den > 0 else float(np.sqrt(np.mean(np.abs(a) ** 2)))


def _setup(fs, out_rate, carriers, n_ch, outputs=N.OUT_AUDIO | N.OUT_DEMOD | N.OUT_IF, **kw):
    bank = ChannelBank(fs, outputs=outputs)
    chans = []
    for c in range(n_ch):
        car = carriers[c % len(carriers)]
        ch = bank.add_channel(out_rate, demod=car["kind"], offset=car["offset"], bandpass=BANDPASS[car["kind"]], **kw)
        chans.append((ch, car))
    return bank, chans


def _oracle_chain(iq, fs, out_rate, car, **kw):
    return oracle.client_chain_run(iq, fs, out_rate, car["offset"], BANDPASS[car["kind"]], KIND[car["kind"]], **kw)


def _check(ch, ref, min_len=100):
    if_ = ch.read_if()
    dm = ch.read_demod()
    au = ch.read_audio()
    assert len(if_) == len(ref["if_"])
    assert len(dm) == len(ref["demod"]) and len(dm) >= min_len
    assert len(au) == len(ref["audio"])
    e_if, e_dm = rel_rms(if_, ref["if_"]), rel_rms(dm, ref["demod"])
    assert e_if <= AUDIO_TOL, ("IF", e_if)
    assert e_dm <= AUDIO_TOL, ("demod", e_dm)
    return e_if, e_dm, rel_rms(au, ref["audio"])


def test_rtl_profile_all_modes(gpu):
    # 2.4 MS/s -> 12 kHz: D = 200, T = 5333, no fractional stage
    fs, out = 2.4e6, 12000
    cars = carrier_plan(6, fs, seed=21)
    n = 5333 + 200 * (750 * 3 + 40)
    iq = make_iq(n, fs, cars, seed=21)
    bank, chans = _setup(fs, out, cars, 6)
    bank.feed(iq)
    worst_agc = 0.0
    for ch, car in chans:
        ref = _oracle_chain(iq, fs, out, car)
        _, _, e_au = _check(ch, ref, min_len=2250)
        worst_agc = max(worst_agc, e_au)
    assert worst_agc < 1e-2        # post-AGC is spec-defined (SURVEY A.11); reported, loosely bounded


def test_c2_shape_fractional(gpu):
    # 10 MS/s -> 12 kHz: D = 833, frac = 1.0004, T = 22223 (BASELINE config 2 shape)
    fs, out = 10e6, 12000
    cars = carrier_plan(3, fs, seed=22)
    n = 22223 + 833 * (750 * 2 + 60)
    iq = make_iq(n, fs, cars, seed=22)
    bank, chans = _setup(fs, out, cars, 3)
    bank.feed(iq)
    for ch, car in chans:
        _check(ch, _oracle_chain(iq, fs, out, car), min_len=1500)


def test_c3_shape_r_split(gpu):
    # 61.44 MS/s -> 12 kHz: D = 5120, T = 136533 (BASELINE config 3 shape): the D-sample block is split over
    # 6 CTAs (r-splits) whose partial sums meet in fir_reduce_kernel
    fs, out = 61.44e6, 12000
    cars = carrier_plan(2, fs, seed=28)
    n = 136533 + 5120 * (750 + 40)
    iq = make_iq(n, fs, cars, seed=28)
    bank, chans = _setup(fs, out, cars, 2)
    bank.feed(iq)
    for ch, car in chans:
        _check(ch, _oracle_chain(iq, fs, out, car), min_len=750)


def test_device_path_matches_host_path(gpu):
    # owrx_bank_process_device (+ pipelined side stream) + owrx_bank_drain == owrx_bank_feed
    import torch
    fs, out = 2.4e6, 12000
    cars = carrier_plan(3, fs, seed=29)
    n = 5333 + 200 * (750 * 2 + 10)
    iq = make_iq(n, fs, cars, seed=29)
    bank, chans = _setup(fs, out, cars, 3)
    bank.feed(iq)
    want = [(ch.read_if(), ch.read_demod(), ch.read_audio()) for ch, _ in chans]
    bank2, chans2 = _setup(fs, out, cars, 3)
    bank2.set_pipelined(True)
    d_iq = torch.from_numpy(iq.view(np.float32)).cuda()
    st = torch.cuda.Stream()
    torch.cuda.synchronize()
    bank2.process_device(d_iq, n, stream=st.cuda_stream)
    bank2.drain()
    for (ch, _), (w_if, w_dm, w_au) in zip(chans2, want):
        assert np.array_equal(ch.read_if(), w_if)
        assert np.array_equal(ch.read_demod(), w_dm)
        assert np.array_equal(ch.read_audio(), w_au)


def test_streaming_ragged_equals_one_shot(gpu):
    fs, out = 2.4e6, 12000
    cars = carrier_plan(3, fs, seed=23)
    n = 5333 + 200 * (750 * 4 + 10)
    iq = make_iq(n, fs, cars, seed=23)
    bank, chans = _setup(fs, out, cars, 3)
    rng = np.random.default_rng(1)
    pos = 0
    while pos < n:
        step = int(rng.integers(1, 250000))
        bank.feed(iq[pos:pos + step])
        pos += step
    for ch, car in chans:
        _check(ch, _oracle_chain(iq, fs, out, car), min_len=3000)


def test_many_channels_two_groups_of_64(gpu):
    # 70 channels -> two CTA channel groups; every channel must still match its own oracle chain
    fs, out = 2.4e6, 12000
    cars = carrier_plan(7, fs, seed=24)
    n = 5333 + 200 * (750 + 20)
    iq = make_iq(n, fs, cars, seed=24)
    bank, chans = _setup(fs, out, cars, 70)
    bank.feed(iq)
    refs = {}
    for i, (ch, car) in enumerate(chans):
        key = car["offset"]
        if key not in refs:
            refs[key] = _oracle_chain(iq, fs, out, car)
        _check(ch, refs[key], min_len=750)


def test_wfm_chain(gpu):
    # 2.0 MS/s -> 250 kHz IF (D = 8) -> 48 kHz audio, tau = 50 us  (csdr/chain/analog.py:55-116)
    fs, out = 2.0e6, 250000
    cars = carrier_plan(2, fs, seed=25, wfm=True, span=0.3)
    n = 213 + 8 * (15625 * 3 + 50)
    iq = make_iq(n, fs, cars, seed=25)
    bank, chans = _setup(fs, out, cars, 2, audio_rate=48000.0, tau=50e-6)
    bank.feed(iq)
    for ch, car in chans:
        ref = _oracle_chain(iq, fs, out, car, audio_rate=48000.0, wfm_tau=50e-6)
        _check(ch, ref, min_len=8000)


def test_retune_bandpass_and_errors(gpu):
    fs, out = 2.4e6, 12000
    bank = ChannelBank(fs, outputs=N.OUT_IF)
    ch = bank.add_channel(out, demod="none")
    cars = carrier_plan(2, fs, seed=26)
    iq = make_iq(5333 + 200 * 800, fs, cars, seed=26)
    ch.setFrequencyOffset(cars[1]["offset"])
    ch.setBandpass(-4000, 4000)
    bank.feed(iq)
    ref = oracle.client_chain_run(iq, fs, out, cars[1]["offset"], (-4000, 4000), oracle.DEMOD_NONE)
    got = ch.read_if()
    assert len(got) == len(ref["if_"]) and rel_rms(got, ref["if_"]) <= AUDIO_TOL
    ch.setBandpass(None, None)              # Selector.setBandpass(None, ...) removes the stage
    with pytest.raises(ValueError):
        N.check(N.lib.owrx_chan_set_shift_rate(bank._h, 999, 0.0))
    with pytest.raises(ValueError):
        ChannelBank(-1.0)
    bank.feed(np.empty(0, np.complex64))    # empty block is a no-op
    assert len(ch.read_if()) == 0


def test_squelch_gate_and_power(gpu):
    fs, out = 2.4e6, 12000
    cars = [dict(offset=100000, amp=0.2, kind="nfm")]
    n = 5333 + 200 * (750 * 8)
    iq = make_iq(n, fs, cars, seed=27)
    iq[len(iq) // 2:] *= np.float32(1e-3)          # signal drops 60 dB half way
    bank = ChannelBank(fs, outputs=N.OUT_DEMOD | N.OUT_IF | N.OUT_POWER)
    ch = bank.add_channel(out, demod="nfm", offset=100000, bandpass=BANDPASS["nfm"])
    ch.setSquelchLevel(-30.0)
    bank.feed(iq)
    if_ = ch.read_if()
    sq, pw = oracle.squelch(if_, 750, 5, 1500, 10 ** (-30 / 10), 4)
    power = ch.read_power()
    assert len(power) == len(pw) and np.allclose(power, pw, rtol=1e-5)
    dm = ch.read_demod()
    ref = oracle.fir_f(oracle.limit(oracle.fm_demod(sq)), oracle.nfm_deemphasis_taps(12000))
    assert len(dm) == len(ref) and rel_rms(dm, ref) <= AUDIO_TOL
    assert np.all(dm[-600:] == 0.0) and np.any(dm[:3000] != 0.0)     # closed squelch emits silence (after the hang)


def test_agc_bit_exact_on_own_demod(gpu):
    # the Agc stage is sample-serial; the GPU evaluates it tile-wise (speculative "no attack" trajectory, attacks
    # applied one at a time).  Given the GPU's OWN pre-AGC samples, the oracle's sample-by-sample recurrence must
    # reproduce the GPU audio bit for bit — including level steps that force runs of consecutive attacks.
    fs, out = 2.4e6, 12000
    cars = carrier_plan(6, fs, seed=31)
    n = 5333 + 200 * (750 * 6 + 13)
    iq = make_iq(n, fs, cars, seed=31)
    iq[n // 3: n // 2] *= np.float32(30.0)            # +29.5 dB step: consecutive attacks
    iq[n // 2: 2 * n // 3] *= np.float32(0.01)        # deep fade: hang, then the long decay ramp
    bank, chans = _setup(fs, out, cars, 6, outputs=N.OUT_AUDIO | N.OUT_DEMOD)
    rng = np.random.default_rng(5)
    pos = 0
    while pos < n:
        step = int(rng.integers(1000, 400000))
        bank.feed(iq[pos:pos + step])
        pos += step
    for ch, car in chans:
        dm, au = ch.read_demod(), ch.read_audio()
        assert len(dm) == len(au) >= 4000
        if car["kind"] == "nfm":
            ref = oracle.agc(dm, 0, 1.0, 3.0)             # analog.py:37-39
        elif car["kind"] == "am":
            ref = oracle.agc(dm, 0, 200.0, 65535.0)       # analog.py:13-15
        else:
            ref = oracle.agc(dm, 0, 1.0, 65535.0)         # analog.py:121-122 (bank default profile: slow)
        assert np.array_equal(au, ref), (car["kind"], int(np.argmax(au != ref)))


def test_retune_and_grow_midstream_direct_equals_fastconv(gpu, monkeypatch):
    # control-path events between feeds — a retune (Shift.setRate: the fast-convolution table column of that channel is
    # rebuilt), then 64 more clients (the group's slot layout and every per-slot table grow) — must leave both
    # evaluations of Shift + FirDecimate in agreement, sample for sample within the audio tolerance
    fs, out = 2.4e6, 12000
    cars = carrier_plan(4, fs, seed=33)
    n = 5333 + 200 * (750 * 3 + 7)
    iq = make_iq(n, fs, cars, seed=33)
    a, b = n // 3 + 11, 2 * n // 3 + 5
    got = {}
    for mode in ("direct", "fastconv", "fastconv_tc"):
        monkeypatch.setenv("OWRX_FIR_MODE", str(N.FIR_MODES[mode]))
        bank, chans = _setup(fs, out, cars, 4, outputs=N.OUT_IF | N.OUT_DEMOD)
        bank.feed(iq[:a])
        chans[1][0].setFrequencyOffset(cars[2]["offset"] + 1234)
        bank.feed(iq[a:b])
        extra = [bank.add_channel(out, demod="usb", offset=cars[i % 4]["offset"] + 50 * i, bandpass=BANDPASS["usb"]) for i in range(64)]
        bank.feed(iq[b:])
        got[mode] = [(ch.read_if(), ch.read_demod()) for ch, _ in chans] + [(extra[0].read_if(), extra[0].read_demod()), (extra[63].read_if(), extra[63].read_demod())]
    for other in ("fastconv", "fastconv_tc"):
        for (if_d, dm_d), (if_f, dm_f) in zip(got["direct"], got[other]):
            assert len(if_d) == len(if_f) > 0 and len(dm_d) == len(dm_f)
            assert rel_rms(if_f, if_d) <= AUDIO_TOL, other
            assert rel_rms(dm_f, dm_d) <= AUDIO_TOL, other


def test_prime_decimation_and_block_edges(gpu):
    # D = 211 (prime: nothing to factor for an FFT over the input index — the polyphase form needs no such FFT) and feeds
    # that end exactly on, one before and one after an overlap-save block boundary (Kb = 230 outputs per block)
    fs, out = 211 * 12000.0, 12000
    cars = carrier_plan(3, fs, seed=34)
    T = 5627                                           # filter_len(0.15 * 12000 / fs)
    for n_k in (230 * 3, 230 * 3 - 1, 230 * 3 + 1, 64, 65):
        n = T + 211 * (n_k - 1)
        iq = make_iq(n, fs, cars, seed=34)
        bank, chans = _setup(fs, out, cars, 3, outputs=N.OUT_IF)
        bank.feed(iq)
        for ch, car in chans:
            ref = oracle.client_chain_run(iq, fs, out, car["offset"], BANDPASS[car["kind"]], KIND[car["kind"]])
            got = ch.read_if()
            assert len(got) == len(ref["if_"]) == n_k
            assert rel_rms(got, ref["if_"]) <= AUDIO_TOL


def test_full_size_block_properties(gpu, fir_mode):
    # BASELINE config 2 at full size (10 MS/s, 2^24-sample block, 64 x 12 kHz channels: 88 overlap-save blocks), checked
    # through size-independent properties: (a) partition invariance — the block fed in two ragged parts gives the same
    # streams as one shot; (b) linearity — every stage up to the selector output is linear, and scaling by 1/2 is exact in
    # float32, so IF(x/2) == IF(x)/2 bit for bit; (c) the two evaluations of Shift + FirDecimate agree (checked in the
    # fastconv run against a direct-form bank on 3 of the channels)
    import torch
    import bench
    fs, out, n, n_ch = 10e6, 12000, 1 << 24, 64
    cars = bench.channel_plan(0, n_ch)
    iq = bench.synth_iq_torch(n, fs, cars, torch.device("cuda", 0)).cpu().numpy().view(np.complex64).reshape(-1)

    def run(x, parts, n_channels=n_ch, mode=None):
        bank = ChannelBank(fs, outputs=N.OUT_IF | N.OUT_DEMOD)
        if mode:
            bank.set_fir_mode(mode)
        chans = [bank.add_channel(out, demod=c["kind"], offset=c["offset"], bandpass=BANDPASS[c["kind"]]) for c in cars[:n_channels]]
        pos = 0
        for p in parts + [len(x)]:
            bank.feed(x[pos:p])
            pos = p
        res = [(ch.read_if(), ch.read_demod()) for ch in chans]
        bank.close()
        return res

    one = run(iq, [])
    n_if = len(one[0][0])
    assert n_if >= 20000 and all(len(i) == n_if for i, _ in one)
    two = run(iq, [5_000_003, 5_000_003 + 777])
    half = run(iq * np.float32(0.5), [])
    for c in range(n_ch):
        assert len(two[c][0]) == n_if and len(two[c][1]) == len(one[c][1])
        # the noise floor of the evaluation itself (block partition differs between the two feeds): FP32-pipe forms 1e-5,
        # bf16x3 tensor-core contraction 3e-5 on the weakest channels (50 dB below the wideband power), 4e-5 with 64-point
        # branch FFTs (six times the overlap-save blocks: measured 3.1e-5; not the size AUTO uses at D = 833); the spec is 1e-4
        floor = 4e-5 if fir_mode.startswith("fastconv_tct_m64") else 3e-5 if fir_mode.startswith("fastconv_tc") else 1e-5
        assert rel_rms(two[c][0], one[c][0]) <= floor, c
        assert rel_rms(two[c][1], one[c][1]) <= AUDIO_TOL, c
        assert np.array_equal(half[c][0], one[c][0] * np.complex64(0.5)), c
    if fir_mode != "direct":
        direct = run(iq, [], n_channels=3, mode="direct")
        for c in range(3):
            assert rel_rms(one[c][0], direct[c][0]) <= AUDIO_TOL, c


def test_read_audio_all_equals_per_channel_reads(gpu):
    fs, out = 2.4e6, 12000
    cars = carrier_plan(5, fs, seed=41)
    iq = make_iq(5333 + 200 * 1500, fs, cars, seed=41)
    per_chan, batched = [], None
    for use_all in (False, True):
        bank, chans = _setup(fs, out, cars, 5, outputs=N.OUT_AUDIO)
        bank.feed(iq)
        if use_all:
            buf = np.zeros((5, 4096), np.float32)
            counts = bank.read_audio_all([ch for ch, _ in chans], buf)
            batched = [buf[i, :counts[i]].copy() for i in range(5)]
            assert bank.read_audio_all([ch for ch, _ in chans], buf) == [0] * 5          # queues are empty now
        else:
            per_chan = [ch.read_audio() for ch, _ in chans]
        bank.close()
    for a, b in zip(per_chan, batched):
        assert len(a) == len(b) > 1000 and np.array_equal(a, b)


def test_deferred_drain_streams_the_same_outputs(gpu):
    # streaming mode (owrx_bank_set_deferred_drain): a feed returns before its last outputs are drained; they arrive with the
    # next feed or flush().  Everything popped in total must equal the synchronous mode bit for bit, including a retune and
    # a new client between feeds (reconfiguration completes the pending feed first) and ADPCM client audio bytes.
    fs, out = 2.4e6, 12000
    cars = carrier_plan(4, fs, seed=61)
    n = 5333 + 200 * 6000
    iq = make_iq(n, fs, cars, seed=61)
    cuts = [0, 400_003, 400_003 + 2_200_000 // 3, 900_001, n]
    got = {}
    for deferred in (False, True):
        bank, chans = _setup(fs, out, cars, 4, outputs=N.OUT_AUDIO | N.OUT_IF)
        chans[3][0].setAudioFormat("adpcm")
        bank.set_deferred_drain(deferred)
        audio = [[] for _ in range(5)]
        if_ = [[] for _ in range(5)]
        raw = []
        extra = None
        for k in range(len(cuts) - 1):
            bank.feed(iq[cuts[k]:cuts[k + 1]])
            if k == 1:
                chans[1][0].setFrequencyOffset(cars[2]["offset"] + 777)
                extra = bank.add_channel(out, demod="usb", offset=cars[0]["offset"] + 300, bandpass=BANDPASS["usb"])
            allch = [c for c, _ in chans] + ([extra] if extra is not None else [])
            for i, c in enumerate(allch):
                audio[i].append(c.read_audio()); if_[i].append(c.read_if())
            raw.append(chans[3][0].read_bytes())
        bank.flush()
        allch = [c for c, _ in chans] + [extra]
        for i, c in enumerate(allch):
            audio[i].append(c.read_audio()); if_[i].append(c.read_if())
        raw.append(chans[3][0].read_bytes())
        got[deferred] = ([np.concatenate(a) for a in audio], [np.concatenate(a) for a in if_], b"".join(bytes(r) for r in raw))
        bank.close()
    for i in range(5):
        assert len(got[True][0][i]) == len(got[False][0][i]) and len(got[True][1][i]) == len(got[False][1][i]) > 0
        assert np.array_equal(got[True][0][i], got[False][0][i]), i
        assert np.array_equal(got[True][1][i], got[False][1][i]), i
    assert got[True][2] == got[False][2] and len(got[True][2]) > 1000


def test_fused_tail_equals_the_seven_kernel_tail(gpu, monkeypatch):
    """tail_front_kernel (Squelch + demodulator front + DcBlock means in one launch, gate from local block powers) against the
    seven-kernel low-rate tail it replaces for short squelch blocks, bit for bit — ragged streaming feeds, a squelched channel,
    all three demodulators"""
    fs, out = 2.4e6, 12000
    cars = carrier_plan(7, fs, seed=61)
    iq = make_iq(5333 + 200 * (750 * 9 + 123), fs, cars, seed=61)
    iq[200 * 750 * 3:200 * 750 * 6] *= 1e-4                       # a quiet stretch: squelched channels close and reopen

    def run(tail_fused):
        monkeypatch.setenv("OWRX_TAIL_FUSED", "1" if tail_fused else "0")
        bank = ChannelBank(fs, outputs=N.OUT_AUDIO | N.OUT_DEMOD | N.OUT_POWER)
        chans = [bank.add_channel(out, demod=c["kind"], offset=c["offset"], bandpass=BANDPASS[c["kind"]]) for c in cars]
        for ch, c in zip(chans[:4], cars):
            ch.setSquelchLevel(10 * np.log10(max(0.3 * c["amp"] ** 2, 1e-12)))
        pos = 0
        for cut in (200 * 2000 + 17, 200 * 2900, 200 * 5100 + 3, len(iq)):
            bank.feed(iq[pos:cut])
            pos = cut
        res = [(ch.read_demod(), ch.read_audio(), ch.read_power()) for ch in chans]
        bank.close()
        return res

    ref = run(False)
    new = run(True)
    assert len(ref[0][0]) >= 750 * 8
    for (d0, a0, p0), (d1, a1, p1) in zip(ref, new):
        assert np.array_equal(d0, d1) and np.array_equal(a0, a1) and np.array_equal(p0, p1)
    assert any((d == 0).any() and (d != 0).any() for d, _, _ in new[:4])      # the gate really closed somewhere
