"""GPU parity of the squelched low-rate tail: Squelch -> demodulator front -> DcBlock / NfmDeemphasis -> Agc, with the gate
closing and reopening across feeds.

The reference is the oracle's stage functions applied to the GPU's OWN IF (read_if), so an error of Shift / FirDecimate /
Bandpass can neither hide nor fake an error of the tail.  Carriers are keyed on and off at squelch-block boundaries and every
squelch level sits at a tenth of its carrier's power, so no gate decision is close to its level (asserted).  Every feed here
stays below one upload chunk (2^21 samples), so one feed is one pass of the low-rate stages, and the per-feed output counts
give the pass boundaries; each test asserts from them and from the oracle's gate sequence that the case it is about happened.
"""
import numpy as np
import pytest

import oracle
from openwebrx_b200 import ChannelBank
from openwebrx_b200 import _native as N
from openwebrx_b200.synth import BANDPASS, make_iq

pytestmark = pytest.mark.gpu

TOL = 1e-4                   # north_star: demodulated audio within 1e-4 relative RMS (float32), pre-AGC
CHUNK = 1 << 21              # host feeds are uploaded and processed in passes of this many samples
HANG_BLOCKS = 2              # Squelch hangLength = 2 x length (csdr/chain/selector.py:124)
AMP = 0.1
POWER = {"nfm": AMP ** 2, "am": 0.5 * AMP ** 2, "usb": 0.5 * AMP ** 2, "wfm": AMP ** 2}   # mean |IF|^2 of a keyed-on carrier
AGC_DEFAULTS = {"nfm": (1.0, 3.0), "am": (200.0, 65535.0), "usb": (1.0, 65535.0)}      # analog.py:13-15, 37-39, 121-122


# ------------------------------------------------------------------------------------------------ signals and schedules
def _geometry(fs, out):
    D, frac, transition, _ = oracle.decimator_params(fs, out)
    return D, frac, oracle.filter_len(transition), oracle.filter_len(320.0 / out), int(out / 16)


def _block_edges(fs, out, n_blocks):
    """input sample at which the IF of squelch block b begins (FirDecimate centre, FractionalDecimator lead and the band-pass
    group delay undone), so that a carrier keyed there fills whole blocks up to a few percent at the edges"""
    D, frac, T, Tb, L = _geometry(fs, out)
    rows = np.arange(n_blocks + 1, dtype=np.float64) * L - (Tb - 1) / 2
    pre = rows * frac + (5.0 if frac != 1.0 else 0.0)
    return np.maximum(np.round(pre * D + (T - 1) / 2).astype(np.int64), 0)


def _keyed_iq(n, fs, out, cars, key, seed):
    """noise floor + carriers; every carrier is on in the squelch blocks where key is True"""
    edges = _block_edges(fs, out, len(key))
    env = np.zeros(n, np.float32)
    for b, on in enumerate(key):
        if on:
            env[min(edges[b], n):min(edges[b + 1], n)] = 1.0
    env[min(edges[-1], n):] = 1.0 if key[-1] else 0.0
    x = make_iq(n, fs, [], seed=seed)
    for c in cars:
        x += make_iq(n, fs, [c], seed=seed, noise=0.0) * env
    return x


def _level_db(kind):
    return 10 * np.log10(0.1 * POWER[kind])


def _feed_all(bank, chans, iq, cuts, mpx=False):
    """feed iq[cuts[i]:cuts[i+1]] one after another; returns per channel the concatenated outputs (the multiplex tap too if
    mpx) and the per-feed demod counts"""
    got = [dict(if_=[], demod=[], audio=[], power=[], mpx=[]) for _ in chans]
    for i in range(len(cuts) - 1):
        assert cuts[i + 1] - cuts[i] <= CHUNK
        bank.feed(iq[cuts[i]:cuts[i + 1]])
        for g, ch in zip(got, chans):
            g["if_"].append(ch.read_if())
            g["demod"].append(ch.read_demod())
            g["audio"].append(ch.read_audio())
            g["power"].append(ch.read_power())
            if mpx:
                g["mpx"].append(ch.read_mpx())
    out = []
    for g in got:
        r = {k: np.concatenate(v) if v else np.empty(0, np.float32) for k, v in g.items()}
        r["counts"] = [len(d) for d in g["demod"]]
        out.append(r)
    return out


def _phase_schedule():
    """(key per block, block count per pass) for 2.4 MS/s -> 12 kHz.  A run of c closed blocks is c + 2 blocks below the level
    (the hang keeps the first two open).  Each run's first below-level block sits at pass block k: k = 0..3 (the pass starts
    with carried hang 2), k = -1 / -2 (the run began in the previous pass: carried hang 1 / 0), k = -(c + 2) (the closed run
    ends with the previous pass: the carrier returns at pass block 0 with carried hang 0)."""
    key, passes = [1, 1, 1], [3]
    for c in (1, 2, 3, 4):
        R = c + 2
        for k in (0, 1, 2, 3):
            key += [1] * k + [0] * R + [1]
            passes.append(k + R + 1)
        for k in (1, 2, R):
            key += [1] + [0] * k
            passes.append(1 + k)
            key += [0] * (R - k) + [1, 1]
            passes.append(R - k + 2)
    return [bool(v) for v in key], passes


def _cuts_for_passes(passes, D, T, L, rng):
    """feed cuts that end pass p exactly after its last block (plus a ragged remainder of rows and samples that stays pending)"""
    cuts, B = [0], 0
    for nb in passes:
        B += nb
        rows = B * L + int(rng.integers(0, L))
        cuts.append(T + D * (rows - 1) + int(rng.integers(0, D)))
    return cuts


# ------------------------------------------------------------------------------------------------ references and checks
def _gate(power, level):
    """Squelch decisions per block from the oracle's block powers; level: one float32 level per block"""
    open_, hang = np.zeros(len(power), bool), 0
    for b, p in enumerate(power):
        if p >= level[b]:
            open_[b], hang = True, HANG_BLOCKS
        elif hang > 0:
            open_[b], hang = True, hang - 1
    return open_


def _hangs(power, level):
    """hang counter after every block (what a pass starting behind that block carries)"""
    h, out = 0, []
    for b, p in enumerate(power):
        h = HANG_BLOCKS if p >= level[b] else max(h - 1, 0)
        out.append(h)
    return out


def _block_powers(if_, L):
    _, pw = oracle.squelch(if_, L, 5, 2 * L, 0.0, 1)
    return pw


def _reference_demod(kind, gated, L, out):
    if kind == "usb":
        return gated.real.astype(np.float32)
    if kind == "am":
        return oracle.dc_block(oracle.am_demod(gated), L)
    return oracle.fir_f(oracle.limit(oracle.fm_demod(gated)), oracle.nfm_deemphasis_taps(out))


def _check_tail(kind, r, level_db, L, out, level_per_block=None):
    """the checks of one squelched channel against the oracle over its own IF; returns (gate per block, block powers)"""
    if_, dm = r["if_"], r["demod"]
    nb = len(if_) // L
    assert len(dm) == nb * L and nb > 0
    pw = _block_powers(if_, L)
    assert len(pw) == nb
    level = np.full(nb, np.float32(10.0 ** (level_db / 10.0)), np.float32) if level_per_block is None else level_per_block
    # the GPU's squelch power (every reportInterval = 4th block) is the oracle's, and no decision is ambiguous
    assert len(r["power"]) == len(pw[::4]) and np.allclose(r["power"], pw[::4], rtol=1e-5)
    assert np.all(np.abs(pw / level - 1.0) >= 1e-3), float(np.min(np.abs(pw / level - 1.0)))
    gate = _gate(pw, level)
    gated = if_[:nb * L] * np.repeat(gate, L).astype(np.complex64)
    ref = _reference_demod(kind, gated, L, out)
    assert len(ref) == len(dm)
    if kind == "usb":
        assert np.array_equal(dm, ref), int(np.argmax(dm != ref))      # pins the gate of every block exactly
    else:
        scale = np.sqrt(np.mean(ref.astype(np.float64) ** 2))
        err = np.sqrt(np.mean(((dm - ref).astype(np.float64) ** 2).reshape(nb, L), axis=1)) / scale
        assert np.all(err <= TOL), (kind, int(np.argmax(err)), float(err.max()))
    # rows the reference gives as exactly 0.0 behind a closed gate are 0.0 on the GPU: for NFM past the de-emphasis tail of the
    # run's first closed row, for AM from the run's second closed block on (DcBlock ramps from the last open block's mean)
    skip = {"nfm": len(oracle.nfm_deemphasis_taps(out)) - 1, "am": L, "usb": 0}[kind]
    silent = _closed_rows(gate, L, skip) & (ref == 0.0)
    assert np.all(dm[silent] == 0.0), (kind, int(np.argmax(silent & (dm != 0.0))))
    assert (~gate).sum() > 0 and silent.sum() >= L // 2        # the gate really closed, and closed rows came out silent
    return gate, pw, level


def _closed_rows(gate, L, skip):
    """rows of closed blocks that lie at least `skip` rows behind the start of their closed run"""
    closed = np.repeat(~gate, L)
    start = np.flatnonzero(closed & ~np.concatenate([[False], closed[:-1]]))
    since = np.arange(len(closed)) - start[np.maximum(np.searchsorted(start, np.arange(len(closed)), side="right") - 1, 0)] \
        if len(start) else np.zeros(len(closed), np.int64)
    return closed & (since >= skip)


def _pass_starts(counts, L):
    return [int(s) for s in np.cumsum([0] + [n // L for n in counts])[:-1]]


def _runs_by_pass(gate, below, counts, L):
    """{(k, c)} over the closed runs that end inside the stream: c closed blocks, the run's first below-level block at block k
    of the pass that holds it, and at block k < 0 of every later pass up to the one the carrier returns in"""
    starts = _pass_starts(counts, L)
    seen, b = set(), 0
    while b < len(gate):
        if gate[b]:
            b += 1
            continue
        e = b
        while e < len(gate) and not gate[e]:
            e += 1
        k0 = b
        while k0 > 0 and below[k0 - 1]:
            k0 -= 1
        if e < len(gate):
            for s in [max(s for s in starts if s <= k0)] + [s for s in starts if k0 < s <= e]:
                seen.add((k0 - s, e - b))
        b = e
    return seen


# ------------------------------------------------------------------------------------------------ (a) gate, hang, DcBlock
@pytest.fixture(scope="module")
def phase_case():
    fs, out = 2.4e6, 12000
    D, frac, T, Tb, L = _geometry(fs, out)
    assert (D, frac, L) == (200, 1.0, 750)
    key, passes = _phase_schedule()
    cuts = _cuts_for_passes(passes, D, T, L, np.random.default_rng(3))
    cars = [dict(offset=-700000, amp=AMP, kind="nfm"), dict(offset=150000, amp=AMP, kind="am"),
            dict(offset=820000, amp=AMP, kind="usb")]
    iq = _keyed_iq(cuts[-1], fs, out, cars, key, seed=81)
    return dict(fs=fs, out=out, L=L, cars=cars, iq=iq, cuts=cuts, key=key, passes=passes)


def test_gate_hang_and_dc_block_at_every_pass_phase(gpu, phase_case):
    """NFM, AM and USB behind a squelch whose closed runs (1-4 blocks) begin at every pass block 0..3, straddle a pass boundary
    with carried hang 0 / 1 / 2, and end exactly at a pass boundary"""
    p = phase_case
    L, out = p["L"], p["out"]
    bank = ChannelBank(p["fs"], outputs=N.OUT_IF | N.OUT_DEMOD | N.OUT_POWER)
    chans = [bank.add_channel(out, demod=c["kind"], offset=c["offset"], bandpass=BANDPASS[c["kind"]]) for c in p["cars"]]
    for ch, c in zip(chans, p["cars"]):
        ch.setSquelchLevel(_level_db(c["kind"]))
    res = _feed_all(bank, chans, p["iq"], p["cuts"])
    bank.close()
    for c, r in zip(p["cars"], res):
        assert [n // L for n in r["counts"]] == p["passes"] and all(n % L == 0 for n in r["counts"])
        gate, pw, level = _check_tail(c["kind"], r, _level_db(c["kind"]), L, out)
        assert np.array_equal(pw >= level, np.array(p["key"][:len(pw)]))        # the keying is what the squelch saw
        seen = _runs_by_pass(gate, pw < level, r["counts"], L)
        want = {(k, cl) for cl in (1, 2, 3, 4) for k in (-(cl + 2), -2, -1, 0, 1, 2, 3)}
        assert want <= seen, sorted(want - seen)
        # carried hang 0, 1 and 2 all occur at a pass start whose block 0 is below the level
        starts = _pass_starts(r["counts"], L)
        hangs = _hangs(pw, level)
        carried = {hangs[s - 1] for s in starts[1:] if pw[s] < level[s]}
        assert carried == {0, 1, 2}, carried


# ------------------------------------------------------------------------------------------------ (b) every tail-front shape
RATES = [16384, 16400, 24000, 32768, 32784, 48000]


@pytest.mark.parametrize("out", RATES)
def test_every_tail_front_shape(gpu, out, monkeypatch):
    """squelch blocks of 1024 (one tail_front CTA), 1025 (a second CTA with one row), 1500, 2048 (the largest fused block),
    2049 (the first unfused one) and 3000 rows, ragged feeds; the fused form and the seven-kernel form both against the oracle,
    and the launch count says which one ran"""
    fs = 2.4e6
    D, frac, T, Tb, L = _geometry(fs, out)
    key = [bool(v) for v in [1, 1, 1, 0, 0, 0, 0, 1, 1, 0, 0, 0, 0, 0, 1, 0, 1, 1, 0, 0, 0, 1, 1, 1]]
    n = int(_block_edges(fs, out, len(key))[-1]) + T + 3 * D
    rng = np.random.default_rng(out)
    cuts = [0]
    while cuts[-1] < n:
        cuts.append(min(n, cuts[-1] + int(rng.integers(CHUNK // 8, CHUNK // 2))))
    cars = [dict(offset=-600000, amp=AMP, kind="nfm"), dict(offset=250000, amp=AMP, kind="am"),
            dict(offset=760000, amp=AMP, kind="usb")]
    iq = _keyed_iq(n, fs, out, cars, key, seed=82)
    launches, results = {}, {}
    for fused in (True, False):
        monkeypatch.setenv("OWRX_TAIL_FUSED", "1" if fused else "0")
        bank = ChannelBank(fs, outputs=N.OUT_IF | N.OUT_DEMOD | N.OUT_POWER)
        chans = [bank.add_channel(out, demod=c["kind"], offset=c["offset"], bandpass=BANDPASS[c["kind"]]) for c in cars]
        for ch, c in zip(chans, cars):
            ch.setSquelchLevel(_level_db(c["kind"]))
        res = _feed_all(bank, chans, iq, cuts)
        launches[fused] = bank.stats()["kernel_launches"]
        bank.close()
        results[fused] = res
        for c, r in zip(cars, res):
            gate, pw, level = _check_tail(c["kind"], r, _level_db(c["kind"]), L, out)
            assert len(pw) >= len(key) - 1 and np.array_equal(pw >= level, np.array(key[:len(pw)]))
            # some pass starts inside a below-level run, i.e. with the hang counter carried from the pass before
            assert any(0 < s < len(pw) and pw[s - 1] < level[s - 1] for s in _pass_starts(r["counts"], L))
    n_passes = sum(1 for k in results[True][0]["counts"] if k)
    assert n_passes >= 4
    # the fused tail is two launches (tail_front + commit) plus demod_back per pass; the seven-kernel tail counts six
    want = 3 * n_passes if L <= 2048 else 0
    assert launches[False] - launches[True] == want, (L, launches)
    for a, b in zip(results[True], results[False]):
        assert np.array_equal(a["demod"], b["demod"]) and np.array_equal(a["power"], b["power"])


# ------------------------------------------------------------------------------------------------ (c) WFM with squelch
def test_wfm_squelch_unfused_tail(gpu):
    """WFM behind a squelch (250 kHz IF: 15 625-row blocks, the seven-kernel tail): demod against squelch -> FmDemod -> Limit ->
    FractionalDecimator(prefiltered) -> WfmDeemphasis of the GPU's IF, the F32 multiplex tap against Limit(FmDemod) of the
    gated IF.  At 32 784 Hz audio a block makes exactly 2049 audio samples, so passes of 1..8 blocks give de-emphasis passes
    of every length mod 8, 2049 = one past 8 x 256 among them"""
    fs, out, tau = 2.0e6, 250000, 50e-6
    D, frac, T, Tb, L = _geometry(fs, out)
    assert (D, frac, L) == (8, 1.0, 15625)
    passes = [3, 1, 2, 3, 4, 5, 6, 7, 8]
    key = [bool(v) for v in [1, 1, 1, 1, 0, 0, 0, 1, 1, 0, 0, 0, 0, 1, 1, 1, 0, 0, 0, 0, 0, 1, 1, 1, 1, 0, 0, 0, 1, 1, 1, 1,
                             1, 0, 0, 0, 0, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1]]
    rng = np.random.default_rng(7)
    cuts = _cuts_for_passes(passes, D, T, L, rng)
    cars = [dict(offset=-450000, amp=AMP, kind="wfm"), dict(offset=420000, amp=AMP, kind="wfm")]
    rates = [48000.0, 32784.0]
    iq = _keyed_iq(cuts[-1], fs, out, cars, key, seed=83)
    bank = ChannelBank(fs, outputs=N.OUT_AUDIO | N.OUT_IF | N.OUT_DEMOD | N.OUT_POWER)
    chans = []
    for c, ar in zip(cars, rates):
        ch = bank.add_channel(out, demod="wfm", offset=c["offset"], bandpass=BANDPASS["wfm"], audio_rate=ar, tau=tau)
        ch.setSquelchLevel(_level_db("wfm"))
        ch.set_mpx("f32")
        chans.append(ch)
    res = _feed_all(bank, chans, iq, cuts, mpx=True)
    bank.close()
    residues, past_256 = set(), False
    for ar, r in zip(rates, res):
        if_ = r["if_"]
        nb = len(if_) // L
        pw = _block_powers(if_, L)
        level = np.full(nb, np.float32(10.0 ** (_level_db("wfm") / 10.0)), np.float32)
        assert len(r["power"]) == len(pw[::4]) and np.allclose(r["power"], pw[::4], rtol=1e-5)
        assert np.all(np.abs(pw / level - 1.0) >= 1e-3)
        gate = _gate(pw, level)
        assert (~gate).sum() >= 3
        gated = if_[:nb * L] * np.repeat(gate, L).astype(np.complex64)
        mpx_ref = oracle.limit(oracle.fm_demod(gated))
        mpx = r["mpx"]
        assert len(mpx) == nb * L
        err = np.sqrt(np.mean(((mpx - mpx_ref).astype(np.float64) ** 2).reshape(nb, L), axis=1)) / np.sqrt(np.mean(mpx_ref.astype(np.float64) ** 2))
        assert np.all(err <= TOL), float(err.max())
        silent = _closed_rows(gate, L, 0)
        assert np.all(mpx_ref[silent] == 0.0) and np.all(mpx[silent] == 0.0) and silent.sum() >= L
        rr = out / ar
        pre = oracle.firdes_lowpass(oracle.filter_len(0.03), 0.5 / (rr - 0.03))
        ref = oracle.wfm_deemphasis(oracle.fractional_decimator_f(mpx_ref, rr, pre), int(ar), tau)
        dm = r["demod"]
        assert len(dm) == len(ref)
        assert np.array_equal(r["audio"], dm)                  # the WFm chain has no Agc
        scale = np.sqrt(np.mean(ref.astype(np.float64) ** 2))
        per = 1024
        nseg = len(ref) // per
        e = np.sqrt(np.mean(((dm[:nseg * per] - ref[:nseg * per]).astype(np.float64) ** 2).reshape(nseg, per), axis=1)) / scale
        assert np.all(e <= TOL), (ar, int(np.argmax(e)), float(e.max()))
        for k in r["counts"]:
            if k:
                residues.add(k % 8)
                past_256 |= k % 256 == 1
    assert residues == set(range(8)) and past_256, (residues, past_256)


# ------------------------------------------------------------------------------------------------ (d) Agc bit for bit
def _agc_steps(agc, dm, counts):
    """run the oracle Agc over dm in the GPU's pass-relative 128-row steps; returns the outputs and per step
    (zeros, live, hang before, hang after, gain after, attack)"""
    out, steps, pos = [], [], 0
    for n in counts:
        for s in range(0, n, 128):
            x = dm[pos + s:pos + min(s + 128, n)]
            h0 = agc.hang
            out.append(agc.process(x))
            live = int(np.count_nonzero(x))
            attack = agc.hang != max(h0 - live, 0)
            steps.append(dict(zeros=len(x) - live, live=live, h0=h0, gain=agc.gain, max=agc.max_gain, attack=attack))
        pos += n
    return (np.concatenate(out) if out else np.empty(0, np.float32)), steps


AGC_CHANNELS = [("nfm", None), ("am", None), ("usb", None), ("usb", (0.05, 10.0)), ("nfm", (50.0, 2.0)), ("am", (50.0, 2.0))]


@pytest.mark.parametrize("profile", ["slow", "fast"])
def test_agc_bit_exact_through_squelch_gaps(gpu, phase_case, profile):
    """the Agc over streams with runs of exact zeros (closed squelch): the GPU's ballot path, the hang counter carried through
    the zeros, explicit gains (one initial gain above the cap) — read_audio equals the oracle Agc over the channel's own
    read_demod, bit for bit"""
    p = phase_case
    L, out = p["L"], p["out"]
    prof = N.AGC_FAST if profile == "fast" else N.AGC_SLOW
    bank = ChannelBank(p["fs"], outputs=N.OUT_AUDIO | N.OUT_DEMOD)
    car = {c["kind"]: c for c in p["cars"]}
    chans = []
    for kind, gains in AGC_CHANNELS:
        c = car[kind]
        ch = bank.add_channel(out, demod=kind, offset=c["offset"], bandpass=BANDPASS[kind], agc_profile=profile)
        ch.setSquelchLevel(_level_db(kind))
        if gains:
            N.check(N.lib.owrx_chan_set_agc(bank._h, ch.id, prof, gains[0], gains[1]))
        chans.append(ch)
    res = _feed_all(bank, chans, p["iq"], p["cuts"])
    bank.close()
    mixed_attack = entered_with_hang = mixed_rising = at_max = False
    for (kind, gains), r in zip(AGC_CHANNELS, res):
        dm, au = r["demod"], r["audio"]
        assert len(au) == len(dm) > 100 * L
        ini, mx = gains if gains else AGC_DEFAULTS[kind]
        ref, steps = _agc_steps(oracle.AgcStream(1 if profile == "fast" else 0, ini, mx), dm, r["counts"])
        assert np.array_equal(au, ref), (kind, gains, int(np.argmax(au != ref)))
        for s in steps:
            if s["zeros"] and s["live"]:
                mixed_attack |= s["attack"]
                mixed_rising |= s["h0"] < s["live"] and not s["attack"]
            at_max |= s["gain"] == s["max"]
        # a closed run (zeros for more than a block) entered with the hang counter running: the counter must survive the zeros
        agc = oracle.AgcStream(1 if profile == "fast" else 0, ini, mx)
        pos = 0
        for i in np.flatnonzero((dm[1:] == 0.0) & (dm[:-1] != 0.0)) + 1:
            agc.process(dm[pos:i])
            pos = i
            if np.all(dm[i:i + L] == 0.0) and i + L < len(dm) and agc.hang > 0:
                entered_with_hang = True
    assert mixed_attack and mixed_rising and entered_with_hang and at_max, (mixed_attack, mixed_rising, entered_with_hang, at_max)


# ------------------------------------------------------------------------------------------------ (e) control events
def test_control_events_against_the_carried_oracle_state(gpu, phase_case):
    """between feeds: a profile switch, a new initial gain (owrx_chan_set_agc), a max gain below the current gain, a re-mode
    NFM -> AM and a new squelch level.  Each takes effect at the first row of the next feed; the audio from there on must be the
    oracle's, run on from the carried state (or a fresh Agc for the re-mode), bit for bit"""
    p = phase_case
    L, out = p["L"], p["out"]
    car = {c["kind"]: c for c in p["cars"]}
    bank = ChannelBank(p["fs"], outputs=N.OUT_AUDIO | N.OUT_DEMOD | N.OUT_IF | N.OUT_POWER)
    kinds = ["usb", "usb", "nfm", "nfm", "usb"]
    chans = []
    for kind in kinds:
        ch = bank.add_channel(out, demod=kind, offset=car[kind]["offset"], bandpass=BANDPASS[kind])
        ch.setSquelchLevel(_level_db(kind))
        chans.append(ch)
    agcs = [oracle.AgcStream(0, *AGC_DEFAULTS[k]) for k in kinds]
    audio_ref = [[] for _ in chans]
    demod_seen = [[] for _ in chans]
    events = {3: "profile", 6: "gain", 9: "max", 12: "remode", 15: "level"}
    at = {}
    level2 = -110.0                                           # below every noise-only block: the gate stays open

    def between(i):
        ev = events.get(i)
        if ev == "profile":
            N.check(N.lib.owrx_chan_set_agc(bank._h, chans[0].id, N.AGC_FAST, 0.0, 0.0))
            agcs[0].set_profile(1)
        elif ev == "gain":
            N.check(N.lib.owrx_chan_set_agc(bank._h, chans[1].id, N.AGC_SLOW, 7.5, 0.0))
            agcs[1].set_initial_gain(7.5)
        elif ev == "max":
            m = float(np.float32(0.6 * agcs[2].gain))
            assert agcs[2].gain > m
            N.check(N.lib.owrx_chan_set_agc(bank._h, chans[2].id, N.AGC_SLOW, 0.0, m))
            agcs[2].set_max_gain(m)
        elif ev == "remode":
            chans[3].setDemodulator("am")
            agcs[3] = oracle.AgcStream(0, *AGC_DEFAULTS["am"])
        elif ev == "level":
            chans[4].setSquelchLevel(level2)
        if ev:
            at[ev] = i + 1

    got = [dict(if_=[], demod=[], audio=[], power=[]) for _ in chans]
    cuts = p["cuts"]
    for i in range(len(cuts) - 1):
        bank.feed(p["iq"][cuts[i]:cuts[i + 1]])
        for j, ch in enumerate(chans):
            d, a = ch.read_demod(), ch.read_audio()
            got[j]["demod"].append(d)
            got[j]["audio"].append(a)
            got[j]["if_"].append(ch.read_if())
            got[j]["power"].append(ch.read_power())
            audio_ref[j].append(agcs[j].process(d))
        between(i)
    bank.close()
    assert set(at) == set(events.values())
    for j, (ch, g) in enumerate(zip(chans, got)):
        au, ref = np.concatenate(g["audio"]), np.concatenate(audio_ref[j])
        assert len(au) == len(ref) > 50 * L
        assert np.array_equal(au, ref), (j, int(np.argmax(au != ref)))
    # the re-mode: from the next feed the demod is a fresh AM chain (DcBlock from zero) over the gated IF
    counts = [len(d) for d in got[3]["demod"]]
    first = sum(counts[:at["remode"]])
    if_ = np.concatenate(got[3]["if_"])
    dm = np.concatenate(got[3]["demod"])
    nb = len(if_) // L
    pw = _block_powers(if_, L)
    level = np.full(nb, np.float32(10.0 ** (_level_db("nfm") / 10.0)), np.float32)
    gate = _gate(pw, level)
    gated = if_[:nb * L] * np.repeat(gate, L).astype(np.complex64)
    am = oracle.dc_block(oracle.am_demod(gated[first:]), L)
    scale = np.sqrt(np.mean(am.astype(np.float64) ** 2))
    assert first % L == 0 and len(am) == len(dm) - first
    assert np.sqrt(np.mean((dm[first:] - am).astype(np.float64) ** 2)) / scale <= TOL
    # the new squelch level: USB demod is the IF gated with the old level up to the event and the new one after it
    counts = [len(d) for d in got[4]["demod"]]
    first = sum(counts[:at["level"]]) // L
    if_ = np.concatenate(got[4]["if_"])
    nb = len(if_) // L
    lv = np.full(nb, np.float32(10.0 ** (_level_db("usb") / 10.0)), np.float32)
    lv[first:] = np.float32(10.0 ** (level2 / 10.0))
    gate = _gate(_block_powers(if_, L), lv)
    assert not gate[:first].all() and gate[first:].all()
    gated = if_[:nb * L] * np.repeat(gate, L).astype(np.complex64)
    assert np.array_equal(np.concatenate(got[4]["demod"]), gated.real.astype(np.float32))


# ------------------------------------------------------------------------------------------------ (f) the bench's C2 block
def test_c2_block_agc_against_the_oracle(gpu):
    """the bench's own device block (2^24 samples at 10 MS/s, 64 channels in one group, one process_device call): every
    channel's audio is the oracle Agc over its own demod; then again with squelch levels on 16 channels (closing some blocks:
    the Agc's sparse path at the launch shape bench.py times) and the FAST profile on 16 others"""
    import torch
    import bench
    fs, out, n = 10e6, 12000, 1 << 24
    L = int(out / 16)
    cars = bench.channel_plan(0, 64)
    d_iq = bench.synth_iq_torch(n, fs, cars, torch.device("cuda", 0))

    def run(setup):
        bank = ChannelBank(fs, outputs=N.OUT_AUDIO | N.OUT_DEMOD | N.OUT_IF)
        chans = []
        for i, c in enumerate(cars):
            level, profile = setup.get(i, (None, "slow"))
            ch = bank.add_channel(out, demod=c["kind"], offset=c["offset"], bandpass=BANDPASS[c["kind"]], agc_profile=profile)
            if level is not None:
                ch.setSquelchLevel(level)
            chans.append(ch)
        st = torch.cuda.Stream()
        torch.cuda.synchronize()
        bank.process_device(d_iq, n, stream=st.cuda_stream)
        bank.join(st.cuda_stream)
        st.synchronize()
        bank.drain()
        res = [(ch.read_if(), ch.read_demod(), ch.read_audio()) for ch in chans]
        bank.close()
        return res

    def check(res, setup):
        for i, (c, (_, dm, au)) in enumerate(zip(cars, res)):
            assert len(dm) == len(au) >= 26 * L
            prof = 1 if setup.get(i, (None, "slow"))[1] == "fast" else 0
            ref = oracle.AgcStream(prof, *AGC_DEFAULTS[c["kind"]]).process(dm)
            assert np.array_equal(au, ref), (i, c["kind"], int(np.argmax(au != ref)))

    plain = run({})
    check(plain, {})
    # squelch levels at the median block power of 16 channels: their gate closes wherever three blocks in a row fall below it
    closing = []
    for i, (if_, _, _) in enumerate(plain):
        pw = _block_powers(if_, L)
        level = np.float32(np.median(pw))
        gate = _gate(pw, np.full(len(pw), level, np.float32))
        if (~gate).any():
            closing.append((i, float(10 * np.log10(level))))
    assert len(closing) >= 16, len(closing)
    setup = {i: (lv, "slow") for i, lv in closing[:16]}
    fast = [i for i in range(64) if i not in setup][:16]
    setup.update({i: (None, "fast") for i in fast})
    sq = run(setup)
    check(sq, setup)
    assert sum(1 for i in setup if setup[i][0] is not None and (sq[i][1] == 0.0).any()) >= 8
