"""ctypes wrapper around oracle/csdr_oracle.c — the CPU restatement of the csdr arithmetic.

TEST INFRASTRUCTURE ONLY.  Importable from tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs; the product packages (openwebrx_b200, pycsdr) never import it.
PARITY UNPINNED against a pycsdr binary (see csdr_oracle.h).
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "libcsdr_oracle.so")

DEMOD_NFM, DEMOD_AM, DEMOD_SSB, DEMOD_WFM, DEMOD_NONE = 0, 1, 2, 3, 4


def build(force=False):
    srcs = [os.path.join(_HERE, f) for f in ("csdr_oracle.c", "csdr_oracle.h", "Makefile")]
    stale = force or not os.path.exists(_SO) or any(os.path.getmtime(s) > os.path.getmtime(_SO) for s in srcs)
    if stale:
        subprocess.run(["make", "-C", _HERE, "-B"], check=True, capture_output=True)
    return _SO


class ChainCfg(C.Structure):
    _fields_ = [("input_rate", C.c_double), ("output_rate", C.c_double), ("offset_hz", C.c_double),
                ("bp_lo_hz", C.c_double), ("bp_hi_hz", C.c_double), ("demod", C.c_int),
                ("audio_rate", C.c_double), ("wfm_tau", C.c_double), ("agc_profile", C.c_int),
                ("fast_shift", C.c_int)]


class ChainCounts(C.Structure):
    _fields_ = [("n_if", C.c_size_t), ("n_demod", C.c_size_t), ("n_audio", C.c_size_t)]


class Agc(C.Structure):
    _fields_ = [("reference", C.c_float), ("attack", C.c_float), ("decay", C.c_float), ("max_gain", C.c_float),
                ("gain", C.c_float), ("hang_time", C.c_int), ("hang_counter", C.c_int)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        try:
            _lib = C.CDLL(_SO)
        except OSError:
            build(force=True)
            _lib = C.CDLL(_SO)
        L = _lib
        vp, sz, i32, f32, f64 = C.c_void_p, C.c_size_t, C.c_int, C.c_float, C.c_double
        L.oc_filter_len.restype = i32; L.oc_filter_len.argtypes = [f64]
        L.oc_firdes_lowpass.argtypes = [vp, i32, f64]
        L.oc_firdes_bandpass.argtypes = [vp, i32, f64, f64]
        L.oc_fft_window_hamming.argtypes = [vp, i32]
        L.oc_nfm_deemphasis_len.restype = i32; L.oc_nfm_deemphasis_len.argtypes = [i32]
        L.oc_nfm_deemphasis_taps.argtypes = [vp, i32, i32]
        L.oc_fft_forward.argtypes = [vp, vp, i32]
        L.oc_fft_adpcm_quantise.argtypes = [vp, vp, i32]
        L.oc_ima_adpcm_encode.argtypes = [vp, i32, vp, vp, vp]
        L.oc_ima_adpcm_decode.argtypes = [vp, i32, vp, vp, vp]
        L.oc_fft_adpcm.argtypes = [vp, vp, i32]
        L.oc_fftchain_run.restype = sz
        L.oc_fftchain_run.argtypes = [vp, sz, i32, i32, i32, f32, i32, vp, sz, vp, vp]
        L.oc_fftchain_run_nf.restype = sz
        L.oc_fftchain_run_nf.argtypes = [vp, sz, i32, i32, i32, f32, i32, vp, sz, vp, vp, f32, f32, f32]
        L.oc_fftchain_params.argtypes = [f64, i32, f64, f64, vp, vp]
        L.oc_decimator_params.argtypes = [f64, f64, vp, vp, vp, vp]
        L.oc_shift.argtypes = [vp, vp, sz, f64, f64, C.c_uint64, i32]
        L.oc_fir_decimate.restype = sz; L.oc_fir_decimate.argtypes = [vp, sz, vp, i32, i32, vp]
        L.oc_fractional_decimator_cf.restype = sz; L.oc_fractional_decimator_cf.argtypes = [vp, sz, f64, vp, sz]
        L.oc_fractional_decimator_f.restype = sz; L.oc_fractional_decimator_f.argtypes = [vp, sz, f64, vp, i32, vp, sz]
        L.oc_bandpass.argtypes = [vp, sz, vp, i32, vp]
        L.oc_squelch.restype = sz; L.oc_squelch.argtypes = [vp, sz, i32, i32, i32, f32, i32, vp, vp, sz, vp]
        L.oc_am_demod.argtypes = [vp, sz, vp]
        L.oc_fm_demod.argtypes = [vp, sz, vp, vp]
        L.oc_limit.argtypes = [vp, sz]
        L.oc_real_part.argtypes = [vp, sz, vp]
        L.oc_dc_block.argtypes = [vp, sz, i32, vp, vp]
        L.oc_fir_f.argtypes = [vp, sz, vp, i32, vp]
        L.oc_wfm_deemphasis.argtypes = [vp, sz, i32, f64, vp, vp]
        L.oc_agc_init.argtypes = [vp, i32, f32, f32]
        L.oc_agc_process.argtypes = [vp, vp, sz, vp]
        L.oc_convert_f_s16.argtypes = [vp, sz, vp]
        L.oc_convert_s16_f.argtypes = [vp, sz, f32, vp]
        L.oc_convert_u8_f.argtypes = [vp, sz, f32, vp]
        L.oc_adpcm_sync_encode.restype = sz; L.oc_adpcm_sync_encode.argtypes = [vp, sz, vp, sz]
        L.oc_client_chain_run.restype = i32
        L.oc_client_chain_run.argtypes = [vp, vp, sz, vp, sz, vp, sz, vp, sz, vp]
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _cf(a):
    a = np.ascontiguousarray(a, dtype=np.complex64)
    return a


# ---------------------------------------------------------------- design
def filter_len(transition):
    return lib().oc_filter_len(float(transition))


def firdes_lowpass(length, cutoff):
    t = np.empty(length, np.float32)
    lib().oc_firdes_lowpass(_p(t), length, float(cutoff))
    return t


def firdes_bandpass(length, lo, hi):
    t = np.empty(length, np.complex64)
    lib().oc_firdes_bandpass(_p(t), length, float(lo), float(hi))
    return t


def fft_window(n):
    w = np.empty(n, np.float32)
    lib().oc_fft_window_hamming(_p(w), n)
    return w


def nfm_deemphasis_taps(sample_rate):
    n = lib().oc_nfm_deemphasis_len(int(sample_rate))
    t = np.empty(n, np.float32)
    lib().oc_nfm_deemphasis_taps(_p(t), n, int(sample_rate))
    return t


def fftchain_params(samp_rate, fft_size, voverlap, fps):
    a, e = C.c_int(), C.c_int()
    lib().oc_fftchain_params(float(samp_rate), int(fft_size), float(voverlap), float(fps), C.byref(a), C.byref(e))
    return a.value, e.value


def decimator_params(input_rate, output_rate):
    d, fr, tr, cu = C.c_int(), C.c_double(), C.c_double(), C.c_double()
    lib().oc_decimator_params(float(input_rate), float(output_rate), C.byref(d), C.byref(fr), C.byref(tr), C.byref(cu))
    return d.value, fr.value, tr.value, cu.value


# ---------------------------------------------------------------- FftChain
def fft_forward(x):
    x = _cf(x)
    out = np.empty_like(x)
    lib().oc_fft_forward(_p(x), _p(out), len(x))
    return out


def fft_adpcm_quantise(db):
    db = np.ascontiguousarray(db, np.float32)
    s = np.empty(len(db) + 10, np.int16)
    lib().oc_fft_adpcm_quantise(_p(db), _p(s), len(db))
    return s


def ima_adpcm_encode(s, index=0, predictor=0):
    s = np.ascontiguousarray(s, np.int16)
    out = np.empty(len(s) // 2, np.uint8)
    ix, pr = C.c_int(index), C.c_int(predictor)
    lib().oc_ima_adpcm_encode(_p(s), len(s), _p(out), C.byref(ix), C.byref(pr))
    return out, ix.value, pr.value


def ima_adpcm_decode(b, index=0, predictor=0):
    b = np.ascontiguousarray(b, np.uint8)
    out = np.empty(len(b) * 2, np.int16)
    ix, pr = C.c_int(index), C.c_int(predictor)
    lib().oc_ima_adpcm_decode(_p(b), len(b), _p(out), C.byref(ix), C.byref(pr))
    return out


def fft_adpcm(db):
    db = np.ascontiguousarray(db, np.float32)
    out = np.empty((len(db) + 10) // 2, np.uint8)
    lib().oc_fft_adpcm(_p(db), _p(out), len(db))
    return out


def fftchain_run(iq, n, every_n, avg, add_db=-70.0, compression="adpcm", noise_filter=None):
    """Returns dict(lines=bytes array [L, line_bytes], s16=[L, n+10] or None, db=[L, n]).
    noise_filter = (alpha, beta, growth): the spec-defined spectral-subtraction stage of BASELINE config 4."""
    iq = _cf(iq)
    comp = 1 if compression == "adpcm" else 0
    fpl = avg if avg > 0 else 1
    nframes = (len(iq) - n) // every_n + 1 if len(iq) >= n else 0
    L = nframes // fpl
    line_bytes = (n + 10) // 2 if comp else 4 * n
    out = np.empty((max(L, 1), line_bytes), np.uint8)
    s16 = np.empty((max(L, 1), n + 10), np.int16)
    db = np.empty((max(L, 1), n), np.float32)
    if noise_filter is not None:
        a, b, g = noise_filter
        got = lib().oc_fftchain_run_nf(_p(iq), len(iq), n, every_n, avg, add_db, comp, _p(out), out.size, _p(s16), _p(db), a, b, g)
    else:
        got = lib().oc_fftchain_run(_p(iq), len(iq), n, every_n, avg, add_db, comp, _p(out), out.size, _p(s16), _p(db))
    assert got == L, (got, L)
    return dict(lines=out[:L], s16=s16[:L] if comp else None, db=db[:L])


# ---------------------------------------------------------------- Selector stages
def shift(x, rate, phase0=0.0, n0=0, fast=False):
    x = _cf(x)
    y = np.empty_like(x)
    lib().oc_shift(_p(x), _p(y), len(x), float(rate), float(phase0), int(n0), int(fast))
    return y


def fir_decimate(x, taps, D):
    x = _cf(x)
    taps = np.ascontiguousarray(taps, np.float32)
    n_out = (len(x) - len(taps)) // D + 1 if len(x) >= len(taps) else 0
    y = np.empty(max(n_out, 1), np.complex64)
    got = lib().oc_fir_decimate(_p(x), len(x), _p(taps), len(taps), D, _p(y))
    return y[:got]


def fractional_decimator_cf(x, rate):
    x = _cf(x)
    y = np.empty(len(x) + 2, np.complex64)
    got = lib().oc_fractional_decimator_cf(_p(x), len(x), float(rate), _p(y), len(y))
    return y[:got]


def fractional_decimator_f(x, rate, prefilter=None):
    x = np.ascontiguousarray(x, np.float32)
    y = np.empty(len(x) + 2, np.float32)
    if prefilter is None:
        got = lib().oc_fractional_decimator_f(_p(x), len(x), float(rate), None, 0, _p(y), len(y))
    else:
        pre = np.ascontiguousarray(prefilter, np.float32)
        got = lib().oc_fractional_decimator_f(_p(x), len(x), float(rate), _p(pre), len(pre), _p(y), len(y))
    return y[:got]


def bandpass(x, taps):
    x = _cf(x)
    taps = _cf(taps)
    y = np.empty_like(x)
    lib().oc_bandpass(_p(x), len(x), _p(taps), len(taps), _p(y))
    return y


def squelch(x, length, decimation, hang_length, level, report_interval):
    x = _cf(x)
    y = np.empty_like(x)
    pw = np.empty(len(x) // max(length, 1) + 1, np.float32)
    npw = C.c_size_t()
    got = lib().oc_squelch(_p(x), len(x), length, decimation, hang_length, level, report_interval,
                           _p(y), _p(pw), len(pw), C.byref(npw))
    return y[:got], pw[:npw.value]


def am_demod(x):
    x = _cf(x)
    y = np.empty(len(x), np.float32)
    lib().oc_am_demod(_p(x), len(x), _p(y))
    return y


def fm_demod(x):
    x = _cf(x)
    y = np.empty(len(x), np.float32)
    last = np.zeros(1, np.complex64)
    lib().oc_fm_demod(_p(x), len(x), _p(y), _p(last))
    return y


def limit(x):
    y = np.array(x, np.float32, copy=True)
    lib().oc_limit(_p(y), len(y))
    return y


def dc_block(x, block):
    x = np.ascontiguousarray(x, np.float32)
    n = len(x) - len(x) % block
    y = np.empty(max(n, 1), np.float32)
    last = C.c_float(0.0)
    lib().oc_dc_block(_p(x), n, block, _p(y), C.byref(last))
    return y[:n]


def fir_f(x, taps):
    x = np.ascontiguousarray(x, np.float32)
    taps = np.ascontiguousarray(taps, np.float32)
    y = np.empty_like(x)
    lib().oc_fir_f(_p(x), len(x), _p(taps), len(taps), _p(y))
    return y


def wfm_deemphasis(x, sample_rate, tau):
    x = np.ascontiguousarray(x, np.float32)
    y = np.empty_like(x)
    st = C.c_float(0.0)
    lib().oc_wfm_deemphasis(_p(x), len(x), int(sample_rate), float(tau), _p(y), C.byref(st))
    return y


def agc(x, profile=0, initial_gain=1.0, max_gain=65535.0):
    x = np.ascontiguousarray(x, np.float32)
    y = np.empty_like(x)
    a = Agc()
    lib().oc_agc_init(C.byref(a), profile, initial_gain, max_gain)
    lib().oc_agc_process(C.byref(a), _p(x), len(x), _p(y))
    return y


class AgcStream:
    """The Agc as a stream: process() carries gain and hang counter from call to call, and the setters change a live
    instance the way the channel bank's control calls do (Agc.setProfile / setInitialGain / setMaxGain on the running
    module).  A new demodulator means a new Agc: build a fresh instance with that kind's defaults."""

    def __init__(self, profile=0, initial_gain=1.0, max_gain=65535.0):
        self._a = Agc()
        lib().oc_agc_init(C.byref(self._a), int(profile), float(initial_gain), float(max_gain))

    def set_profile(self, profile):
        """decay and hang time of the profile; gain and hang counter run on"""
        fresh = Agc()
        lib().oc_agc_init(C.byref(fresh), int(profile), 1.0, 1.0)
        self._a.decay, self._a.hang_time = fresh.decay, fresh.hang_time

    def set_initial_gain(self, gain):
        if gain > 0:
            self._a.gain = gain

    def set_max_gain(self, gain):
        if gain > 0:
            self._a.max_gain = gain

    @property
    def gain(self):
        return self._a.gain

    @property
    def hang(self):
        return self._a.hang_counter

    @property
    def max_gain(self):
        return self._a.max_gain

    def process(self, x):
        x = np.ascontiguousarray(x, np.float32)
        y = np.empty_like(x)
        lib().oc_agc_process(C.byref(self._a), _p(x), len(x), _p(y))
        return y


def convert_raw_iq(raw, fmt, gain=1.0):
    """source-side Convert (+ Gain): raw int16 ("cs16") / uint8 ("cu8") interleaved I, Q -> complex64"""
    raw = np.ascontiguousarray(raw, np.int16 if fmt == "cs16" else np.uint8)
    out = np.empty(raw.size, np.float32)
    (lib().oc_convert_s16_f if fmt == "cs16" else lib().oc_convert_u8_f)(_p(raw), raw.size, gain, _p(out))
    return out.view(np.complex64)


def convert_f_s16(x):
    x = np.ascontiguousarray(x, np.float32)
    y = np.empty(len(x), np.int16)
    lib().oc_convert_f_s16(_p(x), len(x), _p(y))
    return y


def adpcm_sync_encode(s):
    s = np.ascontiguousarray(s, np.int16)
    out = np.empty(len(s) // 2 + 8 * (len(s) // 2002 + 2), np.uint8)
    got = lib().oc_adpcm_sync_encode(_p(s), len(s), _p(out), len(out))
    return out[:got]


def client_chain_run(iq, input_rate, output_rate, offset_hz, bandpass_hz, demod, audio_rate=48000.0,
                     wfm_tau=50e-6, agc_profile=0, fast_shift=False):
    """Returns dict(if_=complex64, demod=float32 (pre-AGC), audio=float32 (post-AGC))."""
    iq = _cf(iq)
    lo, hi = bandpass_hz if bandpass_hz is not None else (1.0, -1.0)
    cfg = ChainCfg(float(input_rate), float(output_rate), float(offset_hz), float(lo), float(hi), int(demod),
                   float(audio_rate), float(wfm_tau), int(agc_profile), int(fast_shift))
    D = int(input_rate / output_rate)
    cap = len(iq) // D + 8
    if_ = np.empty(cap, np.complex64)
    dm = np.empty(cap, np.float32)
    au = np.empty(cap, np.float32)
    cnt = ChainCounts()
    rc = lib().oc_client_chain_run(C.byref(cfg), _p(iq), len(iq), _p(if_), cap, _p(dm), cap, _p(au), cap, C.byref(cnt))
    assert rc == 0
    return dict(if_=if_[:cnt.n_if], demod=dm[:cnt.n_demod], audio=au[:cnt.n_audio])
