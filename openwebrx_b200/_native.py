"""ctypes binding of libowrx_b200.so (include/owrx_b200.h).

There is no CPU fallback: if the library has not been built (`python openwebrx_b200/_build.py` or
`__graft_entry__.build()`), importing this module raises ImportError; if no sm_100 device is usable
every create call raises RuntimeError.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(HERE, "libowrx_b200.so")

OK, E_INVALID, E_CUDA, E_NOMEM, E_OVERFLOW, E_STATE = 0, -1, -2, -3, -4, -5
COMPRESSION_NONE, COMPRESSION_ADPCM = 0, 1
DEMOD_NFM, DEMOD_AM, DEMOD_SSB, DEMOD_WFM, DEMOD_NONE = 0, 1, 2, 3, 4
AGC_SLOW, AGC_FAST = 0, 1
OUT_AUDIO, OUT_DEMOD, OUT_IF, OUT_POWER = 1, 2, 4, 8
IQ_CF32, IQ_CS16, IQ_CU8 = 0, 1, 2
IQ_FORMATS = {"cf32": IQ_CF32, "cs16": IQ_CS16, "cu8": IQ_CU8}
AUDIO_F32, AUDIO_S16, AUDIO_ADPCM = 0, 1, 2
MPX_OFF, MPX_F32, MPX_S16 = 0, 1, 2          # tap formats: the multiplex tap and the audio tap


class ChanSpec(C.Structure):
    _fields_ = [("decimation", C.c_int), ("transition", C.c_double), ("cutoff", C.c_double), ("fraction", C.c_double),
                ("bp_transition", C.c_double), ("squelch_length", C.c_int), ("deemph_rate", C.c_int), ("wfm", C.c_int),
                ("wfm_decimation", C.c_double), ("wfm_audio_rate", C.c_int), ("wfm_tau", C.c_double)]


class BankStats(C.Structure):
    _fields_ = [("input_samples", C.c_uint64), ("channel_samples", C.c_uint64), ("kernel_launches", C.c_uint64),
                ("device_ms", C.c_double), ("h2d_pinned_bytes", C.c_uint64), ("h2d_pageable_bytes", C.c_uint64)]


if not os.path.exists(SO_PATH):
    raise ImportError(
        "libowrx_b200.so is not built (%s). Run `python openwebrx_b200/_build.py`; this package has no CPU fallback."
        % SO_PATH)

lib = C.CDLL(SO_PATH)

_vp, _sz, _i, _f, _d = C.c_void_p, C.c_size_t, C.c_int, C.c_float, C.c_double
_pp = C.POINTER(C.c_void_p)
_psz = C.POINTER(C.c_size_t)

SIGNATURES = {
    "owrx_last_error": (C.c_char_p, []),
    "owrx_version": (C.c_char_p, []),
    "owrx_launch_count": (C.c_uint64, []),
    "owrx_device_count": (_i, [C.POINTER(_i)]),
    "owrx_pinned_alloc": (_i, [_sz, _pp]),
    "owrx_pinned_free": (None, [_vp]),
    "owrx_host_is_pinned": (_i, [_vp]),
    "owrx_wf_get_h2d_bytes": (_i, [_vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "owrx_iq_multicast_store": (_i, [_vp, _vp, _sz, _vp]),
    "owrx_wf_create": (_i, [_i, _i, _i, _i, _f, _i, _pp]),
    "owrx_wf_destroy": (None, [_vp]),
    "owrx_wf_set_every_n_samples": (_i, [_vp, _i]),
    "owrx_wf_set_avg_number": (_i, [_vp, _i]),
    "owrx_wf_set_compression": (_i, [_vp, _i]),
    "owrx_wf_set_noise_filter": (_i, [_vp, _i, _f, _f, _f]),
    "owrx_wf_line_bytes": (_sz, [_vp]),
    "owrx_wf_feed": (_i, [_vp, _vp, _sz]),
    "owrx_wf_feed_fmt": (_i, [_vp, _vp, _sz, _i, _f]),
    "owrx_wf_read_message": (_i, [_vp, _vp, _sz, _psz]),
    "owrx_chan_read_message": (_i, [_vp, _i, _i, _vp, _sz, _psz]),
    "owrx_wf_read": (_i, [_vp, _vp, _sz, _psz]),
    "owrx_wf_process_device": (_i, [_vp, _vp, _sz, _vp, _sz, _vp, _vp, _psz, _vp]),
    "owrx_wf_lines_for": (_sz, [_vp, _sz]),
    "owrx_wf_set_pipelined": (_i, [_vp, _i]),
    "owrx_wf_join": (_i, [_vp, _vp]),
    "owrx_fft_adpcm_encode_device": (_i, [_i, _vp, _i, _sz, _vp, _vp]),
    "owrx_bank_create": (_i, [_i, _d, _pp]),
    "owrx_bank_destroy": (None, [_vp]),
    "owrx_bank_add_channel": (_i, [_vp, _d, C.POINTER(_i)]),
    "owrx_bank_add_channel_ex": (_i, [_vp, C.POINTER(ChanSpec), C.POINTER(_i)]),
    "owrx_chan_set_agc": (_i, [_vp, _i, _i, _f, _f]),
    "owrx_bank_remove_channel": (_i, [_vp, _i]),
    "owrx_bank_channel_count": (_i, [_vp]),
    "owrx_chan_set_shift_rate": (_i, [_vp, _i, _d]),
    "owrx_chan_set_bandpass": (_i, [_vp, _i, _d, _d, _i]),
    "owrx_chan_set_squelch_level": (_i, [_vp, _i, _f]),
    "owrx_chan_set_demod": (_i, [_vp, _i, _i, _d, _d, _i]),
    "owrx_bank_feed": (_i, [_vp, _vp, _sz]),
    "owrx_bank_feed_fmt": (_i, [_vp, _vp, _sz, _i, _f]),
    "owrx_bank_set_deferred_drain": (_i, [_vp, _i]),
    "owrx_bank_flush": (_i, [_vp]),
    "owrx_chan_read_audio": (_i, [_vp, _i, _vp, _sz, _psz]),
    "owrx_chan_read_demod": (_i, [_vp, _i, _vp, _sz, _psz]),
    "owrx_chan_read_if": (_i, [_vp, _i, _vp, _sz, _psz]),
    "owrx_chan_read_power": (_i, [_vp, _i, _vp, _sz, _psz]),
    "owrx_bank_set_outputs": (_i, [_vp, _i]),
    "owrx_chan_set_audio_format": (_i, [_vp, _i, _i]),
    "owrx_chan_read_bytes": (_i, [_vp, _i, _vp, _sz, _psz]),
    "owrx_chan_set_audio_resampler": (_i, [_vp, _i, _i, _i]),
    "owrx_chan_set_mpx": (_i, [_vp, _i, _i]),
    "owrx_chan_read_mpx": (_i, [_vp, _i, _vp, _sz, _psz]),
    "owrx_chan_set_audio_tap": (_i, [_vp, _i, _i]),
    "owrx_chan_read_audio_tap": (_i, [_vp, _i, _vp, _sz, _psz]),
    "owrx_bank_process_device": (_i, [_vp, _vp, _sz, _vp]),
    "owrx_bank_set_pipelined": (_i, [_vp, _i]),
    "owrx_bank_join": (_i, [_vp, _vp]),
    "owrx_bank_drain": (_i, [_vp]),
    "owrx_bank_drain_begin": (_i, [_vp]),
    "owrx_bank_drain_end": (_i, [_vp]),
    "owrx_bank_last_consumed": (_i, [_vp, _psz]),
    "owrx_bank_last_audio_count": (_i, [_vp, _i, _psz]),
    "owrx_bank_last_audio_device": (_i, [_vp, _i, _pp, _psz, _psz]),
    "owrx_bank_get_stats": (_i, [_vp, C.POINTER(BankStats)]),
    "owrx_bank_profile": (_i, [_vp, _i]),
    "owrx_bank_profile_read": (_i, [_vp, C.POINTER(_d), C.POINTER(C.c_uint64), _i]),
    "owrx_bank_profile_read_ex": (_i, [_vp, C.POINTER(_d), C.POINTER(C.c_uint64), _i]),
    "owrx_bank_read_audio_all": (_i, [_vp, C.POINTER(_i), _i, _vp, _sz, _psz]),
    "owrx_bank_set_fir_mode": (_i, [_vp, _i]),
    "owrx_bank_fir_form": (_i, [_vp]),
}
PROF_KINDS = ("k3_direct", "fc_forward", "fc_contract", "fc_inverse", "tail", "agc", "resample", "tap")
FIR_MODES = {"auto": 0, "direct": 1, "fastconv": 2, "fastconv_tc": 3}

for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)          # AttributeError here = header/library mismatch: fail loudly
    _fn.restype = _res
    _fn.argtypes = _args


def last_error():
    return lib.owrx_last_error().decode("utf-8", "replace")


def check(rc):
    """Map the C ABI's error codes onto the exceptions the reference's callers expect
    (ValueError on bad formats/arguments: csdr/chain/__init__.py:69,80; BufferError: :145,151)."""
    if rc == OK:
        return
    msg = last_error()
    if rc == E_INVALID:
        raise ValueError(msg)
    if rc == E_NOMEM:
        raise MemoryError(msg)
    if rc == E_OVERFLOW:
        raise BufferError(msg)
    raise RuntimeError(msg)
