"""ChannelBank — all client channels of one wideband source, batched on the GPU.

Host-side mirror of what the reference builds per client: Selector (csdr/chain/selector.py:89-214)
followed by an analog demodulator chain (csdr/chain/analog.py:11-127); the reference attaches one such
chain per client to the same source ring (owrx/dsp.py:835-837), here they share one pass over HBM.
"""
import ctypes as C

import numpy as np

from . import _native as N
from .params import shift_rate

_KINDS = {"nfm": N.DEMOD_NFM, "am": N.DEMOD_AM, "usb": N.DEMOD_SSB, "lsb": N.DEMOD_SSB, "ssb": N.DEMOD_SSB,
          "wfm": N.DEMOD_WFM, "none": N.DEMOD_NONE}


def _ptr(obj):
    if obj is None:
        return None
    if hasattr(obj, "data_ptr"):
        return obj.data_ptr()
    return int(obj)


class Channel:
    """One client: Selector(inputRate, outputRate) + demodulator. Method names follow Selector's."""

    def __init__(self, bank, cid, output_rate):
        self.bank = bank
        self.id = cid
        self.outputRate = output_rate
        self.frequencyOffset = 0
        self.bandpassCutoffs = [None, None]
        self._mpx = "off"
        self._atap = "off"

    def setFrequencyOffset(self, offset):            # csdr/chain/selector.py:132-140
        self.frequencyOffset = offset
        N.check(N.lib.owrx_chan_set_shift_rate(self.bank._h, self.id, shift_rate(offset, self.bank.inputRate)))

    def setBandpass(self, low_cut, high_cut):        # csdr/chain/selector.py:159-166
        self.bandpassCutoffs = [low_cut, high_cut]
        if low_cut is None or high_cut is None:
            N.check(N.lib.owrx_chan_set_bandpass(self.bank._h, self.id, 0.0, 0.0, 0))
        else:
            N.check(N.lib.owrx_chan_set_bandpass(self.bank._h, self.id, low_cut / self.outputRate,
                                                 high_cut / self.outputRate, 1))

    def setSquelchLevel(self, level_db):             # csdr/chain/selector.py:142-147
        N.check(N.lib.owrx_chan_set_squelch_level(self.bank._h, self.id, float(10.0 ** (level_db / 10.0))))

    def setDemodulator(self, kind, audio_rate=48000.0, tau=50e-6, agc_profile="slow"):
        k = _KINDS[kind] if isinstance(kind, str) else int(kind)
        prof = N.AGC_FAST if str(agc_profile).lower() == "fast" else N.AGC_SLOW
        N.check(N.lib.owrx_chan_set_demod(self.bank._h, self.id, k, float(audio_rate), float(tau), prof))
        if k != N.DEMOD_WFM:
            self._mpx = "off"                        # the library turns the tap off with the WFm chain
        if k == N.DEMOD_NONE:
            self._atap = "off"                       # ... and the audio tap with the demodulator

    def _read(self, fn, width=1):
        chunks = []
        buf = np.empty(65536 * width, np.float32)
        while True:
            n = C.c_size_t()
            N.check(fn(self.bank._h, self.id, buf.ctypes.data_as(C.c_void_p), 65536, C.byref(n)))
            if n.value == 0:
                break
            chunks.append(buf[:n.value * width].copy())
        return np.concatenate(chunks) if chunks else np.empty(0, np.float32)

    def setAudioFormat(self, fmt):
        """'f32' | 's16' (Convert FLOAT->SHORT) | 'adpcm' (Convert + AdpcmEncoder(sync=True)); csdr/chain/clientaudio.py"""
        code = {"f32": N.AUDIO_F32, "s16": N.AUDIO_S16, "adpcm": N.AUDIO_ADPCM}[fmt]
        N.check(N.lib.owrx_chan_set_audio_format(self.bank._h, self.id, code))

    def set_audio_resampler(self, in_rate, out_rate=None):
        """AudioResampler(in_rate, out_rate) + Limit in front of the S16 / ADPCM bytes (csdr/chain/clientaudio.py:6-19; the
        resampler is spec-defined, see owrx_b200.h).  None removes it, as do equal rates.  ValueError for a rejected ratio or
        a channel without a demodulator."""
        if in_rate is None or out_rate is None:
            in_rate = out_rate = 0
        N.check(N.lib.owrx_chan_set_audio_resampler(self.bank._h, self.id, int(in_rate), int(out_rate)))

    def read_message(self, hd=False, cap=1 << 16):
        """queued client-audio bytes as one websocket message: b"\x02" + data (write_dsp_data) or b"\x04" + data
        (write_hd_audio), owrx/connection.py:477-481; None when nothing is queued"""
        buf = np.empty(cap, np.uint8)
        n = C.c_size_t()
        N.check(N.lib.owrx_chan_read_message(self.bank._h, self.id, 0x04 if hd else 0x02, buf.ctypes.data_as(C.c_void_p), buf.size, C.byref(n)))
        return buf[:n.value].tobytes() if n.value else None

    def read_bytes(self):
        chunks = []
        buf = np.empty(1 << 16, np.uint8)
        while True:
            n = C.c_size_t()
            N.check(N.lib.owrx_chan_read_bytes(self.bank._h, self.id, buf.ctypes.data_as(C.c_void_p), buf.size, C.byref(n)))
            if n.value == 0:
                break
            chunks.append(buf[:n.value].copy())
        return np.concatenate(chunks) if chunks else np.empty(0, np.uint8)

    def set_mpx(self, fmt):
        """WFM multiplex tap (the WFm chain's Limit output, csdr/chain/analog.py:62,73-76): "off" | "f32" | "s16" (after
        Convert(FLOAT, SHORT), what the reference's RDS path feeds redsea).  WFM channels only (ValueError otherwise)."""
        codes = {"off": N.MPX_OFF, "f32": N.MPX_F32, "s16": N.MPX_S16}
        if fmt not in codes:
            raise ValueError("unknown multiplex format %r (off | f32 | s16)" % (fmt,))
        code = codes[fmt]
        N.check(N.lib.owrx_chan_set_mpx(self.bank._h, self.id, code))
        self._mpx = fmt

    def read_mpx(self):
        """queued multiplex samples: np.float32 ("f32") or np.int16 ("s16")"""
        return self._read_tap(N.lib.owrx_chan_read_mpx, self._mpx)

    def set_audio_tap(self, fmt):
        """demodulated-audio tap (what a secondary demodulator reads beside the client-audio Converter), at the demodulator
        rate: "off" | "f32" | "s16" (after Convert(FLOAT, SHORT)).  ValueError for an unknown format or a channel without a
        demodulator."""
        codes = {"off": N.MPX_OFF, "f32": N.MPX_F32, "s16": N.MPX_S16}
        if fmt not in codes:
            raise ValueError("unknown audio tap format %r (off | f32 | s16)" % (fmt,))
        N.check(N.lib.owrx_chan_set_audio_tap(self.bank._h, self.id, codes[fmt]))
        self._atap = fmt

    def read_audio_tap(self):
        """queued audio-tap samples: np.float32 ("f32") or np.int16 ("s16")"""
        return self._read_tap(N.lib.owrx_chan_read_audio_tap, self._atap)

    def _read_tap(self, fn, fmt):
        dtype = np.int16 if fmt == "s16" else np.float32
        chunks = []
        buf = np.empty(1 << 18, np.uint8)
        while True:
            n = C.c_size_t()
            N.check(fn(self.bank._h, self.id, buf.ctypes.data_as(C.c_void_p), buf.size, C.byref(n)))
            if n.value == 0:
                break
            chunks.append(buf[:n.value].copy())
        return (np.concatenate(chunks) if chunks else np.empty(0, np.uint8)).view(dtype)

    def read_audio(self):
        return self._read(N.lib.owrx_chan_read_audio)

    def read_audio_into(self, buf):
        """pop queued float32 audio into a caller-owned numpy buffer; returns the sample count"""
        n = C.c_size_t()
        N.check(N.lib.owrx_chan_read_audio(self.bank._h, self.id, buf.ctypes.data_as(C.c_void_p), buf.size, C.byref(n)))
        return n.value

    def read_demod(self):
        return self._read(N.lib.owrx_chan_read_demod)

    def read_if(self):
        return self._read(N.lib.owrx_chan_read_if, 2).view(np.complex64)

    def read_power(self):
        return self._read(N.lib.owrx_chan_read_power)

    def last_audio_count(self):
        n = C.c_size_t()
        N.check(N.lib.owrx_bank_last_audio_count(self.bank._h, self.id, C.byref(n)))
        return n.value

    def last_audio_device(self):
        base, stride, slot = C.c_void_p(), C.c_size_t(), C.c_size_t()
        N.check(N.lib.owrx_bank_last_audio_device(self.bank._h, self.id, C.byref(base), C.byref(stride), C.byref(slot)))
        return base.value, stride.value, slot.value

    def remove(self):
        N.check(N.lib.owrx_bank_remove_channel(self.bank._h, self.id))


class ChannelBank:
    def __init__(self, input_rate, device=0, outputs=N.OUT_AUDIO):
        self.inputRate = input_rate
        h = C.c_void_p()
        N.check(N.lib.owrx_bank_create(device, float(input_rate), C.byref(h)))
        self._h = h
        self.channels = []
        if outputs != N.OUT_AUDIO:
            self.set_outputs(outputs)

    def set_outputs(self, mask):
        N.check(N.lib.owrx_bank_set_outputs(self._h, mask))

    def add_channel(self, output_rate, demod="nfm", offset=0, bandpass=None, **demod_kw):
        cid = C.c_int()
        N.check(N.lib.owrx_bank_add_channel(self._h, float(output_rate), C.byref(cid)))
        ch = Channel(self, cid.value, output_rate)
        ch.setDemodulator(demod, **demod_kw)
        if offset:
            ch.setFrequencyOffset(offset)
        if bandpass is not None:
            ch.setBandpass(*bandpass)
        self.channels.append(ch)
        return ch

    def feed(self, iq):
        """One wideband block from HOST memory (complex64 numpy array, ideally pinned)."""
        iq = np.ascontiguousarray(iq, dtype=np.complex64)
        N.check(N.lib.owrx_bank_feed(self._h, iq.ctypes.data_as(C.c_void_p), iq.size))

    def feed_ptr(self, host_ptr, n_samples, fmt="cf32", gain=1.0):
        if fmt == "cf32" and gain == 1.0:
            N.check(N.lib.owrx_bank_feed(self._h, host_ptr, n_samples))
        else:
            N.check(N.lib.owrx_bank_feed_fmt(self._h, host_ptr, n_samples, N.IQ_FORMATS[fmt], float(gain)))

    def feed_raw(self, raw, fmt, gain=1.0):
        """One wideband block of RAW source samples from host memory: fmt "cs16" (int16 array, interleaved I, Q) or "cu8"
        (uint8, offset binary).  The reference's CPU-side Convert (+ Gain) (owrx/source/fifi_sdr.py:27-28) runs on the GPU."""
        raw = np.ascontiguousarray(raw, dtype=np.int16 if fmt == "cs16" else np.uint8)
        assert raw.size % 2 == 0
        N.check(N.lib.owrx_bank_feed_fmt(self._h, raw.ctypes.data_as(C.c_void_p), raw.size // 2, N.IQ_FORMATS[fmt], float(gain)))

    def set_deferred_drain(self, enable=True):
        """streaming mode: feed() only enqueues (uploads + kernels) and returns; the block's outputs reach the queues at the start
        of the next feed (behind its uploads) or at flush().  The fed host buffer must stay valid until then."""
        N.check(N.lib.owrx_bank_set_deferred_drain(self._h, 1 if enable else 0))

    def flush(self):
        N.check(N.lib.owrx_bank_flush(self._h))

    def process_device(self, iq_dev, n_samples, stream=None):
        N.check(N.lib.owrx_bank_process_device(self._h, _ptr(iq_dev), n_samples, _ptr(stream)))

    def last_consumed(self):
        """samples of the last process_device block every channel is done with: the next block of a continuous stream starts
        there ([carry | new], include/owrx_b200.h)"""
        n = C.c_size_t()
        N.check(N.lib.owrx_bank_last_consumed(self._h, C.byref(n)))
        return n.value

    def stats(self):
        st = N.BankStats()
        N.check(N.lib.owrx_bank_get_stats(self._h, C.byref(st)))
        return dict(input_samples=st.input_samples, channel_samples=st.channel_samples,
                    kernel_launches=st.kernel_launches, device_ms=st.device_ms,
                    h2d_pinned_bytes=st.h2d_pinned_bytes, h2d_pageable_bytes=st.h2d_pageable_bytes)

    def set_pipelined(self, enable=True):
        N.check(N.lib.owrx_bank_set_pipelined(self._h, 1 if enable else 0))

    def join(self, stream=None):
        N.check(N.lib.owrx_bank_join(self._h, _ptr(stream)))

    def drain(self):
        """D2H of the last process_device block into the host queues (then read_audio etc. pop it)"""
        N.check(N.lib.owrx_bank_drain(self._h))

    def drain_begin(self):
        """split-phase drain: enqueue the D2H of the last process_device block; the next block may be issued before drain_end"""
        N.check(N.lib.owrx_bank_drain_begin(self._h))

    def drain_end(self):
        """wait for drain_begin's copies and fill the host queues (no-op without a pending drain_begin)"""
        N.check(N.lib.owrx_bank_drain_end(self._h))

    def profile(self, enable=True):
        N.check(N.lib.owrx_bank_profile(self._h, 1 if enable else 0))

    def profile_read(self, reset=True):
        ms, n = C.c_double(), C.c_uint64()
        N.check(N.lib.owrx_bank_profile_read(self._h, C.byref(ms), C.byref(n), 1 if reset else 0))
        return ms.value, n.value

    def profile_read_ex(self, reset=True):
        """{kind: (ms, launches)} per kernel kind (direct K3 / fast-convolution forward, contract, inverse)"""
        k = len(N.PROF_KINDS)
        ms, n = (C.c_double * k)(), (C.c_uint64 * k)()
        N.check(N.lib.owrx_bank_profile_read_ex(self._h, ms, n, 1 if reset else 0))
        return {name: (ms[i], n[i]) for i, name in enumerate(N.PROF_KINDS)}

    def read_audio_all(self, channels, buf):
        """pop the queued float32 audio of every channel in `channels` with ONE library call: channel i -> buf[i, :counts[i]]
        (buf: C-contiguous float32 [len(channels), cap]); returns the per-channel sample counts"""
        ids = (C.c_int * len(channels))(*[c.id for c in channels])
        counts = (C.c_size_t * len(channels))()
        assert buf.dtype == np.float32 and buf.flags.c_contiguous and buf.shape[0] >= len(channels)
        N.check(N.lib.owrx_bank_read_audio_all(self._h, ids, len(channels), buf.ctypes.data_as(C.c_void_p), buf.shape[1], counts))
        return list(counts)

    def set_fir_mode(self, mode="auto"):
        """how Shift + FirDecimate is evaluated: "auto" | "direct" (K3) | "fastconv" (K3F, FP32 pipe) | "fastconv_tc" (K3F, tcgen05)"""
        N.check(N.lib.owrx_bank_set_fir_mode(self._h, N.FIR_MODES[mode] if isinstance(mode, str) else int(mode)))

    def fir_form(self):
        """the form the latest Shift + FirDecimate pass used: "direct" | "fastconv" | "fastconv_tc" (None before any pass)"""
        v = N.lib.owrx_bank_fir_form(self._h)
        return {1: "direct", 2: "fastconv", 3: "fastconv_tc"}.get(v)

    def close(self):
        if getattr(self, "_h", None):
            N.lib.owrx_bank_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
