"""pycsdr.modules — drop-in for the CPython extension the reference imports (SURVEY Appendix C),
backed by libowrx_b200.so through openwebrx_b200._native (ctypes).  No CPU fallback: the arithmetic of
every hot-path module runs in the CUDA library or not at all.

How it maps onto the GPU.  The reference builds one pycsdr module object per DSP stage and joins
them with Buffers (csdr/chain/__init__.py:21-25); here those objects are *descriptors*.  A runner
thread per source Buffer discovers, lazily (when data flows and the wiring has changed), the chains
hanging off that Buffer and compiles each into a fused plan:

    Fft -> LogPower|LogAveragePower -> FftSwap -> [FftAdpcm]                 -> one owrx_wf_t
    Shift -> FirDecimate -> [FractionalDecimator] -> [Bandpass] -> [Squelch]
          -> [FmDemod Limit NfmDeemphasis Agc | AmDemod DcBlock Agc | RealPart Agc
              | FmDemod Limit FractionalDecimator(FLOAT) WfmDeemphasis]       -> one channel of the
                                                                                 source's owrx_bank_t
All channels reading the same source Buffer share one owrx_bank_feed per block (one H2D copy, one
pass over HBM).  Buffers between fused stages stay virtual; the Buffer after the last fused module
receives the result bytes, and the selector output is materialised only when something else reads it
(e.g. the secondary FFT on ClientDemodulatorChain.selectorBuffer, owrx/dsp.py:49,220-225).
"""
import ctypes as C
import itertools
import logging
import math
import os
import threading
import weakref
from collections import deque

import numpy as np

from .types import AgcProfile, Format

logger = logging.getLogger(__name__)

# owrx/feature.py:213-222 requires csdr_version / version >= 0.18.0
version = "0.18.36"
csdr_version = "0.18.36"

# ring capacity of a Buffer: a reader that falls further behind than this loses the oldest data (a few seconds of the
# fastest source: 61.44 MS/s complex float32 = 491 MB/s)
_BUFFER_CAP_BYTES = 1 << 28


def _native():
    from openwebrx_b200 import _native as N      # raises ImportError if the CUDA library is not built
    return N


# ================================================================================================
# page-locked ingress ring (SURVEY 8f-4 / a19: owrx/source/__init__.py:307-330)
# ================================================================================================
class _PinnedRing:
    """cudaHostAlloc'd arena behind a SOURCE Buffer (one that a GPU runner reads): TcpSource recv()s straight into it and the
    runner hands the copy engine pointers into it, so no pageable bounce copy sits between the socket and HBM.  Chunks are
    never split across the wrap (the allocator skips to offset 0 when the end is too short)."""

    def __init__(self, nbytes):
        N = _native()
        p = C.c_void_p()
        N.check(N.lib.owrx_pinned_alloc(nbytes, C.byref(p)))
        self._free = N.lib.owrx_pinned_free
        self.ptr, self.size, self.head = p.value, int(nbytes), 0
        self.view = memoryview((C.c_ubyte * nbytes).from_address(self.ptr)).cast("B")

    def close(self):
        if self.ptr:
            self.view = None
            self._free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_RING_WAIT_S = 5.0      # how long a writer holds back for a runner that has not consumed the oldest ring chunk


def _ring_bytes():
    return max(1, int(os.environ.get("OWRX_RING_MB", "64"))) << 20


# ================================================================================================
# wiring graph
# ================================================================================================
class _Graph:
    def __init__(self):
        self.lock = threading.RLock()
        self.epoch = 0
        self.modules = weakref.WeakSet()

    def touch(self):
        with self.lock:
            self.epoch += 1

    def consumer_of(self, buffer):
        """the live stage whose reader sits on `buffer` (first one), plus the number of other readers"""
        for m in list(self.modules):
            r = m._reader
            if r is not None and r._buffer is buffer and not m._stopped and not r._stopped:
                return m
        return None


_GRAPH = _Graph()
_STAGE_SEQ = itertools.count()


# ================================================================================================
# Reader / Writer / Buffer  (SURVEY 2.3 first row; owrx/fft.py:70-72, csdr/module/__init__.py:36-53)
# ================================================================================================
class Writer:
    def write(self, data):
        raise NotImplementedError


class Reader:
    """Independent cursor on a Buffer.  read() blocks (GIL released in Condition.wait) and returns all
    currently available bytes as a memoryview; None once stopped."""

    def __init__(self, buffer):
        self._buffer = buffer
        self._pos = buffer._end
        self._stopped = False
        # True while the reader is only a wiring token of a fused (descriptor) stage: the source runner reads the Buffer
        # through its own cursor, nobody ever calls read() on this one, so it must not pin chunks in Buffer._trim
        self._virtual = False

    def getFormat(self):
        return self._buffer._format

    def read(self):
        """next write unit.  Frame granularity is preserved: every Writer.write() surfaces as exactly one
        read() result, because the reference forwards one read() as one WebSocket message and the browser
        decodes each FFT message as exactly one line (owrx/fft.py:70-73, htdocs/openwebrx.js:1124-1131)."""
        return self._read(False)

    def _read(self, everything):
        b = self._buffer
        with b._cond:
            if self._virtual:                 # somebody reads this cursor after all: it counts again, from "now"
                self._virtual = False
                self._pos = max(self._pos, b._end)
            while not self._stopped and self._pos >= b._end:
                b._cond.wait()
            if self._stopped:
                return None
            if self._pos < b._start:          # overrun: a slow reader loses the oldest data (ring semantics)
                self._pos = b._start
            first = self._pos - b._start
            if everything:
                chunks = [b._chunks[i] for i in range(first, len(b._chunks))]
                self._pos = b._end
            else:
                chunks = [b._chunks[first]]
                self._pos += 1
            # a Python reader gets its own copy of ring-backed chunks (the ring region is overwritten later)
            chunks = [c if isinstance(c, bytes) else bytes(b._ring.view[c[0]:c[0] + c[1]]) for c in chunks]
            b._trim()
        if len(chunks) == 1:
            return memoryview(chunks[0])
        return memoryview(b"".join(chunks))

    def _read_views(self):
        """the GPU runner's read: everything that has arrived, as a list of buffers to feed in order — views INTO the page-locked
        ring where the Buffer has one (adjacent chunks merged; zero copy), bytes otherwise.  Ring regions stay reserved
        (the writer will not overwrite them) until _release()."""
        b = self._buffer
        with b._cond:
            while not self._stopped and self._pos >= b._end:
                b._cond.wait()
            if self._stopped:
                return None
            if self._pos < b._start:
                self._pos = b._start
            first = self._pos - b._start
            chunks = [b._chunks[i] for i in range(first, len(b._chunks))]
            self._pos = b._end
            out, runs = [], []
            for c in chunks:
                if isinstance(c, bytes):
                    out.append(memoryview(c))
                elif runs and out and runs[-1] is not None and runs[-1][0] + runs[-1][1] == c[0]:
                    runs[-1][1] += c[1]
                    out[-1] = b._ring.view[runs[-1][0]:runs[-1][0] + runs[-1][1]]
                    continue
                else:
                    out.append(b._ring.view[c[0]:c[0] + c[1]])
                runs.append(None if isinstance(c, bytes) else [c[0], c[1]])
            b._inflight = [tuple(r) for r in runs if r is not None]
            b._trim()
            b._cond.notify_all()
        return out

    def _release(self):
        b = self._buffer
        with b._cond:
            if b._inflight:
                b._inflight = []
                b._cond.notify_all()

    def stop(self):
        with self._buffer._cond:
            self._stopped = True
            self._buffer._cond.notify_all()
        _GRAPH.touch()

    def resume(self):
        with self._buffer._cond:
            self._stopped = False
            self._pos = self._buffer._end
        _GRAPH.touch()


class Buffer(Writer):
    """Single-writer multi-reader byte queue carrying items of one Format."""

    def __init__(self, format=Format.CHAR, *args):
        if not isinstance(format, Format):
            raise ValueError("Buffer needs a pycsdr.types.Format")
        self._format = format
        self._cond = threading.Condition()
        self._chunks = deque()      # bytes objects; chunk i has sequence number _start + i
        self._start = 0
        self._end = 0
        self._bytes = 0
        self._readers = weakref.WeakSet()
        self._runner = None
        # set by the source-side Convert (+ Gain) pump: this COMPLEX_FLOAT buffer physically carries the source's raw
        # samples ("cs16" / "cu8") and the gain to apply; the GPU does the conversion (owrx_*_feed_fmt)
        self._raw = None
        # page-locked storage, enabled when a GPU runner attaches (None: not tried, False: no CUDA device here)
        self._ring = None
        self._inflight = []         # ring regions (offset, length) the runner is feeding from: not to be overwritten

    def getFormat(self):
        return self._format

    def _write_raw(self, data, fmt, gain):
        self._raw = (fmt, float(gain))
        self.write(data)

    def getReader(self):
        r = Reader(self)
        with self._cond:
            self._readers.add(r)
        _GRAPH.touch()            # a new cursor on a Buffer between fused stages makes that Buffer's content needed
        return r

    def write(self, data):
        if self._ring:
            mv = memoryview(data).cast("B")
            step = self._ring.size // 4
            for o in range(0, len(mv), step):
                part = mv[o:o + step]
                off = self._reserve(len(part))
                self._ring.view[off:off + len(part)] = part
                self._commit(off, len(part))
            return
        data = bytes(data)
        if not data:
            return
        with self._cond:
            self._chunks.append(data)
            self._end += 1
            self._bytes += len(data)
            self._trim()
            self._cond.notify_all()

    # ---- page-locked ring (single writer) --------------------------------------------------------
    def _enable_ring(self):
        """called when a GPU runner attaches to this Buffer; without a CUDA device the Buffer stays a plain byte queue"""
        with self._cond:
            if self._ring is None:
                try:
                    self._ring = _PinnedRing(_ring_bytes())
                except Exception as e:        # no device (build container) / out of lockable memory
                    logger.debug("pycsdr-b200: no page-locked ring for this Buffer: %s", e)
                    self._ring = False
        return bool(self._ring)

    def _reserve(self, nbytes):
        """offset of a contiguous writable region of nbytes (<= size / 2) in the ring.  Unread chunks in the way are dropped
        (a slow reader loses the oldest data, as with the reference's ring); regions the runner is feeding from are waited
        for (back-pressure on the socket)."""
        r = self._ring
        if nbytes > r.size // 2:
            raise ValueError("chunk larger than half the ring")
        with self._cond:
            if r.head + nbytes > r.size:
                r.head = 0
            lo, hi = r.head, r.head + nbytes
            while any(a < hi and lo < a + n for a, n in self._inflight):
                self._cond.wait(0.5)
            waited = 0.0
            while self._chunks:
                c = self._chunks[0]
                if isinstance(c, bytes) or not (c[0] < hi and lo < c[0] + c[1]):
                    break
                # the oldest chunk is in the way.  If the GPU runner has not taken it yet, hold the socket back for a moment
                # (TCP back-pressure is gentler than a gap in the stream: the first block also pays CUDA start-up); a consumer
                # that stays away loses the data, as with the reference's ring.
                r = self._runner
                if r is not None and r.is_alive() and not r.reader._stopped and r.reader._pos <= self._start and waited < _RING_WAIT_S:
                    self._cond.wait(0.05)
                    waited += 0.05
                    continue
                self._chunks.popleft()
                self._bytes -= c[1]
                self._start += 1
            return lo

    def _commit(self, off, nbytes):
        if not nbytes:
            return
        with self._cond:
            self._ring.head = off + nbytes
            self._chunks.append((off, nbytes))
            self._end += 1
            self._bytes += nbytes
            self._trim()
            self._cond.notify_all()

    def _trim(self):
        live = [r._pos for r in self._readers if not r._stopped and not r._virtual]
        low = min(live) if live else self._end
        while self._chunks and (self._start < low or self._bytes > _BUFFER_CAP_BYTES):
            c = self._chunks.popleft()
            self._bytes -= len(c) if isinstance(c, bytes) else c[1]
            self._start += 1

    def _extra_readers(self, used):
        with self._cond:
            # virtual readers are wiring tokens of fused stages: only cursors somebody really reads count (a Python pump, or the
            # own reader of a runner that serves heads attached to this Buffer)
            return [r for r in self._readers if r is not used and not r._stopped and not r._virtual]


# ================================================================================================
# module descriptors
# ================================================================================================
class Module:
    """Base of every pycsdr module.  The reference subclasses it with ABCMeta and a no-arg __init__
    (csdr/module/__init__.py:16-20) and relies on the inherited no-op stop() (owrx/dsp.py:143)."""

    def __init__(self, *args, **kwargs):
        pass

    def setReader(self, reader):
        pass

    def setWriter(self, writer):
        pass

    def stop(self):
        pass

    def getInputFormat(self):
        raise NotImplementedError

    def getOutputFormat(self):
        raise NotImplementedError


class _Stage(Module):
    IN = Format.COMPLEX_FLOAT
    OUT = Format.COMPLEX_FLOAT
    HEAD = False

    def __init__(self):
        self._reader = None
        self._writer = None
        self._stopped = False
        self._lock = threading.Lock()
        self._seq = next(_STAGE_SEQ)          # construction order: the walk's tie-break
        _GRAPH.modules.add(self)

    def getInputFormat(self):
        return self.IN

    def getOutputFormat(self):
        return self.OUT

    def setReader(self, reader):
        if reader is not None and isinstance(reader, Reader) and reader.getFormat() is not self.getInputFormat():
            raise ValueError("invalid reader format: %s, expected %s" % (reader.getFormat().name, self.getInputFormat().name))
        self._reader = reader
        self._stopped = False
        if isinstance(reader, Reader):
            reader._virtual = self._consumes_through_runner()
        _GRAPH.touch()
        if self.HEAD and reader is not None:
            _SourceRunner.attach(reader._buffer)

    def _consumes_through_runner(self):
        """descriptor stages never call reader.read(): their data arrives through the source Buffer's runner"""
        return True

    def setWriter(self, writer):
        if isinstance(writer, Buffer) and writer.getFormat() is not self.getOutputFormat():
            raise ValueError("invalid writer format: %s, expected %s" % (writer.getFormat().name, self.getOutputFormat().name))
        self._writer = writer
        _GRAPH.touch()
        # a tail that got its writer completes a chain whose head may already be attached
        head_buf = _find_source(self)
        if head_buf is not None:
            _SourceRunner.attach(head_buf)

    def stop(self):
        self._stopped = True
        _GRAPH.touch()

    def _changed(self):
        self._dirty = True
        _GRAPH.touch()


def _find_source(stage, limit=64):
    """walk upstream through virtual Buffers to the Buffer feeding the chain's head"""
    seen = 0
    while stage is not None and seen < limit:
        r = stage._reader
        if r is None:
            return None
        buf = r._buffer
        up = None
        for m in list(_GRAPH.modules):
            if m._writer is buf and not m._stopped:
                up = m
                break
        if up is None:
            return buf if stage.HEAD else None
        stage = up
        seen += 1
    return None


# ---- waterfall stages (csdr/chain/fft.py:18-22,34-45) -------------------------------------------------
class Fft(_Stage):
    HEAD = True

    def __init__(self, size, every_n_samples=0):
        super().__init__()
        self.size = int(size)
        self.every_n_samples = int(every_n_samples)

    def setEveryNSamples(self, n):
        self.every_n_samples = int(n)
        self._changed()


class LogPower(_Stage):
    OUT = Format.FLOAT

    def __init__(self, add_db=0.0):
        super().__init__()
        self.add_db = float(add_db)
        self.avg_number = 0


class LogAveragePower(_Stage):
    OUT = Format.FLOAT

    def __init__(self, add_db=0.0, fft_size=0, avg_number=1):
        super().__init__()
        self.add_db = float(add_db)
        self.fft_size = int(fft_size)
        self.avg_number = int(avg_number)

    def setAvgNumber(self, n):
        self.avg_number = int(n)
        self._changed()


class FftSwap(_Stage):
    IN = Format.FLOAT
    OUT = Format.FLOAT

    def __init__(self, fft_size):
        super().__init__()
        self.fft_size = int(fft_size)


class FftAdpcm(_Stage):
    IN = Format.FLOAT
    OUT = Format.CHAR

    def __init__(self, fft_size):
        super().__init__()
        self.fft_size = int(fft_size)


# ---- selector stages (csdr/chain/selector.py) ---------------------------------------------------------
class Shift(_Stage):
    HEAD = True

    def __init__(self, rate=0.0):
        super().__init__()
        self.rate = float(rate)

    def setRate(self, rate):
        self.rate = float(rate)
        self._changed()


class FirDecimate(_Stage):
    def __init__(self, decimation, transition=0.05, cutoff=0.5):
        super().__init__()
        self.decimation = int(decimation)
        self.transition = float(transition)
        self.cutoff = float(cutoff)


class FractionalDecimator(_Stage):
    def __init__(self, format, rate, prefilter=False):
        super().__init__()
        if format not in (Format.FLOAT, Format.COMPLEX_FLOAT):
            raise ValueError("unsupported FractionalDecimator format")
        self.format = format
        self.rate = float(rate)
        self.prefilter = bool(prefilter)

    def getInputFormat(self):
        return self.format

    def getOutputFormat(self):
        return self.format


class Bandpass(_Stage):
    def __init__(self, *args, **kwargs):
        super().__init__()
        # Bandpass(transition=, use_fft=True) (selector.py:117) or Bandpass(lo, hi, transition, use_fft=True) (:224)
        self.low = self.high = None
        if len(args) >= 3:
            self.low, self.high, self.transition = float(args[0]), float(args[1]), float(args[2])
        else:
            self.transition = float(kwargs.get("transition", args[0] if args else 0.05))
            if "low_cut" in kwargs:
                self.low, self.high = float(kwargs["low_cut"]), float(kwargs["high_cut"])
        self.use_fft = bool(kwargs.get("use_fft", True))

    def setBandpass(self, low, high):
        self.low, self.high = float(low), float(high)
        self._changed()


class Squelch(_Stage):
    def __init__(self, format=Format.COMPLEX_FLOAT, length=1024, decimation=5, hangLength=0, flushLength=0, reportInterval=1):
        super().__init__()
        self.format = format
        self.length = int(length)
        self.decimation = int(decimation)
        self.hangLength = int(hangLength)
        self.flushLength = int(flushLength)
        self.reportInterval = int(reportInterval)
        self.level = 0.0            # default: open (owrx/dsp.py:281-285 only sets it when it differs)
        self.powerWriter = None

    def getInputFormat(self):
        return self.format

    def getOutputFormat(self):
        return self.format

    def setSquelchLevel(self, level):
        self.level = float(level)
        self._changed()

    def setPowerWriter(self, writer):
        self.powerWriter = writer
        self._changed()


# ---- demodulator stages (csdr/chain/analog.py) --------------------------------------------------------
class AmDemod(_Stage):
    OUT = Format.FLOAT


class FmDemod(_Stage):
    OUT = Format.FLOAT


class RealPart(_Stage):
    OUT = Format.FLOAT


class DcBlock(_Stage):
    IN = Format.FLOAT
    OUT = Format.FLOAT


class Limit(_Stage):
    IN = Format.FLOAT
    OUT = Format.FLOAT

    def __init__(self, maxAmplitude=1.0):
        super().__init__()
        self.maxAmplitude = float(maxAmplitude)


class NfmDeemphasis(_Stage):
    IN = Format.FLOAT
    OUT = Format.FLOAT

    def __init__(self, sampleRate):
        super().__init__()
        self.sampleRate = int(sampleRate)


class WfmDeemphasis(_Stage):
    IN = Format.FLOAT
    OUT = Format.FLOAT

    def __init__(self, sampleRate, tau):
        super().__init__()
        self.sampleRate = int(sampleRate)
        self.tau = float(tau)


class AudioResampler(_Stage):
    """AudioResampler(inputRate, outputRate): the client-audio Converter's rate change (csdr/chain/clientaudio.py:16), fused
    with the Limit and Convert behind it into the channel's audio tail (owrx_chan_set_audio_resampler).  Spec-defined: the
    reference's libsamplerate is not reproduced (DESIGN.md)."""
    IN = Format.FLOAT
    OUT = Format.FLOAT

    def __init__(self, inputRate, outputRate):
        super().__init__()
        self.inputRate = int(inputRate)
        self.outputRate = int(outputRate)


def _resampler_ok(in_rate, out_rate):
    """the library's limit on AudioResampler(in, out): positive rates and at most 65536 prototype taps (owrx_b200.h)"""
    if in_rate <= 0 or out_rate <= 0:
        return False
    g = math.gcd(in_rate, out_rate)
    L = out_rate // g
    df = 0.1 * min(in_rate, out_rate) / (L * in_rate)
    K = math.ceil(((96.0 - 7.95) / (14.36 * df) + 1.0) / L)
    return L * K <= 65536


class Agc(_Stage):
    def __init__(self, format=Format.FLOAT):
        super().__init__()
        self.format = format
        self.profile = AgcProfile.SLOW
        self.initialGain = 0.0
        self.maxGain = 0.0

    def getInputFormat(self):
        return self.format

    def getOutputFormat(self):
        return self.format

    def setProfile(self, profile):
        self.profile = profile
        self._changed()

    def setInitialGain(self, gain):
        self.initialGain = float(gain)
        self._changed()

    def setMaxGain(self, gain):
        self.maxGain = float(gain)
        self._changed()

    def setReference(self, r):
        self._changed()


# ---- modules the reference imports or constructs around the hot path; constructible, not fused ---------
class _Unfused(_Stage):
    """Constructible so that the reference's chains import and wire (SURVEY 8b item 4), but outside the
    accelerated path: data reaching one of these is an error, not a silent CPU fallback."""

    def __init__(self, *args, **kwargs):
        super().__init__()
        self.args, self.kwargs = args, kwargs

    def __getattr__(self, name):
        if name.startswith("set"):
            return lambda *a, **k: None
        raise AttributeError(name)


class Convert(_Unfused):
    """Convert(inFormat, outFormat).  Two uses in the reference: the client-audio Convert(FLOAT, SHORT)
    (csdr/chain/clientaudio.py:12, fused into the audio tail) and the SOURCE-side conversion
    Chain([Convert(COMPLEX_SHORT, COMPLEX_FLOAT), Gain(COMPLEX_FLOAT, 5.0)]) of sources that do not deliver floats
    (owrx/source/fifi_sdr.py:27-28, wired by owrx/source/direct.py:59-71).  The latter never converts on the host: a pump
    thread hands the raw samples on, tagged with their format and the accumulated gain, and the runner of the
    COMPLEX_FLOAT buffer feeds them through owrx_wf_feed_fmt / owrx_bank_feed_fmt (SURVEY 8f-4)."""

    _RAW = {Format.COMPLEX_SHORT: "cs16", Format.COMPLEX_CHAR: "cu8"}

    def __init__(self, inFormat, outFormat):
        super().__init__(inFormat, outFormat)
        self.IN, self.OUT = inFormat, outFormat
        self._pump = None

    def _ingress(self):
        return self.OUT is Format.COMPLEX_FLOAT and self.IN in self._RAW

    def _consumes_through_runner(self):
        return not self._ingress()            # the source-side pump below really reads its reader

    def setReader(self, reader):
        super().setReader(reader)
        if self._ingress() and reader is not None and (self._pump is None or not self._pump.is_alive()):
            self._pump = threading.Thread(target=self._run, args=(reader,), daemon=True, name="pycsdr-b200-ingress")
            self._pump.start()

    def _sink(self):
        """the COMPLEX_FLOAT buffer at the end of Convert [-> Gain ...] and the product of the gains on the way"""
        gain, buf = 1.0, self._writer
        for _ in range(8):
            if not isinstance(buf, Buffer):
                return None, gain
            nxt = _GRAPH.consumer_of(buf)
            if isinstance(nxt, Gain) and nxt.IN is Format.COMPLEX_FLOAT and nxt._writer is not None:
                gain *= nxt.gain
                buf = nxt._writer
                continue
            return buf, gain
        return None, gain

    def _run(self, reader):
        while not self._stopped and self._reader is reader:
            data = reader.read()
            if data is None:
                break
            sink, gain = self._sink()
            if sink is not None:
                sink._write_raw(data, self._RAW[self.IN], gain)


class Gain(_Unfused):
    def __init__(self, format, gain):
        super().__init__(format, gain)
        self.IN = self.OUT = format
        self.gain = float(gain)


class AdpcmEncoder(_Unfused):
    IN = Format.SHORT
    OUT = Format.CHAR

    def __init__(self, sync=False):
        super().__init__(sync=sync)
        self.sync = bool(sync)


class NoiseFilter(_Unfused):
    IN = Format.FLOAT
    OUT = Format.FLOAT


class Afc(_Unfused):
    pass


class TcpSource(Module):
    """TcpSource(port, Format) — owrx/source/__init__.py:310-314: reads the connector's TCP stream into
    its writer.  When the writer is a source Buffer with a page-locked ring (a GPU runner reads it) the socket is
    received straight into the ring: TcpSource -> pinned host ring -> H2D (SURVEY 8f-4)."""

    def __init__(self, port, format):
        import socket
        self._format = format
        self._writer = None
        self._stop = False
        self._sock = socket.create_connection(("127.0.0.1", int(port)))
        self._thread = None

    def getOutputFormat(self):
        return self._format

    def setWriter(self, writer):
        self._writer = writer
        if self._thread is None:
            self._thread = threading.Thread(target=self._run, daemon=True, name="pycsdr-tcpsource")
            self._thread.start()

    def _run(self):
        item = self._format.size
        pending = b""
        while not self._stop:
            w = self._writer
            ring = getattr(w, "_ring", None)
            if ring:
                # the writer is a source Buffer with a page-locked ring: the kernel copies the TCP payload straight into it
                want = min(1 << 20, ring.size // 4)
                off = w._reserve(want)
                k = len(pending)
                ring.view[off:off + k] = pending
                try:
                    got = self._sock.recv_into(ring.view[off + k:off + want])
                except OSError:
                    break
                if not got:
                    break
                n = (k + got) - (k + got) % item
                pending = bytes(ring.view[off + n:off + k + got])       # at most item - 1 bytes of a split sample
                w._commit(off, n)
                self.bytes_direct = getattr(self, "bytes_direct", 0) + n
                continue
            try:
                data = self._sock.recv(1 << 20)
            except OSError:
                break
            if not data:
                break
            pending += data
            n = len(pending) - len(pending) % item
            if n and w is not None:
                w.write(pending[:n])
                pending = pending[n:]

    def stop(self):
        self._stop = True
        try:
            self._sock.close()
        except OSError:
            pass


class ExecModule(Module):
    """ExecModule(inFormat, outFormat, args, ...): pycsdr's base of the modules that run an external decoder process.  In
    OpenWebRX+ the RDS decoder module (RedseaModule, fed by WFm.setMetaWriter through Convert(FLOAT, SHORT)) is described as
    one of them; that base class and wiring have not been checked against OpenWebRX source in this project, so no lines are
    cited.  The WFM tap works whether its consumer is an ExecModule or a Python module reading the Buffer.  This is a host
    process, not DSP: one thread copies the reader into the child's stdin, one copies its stdout into the writer.  stop()
    closes stdin, terminates the child and waits for it, so no process outlives the module."""

    _STOP_WAIT_S = 5.0

    def __init__(self, inFormat, outFormat, args, *rest, **kw):
        import subprocess
        self.IN, self.OUT = inFormat, outFormat
        self._reader = None
        self._writer = None
        self._stopped = False
        self._cond = threading.Condition()
        self._proc = subprocess.Popen([str(a) for a in args], stdin=subprocess.PIPE, stdout=subprocess.PIPE)
        self._threads = [threading.Thread(target=f, daemon=True, name="pycsdr-exec") for f in (self._pump_in, self._pump_out)]
        for t in self._threads:
            t.start()

    def getInputFormat(self):
        return self.IN

    def getOutputFormat(self):
        return self.OUT

    def setReader(self, reader):
        with self._cond:
            old, self._reader = self._reader, reader
            self._cond.notify_all()
        if old is not None and old is not reader:
            old.stop()                             # the module's previous cursor: wakes a stdin pump blocked on it

    def setWriter(self, writer):
        self._writer = writer

    def _pump_in(self):
        while True:
            with self._cond:
                while self._reader is None and not self._stopped:
                    self._cond.wait()
                if self._stopped:
                    break
                reader = self._reader
            data = reader.read()
            if data is None:
                if self._stopped or reader is self._reader:
                    break
                continue                           # setReader() swapped the cursor
            try:
                self._proc.stdin.write(data)
                self._proc.stdin.flush()
            except (OSError, ValueError):          # the child went away / stop() closed stdin
                break

    def _pump_out(self):
        out = self._proc.stdout
        while True:
            data = out.read1(1 << 16)
            if not data:
                break
            w = self._writer
            if w is not None:
                w.write(data)

    def stop(self):
        import subprocess
        with self._cond:
            if self._stopped:
                return
            self._stopped = True
            reader = self._reader
            self._cond.notify_all()
        if reader is not None:
            reader.stop()                          # wakes the stdin pump
        try:
            self._proc.stdin.close()
        except OSError:
            pass
        self._proc.terminate()
        try:
            self._proc.wait(self._STOP_WAIT_S)
        except subprocess.TimeoutExpired:
            self._proc.kill()
            self._proc.wait()
        for t in self._threads:
            t.join(self._STOP_WAIT_S)
        self._proc.stdout.close()


def _unavailable(name):
    def ctor(*a, **k):
        raise NotImplementedError("pycsdr.modules.%s is outside the B200 hot path (SURVEY Appendix C)" % name)
    return type(name, (Module,), {"__init__": lambda self, *a, **k: ctor()})


for _n in ("Lowpass", "Downmix", "Throttle", "SnrSquelch", "SmartSquelch", "TimingRecovery", "DBPskDecoder",
           "VaricodeDecoder", "RttyDecoder", "BaudotDecoder", "MFRttyDecoder", "CwDecoder", "SstvDecoder", "FaxDecoder",
           "SitorBDecoder", "Ccir476Decoder", "DscDecoder", "Ccir493Decoder", "NavtexDecoder"):
    globals()[_n] = _unavailable(_n)


# ================================================================================================
# chain discovery and fused plans
# ================================================================================================
def _float_to_short(m):
    return isinstance(m, Convert) and m.IN is Format.FLOAT and m.OUT is Format.SHORT


def _walk_rank(m):
    """preference of a reader as the stage that continues a chain (_walk)"""
    if not isinstance(m, _Unfused):
        return 3
    if _float_to_short(m):
        w = m._writer
        if isinstance(w, Buffer) and isinstance(_GRAPH.consumer_of(w), AdpcmEncoder):
            return 2
        return 1
    return 0


def _walk(head):
    """the list of stages from `head` downstream through virtual Buffers, and the Buffers between them"""
    chain, links = [head], []
    cur = head
    for _ in range(64):
        w = cur._writer
        if not isinstance(w, Buffer):
            break
        # the stage that continues THIS chain: a Buffer can have further readers that start chains of their own (the secondary
        # FFT and the SecondarySelector on ClientDemodulatorChain.selectorBuffer, owrx/dsp.py:49,188-225) — those are heads
        # A fused stage goes before an unfused one: the WFm chain's tap buffer is read by the FractionalDecimator AND by the
        # RDS path's Convert(FLOAT, SHORT) (csdr/chain/analog.py:62,73-76); the chain goes on through the former.  On the
        # demodulator's audio Buffer a secondary demodulator's Convert(FLOAT, SHORT) sits beside the client-audio Converter: the
        # chain goes on through the AudioResampler (fused), else a Convert(FLOAT, SHORT) feeding an AdpcmEncoder, else any
        # Convert(FLOAT, SHORT); ties go to the older stage, so the choice never depends on the set's iteration order.
        cands = [m for m in list(_GRAPH.modules)
                 if m._reader is not None and m._reader._buffer is w and not m._stopped and not m._reader._stopped and not m.HEAD]
        if not cands:
            break
        nxt = min(cands, key=lambda m: (-_walk_rank(m), m._seq))
        links.append(w)
        chain.append(nxt)
        cur = nxt
    return chain, links


class _WaterfallPlan:
    def __init__(self, chain):
        self.key = None
        self.handle = None
        self.size = None
        self.update(chain)

    @staticmethod
    def match(chain):
        if len(chain) < 3 or not isinstance(chain[0], Fft) or not isinstance(chain[1], (LogPower, LogAveragePower)):
            return None
        if not isinstance(chain[2], FftSwap):
            return None
        n = 3
        if len(chain) > 3 and isinstance(chain[3], FftAdpcm):
            n = 4
        if chain[n - 1]._writer is None:
            return None
        return chain[:n]

    def update(self, chain):
        N = _native()
        fft, avg = chain[0], chain[1]
        comp = N.COMPRESSION_ADPCM if len(chain) == 4 else N.COMPRESSION_NONE
        if self.handle is None or self.size != fft.size:
            self.close()
            h = C.c_void_p()
            N.check(N.lib.owrx_wf_create(0, fft.size, fft.every_n_samples, avg.avg_number, avg.add_db, comp, C.byref(h)))
            self.handle, self.size = h, fft.size
            self.params = (fft.every_n_samples, avg.avg_number, comp)
        else:
            e, a, c = self.params
            if e != fft.every_n_samples:
                N.check(N.lib.owrx_wf_set_every_n_samples(self.handle, fft.every_n_samples))
            if a != avg.avg_number:
                N.check(N.lib.owrx_wf_set_avg_number(self.handle, avg.avg_number))
            if c != comp:
                N.check(N.lib.owrx_wf_set_compression(self.handle, comp))
            self.params = (fft.every_n_samples, avg.avg_number, comp)
        self.writer = chain[-1]._writer
        self.line_bytes = N.lib.owrx_wf_line_bytes(self.handle)
        self.buf = np.empty(self.line_bytes * 64, np.uint8)

    def feed(self, data, raw=None):
        N = _native()
        if raw is None:
            arr = np.frombuffer(data, dtype=np.float32)
            N.check(N.lib.owrx_wf_feed(self.handle, arr.ctypes.data_as(C.c_void_p), arr.size // 2))
        else:
            arr = np.frombuffer(data, dtype=np.uint8)
            fmt, gain = raw
            N.check(N.lib.owrx_wf_feed_fmt(self.handle, arr.ctypes.data_as(C.c_void_p), arr.size // (4 if fmt == "cs16" else 2),
                                           N.IQ_FORMATS[fmt], gain))
        lb = self.line_bytes
        while True:
            n = C.c_size_t()
            N.check(N.lib.owrx_wf_read(self.handle, self.buf.ctypes.data_as(C.c_void_p), self.buf.size, C.byref(n)))
            if n.value == 0:
                break
            for k in range(n.value // lb):
                # one write per line: the browser decodes each message as exactly one line (htdocs/openwebrx.js:1124-1131)
                self.writer.write(self.buf[k * lb:(k + 1) * lb].tobytes())

    def close(self):
        if self.handle is not None:
            _native().lib.owrx_wf_destroy(self.handle)
            self.handle = None


_DEMODS = ("nfm", "am", "ssb", "wfm", "none")


_TAP_WARNED = set()      # ids of tap Buffers whose float reader has been reported as not served


class _ChannelPlan:
    """one client chain = one channel of the source's bank"""

    def __init__(self):
        self.cid = None
        self.spec_key = None

    @staticmethod
    def _tap(writer_stage, nxt, what):
        """a tap of a Buffer inside a fused chain: `writer_stage` writes it, `nxt` (the chain's next stage) reads it, and any other
        reader is a tap consumer.  The WFm chain's multiplex tap (csdr/chain/analog.py:62,73-76: the Limit's Buffer, read by the
        audio path's FractionalDecimator and by the RDS path) and the demodulator's audio Buffer (read by the client-audio
        Converter and by a secondary demodulator) follow the same rules.  A Convert(FLOAT, SHORT) reader is fused: ("s16", the
        Convert's writer).  Any other reader gets the float samples in the Buffer itself: ("f32", that Buffer).  With both kinds
        of reader only the Convert is served (logged once).  (None, None) without a consumer."""
        tap = writer_stage._writer
        if not isinstance(tap, Buffer):
            return None, None
        for m in list(_GRAPH.modules):
            r = m._reader
            if (m is not nxt and _float_to_short(m) and r is not None and r._buffer is tap and not m._stopped and not r._stopped
                    and isinstance(m._writer, Buffer)):
                if tap._extra_readers(nxt._reader) and id(tap) not in _TAP_WARNED:
                    # one tap per channel: the bank delivers one format, and the int16 samples of the Convert win
                    _TAP_WARNED.add(id(tap))
                    logger.warning("pycsdr-b200: the %s has a float reader beside Convert(FLOAT, SHORT); only the "
                                   "Convert is served, the float reader receives nothing", what)
                return "s16", m._writer
        if tap._extra_readers(nxt._reader):
            return "f32", tap
        return None, None

    @staticmethod
    def match(chain):
        """returns dict describing the chain or None if it is not (yet) a complete, supported client chain"""
        i = 0
        d = {}
        if not isinstance(chain[0], Shift) or len(chain) < 2:
            return None
        d["shift"] = chain[0]
        if isinstance(chain[1], FirDecimate):
            d["fir"] = chain[1]
            i = 2
        elif isinstance(chain[1], Bandpass):
            # SecondarySelector: Shift -> Bandpass at the same rate (csdr/chain/selector.py:217-226): a channel with
            # decimation 1 and a one-tap (identity) FirDecimate
            d["fir"] = None
            i = 1
        else:
            return None
        d["frac"] = None
        if i < len(chain) and isinstance(chain[i], FractionalDecimator) and chain[i].format is Format.COMPLEX_FLOAT:
            d["frac"] = chain[i]; i += 1
        d["bandpass"] = None
        if i < len(chain) and isinstance(chain[i], Bandpass):
            d["bandpass"] = chain[i]; i += 1
        d["squelch"] = None
        if i < len(chain) and isinstance(chain[i], Squelch):
            d["squelch"] = chain[i]; i += 1
        d["if_index"] = i - 1          # last selector stage: its writer carries the selector output
        rest = chain[i:]
        kinds = [type(m) for m in rest]
        d["agc"] = None
        if kinds[:4] == [FmDemod, Limit, NfmDeemphasis, Agc]:
            d["demod"], d["deemph"], d["agc"], used = "nfm", rest[2], rest[3], 4
        elif kinds[:3] == [AmDemod, DcBlock, Agc]:
            d["demod"], d["agc"], used = "am", rest[2], 3
        elif kinds[:2] == [RealPart, Agc]:
            d["demod"], d["agc"], used = "ssb", rest[1], 2
        elif kinds[:4] == [FmDemod, Limit, FractionalDecimator, WfmDeemphasis] and rest[2].format is Format.FLOAT:
            d["demod"], d["wfm_frac"], d["wfm_de"], used = "wfm", rest[2], rest[3], 4
            d["mpx"], d["mpx_writer"] = _ChannelPlan._tap(rest[1], rest[2], "WFM tap buffer")
        elif not rest:
            d["demod"], used = "none", 0
        else:
            return None
        # client audio tail (csdr/chain/clientaudio.py:6-35): [AudioResampler + Limit] Convert(FLOAT, SHORT)
        # [+ AdpcmEncoder(sync=True)]
        after = rest[used:]
        d["audio_fmt"] = "f32"
        d["resampler"] = None
        # a second reader of the demodulator's audio Buffer (a secondary demodulator: Convert(FLOAT, SHORT) -> decoder) is
        # served by the audio tap when the chain goes on past that Buffer; with float client audio the Buffer is materialised
        d["atap"], d["atap_writer"] = None, None
        if after and d["demod"] != "none":
            d["atap"], d["atap_writer"] = _ChannelPlan._tap(rest[used - 1], after[0], "demodulator's audio buffer")
        if after and d["demod"] != "none" and isinstance(after[0], AudioResampler):
            rs = after[0]
            if len(after) < 3 or not isinstance(after[1], Limit) or not _resampler_ok(rs.inputRate, rs.outputRate):
                return None
            d["resampler"] = (rs.inputRate, rs.outputRate)
            d["resampler_stages"] = (after[0], after[1])
            after = after[2:]
            used += 2
        if after and d["demod"] != "none":
            cv = after[0]
            if not (isinstance(cv, Convert) and cv.IN is Format.FLOAT and cv.OUT is Format.SHORT):
                return None
            d["audio_fmt"] = "s16"
            used += 1
            if len(after) > 1:
                if not isinstance(after[1], AdpcmEncoder) or len(after) > 2:
                    return None
                d["audio_fmt"] = "adpcm"
                used += 1
        elif after:
            return None
        tail = chain[i + used - 1] if used else chain[d["if_index"]]
        if tail._writer is None:
            return None
        d["tail"] = tail
        d["stages"] = chain[:i + used]
        return d


class _SourceRunner(threading.Thread):
    """one per source Buffer: reads each block once and feeds every fused plan hanging off it"""

    _lock = threading.Lock()

    def __init__(self, buffer):
        super().__init__(daemon=True, name="pycsdr-b200-runner")
        self.buffer = buffer
        self.reader = buffer.getReader()
        self.epoch = -1
        self.wf_plans = {}        # id(Fft stage) -> _WaterfallPlan
        self.bank = None
        self.channels = {}        # id(Shift stage) -> dict(plan state)
        self.unsupported = set()
        self.processed = 0        # sequence number of the source Buffer up to which every plan has been fed and drained

    @classmethod
    def attach(cls, buffer):
        with cls._lock:
            r = buffer._runner
            if r is None or not r.is_alive():
                buffer._enable_ring()
                r = cls(buffer)
                buffer._runner = r
                r.start()
        return r

    # ---------------------------------------------------------------- topology
    def heads(self):
        out = []
        for m in list(_GRAPH.modules):
            r = m._reader
            if m.HEAD and r is not None and r._buffer is self.buffer and not m._stopped and not r._stopped:
                out.append(m)
        return out

    def rebuild(self):
        N = _native()
        self.epoch = _GRAPH.epoch
        live_wf, live_ch = set(), set()
        for head in self.heads():
            chain, links = _walk(head)
            if isinstance(head, Fft):
                m = _WaterfallPlan.match(chain)
                if m is None:
                    continue
                plan = self.wf_plans.get(id(head))
                if plan is None:
                    self.wf_plans[id(head)] = _WaterfallPlan(m)
                else:
                    plan.update(m)
                live_wf.add(id(head))
            elif isinstance(head, Shift):
                d = _ChannelPlan.match(chain)
                if d is None:
                    if len(chain) > 2 and id(head) not in self.unsupported and chain[-1]._writer is not None:
                        self.unsupported.add(id(head))
                        logger.error("pycsdr-b200: client chain %s is not a fusable hot-path chain; it will not run",
                                     [type(m).__name__ for m in chain])
                    continue
                try:
                    self._update_channel(N, head, d, links)
                except (ValueError, BufferError) as e:
                    # one client's spec was rejected by the library (e.g. a band-pass transition out of range): that chain
                    # does not run; every other client of this source keeps running
                    if id(head) not in self.unsupported:
                        self.unsupported.add(id(head))
                        logger.error("pycsdr-b200: client chain %s rejected: %s", [type(m).__name__ for m in chain], e)
                    st = self.channels.pop(id(head), None)
                    if st is not None:
                        N.lib.owrx_bank_remove_channel(self.bank, st["cid"])
                    continue
                live_ch.add(id(head))
        for k in [k for k in self.wf_plans if k not in live_wf]:
            self.wf_plans.pop(k).close()
        for k in [k for k in self.channels if k not in live_ch]:
            st = self.channels.pop(k)
            N.lib.owrx_bank_remove_channel(self.bank, st["cid"])

    def _update_channel(self, N, head, d, links):
        fir, frac, bp, sq = d["fir"], d["frac"], d["bandpass"], d["squelch"]
        sp = N.ChanSpec()
        if fir is not None:
            sp.decimation, sp.transition, sp.cutoff = fir.decimation, fir.transition, fir.cutoff
        else:
            sp.decimation, sp.transition, sp.cutoff = 1, 4.0, 0.5          # filter length odd(int(4/4)) = 1: identity
        sp.fraction = frac.rate if frac is not None else 1.0
        sp.bp_transition = bp.transition if bp is not None else 0.05
        sp.squelch_length = sq.length if sq is not None else 750
        sp.deemph_rate = d["deemph"].sampleRate if d["demod"] == "nfm" else 12000
        sp.wfm = 1 if d["demod"] == "wfm" else 0
        if sp.wfm:
            sp.wfm_decimation = d["wfm_frac"].rate
            sp.wfm_audio_rate = d["wfm_de"].sampleRate
            sp.wfm_tau = d["wfm_de"].tau
        key = (sp.decimation, sp.transition, sp.cutoff, sp.fraction, sp.bp_transition, sp.squelch_length, sp.deemph_rate,
               sp.wfm, sp.wfm_decimation, sp.wfm_audio_rate, sp.wfm_tau, d["demod"], d["audio_fmt"],
               tuple(id(m) for m in d["stages"] if m not in d.get("resampler_stages", ())))
        if self.bank is None:
            h = C.c_void_p()
            N.check(N.lib.owrx_bank_create(0, 1.0, C.byref(h)))     # rates are carried by the explicit specs
            self.bank = h
        st = self.channels.get(id(head))
        if st is not None and st["key"] != key:
            N.lib.owrx_bank_remove_channel(self.bank, st["cid"])
            st = None
        if st is None:
            cid = C.c_int()
            N.check(N.lib.owrx_bank_add_channel_ex(self.bank, C.byref(sp), C.byref(cid)))
            kind = {"nfm": N.DEMOD_NFM, "am": N.DEMOD_AM, "ssb": N.DEMOD_SSB, "wfm": N.DEMOD_WFM, "none": N.DEMOD_NONE}[d["demod"]]
            agc = d.get("agc")
            prof = N.AGC_FAST if (agc is not None and agc.profile is AgcProfile.FAST) else N.AGC_SLOW
            if kind != N.DEMOD_WFM:
                N.check(N.lib.owrx_chan_set_demod(self.bank, cid.value, kind, 0.0, 0.0, prof))
            if agc is not None:
                N.check(N.lib.owrx_chan_set_agc(self.bank, cid.value, prof, agc.initialGain, agc.maxGain))
            fmt = {"f32": N.AUDIO_F32, "s16": N.AUDIO_S16, "adpcm": N.AUDIO_ADPCM}[d["audio_fmt"]]
            N.check(N.lib.owrx_chan_set_audio_format(self.bank, cid.value, fmt))
            st = {"cid": cid.value, "key": key, "rate": None, "bp": None, "level": None, "audio_fmt": d["audio_fmt"]}
            self.channels[id(head)] = st
        cid = st["cid"]
        if st["rate"] != head.rate:
            N.check(N.lib.owrx_chan_set_shift_rate(self.bank, cid, head.rate))
            st["rate"] = head.rate
        bpv = (bp.low, bp.high) if (bp is not None and bp.low is not None) else None
        if st["bp"] != bpv:
            if bpv is None:
                N.check(N.lib.owrx_chan_set_bandpass(self.bank, cid, 0.0, 0.0, 0))
            else:
                N.check(N.lib.owrx_chan_set_bandpass(self.bank, cid, bpv[0], bpv[1], 1))
            st["bp"] = bpv
        level = sq.level if sq is not None else 0.0
        if st["level"] != level:
            N.check(N.lib.owrx_chan_set_squelch_level(self.bank, cid, level))
            st["level"] = level
        # the resampler follows its chain through the setter (a new one starts from empty history)
        if st.get("resampler") != d["resampler"]:
            rin, rout = d["resampler"] or (0, 0)
            N.check(N.lib.owrx_chan_set_audio_resampler(self.bank, cid, rin, rout))
            st["resampler"] = d["resampler"]
        # the multiplex tap follows its consumers through the setter: no rebuild of the channel when RDS comes or goes
        mpx = d.get("mpx")
        if st.get("mpx") != mpx:
            N.check(N.lib.owrx_chan_set_mpx(self.bank, cid, {None: N.MPX_OFF, "f32": N.MPX_F32, "s16": N.MPX_S16}[mpx]))
            st["mpx"] = mpx
        st["mpx_writer"] = d.get("mpx_writer")
        # so does the audio tap: no rebuild when a secondary demodulator comes or goes
        atap = d.get("atap")
        if st.get("atap") != atap:
            N.check(N.lib.owrx_chan_set_audio_tap(self.bank, cid, {None: N.MPX_OFF, "f32": N.MPX_F32, "s16": N.MPX_S16}[atap]))
            st["atap"] = atap
        st["atap_writer"] = d.get("atap_writer")
        st["demod"] = d["demod"]
        st["tail_writer"] = d["tail"]._writer
        st["power_writer"] = sq.powerWriter if sq is not None else None
        # the selector output is materialised only if someone besides the next fused stage reads it
        if_stage = d["stages"][d["if_index"]]
        st["if_writer"] = None
        if d["demod"] != "none" and isinstance(if_stage._writer, Buffer):
            nxt = d["stages"][d["if_index"] + 1]
            if if_stage._writer._extra_readers(nxt._reader):
                st["if_writer"] = if_stage._writer
        mask = 0
        for s in self.channels.values():
            mask |= N.OUT_IF if (s.get("if_writer") is not None or s.get("demod") == "none") else 0
            mask |= N.OUT_AUDIO if (s.get("demod") != "none" and s.get("audio_fmt") == "f32") else 0
            mask |= N.OUT_POWER if s.get("power_writer") is not None else 0
        N.check(N.lib.owrx_bank_set_outputs(self.bank, mask))

    # ---------------------------------------------------------------- data
    def run(self):
        N = None
        idle = 0
        while True:
            self.processed = self.reader._pos
            views = self.reader._read_views()   # the runner batches everything that has arrived (views into the pinned ring)
            if views is None:
                break
            try:
                if N is None:
                    N = _native()
                if self.epoch != _GRAPH.epoch:
                    with _GRAPH.lock:
                        self.rebuild()
                if not self.wf_plans and not self.channels:
                    idle += 1
                    if idle > 64 and not self.heads():
                        with self._lock:
                            self.buffer._runner = None
                        self.reader.stop()
                        break
                    continue
                idle = 0
                raw = self.buffer._raw          # source-side Convert (+ Gain): the buffer carries raw samples
                for data in views:
                    for plan in list(self.wf_plans.values()):
                        plan.feed(data, raw)
                    if self.channels:
                        self._feed_bank(N, data, raw)
            except (ValueError, BufferError):
                # a bad argument on one plan: logged, the source keeps feeding (only CUDA / memory failures are fatal)
                logger.exception("pycsdr-b200 runner: block dropped")
                continue
            except Exception:
                logger.exception("pycsdr-b200 runner failed")
                break
        with self._lock:
            if self.buffer._runner is self:
                self.buffer._runner = None
        self.reader.stop()                      # a dead runner must not pin chunks of the source Buffer
        for p in self.wf_plans.values():
            p.close()
        if self.bank is not None and N is not None:
            N.lib.owrx_bank_destroy(self.bank)
            self.bank = None

    def _drain(self, N, fn, cid, width):
        out = []
        buf = np.empty(65536 * width, np.float32)
        while True:
            n = C.c_size_t()
            N.check(fn(self.bank, cid, buf.ctypes.data_as(C.c_void_p), 65536, C.byref(n)))
            if n.value == 0:
                break
            out.append(buf[:n.value * width].tobytes())
        return b"".join(out)

    def _drain_bytes(self, N, cid, fn=None):
        fn = fn or N.lib.owrx_chan_read_bytes
        out = []
        buf = np.empty(1 << 16, np.uint8)
        while True:
            n = C.c_size_t()
            N.check(fn(self.bank, cid, buf.ctypes.data_as(C.c_void_p), buf.size, C.byref(n)))
            if n.value == 0:
                break
            out.append(buf[:n.value].tobytes())
        return b"".join(out)

    def _feed_bank(self, N, data, raw=None):
        if raw is None:
            arr = np.frombuffer(data, dtype=np.float32)
            N.check(N.lib.owrx_bank_feed(self.bank, arr.ctypes.data_as(C.c_void_p), arr.size // 2))
        else:
            arr = np.frombuffer(data, dtype=np.uint8)
            fmt, gain = raw
            N.check(N.lib.owrx_bank_feed_fmt(self.bank, arr.ctypes.data_as(C.c_void_p), arr.size // (4 if fmt == "cs16" else 2),
                                             N.IQ_FORMATS[fmt], gain))
        for st in list(self.channels.values()):
            cid = st["cid"]
            if st["demod"] == "none":
                b = self._drain(N, N.lib.owrx_chan_read_if, cid, 2)
                if b:
                    st["tail_writer"].write(b)
            else:
                if st.get("audio_fmt", "f32") == "f32":
                    b = self._drain(N, N.lib.owrx_chan_read_audio, cid, 1)
                else:
                    b = self._drain_bytes(N, cid)
                if b:
                    st["tail_writer"].write(b)
                if st.get("if_writer") is not None:
                    bi = self._drain(N, N.lib.owrx_chan_read_if, cid, 2)
                    if bi:
                        st["if_writer"].write(bi)
                if st.get("mpx_writer") is not None:
                    bm = self._drain_bytes(N, cid, N.lib.owrx_chan_read_mpx)
                    if bm:
                        st["mpx_writer"].write(bm)
                if st.get("atap_writer") is not None:
                    ba = self._drain_bytes(N, cid, N.lib.owrx_chan_read_audio_tap)
                    if ba:
                        st["atap_writer"].write(ba)
            if st.get("power_writer") is not None:
                bp = self._drain(N, N.lib.owrx_chan_read_power, cid, 1)
                if bp:
                    st["power_writer"].write(bp)
