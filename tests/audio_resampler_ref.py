"""Reference of the client-audio resampler, AudioResampler(in, out) -> Limit (csdr/chain/clientaudio.py:6-19).  Test
infrastructure only: the product runs audio_resample_kernel (openwebrx_b200/csrc/selector_kernels.cuh).

SPEC-DEFINED: the reference calls libsamplerate, whose converter type and tables are not in the tree, so this restates the
resampler the project defines (DESIGN.md section 7) and is excluded from reference-parity claims:
  L/M = out/in reduced; prototype low-pass at the rate L*in, Kaiser-windowed sinc with a 96 dB stop band (beta = 0.1102 (A - 8.7)),
  transition 0.1 min(in, out) and cutoff 0.45 min(in, out); K = ceil(((A - 7.95) / (14.36 df) + 1) / L) taps per phase, N = L K,
  designed in double and scaled so that sum h = L; ratios with N > 65536 are rejected.
  y[k] = sum_n x[n] h[kM - nL], causal (x[n < 0] = 0): after n inputs exactly ceil(n L / M) outputs exist.  Then Limit (clamp to +-1).
"""
import math

import numpy as np

MAX_TAPS = 65536


def design(in_rate, out_rate):
    """(h float64 [L*K], L, M, K), or None for a rejected ratio"""
    in_rate, out_rate = int(in_rate), int(out_rate)
    if in_rate <= 0 or out_rate <= 0:
        return None
    g = math.gcd(in_rate, out_rate)
    L, M = out_rate // g, in_rate // g
    A = 96.0
    beta = 0.1102 * (A - 8.7)
    f_lo, fs = min(in_rate, out_rate), float(L) * in_rate
    df, fc = 0.1 * f_lo / fs, 0.45 * f_lo / fs
    K = math.ceil(((A - 7.95) / (14.36 * df) + 1.0) / L)
    if L * K > MAX_TAPS:
        return None
    N = L * K
    i = np.arange(N, dtype=np.float64)
    r = 2.0 * i / (N - 1) - 1.0 if N > 1 else np.zeros(1)
    w = np.i0(beta * np.sqrt(np.maximum(0.0, 1.0 - r * r))) / np.i0(beta)
    h = 2.0 * fc * np.sinc(2.0 * fc * (i - (N - 1) / 2.0)) * w
    return h * (L / h.sum()), L, M, K


class Resampler:
    """streaming AudioResampler -> Limit: taps rounded once to float32, float32 accumulation, one output at a time in the
    kernel's tap order (newest input first)"""

    def __init__(self, in_rate, out_rate):
        d = design(in_rate, out_rate)
        if d is None:
            raise ValueError("rejected resampler ratio %d -> %d" % (in_rate, out_rate))
        h, self.L, self.M, self.K = d
        self.hp = h.astype(np.float32).reshape(self.K, self.L).T.copy()      # hp[p, j] = h[p + j L]
        self.hist = np.zeros(self.K - 1, np.float32)                          # the last K - 1 inputs (zeros before the first)
        self.n_in = 0
        self.k_out = 0

    def process(self, x):
        x = np.asarray(x, np.float32)
        buf = np.concatenate([self.hist, x])
        base = self.n_in - (self.K - 1)                                       # absolute index of buf[0]
        n_end = self.n_in + len(x)
        k = np.arange(self.k_out, -(-n_end * self.L // self.M), dtype=np.int64)
        nmax = k * self.M // self.L
        p = k * self.M - nmax * self.L
        acc = np.zeros(len(k), np.float32)
        for j in range(self.K):
            n = nmax - j
            v = np.where(n >= 0, buf[np.maximum(n - base, 0)], np.float32(0))
            acc = (acc + v * self.hp[p, j]).astype(np.float32)
        self.hist = buf[len(buf) - (self.K - 1):] if self.K > 1 else self.hist
        self.n_in = n_end
        self.k_out += len(k)
        return np.clip(acc, -1.0, 1.0).astype(np.float32)


def resample(x, in_rate, out_rate, parts=None):
    """AudioResampler(in, out) -> Limit over x, fed in pieces of the given lengths (default: one piece)"""
    r = Resampler(in_rate, out_rate)
    x = np.asarray(x, np.float32)
    out, o = [], 0
    for n in (list(parts) if parts is not None else []) + [len(x)]:
        n = min(int(n), len(x) - o)
        out.append(r.process(x[o:o + n]))
        o += n
    return np.concatenate(out)
