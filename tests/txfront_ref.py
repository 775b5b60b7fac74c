"""The TX front end's definition, for the tests (test infrastructure only, like oracle/).

gr_mod_base (gr_mod_base.cpp:38,211-290,799-805) runs mod -> rotator_cc(2 pi offset / 1e6) and, when the sink runs at
samp_rate >= 2 Msps, rational_resampler_ccf(N, 1, low_pass(N, samp_rate, 480000, 20000, BLACKMAN_HARRIS)), N = samp_rate / 1e6;
below 2 Msps the rotator feeds the sink directly (N = 1: the rotator alone).

* Rotator: the oracle's exact Q32 NCO (the receive side's rotator) with the TX sign, inc = rint(+offset / 1e6 * 2^32), phase =
  base + inc (n - n_base) over the absolute 1 Msps index, sin / cos from the oracle's qo_sincosf; a retune is phase-continuous.
  Channels whose phase is identically zero pass through unrotated.
* Interpolator: the oracle's resampler arms (arm[p][k] = taps[p + k N], zero padded), each output one sequential fmaf chain,
  oldest sample first; the history holds rotated samples.  Every input item yields exactly N outputs.
* sc16: per component clamp(rint(x * scale), -32768, 32767), one float32 multiply and round-half-even.

The float loops are C (tests/txfront_ref.c, compiled into a temporary directory at first use with the oracle's flags and linked
against the oracle's library for qo_sincosf); the stream state is kept here."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

from oracle import oracle as O

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None
RATES = [1000000] + [k * 1000000 for k in range(2, 57)]


def _lib():
    global _LIB
    if _LIB is None:
        so_oracle = O.build()
        d = tempfile.mkdtemp(prefix="txfront_ref_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libtxfront_ref.so")
        subprocess.check_call(["gcc", "-O2", "-march=x86-64-v3", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared", "-o", so,
                               os.path.join(_HERE, "txfront_ref.c"), so_oracle, "-Wl,-rpath," + os.path.dirname(so_oracle), "-lm"])
        L = C.CDLL(so)
        L.txref_rotate.argtypes = [C.c_void_p, C.c_long, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p]
        L.txref_interp.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_long, C.c_void_p]
        _LIB = L
    return _LIB


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def design_taps(samp_rate):
    """low_pass(N, samp_rate, 480000, 20000, BLACKMAN_HARRIS) of the oracle's firdes restatement."""
    N = samp_rate // 1000000
    return O.low_pass(N, samp_rate, 480000, 20000, O.WIN_BLACKMAN_HARRIS)


class TxFrontend:
    """One channel of the TX front end at device rate samp_rate."""

    def __init__(self, samp_rate):
        if samp_rate not in RATES:
            raise ValueError("TX front end: samp_rate must be 1e6 or a multiple of 1e6 in [2e6, 56e6]")
        self.N = samp_rate // 1000000
        self.n = 0
        self.base = self.inc = self.nbase = 0
        self.ntaps = self.arm_taps = 0
        if self.N > 1:
            h = design_taps(samp_rate)
            self.ntaps = len(h)
            self.arm_taps = -(-len(h) // self.N)
            padded = np.zeros(self.arm_taps * self.N, np.float32)
            padded[:len(h)] = h
            self._arms = np.ascontiguousarray(padded.reshape(self.arm_taps, self.N).T)     # [N][nt]
            self._hist = np.zeros(self.arm_taps - 1, np.complex64)

    def set_carrier_offset(self, hz):
        self.base = (self.base + self.inc * (self.n - self.nbase)) & 0xFFFFFFFF
        self.nbase = self.n
        self.inc = int(np.rint(hz / 1e6 * 4294967296.0)) & 0xFFFFFFFF

    def work(self, iq):
        x = np.ascontiguousarray(iq, np.complex64)
        n = len(x)
        if self.inc or self.base:
            y = np.empty_like(x)
            _lib().txref_rotate(_p(x), n, self.base, self.inc, (self.n - self.nbase) & 0xFFFFFFFF, _p(y))
            x = y
        self.n += n
        if self.N == 1:
            return x.copy()
        w = np.concatenate([self._hist, x])
        out = np.empty(n * self.N, np.complex64)
        if n:
            _lib().txref_interp(_p(self._arms), self.N, self.arm_taps, _p(w), n, _p(out))
        self._hist = w[len(w) - (self.arm_taps - 1):].copy()
        return out


def to_sc16(x, scale):
    """complex64 [..., n] -> int16 [..., 2 n]: per component clamp(rint(x * scale), -32768, 32767)."""
    v = np.ascontiguousarray(x, np.complex64).view(np.float32) * np.float32(scale)
    return np.clip(np.rint(v), -32768, 32767).astype(np.int16)
