"""Front end at device rates >= 2 Msps: host-side mirror of gr_demod_base::set_samp_rate / set_carrier_offset for that case
(/root/reference/src/gr/gr_demod_base.cpp:1220-1225, 1303-1362): rotator at the device rate + rational_resampler_ccf(1, samp_rate / 1e6)
for a batch of channels.  The output stays in HBM in the layout RxBlock.work_device takes."""
import ctypes as C

import numpy as np

from .lib import QrlError, check, load_library


class Frontend:
    def __init__(self, samp_rate, n_channels=1, max_in=1 << 21, device=0):
        self._L = load_library()
        self.n_channels, self.max_in, self.decimation = int(n_channels), int(max_in), int(samp_rate) // 1000000
        self._h = C.c_void_p()
        rc = self._L.qrl_frontend_create(int(samp_rate), self.n_channels, self.max_in, device, C.byref(self._h))
        if rc != 0:
            raise QrlError("qrl_frontend_create failed (%d): %s" % (rc, (self._L.qrl_last_error(None) or b"").decode()))

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._L.qrl_frontend_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, cuda_stream_ptr):
        check(self._L.qrl_frontend_set_stream(self._h, C.c_void_p(cuda_stream_ptr)), self._h, "qrl_frontend_set_stream")

    def set_carrier_offset(self, hz, channel=-1):
        check(self._L.qrl_frontend_set_carrier_offset(self._h, channel, float(hz)), self._h, "qrl_frontend_set_carrier_offset")

    def work(self, iq):
        """iq: complex64 [n_channels, T] at the device rate (host) -> complex64 [n_channels, n_out] at 1 Msps."""
        iq = np.ascontiguousarray(iq, np.complex64)
        if iq.ndim == 1:
            iq = iq[None, :]
        T = iq.shape[1]
        n = C.c_long()
        check(self._L.qrl_frontend_work(self._h, iq.ctypes.data_as(C.c_void_p), T, T, 0, C.byref(n)), self._h, "qrl_frontend_work")
        out = np.zeros((self.n_channels, max(1, n.value)), np.complex64)
        check(self._L.qrl_frontend_read(self._h, out.ctypes.data_as(C.c_void_p), out.shape[1]), self._h, "qrl_frontend_read")
        return out[:, :n.value]

    def work_device(self, dev_ptr, T, stride):
        n = C.c_long()
        check(self._L.qrl_frontend_work(self._h, C.c_void_p(dev_ptr), T, stride, 1, C.byref(n)), self._h, "qrl_frontend_work")
        return n.value

    def out_device(self):
        """(device pointer, stride, items) of the last call's 1 Msps output: pass to RxBlock.work_device(ptr, items, stride)."""
        p, s, n = C.c_void_p(), C.c_long(), C.c_long()
        check(self._L.qrl_frontend_out_device(self._h, C.byref(p), C.byref(s), C.byref(n)), self._h, "qrl_frontend_out_device")
        return p.value, s.value, n.value


class TxFrontend:
    """TX front end: host-side mirror of gr_mod_base's rotator_cc + rational_resampler_ccf(N, 1) pair (/root/reference/src/gr/
    gr_mod_base.cpp:38,211-290,799-805) for a batch of channels.  1 Msps complex64 in (e.g. TxBlock.out_device), N * n items at
    samp_rate out, complex64 ("fc32") or interleaved int16 I/Q ("sc16", per component clamp(rint(x * scale)))."""

    FORMATS = {"fc32": 0, "sc16": 1}

    def __init__(self, samp_rate, n_channels=1, max_in=1 << 20, out_format="fc32", scale=32767.0, device=0):
        if out_format not in self.FORMATS:
            raise ValueError("out_format must be 'fc32' or 'sc16'")
        self._L = load_library()
        self.n_channels, self.max_in, self.interpolation = int(n_channels), int(max_in), int(samp_rate) // 1000000
        self.out_format = out_format
        self._h = C.c_void_p()
        rc = self._L.qrl_txfront_create(int(samp_rate), self.n_channels, self.max_in, self.FORMATS[out_format], float(scale), device, C.byref(self._h))
        if rc != 0:
            raise QrlError("qrl_txfront_create failed (%d): %s" % (rc, (self._L.qrl_last_error(None) or b"").decode()))

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._L.qrl_txfront_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def launches(self):
        return self._L.qrl_txfront_launch_count(self._h)

    def set_stream(self, cuda_stream_ptr):
        check(self._L.qrl_txfront_set_stream(self._h, C.c_void_p(cuda_stream_ptr)), self._h, "qrl_txfront_set_stream")

    def set_carrier_offset(self, hz, channel=-1):
        check(self._L.qrl_txfront_set_carrier_offset(self._h, channel, float(hz)), self._h, "qrl_txfront_set_carrier_offset")

    def read(self, n_out):
        """The last call's output: complex64 [n_channels, n_out] (fc32) or int16 [n_channels, 2 n_out] (sc16)."""
        if self.out_format == "fc32":
            out = np.zeros((self.n_channels, max(1, n_out)), np.complex64)
        else:
            out = np.zeros((self.n_channels, 2 * max(1, n_out)), np.int16)
        check(self._L.qrl_txfront_read(self._h, out.ctypes.data_as(C.c_void_p), max(1, n_out)), self._h, "qrl_txfront_read")
        return out[:, :n_out] if self.out_format == "fc32" else out[:, :2 * n_out]

    def work(self, iq):
        """iq: complex64 [n_channels, n] at 1 Msps (host) -> the n * N items at the device rate (see read)."""
        iq = np.ascontiguousarray(iq, np.complex64)
        if iq.ndim == 1:
            iq = iq[None, :]
        n = C.c_long()
        check(self._L.qrl_txfront_work(self._h, iq.ctypes.data_as(C.c_void_p), iq.shape[1], iq.shape[1], 0, C.byref(n)), self._h, "qrl_txfront_work")
        return self.read(n.value)

    def work_device(self, dev_ptr, n, stride):
        """Device-resident input ([n_channels][stride] complex64 on the handle's GPU, e.g. TxBlock.out_device()); returns N * n."""
        o = C.c_long()
        check(self._L.qrl_txfront_work(self._h, C.c_void_p(dev_ptr), n, stride, 1, C.byref(o)), self._h, "qrl_txfront_work")
        return o.value

    def out_device(self):
        """(device pointer, stride in items, items) of the last call's output; it stays valid until the next work call."""
        p, s, n = C.c_void_p(), C.c_long(), C.c_long()
        check(self._L.qrl_txfront_out_device(self._h, C.byref(p), C.byref(s), C.byref(n)), self._h, "qrl_txfront_out_device")
        return p.value, s.value, n.value
