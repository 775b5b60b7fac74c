"""ctypes binding of libqrl_b200.so (C ABI: include/qrl_b200.h).  Fails loudly if the library is missing."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libqrl_b200.so")
_LIB = None


class QrlError(RuntimeError):
    pass


class KIND:
    DEMOD_NBFM, DEMOD_4FSK, DEMOD_QPSK, DEMOD_BPSK, DEMOD_2FSK, DEMOD_SSB, DEMOD_AM, DEMOD_GMSK, DEMOD_WBFM, DEMOD_M17, DEMOD_DMR, DEMOD_DSSS = 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12
    MOD_4FSK, MOD_QPSK, MOD_NBFM, MOD_BPSK, MOD_2FSK, MOD_SSB, MOD_GMSK, MOD_M17, MOD_DMR, MOD_DSSS, MOD_AM = 101, 102, 103, 104, 105, 106, 107, 108, 109, 110, 111


class PARAM:
    CARRIER_OFFSET_HZ, SQUELCH_DB, FILTER_WIDTH, BB_GAIN, OVERLAP_CALLS, RSSI, CTCSS, AGC_ATTACK, AGC_DECAY, GAIN = 1, 2, 3, 4, 5, 6, 7, 8, 9, 10


# every symbol include/qrl_b200.h declares: (restype, argtypes)
_vp, _i, _l, _d = C.c_void_p, C.c_int, C.c_long, C.c_double
SYMBOLS = {
    "qrl_device_count": (_i, []),
    "qrl_version": (C.c_char_p, []),
    "qrl_last_error": (C.c_char_p, [_vp]),
    "qrl_rx_create": (_i, [_i] * 7 + [_l, _i, C.POINTER(_vp)]),
    "qrl_rx_destroy": (_i, [_vp]),
    "qrl_rx_set_stream": (_i, [_vp, _vp]),
    "qrl_rx_set_param": (_i, [_vp, _i, _i, _d]),
    "qrl_rx_reset": (_i, [_vp]),
    "qrl_rx_work": (_i, [_vp, _vp, _l, _l, _i]),
    "qrl_rx_work_sc16": (_i, [_vp, _vp, _l, _l, C.c_float, _i]),
    "qrl_rx_work_sc8": (_i, [_vp, _vp, _l, _l, C.c_float, _i]),
    "qrl_rx_sync": (_i, [_vp]),
    "qrl_rx_join": (_i, [_vp]),
    "qrl_rx_rssi": (_i, [_vp, C.c_float, _vp]),
    "qrl_rx_num_ports": (_i, [_vp]),
    "qrl_rx_port_itemsize": (_i, [_vp, _i]),
    "qrl_rx_read_port": (_i, [_vp, _i, _vp, _l, _vp, _i]),
    "qrl_rx_port_device": (_i, [_vp, _i, C.POINTER(_vp), C.POINTER(_l), C.POINTER(_vp)]),
    "qrl_rx_launch_count": (_l, [_vp]),
    "qrl_rx_sm_partition": (_i, [_vp, C.POINTER(_i), C.POINTER(_i)]),
    "qrl_rx_profile": (_i, [_vp, _i]),
    "qrl_rx_profile_read": (_i, [_vp, _i, C.POINTER(_d), C.POINTER(_l)]),
    "qrl_tx_create": (_i, [_i] * 7 + [_l, _i, C.POINTER(_vp)]),
    "qrl_tx_destroy": (_i, [_vp]),
    "qrl_tx_set_stream": (_i, [_vp, _vp]),
    "qrl_tx_set_param": (_i, [_vp, _i, _i, _d]),
    "qrl_tx_work": (_i, [_vp, _vp, _l, _l, _i]),
    "qrl_tx_sync": (_i, [_vp]),
    "qrl_tx_read": (_i, [_vp, _vp, _l, C.POINTER(_l), _i]),
    "qrl_tx_out_device": (_i, [_vp, C.POINTER(_vp), C.POINTER(_l), C.POINTER(_l)]),
    "qrl_tx_launch_count": (_l, [_vp]),
    "qrl_tx_profile": (_i, [_vp, _i]),
    "qrl_tx_zero_samples": (_i, [_vp, _i, C.c_longlong, _l]),
    "qrl_mmdvm_rx_create": (_i, [_i, _i, _vp, _i, _i, _l, _i, _vp]),
    "qrl_mmdvm_rx_destroy": (_i, [_vp]),
    "qrl_mmdvm_rx_set_stream": (_i, [_vp, _vp]),
    "qrl_mmdvm_rx_calibrate_rssi": (_i, [_vp, C.c_float]),
    "qrl_mmdvm_rx_work": (_i, [_vp, _vp, _l, _l, _i, _vp]),
    "qrl_mmdvm_rx_sync": (_i, [_vp]),
    "qrl_mmdvm_rx_out_device": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "qrl_mmdvm_rx_read": (_i, [_vp, _vp, _l, _vp, _l, _vp, _vp]),
    "qrl_mmdvm_rx_launch_count": (_l, [_vp]),
    "qrl_mmdvm_tx_create": (_i, [_i, _i, _vp, _i, _i, _l, _i, _vp]),
    "qrl_mmdvm_tx_destroy": (_i, [_vp]),
    "qrl_mmdvm_tx_set_stream": (_i, [_vp, _vp]),
    "qrl_mmdvm_tx_set_bb_gain": (_i, [_vp, C.c_float]),
    "qrl_mmdvm_tx_zero_samples": (_i, [_vp, _i, C.c_longlong, _l]),
    "qrl_mmdvm_tx_work": (_i, [_vp, _vp, _l, _l, _i, _vp]),
    "qrl_mmdvm_tx_sync": (_i, [_vp]),
    "qrl_mmdvm_tx_out_device": (_i, [_vp, _vp, _vp, _vp]),
    "qrl_mmdvm_tx_read": (_i, [_vp, _vp, _l]),
    "qrl_mmdvm_tx_finish": (_i, [_vp, _vp, _l]),
    "qrl_mmdvm_tx_launch_count": (_l, [_vp]),
    "qrl_spectrum_create": (_i, [_i, _i, _i, _l, _i, _vp]),
    "qrl_spectrum_destroy": (_i, [_vp]),
    "qrl_spectrum_set_stream": (_i, [_vp, _vp]),
    "qrl_spectrum_set_enabled": (_i, [_vp, _i]),
    "qrl_spectrum_set_fft_size": (_i, [_vp, _i]),
    "qrl_spectrum_work": (_i, [_vp, _vp, _l, _l, _i]),
    "qrl_spectrum_get": (_i, [_vp, _vp, _l, _i, _vp]),
    "qrl_spectrum_launch_count": (_l, [_vp]),
    "qrl_tx_profile_read": (_i, [_vp, _i, C.POINTER(_d), C.POINTER(_l)]),
    "qrl_frontend_create": (_i, [_i, _i, _l, _i, C.POINTER(_vp)]),
    "qrl_frontend_destroy": (_i, [_vp]),
    "qrl_frontend_set_stream": (_i, [_vp, _vp]),
    "qrl_frontend_set_carrier_offset": (_i, [_vp, _i, _d]),
    "qrl_frontend_work": (_i, [_vp, _vp, _l, _l, _i, C.POINTER(_l)]),
    "qrl_frontend_out_device": (_i, [_vp, C.POINTER(_vp), C.POINTER(_l), C.POINTER(_l)]),
    "qrl_frontend_read": (_i, [_vp, _vp, _l]),
    "qrl_frontend_launch_count": (_l, [_vp]),
    "qrl_txfront_create": (_i, [_i, _i, _l, _i, C.c_float, _i, C.POINTER(_vp)]),
    "qrl_txfront_destroy": (_i, [_vp]),
    "qrl_txfront_set_stream": (_i, [_vp, _vp]),
    "qrl_txfront_set_carrier_offset": (_i, [_vp, _i, _d]),
    "qrl_txfront_work": (_i, [_vp, _vp, _l, _l, _i, C.POINTER(_l)]),
    "qrl_txfront_out_device": (_i, [_vp, C.POINTER(_vp), C.POINTER(_l), C.POINTER(_l)]),
    "qrl_txfront_read": (_i, [_vp, _vp, _l]),
    "qrl_txfront_launch_count": (_l, [_vp]),
    "qrl_firdes_low_pass": (_i, [_d] * 4 + [_i, _vp, _i]),
    "qrl_firdes_low_pass_2": (_i, [_d] * 5 + [_i, _vp, _i]),
    "qrl_firdes_band_pass": (_i, [_d] * 5 + [_i, _vp, _i]),
    "qrl_firdes_complex_band_pass": (_i, [_d] * 5 + [_i, _vp, _i]),
    "qrl_firdes_root_raised_cosine": (_i, [_d] * 4 + [_i, _vp, _i]),
    "qrl_firdes_gaussian": (_i, [_d] * 3 + [_i, _vp, _i]),
    "qrl_design_table": (_i, [C.c_char_p, _vp, _i]),
    "qrl_design_deemph": (_i, [_i, _d, _vp, _vp]),
    "qrl_fir_decim_ccf_device": (_i, [_vp, _i, _i, _vp, _l, _l, _vp, _l, _i, _vp]),
    "qrl_pfb_create": (_i, [_i, _i, _vp, _i, _l, _i, C.POINTER(_vp)]),
    "qrl_pfb_destroy": (_i, [_vp]),
    "qrl_pfb_set_stream": (_i, [_vp, _vp]),
    "qrl_pfb_work": (_i, [_vp, _vp, _l, _l, _i, C.POINTER(_l)]),
    "qrl_pfb_sync": (_i, [_vp]),
    "qrl_pfb_out_device": (_i, [_vp, C.POINTER(_vp), C.POINTER(_l), C.POINTER(_l)]),
    "qrl_pfb_read": (_i, [_vp, _vp, _l]),
    "qrl_pfb_launch_count": (_l, [_vp]),
    "qrl_deframer_create": (_i, [_i, _i, _i, _i, _l, _i, _i, C.POINTER(_vp)]),
    "qrl_deframer_destroy": (_i, [_vp]),
    "qrl_deframer_set_stream": (_i, [_vp, _vp]),
    "qrl_deframer_work": (_i, [_vp, _vp, _vp, _l, _i]),
    "qrl_deframer_record_bytes": (_i, [_vp]),
    "qrl_deframer_read": (_i, [_vp, _vp, _vp, _vp]),
    "qrl_deframer_out_device": (_i, [_vp, C.POINTER(_vp), C.POINTER(_vp)]),
    "qrl_deframer_sync": (_i, [_vp]),
    "qrl_deframer_launch_count": (_l, [_vp]),
    "qrl_deframer_work2": (_i, [_vp, _vp, _vp, _vp, _vp, _l, _i]),
    "qrl_deframer_dropped": (_i, [_vp, _vp]),
    "qrl_frame_build": (_i, [_i, _vp, _l, _vp, _vp, _i, _i, _vp, _l, _vp, _i, _i, _vp]),
    "qrl_dfbb_create": (_i, [_i, _i, _l, _i, C.POINTER(_vp)]),
    "qrl_dfbb_destroy": (_i, [_vp]),
    "qrl_dfbb_set_stream": (_i, [_vp, _vp]),
    "qrl_dfbb_work": (_i, [_vp, _vp, _vp, _l, _i]),
    "qrl_dfbb_out_device": (_i, [_vp, C.POINTER(_vp), C.POINTER(_l), C.POINTER(_vp)]),
    "qrl_dfbb_read": (_i, [_vp, _vp, _l, _vp]),
    "qrl_dfbb_sync": (_i, [_vp]),
    "qrl_dfbb_launch_count": (_l, [_vp]),
}


def load_library():
    """Load libqrl_b200.so (built in-tree by __graft_entry__.build()).  No fallback of any kind."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(_LIB_PATH):
            raise QrlError("libqrl_b200.so is not built (%s missing): run `python __graft_entry__.py build`; "
                           "qradiolink_b200 has no CPU fallback" % _LIB_PATH)
        L = C.CDLL(_LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)     # AttributeError if the ABI lost a symbol
            fn.restype = res
            fn.argtypes = args
        _LIB = L
    return _LIB


def device_count():
    return load_library().qrl_device_count()


def check(rc, handle=None, what=""):
    if rc != 0:
        msg = load_library().qrl_last_error(handle)
        raise QrlError("%s failed (%d): %s" % (what, rc, (msg or b"").decode()))
