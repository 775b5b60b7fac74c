"""qradiolink_b200 -- B200-native batched-channel replacement for QRadioLink's per-mode GNU Radio
demod/mod hier-blocks (src/gr/gr_demod_*.cpp, gr_mod_*.cpp).  The arithmetic runs in hand-written
sm_100a CUDA kernels behind the C ABI in include/qrl_b200.h (libqrl_b200.so); this package is the
Python host side: a ctypes binding plus mirrors of the reference's factory functions and sink blocks.

There is no CPU fallback: importing works anywhere (so the CPU test tier can check the ABI), but
creating a demodulator without a CUDA device raises.
"""
from .lib import (QrlError, load_library, device_count, KIND, PARAM)  # noqa: F401
from .demod import (RxBlock, make_gr_demod_4fsk, make_gr_demod_qpsk, make_gr_demod_nbfm,  # noqa: F401
                    make_gr_demod_bpsk, make_gr_demod_2fsk, make_gr_demod_ssb, make_gr_demod_am, make_gr_demod_gmsk, make_gr_demod_wbfm, make_gr_demod_m17, make_gr_demod_dmr, make_gr_demod_dsss,
                    gr_bit_sink, gr_audio_sink, gr_const_sink, gr_sample_sink)
from .mod import TxBlock, make_gr_mod_4fsk, make_gr_mod_qpsk, make_gr_mod_bpsk, make_gr_mod_2fsk, make_gr_mod_nbfm, make_gr_mod_ssb, make_gr_mod_gmsk, make_gr_mod_m17, make_gr_mod_dmr, make_gr_mod_dsss, make_gr_mod_am  # noqa: F401
from .pfb import PfbChannelizer, PfbSynthesizer, mmdvm_port_map  # noqa: F401
from .framing import Deframer, DeframerBB, MODE_FRAMING, SYNC_1K, SYNC_NARROW, SYNC_WIDE, SYNC_M17, frame  # noqa: F401
from .frontend import Frontend, TxFrontend  # noqa: F401
from .spectrum import Spectrum  # noqa: F401
from .mmdvm import MmdvmDemod, MmdvmMod, MmdvmChannelsRx, MmdvmChannelsTx, mmdvm_tag_item  # noqa: F401
