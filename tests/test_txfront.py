"""CPU tier: the TX front end (gr_mod_base.cpp:38,211-290,799-805: rotator_cc at 1 Msps + xN rational_resampler_ccf to the device
rate).  Its definition (tests/txfront_ref.py) -- tap design, impulse response, chunk invariance, spectrum -- and the library's own host
code and kernels, compiled for host threads by tools/emu/build_emulated_lib.py, against that definition bit for bit."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from tests import txfront_ref as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# device rate -> (designed taps, taps per arm): low_pass(N, samp_rate, 480000, 20000, BLACKMAN_HARRIS)
TAPS = {2000000: (419, 210), 5000000: (1045, 209), 10000000: (2091, 210), 20000000: (4181, 210), 56000000: (11709, 210)}


@pytest.mark.parametrize("samp_rate", sorted(TAPS))
def test_definition_taps_match_the_library_design_helper(qrl, oracle, samp_rate):
    N = samp_rate // 1000000
    t = R.TxFrontend(samp_rate)
    assert (t.ntaps, t.arm_taps) == TAPS[samp_rate]
    BH = oracle.WIN_BLACKMAN_HARRIS
    got = np.zeros(1 << 15, np.float32)
    n = qrl.load_library().qrl_firdes_low_pass(float(N), float(samp_rate), 480000.0, 20000.0, BH, got.ctypes.data_as(C.c_void_p), 1 << 15)
    want = oracle.low_pass(N, samp_rate, 480000, 20000, BH)
    assert n == len(want) == t.ntaps
    assert np.array_equal(got[:n].view(np.uint32), want.view(np.uint32))


@pytest.mark.parametrize("samp_rate", [2000000, 5000000, 10000000])
def test_definition_impulse_response_is_the_designed_filter(oracle, samp_rate):
    N = samp_rate // 1000000
    t = R.TxFrontend(samp_rate)
    x = np.zeros(t.arm_taps + 5, np.complex64)
    x[0] = 1.0
    y = t.work(x)
    h = oracle.low_pass(N, samp_rate, 480000, 20000, oracle.WIN_BLACKMAN_HARRIS)
    assert len(y) == N * len(x)
    assert np.array_equal(y.real[:len(h)], h) and not np.any(y.imag) and not np.any(y[len(h):])


def test_definition_rate_set(oracle):
    assert R.TxFrontend(1000000).ntaps == 0
    for bad in (0, 500000, 1500000, 2500000, 57000000, 64000000):
        with pytest.raises(ValueError):
            R.TxFrontend(bad)


def _tone(n, f, amp=0.7, n0=0):
    return (amp * np.exp(2j * np.pi * f * (np.arange(n) + n0) / 1e6)).astype(np.complex64)


@pytest.mark.parametrize("samp_rate", [1000000, 2000000, 5000000])
def test_definition_is_chunk_invariant(oracle, samp_rate):
    rng = np.random.default_rng(samp_rate // 1000000)
    T = 3000
    x = (0.5 * (rng.standard_normal(T) + 1j * rng.standard_normal(T))).astype(np.complex64)
    one = R.TxFrontend(samp_rate)
    one.set_carrier_offset(120000.0)
    a = one.work(x[:1700])
    one.set_carrier_offset(-33333.0)
    want = np.concatenate([a, one.work(x[1700:])])
    many = R.TxFrontend(samp_rate)
    many.set_carrier_offset(120000.0)
    got, lo = [], 0
    for m in [1, 1, 2, 999, 1, 696, 1, 300, 1, 13, 1, 984]:
        if lo == 1700:
            many.set_carrier_offset(-33333.0)
        got.append(many.work(x[lo:lo + m])); lo += m
    assert lo == T
    got = np.concatenate(got)
    assert len(got) == len(want) == T * (samp_rate // 1000000)
    assert np.array_equal(got, want)


@pytest.mark.parametrize("N", [2, 10])
def test_definition_tone_moves_by_the_offset_and_images_are_80_db_down(oracle, N):
    f, o = 50000.0, 100000.0
    t = R.TxFrontend(N * 1000000)
    t.set_carrier_offset(o)
    skip = 2 * t.arm_taps
    y = t.work(_tone(skip + 1000, f))[N * skip:].astype(np.complex128)
    L = len(y)                                        # N * 1000 samples: 1 kHz bins, every frequency below lands on a bin
    X = np.abs(np.fft.fft(y))
    b = int(round((f + o) / 1e6 * 1000))              # bin of f + o
    assert np.argmax(X) == b
    for k in range(-N, N + 1):
        for s in (1, -1):
            img = (k * 1000 + s * b) % L
            if img != b:
                assert 20 * np.log10(X[img] / X[b]) <= -80.0, (k, s, 20 * np.log10(X[img] / X[b]))


@pytest.mark.parametrize("N", [2, 10])
def test_definition_tx_front_end_into_rx_front_end_returns_the_tone(oracle, N):
    f, o = 40000.0, -150000.0
    tx, rx = R.TxFrontend(N * 1000000), oracle.Frontend(N * 1000000)
    tx.set_carrier_offset(o); rx.set_carrier_offset(o)
    y = rx.work(tx.work(_tone(3000, f)))
    assert len(y) == 3000
    z = y[1000:2000].astype(np.complex128)            # 1 ms at 1 Msps, past both filters' transients: 1 kHz bins
    X = np.abs(np.fft.fft(z))
    b = int(round(f / 1e6 * 1000)) % 1000
    assert np.argmax(X) == b
    assert np.max(np.delete(X, b)) / X[b] < 1e-3


def test_cpp_adapter_header_compiles():
    src = '#include "qrl_b200_gr.hpp"\nint main() { qrl_gr::tx_frontend_b200 t(10000000, 2); std::vector<qrl_gr::gr_complex> v; return t.work(nullptr, 0, 0, v); }\n'
    r = subprocess.run(["g++", "-std=c++17", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), "-x", "c++", "-"], input=src, text=True,
                       capture_output=True)
    assert r.returncode == 0, r.stderr


def test_unsupported_rate_is_refused_naming_it(qrl):
    L = qrl.load_library()
    h = C.c_void_p()
    assert L.qrl_txfront_create(1500000, 1, 1024, 0, 32767.0, 0, C.byref(h)) == -22
    assert b"1500000" in L.qrl_last_error(None)
    assert L.qrl_txfront_create(10000000, 1, 1024, 7, 32767.0, 0, C.byref(h)) == -22
    if qrl.device_count() == 0:
        with pytest.raises(qrl.QrlError) as e:
            qrl.TxFrontend(10000000)
        assert "no CUDA device" in str(e.value)


# ---------------------------------------------------------------- the library's own code under emulation (after the tests above:
# the fixture swaps the library for this module until its end)
@pytest.fixture(scope="module")
def emu_qrl(tmp_path_factory):
    sys.path.insert(0, os.path.join(ROOT, "tools", "emu"))
    from build_emulated_lib import build
    lib_path, n_sites = build(str(tmp_path_factory.mktemp("qrl_emu")))
    import qradiolink_b200 as q
    from qradiolink_b200 import lib as L
    saved = (L._LIB_PATH, L._LIB)
    L._LIB_PATH, L._LIB = lib_path, None
    q.load_library()
    assert L.device_count() == 1
    yield q
    L._LIB_PATH, L._LIB = saved


@pytest.mark.timeout(900)
@pytest.mark.parametrize("samp_rate", [1000000, 2000000, 5000000])
@pytest.mark.parametrize("fmt", ["fc32", "sc16"])
def test_library_matches_definition_under_emulation(emu_qrl, oracle, samp_rate, fmt):
    N, Cn, T = samp_rate // 1000000, 2, 2600
    rng = np.random.default_rng(77 + N)
    X = (0.8 * (rng.standard_normal((Cn, T)) + 1j * rng.standard_normal((Cn, T)))).astype(np.complex64)    # peaks clip in sc16
    scale = 32767.0
    txf = emu_qrl.TxFrontend(samp_rate, n_channels=Cn, max_in=1500, out_format=fmt, scale=scale)
    ref = [R.TxFrontend(samp_rate) for _ in range(Cn)]
    txf.set_carrier_offset(90000.0)
    for r in ref:
        r.set_carrier_offset(90000.0)
    lo, clipped = 0, False
    for i, m in enumerate([1500, 1, 333, 13, 753]):
        if i == 3:                                    # per-channel retune in mid-stream
            txf.set_carrier_offset(-210000.0, channel=1); ref[1].set_carrier_offset(-210000.0)
        got = txf.work(X[:, lo:lo + m])
        for c in range(Cn):
            want = ref[c].work(X[c, lo:lo + m])
            if fmt == "sc16":
                want = R.to_sc16(want, scale)
                assert got.dtype == np.int16
                clipped |= bool(np.any(want == 32767) or np.any(want == -32768))
            assert got.shape[1] == len(want) == (m * N if fmt == "fc32" else 2 * m * N), (i, c)
            assert np.array_equal(got[c], want), (i, c)
        lo += m
    assert lo == T and (clipped or fmt == "fc32")
    with pytest.raises(emu_qrl.QrlError) as e:
        txf.work(np.zeros((Cn, 1501), np.complex64))
    assert "(-34)" in str(e.value)
