"""GPU tier: TX front end (gr_mod_base.cpp:38,211-290,799-805: rotator_cc at 1 Msps + xN interpolator up to the device rate) against
its definition (tests/txfront_ref.py) bit for bit -- ragged chunks, retunes in mid-stream, sc16 output, device-resident chaining behind the modulator -- and a
loop-back through the RX front end and the 4FSK demodulator, all on the device."""
import ctypes as C

import numpy as np
import pytest

from tests import siggen
from tests import txfront_ref as R

pytestmark = pytest.mark.gpu


def _sync():
    import torch
    torch.cuda.synchronize()


@pytest.mark.parametrize("samp_rate", [1000000, 2000000, 5000000, 10000000, 20000000, 56000000])
def test_txfront_matches_definition(qrl, oracle, samp_rate):
    N, Cn = samp_rate // 1000000, 3
    T = min(300000, 1200000 // N)
    big = T // 3
    rng = np.random.default_rng(N)
    n = np.arange(T)
    X = np.stack([(0.6 * np.exp(2j * np.pi * (20000.0 * (c + 1)) * n / 1e6) + 0.05 * (rng.standard_normal(T) + 1j * rng.standard_normal(T))).astype(np.complex64)
                  for c in range(Cn)])
    txf = qrl.TxFrontend(samp_rate, n_channels=Cn, max_in=big)
    ref = [R.TxFrontend(samp_rate) for _ in range(Cn)]
    lo, i, sizes = 0, 0, [big, 1, 7777, 13, 12345]
    offsets = {1: 150000.0, 3: -200000.0}              # retune before chunks 1 and 3
    while lo < T:
        m = min(sizes[i % len(sizes)], T - lo, big)
        if i in offsets:
            txf.set_carrier_offset(offsets[i])
            for r in ref:
                r.set_carrier_offset(offsets[i])
            if i == 3:
                txf.set_carrier_offset(33000.0, channel=1); ref[1].set_carrier_offset(33000.0)
        got = txf.work(X[:, lo:lo + m])
        for c in range(Cn):
            want = ref[c].work(X[c, lo:lo + m])
            assert got.shape[1] == len(want) == m * N, (i, c, got.shape, len(want))
            assert np.array_equal(got[c], want), (i, c)
        lo += m; i += 1
    assert txf.launches == i * (1 if N == 1 else 2)


@pytest.mark.parametrize("samp_rate,scale", [(1000000, 32767.0), (2000000, 32767.0), (10000000, 20000.5)])
def test_sc16_is_the_rounded_fc32_output(qrl, oracle, samp_rate, scale):
    Cn, T = 2, 200000
    rng = np.random.default_rng(3)
    X = (0.9 * (rng.standard_normal((Cn, T)) + 1j * rng.standard_normal((Cn, T)))).astype(np.complex64)     # peaks clip
    f32 = qrl.TxFrontend(samp_rate, n_channels=Cn, max_in=T)
    s16 = qrl.TxFrontend(samp_rate, n_channels=Cn, max_in=T, out_format="sc16", scale=scale)
    for t in (f32, s16):
        t.set_carrier_offset(-75000.0)
    for lo, hi in ((0, 99999), (99999, T)):
        a, b = f32.work(X[:, lo:hi]), s16.work(X[:, lo:hi])
        want = np.clip(np.rint(a.view(np.float32) * np.float32(scale)), -32768, 32767).astype(np.int16)
        assert b.dtype == np.int16 and np.array_equal(b, want)
        assert np.array_equal(b, R.to_sc16(a, scale))
    assert np.any(want == 32767) and np.any(want == -32768)


def _mod_out_device(tx, data):
    """qrl_tx_work on host bytes, output left on the device: (ptr, stride, items)"""
    L = tx._L
    n = data.shape[1]
    assert L.qrl_tx_work(tx._h, data.ctypes.data_as(C.c_void_p), n, n, 0) == 0
    tx.sync()
    p, s, m = C.c_void_p(), C.c_long(), C.c_long()
    assert L.qrl_tx_out_device(tx._h, C.byref(p), C.byref(s), C.byref(m)) == 0
    return p.value, s.value, m.value


def _frames(Cn, nframes, seed):
    streams, payloads = [], []
    for c in range(Cn):
        d, pl = siggen.frames_4fsk(np.random.default_rng(seed + c), nframes)
        streams.append(d); payloads.append(pl)
    n = max(len(d) for d in streams)
    data = np.full((Cn, n), 0xAA, np.uint8)
    for c, d in enumerate(streams):
        data[c, :len(d)] = d
    return data, payloads


def test_chained_behind_the_modulator_on_device(qrl):
    Cn = 2
    data, _ = _frames(Cn, 6, 4100)
    n = data.shape[1]
    tx = qrl.make_gr_mod_4fsk(25, 1000000, 1700, 3500, True, n_channels=Cn, max_items=n)
    iq = qrl.make_gr_mod_4fsk(25, 1000000, 1700, 3500, True, n_channels=Cn, max_items=n).work(data)
    ptr, stride, items = _mod_out_device(tx, data)
    assert items == iq.shape[1]
    dev = qrl.TxFrontend(5000000, n_channels=Cn, max_in=items)
    host = qrl.TxFrontend(5000000, n_channels=Cn, max_in=items)
    for t in (dev, host):
        t.set_carrier_offset(120000.0)
    assert dev.work_device(ptr, items, stride) == 5 * items
    got = dev.read(5 * items)
    assert np.array_equal(got, host.work(iq))


def test_loopback_through_rx_front_end_and_demodulator(qrl, oracle):
    """4FSK TX -> TX front end (10 Msps, +150 / -200 kHz) -> RX front end (10 Msps, same offsets) -> 4FSK RX, device-resident from
    the modulator's output on: every frame comes back, and the bits are those of the same chain through the oracle."""
    Cn, rate, offs = 2, 10000000, (150000.0, -200000.0)
    data, payloads = _frames(Cn, 20, 7000)
    n = data.shape[1]
    tx = qrl.make_gr_mod_4fsk(25, 1000000, 1700, 3500, True, n_channels=Cn, max_items=n)
    ptr, stride, items = _mod_out_device(tx, data)
    txf = qrl.TxFrontend(rate, n_channels=Cn, max_in=items)
    fe = qrl.Frontend(rate, n_channels=Cn, max_in=10 * items)
    for c, o in enumerate(offs):
        txf.set_carrier_offset(o, channel=c); fe.set_carrier_offset(o, channel=c)
    assert txf.work_device(ptr, items, stride) == 10 * items
    _sync()
    p2, s2, n2 = txf.out_device()
    assert fe.work_device(p2, n2, s2) == items
    _sync()
    p3, s3, n3 = fe.out_device()
    rx = qrl.make_gr_demod_4fsk(5, 1000000, 1700, 3000, True, n_channels=Cn, max_samples=n3)
    rx.work_device(p3, n3, s3)
    bits = rx.read_port(2)
    for c in range(Cn):
        good, found = siggen.count_good_frames(bits[c], 0xED89AA, 24, 7, payloads[c])
        assert good >= len(payloads[c]) - 4 and found - good <= 1, (c, good, found)
        x = oracle.Tx(oracle.MOD_4FSK, 25, 1000000, 1700, 3500, 1).work(data[c])
        t, f = R.TxFrontend(rate), oracle.Frontend(rate)
        t.set_carrier_offset(offs[c]); f.set_carrier_offset(offs[c])
        r = oracle.Rx(oracle.DEMOD_4FSK, 5, 1000000, 1700, 3000, 1)
        r.work(f.work(t.work(x)))
        assert np.array_equal(bits[c], r.port(2)), c


def test_error_paths(qrl):
    for bad in (1500000, 57000000, 0):
        with pytest.raises(qrl.QrlError) as e:
            qrl.TxFrontend(bad)
        assert "(-22)" in str(e.value) and str(bad) in str(e.value)
    txf = qrl.TxFrontend(2000000, n_channels=2, max_in=100)
    with pytest.raises(qrl.QrlError) as e:
        txf.work(np.zeros((2, 101), np.complex64))
    assert "(-34)" in str(e.value)
    with pytest.raises(qrl.QrlError):
        txf.set_carrier_offset(1000.0, channel=2)
