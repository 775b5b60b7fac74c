"""CPU tier: pin the ORACLE itself (the known-answer tests the reference never had, SURVEY.md section 4 / 8c)."""
import json
import os

import numpy as np
import pytest
import scipy.signal as ss

from tests import siggen

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_tap_counts_match_survey(oracle):
    O = oracle; BH = O.WIN_BLACKMAN_HARRIS
    assert len(O.low_pass(1, 1e6, 10000, 10000, BH)) == 419          # /50 decimator (nbfm, 4fsk, bpsk)
    assert len(O.low_pass(1, 20000, 3000, 1500, BH)) == 55           # 4FSK-FM channel filter
    assert len(O.low_pass(1, 20000, 4000, 2000, BH)) == 41
    assert len(O.low_pass_2(1, 1e6, 250000, 50000, 60, BH)) == 55    # QPSK-250k /2
    assert len(O.rrc(2, 2, 1, 0.35, 22)) == 23
    assert len(O.low_pass_2(1, 20000, 2500, 3500, 60, BH)) == 15     # nbfm channel filter
    assert len(O.low_pass_2(2, 40000, 3600, 250, 60, BH)) == 437
    assert len(O.low_pass_2(1, 8000, 3500, 200, 35, BH)) == 63
    assert len(O.low_pass(1, 20000, 2000, 100, BH)) == 837
    assert len(O.low_pass(1, 1e6, 4000, 4000, BH)) == 1045           # ssb /125
    assert len(O.low_pass(20, 1e6, 3500, 3500, O.WIN_HAMMING)) == 689


def test_firdes_closed_forms(oracle):
    O = oracle
    h = O.low_pass(1, 1e6, 10000, 10000, O.WIN_BLACKMAN_HARRIS).astype(np.float64)
    assert abs(h.sum() - 1.0) < 1e-6 and np.allclose(h, h[::-1], atol=1e-9)
    # same design via scipy's window + ideal sinc
    n = np.arange(419) - 209
    w = ss.get_window(("blackmanharris"), 419, fftbins=False)
    ideal = np.sinc(2 * 10000 / 1e6 * n) * (2 * 10000 / 1e6) * w
    ideal /= ideal.sum()
    assert np.max(np.abs(ideal - h)) < 2e-7
    hh = O.low_pass(20, 1e6, 3500, 3500, O.WIN_HAMMING).astype(np.float64)
    assert abs(hh.sum() - 20.0) < 1e-4
    r = O.rrc(1.5, 20000, 2000, 0.2, 251).astype(np.float64)
    assert abs(r.sum() - 1.5) < 1e-5 and np.argmax(r) == 125
    # RRC * RRC ~ Nyquist: zero ISI at multiples of the symbol period (10 samples)
    rc = np.convolve(r, r); mid = len(rc) // 2
    isi = np.abs(rc[mid + 10::10]) / rc[mid]
    assert isi.max() < 2e-2
    cb = O.complex_band_pass(1, 20000, -4000, -2000, 4000, O.WIN_BLACKMAN_HARRIS)
    H = np.abs(np.fft.fft(cb, 4096)); f = np.fft.fftfreq(4096, 1 / 20000)
    assert abs(f[np.argmax(H)] - (-3000)) < 100


def test_mmse_table_matches_upstream_rows(oracle):
    t = oracle.table("mmse").reshape(129, 8)
    assert np.array_equal(t[0], [0, 0, 0, 0, 1, 0, 0, 0]) and np.array_equal(t[128], [0, 0, 0, 1, 0, 0, 0, 0])
    # rows 1/128 and 2/128 of gnuradio's interpolator_taps.h
    row1 = [-1.54700e-04, 8.53777e-04, -2.76968e-03, 7.89295e-03, 9.98534e-01, -5.41054e-03, 1.24642e-03, -1.98993e-04]
    row2 = [-3.09412e-04, 1.70888e-03, -5.55134e-03, 1.58840e-02, 9.96891e-01, -1.07209e-02, 2.47942e-03, -3.96391e-04]
    assert np.max(np.abs(t[1] - np.float32(row1))) < 2e-6
    assert np.max(np.abs(t[2] - np.float32(row2))) < 2e-6
    assert np.allclose(t.sum(axis=1), 1.0, atol=2e-3)
    assert np.allclose(t[64], t[64][::-1], atol=1e-6)      # mu = 0.5 is symmetric


def test_sincos_and_atan(oracle):
    x = np.linspace(-7, 7, 2001).astype(np.float32)
    s, c = oracle.sincosf(x)
    assert np.max(np.abs(s - np.sin(x.astype(np.float64)))) < 3e-7
    assert np.max(np.abs(c - np.cos(x.astype(np.float64)))) < 3e-7
    L = oracle.lib()
    rng = np.random.default_rng(0)
    xy = rng.standard_normal((2000, 2)).astype(np.float32)
    got = np.array([L.qo_fast_atan2f(float(y), float(x_)) for x_, y in xy])
    assert np.max(np.abs(got - np.arctan2(xy[:, 1], xy[:, 0]))) < 2e-4   # gr::fast_atan2f accuracy
    assert L.qo_fast_atan2f(0.0, 0.0) == 0.0


def test_deemph_taps_against_compiled_reference(oracle):
    """The taps of the reference's src/gr/emphasis.cpp compiled as-is (the only stand-alone piece, oracle/_ref), as frozen in
    tests/golden/golden_v1.json by tests/golden/make_golden.py."""
    G = json.load(open(os.path.join(ROOT, "tests", "golden", "golden_v1.json")))["emphasis"]
    for fs, tau in ((20000, 50e-6), (8000, 50e-6), (48000, 75e-6)):
        a, b = np.array([float.fromhex(v) for v in G["deemph_%d_%g" % (fs, tau)]]).reshape(2, 2)
        oa, ob = oracle.deemph_taps(fs, tau)
        assert np.array_equal(a, oa) and np.array_equal(b, ob)
        a, b = np.array([float.fromhex(v) for v in G["preemph_%d_%g" % (fs, tau)]]).reshape(2, 2)
        oa, ob = oracle.preemph_taps(fs, tau)
        assert np.array_equal(a, oa) and np.array_equal(b, ob)


def test_fir_orders_and_scipy(oracle):
    O = oracle
    rng = np.random.default_rng(3)
    h = O.low_pass(1, 1e6, 10000, 10000, O.WIN_BLACKMAN_HARRIS)
    x = (rng.standard_normal(20000) + 1j * rng.standard_normal(20000)).astype(np.complex64)
    y = O.fir_decim_ccf(h, 50, x)
    ref = ss.upfirdn(h.astype(np.float64), x.astype(np.complex128), 1, 50)[: len(y)]
    assert len(y) == 400 and np.max(np.abs(y - ref)) < 5e-6
    O.lib().qo_set_fir_order(1)
    y_seq = O.fir_decim_ccf(h, 50, x)
    O.lib().qo_set_fir_order(0)
    rms = np.sqrt(np.mean(np.abs(y - y_seq) ** 2)) / np.sqrt(np.mean(np.abs(y_seq) ** 2))
    assert rms < 1e-6          # the parity order vs plain sequential order: far inside the 1e-5 RMS budget
    # interpolating arm structure (rational_resampler_fff(25,1))
    r = O.rrc(25, 25, 1, 0.2, 250)
    sym = rng.choice([-1.5, -0.5, 0.5, 1.5], 200).astype(np.float32)
    yi = O.fir_fff(r, 25, 1, sym)
    refi = ss.upfirdn(r.astype(np.float64), sym.astype(np.float64), 25, 1)[: len(yi)]
    assert len(yi) == 5000 and np.max(np.abs(yi - refi)) < 1e-5
    # 2/5 audio resampler
    a = O.low_pass_2(2, 40000, 3600, 250, 60, O.WIN_BLACKMAN_HARRIS)
    xa = rng.standard_normal(5000).astype(np.float32)
    ya = O.fir_fff(a, 2, 5, xa)
    refa = ss.upfirdn(a.astype(np.float64), xa.astype(np.float64), 2, 5)[: len(ya)]
    assert len(ya) == 2000 and np.max(np.abs(ya - refa)) < 1e-5


def test_fec_and_lfsr_inverses(oracle):
    O = oracle
    rng = np.random.default_rng(7)
    bits = rng.integers(0, 2, 80 * 40, dtype=np.uint8)
    assert np.array_equal(O.descramble(O.scramble(bits))[8:], bits[:-8])        # 8-bit scrambler latency
    coded = O.cc_encode(bits)
    assert len(coded) == 2 * len(bits)
    # CCSDS generator check: impulse response of {109, 79}
    imp = O.cc_encode(np.array([1, 0, 0, 0, 0, 0, 0], np.uint8)).reshape(-1, 2)
    assert [int(b) for b in imp[:, 0]] == [1, 0, 1, 1, 0, 1, 1] and [int(b) for b in imp[:, 1]] == [1, 1, 1, 1, 0, 0, 1]
    soft = np.where(coded > 0, 255, 0).astype(np.uint8)
    dec = O.cc_decode(soft)
    assert len(dec) == len(bits) - 80 + 80 - 80 or len(dec) % 80 == 0
    assert np.array_equal(dec[6:], bits[: len(dec) - 6])                        # 6-bit decoder latency
    # 3 % channel errors are corrected
    flip = rng.random(len(soft)) < 0.03
    dec2 = O.cc_decode(np.where(flip, 255 - soft, soft).astype(np.uint8))
    assert np.mean(dec2[6:] != bits[: len(dec2) - 6]) < 1e-3


def test_4fsk_loopback_recovers_frames(oracle):
    X, payloads = siggen.gen_4fsk_channels(2, 1 << 20, seed0=1000, snr_db=20.0)
    for c in range(2):
        rx = oracle.Rx(oracle.DEMOD_4FSK, 5, 1000000, 1700, 3000, 1)
        rx.work(X[c])
        good, found = siggen.count_good_frames(rx.port(2), 0xED89AA, 24, 7, payloads[c])
        assert good >= len(payloads[c]) - 4 and found - good <= 1   # first frames fall into clock acquisition


def test_qpsk_loopback_recovers_frames(oracle):
    X, payloads = siggen.gen_qpsk_channels(1, 1 << 18, seed0=2000, snr_db=15.0)
    rx = oracle.Rx(oracle.DEMOD_QPSK, 2, 1000000, 1700, 160000, 0)
    rx.work(X[0])
    good, found = siggen.count_good_frames(rx.port(2), 0xDE98AA, 24, 1516, payloads[0])
    assert good == len(payloads[0]) and good >= 3


def test_chunk_invariance(oracle):
    X, _ = siggen.gen_4fsk_channels(1, 300000, seed0=1234)
    a = oracle.Rx(oracle.DEMOD_4FSK, 5, 1000000, 1700, 3000, 1)
    a.work(X[0])
    b = oracle.Rx(oracle.DEMOD_4FSK, 5, 1000000, 1700, 3000, 1)
    for lo in range(0, 300000, 33333):
        b.work(X[0][lo:lo + 33333])
    for p in (0, 1, 2):
        pa, pb = a.port(p), b.port(p)
        n = min(len(pa), len(pb))
        assert n > 0 and abs(len(pa) - len(pb)) <= 160
        assert np.array_equal(pa[:n], pb[:n])


def test_nbfm_tone(oracle):
    """FM-modulate a 1 kHz tone (numpy) and check the NBFM chain returns a 1 kHz tone at 8 ksps."""
    fs = 1e6; n = np.arange(400000)
    dev = 2000.0
    phase = 2 * np.pi * dev / (2 * np.pi * 1000.0) * np.sin(2 * np.pi * 1000.0 * n / fs)
    x = (0.8 * np.exp(1j * phase)).astype(np.complex64)
    rx = oracle.Rx(oracle.DEMOD_NBFM, 125, 1000000, 1700, 2500, 0)
    rx.work(x)
    audio = rx.port(1)
    assert 3000 < len(audio) <= 3200
    seg = audio[1000:3000].astype(np.float64)
    spec = np.abs(np.fft.rfft(seg * np.hanning(len(seg))))
    f = np.fft.rfftfreq(len(seg), 1 / 8000.0)
    assert abs(f[np.argmax(spec)] - 1000.0) < 10.0
    assert 0.2 < np.std(seg) < 3.0


def test_pfb_channelizer_and_synthesizer_against_float64(oracle):
    """SURVEY 8f row 1: the oracle's polyphase channelizer / synthesizer against an independent float64 statement
    (branch convolution with scipy-free numpy + np.fft), chunk invariance, and the loop-back convention."""
    O = oracle
    M = 10
    taps = O.low_pass_2(1, 250000, 5000, 2000, 60, O.WIN_BLACKMAN_HARRIS)
    assert len(taps) == 341                                   # the reference's prototype (gr_demod_mmdvm_multi2.cpp:56)
    rng = np.random.default_rng(5)
    x = ((rng.standard_normal(4003) + 1j * rng.standard_normal(4003)) * 0.3).astype(np.complex64)
    y = O.PfbChannelizer(M, taps).work(x)
    tpf = (len(taps) + M - 1) // M
    hp = np.zeros(tpf * M); hp[:len(taps)] = taps
    xs = np.concatenate([np.zeros(tpf * M), x.astype(np.complex128)])
    frames = len(x) // M
    u = np.zeros((frames, M), np.complex128)
    for k in range(M):
        s = xs[tpf * M + (M - 1 - k) - (tpf - 1) * M:][::M]   # stream M-1-k with tpf-1 samples of history in front
        u[:, k] = np.convolve(s, hp[k::M])[tpf - 1:tpf - 1 + frames]
    ref = (np.fft.ifft(u, axis=1) * M).T                      # sum_k u_k exp(+j 2 pi k c / M)
    assert y.shape == ref.shape
    assert np.max(np.abs(y - ref)) < 2e-6
    parts = O.PfbChannelizer(M, taps)
    y2 = np.concatenate([parts.work(x[a:b]) for a, b in ((0, 7), (7, 1234), (1234, 1235), (1235, len(x)))], axis=1)
    assert np.array_equal(y, y2)
    # synthesizer: float64 statement of y[nM + i] = sum_t taps[i + tM] v_i[n - t], v = M * ifft(in)
    st = O.low_pass_2(10, 250000, 5000, 2000, 60, O.WIN_BLACKMAN_HARRIS)
    z = ((rng.standard_normal((M, 300)) + 1j * rng.standard_normal((M, 300))) * 0.3).astype(np.complex64)
    w = O.PfbSynthesizer(M, st).work(z)
    sp = np.zeros(tpf * M); sp[:len(st)] = st
    v = np.fft.ifft(z.astype(np.complex128), axis=0) * M
    refw = np.zeros(300 * M, np.complex128)
    for i in range(M):
        refw[i::M] = np.convolve(v[i], sp[i::M])[:300]
    assert np.max(np.abs(w - refw)) < 2e-5
    s2 = O.PfbSynthesizer(M, st)
    assert np.array_equal(w, np.concatenate([s2.work(z[:, :17]), s2.work(z[:, 17:])]))
    # loop-back convention: a channel fed to synthesizer port c comes back on channelizer port c
    zz = np.zeros((M, 800), np.complex64); zz[3] = 1.0; zz[9] = 0.5
    back = O.PfbChannelizer(M, taps).work(O.PfbSynthesizer(M, st).work(zz))
    p = np.abs(back[:, -1])
    assert abs(p[3] - 1.0) < 0.02 and abs(p[9] - 0.5) < 0.02 and np.all(np.delete(p, [3, 9]) < 0.02)


def test_deframer_known_answers(oracle):
    """gr_modem::synchronize / findSync restated (SURVEY 8f row 2): planted frames come back with type and payload,
    non-voice frames take 8 bits less, the register is cleared after a frame, chunking is invisible."""
    O = oracle
    rng = np.random.default_rng(1)
    bits_of = lambda bs: np.unpackbits(np.frombuffer(bytes(bs), np.uint8))  # noqa: E731
    pl = [rng.integers(0, 256, 7, dtype=np.uint8).tobytes() for _ in range(5)]
    text = rng.integers(0, 256, 7, dtype=np.uint8).tobytes()
    parts = [bits_of([0xAA] * 8)]
    for p in pl:
        parts.append(bits_of([0xED, 0x89, 0xAA] + list(p)))
    parts.append(bits_of([0x89, 0xED, 0xAA] + list(text)))
    parts.append(bits_of([0x4C, 0x8A, 0x2B] + [0] * 7))
    b = np.concatenate(parts)
    fr = O.Deframer(2, 64, 7).work(b)
    assert [t for t, _ in fr] == [0xED89] * 5 + [0x89EDAA, 0x4C8A2B]
    assert [p for _, p in fr[:5]] == [bytes([0xAA]) + p for p in pl]        # reserved byte + 7 payload bytes
    assert fr[5][1] == text and len(fr[6][1]) == 7
    d2 = O.Deframer(2, 64, 7)
    fr2 = []
    for a in range(0, len(b), 37):
        fr2 += d2.work(b[a:a + 37])
    assert fr2 == fr
    # voice payloads agree with the plain sync search used elsewhere in the tests
    ff = O.find_frames(b, 0xED89AA, 24, 7)
    assert [f.tobytes() for f in ff][:5] == pl
    # class 1: 8-bit sync, 4-byte frames; a sync word inside a frame is not a sync
    b1 = np.concatenate([bits_of([0x00, 0xB5, 0xB5, 1, 2, 3]), bits_of([0xB5, 9, 8, 7, 6])])
    assert O.Deframer(1, 32, 4).work(b1) == [(0xB5, bytes([0xB5, 1, 2, 3])), (0xB5, bytes([9, 8, 7, 6]))]


def test_rssi_block_known_answers(oracle):
    """rssi_block.cpp:25-45 restated: a constant-envelope tone of amplitude a settles at 10 log10(2000 a^2); chunking is
    invisible; silence reports the nlog10 floor."""
    n = np.arange(30000)
    x = (0.1 * np.exp(2j * np.pi * 0.01 * n)).astype(np.complex64)
    r = oracle.Rssi(0.0)
    v = r.work(x)
    assert abs(v - 10 * np.log10(2000 * 0.01)) < 1e-3
    r2 = oracle.Rssi(0.0)
    for a in range(0, len(x), 777):
        v2 = r2.work(x[a:a + 777])
    assert v2 == v
    assert oracle.Rssi(-10.0).work(np.zeros(100, np.complex64)) == pytest.approx(-190.0, abs=1e-3)


def test_am_and_gmsk_chains_run_and_stream(oracle):
    """The AM and GMSK receive chains (SURVEY 8f row 3) are chunk-size invariant in the oracle, AM audio carries the tone."""
    O = oracle
    T = 1 << 17
    n = np.arange(T)
    aud = 0.5 * np.sin(2 * np.pi * 1000.0 * n / 1e6)
    x = (0.4 * (1.0 + 0.8 * aud) * np.exp(2j * np.pi * 200.0 * n / 1e6)).astype(np.complex64)
    a = O.Rx(O.DEMOD_AM, 125, 1000000, 1700, 5000, 0); a.work(x)
    b = O.Rx(O.DEMOD_AM, 125, 1000000, 1700, 5000, 0)
    for lo in range(0, T, 30011):
        b.work(x[lo:lo + 30011])
    for p in range(2):
        assert np.array_equal(a.port(p, clear=False), b.port(p, clear=False))
    audio = a.port(1)
    assert len(audio) == pytest.approx(T / 125, abs=40) and np.std(audio[300:]) > 0.05
    rng = np.random.default_rng(2)
    y = ((rng.standard_normal(T) + 1j * rng.standard_normal(T)) * 0.1).astype(np.complex64)
    g = O.Rx(O.DEMOD_GMSK, 5, 1000000, 1700, 4000, 0); g.work(y)
    g2 = O.Rx(O.DEMOD_GMSK, 5, 1000000, 1700, 4000, 0)
    for lo in range(0, T, 12345):
        g2.work(y[lo:lo + 12345])
    for p in range(4):
        assert np.array_equal(g.port(p, clear=False), g2.port(p, clear=False))
    assert len(g.port(2)) > 50


def test_gmsk_modem_loops_back_in_the_oracle(oracle):
    """gr_mod_gmsk -> channel -> gr_demod_gmsk (GMSK2K instances): every transmitted voice frame is recovered by one of the
    two decoders (the second sits behind delay(1)); ties the two restatements to each other physically."""
    O = oracle
    from tests import siggen
    rng = np.random.default_rng(5)
    data, pl = siggen.frames_4fsk(rng, 8)
    iq = O.Tx(O.MOD_GMSK, 50, 1000000, 1700, 4000, 0).work(data)
    assert len(iq) == len(data) * 16 * 50 * 5
    x = siggen.channel(iq, rng, fo_hz=30, phase=0.4, delay=123, snr_db=25, amp=0.5, total=len(iq) + 20000)
    rx = O.Rx(O.DEMOD_GMSK, 5, 1000000, 1700, 4000, 0)
    rx.work(x)
    good = max(siggen.count_good_frames(rx.port(p), 0xED89AA, 24, 7, pl)[0] for p in (2, 3))
    assert good == len(pl)


def test_wbfm_chain_streams_and_recovers_the_tone(oracle):
    O = oracle
    T = 1 << 17
    n = np.arange(T)
    x = (0.5 * np.exp(1j * 2 * np.pi * 40000.0 * np.cumsum(np.sin(2 * np.pi * 1000.0 * n / 1e6)) / 1e6)).astype(np.complex64)
    a = O.Rx(O.DEMOD_WBFM, 125, 1000000, 1700, 75000, 0); a.work(x)
    b = O.Rx(O.DEMOD_WBFM, 125, 1000000, 1700, 75000, 0)
    for lo in range(0, T, 23456):
        b.work(x[lo:lo + 23456])
    for p in range(2):
        assert np.array_equal(a.port(p, clear=False), b.port(p, clear=False))
    assert len(a.port(0, clear=False)) == (T + 4) // 5
    audio = a.port(1)
    f = np.abs(np.fft.rfft(audio[100:] * np.hanning(len(audio) - 100)))
    assert abs(np.argmax(f) * 8000.0 / (len(audio) - 100) - 1000.0) < 20.0


def test_m17_chain_streams(oracle):
    """gr_demod_m17 restated (x3/125 to 24 ksps, 4FSK, hard bits): chunk-size invariant, 2 bits per symbol, 3/125 of the input rate."""
    O = oracle
    from tests.golden import cases
    x = cases._sig_m17(O, None)[0][:200000]
    a = O.Rx(O.DEMOD_M17, 125, 1000000, 1700, 9000, 0); a.work(x)
    b = O.Rx(O.DEMOD_M17, 125, 1000000, 1700, 9000, 0)
    for lo in range(0, len(x), 33331):
        b.work(x[lo:lo + 33331])
    for p in range(3):
        assert np.array_equal(a.port(p, clear=False), b.port(p, clear=False))
    assert len(a.port(0, clear=False)) == (len(x) * 3 + 124) // 125
    assert len(a.port(2, clear=False)) == 2 * len(a.port(1, clear=False))


def test_m17_modem_loops_back_in_the_oracle(oracle):
    """gr_mod_m17 -> channel -> gr_demod_m17 restated: after acquisition the hard bits of port 2 are the transmitted bits (the
    TX map {2,3,1,0} and the RX map {3,1,2,0} are inverse through the phase modulator / slicer pair)."""
    O = oracle
    from tests import siggen
    rng = np.random.default_rng(4)
    data = rng.integers(0, 256, 300, dtype=np.uint8)
    iq = O.Tx(O.MOD_M17, 125, 1000000, 1700, 9000, 0).work(data)
    assert len(iq) == len(data) * 4 * 5 * 125 // 3
    x = siggen.channel(iq, rng, fo_hz=40, phase=0.3, delay=211, snr_db=30, amp=0.5, total=len(iq) + 30000)
    rx = O.Rx(O.DEMOD_M17, 125, 1000000, 1700, 9000, 0)
    rx.work(x)
    bits, tx_bits = rx.port(2), np.unpackbits(data)
    best = 0.0
    for off in range(60, 160):                        # demodulator latency in bits; the last ~60 bits ride on the filter tails
        n = min(len(bits) - off, len(tx_bits)) - 100
        best = max(best, float(np.mean(bits[off:off + n] == tx_bits[:n])))
    assert best == 1.0


def test_dmr_chain_streams_and_locks(oracle):
    """gr_demod_dmr restated (oracle only so far: x3/125 to 24 ksps, RRC 0.2, symbol_sync_ff with the PLAIN Mueller & Mueller TED,
    float port 3): chunk-size invariant, and -- fed the M17 modulator's 4FSK burst, same symbol rate and maps -- its timing
    loop locks and the hard bits follow the transmitted ones (the 0.5 vs 0.2 roll-off mismatch leaves a little ISI)."""
    O = oracle
    from tests import siggen
    rng = np.random.default_rng(4)
    data = rng.integers(0, 256, 300, dtype=np.uint8)
    iq = O.Tx(O.MOD_M17, 125, 1000000, 1700, 9000, 0).work(data)
    x = siggen.channel(iq, rng, fo_hz=40, phase=0.3, delay=211, snr_db=30, amp=0.5, total=len(iq) + 30000)
    a = O.Rx(O.DEMOD_DMR, 5, 1000000, 0, 0, 0); a.work(x)
    b = O.Rx(O.DEMOD_DMR, 5, 1000000, 0, 0, 0)
    for lo in range(0, len(x), 33331):
        b.work(x[lo:lo + 33331])
    for p in range(4):
        assert np.array_equal(a.port(p, clear=False), b.port(p, clear=False))
    assert a.port(3, clear=False).dtype == np.float32
    assert len(a.port(0, clear=False)) == len(a.port(3, clear=False)) == (len(x) * 3 + 124) // 125
    assert len(a.port(2, clear=False)) == 2 * len(a.port(1, clear=False))
    bits, tx_bits = a.port(2), np.unpackbits(data)
    best = 0.0
    for off in range(40, 200):
        n = min(len(bits) - off, len(tx_bits)) - 100
        best = max(best, float(np.mean(bits[off:off + n] == tx_bits[:n])))
    assert best > 0.97


def test_frame_and_m17_deframer_restatements(oracle):
    """gr_modem::frame (gr_modem.cpp:904-961) and the M17 branch of findSync (:1187-1207), oracle level: known answers."""
    O = oracle
    assert bytes(O.frame(b"\x01\x02", 0xED89)) == b"\xED\x89\xAA\x01\x02"
    assert bytes(O.frame(b"\x01\x02", 0xED89, one_k_mode=True)) == b"\xB5\x01\x02"
    assert bytes(O.frame(b"\x07", 0xDE98AA, burst_ip=True)) == b"\xAA" * 10 + b"\xDE\x98\xAA\x07"
    assert bytes(O.frame(b"\x07", 0xDE98AA)) == b"\xDE\x98\xAA\x07"
    assert bytes(O.frame(b"\x09", 0x8CC8DD)) == b"\x09"                      # callsign / end frames get no sync word from frame()
    rng = np.random.default_rng(5)
    payload = rng.integers(0, 256, 7, dtype=np.uint8).tobytes()
    bits = np.unpackbits(np.concatenate([np.full(3, 0xAA, np.uint8), O.frame(payload, 0xED89), np.full(4, 0xAA, np.uint8)]))
    fr = O.Deframer(2, 64, 7).work(bits)
    assert fr == [(0xED89, b"\xAA" + payload)]
    m17 = np.unpackbits(np.array([0x00, 0x55, 0xF7] + list(range(46)) + [0x55, 0x5D, 0x55, 0x5D] + [0xFF] * 46, np.uint8))
    fr = O.Deframer(4, 46 * 8, 46).work(m17)
    assert [t for t, _ in fr] == [0x55F7, 0x555D555D] and fr[0][1] == bytes(range(46)) and fr[1][1] == b"\xFF" * 46


def test_dmr_modulator_restatement(oracle):
    """gr_mod_dmr restated (gr_mod_dmr.cpp:27-93): chunk invariant incl. the "zero_samples" tags, 125/3 output items per 24 ksps
    item, the gr_zero_idle_bursts history shows as 1439 items (60 ms) of silence in front, a tag clears exactly its count `delay`
    items before the tagged byte's first item, and the burst loops back through the restated DMR receiver (same pulse, 0.2)."""
    O = oracle
    from tests import siggen
    rng = np.random.default_rng(41)
    data = rng.integers(0, 256, 400, dtype=np.uint8)
    a = O.Tx(O.MOD_DMR, 125, 1000000, 1700, 5000, 0)
    a.zero_samples(100, 720); a.zero_samples(110, 100); a.zero_samples(1, 50); a.zero_samples(300, 333)
    ya = a.work(data)
    assert len(ya) == (len(data) * 20 * 125 + 2) // 3
    b = O.Tx(O.MOD_DMR, 125, 1000000, 1700, 5000, 0)
    b.zero_samples(100, 720); b.zero_samples(110, 100); b.zero_samples(1, 50); b.zero_samples(300, 333)
    yb = np.concatenate([b.work(data[lo:lo + 37]) for lo in range(0, len(data), 37)])
    assert np.array_equal(ya.view(np.uint32), yb.view(np.uint32))
    # where the 24 ksps stream is zero, the x125/3 interpolator's output is zero once its 33-tap arms are flushed
    up = 125 / 3
    head = int(1439 * up) - 10
    assert np.all(ya[:head] == 0) and np.any(ya[head + 40 * 42:head + 80 * 42] != 0)
    s0, s1 = 100 * 20 - 62, 110 * 20 - 62                    # tag 2 overrides tag 1: zero [s0, s1) then [s1, s1 + 100)
    z = np.abs(ya[int((s0 + 40) * up):int((s1 + 100 - 5) * up)])
    assert np.all(z == 0)
    assert np.all(np.abs(ya[int((s1 + 100 + 40) * up):int((s1 + 100 + 300) * up)]) > 0.5)
    assert np.all(np.abs(ya[int((1439 + 40) * up):int((1439 + 200) * up)]) > 0.5)      # the tag on byte 1 (item 20 < delay) is ignored
    # loop-back: no tags
    iq = O.Tx(O.MOD_DMR, 125, 1000000, 1700, 5000, 0).work(data)
    x = siggen.channel(iq, rng, fo_hz=30, phase=0.2, delay=97, snr_db=30, amp=0.5, total=len(iq) + 30000)
    rx = O.Rx(O.DEMOD_DMR, 5, 1000000, 0, 0, 0)
    rx.work(x)
    bits, tx_bits = rx.port(2), np.unpackbits(data)
    best = 0.0
    for off in range(2 * 1439 // 5 - 200, 2 * 1439 // 5 + 400):
        n = min(len(bits) - off, len(tx_bits)) - 900           # the last 1439 items (576 bits) are still in the zero-idle delay line, filter tails
        if n > 1000:
            best = max(best, float(np.mean(bits[off + 200:off + n] == tx_bits[200:n])))       # first 200 bits: loops pulling in
    assert best == 1.0, best


def test_spectrum_restatement_against_numpy(oracle):
    """The oracle's display spectrum (rx_fft_c restated) against an independent float64 statement: window x fft -> 10 log10 |X / N|^2,
    fft-shifted; the trigger sits at the first sample AFTER the buffer filled."""
    O = oracle
    rng = np.random.default_rng(62)
    N = 4096
    x = (rng.standard_normal(3 * N) + 1j * rng.standard_normal(3 * N)).astype(np.complex64) * 0.2
    s = O.Spectrum(N, O.WIN_BLACKMAN_HARRIS)
    s.set_enabled(True)
    s.work(x[:N]); assert s.get() is None                       # full, but the FFT runs with the next sample
    s.work(x[N:N + 1])
    g = s.get()
    w = np.empty(N, np.float32); O.lib().qo_window_build(O.WIN_BLACKMAN_HARRIS, N, w.ctypes.data_as(__import__("ctypes").c_void_p))
    X = np.fft.fft((x[:N] * w).astype(np.complex64).astype(np.complex128)) / N
    want = np.fft.fftshift(10 * np.log10(np.abs(X) ** 2))
    assert np.max(np.abs(g - want)) < 2e-4


def test_dsss_modem_loops_back_in_the_oracle(oracle):
    """gr_mod_dsss -> channel -> gr_demod_dsss restated (gr_mod_dsss.cpp:27-93, gr_demod_dsss.cpp:32-124; 8 bit/s, Barker-13, one
    input byte = 10^6 output samples): chunk-size invariant on both sides, port rates 5200 / 16 / 8 / 8 per second, and one of the
    two decoders (the symbol-pair alignment of the rate-1/2 code is unknown: the second runs one soft bit late) returns the
    transmitted bits exactly."""
    O = oracle
    rng = np.random.default_rng(5)
    data = rng.integers(0, 256, 40, dtype=np.uint8)
    iq = O.Tx(O.MOD_DSSS, 25, 1000000, 1700, 150, 0).work(data)
    assert len(iq) == len(data) * 1000000
    t2 = O.Tx(O.MOD_DSSS, 25, 1000000, 1700, 150, 0)
    iq2 = np.concatenate([t2.work(data[a:b]) for a, b in ((0, 1), (1, 4), (4, 5))])
    assert np.array_equal(iq[:len(iq2)].view(np.uint32), iq2.view(np.uint32))
    n = np.arange(len(iq))
    x = (iq * 0.5 + 0.01 * (rng.standard_normal(len(iq)) + 1j * rng.standard_normal(len(iq)))).astype(np.complex64)
    x = (x * np.exp(2j * np.pi * 0.5 * n / 1e6 + 0.3j)).astype(np.complex64)
    a = O.Rx(O.DEMOD_DSSS, 25, 1000000, 1700, 150, 0); a.work(x)
    b = O.Rx(O.DEMOD_DSSS, 25, 1000000, 1700, 150, 0)
    for lo in range(0, len(x), 3333331):
        b.work(x[lo:lo + 3333331])
    pa = [a.port(p) for p in range(4)]
    for p in range(4):
        assert np.array_equal(pa[p], b.port(p)), p
    assert len(pa[0]) == len(x) // 50 * 13 // 50 and abs(len(pa[1]) - 16 * 40) < 30 and len(pa[2]) == len(pa[3]) == 240
    bits = np.unpackbits(data)
    best = 0.0
    for port in (2, 3):
        for off in range(0, 40):
            m = min(len(pa[port]) - off, len(bits))
            best = max(best, float(np.mean(pa[port][off:off + m] == bits[:m])))
    assert best == 1.0


def test_mmdvm_channel_chains_restated(oracle):
    """gr_mod_mmdvm_multi2 -> gr_demod_mmdvm_multi2, one channel each side of the filter bank (25 ksps complex <-> int16 at 24 ksps):
    rates 25/24 and 24/25, chunk invariance on both sides, RSSI tags every 300 items, and the discriminator returns the modulating
    samples (the 12.5 kHz deviation maps full-scale int16 onto +-pi/... of phase step; the round trip gain is 1)."""
    O = oracle
    rng = np.random.default_rng(91)
    n = 24000
    t = np.arange(n)
    s = (3000 * np.sin(2 * np.pi * 1200 * t / 24000) + 1500 * np.sin(2 * np.pi * 300 * t / 24000 + 0.7)).astype(np.int16)
    a = O.MmdvmTx(5000); ya = a.work(s)
    assert len(ya) == n * 25 // 24
    b = O.MmdvmTx(5000)
    yb = np.concatenate([b.work(s[lo:lo + 777]) for lo in range(0, n, 777)])
    assert np.array_equal(ya.view(np.uint32), yb.view(np.uint32))
    assert 0.6 < np.abs(ya[2000:]).mean() <= 0.81            # x0.8 behind the 5 kHz channel filter (the FM signal is a little wider)
    r1 = O.MmdvmRx(5000); o1, db1, at1 = r1.work(ya)
    assert len(o1) == len(ya) * 24 // 25
    r2 = O.MmdvmRx(5000)
    parts = [r2.work(ya[lo:lo + 1001]) for lo in range(0, len(ya), 1001)]
    assert np.array_equal(o1, np.concatenate([p[0] for p in parts]))
    assert np.array_equal(db1, np.concatenate([p[1] for p in parts])) and np.array_equal(at1, np.concatenate([p[2] for p in parts]))
    assert len(db1) == len(o1) // 300 and np.array_equal(at1, np.arange(len(db1)) * 300 + 299)
    # discriminator output against the modulating samples: the chain delay is not a whole number of 24 ksps items (two 819-tap
    # resamplers at 600 kHz), so compare the two tones' amplitudes (least squares over the steady state) and the residual
    seg = o1[2000:22000].astype(np.float64)
    tt = np.arange(len(seg))
    A = np.stack([np.sin(2 * np.pi * 1200 * tt / 24000), np.cos(2 * np.pi * 1200 * tt / 24000),
                  np.sin(2 * np.pi * 300 * tt / 24000), np.cos(2 * np.pi * 300 * tt / 24000), np.ones(len(seg))], 1)
    coef, *_ = np.linalg.lstsq(A, seg, rcond=None)
    assert abs(np.hypot(coef[0], coef[1]) - 3000) < 30 and abs(np.hypot(coef[2], coef[3]) - 1500) < 15, coef
    assert np.sqrt(np.mean((seg - A @ coef) ** 2)) < 80          # int16 units (2 % of the signal): FM through two 5 kHz channel filters


def test_mmdvm_tx_zero_idle_restated(oracle):
    """gr_zero_idle_bursts(0) on the MMDVM modulators (the block itself is pinned to the compiled reference in test_oracle_ref.py):
    behind the x25/24 resampler of gr_mod_mmdvm_multi2 the tagged stretches of the plain output are cleared and nothing else changes;
    in front of the filter of gr_mod_mmdvm the output is the plain one away from the cleared stretch and exactly zero deep inside it;
    results do not depend on the chunking."""
    n = 6000
    rng = np.random.default_rng(9810)
    s = (6000 * np.sin(2 * np.pi * 700 * np.arange(n) / 24000) + rng.integers(-200, 200, n)).astype(np.int16)
    # multi2: tags on 25 ksps items; the second overrides the first's running count
    plain = oracle.MmdvmTx(5000).work(s)
    o = oracle.MmdvmTx(5000)
    o.zero_samples(1000, 900); o.zero_samples(1500, 100); o.zero_samples(4000, 50)
    got = np.concatenate([o.work(s[a:b]) for a, b in ((0, 1), (1, 1000), (1000, 1001), (1001, n))])
    want = plain.copy(); want[1000:1600] = 0; want[4000:4050] = 0
    assert len(got) == n * 25 // 24 and np.array_equal(got.view(np.uint32), want.view(np.uint32))
    # a tag registered after its item has gone out clears what is left of its count
    o = oracle.MmdvmTx(5000)
    first = o.work(s[:2400])                                  # 2500 items out
    o.zero_samples(2400, 300)                                 # 100 of them are gone already
    got = np.concatenate([first, o.work(s[2400:])])
    want = plain.copy(); want[2500:2700] = 0
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    # single-channel block: the cleared stretch passes the low-pass and the x125/12 resampler
    plain1 = oracle.MmdvmTx(5000, single=True).work(s)
    o = oracle.MmdvmTx(5000, single=True)
    o.zero_samples(2000, 1500)
    got1 = np.concatenate([o.work(s[a:b]) for a, b in ((0, 777), (777, 2000), (2000, 2001), (2001, n))])
    assert len(got1) == len(plain1) == n * 125 // 12
    r = 125 / 12
    assert np.array_equal(got1[:int(1900 * r)], plain1[:int(1900 * r)])            # before the stretch (minus nothing: the chain is causal)
    assert np.all(got1[int(2200 * r):int(3450 * r)] == 0)                          # deep inside: filters flushed, exactly zero
    assert np.array_equal(got1[int(3800 * r):], plain1[int(3800 * r):])            # well behind it the histories hold plain items again
    assert not np.array_equal(got1, plain1)
