"""Pins the oracle (and the host-side sink restatements) to REFERENCE CODE: tests/golden/ref_blocks_v1.json and
ref_cessb_clipper_v1.npy hold what the reference's src/gr/{gr_4fsk_discriminator, gr_deframer_bb, gr_bit_sink, gr_audio_sink,
gr_const_sink, gr_sample_sink, gr_zero_idle_bursts, rx_fft, dsss_decoder_cc_impl, rssi_tag_block, cessb/clipper_cc_impl,
cessb/stretcher_cc_impl}, compiled UNMODIFIED against the runtime stand-in in oracle/gr_stub/ (oracle/Makefile target `ref`;
oracle/ref_blocks_shim.cpp plays the scheduler), returned for the seeded inputs and call schedules of tests/golden/ref_cases.py
(tests/golden/make_ref_golden.py).  CPU tier."""
import ctypes as C
import importlib
import json
import os

import numpy as np
import pytest

from oracle import oracle as O
from tests.golden import ref_cases as RC
from tests.golden.ref_cases import sha

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
G = json.load(open(os.path.join(GOLDEN, "ref_blocks_v1.json")))


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def test_discriminator_is_the_reference_block():
    m = RC.disc4_input()
    n = m.shape[1]
    got = np.zeros(2 * n, np.float32)
    O.lib().qo_disc4(_p(m[0]), _p(m[1]), _p(m[2]), _p(m[3]), n, _p(got))
    assert len(got) == G["disc4"]["n"] and sha(got) == G["disc4"]["sha256"]
    assert np.any(got == 0.0) and len(np.unique(got)) == 3      # -0.707107, 0, +0.707107 all occur


def test_cessb_clipper_against_the_reference_block():
    x = RC.cessb_clipper_input()
    n = len(x)
    ref = np.load(os.path.join(GOLDEN, "ref_cessb_clipper_v1.npy"))
    assert G["cessb_clipper"]["returned"] == n and ref.shape == (n,) and ref.dtype == np.complex64
    got = np.zeros(n, np.complex64)
    O.lib().qo_cessb_clipper(_p(x), n, C.c_float(0.95), _p(got))
    # magnitude path (sqrt, min) is IEEE on both sides; the phase goes through cos / sin, libm (VOLK generic) in the compiled
    # reference vs the oracle's fixed polynomial: 3e-7 each (tests/test_oracle.py::test_sincos_and_atan)
    assert np.max(np.abs(ref - got)) < 5e-7
    assert np.max(np.abs(np.abs(ref) - np.abs(got))) < 2e-7 and np.max(np.abs(got)) <= 0.95 + 1e-6
    small = np.abs(x) < 0.9
    assert np.max(np.abs(np.abs(got[small]) - np.abs(x[small]))) < 3e-7      # below the clip level only the rounding of cos/sin


@pytest.mark.parametrize("chunk", [1024, 3072])
def test_cessb_stretcher_is_the_reference_block_bit_for_bit(chunk):
    x = RC.cessb_stretcher_input()
    n = len(x)
    want = G["cessb_stretcher"][str(chunk)]
    got = np.zeros(n, np.complex64)
    n_got = O.lib().qo_cessb_stretcher(_p(x), n, _p(got))
    n_ref = want["n"]
    assert n_got == n - 2 and n_ref == 9 * 1024
    assert sha(got[:n_ref]) == want["sha256"]                    # the reference block, in either chunking, gave these bits
    assert np.any(np.abs(got[:n_ref]) < np.abs(x[:n_ref]) * 0.9)                           # the stretcher did act


@pytest.mark.parametrize("modem_type", [1, 2, 3])
def test_gr_deframer_bb_is_the_reference_block(modem_type):
    d = O.DeframerBB(modem_type)
    got = np.concatenate([d.work(chunk) for chunk in RC.deframer_chunks(modem_type)])
    want = G["deframer"][str(modem_type)]
    assert len(got) > 1000 and len(got) == want["n"] and sha(got) == want["sha256"]


@pytest.mark.parametrize("kind", ["bit", "audio", "const"])
def test_sink_restatements_follow_the_reference_sinks(kind):
    """qradiolink_b200.demod.gr_*_sink (what the Python host side polls) against the compiled gr_*_sink.cpp, random schedules."""
    demod = importlib.import_module("qradiolink_b200.demod")
    mine = getattr(demod, "gr_%s_sink" % kind)()
    want = G["sinks"][kind]
    works, gets = iter(want["work"]), iter(want["get"])
    for x in RC.sink_ops(kind):
        if x is not None:
            assert next(works) == mine.work(x)
        else:
            k, digest = next(gets)
            m = mine.get_data()
            if k < 0:
                assert m is None
            else:
                assert m is not None and len(m) == k and sha(m) == digest
    assert next(works, None) is None and next(gets, None) is None


def test_sample_sink_restatement_follows_the_reference_sink():
    """qradiolink_b200.demod.gr_sample_sink against the compiled gr_sample_sink.cpp: enable, window changes (odd sizes), the 524288-item
    drop rule, random schedules."""
    demod = importlib.import_module("qradiolink_b200.demod")
    mine = demod.gr_sample_sink()
    want = G["sample_sink"]
    works, gets = iter(want["work"]), iter(want["get"])
    for op in RC.sample_sink_ops():
        if op[0] == "enable":
            mine.set_enabled(True)
        elif op[0] == "work":
            assert next(works) == mine.work(op[1])
        elif op[0] == "window":
            mine.set_sample_window(op[1])
        else:
            k, digest = next(gets)
            m = mine.get_data()
            if k < 0:
                assert m is None
            else:
                assert m is not None and len(m) == k and sha(m) == digest
    assert next(works, None) is None and next(gets, None) is None


def test_zero_idle_bursts_is_the_reference_block():
    """gr_zero_idle_bursts.cpp compiled unmodified (stream tags through the stand-in's get_tags_in_window): delay of history-1 items,
    a counter loaded `delay` items before the tagged one, later tags overriding a running count.  Tags are kept at least `delay`
    items inside their work() window -- the only place the restatement deviates (it also honours the ones the reference drops)."""
    x, to, tv, _ = RC.zero_idle_input()
    n = len(x)
    got = O.zero_idle(x, RC.ZERO_IDLE_DELAYS[0], to, tv)
    assert G["zero_idle"]["62"]["done"] == n and sha(got) == G["zero_idle"]["62"]["sha256"]
    assert np.count_nonzero(got == 0) > 1439 + 500 and np.all(got[:1439] == 0)
    nz = got[1439:] != 0
    assert np.array_equal(got[1439:][nz], x[:n - 1439][nz])              # what is not zeroed is the input, 1439 items late
    # delay = 0: no history, pure pass-through + tags at their own item
    got0 = O.zero_idle(x, 0, to, tv)
    assert G["zero_idle"]["0"]["done"] == n and sha(got0) == G["zero_idle"]["0"]["sha256"]


@pytest.mark.parametrize("n_fft", [1024, 32768])
def test_rx_fft_restatement_follows_the_reference_block(n_fft):
    """rx_fft.cpp compiled unmodified (FFTW replaced by the oracle's own DFT in the stand-in, so this pins the buffering, windowing,
    d_push drop rule, power-spectrum kernel and fft-shift, not FFTW's rounding): same points after every get, for ragged work()
    sizes incl. calls longer than the FFT, calls while a spectrum is pending, disable / enable and a change of size."""
    s = O.Spectrum(n_fft, O.WIN_BLACKMAN_HARRIS)
    gets = iter(G["rx_fft"][str(n_fft)])
    size, got_any = n_fft, 0
    for op in RC.rx_fft_ops(n_fft):
        if op[0] == "work":
            s.work(op[1])
        elif op[0] == "enable":
            s.set_enabled(True)
        elif op[0] == "size":
            s.set_fft_size(op[1]); size = op[1]
        elif op[0] == "drain":
            s.get()
        else:
            nr, digest = next(gets)
            g = s.get()
            assert (nr == 0) == (g is None)
            if g is not None:
                assert nr == size and len(g) == nr and sha(g) == digest
                if size == n_fft:
                    got_any += 1
                    peak = int(np.argmax(g))
                    assert abs(peak - (n_fft // 2 + round(RC.RX_FFT_FREQ * n_fft))) <= 1
    assert next(gets, None) is None
    assert got_any >= 3 and size == n_fft // 2 and g is not None                 # the last get came after the change of size


def test_dsss_decoder_restatement_is_the_reference_block():
    """dsss_decoder_cc_impl.cc compiled unmodified: the matched-filter taps its constructor builds, and general_work over a buffer laid
    out the way the restatement DEFINES the region in front of the declared history (the stream's own older items, zeros at the
    start): same symbols bit for bit, for several scheduler chunkings of the reference and several of the restatement."""
    want = G["dsss_decoder"]
    sps, N = RC.DSSS_SPS, RC.DSSS_HISTORY
    assert want["history"] == N
    nt = N + 11 * sps
    tq = np.zeros(2 * nt, np.float32)
    O.lib().qo_dsss_decoder_taps(_p(RC.BARKER_13), 13, sps, _p(tq))
    assert want["n_taps"] == nt and sha(tq) == want["taps_sha256"]
    x, n_sym = RC.dsss_input()
    n = len(x)
    got = np.zeros(n_sym + 4, np.complex64)
    for chunk in (n, 1000, 77):
        m = O.lib().qo_dsss_decoder_run(_p(RC.BARKER_13), 13, sps, _p(x), n, chunk, _p(got), len(got))
        if chunk == n:
            first, m0 = got[:m].copy(), m
        assert m == m0 and np.array_equal(got[:m].view(np.uint32), first.view(np.uint32)), chunk
    # reference: fed one, three and all symbols' worth of input per general_work call
    assert m0 == want["n_symbols"]
    for per_call, digest in want["symbols_sha256"].items():
        assert sha(first) == digest, per_call
    assert m0 >= n_sym - 2


def test_rssi_tag_rule_is_the_reference_block():
    """rssi_tag_block.cpp compiled unmodified (add_item_tag through the stand-in): an "RSSI" tag every 300 items, value and offset, for
    several scheduler chunkings; the float accumulation order is the block's (sequential)."""
    x = RC.rssi_input()
    n = len(x)
    db_o = np.zeros(64, np.float32); at_o = np.zeros(64, np.int64)
    k = O.lib().qo_rssi_tags_run(_p(x), n, -3.5, _p(db_o), _p(at_o), 64)
    assert k == n // 300
    assert len(G["rssi_tags"]) == len(RC.RSSI_CHUNKINGS)
    for want in G["rssi_tags"]:
        db_r = np.array([float.fromhex(v) for v in want["db"]], np.float32)
        assert want["n"] == k and want["offsets"] == [int(v) for v in at_o[:k]] and np.array_equal(db_r.view(np.uint32), db_o[:k].view(np.uint32))
    assert np.array_equal(at_o[:k], np.arange(k) * 300 + 299)
