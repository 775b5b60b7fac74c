"""Generates tests/golden/ref_blocks_v1.json and tests/golden/ref_cessb_clipper_v1.npy -- what the reference's own GNU Radio
blocks return for the seeded inputs and call schedules of tests/golden/ref_cases.py.

The blocks are the reference's src/gr/{gr_4fsk_discriminator, gr_deframer_bb, gr_bit_sink, gr_audio_sink, gr_const_sink,
gr_sample_sink, gr_zero_idle_bursts, rx_fft, dsss_decoder_cc_impl, rssi_tag_block, cessb/clipper_cc_impl,
cessb/stretcher_cc_impl}, compiled unmodified against the runtime stand-in in oracle/gr_stub/ into
oracle/_ref/libqrl_ref_blocks.so (oracle/Makefile target `ref`, which needs the reference source tree).  The answers are
committed so that tests/test_oracle_ref.py can pin the oracle and the host-side sink restatements to them anywhere.
Outputs compared bit for bit are recorded as SHA-256 of their bytes; the clipper, compared within a tolerance, in full.

Run from the repo root after `make -C oracle REF=<reference source tree>`:  python tests/golden/make_ref_golden.py
"""
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import oracle as O  # noqa: E402
from tests.golden import ref_cases as RC  # noqa: E402
from tests.golden.ref_cases import sha  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def disc4(R):
    m = RC.disc4_input()
    n = m.shape[1]
    ref = np.zeros(2 * n, np.float32)
    R.ref_disc4(_p(m[0]), _p(m[1]), _p(m[2]), _p(m[3]), n, _p(ref))
    return {"n": int(len(ref)), "sha256": sha(ref)}


def cessb_clipper(R):
    x = RC.cessb_clipper_input()
    ref = np.zeros(len(x), np.complex64)
    k = R.ref_cessb_clipper(_p(x), len(x), 0.95, _p(ref))
    np.save(os.path.join(GOLDEN, "ref_cessb_clipper_v1.npy"), ref)
    return {"returned": int(k)}


def cessb_stretcher(R):
    x = RC.cessb_stretcher_input()
    out = {}
    for chunk in (1024, 3072):
        ref = np.zeros(len(x), np.complex64)
        k = R.ref_cessb_stretcher(_p(x), len(x), chunk, _p(ref))
        out[str(chunk)] = {"n": int(k), "sha256": sha(ref[:k])}
    return out


def deframer(R):
    out = {}
    for modem_type in (1, 2, 3):
        h = R.ref_dfbb_create(modem_type)
        ref = []
        for chunk in RC.deframer_chunks(modem_type):
            buf = np.zeros(4 * len(chunk) + 64, np.uint8)
            k = R.ref_dfbb_work(h, _p(chunk), len(chunk), _p(buf), len(buf))
            ref.append(buf[:k].copy())
        R.ref_block_destroy(h)
        ref = np.concatenate(ref)
        out[str(modem_type)] = {"n": int(len(ref)), "sha256": sha(ref)}
    return out


def sinks(R):
    out = {}
    for kind in ("bit", "audio", "const"):
        h = getattr(R, "ref_%s_sink_create" % kind)()
        work, get = getattr(R, "ref_%s_sink_work" % kind), getattr(R, "ref_%s_sink_get" % kind)
        buf = np.zeros(RC.SINK_GET_CAP[kind], RC.SINK_DTYPE[kind])
        rec = {"work": [], "get": []}
        for x in RC.sink_ops(kind):
            if x is not None:
                rec["work"].append(int(work(h, _p(x), len(x))))
            else:
                k = int(get(h, _p(buf), len(buf)))
                rec["get"].append([k, sha(buf[:k]) if k >= 0 else None])
        R.ref_block_destroy(h)
        out[kind] = rec
    return out


def sample_sink(R):
    h = R.ref_sample_sink_create()
    buf = np.zeros(RC.SAMPLE_SINK_GET_CAP, np.complex64)
    rec = {"work": [], "get": []}
    for op in RC.sample_sink_ops():
        if op[0] == "enable":
            R.ref_sample_sink_set_enabled(h, 1)
        elif op[0] == "work":
            rec["work"].append(int(R.ref_sample_sink_work(h, _p(op[1]), len(op[1]))))
        elif op[0] == "window":
            R.ref_sample_sink_set_window(h, op[1])
        else:
            k = int(R.ref_sample_sink_get(h, _p(buf), len(buf)))
            rec["get"].append([k, sha(buf[:k]) if k >= 0 else None])
    R.ref_block_destroy(h)
    return rec


def zero_idle(R):
    x, to, tv, chunks = RC.zero_idle_input()
    ch = chunks.astype(np.dtype("l"))
    out = {}
    for delay in RC.ZERO_IDLE_DELAYS:
        ref = np.zeros(len(x), np.complex64)
        done = R.ref_zero_idle(_p(x), len(x), delay, _p(to), _p(tv), len(to), _p(ch), len(ch), _p(ref))
        out[str(delay)] = {"done": int(done), "sha256": sha(ref)}
    return out


def rx_fft(R):
    out = {}
    for n_fft in (1024, 32768):
        h = R.ref_rx_fft_create(n_fft, O.WIN_BLACKMAN_HARRIS)
        pts = np.empty(n_fft, np.float32)
        gets = []
        for op in RC.rx_fft_ops(n_fft):
            if op[0] == "work":
                R.ref_rx_fft_work(h, _p(op[1]), len(op[1]))
            elif op[0] == "enable":
                R.ref_rx_fft_set_enabled(h, 1)
            elif op[0] == "size":
                R.ref_rx_fft_set_fft_size(h, op[1])
            elif op[0] == "drain":
                R.ref_rx_fft_get(h, _p(pts))
            else:
                nr = int(R.ref_rx_fft_get(h, _p(pts)))
                gets.append([nr, sha(pts[:nr]) if nr else None])
        R.ref_block_destroy(h)
        out[str(n_fft)] = gets
    return out


def dsss_decoder(R):
    sps, N = RC.DSSS_SPS, RC.DSSS_HISTORY
    h = R.ref_dsss_decoder_create(_p(RC.BARKER_13), 13, C.c_float(sps))
    history = int(R.ref_dsss_decoder_history(h))
    nt = N + 11 * sps
    taps = np.zeros(2 * nt, np.float32)
    n_taps = int(R.ref_dsss_decoder_taps(h, _p(taps), nt))
    x, n_sym = RC.dsss_input()
    # the number of symbols is the one the restatement defines for this stream (its region in front of the declared history)
    got = np.zeros(n_sym + 4, np.complex64)
    m0 = int(O.lib().qo_dsss_decoder_run(_p(RC.BARKER_13), 13, sps, _p(x), len(x), len(x), _p(got), len(got)))
    # reference: buffer = [2N - 1 zeros][x][slack]; output m is called with `in` = item m N - (N - 1) (history N), one or more per call
    buf = np.concatenate([np.zeros(2 * N - 1, np.complex64), x, np.zeros(2 * N, np.complex64)])
    symbols = {}
    for per_call in (1, 3, m0):
        ref = np.zeros(m0, np.complex64)
        done = 0
        while done < m0:
            k = min(per_call, m0 - done)
            cons = C.c_long()
            out = np.zeros(k, np.complex64)
            assert R.ref_dsss_decoder_work(h, _p(buf[(2 * N - 1) + done * N - (N - 1):]), k, _p(out), C.byref(cons)) == k and cons.value == k * N
            ref[done:done + k] = out
            done += k
        symbols["all" if per_call == m0 else str(per_call)] = sha(ref)
    R.ref_block_destroy(h)
    return {"history": history, "n_taps": n_taps, "taps_sha256": sha(taps), "n_symbols": m0, "symbols_sha256": symbols}


def rssi_tags(R):
    x = RC.rssi_input()
    out = []
    for chunks in RC.RSSI_CHUNKINGS:
        ch = np.array(chunks, np.dtype("l"))
        db = np.zeros(64, np.float32); at = np.zeros(64, np.int64)
        k = int(R.ref_rssi_tags(_p(x), len(x), C.c_float(-3.5), _p(ch), len(ch), _p(db), _p(at), 64))
        out.append({"n": k, "offsets": [int(v) for v in at[:k]], "db": [float.hex(float(v)) for v in db[:k]]})
    return out


def main():
    R = O.ref_blocks()
    if R is None:
        raise SystemExit("oracle/_ref/libqrl_ref_blocks.so missing: run `make -C oracle REF=<reference source tree>`")
    out = {"version": 1, "generator": "tests/golden/make_ref_golden.py"}
    for name, fn in (("disc4", disc4), ("cessb_clipper", cessb_clipper), ("cessb_stretcher", cessb_stretcher), ("deframer", deframer),
                     ("sinks", sinks), ("sample_sink", sample_sink), ("zero_idle", zero_idle), ("rx_fft", rx_fft),
                     ("dsss_decoder", dsss_decoder), ("rssi_tags", rssi_tags)):
        out[name] = fn(R)
    path = os.path.join(GOLDEN, "ref_blocks_v1.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
