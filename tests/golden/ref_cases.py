"""Seeded inputs and call schedules shared by tests/golden/make_ref_golden.py (which drives the reference's own GNU Radio blocks,
compiled unmodified into oracle/_ref/libqrl_ref_blocks.so, and freezes what they return) and tests/test_oracle_ref.py (which
checks the oracle and the host-side sink restatements against the frozen answers).  Test infrastructure only.

A schedule is a generator of operations, so that both sides make exactly the same calls with exactly the same data."""
import hashlib

import numpy as np

BARKER_13 = np.array([1, 1, 1, 1, 1, 0, 0, 1, 1, 0, 1, 0, 1], np.int32)
DSSS_SPS, DSSS_HISTORY = 25, 325
DEFRAMER_WORDS = [(0xED89, 16), (0x89ED, 16), (0x98DE, 16), (0xED77, 16), (0x8CC8, 16), (0x4C8A2B, 24), (0xB5, 8)]
SINK_DTYPE = {"bit": np.uint8, "audio": np.float32, "const": np.complex64}
SINK_GET_CAP = {"bit": 1 << 21, "audio": 1 << 14, "const": 1 << 14}
SAMPLE_SINK_GET_CAP = 1 << 20
ZERO_IDLE_DELAYS = (62, 0)
RSSI_CHUNKINGS = ([7000], [299, 1, 300, 301, 5000, 2000], [7] * 1001)


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def disc4_input():
    rng = np.random.default_rng(11)
    n = 20000
    m = rng.random((4, n)).astype(np.float32)
    m[:, :2000] = np.round(m[:, :2000] * 4) / 4          # many exact ties: the strict-greater rule decides
    m[:, 2000:2100] = 0.0
    return m


def cessb_clipper_input():
    rng = np.random.default_rng(12)
    n = 8 * 1024
    x = ((rng.standard_normal(n) + 1j * rng.standard_normal(n)) * rng.choice([0.05, 0.5, 1.5], n)).astype(np.complex64)
    x[:16] = 0
    return x


def cessb_stretcher_input():
    rng = np.random.default_rng(13)
    n = 9 * 1024 + 2
    return ((rng.standard_normal(n) + 1j * rng.standard_normal(n)) * rng.choice([0.1, 0.6, 1.2], n)).astype(np.complex64)


def _planted_bits(rng, n, words):
    bits = rng.integers(0, 2, n, dtype=np.uint8)
    pos = 50
    while pos + 500 < n:
        w, nb = words[int(rng.integers(0, len(words)))]
        bits[pos:pos + nb] = [(w >> (nb - 1 - k)) & 1 for k in range(nb)]
        pos += int(rng.integers(100, 700))
    return bits


def deframer_chunks(modem_type):
    """Random bits with sync words planted in them, cut into ragged work() calls."""
    rng = np.random.default_rng(20 + modem_type)
    bits = _planted_bits(rng, 60000, DEFRAMER_WORDS)
    pos = 0
    while pos < len(bits):
        m = int(rng.integers(1, 3000))
        yield np.ascontiguousarray(bits[pos:pos + m])
        pos += m


def sink_ops(kind):
    """400 random steps: an array = one work() call with it, None = one get_data() poll."""
    rng = np.random.default_rng({"bit": 31, "audio": 32, "const": 33}[kind])
    big = {"bit": 400000, "audio": 3000, "const": 120}[kind]
    for _ in range(400):
        if rng.random() < 0.6:
            n = int(rng.integers(0, big))
            if kind == "bit":
                yield rng.integers(0, 2, n, dtype=np.uint8)
            elif kind == "audio":
                yield rng.standard_normal(n).astype(np.float32)
            else:
                yield (rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64)
        else:
            yield None


def sample_sink_ops():
    """gr_sample_sink: enable at step 5, ("work", x), ("window", w) and ("get",) in a random schedule."""
    rng = np.random.default_rng(34)
    for step in range(300):
        r = rng.random()
        if step == 5:
            yield ("enable",)
        if r < 0.55:
            n = int(rng.integers(0, 200000))
            yield ("work", (rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64))
        elif r < 0.65:
            yield ("window", int(rng.integers(1, 30000)))
        else:
            yield ("get",)


def zero_idle_input():
    """(x, tag offsets, tag values, work() chunk sizes); tags are kept at least 62 items inside their work() window."""
    rng = np.random.default_rng(31)
    n, delay = 30000, ZERO_IDLE_DELAYS[0]
    x = (rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64)
    chunks = np.array([4096, 1000, 8192, 5000, 20000], np.int64)
    edges = np.concatenate([[0], np.cumsum(chunks)])
    tag_items, tag_vals = [], []
    for k in range(len(chunks)):
        lo, hi = edges[k], min(edges[k + 1], n)
        if hi - lo < 400:
            continue
        for j in range(3):
            tag_items.append(int(lo + delay + rng.integers(0, hi - lo - delay)))
            tag_vals.append(int(rng.integers(1, 900)))
    tag_items.append(tag_items[0] + 5); tag_vals.append(3)           # overrides a running count with a short one
    tag_items.append(30); tag_vals.append(500)                        # item < delay: never matches
    return x, np.array(tag_items, np.int64), np.array(tag_vals, np.int64), chunks


RX_FFT_FREQ = 0.1234


def rx_fft_ops(n_fft):
    """rx_fft_c: ("work", x) before and after enabling, ("get",) polls whose answer is compared, ("size", n) and ("drain",), a poll
    whose answer is not compared (the first one after a change of size)."""
    rng = np.random.default_rng(61)
    n = n_fft * 9 + 777
    t = np.arange(n)
    x = (0.3 * np.exp(2j * np.pi * RX_FFT_FREQ * t) + 0.05 * (rng.standard_normal(n) + 1j * rng.standard_normal(n))).astype(np.complex64)
    x[5000:5050] = 0
    sizes = [n_fft // 3, 17, n_fft, n_fft // 2 + 5, 2 * n_fft + 9, 100, n_fft - 1, 3 * n_fft]
    lo = 0
    for step, m in enumerate(sizes):
        if step == 0:
            yield ("work", x[lo:lo + 50])                                # not enabled yet: dropped
            yield ("enable",)
        m = min(m, n - lo)
        yield ("work", x[lo:lo + m])
        lo += m
        if step % 2 == 1:
            yield ("get",)
    yield ("size", n_fft // 2)
    yield ("drain",)
    yield ("work", x[:n_fft])
    yield ("get",)


def dsss_input():
    """A spread BPSK stream + noise so that the maximum is well defined, plus a stretch of exact zeros."""
    rng = np.random.default_rng(71)
    n_sym = 40
    chips = np.repeat(np.where(BARKER_13 > 0, 1.0, -1.0), DSSS_SPS)
    bits = rng.integers(0, 2, n_sym) * 2 - 1
    x = np.concatenate([b * chips for b in bits]).astype(np.complex64) * np.exp(0.4j).astype(np.complex64)
    x = (x + 0.3 * (rng.standard_normal(len(x)) + 1j * rng.standard_normal(len(x)))).astype(np.complex64)
    x[3000:3400] = 0
    return x, n_sym


def rssi_input():
    rng = np.random.default_rng(81)
    n = 7000
    return ((rng.standard_normal(n) + 1j * rng.standard_normal(n)) * np.repeat(rng.uniform(1e-4, 2.0, n // 100), 100)).astype(np.complex64)
