"""TX front end throughput (qrl_txfront: rotator at 1 Msps + xN interpolator to the device rate) on one GPU; prints one JSON line.

Kernel leg: 64 channels x 2^20 input items per call, input resident in HBM, at 2, 10, 20 and 56 Msps, fc32 and sc16 output.  Each
shape is warmed up, then called back to back on one stream until the CUDA events around the calls span at least --min-seconds of
device time.  The outputs (1 to 30 GB per call) are far larger than L2, so every call writes HBM.  Work and bytes are computed from
the shapes: 2 NT lane-FMAs per output sample (NT = taps per arm, an FFMA2 counts two), and 8 (fc32) or 4 (sc16) bytes written per
output sample.  The FP32 ceiling is SMs x 128 lanes x the maximum SM clock nvidia-smi reports; the kernel is FP32-bound (its HBM
write rate is an order of magnitude below the card's), so the share of that ceiling is the figure of merit.

End-to-end leg: the same call from a pinned host buffer (H2D of the 1 Msps input, the kernels, D2H of the device-rate output into a
pinned host buffer), host clock around work + read, fc32 against sc16, 16 channels at 10 Msps.

usage: python tools/txfront_bench.py [--rates 2,10,20,56] [--channels 64] [--items 1048576] [--min-seconds 1.0] [--out FILE]"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=clocks.max.sm,power.limit,name", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    clk, pwr, name = [s.strip() for s in q.split(",", 2)]
    return float(clk), float(pwr), name


def arm_taps(rate):
    """taps per arm of low_pass(N, rate, 480000, 20000, BLACKMAN_HARRIS), from the library's host-side design helper"""
    import qradiolink_b200 as q
    N = rate // 1000000
    h = (C.c_float * (1 << 15))()
    n = q.load_library().qrl_firdes_low_pass(float(N), float(rate), 480000.0, 20000.0, 5, C.cast(h, C.c_void_p), 1 << 15)
    return -(-n // N)


def kernel_leg(q, torch, rate, fmt, Cn, n, min_s, ceiling):
    N = rate // 1000000
    x = (torch.randn(Cn, n, dtype=torch.complex64, device="cuda") * 0.5).contiguous()
    t = q.TxFrontend(rate, n_channels=Cn, max_in=n, out_format=fmt)
    s = torch.cuda.Stream()                              # the handle's launches and the events on one (non-default) stream
    t.set_stream(s.cuda_stream)
    torch.cuda.synchronize()
    for _ in range(2):
        t.work_device(x.data_ptr(), n, n)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.perf_counter()
    e0.record(s); t.work_device(x.data_ptr(), n, n); e1.record(s); e1.synchronize()
    one = e0.elapsed_time(e1)
    assert one >= 0.5 * (time.perf_counter() - w0) * 1e3 - 1.0, "events do not bracket the launches"
    reps = min(1000, max(3, int(min_s * 1000.0 / one) + 1))
    l0 = t.launches
    e0.record(s)
    for _ in range(reps):
        t.work_device(x.data_ptr(), n, n)
    e1.record(s); e1.synchronize()
    ms = e0.elapsed_time(e1) / reps
    launches = (t.launches - l0) // reps
    t.close(); del x; torch.cuda.empty_cache()
    nt = arm_taps(rate)
    outs = Cn * n * N
    fma = 2.0 * nt * outs
    wbytes = outs * (8 if fmt == "fc32" else 4)
    return {"samp_rate": rate, "N": N, "format": fmt, "channels": Cn, "items_in": n, "taps_per_arm": nt, "calls_timed": reps,
            "device_seconds": round(ms * reps / 1000.0, 3), "launches_per_call": launches, "ms_per_call": round(ms, 3),
            "out_gsamples_per_s": round(outs / ms / 1e6, 2), "lane_fma_per_call": fma, "tflops_fma": round(2 * fma / ms / 1e9, 2),
            "share_of_fp32_ceiling": round(fma / (ms / 1000.0) / ceiling, 3), "hbm_bytes_written": wbytes,
            "write_gb_per_s": round(wbytes / ms / 1e6, 1)}


def e2e_leg(q, torch, rate, fmt, Cn, n, reps=5):
    N = rate // 1000000
    x = (torch.randn(Cn, n, dtype=torch.complex64) * 0.5).pin_memory()
    dt = torch.complex64 if fmt == "fc32" else torch.int16
    out = torch.empty((Cn, n * N * (1 if fmt == "fc32" else 2)), dtype=dt).pin_memory()
    t = q.TxFrontend(rate, n_channels=Cn, max_in=n, out_format=fmt)
    L = t._L
    no = C.c_long()

    def call():
        assert L.qrl_txfront_work(t._h, C.c_void_p(x.data_ptr()), n, n, 0, C.byref(no)) == 0
        assert L.qrl_txfront_read(t._h, C.c_void_p(out.data_ptr()), no.value) == 0

    call(); call()
    t0 = time.perf_counter()
    for _ in range(reps):
        call()
    sec = (time.perf_counter() - t0) / reps
    t.close()
    d2h = Cn * n * N * (8 if fmt == "fc32" else 4)
    return {"samp_rate": rate, "format": fmt, "channels": Cn, "items_in": n, "ms_per_call": round(sec * 1e3, 2),
            "out_gsamples_per_s": round(Cn * n * N / sec / 1e9, 3), "d2h_bytes": d2h, "h2d_bytes": Cn * n * 8}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rates", default="2,10,20,56")
    ap.add_argument("--channels", type=int, default=64)
    ap.add_argument("--items", type=int, default=1 << 20)
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--e2e-channels", type=int, default=16)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import qradiolink_b200 as q
    if q.device_count() < 1 or not torch.cuda.is_available():
        raise SystemExit("txfront_bench needs a CUDA device")
    clk, pwr, name = gpu_info()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    ceiling = sms * 128 * clk * 1e6                      # lane-FMAs per second
    res = {"tool": "txfront_bench", "gpu": name, "power_limit_w": pwr, "sm_clock_max_mhz": clk, "sms": sms,
           "fp32_ceiling_lane_fma_per_s": ceiling, "bound": "FP32 (FMA pipe)", "kernel": [], "end_to_end": []}
    for r in [int(v) * 1000000 for v in a.rates.split(",")]:
        for fmt in ("fc32", "sc16"):
            res["kernel"].append(kernel_leg(q, torch, r, fmt, a.channels, a.items, a.min_seconds, ceiling))
            print(json.dumps(res["kernel"][-1]), file=sys.stderr, flush=True)
    for fmt in ("fc32", "sc16"):
        res["end_to_end"].append(e2e_leg(q, torch, 10000000, fmt, a.e2e_channels, a.items))
        print(json.dumps(res["end_to_end"][-1]), file=sys.stderr, flush=True)
    line = json.dumps(res)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        open(a.out, "w").write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
