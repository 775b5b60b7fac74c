#!/usr/bin/env python
"""bench.py -- benchmark of the hot path (BASELINE.json metric: RX IQ Msamples/s, batched channels).

Headline workload (BASELINE.json configs[1]): 64 channels of 4FSK-2k RX (RRC + clock recovery + Viterbi), 1 Msps per
channel, per GPU (weak scaling: every rank runs its own 64 channels; channels are independent, so there is no data-path
collective).  One STEP = CALLS_PER_STEP streaming qrl_rx_work calls, each over a [64][2^22] gr_complex slab resident in
HBM (2.1 GB per call, far beyond the 126 MB L2), i.e. 268 s of air time per channel per step -- long enough that the
K timed steps the driver asks for cover more than a second of device time.

  python bench.py --gpus N --steps K --warmup W            our CUDA path: device-resident `value`, host-buffer `e2e`,
                                                           plus a `configs` block with the other BASELINE configurations
  python bench.py --impl reference ...                     the CPU restatement of the reference chain (oracle port)
  python bench.py ... --dump-outputs DIR                   also writes what the timed path computed to DIR/*.npy (dump_outputs)

Prints ONE JSON line (rank 0).  The CPU oracle is used here only as the checker (parity spot checks on the very buffers
that were timed) and as the timed CPU baseline; nothing on the GPU arm's timed path touches it.
"""
import argparse
import ctypes as Ct
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CHANNELS = 64
T_CALL = 1 << 22
CALLS_PER_STEP = 64
D1 = 50
ALG_BYTES_PER_SAMPLE = 8.0 * (1.0 + 1.0 / D1)      # stage 1: read 8 B, write 8/D B per input sample (SURVEY 8d)
N_BASES = 8
WORKLOAD = ("64ch 4FSK-2k-FM RX (make_gr_demod_4fsk(5,1e6,1700,3000,true)): /50 polyphase FIR + LPF + quad demod + RRC + "
            "symbol sync + CCSDS Viterbi + descrambler, 1 Msps/ch")
METRIC = "RX IQ Msamples/s (batched channels)"


def headline_config(world):
    """Identical in both arms (the driver compares them)."""
    return {"workload": WORKLOAD, "channels_per_gpu": CHANNELS, "samples_per_channel_per_call": T_CALL,
            "calls_per_step": CALLS_PER_STEP, "samples_per_channel_per_step": T_CALL * CALLS_PER_STEP,
            "l2": "inputs 2.1 GB per call > 126 MB L2, no flush", "parallelism": "channel-sharded x%d, no data-path collective" % world}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def host_cores():
    """Threads this process may really use: scheduler affinity, capped by the cgroup CPU quota when there is one."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    quota = float(txt[0]) / float(txt[1])
            else:
                q = float(txt[0])
                if q > 0:
                    quota = q / float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            break
        except Exception:  # noqa: BLE001
            continue
    used = n if quota is None else max(1, min(n, int(quota)))
    return used, {"sched_affinity": n, "cgroup_quota_cpus": quota, "cpu_count": os.cpu_count()}


def bind_to_gpu_numa(torch, local):
    """Restrict this rank to the CPUs next to its GPU (sysfs local_cpulist of the GPU's PCI function) so that the pinned slab of the
    e2e leg is first-touched on the GPU's NUMA node and the H2D copy does not cross the socket link.  Returns (old affinity, info)."""
    try:
        p = torch.cuda.get_device_properties(local)
        bdf = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        base = "/sys/bus/pci/devices/" + bdf
        node = int(open(base + "/numa_node").read().strip())
        cpus = set()
        for part in open(base + "/local_cpulist").read().strip().split(","):
            if "-" in part:
                a, b = part.split("-"); cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        old = os.sched_getaffinity(0)
        use = cpus & old
        if not use:
            return None, {"pci": bdf, "numa_node": node, "bound": False, "why": "no allowed CPU on that node"}
        os.sched_setaffinity(0, use)
        return old, {"pci": bdf, "numa_node": node, "bound": True, "cpus": len(use)}
    except Exception as e:  # noqa: BLE001
        return None, {"bound": False, "why": "%s: %s" % (type(e).__name__, e)}


class ClockSampler(threading.Thread):
    """nvidia-smi style clock / throttle-reason samples during the timed region (pynvml)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples, self.reasons = index, False, [], set()
        self.max_mhz = None
        self.armed = False                 # only samples taken while armed (the timed region) count
        self.ready = threading.Event()     # NVML is initialised: the first sample can be taken at once

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {
                getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
                getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
                getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
                getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            }
            self.ready.set()
            while not self.stop_flag:
                if not self.armed:
                    time.sleep(0.0005)
                    continue
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
                time.sleep(0.002)
        except Exception as e:  # noqa: BLE001
            self.reasons.add("sampler_error:%s" % type(e).__name__)
            self.ready.set()

    def result(self):
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ============================================================================================== CPU arm (oracle)
def oracle_4fsk_inputs(n_threads, t_samples):
    """Per-thread 4FSK-2k-FM bursts made by the ORACLE's own modulator (the reference arm never touches the product library)."""
    from oracle import oracle as O
    rng = np.random.default_rng(1000)
    data = np.concatenate([np.full(8, 0xAA, np.uint8)] +
                          [np.concatenate([np.array([0xED, 0x89, 0xAA], np.uint8), rng.integers(0, 256, 7, dtype=np.uint8)])
                           for _ in range(t_samples // 40000 + 2)])
    base = O.Tx(O.MOD_4FSK, 25, 1000000, 1700, 3500, 1).work(data)[:t_samples]
    if len(base) < t_samples:
        base = np.concatenate([base, np.zeros(t_samples - len(base), np.complex64)])
    xs = []
    for i in range(n_threads):
        noise = (rng.standard_normal(t_samples) + 1j * rng.standard_normal(t_samples)) * 0.04
        xs.append((0.8 * np.roll(base, 37 * i) + noise).astype(np.complex64))
    return xs


def cpu_rate(make_worker, n_threads, seconds, units_per_iter):
    """n_threads threads, each with its own oracle object, loop `iter()` until `seconds` elapse; returns units/s/1e6, wall time.
    (ctypes releases the GIL inside the oracle calls, so the threads really run in parallel.)"""
    done = [0] * n_threads
    t_end = [0.0]
    workers = [make_worker(i) for i in range(n_threads)]

    def run(i):
        w = workers[i]
        while time.perf_counter() < t_end[0]:
            w()
            done[i] += units_per_iter

    t_end[0] = time.perf_counter() + min(0.5, seconds / 4)       # warm-up pass
    th = [threading.Thread(target=run, args=(i,)) for i in range(n_threads)]
    [t.start() for t in th]; [t.join() for t in th]
    done[:] = [0] * n_threads
    t0 = time.perf_counter()
    t_end[0] = t0 + seconds
    th = [threading.Thread(target=run, args=(i,)) for i in range(n_threads)]
    [t.start() for t in th]; [t.join() for t in th]
    dt = time.perf_counter() - t0
    return sum(done) / dt / 1e6, dt


def cpu_rx_chain_rate(kind, args, xs, seconds, n_threads):
    from oracle import oracle as O
    O.lib()

    def mk(i):
        rx = O.Rx(kind, *args)
        x = xs[i % len(xs)]
        nports = 2 if kind in (O.DEMOD_NBFM,) else 3

        def it():
            rx.work(x)
            for p in range(nports):
                rx.port(p)
        return it
    return cpu_rate(mk, n_threads, seconds, len(xs[0]))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cores, core_info = host_cores()
    from oracle import oracle as O
    t_s = 1 << 20
    xs = oracle_4fsk_inputs(min(cores, 16), t_s)
    rates = []
    for i in range(args.warmup + args.steps):
        # one step = a bounded sample of the workload: every usable host thread demodulates 2^20-sample chunks of its own channel
        r, dt = cpu_rx_chain_rate(O.DEMOD_4FSK, (5, 1000000, 1700, 3000, 1), xs, 1.0, cores)
        if i >= args.warmup:
            rates.append((r, dt))
    v = float(np.mean([r for r, _ in rates]))
    sample = ("%d host threads (affinity/cgroup: %s), one channel per thread, 2^20-sample chunks of the 4FSK-2k-FM RX chain for ~1 s per "
              "step; CPU oracle port of the reference GNU Radio chain (GNU Radio/VOLK not installable here)" % (cores, json.dumps(core_info)))
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "Msamples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": float(np.mean([dt for _, dt in rates]) * 1e3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": headline_config(world),
        "cpu_baseline": {"value": v, "unit": "Msamples/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ============================================================================================== GPU arm helpers
def timed_calls(fn, k, stream, torch, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(k):
        fn()
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / k



def latency_bound_block(kernel, what, stage_ms_per_call, items_per_channel_per_call, clocks, chain_cycles, chain_source):
    """SURVEY 8d: the loop stages are latency bound -- what is reported for them is cycles of the loop-carried chain per item, live from the
    stage's CUDA-event time and the SM clock sampled under load, beside the chain's own schedule (the same recurrence alone in a
    kernel, tools/microbench/lone_warp.cu / ncu of the single launch: it runs at the sum of ptxas' stall counts)."""
    try:
        mhz = (clocks or {}).get("sm_mhz") or (clocks or {}).get("sm_max_mhz") or 1965
        cyc = stage_ms_per_call * 1e-3 * mhz * 1e6 / items_per_channel_per_call
        return {"kernel": kernel, "bound": "latency (loop-carried dependency chain, one warp per 32 channels)", "what": what,
                "items_per_channel_per_call": items_per_channel_per_call, "stage_ms_per_call": stage_ms_per_call, "sm_mhz": mhz,
                "cycles_per_item_in_step": cyc, "chain_cycles_alone": chain_cycles, "frac_of_chain_schedule": chain_cycles / cyc if cyc > 0 else None,
                "chain_source": chain_source}
    except Exception as e:  # noqa: BLE001
        return {"kernel": kernel, "error": "%s: %s" % (type(e).__name__, e)}

def rx_stage_ms(L, blk, names=("stage1_fir", "chan_filter", "demod_or_loop", "symbol_sync_or_audio", "viterbi", "soft_epilogue")):
    out = {}
    for s, name in enumerate(names):
        m, n = Ct.c_double(), Ct.c_long()
        L.qrl_rx_profile_read(blk._h, s, Ct.byref(m), Ct.byref(n))
        out[name] = (m.value, n.value)
    return out


DUMP_BUDGET = 63 << 20      # array bytes; the .npy headers, counts and channel list stay inside the last MB of 64 MB


def dump_outputs(blk, out_dir):
    """What the step's last qrl_rx_work call left on every output port, i.e. what read_port() hands a caller (each call replaces
    the ports; the state carried from all earlier calls is in them), as float32 DIR/port<p>.npy: the channels' items back to back,
    [items] for bit and float ports, [items, 2] (I, Q) for complex ones; DIR/counts.npy (float64 [ports, channels]) holds each
    channel's item count, so channel i of port p is the counts[p, i] items after the first sum(counts[p, :i]).  Channels whose ports
    do not all fit DUMP_BUDGET are left out by a fixed seeded draw; DIR/channels.npy lists the ones written."""
    ports = [blk.read_port(p) for p in range(blk.nports)]
    C = blk.n_channels
    bytes_per_channel = sum(max(len(v) for v in port) * (8 if port[0].dtype == np.complex64 else 4) for port in ports)
    n_keep = min(C, DUMP_BUDGET // max(1, bytes_per_channel))
    chans = np.arange(C) if n_keep == C else np.sort(np.random.default_rng(0).choice(C, n_keep, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "channels.npy"), chans.astype(np.float64))
    np.save(os.path.join(out_dir, "counts.npy"), np.array([[len(port[c]) for c in chans] for port in ports], np.float64))
    for p, port in enumerate(ports):
        a = np.concatenate([port[c] for c in chans])
        a = a.view(np.float32).reshape(-1, 2) if a.dtype == np.complex64 else a.astype(np.float32)
        np.save(os.path.join(out_dir, "port%d.npy" % p), a)


def parity_bits(blk, X, oracle_kind, oracle_args, channels, port=2, float_port=0):
    """Spot check on the buffers that were just timed: channels `channels` of X through the CPU oracle, decoded bits must be
    identical to what the GPU produced for the same call (fresh handles on both sides are compared by the caller)."""
    from oracle import oracle as O
    got_bits = blk.read_port(port)
    got_f = blk.read_port(float_port)
    res = {"channels": list(map(int, channels)), "bits_equal": True, "bits_compared": 0, "float_rms_max": 0.0}

    def one(c):
        rx = O.Rx(oracle_kind, *oracle_args)
        rx.work(X[c].cpu().numpy())
        return rx.port(port), rx.port(float_port)
    outs = {}
    th = [threading.Thread(target=lambda c=c: outs.__setitem__(c, one(c))) for c in channels]
    [t.start() for t in th]; [t.join() for t in th]
    for c in channels:
        wb, wf = outs[c]
        res["bits_equal"] = bool(res["bits_equal"] and len(wb) == len(got_bits[c]) and np.array_equal(wb, got_bits[c]))
        res["bits_compared"] += int(len(wb))
        if len(wf) and len(wf) == len(got_f[c]):
            rms = float(np.sqrt(np.mean(np.abs(got_f[c] - wf) ** 2)) / max(1e-30, np.sqrt(np.mean(np.abs(wf) ** 2))))
            res["float_rms_max"] = max(res["float_rms_max"], rms)
        else:
            res["bits_equal"] = False
    return res


def qpsk_inputs(q, torch, dev, C, T, seed):
    """[C][T] QPSK-250k bursts made by the product's own modulator on the GPU (x0.5) + AWGN."""
    rng = np.random.default_rng(seed)
    nb = T // 32
    tx = q.make_gr_mod_qpsk(4, 1000000, 1700, 160000, n_channels=C, max_items=nb, device=dev.index)
    d = torch.from_numpy(rng.integers(0, 256, (C, nb), dtype=np.uint8)).to(dev)
    tx.work_device(d.data_ptr(), nb, nb); tx.sync()
    L = q.load_library()
    Xt = torch.empty((C, nb * 32), dtype=torch.complex64, device=dev)
    n2 = Ct.c_long()
    assert L.qrl_tx_read(tx._h, Ct.c_void_p(Xt.data_ptr()), nb * 32, Ct.byref(n2), 1) == 0
    X = (Xt[:, :T] * 0.5).contiguous()
    X += torch.view_as_complex(torch.randn((C, T, 2), device=dev) * 0.03)
    tx.close()
    return X


def nbfm_inputs(torch, dev, C, T):
    n_ = torch.arange(T, device=dev, dtype=torch.float64)
    audio = 0.6 * torch.sin(2 * np.pi * 1000.0 * n_ / 1e6) + 0.4 * torch.sin(2 * np.pi * 2200.0 * n_ / 1e6)
    ph = 2 * np.pi * 2000.0 * torch.cumsum(audio, 0) / 1e6
    x = (0.8 * torch.polar(torch.ones_like(ph), ph)).to(torch.complex64)
    X = x.repeat(C, 1).contiguous()
    X += torch.view_as_complex(torch.randn((C, T, 2), device=dev) * 0.01)
    return X


def rx_config_block(q, torch, dev, name, make, make_args, okind, oargs, X, alg_bytes, kernel_name, k, cpu_seconds, cores,
                    float_port=0, bits_port=2, parity_ch=(0, 1, 2), cpu_threads=None):
    """value / roofline / cpu_baseline / parity for one RX configuration, inputs resident in HBM."""
    L = q.load_library()
    C, T = X.shape
    peak, _ = peaks()
    stream = torch.cuda.current_stream()
    blk = make(*make_args, n_channels=C, max_samples=T, device=dev.index)
    blk.set_stream(stream.cuda_stream)
    blk.work_device(X.data_ptr(), T, T)
    torch.cuda.synchronize()
    parity = None
    if okind is not None:
        if bits_port is None:
            parity = parity_float(blk, X, okind, oargs, [c for c in parity_ch if c < C], float_port)
        else:
            parity = parity_bits(blk, X, okind, oargs, [c for c in parity_ch if c < C], bits_port, float_port)
    L.qrl_rx_profile(blk._h, 1)
    ms = timed_calls(lambda: blk.work_device(X.data_ptr(), T, T), k, stream, torch, warm=1)
    st = rx_stage_ms(L, blk)
    L.qrl_rx_profile(blk._h, 0)
    fir_ms, fir_n = st["stage1_fir"]
    fir_avg = fir_ms / max(1, fir_n)
    per_call = max(1, fir_n // (k + 1))
    alg = alg_bytes * C * T / per_call
    res = {"workload": name, "channels": C, "samples_per_channel_per_call": T, "ms_per_call": ms,
           "value": C * T / ms / 1e3, "unit": "Msamples/s", "realtime_factor_per_channel": T / ms / 1e3,
           "stage_ms_per_call": {n: v[0] / (k + 1) for n, v in st.items()},
           "roofline": {"kernel": kernel_name, "bound": "hbm", "achieved": alg / (fir_avg * 1e-3) / 1e9 if fir_avg > 0 else 0.0,
                        "peak": peak, "unit": "GB/s", "frac": (alg / (fir_avg * 1e-3) / 1e9 / peak) if fir_avg > 0 else 0.0,
                        "algorithmic_bytes_per_launch": alg, "avg_launch_ms": fir_avg, "launches_per_call": per_call,
                        "whole_chain_frac": alg_bytes * C * T / (ms * 1e-3) / 1e9 / peak},
           "parity_vs_oracle": parity}
    if cpu_seconds > 0 and okind is not None:
        nthr = cpu_threads or cores
        xs = [X[c % C, : 1 << 20].cpu().numpy().copy() for c in range(min(nthr, 8))]
        v, dt = cpu_rx_chain_rate(okind, oargs, xs, cpu_seconds, nthr)
        res["cpu_baseline"] = {"value": v, "unit": "Msamples/s", "cores": nthr, "kind": "port",
                               "sample": "%d host threads x 2^20-sample chunks of the same chain (CPU oracle port) for %.1f s" % (nthr, dt)}
        res["gpu_over_cpu"] = res["value"] / v if v > 0 else None
    blk.close()
    return res


def parity_float(blk, X, oracle_kind, oracle_args, channels, float_port):
    from oracle import oracle as O
    res = {"channels": list(map(int, channels)), "float_rms_max": 0.0, "items_compared": 0, "lengths_equal": True}
    for port in (0, float_port):
        got = blk.read_port(port)
        for c in channels:
            rx = O.Rx(oracle_kind, *oracle_args)
            rx.work(X[c].cpu().numpy())
            w = rx.port(port)
            if len(w) != len(got[c]) or len(w) == 0:
                res["lengths_equal"] = False
                continue
            rms = float(np.sqrt(np.mean(np.abs(got[c] - w) ** 2)) / max(1e-30, np.sqrt(np.mean(np.abs(w) ** 2))))
            res["float_rms_max"] = max(res["float_rms_max"], rms)
            res["items_compared"] += int(len(w))
        if float_port == 0:
            break
    return res


def tx_config_block(q, torch, dev, cores, cpu_seconds):
    """BASELINE config 5: 64 ch 4FSK TX (1024 bytes/ch -> 4 096 000 output samples/ch at 1 Msps), IQ compared with the oracle."""
    from oracle import oracle as O
    L = q.load_library()
    peak, _ = peaks()
    C, n = 64, 1024
    rng = np.random.default_rng(5000)
    stream = torch.cuda.current_stream()
    tx = q.make_gr_mod_4fsk(25, 1000000, 1700, 3500, True, n_channels=C, max_items=n)
    tx.set_stream(stream.cuda_stream)
    data_h = rng.integers(0, 256, (C, n), dtype=np.uint8)
    data = torch.from_numpy(data_h).to(dev)
    nout = n * 4000
    # parity on the first call of a fresh handle: 3 channels, full length, against the oracle's modulator
    tx.work_device(data.data_ptr(), n, n); tx.sync()
    out = torch.empty((C, nout), dtype=torch.complex64, device=dev)
    n2 = Ct.c_long()
    assert L.qrl_tx_read(tx._h, Ct.c_void_p(out.data_ptr()), nout, Ct.byref(n2), 1) == 0 and n2.value == nout
    rms_max, ident = 0.0, True
    for c in (0, 31, 63):
        w = O.Tx(O.MOD_4FSK, 25, 1000000, 1700, 3500, 1).work(data_h[c])
        g = out[c].cpu().numpy()
        ident = ident and len(w) == len(g) and np.array_equal(w.view(np.float32), g.view(np.float32))
        if len(w) == len(g):
            rms_max = max(rms_max, float(np.sqrt(np.mean(np.abs(g - w) ** 2)) / np.sqrt(np.mean(np.abs(w) ** 2))))
    del out
    L.qrl_tx_profile(tx._h, 1)
    k = 10
    ms = timed_calls(lambda: tx.work_device(data.data_ptr(), n, n), k, stream, torch, warm=1)
    m, cnt = Ct.c_double(), Ct.c_long()
    L.qrl_tx_profile_read(tx._h, 2, Ct.byref(m), Ct.byref(cnt))
    st = {}
    for s, nm in enumerate(("bit_chain", "shape_fm", "interp_fir")):
        mm, cc = Ct.c_double(), Ct.c_long()
        L.qrl_tx_profile_read(tx._h, s, Ct.byref(mm), Ct.byref(cc))
        st[nm] = mm.value / (k + 1)
    L.qrl_tx_profile(tx._h, 0)
    per_call = max(1, cnt.value // (k + 1))
    avg = m.value / max(1, cnt.value)
    alg = 8.0 * C * nout / per_call
    res = {"workload": "64ch 4FSK-2k-FM TX (make_gr_mod_4fsk(25,1e6,1700,3500,true)): scrambler + CCSDS encoder + RRC x25 + FM + x20 interpolating FIR (689 taps)",
           "channels": C, "out_samples_per_channel_per_call": nout, "ms_per_call": ms, "value": C * nout / ms / 1e3, "unit": "Msamples/s (output)",
           "stage_ms_per_call": st,
           "roofline": {"kernel": "interp_fir_ccf_rt_kernel<20,35,8,16>", "bound": "hbm", "achieved": alg / (avg * 1e-3) / 1e9 if avg > 0 else 0.0,
                        "peak": peak, "unit": "GB/s", "frac": (alg / (avg * 1e-3) / 1e9 / peak) if avg > 0 else 0.0,
                        "algorithmic_bytes_per_launch": alg, "avg_launch_ms": avg, "launches_per_call": per_call,
                        "whole_chain_frac": 8.0 * C * nout / (ms * 1e-3) / 1e9 / peak},
           "parity_vs_oracle": {"channels": [0, 31, 63], "iq_bit_identical": bool(ident), "iq_rms_max": rms_max, "samples_compared": 3 * nout}}
    if cpu_seconds > 0:
        def mk(i):
            t = O.Tx(O.MOD_4FSK, 25, 1000000, 1700, 3500, 1)
            d = data_h[i % C][:256]
            return lambda: t.work(d)
        v, dt = cpu_rate(mk, cores, cpu_seconds, 256 * 4000)
        res["cpu_baseline"] = {"value": v, "unit": "Msamples/s (output)", "cores": cores, "kind": "port",
                               "sample": "%d host threads x 256-byte bursts through the oracle's 4FSK modulator for %.1f s" % (cores, dt)}
        res["gpu_over_cpu"] = res["value"] / v if v > 0 else None
    tx.close()
    return res


def pfb_config_block(q, torch, dev, cores, cpu_seconds):
    """SURVEY 8f row 1: pfb_channelizer_ccf(10, 341-tap prototype), wideband stream resident in HBM (16 algorithmic B/sample)."""
    from oracle import oracle as O
    L = q.load_library()
    peak, _ = peaks()
    M, n_t = 10, 341
    taps = np.zeros(n_t, np.float32)
    assert L.qrl_firdes_low_pass_2(1.0, 250000.0, 5000.0, 2000.0, 60.0, 5, taps.ctypes.data_as(Ct.c_void_p), n_t) == n_t
    stream = torch.cuda.current_stream()
    N = 1 << 27
    x = torch.view_as_complex(torch.randn((N, 2), device=dev) * 0.3)
    ch = q.PfbChannelizer(M, taps, max_in=N)
    ch.set_stream(stream.cuda_stream)
    # parity: first 2^20 wideband samples of a fresh handle against the oracle channelizer (float tolerance 1e-5 RMS)
    n_chk = 1 << 20
    y = ch.work(x[:n_chk].cpu().numpy())
    w = O.PfbChannelizer(M, taps).work(x[:n_chk].cpu().numpy())
    ncol = min(y.shape[1], w.shape[1])
    rms = float(np.sqrt(np.mean(np.abs(y[:, :ncol] - w[:, :ncol]) ** 2)) / np.sqrt(np.mean(np.abs(w[:, :ncol]) ** 2)))
    ch.close()
    ch = q.PfbChannelizer(M, taps, max_in=N)
    ch.set_stream(stream.cuda_stream)
    ms = timed_calls(lambda: ch.work_device(x.data_ptr(), N), 5, stream, torch, warm=2)
    res = {"workload": "pfb_channelizer_ccf(10, 341 taps) behind stream_to_streams(10) (gr_demod_mmdvm_multi2.cpp:98-107)", "wideband_samples_per_call": N,
           "ms_per_call": ms, "value": N / ms / 1e3, "unit": "Msamples/s (wideband)",
           "roofline": {"kernel": "pfb_channelizer_m10_kernel", "bound": "hbm", "achieved": 16.0 * N / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                        "frac": 16.0 * N / (ms * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_launch": 16.0 * N, "avg_launch_ms": ms,
                        "fp32_tflops": 2 * (2 * 35 + 4 * M) * N / ms / 1e9},
           "parity_vs_oracle": {"wideband_samples": n_chk, "columns_compared": int(ncol), "rms": rms, "tolerance": 1e-5}}
    ch.close()
    if cpu_seconds > 0:
        xh = x[: 1 << 18].cpu().numpy()

        def mk(i):
            c = O.PfbChannelizer(M, taps)
            return lambda: c.work(xh)
        v, dt = cpu_rate(mk, cores, cpu_seconds, len(xh))
        res["cpu_baseline"] = {"value": v, "unit": "Msamples/s (wideband)", "cores": cores, "kind": "port",
                               "sample": "%d host threads x 2^18-sample chunks through the oracle channelizer for %.1f s" % (cores, dt)}
        res["gpu_over_cpu"] = res["value"] / v if v > 0 else None
    del x
    return res


def spectrum_config_block(q, torch, dev, cores, cpu_seconds):
    """SURVEY 8f row 4: rx_fft_c (32768 points, Blackman-Harris) for 64 streams at once, samples resident in HBM.  One call = N + 1 samples
    per stream after a get: fill, window, FFT, dB, shift.  Algorithmic bytes per spectrum: 8 N read + 4 N written."""
    from oracle import oracle as O
    peak, _ = peaks()
    S, N = 64, 32768
    stream = torch.cuda.current_stream()
    x = torch.view_as_complex(torch.randn((S, 2 * N, 2), device=dev) * 0.2)
    x += 0.3 * torch.polar(torch.ones(2 * N, device=dev), 2 * np.pi * 0.1234 * torch.arange(2 * N, device=dev))
    sp = q.Spectrum(N, 5, n_streams=S, max_samples=2 * N)
    sp.set_stream(stream.cuda_stream)
    sp.set_enabled(True)
    out = torch.empty((S, N), dtype=torch.float32, device=dev)
    L = q.load_library()
    nfft = Ct.c_uint()

    def call():
        sp.work_device(x.data_ptr(), N + 1, x.shape[1])
        assert L.qrl_spectrum_get(sp._h, Ct.c_void_p(out.data_ptr()), N, 1, Ct.byref(nfft)) == 0 and nfft.value == N

    call()
    o = O.Spectrum(N, O.WIN_BLACKMAN_HARRIS); o.set_enabled(True)
    o.work(x[5, :N + 1].cpu().numpy())
    want, got = o.get(), out[5].cpu().numpy()
    ag, aw = 10.0 ** (got.astype(np.float64) / 20), 10.0 ** (want.astype(np.float64) / 20)
    ms = timed_calls(call, 20, stream, torch, warm=3)
    alg = 12.0 * N * S
    res = {"workload": "rx_fft_c(32768, Blackman-Harris) x 64 streams: fill + window + four-step FFT + power spectrum (dB) + fft-shift, and the D2D get",
           "ms_per_call": ms, "value": S / (ms * 1e-3), "unit": "spectra/s",
           "roofline": {"kernel": "spectrum_pass_a_kernel + spectrum_pass_b_kernel", "bound": "hbm", "achieved": alg / (ms * 1e-3) / 1e9, "peak": peak,
                        "unit": "GB/s", "frac": alg / (ms * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_launch": alg, "avg_launch_ms": ms,
                        "note": "whole call (5 launches + a D2D copy), not one kernel: 25 MB of algorithmic traffic per call is launch-latency territory"},
           "parity_vs_oracle": {"stream": 5, "max_db_err_within_40db_of_peak": float(np.max(np.abs(got - want)[want > want.max() - 40])),
                                "amplitude_rms_rel": float(np.sqrt(np.mean((ag - aw) ** 2)) / np.sqrt(np.mean(aw ** 2))), "tolerance_rms": 1e-5}}
    sp.close()
    if cpu_seconds > 0:
        xh = x[0, :N + 1].cpu().numpy()

        def mk(i):
            c = O.Spectrum(N, O.WIN_BLACKMAN_HARRIS); c.set_enabled(True)
            buf = np.empty(N, np.float32)

            def it():
                c.work(xh); c.get()
            return it
        v, dt = cpu_rate(mk, cores, min(cpu_seconds, 2.0), 1)
        res["cpu_baseline"] = {"value": v * 1e6, "unit": "spectra/s", "cores": cores, "kind": "port",
                               "sample": "%d host threads, one 32768-point spectrum per iteration through the oracle (double-precision radix-2) for %.1f s" % (cores, dt)}
    return res


def mmdvm_config_block(q, torch, dev, cores, cpu_seconds):
    """gr_demod_mmdvm_multi2 without its protocol sink: 250 ksps wideband -> pfb_channelizer(10) -> 7 x (24/25 resampler, low-pass, RSSI,
    discriminator, int16), everything resident in HBM.  Batched over `B` independent wideband streams by running B handles back to back
    would only repeat the number: one stream, long call."""
    from oracle import oracle as O
    from qradiolink_b200.mmdvm import _low_pass_2
    L = q.load_library()
    peak, _ = peaks()
    stream = torch.cuda.current_stream()
    N = 1 << 26
    x = torch.view_as_complex(torch.randn((N, 2), device=dev) * 0.05)
    tt = torch.arange(N, device=dev, dtype=torch.float64)
    for p in (0, 1, 2, 3, 9, 8, 7):
        f = p * 25000.0 if p < 5 else (p - 10) * 25000.0
        x += (0.1 * torch.polar(torch.ones(N, device=dev, dtype=torch.float64), 2 * np.pi * ((f + 900.0) * tt / 250000.0 % 1.0))).to(torch.complex64)
    dem = q.MmdvmDemod(7, 5000, max_in=N)
    dem.channelizer.set_stream(stream.cuda_stream); dem.channels.set_stream(stream.cuda_stream)
    cnt = Ct.c_long()

    def call():
        pf = dem.channelizer
        assert L.qrl_pfb_work(pf._h, Ct.c_void_p(x.data_ptr()), N, 0, 1, Ct.byref(cnt)) == 0
        ptr, stride, items = pf.out_device()
        dem.channels.work_device(ptr, items, stride)

    ms = timed_calls(call, 5, stream, torch, warm=2)
    # parity on the head of a fresh stream
    n_chk = 1 << 20
    d2 = q.MmdvmDemod(7, 5000, max_in=n_chk)
    xh = x[:n_chk].cpu().numpy()
    got = d2.work(xh)[0]
    taps = _low_pass_2(L, 1, 250000, 5000, 2000, 60)
    chan = O.PfbChannelizer(10, taps).work(xh)
    ok = True
    for c, p in enumerate(q.mmdvm_port_map(7)):
        want = O.MmdvmRx(5000).work(chan[p])[0]
        m = min(got.shape[1], len(want))
        ok = ok and bool(np.array_equal(got[c, :m], want[:m]))
    d2.close()
    alg = (8.0 + 7 * 0.096 * 2) * N             # 8 B per wideband sample in, 7 x int16 at 24 / 250 of the rate out
    res = {"workload": "gr_demod_mmdvm_multi2 up to gr_mmdvm_sink: pfb_channelizer_ccf(10, 341 taps) + 7 x (rational_resampler 24/25 (819 taps), 33-tap low-pass, RSSI, quadrature demod, float_to_short), 250 ksps wideband",
           "wideband_samples_per_call": N, "ms_per_call": ms, "value": N / ms / 1e3, "unit": "Msamples/s (wideband)",
           "real_time_factor": N / ms / 1e3 * 1e6 / 250000.0,
           "roofline": {"kernel": "pfb_channelizer_m10_kernel (+ the per-channel kernels)", "bound": "hbm", "achieved": alg / (ms * 1e-3) / 1e9, "peak": peak,
                        "unit": "GB/s", "frac": alg / (ms * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_launch": alg, "avg_launch_ms": ms,
                        "note": "whole chain; the channelizer is FP32-pipe bound (see pfb_channelizer_m10)"},
           "parity_vs_oracle": {"wideband_samples": n_chk, "channels": 7, "int16_equal": ok}}
    dem.close()
    if cpu_seconds > 0:
        xs = x[: 1 << 18].cpu().numpy()

        def mk(i):
            ch = O.PfbChannelizer(10, taps)
            rxs = [O.MmdvmRx(5000) for _ in range(7)]
            ports = q.mmdvm_port_map(7)

            def it():
                y = ch.work(xs)
                for r, p in zip(rxs, ports):
                    r.work(y[p])
            return it
        v, dt = cpu_rate(mk, cores, min(cpu_seconds, 3.0), len(xs))
        res["cpu_baseline"] = {"value": v, "unit": "Msamples/s (wideband)", "cores": cores, "kind": "port",
                               "sample": "%d host threads x 2^18-sample wideband chunks through the oracle channelizer + 7 channel chains for %.1f s" % (cores, dt)}
        res["gpu_over_cpu"] = res["value"] / v if v > 0 else None
    del x
    return res


def mixed_config_block(q, torch, dev, dist, rank, world, synth, k=4):
    """BASELINE config 4: 1024 channels, ch % 3 -> {NBFM, 4FSK-FM, QPSK-250k}, T = 2^21, sharded by mode then by rank
    (qradiolink_b200.sharding): 128 channels per GPU = three handles per rank running concurrently on three streams.  With fewer than
    8 ranks the channel count scales with the ranks (weak scaling: 128 per GPU)."""
    from qradiolink_b200 import sharding
    T = 1 << 21
    total = 128 * world
    modes = [("nbfm", "4fsk", "qpsk")[c % 3] for c in range(total)]
    mine = sharding.shard_channels(modes, world, rank)
    streams = {m: torch.cuda.Stream(device=dev) for m in ("nbfm", "4fsk", "qpsk")}
    blocks, inputs = {}, {}
    for m in ("nbfm", "4fsk", "qpsk"):
        C = len(mine.get(m, []))
        if C == 0:
            continue
        if m == "nbfm":
            X = nbfm_inputs(torch, dev, C, T)
            blk = q.make_gr_demod_nbfm(125, 1000000, 1700, 2500, n_channels=C, max_samples=T, device=dev.index)
        elif m == "4fsk":
            bases = [synth.burst_4fsk(3000 + 97 * rank + i, T) for i in range(4)]
            X = synth.batch_on_device(bases, C, seed=777 + rank, device=dev)
            blk = q.make_gr_demod_4fsk(5, 1000000, 1700, 3000, True, n_channels=C, max_samples=T, device=dev.index)
        else:
            X = qpsk_inputs(q, torch, dev, C, T, 3000 + rank)
            blk = q.make_gr_demod_qpsk(2, 1000000, 1700, 160000, n_channels=C, max_samples=T, device=dev.index)
        blk.set_stream(streams[m].cuda_stream)
        blocks[m], inputs[m] = blk, X
    torch.cuda.synchronize()

    def step():
        for m, blk in blocks.items():
            blk.work_device(inputs[m].data_ptr(), T, T)

    main = torch.cuda.current_stream()
    for _ in range(2):
        step()
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for s in streams.values():
        s.wait_stream(main)
    e0.record(main)
    for s in streams.values():
        s.wait_stream(main)
    for _ in range(k):
        step()
    for s in streams.values():
        main.wait_stream(s)
    e1.record(main)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / k
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if dist:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    per_mode = {}
    for m, blk in blocks.items():
        s = streams[m]
        with torch.cuda.stream(s):
            per_mode[m] = {"channels": int(inputs[m].shape[0]),
                           "ms_per_call_alone": timed_calls(lambda: blk.work_device(inputs[m].data_ptr(), T, T), 2, s, torch, warm=0)}
    res = {"workload": "1024ch mixed NBFM / 4FSK-2k-FM / QPSK-250k RX (ch % 3), T=2^21 per call, sharded by mode then rank, 128 ch per GPU",
           "channels_total": total, "channels_this_rank": {m: len(v) for m, v in mine.items()}, "samples_per_channel_per_call": T,
           "ms_per_call": ms_max, "value": total * T / ms_max / 1e3, "unit": "Msamples/s", "n_gpus": world,
           "per_mode_on_rank0": per_mode, "collective": "none on the data path (per-GPU ingest); rank-0 fan-out / fan-in timed separately in `fanout`"}
    for blk in blocks.values():
        blk.close()
    return res, inputs


def fanout_block(torch, dev, dist, rank, world, n_ch=128, T=1 << 21):
    """north_star's optional rank-0 ingest: a [world*n_ch][T] slab on rank 0 is scattered to per-rank slices with grouped NCCL
    send/recv over NVLink, and per-channel results (here 1 KiB of decoded bits per channel-call) are gathered back.  Timed
    separately from the demodulation: with per-GPU ingest it is not on the path at all."""
    if not dist or world < 2:
        return None
    slab = torch.empty((n_ch, T), dtype=torch.complex64, device=dev)
    src = torch.randn((world * n_ch, 8), device=dev) if rank == 0 else None     # placeholder so rank 0 owns something real below
    full = None
    if rank == 0:
        full = torch.view_as_complex(torch.randn((world * n_ch, T // 8, 2), device=dev)).repeat(1, 8).contiguous()
    bits = torch.zeros((n_ch, 1024), dtype=torch.uint8, device=dev)
    gathered = torch.empty((world * n_ch, 1024), dtype=torch.uint8, device=dev) if rank == 0 else None
    del src

    def scatter():
        ops = []
        if rank == 0:
            slab.copy_(full[:n_ch])
            for r in range(1, world):
                ops.append(dist.P2POp(dist.isend, full[r * n_ch:(r + 1) * n_ch], r))
        else:
            ops.append(dist.P2POp(dist.irecv, slab, 0))
        if ops:
            for w in dist.batch_isend_irecv(ops):
                w.wait()

    def gather():
        ops = []
        if rank == 0:
            gathered[:n_ch].copy_(bits)
            for r in range(1, world):
                ops.append(dist.P2POp(dist.irecv, gathered[r * n_ch:(r + 1) * n_ch], r))
        else:
            ops.append(dist.P2POp(dist.isend, bits, 0))
        if ops:
            for w in dist.batch_isend_irecv(ops):
                w.wait()

    out = {}
    for name, fn, nbytes in (("scatter_iq", scatter, (world - 1) * n_ch * T * 8), ("gather_bits", gather, (world - 1) * n_ch * 1024)):
        fn(); torch.cuda.synchronize(); dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(3):
            fn()
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / 3], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        out[name] = {"ms": float(t.item()), "bytes_over_nvlink": int(nbytes), "GBps": nbytes / (float(t.item()) * 1e-3) / 1e9}
    del full, slab
    return out


# ============================================================================================== GPU arm
def run_ours(args):
    import torch
    import qradiolink_b200 as q
    from qradiolink_b200 import synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if q.device_count() < 1:
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        import datetime
        # a rank that dies must not leave the others waiting ten minutes on the box
        dist.init_process_group("nccl", device_id=torch.device("cuda", local), timeout=datetime.timedelta(seconds=180))
    dev = torch.device("cuda", local)
    cores, core_info = host_cores()

    C, T = CHANNELS, T_CALL
    bases = [synth.burst_4fsk(1000 + 97 * rank + i, T) for i in range(N_BASES)]
    X = synth.batch_on_device(bases, C, seed=4242 + rank, device=dev)
    torch.cuda.synchronize()

    stream = torch.cuda.Stream(device=dev)          # a real (non-null) stream shared by torch events and the library
    torch.cuda.set_stream(stream)
    L = q.load_library()

    # ---- parity spot check at full size on the buffer that is timed below (fresh handle, one call, 3 channels, oracle as checker)
    parity = None
    if rank == 0 and not args.no_parity:
        from oracle import oracle as O
        chk = q.make_gr_demod_4fsk(5, 1000000, 1700, 3000, True, n_channels=C, max_samples=T, device=local)
        chk.set_stream(stream.cuda_stream)
        chk.work_device(X.data_ptr(), T, T)
        parity = parity_bits(chk, X, O.DEMOD_4FSK, (5, 1000000, 1700, 3000, 1), [0, 21, 63])
        chk.close()

    blk = q.make_gr_demod_4fsk(5, 1000000, 1700, 3000, True, n_channels=C, max_samples=T, device=local)
    blk.set_stream(stream.cuda_stream)
    overlap = not args.no_overlap
    if overlap:
        # streaming use: the loop / FEC tail of call k runs under the parallel stages of call k+1 (QRL_PARAM_OVERLAP_CALLS);
        # qrl_rx_join before the closing event puts every call's tail inside the timed region
        blk.set_overlap(True)

    def step_device():
        for _ in range(CALLS_PER_STEP):
            blk.work_device(X.data_ptr(), T, T)

    sm_a, sm_b = Ct.c_int(), Ct.c_int()
    L.qrl_rx_sm_partition(blk._h, Ct.byref(sm_a), Ct.byref(sm_b))
    warm = max(args.warmup, 3)
    for _ in range(warm):
        step_device()
    torch.cuda.synchronize()
    n_bits = int(np.sum(blk.read_port_counts(2)))

    # ---- timed region: K steps
    L.qrl_rx_profile(blk._h, 1)
    launches0 = blk.launches
    sampler = ClockSampler(local)
    sampler.start()
    sampler.ready.wait(10.0)
    if dist:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.armed = True
    e0.record(stream)
    for _ in range(args.steps):
        step_device()
    blk.join()
    e1.record(stream)
    torch.cuda.synchronize()
    sampler.armed = False
    if dist:
        dist.barrier()
    sampler.stop_flag = True
    sampler.join()
    ms = e0.elapsed_time(e1)
    launches = blk.launches - launches0
    stage = rx_stage_ms(L, blk)
    L.qrl_rx_profile(blk._h, 0)
    t_ms = torch.tensor([ms], device=dev, dtype=torch.float64)
    if dist:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms_max = float(t_ms.item())
    n_calls = args.steps * CALLS_PER_STEP
    value = world * C * T * n_calls / (ms_max * 1e-3) / 1e6
    if args.dump_outputs and rank == 0:
        dump_outputs(blk, args.dump_outputs)

    # ---- e2e: the reference-facing call with HOST buffers: H2D of the gr_complex slab + D2H of the decoded bits, every call
    old_aff, numa = bind_to_gpu_numa(torch, local)
    Xh = torch.empty((C, T), dtype=torch.complex64, pin_memory=True)
    Xh.copy_(X)
    bits_cap = int(blk.read_port_counts(2).max()) + 256
    out_bits = torch.empty((C, bits_cap), dtype=torch.uint8, pin_memory=True)
    out_cnt = np.zeros(C, np.int32)
    e2e_calls = 6

    def call_host():
        rc = L.qrl_rx_work(blk._h, Ct.c_void_p(Xh.data_ptr()), T, T, 0)
        assert rc == 0
        rc = L.qrl_rx_read_port(blk._h, 2, Ct.c_void_p(out_bits.data_ptr()), bits_cap, out_cnt.ctypes.data_as(Ct.c_void_p), 0)
        assert rc == 0

    call_host()
    if dist:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    e0.record(stream)
    for _ in range(e2e_calls):
        call_host()
    e1.record(stream)
    torch.cuda.synchronize()
    e2e_ms = max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3)
    t2 = torch.tensor([e2e_ms], device=dev, dtype=torch.float64)
    if dist:
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
    e2e_value = world * C * T * e2e_calls / (float(t2.item()) * 1e-3) / 1e6
    del Xh

    # ---- the same end-to-end call fed with the SDR's wire format (int16 I/Q, 4 B per sample: qrl_rx_work_sc16), reported beside e2e
    e2e_sc16 = None
    try:
        Xq = torch.empty((C, T, 2), dtype=torch.int16, pin_memory=True)
        Xq.copy_(torch.view_as_real(X).mul(20000.0).round_().clamp_(-32768, 32767).to(torch.int16))
        sc = Ct.c_float(1.0 / 32767.0)

        def call_host16():
            rc = L.qrl_rx_work_sc16(blk._h, Ct.c_void_p(Xq.data_ptr()), T, T, sc, 0)
            assert rc == 0
            rc = L.qrl_rx_read_port(blk._h, 2, Ct.c_void_p(out_bits.data_ptr()), bits_cap, out_cnt.ctypes.data_as(Ct.c_void_p), 0)
            assert rc == 0

        call_host16()
        bits16 = int(out_cnt.sum())
        if dist:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        e0.record(stream)
        for _ in range(e2e_calls):
            call_host16()
        e1.record(stream)
        torch.cuda.synchronize()
        ms16 = max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3)
        t3 = torch.tensor([ms16], device=dev, dtype=torch.float64)
        if dist:
            dist.all_reduce(t3, op=dist.ReduceOp.MAX)
        e2e_sc16 = {"value": world * C * T * e2e_calls / (float(t3.item()) * 1e-3) / 1e6, "unit": "Msamples/s",
                    "h2d_bytes_per_call": int(C * T * 4), "decoded_bits_per_call": bits16,
                    "note": "qrl_rx_work_sc16: pinned int16 I/Q slab (x20000, the SDR's wire format) -> device conversion float(v)/32767 -> same chain"}
        del Xq
        # int8 I/Q (HackRF-class front ends): 2 B per sample
        X8 = torch.empty((C, T, 2), dtype=torch.int8, pin_memory=True)
        X8.copy_(torch.view_as_real(X).mul(100.0).round_().clamp_(-128, 127).to(torch.int8))
        sc8 = Ct.c_float(1.0 / 128.0)

        def call_host8():
            rc = L.qrl_rx_work_sc8(blk._h, Ct.c_void_p(X8.data_ptr()), T, T, sc8, 0)
            assert rc == 0
            rc = L.qrl_rx_read_port(blk._h, 2, Ct.c_void_p(out_bits.data_ptr()), bits_cap, out_cnt.ctypes.data_as(Ct.c_void_p), 0)
            assert rc == 0

        call_host8()
        bits8 = int(out_cnt.sum())
        if dist:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        e0.record(stream)
        for _ in range(e2e_calls):
            call_host8()
        e1.record(stream)
        torch.cuda.synchronize()
        ms8 = max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3)
        t4 = torch.tensor([ms8], device=dev, dtype=torch.float64)
        if dist:
            dist.all_reduce(t4, op=dist.ReduceOp.MAX)
        e2e_sc16["sc8"] = {"value": world * C * T * e2e_calls / (float(t4.item()) * 1e-3) / 1e6, "unit": "Msamples/s",
                           "h2d_bytes_per_call": int(C * T * 2), "decoded_bits_per_call": bits8,
                           "note": "qrl_rx_work_sc8: pinned int8 I/Q slab (x100) -> float(v)/128 on the device -> same chain"}
        del X8
    except Exception as e:  # noqa: BLE001
        e2e_sc16 = {"error": "%s: %s" % (type(e).__name__, e)}
    if old_aff is not None:
        os.sched_setaffinity(0, old_aff)
    blk.close()

    # ---- the other BASELINE configurations (config 4 on every rank; the single-GPU ones on rank 0 at N = 1)
    configs = {}
    if not args.headline_only:
        try:
            cfg4, _ = mixed_config_block(q, torch, dev, dist, rank, world, synth)
            fo = fanout_block(torch, dev, dist, rank, world)
            if fo:
                cfg4["fanout"] = fo
            configs["cfg4_mixed_1024ch_sharded"] = cfg4
        except Exception as e:  # noqa: BLE001
            configs["cfg4_mixed_1024ch_sharded"] = {"error": "%s: %s" % (type(e).__name__, e)}

    if rank != 0:
        if dist:
            dist.destroy_process_group()
        return

    if world == 1 and not args.headline_only:
        from oracle import oracle as O
        cs = 0.0 if args.no_cpu else 4.0
        try:
            Xn = nbfm_inputs(torch, dev, 1, 1 << 22)
            configs["cfg1_nbfm_1ch"] = rx_config_block(q, torch, dev, "1ch NBFM RX (make_gr_demod_nbfm(125,1e6,1700,2500)), T=2^22", q.make_gr_demod_nbfm,
                                                       (125, 1000000, 1700, 2500), O.DEMOD_NBFM, (125, 1000000, 1700, 2500), Xn, 8.16,
                                                       "fir_decim_poly_kernel<50,9,8,128,8>", 5, cs, cores, float_port=1, bits_port=None, parity_ch=(0,), cpu_threads=1)
            del Xn
            Xn = nbfm_inputs(torch, dev, 64, 1 << 22)
            configs["cfg1_nbfm_64ch"] = rx_config_block(q, torch, dev, "64ch NBFM RX (same block, batched), T=2^22", q.make_gr_demod_nbfm,
                                                        (125, 1000000, 1700, 2500), O.DEMOD_NBFM, (125, 1000000, 1700, 2500), Xn, 8.16,
                                                        "fir_decim_poly_kernel<50,9,8,128,8>", 3, cs, cores, float_port=1, bits_port=None, parity_ch=(0, 33, 63))
            del Xn
        except Exception as e:  # noqa: BLE001
            configs["cfg1_nbfm_1ch"] = {"error": "%s: %s" % (type(e).__name__, e)}
        try:
            Xq = qpsk_inputs(q, torch, dev, 256, 1 << 20, 2000)
            configs["cfg3_qpsk250k_256ch"] = rx_config_block(q, torch, dev, "256ch QPSK-250k RX (make_gr_demod_qpsk(2,1e6,1700,160000)): /2 FIR + RRC + agc2 + Costas + symbol sync + Costas + CCSDS Viterbi, T=2^20 per call",
                                                             q.make_gr_demod_qpsk, (2, 1000000, 1700, 160000), O.DEMOD_QPSK, (2, 1000000, 1700, 160000), Xq, 12.0,
                                                             "fir_decim2_kernel<56,8,128>", 3, cs, cores, float_port=1, bits_port=2, parity_ch=(0, 100, 255))
            del Xq
            sweep = {}
            for Cq in (1024, 4096):
                Xq = qpsk_inputs(q, torch, dev, Cq, 1 << 18, 2100 + Cq)
                r = rx_config_block(q, torch, dev, "QPSK-250k RX channel sweep", q.make_gr_demod_qpsk, (2, 1000000, 1700, 160000), None, None, Xq, 12.0,
                                    "fir_decim2_kernel<56,8,128>", 2, 0.0, cores)
                sweep[str(Cq)] = {"Msamples_per_s": r["value"], "ms_per_call": r["ms_per_call"], "samples_per_channel_per_call": 1 << 18}
                del Xq
            configs["cfg3_qpsk250k_256ch"]["channel_sweep"] = sweep
        except Exception as e:  # noqa: BLE001
            configs["cfg3_qpsk250k_256ch"] = {"error": "%s: %s" % (type(e).__name__, e)}
        try:
            configs["cfg5_4fsk_tx_64ch"] = tx_config_block(q, torch, dev, cores, cs)
        except Exception as e:  # noqa: BLE001
            configs["cfg5_4fsk_tx_64ch"] = {"error": "%s: %s" % (type(e).__name__, e)}
        try:
            configs["pfb_channelizer_m10"] = pfb_config_block(q, torch, dev, cores, cs)
        except Exception as e:  # noqa: BLE001
            configs["pfb_channelizer_m10"] = {"error": "%s: %s" % (type(e).__name__, e)}
        try:
            configs["mmdvm_demod_7ch"] = mmdvm_config_block(q, torch, dev, cores, cs)
        except Exception as e:  # noqa: BLE001
            configs["mmdvm_demod_7ch"] = {"error": "%s: %s" % (type(e).__name__, e)}
        try:
            configs["spectrum_32k_64streams"] = spectrum_config_block(q, torch, dev, cores, cs)
        except Exception as e:  # noqa: BLE001
            configs["spectrum_32k_64streams"] = {"error": "%s: %s" % (type(e).__name__, e)}
        try:
            # config 2 with more channels per GPU: the 64-channel step is the latency of two loop warps; the machine has room
            sweep = {}
            for Cs in (256, 1024):
                Xs = synth.batch_on_device(bases[:4], Cs, seed=99, device=dev) if Cs * T * 8 < 40e9 else None
                Ts = T
                if Xs is None:
                    continue
                b2 = q.make_gr_demod_4fsk(5, 1000000, 1700, 3000, True, n_channels=Cs, max_samples=Ts, device=local)
                b2.set_stream(stream.cuda_stream)
                b2.set_overlap(True)
                ms2 = timed_calls(lambda: b2.work_device(Xs.data_ptr(), Ts, Ts), 6, stream, torch, warm=3)
                b2.join(); torch.cuda.synchronize()
                sweep[str(Cs)] = {"Msamples_per_s": Cs * Ts / ms2 / 1e3, "ms_per_call": ms2,
                                  "whole_chain_frac_of_hbm_peak": ALG_BYTES_PER_SAMPLE * Cs * Ts / (ms2 * 1e-3) / 1e9 / peaks()[0]}
                b2.close(); del Xs
            configs["cfg2_channel_sweep"] = sweep
        except Exception as e:  # noqa: BLE001
            configs["cfg2_channel_sweep"] = {"error": "%s: %s" % (type(e).__name__, e)}

    # ---- roofline of the dominant kernel (stage-1 polyphase decimating FIR), live CUDA-event time
    peak, peak_src = peaks()
    fir_ms, fir_n = stage["stage1_fir"]
    fir_avg_s = fir_ms / max(1, fir_n) * 1e-3
    launches_per_call = max(1, fir_n // n_calls)
    alg_bytes = ALG_BYTES_PER_SAMPLE * C * T / launches_per_call
    achieved = alg_bytes / fir_avg_s / 1e9 if fir_avg_s > 0 else 0.0
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "fir_traffic_bytes.json")
    if os.path.exists(tp):      # ncu --set full capture (profiles/): DRAM bytes per input sample x samples per launch
        tj = json.load(open(tp))
        traffic = tj.get("per_sample") * C * T / launches_per_call
        traffic_src = tj.get("source")

    cpu_line = None
    if world == 1 and not args.no_cpu:
        from oracle import oracle as O
        xs = oracle_4fsk_inputs(min(cores, 16), 1 << 20)
        v, dt = cpu_rx_chain_rate(O.DEMOD_4FSK, (5, 1000000, 1700, 3000, 1), xs, 8.0, cores)
        cpu_line = {"value": v, "unit": "Msamples/s", "cores": cores, "kind": "port", "cores_detail": core_info,
                    "sample": "%d host threads, one channel per thread, 2^20-sample chunks of the same 4FSK-2k-FM chain (CPU oracle port) for %.0f s" % (cores, dt)}

    cfg = headline_config(world)
    line = {
        "metric": METRIC, "value": value, "unit": "Msamples/s", "n_gpus": world,
        "steps": args.steps, "warmup": warm, "ms_per_step": ms_max / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": cfg,
        "impl_notes": {"calls": ("overlapped: tail of call k under call k+1 (QRL_PARAM_OVERLAP_CALLS), joined before the closing event" if overlap else "serialised"),
                       "decoded_bits_per_call": n_bits, "sm_partition": {"loop_fec_sms": sm_a.value, "parallel_sms": sm_b.value},
                       "timed_region_s": ms_max * 1e-3, "ms_per_call": ms_max / n_calls},
        "clocks": sampler.result(),
        "e2e": {"value": e2e_value, "unit": "Msamples/s", "h2d_bytes_per_step": int(C * T * 8) * CALLS_PER_STEP,
                "d2h_bytes_per_step": int(C * bits_cap + 4 * C) * CALLS_PER_STEP,
                "measured_over_calls": e2e_calls, "h2d_bytes_per_call": int(C * T * 8), "d2h_bytes_per_call": int(C * bits_cap + 4 * C),
                "note": "pinned host slab -> qrl_rx_work (H2D inside the call) -> qrl_rx_read_port of the decoded bits (D2H), every call; PCIe-bound at 8 B/sample",
                "numa": numa, "sc16_ingest": e2e_sc16},
        "gpu_launches": int(launches),
        "roofline": {"kernel": "fir_decim_poly_kernel<50,9,8,128,8>", "bound": "hbm", "achieved": achieved, "peak": peak,
                     "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": alg_bytes, "avg_launch_ms": fir_avg_s * 1e3,
                     "launches_per_call": launches_per_call,
                     "whole_chain_frac": ALG_BYTES_PER_SAMPLE * C * T * n_calls / (ms_max * 1e-3) / 1e9 / peak},
        "stage_ms_per_call": {n: v[0] / n_calls for n, v in stage.items()},
        "parity_vs_oracle": parity,
        "configs": configs,
    }
    line["latency_bound"] = latency_bound_block(
        "symsync_kernel<1,SL_RECT4,EPI_EXT_4FSK_FM,512,2,1,LOOP_SYMSYNC,2>", "symbol_sync_ff recurrence (MMSE interpolation -> TED -> loop filter), the stage that IS the step",
        line["stage_ms_per_call"].get("symbol_sync_or_audio", 0.0), T / 500.0, line["clocks"], 203.0,
        "ncu --set full of one launch over the whole call, profiles/r02_final2_ncu_full_summary.csv: 891.7 us for 8613 symbols")
    try:
        c3 = configs.get("cfg3_qpsk250k_256ch")
        if isinstance(c3, dict) and "stage_ms_per_call" in c3:
            c3["latency_bound"] = latency_bound_block(
                "agc_costas_kernel<128,2,4,1>", "agc2_cc -> costas_loop_cc(order 4, snr) per sample at 500 ksps, the stage that bounds the QPSK chain",
                c3["stage_ms_per_call"].get("demod_or_loop", 0.0), c3["samples_per_channel_per_call"] / 2.0, line["clocks"], 202.6,
                "the Costas recurrence alone in a kernel, tools/microbench/lone_warp.cu, profiles/r02_t_symsync_prefetch_costas_select.txt")
    except Exception:  # noqa: BLE001
        pass
    if cpu_line:
        line["cpu_baseline"] = cpu_line
    print(json.dumps(line))
    if dist:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-overlap", action="store_true", help="serialise qrl_rx_work calls (no QRL_PARAM_OVERLAP_CALLS)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline legs (profiling runs)")
    ap.add_argument("--no-parity", action="store_true", help="skip the full-size parity spot checks")
    ap.add_argument("--headline-only", action="store_true", help="config 2 only (no `configs` block)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the output ports of the timed path's last "
                    "call to DIR/*.npy (float32, rank 0, at most 64 MB; inputs are seeded, so runs with the same arguments compare)")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
