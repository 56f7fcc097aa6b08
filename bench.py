#!/usr/bin/env python3
"""bench.py -- the divANS batched-decode benchmark (BASELINE.json metric: decompressed MB/s on batched 64 KiB streams).

  python bench.py [--gpus N] [--steps K] [--warmup W]            our arm (CUDA kernels through the C ABI)
  python bench.py --impl reference [...]                         the reference arm: the CPU decoder on the host cores

A "step" = one pass of the hot path over one batch: every rank decodes its shard of independent streams
(N = 1: BASELINE configs[1], 4096 x 64 KiB synthetic-text streams; N > 1: configs[2], 8192 streams per GPU -- weak scaling: the
per-GPU batch is fixed as N grows).
`value` times K steps with inputs resident in HBM (CUDA events on the launching stream, max over ranks);
`e2e` repeats the measurement through the host-buffer C-ABI call (pinned host memory, H2D + D2H inside the timed
region).  `roofline` is computed for the stream-decode kernel from its own CUDA-event time; `cpu_baseline` times the
CPU oracle (restatement of the reference algorithm; the Rust reference cannot be built in this image) on a bounded
sample of the same streams.  `populations` repeats the device-resident measurement for the other encodings of the same raw
streams (SURVEY 8d: L = literal-only, the headline; Z = LZ77 command streams; dynamic context mixing 2; UTF8 context mode), each
checked bit-exact against the raw input.  With N > 1, `scattered_e2e` times the sharded API (divans_b200.sharding.ShardedDecoder):
rank 0 owns the whole host batch, scatters it over NVLink, every rank decodes, rank 0 gathers.
  python bench.py --workload entropy       BASELINE configs[4]: 128 x 1 MiB Bernoulli streams per GPU, p in {0.5, 0.9, 0.99}
  python bench.py --dump-outputs DIR       also write what the last timed step decoded (rank 0) to DIR/*.npy, so that two builds
                                           can be compared output for output (the inputs are seeded: same arguments, same inputs)
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

STREAM_BYTES = 65536
STREAMS_PER_GPU = 4096           # N = 1 (BASELINE configs[1])
STREAMS_PER_GPU_SCALING = 8192   # N > 1 (BASELINE configs[2]: 65536 streams at 8 GPUs)
DUMP_STREAMS = 128               # --dump-outputs: 128 x 64 KiB decoded bytes as float32 = 32 MiB (all 4096 would be 1 GiB)
METRIC = "decompressed MB/s (batched 64KiB streams)"
UNIT = "MB/s"


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """SM clock / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe): NVML in-process every
    ~10 ms when nvidia_ml_py is importable, else the `nvidia-smi --query-gpu` line the recipe gives (one call ~0.1 s)."""

    def __init__(self, index, uuid=None):
        super().__init__(daemon=True)
        self.index, self.uuid, self.samples, self._halt = index, uuid, [], threading.Event()
        self.source = "nvidia-smi"
        self.q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
                  "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        self._nv = None
        try:
            import pynvml
            pynvml.nvmlInit()
            h = None
            if uuid:
                try:
                    h = pynvml.nvmlDeviceGetHandleByUUID(uuid if isinstance(uuid, bytes) else str(uuid).encode())
                except Exception:
                    h = None
            if h is None:
                h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self._max = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
            self._nv, self._h, self.source = pynvml, h, "nvml"
        except Exception:
            self._nv = None

    def _nvml_sample(self):
        nv = self._nv
        mhz = float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
        try:
            bits = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self._h))
        except Exception:
            bits = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h))
        act = lambda m: "Active" if bits & m else "Not Active"   # nvml.h: SwPowerCap 0x4, HwSlowdown 0x8, SwThermal 0x20, HwThermal 0x40
        return [str(mhz), str(self._max), "", act(0x8), act(0x40), act(0x20), act(0x4)]

    def run(self):
        while not self._halt.is_set():
            try:
                if self._nv is not None:
                    self.samples.append(self._nvml_sample())
                    self._halt.wait(0.01)
                    continue
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                self._nv = None if self._nv is not None and not self.samples else self._nv
            self._halt.wait(0.1)

    def stop(self):
        self._halt.set()
        self.join(timeout=6)
        sm, mx, reasons = [], 0, set()
        for s in self.samples:
            try:
                sm.append(float(s[0])); mx = max(mx, float(s[1]))
            except Exception:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], s[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm),
                "source": self.source}


def make_inputs(rank, n_streams, engine=None):
    """Synthetic-text streams of this rank's shard (seeded by global stream index) and their compressed form.
    Compression is done by the product's own GPU encoder when it is available; the oracle is only the CPU baseline."""
    from divans_b200 import synth
    blob, off, ln = synth.text_streams(n_streams, STREAM_BYTES, seed=0xD1FA15 + 7919 * rank)
    return blob, off, ln


def encode_inputs(blob, off, ln, engine):
    import divans_b200
    n = len(off)
    cap = np.full(n, STREAM_BYTES + STREAM_BYTES // 2 + 70144, np.uint64)
    eoff = np.arange(n, dtype=np.uint64) * cap[0]
    out = np.zeros(int(cap.sum()), np.uint8)
    out_len, status = engine.encode_batch_host(blob, off, ln, out, eoff, cap, divans_b200.encode_options())
    assert (status == 0).all()
    gen = "divans_b200 GPU encoder (divans_b200_encode_batch_host)"
    # compact to 16-byte aligned offsets
    pad = (out_len + np.uint64(15)) & ~np.uint64(15)
    coff = np.zeros(n, np.uint64)
    coff[1:] = np.cumsum(pad)[:-1]
    comp = np.zeros(int(pad.sum()) + 64, np.uint8)
    for i in range(n):
        comp[int(coff[i]): int(coff[i] + out_len[i])] = out[int(eoff[i]): int(eoff[i] + out_len[i])]
    return comp, coff, out_len.astype(np.uint64), gen


def _pin_all_cores():
    """the CPU arm uses every core the process may run on, and says so"""
    try:
        cores = sorted(os.sched_getaffinity(0))
        os.sched_setaffinity(0, cores)
        return len(cores)
    except Exception:
        return os.cpu_count() or 1


def _oracle_times(O, comp, coff, clen, off, ln, threads, reps):
    """seconds per pass (median of `reps`) of the oracle's threaded batch decoder over the given streams, after one warm pass
    (the per-thread prior tables are touched once: first-touch page placement is not what the arm measures)"""
    O.decode_batch(comp, coff, clen, off, ln, threads)
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out, out_len, status = O.decode_batch(comp, coff, clen, off, ln, threads)
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), out, status


def cpu_baseline(comp, coff, clen, raw_blob, off, ln, n_sample, threads):
    from oracle import oracle_py as O
    n = min(n_sample, len(coff))
    dt, out, status = _oracle_times(O, comp, coff[:n], clen[:n], off[:n], ln[:n], threads, 3)
    n1 = min(n, 48)
    dt1, _, _ = _oracle_times(O, comp, coff[:n1], clen[:n1], off[:n1], ln[:n1], 1, 1)
    ok = bool((status == 0).all() and (out[: n * STREAM_BYTES] == raw_blob[: n * STREAM_BYTES]).all())
    return {"value": n * STREAM_BYTES / dt / 1e6, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": "%d of the benchmark's 64 KiB streams, oracle decode_batch, median of 3 passes of %.2f s after a warm pass" % (n, dt),
            "single_thread_value": n1 * STREAM_BYTES / dt1 / 1e6, "bit_exact_vs_input": ok}, out


def run_reference_arm(args):
    """--impl reference: the reference's CPU implementation of the path (the oracle port: the Rust crate cannot be compiled in
    this image) on all host threads, same workload / metric.  Every step decodes the same fixed sample (2048 streams) after one
    untimed warm pass per thread pool; the line reports the MEDIAN step (a CPU arm on a shared host moves a lot between
    boxes: the median of >= 5 steps and the fixed sample are what keep it comparable) and the single-thread figure."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import oracle_py as O
    O.build()
    threads = _pin_all_cores()
    n_sample = int(os.environ.get("DIVANS_BENCH_REF_STREAMS", "2048"))
    blob, off, ln = make_inputs(0, n_sample)
    enc, eoff, elen = O.encode_batch(blob, off, ln, O.options(), threads)
    for _ in range(max(1, args.warmup)):
        O.decode_batch(enc, eoff, elen, off, ln, threads)
    steps = max(5, args.steps)
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        out, out_len, status = O.decode_batch(enc, eoff, elen, off, ln, threads)
        ts.append(time.perf_counter() - t0)
    assert (status == 0).all() and (out[: blob.size] == blob).all()
    dt = float(np.median(ts))
    n1 = min(n_sample, 48)
    dt1, _, _ = _oracle_times(O, enc, eoff[:n1], elen[:n1], off[:n1], ln[:n1], 1, 1)
    v = blob.size / dt / 1e6
    streams = args.streams or (STREAMS_PER_GPU if args.gpus == 1 else STREAMS_PER_GPU_SCALING)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup,
            "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "i16/u64",
            "data": "synthetic",
            "config": {"workload": "%d independent 64 KiB synthetic-text divANS streams per GPU (BASELINE configs[%d]), literal-only "
                                   "encoding (1 PredictionMode + 1 Literal command)" % (streams, 1 if args.gpus == 1 else 2),
                       "streams_per_gpu": streams, "stream_bytes": STREAM_BYTES,
                       "sample": "each step decodes the same fixed sample of %d of these streams on the host CPU; value = median step" % n_sample},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                             "sample": "%d streams per step, %d pinned host threads, median of %d steps (min %.3f s, max %.3f s)"
                                       % (n_sample, threads, steps, min(ts), max(ts)),
                             "single_thread_value": n1 * STREAM_BYTES / dt1 / 1e6},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


def _device_decode_ms(eng, torch, dev, stream, comp, coff, clen, raw_blob, off, ln, steps, flags=0):
    """device-resident decode of one population: K steps timed with CUDA events on `stream`; returns (ms per step, decode-kernel
    ms, bit-exact vs the raw input)"""
    n = len(coff)
    d_in = torch.from_numpy(comp).to(dev)
    d_in_off, d_in_len = torch.from_numpy(coff.astype(np.int64)).to(dev), torch.from_numpy(clen.astype(np.int64)).to(dev)
    d_out = torch.zeros(int(ln.sum()) + 256, dtype=torch.uint8, device=dev)
    d_out_off, d_out_cap = torch.from_numpy(off.astype(np.int64)).to(dev), torch.from_numpy(ln.astype(np.int64)).to(dev)
    d_out_len, d_status = torch.zeros(n, dtype=torch.int64, device=dev), torch.zeros(n, dtype=torch.int32, device=dev)

    def step():
        eng.decode_batch_device(d_in.data_ptr(), d_in_off.data_ptr(), d_in_len.data_ptr(), d_out.data_ptr(), d_out_off.data_ptr(),
                                d_out_cap.data_ptr(), d_out_len.data_ptr(), d_status.data_ptr(), n, d_in.numel(), flags, stream.cuda_stream)
    for _ in range(2):
        step()
    torch.cuda.synchronize()
    ok = bool((d_status == 0).all()) and bool((d_out[: int(ln.sum())].cpu().numpy() == raw_blob[: int(ln.sum())]).all())
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        step()
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps, eng.last_main_kernel_ms(), ok


def dump_outputs(path, d_out, d_out_len, d_status, n):
    """What a caller of decode_batch_device receives from one step: status and decoded length of every stream, and the decoded
    bytes of a fixed, seeded sample of DUMP_STREAMS streams (stream_index.npy names them), one row per stream."""
    import torch
    os.makedirs(path, exist_ok=True)
    pick = np.sort(np.random.default_rng(0).choice(n, size=min(n, DUMP_STREAMS), replace=False))
    rows = d_out[: n * STREAM_BYTES].view(n, STREAM_BYTES)[torch.from_numpy(pick).to(d_out.device)]
    np.save(os.path.join(path, "decoded.npy"), rows.cpu().numpy().astype(np.float32))
    np.save(os.path.join(path, "stream_index.npy"), pick.astype(np.float64))
    np.save(os.path.join(path, "out_len.npy"), d_out_len.cpu().numpy().astype(np.float64))
    np.save(os.path.join(path, "status.npy"), d_status.cpu().numpy().astype(np.float64))


def _compact(out, eoff, out_len):
    n = len(out_len)
    pad = (out_len + np.uint64(15)) & ~np.uint64(15)
    coff = np.zeros(n, np.uint64)
    coff[1:] = np.cumsum(pad)[:-1]
    comp = np.zeros(int(pad.sum()) + 64, np.uint8)
    for i in range(n):
        comp[int(coff[i]): int(coff[i] + out_len[i])] = out[int(eoff[i]): int(eoff[i] + out_len[i])]
    return comp, coff, out_len.astype(np.uint64)


def measure_populations(eng, torch, dev, stream, blob, off, ln, steps=3):
    """SURVEY 8d: the same raw streams under the other encodings.  Inputs are produced by the product's own GPU encoder (Z: the
    library's greedy LZ77 command generator + the GPU command-list encoder)."""
    import divans_b200
    n = len(off)
    cap = np.full(n, STREAM_BYTES + STREAM_BYTES // 2 + 70144, np.uint64)
    eoff = np.arange(n, dtype=np.uint64) * cap[0]
    out = np.zeros(int(cap.sum()), np.uint8)
    pops = {}

    def run(name, desc, opts, cmds=None, flags=0):
        if cmds is None:
            out_len, status = eng.encode_batch_host(blob, off, ln, out, eoff, cap, opts)
        else:
            out_len, status = eng.encode_batch_host(cmds[0], cmds[1], cmds[2], out, eoff, cap, opts, cmds=True)
        assert (status == 0).all(), name
        comp, coff, clen = _compact(out, eoff, out_len)
        ms, kms, ok = _device_decode_ms(eng, torch, dev, stream, comp, coff, clen, blob, off, ln, steps, flags)
        pops[name] = {"encoding": desc, "ms_per_step": ms, "decode_kernel_ms": kms, "value": float(ln.sum()) / ms / 1e3, "unit": UNIT,
                      "compressed_bytes": int(clen.sum()), "bit_exact": ok, "steps": steps}

    run("Z_lz77_window16", "LZ77 command streams (greedy hash-chain matcher, window 16, min match 4; UTF8 context mode, mixing value 4): copy-dominated, like the reference's default compressor output",
        divans_b200.encode_options(window_size=16), cmds=divans_b200.lz77_cmds_batch(blob, off, ln, 16, 2, 4))
    run("L_dcm2", "literal-only, dynamic_context_mixing=2 (two priors mixed and the weights adapted per nibble)", divans_b200.encode_options(dynamic_context_mixing=2))
    run("L_utf8", "literal-only, UTF8 context mode, mixing value 1", divans_b200.encode_options(literal_pred_mode=2, literal_mixing_value=1))
    run("L_blend", "literal-only, coded with the reference's feature=\"blend\" probability model (BlendCDF16; generic per-nibble path, no literal fast loop)",
        divans_b200.encode_options(cdf_model=divans_b200.CDF_BLEND), flags=divans_b200.FLAG_CDF_BLEND)
    return pops


def run_entropy(args, eng, rank, world, dev):
    """BASELINE configs[4]: 1 MiB Bernoulli-bit streams, 128 per GPU, p in {0.5, 0.9, 0.99}; device-resident decode."""
    import torch
    import torch.distributed as dist
    import divans_b200
    from divans_b200 import synth
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    n, sb = 128, 1 << 20
    res, tot_bytes, tot_ms = {}, 0.0, 0.0
    for pr in (0.5, 0.9, 0.99):
        blob, off, ln = synth.bernoulli_streams(n, sb, pr, seed=0xB17 + 1000 * rank)
        cap = np.full(n, sb + sb // 2 + 70144, np.uint64)
        eoff = np.arange(n, dtype=np.uint64) * cap[0]
        out = np.zeros(int(cap.sum()), np.uint8)
        out_len, status = eng.encode_batch_host(blob, off, ln, out, eoff, cap, divans_b200.encode_options())
        assert (status == 0).all()
        comp, coff, clen = _compact(out, eoff, out_len)
        ms, kms, ok = _device_decode_ms(eng, torch, dev, stream, comp, coff, clen, blob, off, ln, max(2, args.steps // 3))
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t[0])
        res["p=%.2f" % pr] = {"ms_per_step": ms, "value": world * n * sb / ms / 1e3, "unit": UNIT, "ratio": float(clen.sum()) / (n * sb), "bit_exact": ok}
        tot_bytes += world * n * sb
        tot_ms += ms
    if rank == 0:
        print(json.dumps({"metric": METRIC, "value": tot_bytes / tot_ms / 1e3, "unit": UNIT, "n_gpus": world, "steps": max(2, args.steps // 3),
                          "warmup": 2, "ms_per_step": tot_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "i16/u64",
                          "data": "synthetic",
                          "config": {"workload": "entropy sweep (BASELINE configs[4]): %d x 1 MiB Bernoulli-bit streams per GPU, p in {0.5, 0.9, 0.99}, "
                                                 "literal-only encoding" % n, "lanes_per_stream": eng.last_lanes()}, "sweep": res}))
    eng.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--streams", type=int, default=0, help="streams per GPU (default: 4096 at N=1, 8192 at N>1)")
    ap.add_argument("--workload", default="text", choices=["text", "entropy"])
    ap.add_argument("--skip-populations", action="store_true")
    ap.add_argument("--lanes", type=int, default=int(os.environ.get("DIVANS_B200_LPS", "0")), help="lanes per stream: 16 / 8 (v2 engine), 32 / 116 (round-1 kernels); 0 = by batch size")
    ap.add_argument("--cpu-sample", type=int, default=0, help="streams in the cpu_baseline sample (0 = auto)")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step decoded to DIR/*.npy (float32 / float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "text"):
        ap.error("--dump-outputs writes the outputs of the text workload on the GPU (--impl ours --workload text)")
    if args.impl == "reference":
        return run_reference_arm(args)

    import torch
    import torch.distributed as dist
    import divans_b200
    from divans_b200 import sharding

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if args.warmup < 3:
        args.warmup = 3

    if not args.streams:
        args.streams = STREAMS_PER_GPU if world == 1 else STREAMS_PER_GPU_SCALING
    eng = divans_b200.Engine(local_rank, 0, args.lanes)   # 0: the library picks 16 lanes per stream while the batch is resident, else 8
    if args.workload == "entropy":
        return run_entropy(args, eng, rank, world, dev)
    n = args.streams
    blob, off, ln = make_inputs(rank, n)
    comp, coff, clen, generator = encode_inputs(blob, off, ln, eng)
    comp_bytes = int(clen.sum())
    out_bytes = int(ln.sum())

    # ---- device-resident arm ----
    d_in = torch.from_numpy(comp).to(dev)
    d_in_off = torch.from_numpy(coff.astype(np.int64)).to(dev)
    d_in_len = torch.from_numpy(clen.astype(np.int64)).to(dev)
    d_out = torch.zeros(out_bytes + 256, dtype=torch.uint8, device=dev)
    d_out_off = torch.from_numpy(off.astype(np.int64)).to(dev)
    d_out_cap = torch.from_numpy(ln.astype(np.int64)).to(dev)
    d_out_len = torch.zeros(n, dtype=torch.int64, device=dev)
    d_status = torch.zeros(n, dtype=torch.int32, device=dev)
    stream = torch.cuda.Stream(device=dev)          # a non-default stream: its handle is what the C ABI launches on
    torch.cuda.set_stream(stream)

    def step_device():
        eng.decode_batch_device(d_in.data_ptr(), d_in_off.data_ptr(), d_in_len.data_ptr(), d_out.data_ptr(), d_out_off.data_ptr(),
                                d_out_cap.data_ptr(), d_out_len.data_ptr(), d_status.data_ptr(), n, d_in.numel(), 0, stream.cuda_stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step_device()
    barrier()
    assert bool((d_status == 0).all()) and bool((d_out_len == STREAM_BYTES).all()), "decode failed"
    assert bool((d_out[:out_bytes].cpu().numpy() == blob).all()), "GPU output differs from the original input"
    args.lanes = eng.last_lanes()                    # the layout the library used for this batch size
    launches0 = eng.launch_count
    try:
        dev_uuid = "GPU-" + str(torch.cuda.get_device_properties(local_rank).uuid)
    except Exception:
        dev_uuid = None
    sampler = ClockSampler(local_rank, dev_uuid)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    main_ms = []
    barrier()
    ev0.record(stream)
    for _ in range(args.steps):
        step_device()
    ev1.record(stream)
    barrier()
    clocks = sampler.stop()
    dev_ms = ev0.elapsed_time(ev1)
    launches = eng.launch_count - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, d_out, d_out_len, d_status, n)
    # the decode kernel's own duration (CUDA events inside the library, on the same stream), one extra untimed pass
    for _ in range(3):
        step_device()
        torch.cuda.synchronize()
        main_ms.append(eng.last_main_kernel_ms())
    kern_ms = float(np.median(main_ms))

    # ---- the other encodings of the same raw streams (rank 0's shard; device-resident, 3 steps each) ----
    populations = None
    if rank == 0 and not args.skip_populations:
        populations = measure_populations(eng, torch, dev, stream, blob, off, ln)

    # ---- supplementary: the GPU encoder on the same shard, raw inputs resident in HBM (BASELINE configs[3] shape) ----
    d_raw = torch.from_numpy(blob).to(dev)
    ecap = STREAM_BYTES + STREAM_BYTES // 2 + 70144
    d_eout = torch.zeros(n * ecap, dtype=torch.uint8, device=dev)
    d_eoff = (torch.arange(n, dtype=torch.int64, device=dev) * ecap)
    d_ecap = torch.full((n,), ecap, dtype=torch.int64, device=dev)
    d_elen = torch.zeros(n, dtype=torch.int64, device=dev)
    d_est = torch.zeros(n, dtype=torch.int32, device=dev)
    def run_encode(eopts, expect_bytes=None):
        def step_encode():
            eng.encode_batch_device(n, d_raw.data_ptr(), d_out_off.data_ptr(), d_out_cap.data_ptr(), STREAM_BYTES, d_eout.data_ptr(),
                                    d_eoff.data_ptr(), d_ecap.data_ptr(), d_elen.data_ptr(), d_est.data_ptr(), eopts, stream.cuda_stream)
        step_encode()
        torch.cuda.synchronize()
        assert bool((d_est == 0).all()), "GPU encoder failed"
        if expect_bytes is not None:
            assert int(d_elen.sum()) == expect_bytes, "GPU encoder (device API) disagrees with the host API"
        ee0, ee1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ee0.record(stream)
        for _ in range(enc_steps):
            step_encode()
        ee1.record(stream)
        torch.cuda.synchronize()
        return ee0.elapsed_time(ee1) / enc_steps, eng.last_main_kernel_ms(), int(d_elen.sum())
    enc_steps = 3
    enc_ms, enc_model_ms, _ = run_encode(divans_b200.encode_options(), comp_bytes)                       # reference defaults
    enc2_ms, enc2_model_ms, enc2_bytes = run_encode(divans_b200.encode_options(dynamic_context_mixing=2))   # BASELINE configs[3] option
    del d_eout

    # ---- end-to-end arm: host buffers (pinned), H2D + D2H of EVERY step inside the timed region, through the public host
    # API.  Headline: the pipelined call (decode_batch_host_async / wait: at most two batches in flight, each step has its
    # own output buffer, the copies of one step overlap the kernels of its neighbours); the blocking call is reported too.
    h_in = [torch.from_numpy(comp).pin_memory() for _ in range(2)]
    h_out = [torch.zeros(out_bytes + 256, dtype=torch.uint8).pin_memory() for _ in range(2)]
    h_in_np, h_out_np_l = [t.numpy() for t in h_in], [t.numpy() for t in h_out]
    h_out_np = h_out_np_l[0]
    for _ in range(2):
        eng.decode_batch_host(h_in_np[0], coff, clen, h_out_np, off, ln)
    barrier()
    t0 = time.perf_counter()
    sync_steps = 3
    for _ in range(sync_steps):
        out_len_h, status_h = eng.decode_batch_host(h_in_np[0], coff, clen, h_out_np, off, ln)
    torch.cuda.synchronize()
    e2e_sync_s = (time.perf_counter() - t0) / sync_steps
    assert (status_h == 0).all() and (h_out_np[:out_bytes] == blob).all()
    for k in range(2):      # warm the two pipeline lanes (their device buffers are allocated on first use)
        eng.decode_batch_host_async(h_in_np[k], coff, clen, h_out_np_l[k], off, ln).wait()
    h_out_np_l[1][:out_bytes] = 0
    barrier()
    e2e_steps = max(4, args.steps)
    t0 = time.perf_counter()
    pend, results = [], []
    for k in range(e2e_steps):
        pend.append(eng.decode_batch_host_async(h_in_np[k & 1], coff, clen, h_out_np_l[k & 1], off, ln))
        if len(pend) == 2:
            results.append(pend.pop(0).wait())
    while pend:
        results.append(pend.pop(0).wait())
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    assert all((st == 0).all() and (ol == STREAM_BYTES).all() for ol, st in results)
    assert (h_out_np_l[0][:out_bytes] == blob).all() and (h_out_np_l[1][:out_bytes] == blob).all()

    # ---- N > 1: the sharded API.  Rank 0 owns the whole job's host batch (pinned), ShardedDecoder scatters it over NVLink,
    # every rank decodes its byte-balanced shard in HBM, rank 0 gathers and copies the result to the host. ----
    scattered = None
    if world > 1:
        sd = sharding.ShardedDecoder(eng, device=dev)
        sizes = torch.tensor([comp.size, n], dtype=torch.int64, device=dev)
        all_sizes = [torch.zeros(2, dtype=torch.int64, device=dev) for _ in range(world)]
        dist.all_gather(all_sizes, sizes)
        g_comp = [torch.zeros(int(a[0]), dtype=torch.uint8, device=dev) if rank == 0 else None for a in all_sizes]
        g_len = [torch.zeros(int(a[1]), dtype=torch.int64, device=dev) if rank == 0 else None for a in all_sizes]
        g_off = [torch.zeros(int(a[1]), dtype=torch.int64, device=dev) if rank == 0 else None for a in all_sizes]
        # (shards differ in compressed size: point-to-point transfers, not dist.gather, which wants equal shapes)
        mine = [torch.from_numpy(comp).to(dev), torch.from_numpy(clen.astype(np.int64)).to(dev), torch.from_numpy(coff.astype(np.int64)).to(dev)]
        if rank == 0:
            for dst_list, t in zip((g_comp, g_len, g_off), mine):
                dst_list[0].copy_(t)
            for r in range(1, world):
                for dst_list in (g_comp, g_len, g_off):
                    dist.recv(dst_list[r], src=r)
        else:
            for t in mine:
                dist.send(t, dst=0)
        if rank == 0:
            base = np.concatenate([[0], np.cumsum([int(a[0]) for a in all_sizes])[:-1]])
            job_blob = torch.cat(g_comp).cpu().pin_memory()
            job_off = np.concatenate([g_off[r].cpu().numpy() + base[r] for r in range(world)])
            job_len = np.concatenate([g_len[r].cpu().numpy() for r in range(world)])
            job_cap = np.full(job_len.size, STREAM_BYTES, np.int64)
            del g_comp
        sc_steps = 3
        for k in range(1 + sc_steps):
            barrier()
            t0 = time.perf_counter()
            r = sd.decode(job_blob, job_off, job_len, job_cap) if rank == 0 else sd.decode()
            barrier()
            if k == 0:
                if rank == 0:
                    o, oo, ol, st_ = r
                    assert bool((st_ == 0).all()) and bool((ol == STREAM_BYTES).all())
                    assert bool((o[: n * STREAM_BYTES].numpy() == blob).all()), "sharded decode differs from the input"
                t_sc = []
            else:
                t_sc.append(time.perf_counter() - t0)
        if rank == 0:
            scattered = {"value": float(job_len.size) * STREAM_BYTES / float(np.median(t_sc)) / 1e6, "unit": UNIT, "steps": sc_steps,
                         "h2d_bytes_per_step": int(job_blob.numel()), "d2h_bytes_per_step": int(job_len.size) * STREAM_BYTES,
                         "api": "divans_b200.sharding.ShardedDecoder: rank 0 holds the job's host batch; partition_by_bytes, NCCL send/recv scatter, "
                                "device decode per rank, NCCL gather, one D2H on rank 0 (wall clock around the collective call)",
                         "shard_bytes": sd.last.get("shard_bytes")}

    tt = torch.tensor([dev_ms, e2e_s * 1e3, e2e_sync_s * 1e3], dtype=torch.float64, device=dev)
    uu = torch.tensor([float(out_bytes)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dist.all_reduce(uu, op=dist.ReduceOp.SUM)
    dev_ms_max, e2e_ms_max, e2e_sync_ms_max = float(tt[0]), float(tt[1]), float(tt[2])
    total_out = float(uu[0])

    if rank == 0:
        peak, peak_src = _peaks()
        value = total_out * args.steps / (dev_ms_max / 1e3) / 1e6
        e2e_v = total_out * e2e_steps / (e2e_ms_max / 1e3) / 1e6
        alg_bytes = comp_bytes + out_bytes     # per launch of the decode kernel on this rank (SURVEY 8d: B_alg)
        achieved = alg_bytes / (kern_ms / 1e3) / 1e9
        # dram bytes of the decode kernel come from an ncu capture (profiles/traffic.json); they are only reported when that capture
        # was made with the kernel version this library was built from
        traffic, traffic_note = None, "no capture"
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            try:
                tj = json.load(open(tp))
                entries = tj.get("entries", [tj])
                mine = [e for e in entries if int(e.get("lanes_per_stream", 0)) == args.lanes and int(e.get("streams", 0)) == n]
                if mine and mine[0].get("kernel_version") == divans_b200.kernel_version():
                    traffic, traffic_note = mine[0].get("decode_kernel_dram_bytes_per_launch"), mine[0].get("source")
                elif mine:
                    traffic_note = "profiles/traffic.json holds kernel %s for this layout, this library is %s: not reported" % (
                        mine[0].get("kernel_version"), divans_b200.kernel_version())
                else:
                    traffic_note = "profiles/traffic.json has no capture for %d lanes per stream x %d streams: not reported" % (args.lanes, n)
            except Exception:
                traffic = None
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "i16/u64", "data": "synthetic",
            "config": {"workload": "%d independent 64 KiB synthetic-text divANS streams per GPU (BASELINE configs[%d]), literal-only "
                                   "encoding (1 PredictionMode + 1 Literal command)" % (n, 1 if world == 1 else 2),
                       "streams_per_gpu": n, "stream_bytes": STREAM_BYTES, "compressed_bytes_per_gpu": comp_bytes,
                       "lanes_per_stream": args.lanes, "parallelism": "dp%d (streams sharded, no data-path collective)" % world,
                       "l2_policy": "inputs+outputs+model state per step (>0.39 GB + prior arena) exceed the 126 MB L2; no explicit flush",
                       "input_generator": generator},
            "e2e": {"value": e2e_v, "unit": UNIT, "h2d_bytes_per_step": comp_bytes + 4 * 8 * n, "d2h_bytes_per_step": out_bytes + 12 * n,
                    "steps": e2e_steps, "api": "divans_b200_decode_batch_host_async / _wait (two batches in flight, pinned host buffers)",
                    "blocking_call_value": total_out / e2e_sync_ms_max * 1e3 / 1e6, "blocking_call_api": "divans_b200_decode_batch_host"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": "dv::decode_kernel_v2<%d>" % args.lanes if args.lanes in (8, 16) else "dv::decode_kernel<%d>" % (args.lanes % 100), "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_note, "peak_source": peak_src,
                         "kernel_version": divans_b200.kernel_version(),
                         "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": kern_ms},
        }
        line["encode"] = {"metric": "batched_encode_throughput_raw", "unit": UNIT, "steps": enc_steps, "n_gpus": 1,
                          "dynamic_context_mixing_2": {"value": out_bytes / (enc2_ms / 1e3) / 1e6, "ms_per_step": enc2_ms,
                                                       "model_kernel_ms": enc2_model_ms, "compressed_bytes": enc2_bytes},
                          "default_options": {"value": out_bytes / (enc_ms / 1e3) / 1e6, "ms_per_step": enc_ms,
                                              "model_kernel_ms": enc_model_ms, "compressed_bytes": comp_bytes},
                          "note": "rank 0's shard (%d x 64 KiB; BASELINE configs[3] is 4096 x 64 KiB), inputs and outputs resident in HBM; "
                                  "literal-only command generator (the brotli quality-11 command selection is out of scope)" % n}
        if populations is not None:
            line["populations"] = populations
        if scattered is not None:
            line["scattered_e2e"] = scattered
        if not args.skip_cpu and world == 1:
            threads = _pin_all_cores()
            ns = args.cpu_sample or 2048
            cb, cpu_out = cpu_baseline(comp, coff, clen, blob, off, ln, ns, threads)
            nn = min(ns, n)
            cb["gpu_bit_exact_vs_oracle"] = bool((cpu_out[: nn * STREAM_BYTES] == h_out_np[: nn * STREAM_BYTES]).all())
            line["cpu_baseline"] = cb
        print(json.dumps(line))
    eng.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
