#!/usr/bin/env python
"""bench.py -- log lines/sec through the B200 detector (BASELINE.json metric).

Workload (BASELINE config 2 shape, windows as in config 4): every GPU owns 17 synthetic messages of
65 536 audit records x 256 B (16 MiB each, 272 MiB > the 126 MB L2).  Message 0 is the anomaly-free
training window (untimed).  A STEP is one WINDOW of 8 consecutive detection messages (512k records,
128 MiB) and, with more than one GPU, ONE NCCL sum-all-reduce of the window's statistics
(SURVEY.md 8d, config 4); the timed steps cycle over the 16 detection messages.  Multi-GPU: the
stream shards by message across ranks (weak scaling), no data-path collective.

  value     lines/s, messages resident in HBM when the timed region starts, CUDA events on the
            launching stream, max over ranks.
  e2e       the same metric through the reference-facing plugin call:
            B200NewValueDetector.process(message in PINNED HOST memory) -> compact result bytes,
            H2D + kernel + D2H inside the timed region; `abi_pipelined` = the C-ABI two-slot path
            (dm_submit_lines / dm_collect) beside it.
  roofline  the tokenizer+detector kernel (one launch per message): algorithmic bytes per launch
            (record bytes + 1 B flag + 4 B score per record) / average launch duration over the
            timed region, against MEASURED_PEAKS.json.
  cpu_baseline  rank 0, N=1: the oracle's C restatement on all host cores (pinned pthreads, median
            of 5 x 2 s) and, as `reference_engine`, the reference's OWN Engine/Service per record.
  extra.configs  BASELINE configs 3 (through NNG-framed sockets), 4 (windows; = this run) and 5
            (variable-length records) measured in the same run.

`--impl reference` times the CPU restatement with all host threads on the same config (the
reference is pure Python whose detector arithmetic is not vendored; DESIGN.md "Reference arm").
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

LINES_PER_MSG = 65536
LINE_BYTES = 256
N_DETECT = 16                 # detection messages per GPU
WINDOW_MSGS = 8               # messages per window = per step
METRIC = "log lines/sec through detector"
UNIT = "lines/s"


def workload_config(world: int) -> dict:
    """The same dict in both arms (`--impl b200` and `--impl reference`)."""
    return {
        "workload": "config2 shape in config4 windows: detector on synthetic audit records, 64k records x 256 B per "
                    "message (16 MiB), K=5 monitored fields, p=1e-3 anomalies; step = one window of 8 messages "
                    "(512k records) + one statistics all-reduce when n_gpus > 1",
        "lines_per_message": LINES_PER_MSG, "line_bytes": LINE_BYTES, "messages_per_window": WINDOW_MSGS,
        "detect_messages_per_gpu": N_DETECT, "training_window_lines": LINES_PER_MSG,
        "l2_policy": "inputs larger than L2 (16 x 16 MiB cycled per GPU)",
        "parallelism": f"shard-by-message x{world}, 1 stats all-reduce per window" if world > 1 else "single GPU",
    }


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


KERNEL_SOURCES = ("dm_kernels_stream.cuh", "dm_kernels_index.cuh", "dm_device.cuh", "dm_hash.h")


def _csrc_sha() -> str:
    """Fingerprint of the sources of the dominant kernel (dm_k_stream and what it includes): ties the ncu numbers under
    profiles/ to the code they were taken on."""
    h = hashlib.sha256()
    d = os.path.join(ROOT, "detectmateservice_b200", "csrc")
    for f in KERNEL_SOURCES:
        h.update(f.encode())
        h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


def _make_messages(seed_offset: int, n_detect: int = N_DETECT, lines: int = LINES_PER_MSG, varlen: bool = False):
    from detectmateservice_b200.synth import SEED, AuditSynth
    g = AuditSynth(SEED + seed_offset)
    gen = g.batch_varlen if varlen else (lambda n, inject: g.batch(n, inject=inject, line_bytes=LINE_BYTES))
    msgs = [gen(lines, inject=False)[0]]
    for _ in range(n_detect):
        msgs.append(gen(lines, inject=True)[0])
    return msgs


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU during the timed region (NVML)."""

    def __init__(self, index: int, period: float = 0.001):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self._halt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.nv = None

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {}
        for attr, name in (("nvmlClocksThrottleReasonSwPowerCap", "sw_power_cap"),
                           ("nvmlClocksThrottleReasonHwSlowdown", "hw_slowdown"),
                           ("nvmlClocksThrottleReasonSwThermalSlowdown", "sw_thermal_slowdown"),
                           ("nvmlClocksThrottleReasonHwThermalSlowdown", "hw_thermal_slowdown"),
                           ("nvmlClocksThrottleReasonHwPowerBrakeSlowdown", "hw_power_brake")):
            if hasattr(nv, attr):
                names[getattr(nv, attr)] = name
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._halt.wait(self.period)

    def finish(self):
        self._halt.set()
        if self.is_alive():
            self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------
# CPU legs (the oracle and the reference engine are executed HERE and nowhere else in the product)
# ------------------------------------------------------------------------------------------
def _cpu_port_rates(msgs, threads: int, min_seconds: float, samples: int):
    """C restatement on `threads` pinned worker threads: (threads used, rates per sample)."""
    from detectmateservice_b200.synth import MONITORED_KEYS
    from oracle import native
    native.build()
    keys = [k.encode() for k in MONITORED_KEYS]
    used, rates, _ = native.bench_threads(keys, msgs[0], msgs[1], threads, min_seconds, samples)
    return used, rates


def _reference_engine_leg(msgs, seconds: float = 4.0):
    """The reference's own Service.process / Engine loop per record (BASELINE.md section 4)."""
    from detectmateservice_b200.synth import MONITORED_KEYS
    from oracle import ref_engine, rtok
    if ref_engine.reference_path() is None:
        return {"unavailable": "reference service not in oracle/_ref (make -C oracle ref)"}
    train = rtok.split_records(msgs[0][:LINE_BYTES * 2000])
    # (anomaly-free records: an alert would be answered on the feeder's socket)
    detect = rtok.split_records(msgs[0][LINE_BYTES * 2000:LINE_BYTES * 6000])
    out = {"granularity": "one record per message (the reference's native granularity, engine.py:159-217)",
           "source": ref_engine.reference_path().replace(ROOT + os.sep, "")}
    try:
        rate1, n1 = ref_engine.inprocess_rate(MONITORED_KEYS, train, detect, seconds)
        out["service_process_1_thread"] = rate1
        cores = os.cpu_count() or 1
        p = max(1, cores // 2)                      # one service + one sender process per pair of cores
        rate_p, n_p, secs = ref_engine.ipc_rate(MONITORED_KEYS, train, detect, p, seconds)
        out["engine_ipc_processes"] = p
        out["engine_ipc_box"] = rate_p
        out["engine_ipc_per_service"] = rate_p / p
        out["sample"] = f"{n1} records in-process ({seconds:.0f} s); {n_p} records over {p} ipc services ({secs:.1f} s)"
    except Exception as e:                          # a measurement leg must not take the bench line down
        out["error"] = f"{type(e).__name__}: {e}"
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    threads = os.cpu_count() or 1
    msgs = _make_messages(0, n_detect=1)
    step_s = 1.0                                     # one step = a 1 s sample of the same workload on all host threads
    used, _ = _cpu_port_rates(msgs, threads, 0.3, max(1, min(args.warmup, 3)))
    used, rates = _cpu_port_rates(msgs, threads, step_s, args.steps)
    value = float(np.median(rates))
    lines_per_step = WINDOW_MSGS * LINES_PER_MSG
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * lines_per_step / value, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": workload_config(world),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": used, "kind": "port",
                         "sample": f"median of {args.steps} samples of {step_s:.0f} s on {used} pinned threads, C restatement "
                                   f"oracle/c/dm_oracle.c (the reference's detector source is not vendored); ms_per_step = "
                                   f"one window of {lines_per_step} records at that rate",
                         "spread": [float(min(rates)), float(max(rates))]},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------
def _component(device: int, max_batch_bytes: int):
    from detectmateservice_b200.component import B200NewValueDetector
    from detectmateservice_b200.synth import MONITORED_KEYS
    cfg = {"detectors": {"B200NewValueDetector": {
        "method_type": "new_value_detector", "data_use_training": LINES_PER_MSG, "auto_config": False,
        "params": {"output_format": "compact", "input_format": "raw_lines", "max_batch_bytes": max_batch_bytes,
                   "device": device, "table_log2_slots": 16},
        "global": {"g": {"header_variables": [{"pos": k} for k in MONITORED_KEYS]}}}}}
    return B200NewValueDetector(config=cfg)


def _config3_engine(h_msgs, nbytes, device: int, seconds: float = 2.0):
    """BASELINE config 3: sender -> NNG PAIR0 (ipc) -> DetectorEngine(B200NewValueDetector) -> sink."""
    import pynng
    from detectmateservice_b200.compat import ipc_tempdir
    from detectmateservice_b200.service import DetectorEngine
    comp = _component(device, max(nbytes) + 4096)
    tmp = ipc_tempdir("dmcfg3")
    eng_addr, out_addr = f"ipc://{tmp}/det.ipc", f"ipc://{tmp}/out.ipc"
    sink = pynng.Pair0(listen=out_addr, recv_timeout=30000)
    lines = [0]
    res = {}
    try:
        with DetectorEngine(comp, eng_addr, out_addr=[out_addr]) as eng:
            time.sleep(0.3)
            with pynng.Pair0(dial=eng_addr, block_on_dial=True) as tx:
                tx.send(memoryview(h_msgs[0].numpy()))    # training window
                sink.recv()
                sent = [0]
                stop = threading.Event()

                def feeder():
                    i = 0
                    while not stop.is_set():
                        tx.send(memoryview(h_msgs[1 + (i % N_DETECT)].numpy()))
                        sent[0] += 1
                        i += 1
                th = threading.Thread(target=feeder, daemon=True)
                t0 = time.perf_counter()
                th.start()
                got = 0
                while time.perf_counter() - t0 < seconds:
                    out = sink.recv()
                    got += 1
                    lines[0] += int(np.frombuffer(out[:4], dtype="<u4")[0])
                dt = time.perf_counter() - t0
                stop.set()
                # drain what is in flight so that the sender thread can finish
                sink.recv_timeout = 500
                try:
                    while True:
                        sink.recv()
                except pynng.Timeout:
                    pass
                th.join(timeout=5)
            res = {"lines_per_s": lines[0] / dt, "messages": got, "seconds": dt, "errors": eng.counters.get("errors"),
                   "topology": "sender thread -> ipc PAIR0 -> DetectorEngine(B200NewValueDetector, compact output) -> ipc PAIR0 -> sink",
                   "transport": "python SP/PAIR0 shim (detectmateservice_b200/shims/pynng.py), frames received into pinned slots"}
    except Exception as e:
        res = {"error": f"{type(e).__name__}: {e}"}
    finally:
        sink.close()
        comp.close()
    return res


def _dump_outputs(out_dir: str, rank: int, world: int, arrays: dict) -> None:
    """--dump-outputs: DIR/<name>.npy for every array (DIR/<name>_rank<r>.npy when n_gpus > 1)."""
    os.makedirs(out_dir, exist_ok=True)
    sfx = f"_rank{rank}" if world > 1 else ""
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}{sfx}.npy"), a)


def run_gpu(args):
    import torch
    import torch.distributed as dist
    from detectmateservice_b200 import _lib
    from detectmateservice_b200.detector import DeviceDetector
    from detectmateservice_b200.synth import MONITORED_KEYS

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # stdout carries the one JSON line: NCCL's own log (NCCL_DEBUG is left as the caller set it) goes to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    _lib.load()

    msgs = _make_messages(1000 * rank)
    nbytes = [len(m) for m in msgs]
    n_lines_msg = [m.count(b"\n") for m in msgs]
    det = DeviceDetector(MONITORED_KEYS, device=local_rank, max_batch_bytes=max(nbytes) + 4096,
                         max_lines=LINES_PER_MSG + 16, table_log2_slots=16)
    # The device-resident messages are written once, below, and never again: consecutive calls may overlap
    # (dm_set_overlap, include/dmdetect.h)
    det.set_overlap(True)
    # a dedicated non-default stream: the C ABI treats a NULL stream as "the handle's own stream", and torch's
    # default stream IS NULL -- events must sit on the launching stream.
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    sp = stream.cuda_stream
    assert sp != 0

    from detectmateservice_b200.numa import bound_to_gpu_node
    d_msgs, h_msgs = [], []
    with bound_to_gpu_node(local_rank) as numa_cpus:
        for m in msgs:
            t = torch.zeros(len(m) + 64, dtype=torch.uint8, device=dev)
            src = torch.frombuffer(bytearray(m), dtype=torch.uint8)
            t[:len(m)].copy_(src)
            d_msgs.append(t)
            hp = torch.empty(len(m), dtype=torch.uint8, pin_memory=True)
            hp.copy_(src)
            h_msgs.append(hp)
    # the set-up just wrote these buffers: evict them from the CPU caches, else the H2D copies of whichever buffers
    # are still cached run at a fraction of the link rate (dmdetect.cu, dm_host_cache_flush)
    for hp in h_msgs:
        _lib.check(_lib.load().dm_host_cache_flush(hp.data_ptr(), hp.numel()))
    cap = LINES_PER_MSG + 16
    d_flags = torch.zeros(cap, dtype=torch.uint8, device=dev)
    d_scores = torch.zeros(cap, dtype=torch.float32, device=dev)
    # the timed steps give every message of a window its own result rows: after a step the caller holds the flags and
    # scores of all of its messages
    w_flags = torch.zeros((WINDOW_MSGS, cap), dtype=torch.uint8, device=dev)
    w_scores = torch.zeros((WINDOW_MSGS, cap), dtype=torch.float32, device=dev)
    w_out = [(w_flags[m].data_ptr(), w_scores[m].data_ptr()) for m in range(WINDOW_MSGS)]
    from detectmateservice_b200.window import DeviceWindow
    dwin = DeviceWindow(det, rank, world, dev)
    if world > 1 and os.environ.get("DM_WINDOW", "native") == "native":
        dwin.init_native(n_comms=2)

    # the per-window exchange runs on a side stream: in steady state it carries statistics only and gates
    # nothing, so it overlaps the next window's kernels (two communicators: two windows' all-reduces in flight)
    sides = [torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)]
    win_n = [0]
    win_ev = torch.cuda.Event()

    def window(with_keys: bool):
        if with_keys:
            dwin.exchange(True, sp)                 # training window: detection must wait for it
            return
        sd = sides[win_n[0] % 2]
        win_n[0] += 1
        win_ev.record(stream)
        sd.wait_event(win_ev)
        if getattr(dwin, "native", False):
            dwin.exchange(False, sd.cuda_stream)
        else:
            with torch.cuda.stream(sd):
                dwin.exchange(False, sd.cuda_stream)

    # training window (untimed): every rank learns its message 0, then one exchange with keys
    det.enqueue_device(d_msgs[0].data_ptr(), nbytes[0], n_lines_msg[0], d_flags.data_ptr(), d_scores.data_ptr(), cap, sp)
    window(True)
    det.sync()

    def step(i: int):
        """One window: 8 messages, then (multi-GPU) one all-reduce of the window's statistics."""
        n = 0
        for m in range(WINDOW_MSGS):
            j = 1 + ((i * WINDOW_MSGS + m) % N_DETECT)
            det.enqueue_device(d_msgs[j].data_ptr(), nbytes[j], 0, w_out[m][0], w_out[m][1], cap, sp)
            n += n_lines_msg[j]
        if world > 1:
            window(False)
        return n

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- value: device-resident, CUDA events on the launching stream ----------------------
    for i in range(args.warmup):
        step(i)
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    _, _, launches0 = det.profile_read()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    lines_timed = 0
    barrier()
    e0.record(stream)
    for i in range(args.steps):
        lines_timed += step(i)
    stream.wait_stream(sides[0])                     # the last windows' all-reduces are part of the job
    stream.wait_stream(sides[1])
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    _, _, launches1 = det.profile_read()
    if args.dump_outputs:                            # the last timed step's results, before the steps below overwrite them
        last = [1 + (((args.steps - 1) * WINDOW_MSGS + m) % N_DETECT) for m in range(WINDOW_MSGS)]
        _dump_outputs(args.dump_outputs, rank, world, {
            "flags": np.stack([w_flags[m, :n_lines_msg[j]].cpu().numpy() for m, j in enumerate(last)]).astype(np.float32),
            "scores": np.stack([w_scores[m, :n_lines_msg[j]].cpu().numpy() for m, j in enumerate(last)])})
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    tot = torch.tensor([float(lines_timed)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    # The timed region is a few milliseconds, shorter than one NVML query: the same steps are kept running for
    # about another quarter of a second (untimed) under the sampler, so that clocks / throttle reasons are seen under
    # load.  Every rank runs the SAME number of steps (each ends in a collective), derived from the agreed step time.
    n_soak = int(min(20000, max(8, 250.0 / max(float(t.item()) / args.steps, 1e-3))))
    for k in range(n_soak):
        step(k)
        if k % 8 == 7:
            stream.synchronize()
    torch.cuda.synchronize()
    clocks = sampler.finish()
    clocks["window"] = f"timed region + {n_soak} more of the same steps (~0.25 s)"
    n_anom_last = det.sync()[1]
    ms_max, lines_all = float(t.item()), float(tot.item())
    value = lines_all / (ms_max * 1e-3)

    # ---- roofline: the tokenizer+detector kernel, one launch per message --------------------
    # (a) average launch duration over the timed region above (launches overlap, as in production);
    # (b) one launch at a time, event pair inside the library, nothing else on the GPU.
    n_launch = args.steps * WINDOW_MSGS
    alg_bytes = sum(nbytes[1 + (k % N_DETECT)] + 5 * n_lines_msg[1 + (k % N_DETECT)] for k in range(n_launch)) / n_launch
    kernel_ms = ms / n_launch
    det.set_overlap(False)
    det.profile_enable(True)
    for k in range(16):
        j = 1 + (k % N_DETECT)
        det.enqueue_device(d_msgs[j].data_ptr(), nbytes[j], 0, d_flags.data_ptr(), d_scores.data_ptr(), cap, sp)
    k_ms, k_n, _ = det.profile_read()
    det.profile_enable(False)
    det.set_overlap(True)
    peak, peak_src = _peaks()
    achieved = alg_bytes / (kernel_ms * 1e-3) / 1e9
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "r02_stream_traffic.json")
    if os.path.exists(tp):
        try:
            tj = json.load(open(tp))
            if tj.get("csrc_sha") == _csrc_sha():
                traffic, traffic_src = tj.get("dram_bytes_per_launch"), "profiles/r02_stream_traffic.json (ncu --set full of this build)"
            else:
                traffic_src = "profiles/r02_stream_traffic.json is from another build of the kernels: not reported"
        except Exception:
            pass
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "kernel": "dm_k_stream<false,false> (one launch per 64k-record message)",
                "kernel_ms": kernel_ms, "kernel_ms_definition": "timed region / launches (consecutive launches overlap)",
                "kernel_ms_isolated": (k_ms / k_n) if k_n else None,
                "algorithmic_bytes_per_launch": alg_bytes, "csrc_sha": _csrc_sha()}

    # ---- e2e: the plugin call with PINNED HOST buffers, H2D + D2H inside the timed region -----
    torch.cuda.synchronize()
    comp = _component(local_rank, max(nbytes) + 4096)
    from detectmateservice_b200.component import decode_compact
    comp.process(memoryview(h_msgs[0].numpy()))                      # training window
    e2e_steps = max(2, min(args.steps, 24))

    def e2e_window(i: int) -> int:
        n = 0
        for m in range(WINDOW_MSGS):
            j = 1 + ((i * WINDOW_MSGS + m) % N_DETECT)
            out = comp.process(memoryview(h_msgs[j].numpy()))        # bytes: [u32 n][n x u8 flag][n x f32 score]
            n += int.from_bytes(out[:4], "little")
        return n
    for i in range(2):
        e2e_window(i)
    barrier()
    t0 = time.perf_counter()
    e2e_lines = 0
    for i in range(e2e_steps):
        e2e_lines += e2e_window(i)
    barrier()
    dt = time.perf_counter() - t0
    t = torch.tensor([dt], dtype=torch.float64, device=dev)
    tot = torch.tensor([float(e2e_lines)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    e2e_value = float(tot.item()) / float(t.item())
    # parity spot check of the plugin path against the device-resident path
    f_chk, s_chk = decode_compact(comp.process(memoryview(h_msgs[1].numpy())))
    det.enqueue_device(d_msgs[1].data_ptr(), nbytes[1], 0, d_flags.data_ptr(), d_scores.data_ptr(), cap, sp)
    det.sync()
    same = bool((d_flags[:n_lines_msg[1]].cpu().numpy() == f_chk).all())
    comp.close()

    # the C-ABI two-slot path beside it: message i+1 crosses PCIe while message i runs
    pipe_steps = e2e_steps * WINDOW_MSGS

    def pipe_loop(n_steps: int) -> int:
        lines = 0
        for i in range(n_steps):
            slot = i & 1
            if i >= 2:
                f, s = det.collect(slot)
                lines += f.size
            det.submit(h_msgs[1 + (i % N_DETECT)].numpy(), 0, slot)
        for i in range(max(0, n_steps - 2), n_steps):
            f, s = det.collect(i & 1)
            lines += f.size
        return lines
    with bound_to_gpu_node(local_rank):              # the library's pinned result buffers are created here
        pipe_loop(4)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    pipe_lines = pipe_loop(pipe_steps)
    torch.cuda.synchronize()
    pipe_dt = time.perf_counter() - t0
    # plain H2D bandwidth of the same pinned buffers, for context
    t0 = time.perf_counter()
    for i in range(8):
        d_msgs[1 + i][:nbytes[1 + i]].copy_(h_msgs[1 + i], non_blocking=True)
    torch.cuda.synchronize()
    h2d_gbs = sum(nbytes[1:9]) / (time.perf_counter() - t0) / 1e9
    e2e = {"value": e2e_value, "unit": UNIT,
           "h2d_bytes_per_step": WINDOW_MSGS * nbytes[1], "d2h_bytes_per_step": WINDOW_MSGS * (5 * n_lines_msg[1] + 4 + 32),
           "steps": e2e_steps, "ms_per_step": 1e3 * float(t.item()) / e2e_steps,
           "api": "B200NewValueDetector.process(memoryview of a pinned host message) -> compact bytes, one call per message "
                  "(detectmateservice_b200/component.py; the reference calls it from Service.process, core.py:201-203)",
           "matches_device_resident_flags": same,
           "abi_pipelined": {"value": pipe_lines / pipe_dt, "unit": UNIT, "messages": pipe_steps,
                             "api": "dm_submit_lines / dm_collect, two slots (include/dmdetect.h)"},
           "h2d_gbs_pinned": h2d_gbs, "pinned_numa_local_cpus": len(numa_cpus) if numa_cpus else None}

    # ---- the other BASELINE configs, same run --------------------------------------------------
    extra = {"configs": {}}
    extra["configs"]["config4_windows"] = {
        "note": "this run: windows of 8 x 64k records, one NCCL all-reduce per window when n_gpus > 1",
        "lines_processed_timed": lines_all, "lines_per_s": value, "n_gpus": world}
    if not args.no_extra:
        # config 5: variable-length records (32 B - 4 KB mixture), device-resident, every rank its own messages
        try:
            vmsgs = _make_messages(3 + 1000 * rank, n_detect=4, lines=LINES_PER_MSG, varlen=True)
            vdet = DeviceDetector(MONITORED_KEYS, device=local_rank, max_batch_bytes=max(len(m) for m in vmsgs) + 4096,
                                  max_lines=LINES_PER_MSG + 16, table_log2_slots=16)
            vdet.set_overlap(True)
            vd = []
            for m in vmsgs:
                tt = torch.zeros(len(m) + 64, dtype=torch.uint8, device=dev)
                tt[:len(m)].copy_(torch.frombuffer(bytearray(m), dtype=torch.uint8))
                vd.append(tt)
            vdet.enqueue_device(vd[0].data_ptr(), len(vmsgs[0]), LINES_PER_MSG, d_flags.data_ptr(), d_scores.data_ptr(), cap, sp)
            vdet.sync()
            v_steps = 24
            for k in range(4):
                vdet.enqueue_device(vd[1 + k % 4].data_ptr(), len(vmsgs[1 + k % 4]), 0, d_flags.data_ptr(), d_scores.data_ptr(), cap, sp)
            # (the library picks the candidate re-check per message from the last message it has SEEN finish: let the
            # warm-up finish, as a stream that arrives over time would)
            vdet.sync()
            vdet.enqueue_device(vd[1].data_ptr(), len(vmsgs[1]), 0, d_flags.data_ptr(), d_scores.data_ptr(), cap, sp)
            barrier()
            v0, v1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            v0.record(stream)
            vb = 0
            for k in range(v_steps):
                j = 1 + k % 4
                vdet.enqueue_device(vd[j].data_ptr(), len(vmsgs[j]), 0, d_flags.data_ptr(), d_scores.data_ptr(), cap, sp)
                vb += len(vmsgs[j]) + 5 * LINES_PER_MSG
            v1.record(stream)
            barrier()
            vms = v0.elapsed_time(v1)
            tv = torch.tensor([vms], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tv, op=dist.ReduceOp.MAX)
            vms = float(tv.item())
            extra["configs"]["config5_varlen"] = {
                "lines_per_s": world * v_steps * LINES_PER_MSG / (vms * 1e-3), "n_gpus": world,
                "mean_record_bytes": float(np.mean([len(m) for m in vmsgs[1:]])) / LINES_PER_MSG,
                "candidate_recheck": "chained" if vdet.stream_recheck_chained() else "one by one",
                "roofline": {"bound": "hbm", "achieved": vb / (vms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                             "frac": vb / (vms * 1e-3) / 1e9 / peak},
                "workload": "64k records per message, lengths 32 B - 4 KB (70/25/5 % log-uniform mixture), quoted values with "
                            "monitored-key look-alikes; 4 messages cycled, device-resident"}
            vdet.close()
        except Exception as e:
            extra["configs"]["config5_varlen"] = {"error": f"{type(e).__name__}: {e}"}
        # config 3: through NNG-framed sockets (rank 0 only: one service per GPU would each look the same)
        if rank == 0:
            extra["configs"]["config3_nng_pipeline"] = _config3_engine(h_msgs, nbytes, local_rank)
        barrier()

    # ---- CPU baselines (rank 0, N=1 only) ----------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cores = os.cpu_count() or 1
        used, rates = _cpu_port_rates(msgs, cores, 2.0, 5)
        _, one = _cpu_port_rates(msgs, 1, 1.0, 3)
        cpu = {"value": float(np.median(rates)), "unit": UNIT, "cores": used, "kind": "port",
               "sample": f"median of 5 samples of 2 s on {used} pinned threads, each thread its own trained detector over its shard "
                         f"of one 64k-record message; oracle/c/dm_oracle.c (the reference's detector, detectmatelibrary, is not vendored)",
               "spread": [float(min(rates)), float(max(rates))],
               "single_thread": float(np.median(one)),
               "reference_engine": _reference_engine_leg(msgs)}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic", "config": workload_config(world),
            "e2e": e2e, "gpu_launches": int(launches1 - launches0), "clocks": clocks, "roofline": roofline,
            "extra": extra, "anomalies_last_message": int(n_anom_last),
        }
        if cpu is not None:
            line["cpu_baseline"] = cpu
        print(json.dumps(line))
    det.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline legs")
    ap.add_argument("--no-extra", action="store_true", help="skip the config 3 / config 5 legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's results to DIR: flags.npy and scores.npy, float32, one row per "
                         "message of the window (%d x %d records)" % (WINDOW_MSGS, LINES_PER_MSG))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    if os.environ.get("DM_BENCH_WATCHDOG"):                    # a hung run says where: all threads' stacks every N seconds
        import faulthandler
        faulthandler.dump_traceback_later(float(os.environ["DM_BENCH_WATCHDOG"]), repeat=True, file=sys.stderr)
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)
    return run_gpu(args)


if __name__ == "__main__":
    sys.exit(main())
