"""The reference's OWN `Engine._run_loop` + `Service.process`, driven one record per message with
the CPU oracle as its library component (BASELINE.md section 4).  MEASUREMENT INFRASTRUCTURE:
only bench.py's CPU legs and tests/ use this module.

Where the reference comes from: `oracle/_ref` (the unmodified reference service, put there by
`make -C oracle ref` in build()); its two missing
third-party imports (`pynng`, `detectmatelibrary.common.*`) are this repo's stand-ins
(detectmateservice_b200/shims), real packages win when installed.

Two figures, as the reference is deployed (one single-threaded service per process,
/root/reference/src/service/features/engine.py:80-82):
  inprocess_rate  one thread calling Service.process(record) in a loop (metrics + delegate,
                  /root/reference/src/service/core.py:176-206);
  ipc_rate        P service processes, each with its engine loop on its own ipc PAIR0 socket
                  (engine.py:153-217), each fed by its own sender process with 1/P of the stream.
"""
from __future__ import annotations

import multiprocessing as mp
import os
import socket
import sys
import tempfile
import time
from typing import List, Optional, Tuple

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_DIR = os.path.join(ROOT, "oracle", "_ref")


def reference_path() -> Optional[str]:
    return REF_DIR if os.path.isdir(os.path.join(REF_DIR, "service")) else None


def _setup_imports() -> str:
    p = reference_path()
    if p is None:
        raise RuntimeError("the reference service is not in oracle/_ref (make -C oracle ref)")
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    if p not in sys.path:
        sys.path.insert(0, p)
    from detectmateservice_b200.compat import install_shims
    install_shims()
    return p


def _component_class():
    """CoreComponent (the reference's plugin base) around oracle.nvd.NewValueDetectorOracle: one raw
    record per process() call, alerts as DetectorSchema bytes, None otherwise."""
    _setup_imports()
    from detectmatelibrary.common.core import CoreComponent
    from oracle.nvd import NewValueDetectorOracle

    class OracleNewValueDetector(CoreComponent):
        def __init__(self, name: str = "OracleNewValueDetector", config=None, **kw):
            super().__init__(name=name, config=None)
            self.det = NewValueDetectorOracle(name="NewValueDetector", config=_CFG)

        def process(self, data: bytes) -> Optional[bytes]:
            line = bytes(data).rstrip(b"\n")
            flag, score, alerts = self.det.step_line(line)
            if not flag:
                return None
            return self.det.make_output({"logID": ""}, score, alerts).SerializeToString()

    return OracleNewValueDetector


_CFG = {"data_use_training": 0, "global": {"g": {"header_variables": []}}}


def configure(keys: List[str], data_use_training: int) -> None:
    _CFG["data_use_training"] = int(data_use_training)
    _CFG["global"] = {"g": {"header_variables": [{"pos": k} for k in keys]}}


# the dotted path the reference's loader imports (component_loader.py:34-43)
def OracleNewValueDetector(*a, **k):                      # noqa: N802  (a class factory behind a class-like name)
    return _component_class()(*a, **k)


def _free_port() -> int:
    with socket.socket(socket.AF_INET, socket.SOCK_STREAM) as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def make_service(addr: Optional[str], tmp: str, autostart: bool):
    """The unmodified reference Service with the oracle component installed as its library component."""
    _setup_imports()
    from service.core import Service
    from service.settings import ServiceSettings

    class OracleService(Service):
        component_type = "oracle_new_value_detector"      # class attribute: skips resolver / loader (core.py:85-86)

    settings = ServiceSettings(component_name="oracle-nvd", engine_addr=addr, log_dir=os.path.join(tmp, "logs"),
                               log_to_file=False, log_to_console=False, log_level="ERROR", http_port=_free_port(),
                               engine_autostart=False)
    svc = OracleService(settings=settings)
    svc.library_component = _component_class()()
    if autostart:
        svc.start()
    return svc


def inprocess_rate(keys: List[str], train_lines: List[bytes], detect_lines: List[bytes], seconds: float = 5.0
                   ) -> Tuple[float, int]:
    """records/s of Service.process() on one thread; (rate, records timed)."""
    configure(keys, len(train_lines))
    with tempfile.TemporaryDirectory() as tmp:
        svc = make_service(f"inproc://dm-ref-engine-{os.getpid()}", tmp, autostart=False)
        for l in train_lines:
            svc.process(l)
        n, t0 = 0, time.perf_counter()
        deadline = t0 + seconds
        while time.perf_counter() < deadline:
            for l in detect_lines:
                svc.process(l)
            n += len(detect_lines)
        dt = time.perf_counter() - t0
        try:
            svc.stop()
        except Exception:
            pass
    return n / dt, n


def _service_proc(addr: str, keys: List[str], n_train: int, ready, done) -> None:
    configure(keys, n_train)
    with tempfile.TemporaryDirectory() as tmp:
        svc = make_service(addr, tmp, autostart=True)
        ready.set()
        done.wait()
        try:
            svc.stop()
        except Exception:
            pass


_SYNC = b"type=SYNC_%d msg=audit(1.000:1): res=sync"


def _feeder_proc(addr: str, train_lines: List[bytes], detect_lines: List[bytes], seconds: float, start, out_q) -> None:
    _setup_imports()
    import pynng
    with pynng.Pair0(dial=addr, recv_timeout=60000, block_on_dial=True) as s:
        for l in train_lines:
            s.send(l)
        serial = 0

        def sync():
            nonlocal serial
            serial += 1
            s.send(_SYNC % serial)           # a value nobody has seen: the service answers with an alert once every
            s.recv()                          # earlier record is through its (sequential) engine loop
        sync()
        start.wait()
        n, t0 = 0, time.perf_counter()
        deadline = t0 + seconds
        while time.perf_counter() < deadline:
            for l in detect_lines:
                s.send(l)
            n += len(detect_lines)
        sync()
        out_q.put((n, time.perf_counter() - t0))


def ipc_rate(keys: List[str], train_lines: List[bytes], detect_lines: List[bytes], n_services: int, seconds: float = 5.0
             ) -> Tuple[float, int, float]:
    """records/s of n_services reference services (own process, own ipc socket, own feeder process):
    (aggregate rate, records timed, slowest feeder's seconds)."""
    from detectmateservice_b200.compat import ipc_tempdir
    ctx = mp.get_context("spawn")
    tmp = ipc_tempdir("dmref")
    start = ctx.Event()
    done = ctx.Event()
    out_q = ctx.Queue()
    svcs, feeders, readies = [], [], []
    # (anomalous records would be answered and fill the feeder's receive queue: feed anomaly-free records only)
    for i in range(n_services):
        addr = f"ipc://{tmp}/svc{i}.ipc"
        ready = ctx.Event()
        p = ctx.Process(target=_service_proc, args=(addr, keys, len(train_lines), ready, done), daemon=True)
        p.start()
        svcs.append(p)
        readies.append((addr, ready))
    for addr, ready in readies:
        if not ready.wait(120):
            raise RuntimeError("a reference service did not come up")
    for addr, _ in readies:
        f = ctx.Process(target=_feeder_proc, args=(addr, train_lines, detect_lines, seconds, start, out_q), daemon=True)
        f.start()
        feeders.append(f)
    time.sleep(1.0 + 0.02 * n_services)          # feeders connect and train their service
    start.set()
    results = [out_q.get(timeout=seconds * 20 + 120) for _ in feeders]
    done.set()
    for p in feeders + svcs:
        p.join(timeout=10)
    n = sum(r[0] for r in results)
    slowest = max(r[1] for r in results)
    return n / slowest, n, slowest
