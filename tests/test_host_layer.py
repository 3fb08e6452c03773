"""Host layer on CPU: SP/PAIR0 transport, wire codec, engine mirror, component plumbing.

The component's DeviceDetector needs a GPU; here it is replaced by a test double backed by
the oracle so that everything AROUND the kernels (config parsing, framing, alert
materialisation, training counter, engine semantics, the unmodified reference service) is
exercised without a device.  test_gpu_component.py runs the same component on the real
library.
"""
import json
import os
import socket
import struct
import sys
import threading
import time

import numpy as np
import pytest

from detectmateservice_b200 import wire
from detectmateservice_b200.compat import install_shims

install_shims()
import pynng  # noqa: E402

from oracle import schemas as oschemas  # noqa: E402
from oracle.native import NativeOracle  # noqa: E402

from oracle.ref_engine import REF_DIR as REF_SRC  # noqa: E402


# ------------------------------------------------------------------------------------------
# wire codec vs protobuf's own
# ------------------------------------------------------------------------------------------
def test_wire_parser_schema_matches_protobuf(golden_dir):
    g = json.load(open(os.path.join(golden_dir, "parser_fixture1.json")))
    blob = bytes.fromhex(g["wire_hex"])
    rec = wire.decode_parser_schema(blob)
    assert rec["EventID"] == 1 and rec["variables"] == ["john", "192.168.1.100"]
    assert rec["logFormatVariables"] == g["fields"]["logFormatVariables"] and rec["logID"] == "1"
    assert wire.encode_parser_schema(g["fields"]) == blob          # byte-identical (sorted map, field order)
    assert wire.looks_like_parser_schema(blob)
    assert not wire.looks_like_parser_schema(b"type=USER_ACCT msg=audit(1.0:1): pid=1\n")
    assert not wire.looks_like_parser_schema(b"\n\n")


def test_wire_detector_schema_roundtrip_with_protobuf():
    blob = wire.encode_detector_schema("NewValueDetector", "new_value_detector", "10", 1773848383, ["id2"], 1.0,
                                       [1773848383], "d", 1773848383, {"Global - URL": "Unknown value: '/foobar'"})
    m = oschemas.DetectorSchema()
    m.ParseFromString(blob)
    assert m.detectorID == "NewValueDetector" and m.alertID == "10" and m.score == 1.0
    assert list(m.logIDs) == ["id2"] and list(m.extractedTimestamps) == [1773848383]
    assert dict(m.alertsObtain) == {"Global - URL": "Unknown value: '/foobar'"}
    assert getattr(m, "__version__") == "1.0.0"
    assert m.SerializeToString(deterministic=True) == blob       # same bytes as protobuf's encoder
    back = wire.decode_detector_schema(blob)
    assert back["score"] == 1.0 and back["alertsObtain"] == dict(m.alertsObtain)
    assert wire.split_delimited(wire.frame_delimited([blob, b"", blob])) == [blob, b"", blob]


# ------------------------------------------------------------------------------------------
# SP / PAIR0 transport
# ------------------------------------------------------------------------------------------
def test_pair0_wire_format_tcp_and_ipc(sock_dir):
    """The bytes on the wire are NNG's: 8-byte SP header, PAIR0 = 0x0010, be64 length frames
    (ipc frames carry a leading 0x01)."""
    if not getattr(pynng, "__shim__", False):
        pytest.skip("real pynng installed")
    for addr in ("tcp://127.0.0.1:0", f"ipc://{sock_dir}/w.ipc"):
        srv = pynng.Pair0(recv_timeout=2000)
        if addr.startswith("tcp"):
            s0 = socket.socket()
            s0.bind(("127.0.0.1", 0))
            port = s0.getsockname()[1]
            s0.close()
            addr = f"tcp://127.0.0.1:{port}"
            srv.listen(addr)
            raw = socket.create_connection(("127.0.0.1", port))
            ipc = False
        else:
            srv.listen(addr)
            raw = socket.socket(socket.AF_UNIX)
            raw.connect(addr[len("ipc://"):])
            ipc = True
        raw.sendall(b"\x00SP\x00\x00\x10\x00\x00")
        assert raw.recv(8) == b"\x00SP\x00\x00\x10\x00\x00"
        raw.sendall((b"\x01" if ipc else b"") + struct.pack(">Q", 5) + b"hello")
        assert srv.recv() == b"hello"
        srv.send(b"yo")
        want = (b"\x01" if ipc else b"") + struct.pack(">Q", 2) + b"yo"
        got = b""
        while len(got) < len(want):
            got += raw.recv(64)
        assert got == want
        raw.close()
        srv.close()


def test_pair0_semantics(sock_dir):
    addr = f"ipc://{sock_dir}/p.ipc"
    with pynng.Pair0(recv_timeout=100) as a:
        with pytest.raises(pynng.TryAgain):
            a.send(b"x", block=False)                      # no peer
        a.listen(addr)
        with pytest.raises(pynng.Timeout):
            a.recv()
        with pynng.Pair0(dial=addr, recv_timeout=1000) as b:
            b.send(b"ping")
            assert a.recv() == b"ping"
            a.send(b"pong")
            assert b.recv() == b"pong"
            big = os.urandom(1 << 20)                      # 1 MiB (tests/test_engine_multi_output.py:429)
            b.send(big)
            a.recv_timeout = 5000
            assert a.recv() == big
            for i in range(100):
                b.send(b"%d" % i)
            assert [a.recv() for _ in range(100)] == [b"%d" % i for i in range(100)]
    with pytest.raises(pynng.NNGException):
        a.send(b"closed")


def test_pair0_late_binding_and_reconnect(sock_dir):
    addr = f"ipc://{sock_dir}/late.ipc"
    out = pynng.Pair0()
    out.dial(addr, block=False)                            # nobody listens yet
    with pytest.raises(pynng.TryAgain):
        out.send(b"early", block=False)
    with pynng.Pair0(listen=addr, recv_timeout=2000) as lis:
        deadline = time.time() + 3
        while time.time() < deadline:
            try:
                out.send(b"late", block=False)
                break
            except pynng.TryAgain:
                time.sleep(0.02)
        assert lis.recv() == b"late"
    out.close()


def test_pair0_nonblocking_send_queues_and_oversize_frames(sock_dir):
    """send(block=False) to a connected peer that is not draining does not drop (the reference's
    fan-out, engine.py:234-243, relies on it: tests/test_service_multi_output_integration.py:298-318);
    unknown transports are NotSupported; recv_max_size closes the connection on an oversized frame."""
    addr = f"ipc://{sock_dir}/q.ipc"
    with pynng.Pair0(listen=addr, recv_timeout=2000) as rx, pynng.Pair0(recv_timeout=2000) as tx:
        tx.send_buffer_size = 0
        tx.dial(addr, block=True)
        time.sleep(0.05)
        big = b"y" * (300 << 10)                       # larger than a unix socket buffer: must be queued, not dropped
        for i in range(300):
            tx.send(b"msg %d" % i, block=False)
        tx.send(big, block=False)
        tx.send(b"after", block=False)
        for i in range(300):
            assert rx.recv() == b"msg %d" % i
        assert rx.recv() == big and rx.recv() == b"after"
    with pytest.raises(pynng.exceptions.NotSupported):
        pynng.Pair0(listen="invalid://address")
    addr2 = f"ipc://{sock_dir}/m.ipc"
    with pynng.Pair0(listen=addr2, recv_timeout=300) as rx, pynng.Pair0(dial=addr2) as tx:
        rx.recv_max_size = 1024
        time.sleep(0.05)
        tx.send(b"a" * 1024)
        assert rx.recv() == b"a" * 1024
        tx.send(b"b" * 1025)                           # over the limit: dropped with the connection
        with pytest.raises(pynng.Timeout):
            rx.recv()


def test_inproc_transport():
    with pynng.Pair0(listen="inproc://t1", recv_timeout=500) as a, pynng.Pair0(dial="inproc://t1", recv_timeout=500) as b:
        b.send(b"abc")
        assert a.recv() == b"abc"
        a.send(b"def")
        assert b.recv() == b"def"
    with pytest.raises(pynng.NNGException):
        pynng.Pair0(listen="ws://127.0.0.1:1")


# ------------------------------------------------------------------------------------------
# engine mirror: the observable behaviour of Engine._run_loop
# ------------------------------------------------------------------------------------------
class _Upper:
    def process(self, raw):
        if raw == b"boom":
            raise RuntimeError("boom")
        return None if raw == b"skip" else raw.upper()


def test_engine_mirror_reply_none_exception_and_fanout(sock_dir):
    from detectmateservice_b200.service import DetectorEngine
    eng_addr = f"ipc://{sock_dir}/e.ipc"
    with DetectorEngine(_Upper(), eng_addr) as eng:
        with pynng.Pair0(dial=eng_addr, recv_timeout=1000) as c:
            c.send(b"hi")
            assert c.recv() == b"HI"                       # no outputs: reply on the input socket
            c.send(b"skip")
            c.recv_timeout = 150
            with pytest.raises(pynng.Timeout):
                c.recv()                                   # None => nothing sent
            c.send(b"boom")
            with pytest.raises(pynng.Timeout):
                c.recv()                                   # exception => dropped, loop continues
            c.recv_timeout = 1000
            c.send(b"again")
            assert c.recv() == b"AGAIN"
        assert eng.counters["errors"] == 1 and eng.counters["messages"] == 4
    outs = [f"ipc://{sock_dir}/o{i}.ipc" for i in range(3)]
    sinks = [pynng.Pair0(listen=o, recv_timeout=2000) for o in outs[:2]]      # third output never comes up
    eng2_addr = f"ipc://{sock_dir}/e2.ipc"
    with DetectorEngine(_Upper(), eng2_addr, out_addr=outs) as eng:
        time.sleep(0.3)
        with pynng.Pair0(dial=eng2_addr) as c:
            for i in range(10):
                c.send(b"m%d" % i)
            for s in sinks:
                assert [s.recv() for _ in range(10)] == [b"M%d" % i for i in range(10)]
        assert eng.counters["dropped_bytes"] > 0           # the dead output drops, the others deliver
    for s in sinks:
        s.close()


# ------------------------------------------------------------------------------------------
# component plumbing with an oracle-backed device double
# ------------------------------------------------------------------------------------------
class FakeDevice:
    """Stands in for DeviceDetector on a box without a GPU (tests only)."""

    def close(self):
        self.closed = True

    def __init__(self, keys):
        self.keys = [bytes(k) for k in keys]
        self.oracle = NativeOracle([k if not k.startswith(b"\x01") else b"\x02unused%d" % i for i, k in enumerate(self.keys)])
        self.known = [set() for _ in self.keys]
        self.last_n_anomalies = 0
        self._an = []
        self.closed = False

    def process_lines(self, buf, n_train_lines=0, copy=True):
        f, s, m = self.oracle.process(bytes(buf), n_train_lines, want_masks=True)
        arr = np.frombuffer(bytes(buf), dtype=np.uint8)
        starts = np.concatenate([[0], np.nonzero(arr == 10)[0] + 1])
        self._an = [(int(i), int(m[i]), int(starts[i])) for i in np.nonzero(f)[0]]
        self.last_n_anomalies = len(self._an)
        return f, s

    def anomalies(self):
        return self._an

    def process_values(self, records, n_train_records=0, record_bytes=0):
        flags, scores, masks = [], [], []
        for r, vals in enumerate(records):
            m = 0
            for f, v in vals:
                if r < n_train_records:
                    self.known[f].add(v)
                elif v not in self.known[f]:
                    m |= 1 << f
            flags.append(1 if m else 0)
            scores.append(float(bin(m).count("1")))
            masks.append(m)
        self.last_n_anomalies = sum(flags)
        return np.array(flags, np.uint8), np.array(scores, np.float32), np.array(masks, np.uint32)


def _component(cfg, name="B200NewValueDetector"):
    from detectmateservice_b200.component import B200NewValueDetector
    c = B200NewValueDetector(name=name, config=cfg)
    c._det = FakeDevice([m.key for m in c.monitors])
    c.clock = lambda: 1773848383
    return c


def test_component_record_mode_docs_golden(golden_dir):
    """The documented example (docs/getting_started.md:423-435,510) through the plugin surface."""
    g = json.load(open(os.path.join(golden_dir, "docs_golden.json")))
    cfg = dict(g["config"], parsers=None, readers=None)       # what core.py:127-133 hands the component
    comp = _component(cfg)
    outs = []
    for i, url in enumerate(g["urls"]):
        rec = {"EventID": 0, "logID": f"id{i}", "logFormatVariables": {"URL": url, "Time": "18/Mar/2026:11:43:30 +0000"}}
        outs.append(comp.process(wire.encode_parser_schema(rec)))
    assert outs[0] is None and outs[1] is None
    m = oschemas.DetectorSchema()
    m.ParseFromString(outs[2])
    e = g["expected"]
    assert (m.detectorID, m.detectorType, m.alertID, m.score, m.description) == (
        e["detectorID"], e["detectorType"], e["alertID"], e["score"], e["description"])
    assert dict(m.alertsObtain) == e["alertsObtain"] and list(m.logIDs) == ["id2"]
    assert list(m.extractedTimestamps) == [1773848383] and getattr(m, "__version__") == "1.0.0"


def test_component_matches_oracle_on_record_stream():
    from oracle.nvd import NewValueDetectorOracle
    cfg = {"detectors": {"NewValueDetector": {
        "method_type": "new_value_detector", "data_use_training": 3, "auto_config": False, "params": {},
        "global": {"g": {"header_variables": [{"pos": "level"}]}},
        "events": {1: {"test": {"params": {}, "variables": [{"pos": 0, "name": "var1"}],
                                "header_variables": [{"pos": "user"}]}}}}}}
    comp = _component(cfg)
    orc = NewValueDetectorOracle(config=cfg, clock=lambda: 1773848383)
    recs = [
        {"EventID": 1, "logID": "1", "variables": ["a"], "logFormatVariables": {"level": "INFO", "user": "x", "Time": "1634567890"}},
        {"EventID": 2, "logID": "2", "variables": ["zzz"], "logFormatVariables": {"level": "WARN"}},
        {"EventID": 1, "logID": "3", "variables": ["b"], "logFormatVariables": {"level": "INFO", "user": "y"}},
        {"EventID": 1, "logID": "4", "variables": ["c"], "logFormatVariables": {"level": "ERR", "user": "x", "Time": "1634567891"}},
        {"EventID": 2, "logID": "5", "variables": ["c"], "logFormatVariables": {"level": "INFO"}},
        {"EventID": 1, "logID": "6", "variables": ["a"], "logFormatVariables": {"level": "WARN", "user": "q"}},
    ]
    for r in recs:
        blob = wire.encode_parser_schema(r)
        got, want = comp.process(blob), orc.process(blob)
        assert (got is None) == (want is None)
        if got is not None:
            a, b = oschemas.DetectorSchema(), oschemas.DetectorSchema()
            a.ParseFromString(got)
            b.ParseFromString(want)
            assert dict(a.alertsObtain) == dict(b.alertsObtain) and a.score == b.score and a.alertID == b.alertID
            assert list(a.extractedTimestamps) == list(b.extractedTimestamps) and list(a.logIDs) == list(b.logIDs)


def test_component_raw_mode_alerts_and_compact(golden_dir):
    from detectmateservice_b200.component import decode_compact
    exp = json.load(open(os.path.join(golden_dir, "audit_sample.expected.json")))
    buf = open(os.path.join(golden_dir, "audit_sample.log"), "rb").read()
    base = {"method_type": "new_value_detector", "data_use_training": exp["n_train"], "auto_config": False,
            "global": {"g": {"header_variables": [{"pos": k} for k in exp["keys"]]}}}
    comp = _component({"detectors": {"B200NewValueDetector": dict(base, params={"output_format": "compact"})}})
    f, s = decode_compact(comp.process(buf))
    assert f.tolist() == exp["flags"] and s.tolist() == exp["scores"]
    comp = _component({"detectors": {"B200NewValueDetector": base}})
    half = buf[:buf.index(b"\n", len(buf) // 2) + 1]
    out1 = comp.process(half)                                   # training window + some detection
    rest = bytearray(buf[len(half):])
    out2 = comp.process(memoryview(rest)[:len(rest) // 2 + 1 + rest[len(rest) // 2:].index(b"\n")])
    out2b = comp.process(rest[len(rest) // 2 + 1 + rest[len(rest) // 2:].index(b"\n"):])   # any bytes-like is accepted
    alerts = [wire.decode_detector_schema(b) for o in (out1, out2, out2b) if o for b in wire.split_delimited(o)]
    want_idx = [i for i, fl in enumerate(exp["flags"]) if fl]
    assert [int(a["logIDs"][0]) for a in alerts] == want_idx
    assert [a["score"] for a in alerts] == [exp["scores"][i] for i in want_idx]
    assert [a["alertID"] for a in alerts] == [str(10 + i) for i in range(len(want_idx))]
    first = alerts[0]
    assert first["detectorID"] == "NewValueDetector" and first["detectorType"] == "new_value_detector"
    assert all(k.startswith("Global - ") and v.startswith("Unknown value: '") for k, v in first["alertsObtain"].items())
    assert first["extractedTimestamps"][0] > 1600000000        # audit stamp seconds (R-tok L7)
    # a message holding ONE anomalous record yields a bare DetectorSchema (fluentout parses one per message)
    one = comp.process(b"type=NEVER_SEEN msg=audit(1642723741.072:1): pid=1\n")
    assert wire.decode_detector_schema(one)["alertsObtain"] == {"Global - type": "Unknown value: 'NEVER_SEEN'"}
    assert comp.process(b"type=USER_ACCT msg=audit(1642723741.072:2): pid=1\n") is None


def test_component_config_validation():
    from detectmateservice_b200.component import B200NewValueDetector, parse_monitors, select_component_config
    cfg = select_component_config({"detectors": {"X": {"params": {"all_threshold": 1, "device": 3}, "global": {}}}}, "X")
    assert cfg["threshold"] == 1 and cfg["device"] == 3 and "params" not in cfg
    with pytest.raises(ValueError):
        B200NewValueDetector(config={"detectors": {"B200NewValueDetector": {"auto_config": True}}})
    with pytest.raises(ValueError):
        B200NewValueDetector(config={"detectors": {"B200NewValueDetector": {"params": {"input_format": "xml"}}}})
    mons = parse_monitors({"global": {"g": {"header_variables": [{"pos": "type"}, {"pos": "a b"}]}},
                           "events": {"7": {"i": {"variables": [{"pos": 2, "name": "v"}]}}}})
    assert [m.alert_key for m in mons] == ["Global - type", "Global - a b", "EventID 7 - v"]
    assert mons[0].key == b"type" and mons[1].key.startswith(b"\x01") and mons[2].key.startswith(b"\x01")
    from detectmatelibrary.common.core import CoreComponent
    assert isinstance(B200NewValueDetector(config={}), CoreComponent)


def test_process_records_retries_with_room_for_empty_records():
    """DeviceDetector.process_records sizes its outputs for records of >= 2 bytes and tries again, one entry per byte,
    when the library reports that the batch holds more (a batch of empty ParserSchema records: one zero byte each)."""
    import ctypes as C
    from detectmateservice_b200 import _lib
    from detectmateservice_b200.detector import DeviceDetector
    calls = []

    class StubLib:
        def dm_process_records(self, h, buf, nbytes, n_train, flags_p, scores_p, masks_p, cap, n_rec, n_anom):
            calls.append(cap)
            n = buf.count(b"\0")                                  # (every record of the stub batch is empty)
            if n > cap:
                return _lib.DM_ERR_CAPACITY
            C.cast(n_rec, C.POINTER(C.c_uint64))[0] = n
            C.cast(n_anom, C.POINTER(C.c_uint64))[0] = 0
            return _lib.DM_OK

    d = object.__new__(DeviceDetector)
    d._lib, d._h = StubLib(), None
    f, s_, m = d.process_records(b"\0" * 10)
    assert calls == [6, 11] and f.size == 10 and s_.size == 10 and m.size == 10
    calls.clear()
    f, _, _ = d.process_records(b"\0\0")
    assert calls == [2] and f.size == 2


def test_training_window_ends_even_when_the_table_is_full():
    """DM_ERR_TABLE_FULL on a training message: the engine drops the message (the exception propagates), but its
    records count as seen, so the training window ends instead of failing forever."""
    from detectmateservice_b200._lib import DmError, DM_ERR_TABLE_FULL, DM_ERR_CUDA
    from detectmateservice_b200.component import B200NewValueDetector

    class FullDevice(FakeDevice):
        def __init__(self, keys, code):
            super().__init__(keys)
            self.code = code

        def process_lines(self, *a, **k):
            raise DmError(self.code, "known-set table over its load limit")

    cfg = {"detectors": {"B200NewValueDetector": {"method_type": "new_value_detector", "data_use_training": 3,
                                                  "global": {"g": {"header_variables": [{"pos": "type"}]}}}}}
    c = B200NewValueDetector(config=cfg)
    c._det = FullDevice([m.key for m in c.monitors], DM_ERR_TABLE_FULL)
    with pytest.raises(DmError):
        c.process(b"type=A\ntype=B\n")
    assert c.n_seen == 2
    with pytest.raises(DmError):
        c.process(b"type=C\ntype=D")
    assert c.n_seen == 4                                          # training (3 records) is over
    c._det = FullDevice([m.key for m in c.monitors], DM_ERR_CUDA)
    c.n_seen = 0
    with pytest.raises(DmError):
        c.process(b"type=A\n")
    assert c.n_seen == 0                                          # any other failure: the message simply did not happen


def test_component_reconfigure_decides_what_has_to_be_rebuilt():
    """reconfigure(): scalar parameters apply in place, a change of the monitored fields / log_format / geometry asks
    for a new device configuration (no device is touched here: the handle is created lazily)."""
    from detectmateservice_b200.component import B200NewValueDetector
    base = {"method_type": "new_value_detector", "data_use_training": 5,
            "global": {"g": {"header_variables": [{"pos": "type"}, {"pos": "res"}]}}}
    c = B200NewValueDetector(config={"detectors": {"B200NewValueDetector": base}})
    c.n_seen = 3
    assert c.reconfigure({"detectors": {"B200NewValueDetector": dict(base, data_use_training=9,
                                                                       params={"output_format": "compact"})}}) is False
    assert (c.data_use_training, c.output_format, c.n_seen) == (9, "compact", 3)
    assert c.reconfigure({"detectors": {"B200NewValueDetector": dict(base, **{"global": {"g": {"header_variables": [{"pos": "type"}]}}})}}) is True
    assert [m.pos for m in c.monitors] == ["type"] and c.n_seen == 0 and c.data_use_training == 5
    assert c.reconfigure({"detectors": {"B200NewValueDetector": dict(base, **{"global": {"g": {"header_variables": [{"pos": "type"}]}}},
                                                                       params={"log_format": "type=<type> <Content>"})}}) is True
    assert c.logformat is not None
    with pytest.raises(ValueError):
        c.reconfigure({"detectors": {"B200NewValueDetector": {"auto_config": True}}})
    assert c.logformat is not None                               # a rejected configuration changes nothing


@pytest.mark.skipif(not os.path.isdir(REF_SRC), reason="the reference service is not in oracle/_ref (make -C oracle ref)")
def test_service_subclass_forwards_reconfigure(tmp_path, sock_dir, monkeypatch):
    """Service.reconfigure (core.py:299-345) stores the new configuration; the B200 subclass hands it to the
    detector before the next message (the device handle is a double here)."""
    import yaml
    monkeypatch.syspath_prepend(REF_SRC)
    from service.settings import ServiceSettings
    from detectmateservice_b200.service import b200_detector_service
    def det_cfg(keys, n_train):
        return {"detectors": {"B200NewValueDetector": {"method_type": "new_value_detector", "auto_config": False,
                "data_use_training": n_train, "global": {"g": {"header_variables": [{"pos": k} for k in keys]}}}}}
    cfg_file = tmp_path / "detector_config.yaml"
    cfg_file.write_text(yaml.safe_dump(det_cfg(["type"], 1)))
    Svc = b200_detector_service()
    svc = Svc(settings=ServiceSettings(component_name="b200-reconf", engine_addr=f"ipc://{sock_dir}/r.ipc", config_file=cfg_file,
                                       log_dir=tmp_path / "logs", log_to_file=False, log_to_console=False, http_port=18127,
                                       engine_autostart=False))
    try:
        assert [m.pos for m in svc.detector.monitors] == ["type"]
        svc.detector._det = FakeDevice([m.key for m in svc.detector.monitors])
        assert svc.process(b"type=A res=ok\n") is None                       # training record
        assert svc.reconfigure(det_cfg(["type", "res"], 1), persist=True) == "reconfigure: ok"
        assert [m.pos for m in svc.detector.monitors] == ["type"]            # not before the next message
        real_reconf = svc.detector.reconfigure

        def reconf(cfg):
            rebuilt = real_reconf(cfg)
            svc.detector._det = FakeDevice([m.key for m in svc.detector.monitors])
            return rebuilt
        svc.detector.reconfigure = reconf
        assert svc.process(b"type=A res=ok\n") is None                       # rebuilt: trains again
        assert [m.pos for m in svc.detector.monitors] == ["type", "res"] and svc._pending_config is None
        out = svc.process(b"type=A res=bad\n")
        assert wire.decode_detector_schema(out)["alertsObtain"] == {"Global - res": "Unknown value: 'bad'"}
        assert "res" in cfg_file.read_text()                                 # persisted by the reference's manager
    finally:
        try:
            svc.stop()
        except Exception:
            pass


# ------------------------------------------------------------------------------------------
# the UNMODIFIED reference service, with the shims, loading the B200 component
# ------------------------------------------------------------------------------------------
@pytest.mark.skipif(not os.path.isdir(REF_SRC), reason="the reference service is not in oracle/_ref (make -C oracle ref)")
def test_reference_service_loads_b200_component(tmp_path, sock_dir, monkeypatch, golden_dir):
    import yaml
    monkeypatch.syspath_prepend(REF_SRC)
    from service.core import Service                     # reference code, imported unmodified
    from service.settings import ServiceSettings
    from service.features.component_loader import ComponentLoader
    import detectmateservice_b200.component as comp_mod

    g = json.load(open(os.path.join(golden_dir, "docs_golden.json")))
    cfg_file = tmp_path / "detector_config.yaml"
    det_cfg = dict(g["config"]["detectors"]["NewValueDetector"])
    cfg_file.write_text(yaml.safe_dump({"detectors": {"B200NewValueDetector": det_cfg}}))
    # the component is created by the reference's loader; give it the oracle-backed double
    real_init = comp_mod.B200NewValueDetector.__init__

    def init(self, *a, **k):
        real_init(self, *a, **k)
        self._det = FakeDevice([m.key for m in self.monitors])
    monkeypatch.setattr(comp_mod.B200NewValueDetector, "__init__", init)

    addr = f"ipc://{sock_dir}/svc.ipc"
    settings = ServiceSettings(component_type="detectmateservice_b200.component.B200NewValueDetector",
                               component_name="b200-det", engine_addr=addr, config_file=cfg_file,
                               log_dir=tmp_path / "logs", log_to_file=False, log_to_console=False,
                               http_port=18123, engine_autostart=False)
    svc = Service(settings=settings)
    assert isinstance(svc.library_component, comp_mod.B200NewValueDetector)
    assert settings.component_config_class.endswith("B200NewValueDetectorConfig")   # found by the resolver
    svc.start()
    try:
        with pynng.Pair0(dial=addr, recv_timeout=300) as c:
            for i, url in enumerate(g["urls"]):
                rec = {"EventID": 0, "logID": f"id{i}", "logFormatVariables": {"URL": url}}
                c.send(wire.encode_parser_schema(rec))
                if i < 2:
                    with pytest.raises(pynng.Timeout):
                        c.recv()                          # training => no reply (engine.py:196-198)
                else:
                    alert = wire.decode_detector_schema(c.recv())
                    assert alert["alertsObtain"] == g["expected"]["alertsObtain"] and alert["alertID"] == "10"
    finally:
        svc.stop()
    inst = ComponentLoader.load_component("detectmateservice_b200.component.B200NewValueDetector", {})
    assert isinstance(inst, comp_mod.B200NewValueDetector)


def test_component_chunks_messages_larger_than_the_device_batch(golden_dir):
    from detectmateservice_b200.component import decode_compact
    exp = json.load(open(os.path.join(golden_dir, "audit_sample.expected.json")))
    buf = open(os.path.join(golden_dir, "audit_sample.log"), "rb").read()
    base = {"method_type": "new_value_detector", "data_use_training": exp["n_train"], "auto_config": False,
            "global": {"g": {"header_variables": [{"pos": k} for k in exp["keys"]]}}}
    whole = _component({"detectors": {"B200NewValueDetector": base}})
    small = _component({"detectors": {"B200NewValueDetector": dict(base, params={"max_batch_bytes": 5000})}})
    a = [wire.decode_detector_schema(b) for b in wire.split_delimited(whole.process(buf))]
    b = [wire.decode_detector_schema(x) for x in wire.split_delimited(small.process(buf))]
    assert [(x["logIDs"], x["alertID"], x["alertsObtain"]) for x in a] == [(x["logIDs"], x["alertID"], x["alertsObtain"]) for x in b]
    comp = _component({"detectors": {"B200NewValueDetector": dict(base, params={"max_batch_bytes": 3000, "output_format": "compact"})}})
    f, s = decode_compact(comp.process(buf))
    assert f.tolist() == exp["flags"] and s.tolist() == exp["scores"]
    with pytest.raises(ValueError):
        _component({"detectors": {"B200NewValueDetector": dict(base, params={"max_batch_bytes": 100})}}).process(buf)


# ------------------------------------------------------------------------------------------
# BASELINE config 1: reader -> parser -> detector over the sample audit log, one process,
# chained over the transport exactly like docker-compose.yml:16-40 chains the services
# (out_addr of one stage = engine_addr of the next).  No GPU: the detector's device is the
# oracle-backed double; reader and parser are minimal stand-ins for the library's
# LogFileReader / MatcherParser (not on the hot path) that speak the real wire schemas.
# ------------------------------------------------------------------------------------------
class _ReaderStage:
    """`read` request -> next log line as LogSchema-like ParserSchema input (one per message)."""

    def __init__(self, lines):
        self.lines, self.i = lines, 0

    def process(self, raw):
        if self.i >= len(self.lines):
            return None
        line = self.lines[self.i]
        self.i += 1
        return b"%d\t" % self.i + line                       # logID \t raw line


class _ParserStage:
    """raw line -> ParserSchema whose logFormatVariables hold every key=value field (R-tok)."""

    def process(self, raw):
        from oracle import rtok
        log_id, line = raw.split(b"\t", 1)
        fields = {k.decode("latin-1"): v.decode("latin-1") for k, v in rtok.tokenize_line(line).items()}
        t = rtok.line_time(line)
        if t is not None:
            fields["Time"] = t.decode()
        return wire.encode_parser_schema({"EventID": 0, "logID": log_id.decode(), "log": line.decode("latin-1"),
                                          "logFormatVariables": fields})


def test_config1_reader_parser_detector_pipeline(sock_dir, golden_dir):
    from detectmateservice_b200.service import DetectorEngine
    exp = json.load(open(os.path.join(golden_dir, "audit_sample.expected.json")))
    lines = open(os.path.join(golden_dir, "audit_sample.log"), "rb").read().split(b"\n")[:-1]
    cfg = {"detectors": {"B200NewValueDetector": {
        "method_type": "new_value_detector", "data_use_training": exp["n_train"], "auto_config": False,
        "global": {"g": {"header_variables": [{"pos": k} for k in exp["keys"]]}}}}}
    det = _component(cfg)
    a_reader, a_parser, a_det, a_out = (f"ipc://{sock_dir}/{n}.ipc" for n in ("reader", "parser", "detector", "out"))
    sink = pynng.Pair0(listen=a_out, recv_timeout=300)
    with DetectorEngine(det, a_det, out_addr=[a_out]) as e_det, \
            DetectorEngine(_ParserStage(), a_parser, out_addr=[a_det]), \
            DetectorEngine(_ReaderStage(lines), a_reader, out_addr=[a_parser]):
        time.sleep(0.4)                                       # background dials connect
        alerts = []
        with pynng.Pair0(dial=a_reader) as trigger:
            for i in range(len(lines)):
                trigger.send(b"read")
                # the engines drop on a full output queue (engine.py:233-241), like the
                # reference: pace the source on the last stage's message counter
                t_end = time.monotonic() + 5
                while e_det.counters["messages"] <= i and time.monotonic() < t_end:
                    time.sleep(0.0005)
                assert e_det.counters["messages"] == i + 1
                if exp["flags"][i]:
                    alerts.append(wire.decode_detector_schema(sink.recv()))
            with pytest.raises(pynng.Timeout):
                sink.recv()                                   # nothing else was sent
    sink.close()
    want = [i for i, f in enumerate(exp["flags"]) if f]
    assert [int(a["logIDs"][0]) - 1 for a in alerts] == want
    assert [a["score"] for a in alerts] == [exp["scores"][i] for i in want]
    keys = exp["keys"]
    for a, i in zip(alerts, want):
        assert sorted(a["alertsObtain"]) == sorted(f"Global - {keys[b]}" for b in range(len(keys)) if exp["masks"][i] >> b & 1)
        assert a["extractedTimestamps"][0] > 1600000000


def test_engine_lends_receive_frames(sock_dir, golden_dir):
    """alloc_frame / release_frame: the engine hands the transport the processor's receive
    buffers for large messages and gives each one back after process() (also on errors)."""
    from detectmateservice_b200.service import DetectorEngine

    class Lender:
        accepts_bytes_like = True

        def __init__(self):
            self.slots = [bytearray(1 << 20) for _ in range(2)]
            self.busy = [False, False]
            self.n_seen = 0
            self.seen, self.kinds, self.lent, self.released = [], [], 0, 0

        def alloc_frame(self, n):
            for i, b in enumerate(self.busy):
                if not b and n <= len(self.slots[i]):
                    self.busy[i] = True
                    self.lent += 1
                    return memoryview(self.slots[i])[:n]
            return None

        def release_frame(self, frame):
            if isinstance(frame, memoryview):
                i = [j for j, s in enumerate(self.slots) if frame.obj is s][0]
                self.busy[i] = False
                self.released += 1

        def process(self, raw):
            self.n_seen += 1
            self.kinds.append(type(raw).__name__)
            self.seen.append(bytes(raw[:8]) + bytes(raw[-8:]))
            if bytes(raw[:4]) == b"boom":
                raise RuntimeError("boom")
            return None

    p = Lender()
    addr = f"ipc://{sock_dir}/lend.ipc"
    msgs = [bytes([65 + i]) * (200000 + i) for i in range(6)] + [b"boom" * 50000, b"small", b"Z" * (2 << 20)]
    with DetectorEngine(p, addr) as e, pynng.Pair0(dial=addr) as s:
        time.sleep(0.2)
        for i, m in enumerate(msgs):
            s.send(m)
            t_end = time.monotonic() + 5                      # paced: a free slot for every frame
            while e.counters["messages"] <= i and time.monotonic() < t_end:
                time.sleep(0.002)
        time.sleep(0.05)
        assert e.counters["messages"] == len(msgs) and e.counters["errors"] == 1
    assert p.seen == [m[:8] + m[-8:] for m in msgs]              # content and order intact
    assert p.kinds[:7] == ["memoryview"] * 7                      # large frames landed in lent slots
    assert p.kinds[7] == "bytes"                                  # small frames are plain bytes
    assert p.kinds[8] == "bytearray"                              # too large for a slot -> transport allocates
    assert p.lent == 7 and p.released == 7 and p.busy == [False, False]


def test_numa_helpers(tmp_path):
    from detectmateservice_b200 import numa
    assert numa.parse_cpulist("0-3,8,10-11\n") == {0, 1, 2, 3, 8, 10, 11}
    assert numa.parse_cpulist("") == set()
    with numa.bound_to_gpu_node(0) as cpus:                # no GPU here: topology unknown, affinity untouched
        assert cpus is None or isinstance(cpus, set)
    assert os.sched_getaffinity(0) == os.sched_getaffinity(0)
