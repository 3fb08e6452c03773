"""The reference-facing plugin (B200NewValueDetector) on the real CUDA library.  Needs a B200."""
import json
import os
import time

import numpy as np
import pytest

from detectmateservice_b200 import wire
from oracle.native import NativeOracle
from oracle.nvd import NewValueDetectorOracle
from oracle import schemas as oschemas

pytestmark = pytest.mark.gpu


def _comp(cfg, name="B200NewValueDetector"):
    from detectmateservice_b200.component import B200NewValueDetector
    c = B200NewValueDetector(name=name, config=cfg)
    c.clock = lambda: 1773848383
    return c


def test_record_mode_docs_golden(golden_dir):
    g = json.load(open(os.path.join(golden_dir, "docs_golden.json")))
    comp = _comp(dict(g["config"], parsers=None, readers=None))
    outs = []
    for i, url in enumerate(g["urls"] + ["/hello", "/foobar"]):
        rec = {"EventID": 0, "logID": f"id{i}", "logFormatVariables": {"URL": url, "Time": "1634567890"}}
        outs.append(comp.process(wire.encode_parser_schema(rec)))
    assert [o is not None for o in outs] == [False, False, True, False, True]
    a = wire.decode_detector_schema(outs[2])
    e = g["expected"]
    assert a["alertsObtain"] == e["alertsObtain"] and a["alertID"] == "10" and a["score"] == 1.0
    assert a["detectorID"] == e["detectorID"] and a["description"] == e["description"]
    assert a["extractedTimestamps"] == [1634567890]
    assert wire.decode_detector_schema(outs[4])["alertID"] == "11"        # detection never inserts
    st = comp.stats()
    assert st["lines"] == 5 and st["train_lines"] == 2 and st["anomalies"] == 2 and st["known_keys"] == 2
    comp.close()


def test_record_mode_matches_oracle_on_events_config():
    cfg = {"detectors": {"NewValueDetector": {
        "method_type": "new_value_detector", "data_use_training": 40, "auto_config": False, "params": {},
        "global": {"g": {"header_variables": [{"pos": "level"}]}},
        "events": {1: {"t": {"params": {}, "variables": [{"pos": 0, "name": "var1"}], "header_variables": [{"pos": "user"}]}},
                   2: {"t": {"variables": [{"pos": 1}]}}}}}}
    comp = _comp(cfg)
    orc = NewValueDetectorOracle(config=cfg, clock=lambda: 1773848383)
    r = np.random.Generator(np.random.PCG64(3))
    n_alerts = 0
    for i in range(200):
        rec = {"EventID": int(r.integers(1, 4)), "logID": str(i),
               "variables": ["v%d" % r.integers(0, 6), "w%d" % r.integers(0, 9 if i > 60 else 4)],
               "logFormatVariables": {"level": ["INFO", "WARN", "ERR", "DBG"][int(r.integers(0, 4 if i > 60 else 2))],
                                      "user": "u%d" % r.integers(0, 5)}}
        blob = wire.encode_parser_schema(rec)
        got, want = comp.process(blob), orc.process(blob)
        assert (got is None) == (want is None), i
        if got is not None:
            n_alerts += 1
            a = wire.decode_detector_schema(got)
            b = oschemas.DetectorSchema()
            b.ParseFromString(want)
            assert a["alertsObtain"] == dict(b.alertsObtain) and a["score"] == b.score and a["alertID"] == b.alertID
    assert n_alerts > 10
    comp.close()


def test_raw_mode_alerts_audit_sample(golden_dir):
    from detectmateservice_b200.component import decode_compact
    exp = json.load(open(os.path.join(golden_dir, "audit_sample.expected.json")))
    buf = open(os.path.join(golden_dir, "audit_sample.log"), "rb").read()
    base = {"method_type": "new_value_detector", "data_use_training": exp["n_train"], "auto_config": False,
            "global": {"g": {"header_variables": [{"pos": k} for k in exp["keys"]]}}}
    comp = _comp({"detectors": {"B200NewValueDetector": dict(base, params={"output_format": "compact"})}})
    f, s = decode_compact(comp.process(buf))
    assert f.tolist() == exp["flags"] and s.tolist() == exp["scores"]
    comp.close()
    comp = _comp({"detectors": {"B200NewValueDetector": base}})
    half = buf[:buf.index(b"\n", len(buf) // 2) + 1]
    outs = [comp.process(half), comp.process(buf[len(half):])]
    alerts = [wire.decode_detector_schema(b) for o in outs if o for b in wire.split_delimited(o)]
    want_idx = [i for i, fl in enumerate(exp["flags"]) if fl]
    assert [int(a["logIDs"][0]) for a in alerts] == want_idx
    assert [a["score"] for a in alerts] == [exp["scores"][i] for i in want_idx]
    keys = exp["keys"]
    for a, i in zip(alerts, want_idx):
        assert sorted(a["alertsObtain"]) == sorted(f"Global - {keys[b]}" for b in range(len(keys)) if exp["masks"][i] >> b & 1)
    comp.close()


def test_engine_pipeline_raw_messages(sock_dir):
    """sender -> [ipc] -> DetectorEngine(B200NewValueDetector) -> [ipc] -> sink, 64k-record messages
    (BASELINE config 3 topology at small scale)."""
    import pynng
    from detectmateservice_b200.service import DetectorEngine
    from detectmateservice_b200.component import decode_compact
    from detectmateservice_b200.synth import AuditSynth, MONITORED_KEYS
    g = AuditSynth(seed=77)
    msgs = [g.batch(8192, inject=False)[0]] + [g.batch(8192, inject=True)[0] for _ in range(5)]
    keys = [k.encode() for k in MONITORED_KEYS]
    orc = NativeOracle(keys)
    want = [orc.process(msgs[0], 8192)] + [orc.process(m, 0) for m in msgs[1:]]
    cfg = {"detectors": {"B200NewValueDetector": {
        "method_type": "new_value_detector", "data_use_training": 8192, "auto_config": False,
        "params": {"output_format": "compact", "max_batch_bytes": 4 << 20},
        "global": {"g": {"header_variables": [{"pos": k} for k in MONITORED_KEYS]}}}}}
    comp = _comp(cfg)
    eng_addr, out_addr = f"ipc://{sock_dir}/det.ipc", f"ipc://{sock_dir}/out.ipc"
    sink = pynng.Pair0(listen=out_addr, recv_timeout=20000)
    with DetectorEngine(comp, eng_addr, out_addr=[out_addr]) as eng:
        time.sleep(0.3)
        with pynng.Pair0(dial=eng_addr) as tx:
            for m, (wf, ws, _) in zip(msgs, want):
                tx.send(m)
                f, s = decode_compact(sink.recv())
                assert (f == wf).all() and (s == ws).all()
        assert eng.counters["errors"] == 0 and eng.counters["processed_lines"] == 6 * 8192
        # the frames were received straight into the component's pinned slots, all returned
        assert comp._frames and len(comp._frames) == comp.FRAME_SLOTS and not any(b for _, _, b in comp._frames)
        assert all(t.is_pinned() for t, _, _ in comp._frames)
        # burst: more messages in flight than slots -> the reader stalls on a slot, nothing is lost
        comp.reset_state()
        with pynng.Pair0(dial=eng_addr) as tx:
            time.sleep(0.2)
            for m in msgs:
                tx.send(m)
            for wf, ws, _ in want:
                f, s = decode_compact(sink.recv())
                assert (f == wf).all() and (s == ws).all()
        assert eng.counters["errors"] == 0 and not any(b for _, _, b in comp._frames)
    sink.close()
    comp.close()


def test_large_messages_are_pipelined_and_match_the_oracle():
    """Large messages are cut at record boundaries into pieces that overlap copy and compute
    (component._detect_pipelined): same flags, scores and alerts as the oracle on the whole message."""
    from detectmateservice_b200.component import decode_compact
    from detectmateservice_b200.synth import AuditSynth, MONITORED_KEYS
    g = AuditSynth(seed=99)
    train, _ = g.batch(8192, inject=False)
    msgs = [g.batch(40000, inject=True)[0], g.batch_varlen(30000, inject=True)[0]]        # ~10 MiB each
    keys = [k.encode() for k in MONITORED_KEYS]
    base = {"method_type": "new_value_detector", "data_use_training": 8192, "auto_config": False,
            "global": {"g": {"header_variables": [{"pos": k} for k in MONITORED_KEYS]}}}
    for fmt in ("compact", "alerts"):
        orc = NativeOracle(keys)
        orc.process(train, 8192)
        comp = _comp({"detectors": {"B200NewValueDetector": dict(base, params={"output_format": fmt, "max_batch_bytes": 32 << 20})}})
        comp.PIPE_MIN_BYTES = comp.PIPE_PIECE_BYTES = 4 << 20          # (the defaults only cut much larger messages)
        assert comp.process(train) is None or fmt == "compact"
        lines_before = 8192
        for m in msgs:
            assert len(m) >= comp.PIPE_MIN_BYTES
            wf, ws, wm = orc.process(m, 0, want_masks=True)
            out = comp.process(m)
            if fmt == "compact":
                f, s = decode_compact(out)
                assert (f == wf).all() and (s == ws).all()
            else:
                alerts = [wire.decode_detector_schema(b) for b in wire.split_delimited(out)]
                idx = np.flatnonzero(wf)
                assert [int(a["logIDs"][0]) - lines_before for a in alerts] == idx.tolist()
                assert [a["score"] for a in alerts] == ws[idx].tolist()
                for a, i in zip(alerts, idx):
                    assert sorted(a["alertsObtain"]) == sorted(f"Global - {MONITORED_KEYS[b]}" for b in range(5) if wm[i] >> b & 1)
            lines_before += wf.size
        comp.close()


def test_reconfigure_rebuilds_the_device_configuration(golden_dir):
    """Service.reconfigure -> component.reconfigure (core.py:299-345): new monitored fields take effect on the
    next message, with fresh training; scalar changes keep the learnt state."""
    from detectmateservice_b200.component import decode_compact
    def cfg(keys, n_train):
        return {"detectors": {"B200NewValueDetector": {"method_type": "new_value_detector", "data_use_training": n_train,
                "global": {"g": {"header_variables": [{"pos": k} for k in keys]}}, "params": {"output_format": "compact"}}}}
    train = b"type=A res=ok\ntype=B res=ok\n"
    probe = b"type=A res=bad\ntype=C res=ok\n"
    comp = _comp(cfg(["type"], 2))
    comp.process(train)
    assert decode_compact(comp.process(probe))[0].tolist() == [0, 1]
    assert comp.reconfigure(cfg(["type"], 2)) is False           # nothing changed: state kept
    assert decode_compact(comp.process(probe))[0].tolist() == [0, 1]
    assert comp.reconfigure(cfg(["type", "res"], 2)) is True     # a new monitored field: rebuilt, trains again
    comp.process(train)
    f, s = decode_compact(comp.process(probe))
    assert f.tolist() == [1, 1] and s.tolist() == [1.0, 1.0]
    o = NativeOracle([b"type", b"res"])
    o.process(train, 2)
    assert o.process(probe, 0)[0].tolist() == [1, 1]
    comp.close()
