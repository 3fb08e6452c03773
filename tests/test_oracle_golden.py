"""The oracle against every golden vector the reference holds for this path (CPU only)."""
import gzip
import json
import os

import numpy as np
import pytest

from oracle import fingerprint, native, rtok
from oracle.nvd import DummyDetectorOracle, NewValueDetectorOracle
from oracle.schemas import DetectorSchema, ParserSchema, parser_schema_from_dict


def _rec(url, i):
    return parser_schema_from_dict({"EventID": 0, "logID": f"id{i}",
                                    "logFormatVariables": {"URL": url, "Time": "18/Mar/2026:11:43:30 +0000"}}
                                   ).SerializeToString()


def test_docs_golden_new_value_detector(golden_dir):
    """docs/getting_started.md:423-435,498-510: train on /hello,/world; /foobar alerts."""
    g = json.load(open(os.path.join(golden_dir, "docs_golden.json")))
    det = NewValueDetectorOracle(config=g["config"], clock=lambda: 1773848383)
    outs = [det.process(_rec(u, i)) for i, u in enumerate(g["urls"])]
    assert outs[0] is None and outs[1] is None and outs[2] is not None
    m = DetectorSchema()
    m.ParseFromString(outs[2])
    e = g["expected"]
    assert getattr(m, "__version__") == e["__version__"]
    assert m.detectorID == e["detectorID"] and m.detectorType == e["detectorType"]
    assert m.alertID == e["alertID"] and m.score == e["score"] and m.description == e["description"]
    assert dict(m.alertsObtain) == e["alertsObtain"]
    assert list(m.logIDs) == ["id2"] and m.detectionTimestamp == 1773848383
    assert list(m.extractedTimestamps) == [1773848383]      # unparseable Time -> detection time
    # a known value after training stays silent; detection never inserts
    assert det.process(_rec("/hello", 3)) is None
    again = det.process(_rec("/foobar", 4))
    m2 = DetectorSchema()
    m2.ParseFromString(again)
    assert m2.alertID == "11"


def test_dummy_detector_pattern():
    """tests/library_integration/test_detector_integration.py:83-84,89-115,143-144."""
    det = DummyDetectorOracle()
    msg = parser_schema_from_dict({"EventID": 1, "logID": "1"}).SerializeToString()
    outs = [det.process(msg) for _ in range(3)]
    assert [o is not None for o in outs] == [False, True, False]
    m = DetectorSchema()
    m.ParseFromString(outs[1])
    assert m.score == 1.0 and m.description == "Dummy detection process"
    assert "Anomaly detected by DummyDetector" in m.alertsObtain["type"]


def test_audit_sample_expected(golden_dir):
    exp = json.load(open(os.path.join(golden_dir, "audit_sample.expected.json")))
    buf = open(os.path.join(golden_dir, "audit_sample.log"), "rb").read()
    keys = [k.encode() for k in exp["keys"]]
    o = native.NativeOracle(keys)
    f, s, m = o.process(buf, exp["n_train"], want_masks=True)
    assert f.tolist() == exp["flags"] and s.tolist() == exp["scores"] and m.tolist() == exp["masks"]
    assert [o.known_count(i) for i in range(len(keys))] == exp["known_counts"]


def test_audit_stats(golden_dir):
    st = json.load(open(os.path.join(golden_dir, "audit_stats.json")))
    assert st["records"] == 2316 and st["bytes"] == 420842 and st["len_min"] == 127 and st["len_max"] == 311
    assert st["types"]["CRED_ACQ"] == 308 and len(st["types"]) == 15
    raw = gzip.decompress(open(os.path.join(golden_dir, "audit.log.gz"), "rb").read())    # the reference's full audit.log
    assert len(rtok.split_records(raw)) == st["records"] and len(raw) == st["bytes"]


def test_rtok_rules():
    line = (b"type=USER_ACCT msg=audit(1642723741.072:375): pid=10125 uid=0 auid=4294967295 ses=4294967295 "
            b"msg='op=PAM:accounting acct=\"root\" exe=\"/usr/sbin/cron\" hostname=? addr=? terminal=cron res=success'")
    f = rtok.tokenize_line(line)
    assert f[b"type"] == b"USER_ACCT" and f[b"msg"] == b"audit(1642723741.072:375):"      # first msg wins (L6)
    assert f[b"op"] == b"PAM:accounting" and f[b"acct"] == b'"root"' and f[b"res"] == b"success'"
    assert rtok.line_time(line) == b"1642723741.072"
    f = rtok.tokenize_line(b'info="same as a=b, skipping" x=it\'s=5 a=b=c  d= =e "q r"=1')
    assert f == {b"info": b'"same as a=b, skipping"', b"x": b"it's=5", b"s": b"5", b"a": b"b=c", b"d": b""}
    assert rtok.split_records(b"a\n\nb") == [b"a", b"", b"b"] and rtok.split_records(b"a\n") == [b"a"]
    assert rtok.split_records(b"") == [] and rtok.split_records(b"\n") == [b""]


def test_python_and_c_oracle_agree_on_fuzz():
    from util import FUZZ_KEYS, fuzz_lines
    buf = fuzz_lines(7, 3000)
    cfg = {"data_use_training": 1000,
           "global": {"g": {"header_variables": [{"pos": k.decode()} for k in FUZZ_KEYS]}}}
    py = NewValueDetectorOracle(config=cfg)
    pf, ps = py.process_lines(buf)
    c = native.NativeOracle(FUZZ_KEYS)
    cf, cs, _ = c.process(buf, 1000)
    assert cf.tolist() == pf and cs.tolist() == ps
    assert sum(pf) > 50                       # the fuzz really exercises detections
    for i in range(len(FUZZ_KEYS)):
        assert sorted(c.known_values(i)) == sorted(py.known[i])
    py.known_keys()                           # fingerprint-collision audit


def test_fp64_c_matches_python():
    r = np.random.Generator(np.random.PCG64(1))
    for n in list(range(0, 40)) + [63, 64, 65, 255, 1000]:
        v = r.integers(0, 256, n, dtype=np.uint8).tobytes()
        assert native.fp64(v) == fingerprint.fp64(v)
    assert fingerprint.fp64(b"success'") == 0x183383F8678A370B
    assert fingerprint.table_key(3, b"x") != fingerprint.table_key(4, b"x")
