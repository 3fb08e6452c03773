#!/usr/bin/env python
"""Generate tests/golden/* from the reference checkout (run in the build container only;
/root/reference does not exist on the GPU box, the committed fixtures travel instead).

  audit_sample.log            a 420-record subset of the reference's sample audit log
                              (tests/library_integration/audit.log): the first 250 records,
                              every record of the 7 rare types, and the last 100 records.
  audit_sample.expected.json  flags / scores / unknown-field masks of the oracle
                              (oracle/nvd.py, R-spec) with the first 200 records as training
                              data and monitors type, exe, terminal, acct, res.
  parser_fixture1.json        field values + 201-byte wire image of the first ParserSchema
                              fixture (library_integration_base_fixtures.py:27-43).
  docs_golden.json            the documented NewValueDetector example
                              (docs/getting_started.md:423-435,510).
  audit_stats.json            probe statistics of the full audit.log (SURVEY 8c iv).
  audit_templates.txt         the nine `<*>` templates of the reference's parser test data
                              (tests/library_integration/audit_templates.txt; test DATA, copied
                              verbatim as a fixture like audit_sample.log).
  audit.log.gz                the full audit.log itself, gzip-compressed (test DATA).
  schemas_descriptor.json     the FileDescriptorProto the reference embeds in
                              container/fluentout/schemas_pb.rb:8, as hex.
"""
import collections
import gzip
import json
import os
import re
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
REF = "/root/reference"
OUT = os.path.join(ROOT, "tests", "golden")

from oracle.nvd import NewValueDetectorOracle  # noqa: E402
from oracle import rtok  # noqa: E402
from oracle.schemas import parser_schema_from_dict  # noqa: E402

KEYS = ["type", "exe", "terminal", "acct", "res"]
N_TRAIN = 200


def _ruby_unescape(s: str) -> bytes:
    """The bytes of a double-quoted Ruby string literal's body."""
    out = bytearray()
    i = 0
    simple = {"n": 10, "r": 13, "t": 9, '"': 34, "\\": 92, "e": 27, "a": 7, "b": 8, "f": 12, "v": 11, "0": 0, "#": 35}
    while i < len(s):
        c = s[i]
        if c != "\\":
            out += c.encode("latin-1")
            i += 1
            continue
        n = s[i + 1]
        if n == "x":
            m = re.match(r"[0-9a-fA-F]{1,2}", s[i + 2:i + 4])
            out.append(int(m.group(0), 16))
            i += 2 + len(m.group(0))
        elif n in "01234567":
            m = re.match(r"[0-7]{1,3}", s[i + 1:i + 4])
            out.append(int(m.group(0), 8))
            i += 1 + len(m.group(0))
        else:
            out.append(simple[n])
            i += 2
    return bytes(out)


def main() -> None:
    os.makedirs(OUT, exist_ok=True)
    with open(os.path.join(REF, "tests/library_integration/audit_templates.txt"), "rb") as f:
        open(os.path.join(OUT, "audit_templates.txt"), "wb").write(f.read())
    raw = open(os.path.join(REF, "tests/library_integration/audit.log"), "rb").read()
    open(os.path.join(OUT, "audit.log.gz"), "wb").write(gzip.compress(raw, compresslevel=9, mtime=0))
    lines = rtok.split_records(raw)
    counts = collections.Counter(l.split(b" ")[0][5:].decode() for l in lines)
    rare = {t for t, c in counts.items() if c <= 4}
    pick = sorted(set(range(250)) | {i for i, l in enumerate(lines) if l.split(b" ")[0][5:].decode() in rare}
                  | set(range(len(lines) - 100, len(lines))))
    sample = b"".join(lines[i] + b"\n" for i in pick)
    open(os.path.join(OUT, "audit_sample.log"), "wb").write(sample)

    cfg = {"detectors": {"NewValueDetector": {
        "method_type": "new_value_detector", "data_use_training": N_TRAIN, "auto_config": False,
        "global": {"global_instance": {"header_variables": [{"pos": k} for k in KEYS]}}}}}
    det = NewValueDetectorOracle(config=cfg)
    flags, scores, masks = [], [], []
    for line in rtok.split_records(sample):
        f, s, alerts = det.step_line(line)
        flags.append(int(f))
        scores.append(s)
        m = 0
        for i, k in enumerate(KEYS):
            if f"Global - {k}" in alerts:
                m |= 1 << i
        masks.append(m)
    json.dump({"keys": KEYS, "n_train": N_TRAIN, "n_records": len(flags), "flags": flags, "scores": scores,
               "masks": masks, "known_counts": [len(s) for s in det.known]},
              open(os.path.join(OUT, "audit_sample.expected.json"), "w"))

    lens = [len(l) + 1 for l in lines]
    json.dump({"records": len(lines), "bytes": len(raw), "len_min": min(lens) - 1, "len_max": max(lens) - 1,
               "types": dict(counts)}, open(os.path.join(OUT, "audit_stats.json"), "w"), indent=1, sort_keys=True)

    fx = {"parserType": "LogParser", "parserID": "parser_001", "EventID": 1,
          "template": "User <*> logged in from <*>", "variables": ["john", "192.168.1.100"],
          "parsedLogID": "101", "logID": "1", "log": "User john logged in from 192.168.1.100",
          "logFormatVariables": {"username": "john", "ip": "192.168.1.100", "Time": "1634567890"},
          "receivedTimestamp": 1634567890, "parsedTimestamp": 1634567891}
    wire = parser_schema_from_dict(fx).SerializeToString(deterministic=True)
    json.dump({"fields": fx, "wire_hex": wire.hex(), "wire_len": len(wire)},
              open(os.path.join(OUT, "parser_fixture1.json"), "w"), indent=1)

    json.dump({
        "config": {"detectors": {"NewValueDetector": {
            "method_type": "new_value_detector", "data_use_training": 2, "auto_config": False,
            "global": {"global_instance": {"header_variables": [{"pos": "URL"}]}}}}},
        "urls": ["/hello", "/world", "/foobar"],
        "expected": {"__version__": "1.0.0", "detectorID": "NewValueDetector", "detectorType": "new_value_detector",
                     "alertID": "10", "score": 1.0,
                     "description": "NewValueDetector detects values not encountered in training as anomalies.",
                     "alertsObtain": {"Global - URL": "Unknown value: '/foobar'"}}},
        open(os.path.join(OUT, "docs_golden.json"), "w"), indent=1)

    rb = open(os.path.join(REF, "container/fluentout/schemas_pb.rb"), "r", encoding="latin-1").read()
    lit = re.search(r'descriptor_data = "((?:[^"\\]|\\.)*)"', rb, re.S).group(1)
    json.dump({"source": "container/fluentout/schemas_pb.rb:8 (descriptor_data)", "file_descriptor_hex": _ruby_unescape(lit).hex()},
              open(os.path.join(OUT, "schemas_descriptor.json"), "w"), indent=1)
    print("golden written:", sorted(os.listdir(OUT)), "sample records:", len(pick), "anomalies:", sum(flags))


if __name__ == "__main__":
    main()
