"""The UNMODIFIED reference service (oracle/_ref, see oracle/Makefile) around the real
CUDA library.  Needs a B200.  Covers SURVEY.md 8(a3), 8(b): both plugin routes -- the component loader
(settings.component_type = dotted path; /root/reference/src/service/features/component_loader.py:34-55) and the
Service subclass (core.py:64-69,85-86) -- with the reference's own metrics (core.py:184-200) asserted."""
import json
import os
import sys
import time

import numpy as np
import pytest

from detectmateservice_b200 import wire
from detectmateservice_b200.compat import install_shims
from oracle.native import NativeOracle
from oracle.ref_engine import reference_path as _reference_src

pytestmark = pytest.mark.gpu


needs_ref = pytest.mark.skipif(_reference_src() is None, reason="the reference service is not in oracle/_ref (make -C oracle ref)")


def _metric(counter, **labels):
    return counter.labels(**labels)._value.get()


@needs_ref
def test_reference_service_loads_the_cuda_component(tmp_path, sock_dir, monkeypatch, golden_dir):
    import yaml
    monkeypatch.syspath_prepend(_reference_src())
    install_shims()
    import pynng
    from service.core import Service, data_processed_lines_total, data_processed_bytes_total
    from service.settings import ServiceSettings
    import detectmateservice_b200.component as comp_mod

    g = json.load(open(os.path.join(golden_dir, "docs_golden.json")))
    cfg_file = tmp_path / "detector_config.yaml"
    det_cfg = dict(g["config"]["detectors"]["NewValueDetector"])
    cfg_file.write_text(yaml.safe_dump({"detectors": {"B200NewValueDetector": det_cfg}}))
    addr = f"ipc://{sock_dir}/svc.ipc"
    settings = ServiceSettings(component_type="detectmateservice_b200.component.B200NewValueDetector",
                               component_name="b200-det-gpu", engine_addr=addr, config_file=cfg_file,
                               log_dir=tmp_path / "logs", log_to_file=False, log_to_console=False,
                               http_port=18231, engine_autostart=False)
    svc = Service(settings=settings)
    assert isinstance(svc.library_component, comp_mod.B200NewValueDetector)
    labels = dict(component_type=svc.component_type, component_id=svc.component_id)
    lines0, bytes0 = _metric(data_processed_lines_total, **labels), _metric(data_processed_bytes_total, **labels)
    svc.start()
    sent = 0
    try:
        with pynng.Pair0(dial=addr, recv_timeout=2000) as c:
            time.sleep(0.2)
            for i, url in enumerate(g["urls"]):
                rec = {"EventID": 0, "logID": f"id{i}", "logFormatVariables": {"URL": url}}
                blob = wire.encode_parser_schema(rec)
                sent += len(blob)
                c.send(blob)
                if i < 2:
                    c.recv_timeout = 500
                    with pytest.raises(pynng.Timeout):
                        c.recv()                          # training => no reply (engine.py:196-198)
                else:
                    c.recv_timeout = 5000
                    alert = wire.decode_detector_schema(c.recv())
                    assert alert["alertsObtain"] == g["expected"]["alertsObtain"] and alert["alertID"] == "10"
    finally:
        svc.stop()
    assert svc.library_component.det.stats()["lines"] == len(g["urls"])         # the records went through the GPU
    # (the reference counts b"\n" bytes per message, core.py:190: a ParserSchema holds some -- tag 0x0a)
    assert _metric(data_processed_lines_total, **labels) - lines0 >= len(g["urls"])
    assert _metric(data_processed_bytes_total, **labels) - bytes0 == sent
    svc.library_component.close()


@needs_ref
def test_service_subclass_route_on_raw_batches(tmp_path, sock_dir, monkeypatch):
    """b200_detector_service(): a Service subclass whose process() keeps the base class's metrics; fed with raw
    key=value batches (one message = many records), checked against the oracle."""
    monkeypatch.syspath_prepend(_reference_src())
    install_shims()
    from service.core import data_processed_lines_total
    from service.settings import ServiceSettings
    from detectmateservice_b200.component import decode_compact
    from detectmateservice_b200.service import b200_detector_service
    from detectmateservice_b200.synth import AuditSynth, MONITORED_KEYS

    g = AuditSynth(seed=123)
    train, _ = g.batch(4096, inject=False)
    msgs = [g.batch(4096, inject=True)[0] for _ in range(3)]
    keys = [k.encode() for k in MONITORED_KEYS]
    orc = NativeOracle(keys)
    orc.process(train, 4096)
    cfg = {"detectors": {"B200NewValueDetector": {
        "method_type": "new_value_detector", "data_use_training": 4096, "auto_config": False,
        "params": {"output_format": "compact", "max_batch_bytes": 4 << 20},
        "global": {"g": {"header_variables": [{"pos": k} for k in MONITORED_KEYS]}}}}}
    Svc = b200_detector_service()
    settings = ServiceSettings(component_name="b200-subclass", engine_addr=f"ipc://{sock_dir}/sub.ipc",
                               log_dir=tmp_path / "logs", log_to_file=False, log_to_console=False,
                               http_port=18232, engine_autostart=False)
    svc = Svc(settings=settings, component_config=cfg)
    labels = dict(component_type=svc.component_type, component_id=svc.component_id)
    lines0 = _metric(data_processed_lines_total, **labels)
    try:
        f, s = decode_compact(svc.process(train))
        assert not f.any()
        for m in msgs:
            wf, ws, _ = orc.process(m, 0)
            f, s = decode_compact(svc.process(m))
            assert (f == wf).all() and (s == ws).all()
    finally:
        svc.detector.close()
        try:
            svc.stop()
        except Exception:
            pass
    assert _metric(data_processed_lines_total, **labels) - lines0 == 4 * 4096
