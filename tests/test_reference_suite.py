"""The reference's OWN test-suite (everything but tests/library_integration, which needs the
un-vendored detectmatelibrary components) run against this repo's stand-ins for the two
packages that cannot be installed offline: `pynng` (SP/PAIR0 transport) and the two
`detectmatelibrary` base modules.  The suite and the service it tests are the copies build()
puts under oracle/_ref (oracle/Makefile); without them this test skips.

Bar: 0 failures, 0 collection errors.
"""
import os
import shutil
import subprocess
import sys

import pytest

from detectmateservice_b200.compat import ipc_tempdir
from oracle.ref_engine import REF_DIR as REF

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.skipif(not os.path.isdir(os.path.join(REF, "tests")), reason="the reference test-suite is not in oracle/_ref")
def test_reference_suite_passes_on_the_shims(tmp_path):
    shims = os.path.join(ROOT, "detectmateservice_b200", "shims")
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join([REF, shims, env.get("PYTHONPATH", "")])
    env.pop("DM_KERNEL", None)
    # the suite's tests listen on ipc:// sockets under their tmp_path: keep it short enough for an AF_UNIX address
    basetemp = ipc_tempdir()
    cmd = [sys.executable, "-m", "pytest", os.path.join(REF, "tests"), "-q", "-x", "-p", "no:cacheprovider",
           "--rootdir", str(tmp_path), "--basetemp", os.path.join(basetemp, "t"), "--timeout", "120"]
    try:
        res = subprocess.run(cmd, cwd=str(tmp_path), env=env, capture_output=True, text=True, timeout=1500)
    finally:
        shutil.rmtree(basetemp, ignore_errors=True)
    tail = "\n".join((res.stdout + res.stderr).splitlines()[-40:])
    assert res.returncode == 0, "reference suite on the shims:\n" + tail
    assert " passed" in res.stdout and "error" not in res.stdout.splitlines()[-1].lower(), tail
