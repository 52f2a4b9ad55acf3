"""GPU: the ctypes stub of INTEGRATION.md, verbatim, patched into the reference's MP3Parser / MP3Encoder surface (the package's
mirror of those classes): every codec call of the facade goes through the stub, and the artefacts equal the pure-Python
reference's by sha256."""
import json
import os
import subprocess
import sys

import pytest

from conftest import PKG, ROOT, golden_path

pytestmark = pytest.mark.gpu


def test_reference_classes_over_the_stub(built):
    env = dict(os.environ)
    env["LD_LIBRARY_PATH"] = os.path.join(PKG, "lib") + os.pathsep + env.get("LD_LIBRARY_PATH", "")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "integration_stub_runner.py")], env=env, capture_output=True,
                       text=True, timeout=900)
    assert p.returncode == 0, p.stderr[-3000:]
    line = [ln for ln in p.stdout.splitlines() if ln.startswith("RESULT ")][-1]
    out = json.loads(line[7:])
    fac = json.load(open(golden_path("ref_facade.json")))
    assert out["calls"] == {"parse_file": 7, "encode": 5}      # every decode / encode of the facade went through the stub
    for k in ("decode_returns", "out_wav_sha256", "enc320_sha256", "enc128_sha256", "hide_ddd_returns", "hid_sha256",
              "hide_long_returns", "hid_long_sha256", "cleared_sha256", "reveal_hid", "reveal_cleared", "reveal_test_mp3"):
        assert out[k] == fac[k], k
    assert out["batch_binding_equals_single"]      # INTEGRATION.md's m3s_decode binding: N files in one call == N single-file calls
