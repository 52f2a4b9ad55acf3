"""Runs in a subprocess of tests/test_integration_stub.py: the ctypes stub and the call-site replacements printed in
INTEGRATION.md -- taken VERBATIM from the markdown -- patched into the package's MP3Parser / MP3Encoder, which carry the
reference's class and private attribute names, so the replacements apply to them unchanged.  The facade is then driven through
the stub the way the reference's own test cases drive it (tests/steganography_test.py:15-60), and the artefacts are hashed for a
byte comparison with those the pure-Python reference produced (tests/golden/ref_facade.json).  Needs a B200; prints one JSON
object."""
import hashlib
import json
import os
import re
import shutil
import sys
import tempfile
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "mp3-steganography-lib_b200")


def main():
    sys.path.insert(0, PKG)
    md = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    blocks = re.findall(r"```python\n(.*?)```", md, flags=re.S)
    stub_src = next(b for b in blocks if "mp3stego/_b200.py" in b.splitlines()[0] and "continued" not in b.splitlines()[0])
    batch_src = next(b for b in blocks if "mp3stego/_b200.py (continued)" in b.splitlines()[0])
    sites_src = next(b for b in blocks if "mp3stego/decoder/MP3_Parser.py" in b.splitlines()[0])
    import numpy as np
    import mp3stego_b200
    import mp3stego_b200.decoder as mp
    import mp3stego_b200.encoder as me
    stub = types.ModuleType("mp3stego._b200")          # "new file in the reference tree"
    exec(compile(stub_src, "INTEGRATION.md:_b200", "exec"), stub.__dict__)
    from scipy.io.wavfile import write
    ns = {"_b200": stub, "np": np, "write": write}
    exec(compile(sites_src, "INTEGRATION.md:call_sites", "exec"), ns)
    calls = {"parse_file": 0, "encode": 0}

    def counted(name, fn):
        def w(self, *a, **k):
            calls[name] += 1
            return fn(self, *a, **k)
        return w

    mp.MP3Parser.parse_file = counted("parse_file", ns["parse_file"])
    mp.MP3Parser.write_to_wav = ns["write_to_wav"]
    mp.MP3Parser.get_bitrate = ns["get_bitrate"]
    me.MP3Encoder.encode = counted("encode", ns["encode"])

    work = tempfile.mkdtemp(prefix="m3s_stub_")
    shutil.copy(os.path.join(ROOT, "tests", "golden", "test.mp3"), os.path.join(work, "test.mp3"))
    os.chdir(work)
    s = mp3stego_b200.Steganography(quiet=True)
    sha = lambda p: hashlib.sha256(open(p, "rb").read()).hexdigest()   # noqa: E731
    out = {"calls": calls}
    out["decode_returns"] = s.decode_mp3_to_wav("test.mp3", "o.wav")
    out["out_wav_sha256"] = sha("o.wav")
    s.encode_wav_to_mp3("o.wav", "e320.mp3", 320)
    out["enc320_sha256"] = sha("e320.mp3")
    s.encode_wav_to_mp3("o.wav", "e128.mp3", 128)
    out["enc128_sha256"] = sha("e128.mp3")
    out["hide_ddd_returns"] = s.hide_message("test.mp3", "hid.mp3", "ddd")
    out["hid_sha256"] = sha("hid.mp3")
    out["hide_long_returns"] = s.hide_message("test.mp3", "long.mp3", "ddd" * 100)
    out["hid_long_sha256"] = sha("long.mp3")
    s.clear_file("hid.mp3", "cleared.mp3")
    out["cleared_sha256"] = sha("cleared.mp3")
    for name, mp3 in (("reveal_hid", "hid.mp3"), ("reveal_cleared", "cleared.mp3"), ("reveal_test_mp3", "test.mp3")):
        s.reveal_massage(mp3, "r.txt")
        out[name] = open("r.txt").read()
    # the batch binding of INTEGRATION.md (m3s_decode: one pipelined call for N files) against the single-file stub
    exec(compile(batch_src, "INTEGRATION.md:_b200_batch", "exec"), stub.__dict__)
    blobs = [open(p, "rb").read() for p in ("test.mp3", "hid.mp3", "cleared.mp3")]
    many = stub.parse_files(blobs, [0, 0, 0])
    same = True
    for b, m in zip(blobs, many):
        one = stub.parse_file(b, 0)
        same = same and one[0] == m[0] and np.array_equal(one[1], m[1]) and one[2:] == m[2:]
    out["batch_binding_equals_single"] = bool(same)
    os.chdir(ROOT)
    shutil.rmtree(work, ignore_errors=True)
    print("RESULT " + json.dumps(out))


if __name__ == "__main__":
    main()
