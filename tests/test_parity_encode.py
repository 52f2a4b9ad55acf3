"""GPU: encode (+hide) parity of the CUDA path (through the C ABI) against the oracle and the reference-generated
golden vectors.  Gates: MDCT spectra, quantised values, side-info fields, table choices, hide_str_offset and the
MP3 byte stream are all bit-exact."""
import hashlib
import json
import os

import numpy as np
import pytest

from conftest import SYNTH_CASES, golden_path, load_npz, synth_wav

pytestmark = pytest.mark.gpu


def _wav_pcm(path):
    raw = open(path, "rb").read()
    i = raw.find(b"data")
    return np.frombuffer(raw[i + 8:], dtype=np.int16).reshape(-1, 2)


def _encode(handle, clips, bitrate, payloads=None, taps=True, sr=44100):
    pcm = np.concatenate([c.reshape(-1) for c in clips]).astype(np.int16)
    ns = [c.shape[0] for c in clips]
    res = handle.encode(pcm, ns, sr, bitrate, payloads=payloads, taps=taps)
    outs = []
    fb = np.concatenate([[0], np.cumsum([n // 1152 for n in ns])])
    for i in range(len(clips)):
        o = int(res["mp3_off"][i])
        d = dict(mp3=bytes(res["mp3"][o:o + int(res["out_len"][i])]), hide_str_offset=int(res["hide_str_offset"][i]))
        if taps:
            for k in ("mdct", "ix", "info", "scfsi"):
                d[k] = res[k][fb[i]:fb[i + 1]]
        outs.append(d)
    return outs


def _check_taps(got, ref, n_mdct=None):
    m = ref["mdct"] if n_mdct is None else ref["mdct"][:n_mdct]
    assert np.array_equal(got["mdct"][:len(m)], m), "MDCT spectra differ"
    assert np.array_equal(got["scfsi"], ref["scfsi"]), "scfsi differs"
    bad = np.argwhere(got["info"][..., :16] != ref["info"][..., :16])
    assert bad.size == 0, f"side info differs at (frame, gr, ch, field) {bad[:6].tolist()}"
    assert np.array_equal(got["ix"], ref["ix"]), "quantised values differ"


def _clicks(seed, n, amp):
    rng = np.random.default_rng(seed)
    y = np.zeros((n, 2), np.int16)
    idx = rng.integers(0, n, size=n // 200)
    y[idx, 0] = amp
    y[idx[::2], 1] = -amp
    return y


@pytest.mark.parametrize("case", SYNTH_CASES)
def test_synth_vs_reference_golden(handle, case):
    """Bytes, hide_str_offset and every tap equal what the unmodified reference produced."""
    z = load_npz(f"ref_synth_{case}.npz")
    bits = str(z["hide_bits"])
    got = _encode(handle, [z["pcm_in"]], int(z["bitrate"]), payloads=[bits] if bits else None)[0]
    ref = dict(mdct=z["mdct"], ix=z["ix"].astype(np.int32), info=z["info"], scfsi=z["scfsi"].astype(np.int32))
    _check_taps(got, ref, n_mdct=3)
    assert got["hide_str_offset"] == int(z["hide_str_offset"])
    assert got["mp3"] == z["mp3"].tobytes(), "MP3 bytes differ"


def test_facade_goldens(handle):
    """SURVEY 8(c): the reference's own WAV -> 320k / 128k / hide('ddd') / hide('ddd'*100) artefacts, by sha256."""
    fac = json.load(open(golden_path("ref_facade.json")))
    wav = _wav_pcm(golden_path("ref_test_out.wav"))
    sha = lambda b: hashlib.sha256(b).hexdigest()  # noqa: E731
    from oracle import oracle as O
    assert sha(_encode(handle, [wav], 320, taps=False)[0]["mp3"]) == fac["enc320_sha256"]
    assert sha(_encode(handle, [wav], 128, taps=False)[0]["mp3"]) == fac["enc128_sha256"]
    bits = O.str_to_bits("3#ddd")
    g = _encode(handle, [wav], 320, payloads=[bits], taps=False)[0]
    assert sha(g["mp3"]) == fac["hid_sha256"]
    assert (g["hide_str_offset"] < len(bits) - 1) == fac["hide_ddd_returns"]
    long_bits = O.str_to_bits("300#" + "ddd" * 100)
    g = _encode(handle, [wav], 320, payloads=[long_bits], taps=False)[0]
    assert sha(g["mp3"]) == fac["hid_long_sha256"]
    assert (g["hide_str_offset"] < len(long_bits) - 1) == fac["hide_long_returns"]


@pytest.mark.parametrize("bitrate", [32, 64, 128, 192, 320])
def test_batch_vs_oracle(handle, oracle, bitrate):
    """A batch of clips of different lengths, half of them hiding, vs the oracle clip by clip."""
    rng = np.random.default_rng(bitrate)
    clips = [synth_wav(300 + bitrate + k, n) for k, n in enumerate([3, 17, 40, 9, 1])]
    payloads = ["".join(rng.choice(["0", "1"], size=n)) for n in (0, 2000, 37, 0, 8)]
    got = _encode(handle, clips, bitrate, payloads=payloads)
    for c, p, g in zip(clips, payloads, got):
        ref = oracle.encode(c, 44100, bitrate, p)
        _check_taps(g, ref)
        assert g["hide_str_offset"] == ref["hide_str_offset"]
        assert g["mp3"] == ref["mp3"]


@pytest.mark.parametrize("sr", [48000, 32000])
def test_other_sample_rates(handle, oracle, sr):
    clips = [synth_wav(77, 12, sr=sr)]
    bits = "10" * 300
    g = _encode(handle, clips, 128, payloads=[bits], sr=sr)[0]
    ref = oracle.encode(clips[0], sr, 128, bits)
    _check_taps(g, ref)
    assert g["mp3"] == ref["mp3"] and g["hide_str_offset"] == ref["hide_str_offset"]


def test_quiet_silent_and_loud(handle, oracle):
    """Digital silence (rate loop skipped, stale ix / step / addresses), fades (big_values == 0 probes, A.E6),
    full-scale noise and a square wave (large quantised values -> linbits tables and the double-precision path)."""
    rng = np.random.default_rng(5)
    n = 12 * 1152
    t = np.arange(n) / 44100.0
    silence = np.zeros((n, 2), np.int16)
    fade = (np.linspace(0, 1, n)[:, None] ** 6 * 300 * np.sin(2 * np.pi * 700 * t)[:, None] * np.ones((1, 2))).astype(np.int16)
    gaps = synth_wav(8, 12).copy()
    gaps[1152 * 3:1152 * 6] = 0
    gaps[1152 * 8:1152 * 9, 1] = 0
    loud = rng.integers(-32768, 32767, size=(n, 2)).astype(np.int16)
    square = (np.sign(np.sin(2 * np.pi * 90 * t)) * 32000).astype(np.int16)[:, None] * np.ones((1, 2), np.int16)
    tiny = rng.integers(-2, 3, size=(n, 2)).astype(np.int16)
    # very quiet material: the FIRST probes of a granule already find big_values == 0 among non-zero values, so the table
    # search runs over the slot's stale address1..3 of an earlier frame (A.E6) -- the granules the parallel rate loop hands
    # to its sequential resolve kernel
    hush = np.random.default_rng(6).integers(-6, 7, size=(n, 2)).astype(np.int16)
    clicks = _clicks(48, n, 48)
    clicks1 = _clicks(1, n, 1)
    clips = [silence, fade, gaps, loud, square, tiny, hush, clicks, clicks1]
    bits = "1100101" * 400
    for br in (128, 320):
        got = _encode(handle, clips, br, payloads=[bits] * len(clips))
        for c, g in zip(clips, got):
            ref = oracle.encode(c, 44100, br, bits)
            _check_taps(g, ref)
            assert g["hide_str_offset"] == ref["hide_str_offset"]
            assert g["mp3"] == ref["mp3"]


def test_chunked_equals_single(built, oracle):
    """Long batches advance through frame windows with the rate-loop state carried between them; the bytes must not
    depend on the window size."""
    from mp3stego_b200 import _lib
    os.environ["M3S_ENC_CHUNK_FRAMES"] = "40"
    try:
        h = _lib.Handle(0)
    finally:
        del os.environ["M3S_ENC_CHUNK_FRAMES"]
    gaps = synth_wav(9, 30).copy()
    gaps[1152 * 7:1152 * 13] = 0
    clips = [synth_wav(1, 30), gaps, synth_wav(3, 11), _clicks(64, 30 * 1152, 64), _clicks(7, 17 * 1152, 3)]
    bits = ["01" * 500, "1" * 77, "", "110" * 300, "10" * 20]
    got = _encode(h, clips, 128, payloads=bits, taps=False)
    for c, p, g in zip(clips, bits, got):
        ref = oracle.encode(c, 44100, 128, p, taps=False)
        assert g["mp3"] == ref["mp3"] and g["hide_str_offset"] == ref["hide_str_offset"]
    h.close()


def test_mixed_payload_batch_vs_oracle(handle, oracle):
    """A tone hiding a long payload, quiet clicks hiding another and a short plain clip in one batch: the oracle's bytes, taps
    and offsets."""
    clips = [synth_wav(21, 14), _clicks(5, 9 * 1152, 9), synth_wav(22, 5)]
    bits = ["011" * 200, "10" * 300, ""]
    for c, p, g in zip(clips, bits, _encode(handle, clips, 128, payloads=bits)):
        ref = oracle.encode(c, 44100, 128, p)
        _check_taps(g, ref)
        assert g["mp3"] == ref["mp3"] and g["hide_str_offset"] == ref["hide_str_offset"]


def _analysis_edge_clips():
    """Clips long enough to span several slot blocks and runs of the analysis kernel, with silence, a few-LSB stretch and clicks
    so that the folded kernel's correction pass runs (MP3_Encoder.py:322-370, :652-758); and their payloads."""
    quiet = synth_wav(31, 40).copy()
    quiet[1152 * 5:1152 * 9] = 0
    quiet[1152 * 9:1152 * 12] = (quiet[1152 * 9:1152 * 12] >> 13).astype(np.int16)   # a few LSBs: windowed values with many zero low bits
    clips = [synth_wav(30, 150), quiet, _clicks(11, 33 * 1152, 5), np.zeros((7 * 1152, 2), np.int16)]
    return clips, ["0110" * 900, "1" * 300, "10" * 200, ""]


def test_analysis_correction_pass(handle, oracle):
    """The analysis kernel computes equal truncated products once and corrects the sums where an input has many zero low bits:
    on the edge clips it gives the oracle's MDCT lines, taps, bytes and offsets."""
    clips, bits = _analysis_edge_clips()
    for c, p, g in zip(clips, bits, _encode(handle, clips, 128, payloads=bits)):
        ref = oracle.encode(c, 44100, 128, p)
        _check_taps(g, ref)
        assert g["mp3"] == ref["mp3"] and g["hide_str_offset"] == ref["hide_str_offset"]


def test_edge_clips_in_64_frame_chunks(built, oracle, monkeypatch):
    """The edge clips through the chunk pipeline (M3S_ENC_CHUNK_FRAMES=64: the analysis of chunk k + 1 queued behind the packing
    of chunk k, the rate-loop state carried across chunks): the oracle's bytes and offsets (the taps need a single-chunk batch)."""
    from mp3stego_b200 import _lib
    monkeypatch.setenv("M3S_ENC_CHUNK_FRAMES", "64")
    clips, bits = _analysis_edge_clips()
    h = _lib.Handle(0)
    got = _encode(h, clips, 128, payloads=bits, taps=False)
    h.close()
    for c, p, g in zip(clips, bits, got):
        ref = oracle.encode(c, 44100, 128, p, taps=False)
        assert g["mp3"] == ref["mp3"] and g["hide_str_offset"] == ref["hide_str_offset"]


def test_chunked_regular_batch_host_and_device(built, oracle):
    """Equal-length clips take the strided (2-D) PCIe staging path of the host pipeline; host and device buffers and the
    oracle must agree byte for byte across chunk boundaries."""
    import torch
    from mp3stego_b200 import _lib
    os.environ["M3S_ENC_CHUNK_FRAMES"] = "28"     # 4 clips x 7 frames per chunk -> 4 chunks, the last one ragged
    try:
        h = _lib.Handle(0)
    finally:
        del os.environ["M3S_ENC_CHUNK_FRAMES"]
    clips = [synth_wav(40 + k, 23) for k in range(4)]
    bits = ["0110" * 300, "", "1" * 50, "10" * 400]
    got = _encode(h, clips, 128, payloads=bits, taps=False)
    pcm = np.concatenate([c.reshape(-1) for c in clips]).astype(np.int16)
    res = h.encode(torch.from_numpy(pcm).cuda(), [c.shape[0] for c in clips], 44100, 128, payloads=bits)
    dev_mp3 = res["mp3"].cpu().numpy()
    for i, (c, p, g) in enumerate(zip(clips, bits, got)):
        ref = oracle.encode(c, 44100, 128, p, taps=False)
        assert g["mp3"] == ref["mp3"] and g["hide_str_offset"] == ref["hide_str_offset"]
        o = int(res["mp3_off"][i])
        assert bytes(dev_mp3[o:o + int(res["out_len"][i])]) == ref["mp3"]
    h.close()


def test_hide_reveal_roundtrip_at_scale(handle, oracle):
    """Size-independent property at BASELINE configs[2] scale (3-minute clips): what encode hides, decode reveals."""
    rng = np.random.default_rng(1)
    clips = [synth_wav(500 + k, 6890 // 10) for k in range(4)]   # 689 frames each (18 s); the full 3-min shape runs in bench.py
    msgs = ["".join(chr(c) for c in rng.integers(32, 127, size=1200)) for _ in clips]
    bits = [oracle.str_to_bits(f"{len(m)}#{m}") for m in msgs]
    got = _encode(handle, clips, 128, payloads=bits, taps=False)
    blobs = [g["mp3"] for g in got]
    data = np.frombuffer(b"".join(blobs), np.uint8)
    off = np.concatenate([[0], np.cumsum([len(b) for b in blobs])])
    handle.decode_scan(data, off)
    _, revealed = handle.decode_reveal()
    for g, b, m, r in zip(got, bits, msgs, revealed):
        used = g["hide_str_offset"]
        assert r[:min(used, len(b))] == b[:min(used, len(b))]
        if used >= len(b):
            assert oracle.reveal_parse(r) == m


def _random_clip(rng, sr):
    """Tone + noise under a random piecewise envelope: loud stretches, near-silent ones (a few LSB), digital silence and clicks in one
    clip, so that coded, silent and stale-address granules (A.E6) follow each other within a slot."""
    n_frames = int(rng.integers(1, 31))
    n = n_frames * 1152
    t = np.arange(n) / sr
    f = rng.uniform(60, 6000, 2)
    x = np.stack([np.sin(2 * np.pi * f[c] * t) + rng.uniform(0, 0.3) * rng.standard_normal(n) for c in range(2)], axis=1)
    env = np.zeros(n)
    pos = 0
    while pos < n:
        seg = int(rng.integers(200, 4000))
        kind = rng.integers(0, 5)
        env[pos:pos + seg] = (0.0, rng.uniform(1, 8) / 32767, rng.uniform(0.001, 0.02), rng.uniform(0.1, 0.6), 0.99)[kind]
        pos += seg
    y = (x * env[:, None] * 32767).astype(np.int16)
    for _ in range(int(rng.integers(0, 4))):
        y[int(rng.integers(0, n)), int(rng.integers(0, 2))] = int(rng.integers(-32768, 32768))
    return y


@pytest.mark.parametrize("seed", [11, 12, 13, 14])
def test_random_clips_vs_oracle(handle, oracle, seed):
    """Randomised batches: bitrate, sample rate, clip lengths, envelopes and payload lengths (none, ending inside the clip -- the
    two-, one- and zero-bit variants of the rate loop -- or longer than the capacity), vs the oracle clip by clip, taps included."""
    rng = np.random.default_rng(seed)
    sr = int(rng.choice([44100, 44100, 48000, 32000]))
    bitrate = int(rng.choice([32, 48, 64, 96, 128, 160, 224, 320]))
    clips = [_random_clip(rng, sr) for _ in range(10)]
    payloads = []
    for c in clips:
        cap = 12 * (c.shape[0] // 1152)
        k = rng.integers(0, 4)
        ln = (0, int(rng.integers(1, 12)), int(rng.integers(1, max(2, cap))), 3 * cap + 40)[k]
        payloads.append("".join(rng.choice(["0", "1"], size=ln)) if ln else "")
    got = _encode(handle, clips, bitrate, payloads=payloads, sr=sr)
    for i, (c, p, g) in enumerate(zip(clips, payloads, got)):
        ref = oracle.encode(c, sr, bitrate, p)
        _check_taps(g, ref)
        assert g["hide_str_offset"] == ref["hide_str_offset"], (seed, i)
        assert g["mp3"] == ref["mp3"], (seed, i)
