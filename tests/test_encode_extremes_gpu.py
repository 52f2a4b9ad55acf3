"""GPU: the encode edge corpus (tests/encgen.py) through the CUDA encoder, held to the oracle clip by clip.

- One batch per (sample rate, bitrate): bytes, hide_str_offset, MDCT spectra, quantised values, side info and scfsi equal.
- The same batches through the chunk pipeline (M3S_ENC_CHUNK_FRAMES 64 and 37), from host and from device buffers: bytes and
  hide_str_offset equal.
- The GPU's MP3s decoded with the exact (float64) decode: reveal bits equal to the oracle's decode of the same bytes, int16 PCM
  equal by the float64 rule of tests/test_decode_extremes_gpu.py.
- Clips whose step search runs past the end of the step table (SURVEY A.E13), alone and inside batches of good clips: the call
  fails with M3S_ERR_ARG naming the clip and frame, the Python layers raise IndexError, and the same handle then encodes a
  good batch correctly."""
import numpy as np
import pytest

import encgen
from test_decode_extremes_gpu import _check_exact_loud

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def clips():
    return encgen.extreme_clips(0)


@pytest.fixture(scope="module")
def refs(oracle, clips):
    return {c["name"]: oracle.encode(c["pcm"], c["sr"], c["br"], c["bits"]) for c in clips[0]}


def _encode(h, group, taps=True, device=False):
    pcm = np.concatenate([c["pcm"].reshape(-1) for c in group]).astype(np.int16)
    ns = [c["pcm"].shape[0] for c in group]
    if device:
        import torch
        pcm = torch.from_numpy(pcm).cuda()
    res = h.encode(pcm, ns, group[0]["sr"], group[0]["br"], payloads=[c["bits"] for c in group], taps=taps)
    mp3 = res["mp3"].cpu().numpy() if device else res["mp3"]
    fb = np.concatenate([[0], np.cumsum([n // 1152 for n in ns])])
    outs = []
    for i in range(len(group)):
        o = int(res["mp3_off"][i])
        d = dict(mp3=bytes(mp3[o:o + int(res["out_len"][i])]), hide_str_offset=int(res["hide_str_offset"][i]))
        if taps:
            for k in ("mdct", "ix", "info", "scfsi"):
                d[k] = res[k][fb[i]:fb[i + 1]]
        outs.append(d)
    return outs


@pytest.fixture(scope="module")
def gpu_encoded(handle, clips):
    out = {}
    for _, group in encgen.by_rate(clips[0]).items():
        for c, g in zip(group, _encode(handle, group)):
            out[c["name"]] = g
    return out


def test_corpus_vs_oracle(clips, refs, gpu_encoded):
    for c in clips[0]:
        g, r = gpu_encoded[c["name"]], refs[c["name"]]
        what = c["name"]
        assert np.array_equal(g["mdct"], r["mdct"]), f"{what}: MDCT spectra differ"
        assert np.array_equal(g["scfsi"], r["scfsi"]), f"{what}: scfsi differs"
        bad = np.argwhere(g["info"][..., :16] != r["info"][..., :16])
        assert bad.size == 0, f"{what}: side info differs at (frame, gr, ch, field) {bad[:6].tolist()}"
        assert np.array_equal(g["ix"], r["ix"]), f"{what}: quantised values differ"
        assert g["hide_str_offset"] == r["hide_str_offset"], what
        assert g["mp3"] == r["mp3"], f"{what}: MP3 bytes differ"


@pytest.mark.parametrize("device", [False, True], ids=["host", "device"])
@pytest.mark.parametrize("chunk", [64, 37])
def test_corpus_in_chunks(built, clips, refs, monkeypatch, chunk, device):
    from mp3stego_b200 import _lib
    monkeypatch.setenv("M3S_ENC_CHUNK_FRAMES", str(chunk))
    h = _lib.Handle(0)
    try:
        for (sr, br), group in encgen.by_rate(clips[0]).items():
            for c, g in zip(group, _encode(h, group, taps=False, device=device)):
                r = refs[c["name"]]
                assert g["mp3"] == r["mp3"] and g["hide_str_offset"] == r["hide_str_offset"], (c["name"], chunk, device)
    finally:
        h.close()


def test_decode_of_gpu_encodes(handle, oracle, clips, gpu_encoded):
    names = [c["name"] for c in clips[0]]
    blobs = [gpu_encoded[n]["mp3"] for n in names]
    data = np.frombuffer(b"".join(blobs), np.uint8)
    off = np.concatenate([[0], np.cumsum([len(b) for b in blobs])]).astype(np.int64)
    res = handle.decode(data, off, exact=True)
    bits = handle.reveal_strings(res)
    for i, (n, b) in enumerate(zip(names, blobs)):
        ref = oracle.decode(b)
        assert int(res["n_frames"][i]) == ref["n_frames"], n
        assert bits[i] == ref["bits"], f"{n}: reveal bits differ"
        pcm = res["pcm"][int(res["pcm_off"][i]):int(res["pcm_off"][i + 1])].reshape(-1, 2)
        _check_exact_loud(dict(pcm=pcm), ref, f"{n}: exact decode")


def _overrun_frame(oracle, c):
    r = oracle.encode(c["pcm"], c["sr"], c["br"], c["bits"], taps=False)
    assert r["status"] == -3
    return r["n_frames"]


def test_overrun_clips_fail_the_call(built, oracle, clips, refs):
    from mp3stego_b200 import _lib
    corpus, overrun = clips
    h = _lib.Handle(0)
    try:
        for c in overrun:
            f = _overrun_frame(oracle, c)
            # alone
            with pytest.raises(IndexError, match=f"clip 0 frame {f}: .*{_lib.STEP_TABLE_OVERRUN}"):
                _encode(h, [c], taps=False)
            assert h._L.m3s_last_error(h._h).decode().startswith(f"encode: clip 0 frame {f}:")
            # inside a batch of good clips of the same rates: the whole batch fails, naming the clip
            good = [g for g in corpus if g["sr"] == c["sr"] and g["br"] == c["br"]][:6]
            k = len(good) // 2
            with pytest.raises(IndexError, match=f"clip {k} frame {f}: "):
                _encode(h, good[:k] + [c] + good[k:], taps=False)
            # the same handle then encodes the good clips exactly
            for g, out in zip(good, _encode(h, good)):
                r = refs[g["name"]]
                assert out["mp3"] == r["mp3"] and out["hide_str_offset"] == r["hide_str_offset"], g["name"]
                assert np.array_equal(out["info"][..., :16], r["info"][..., :16]), g["name"]
    finally:
        h.close()


def test_overrun_through_the_file_and_class_api(handle, oracle, clips, tmp_path):
    from mp3stego_b200 import encoder, files
    from mp3stego_b200.wavio import WavReader, write_wav
    corpus, overrun = clips
    c = overrun[0]
    good = next(g for g in corpus if g["sr"] == c["sr"] and g["br"] == c["br"] and g["pcm"].shape[0] == 1152)
    paths = []
    for i, x in enumerate((good, c)):
        p = str(tmp_path / f"in{i}.wav")
        write_wav(p, x["sr"], x["pcm"])
        paths.append(p)
    outs = [str(tmp_path / f"out{i}.mp3") for i in range(2)]
    with pytest.raises(IndexError, match=f"clip 1 frame {_overrun_frame(oracle, c)}: "):
        files.encode_files(handle, paths, outs, bitrate=c["br"])
    with pytest.raises(IndexError, match="past the end of the step table"):
        encoder.MP3Encoder(WavReader(paths[1], c["br"])).encode()
    # and a good file after it
    assert files.encode_files(handle, paths[:1], outs[:1], bitrate=c["br"]) == [False]
    assert open(outs[0], "rb").read() == oracle.encode(good["pcm"], good["sr"], good["br"], "", taps=False)["mp3"]
