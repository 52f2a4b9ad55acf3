"""GPU: clips of different sample rates and bitrates in ONE encode call (m3s_encode_mixed), held to the oracle clip by clip.

- The whole edge corpus of tests/encgen.py (42 rate pairs, 1..300 frames, 320 one-frame clips) shuffled so that neighbouring
  clips differ in rate, in one single-chunk call: bytes, hide_str_offset, MDCT, quantised values, side info and scfsi in the
  caller's clip order.
- The same call through 64- and 37-frame chunks, from host and from device buffers.
- A single rate pair through the mixed entry point: the same bytes and kernel launches as m3s_encode.
- Overrunning clips (SURVEY A.E13) among good clips of other rates: IndexError naming the caller's clip index and frame.
- Unsupported rates: M3S_ERR_ARG naming the clip, nothing launched.
- hide_batch / clear_batch over files of all three sample rates and several bitrates: one encode call, the oracle chain's bytes.
- files.encode_files with per-file bitrates."""
import numpy as np
import pytest

import encgen
from conftest import synth_wav

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def clips():
    return encgen.extreme_clips(0)


@pytest.fixture(scope="module")
def shuffled(clips):
    corpus = clips[0]
    return [corpus[i] for i in np.random.default_rng(11).permutation(len(corpus))]


@pytest.fixture(scope="module")
def refs(oracle, clips):
    return {c["name"]: oracle.encode(c["pcm"], c["sr"], c["br"], c["bits"]) for c in clips[0]}


def _encode(h, group, taps=True, device=False, mixed=True):
    pcm = np.concatenate([c["pcm"].reshape(-1) for c in group]).astype(np.int16)
    ns = [c["pcm"].shape[0] for c in group]
    if device:
        import torch
        pcm = torch.from_numpy(pcm).cuda()
    sr = [c["sr"] for c in group] if mixed else group[0]["sr"]
    br = [c["br"] for c in group] if mixed else group[0]["br"]
    res = h.encode(pcm, ns, sr, br, payloads=[c["bits"] for c in group], taps=taps)
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


def _handle(monkeypatch, chunk=None):
    from mp3stego_b200 import _lib
    if chunk is not None:
        monkeypatch.setenv("M3S_ENC_CHUNK_FRAMES", str(chunk))
    return _lib.Handle(0)


def test_shuffled_corpus_in_one_call(built, monkeypatch, shuffled, refs):
    pairs = [(c["sr"], c["br"]) for c in shuffled]
    assert len(set(pairs)) == 42 and sum(c["pcm"].shape[0] for c in shuffled) // 1152 > 2800
    assert sum(a != b for a, b in zip(pairs, pairs[1:])) > 0.6 * len(pairs)
    h = _handle(monkeypatch, 1 << 22)   # one chunk: the taps need it
    try:
        for c, g in zip(shuffled, _encode(h, shuffled)):
            r, what = refs[c["name"]], c["name"]
            assert np.array_equal(g["mdct"], r["mdct"]), f"{what}: MDCT spectra differ"
            assert np.array_equal(g["scfsi"], r["scfsi"]), f"{what}: scfsi differs"
            bad = np.argwhere(g["info"][..., :16] != r["info"][..., :16])
            assert bad.size == 0, f"{what}: side info differs at (frame, gr, ch, field) {bad[:6].tolist()}"
            assert np.array_equal(g["ix"], r["ix"]), f"{what}: quantised values differ"
            assert g["hide_str_offset"] == r["hide_str_offset"], what
            assert g["mp3"] == r["mp3"], f"{what}: MP3 bytes differ"
    finally:
        h.close()


@pytest.mark.parametrize("device", [False, True], ids=["host", "device"])
@pytest.mark.parametrize("per_clip", [False, True], ids=["budget", "per_clip"])
@pytest.mark.parametrize("chunk", [64, 37])
def test_shuffled_corpus_in_chunks(built, monkeypatch, shuffled, refs, chunk, per_clip, device):
    # M3S_ENC_CHUNK_FRAMES = 64 / 37 frames in all (one frame per clip and chunk), or 64 / 37 frames per clip: clips of 1..300
    # frames run out in different chunks, and so do whole sample-rate groups
    h = _handle(monkeypatch, chunk * len(shuffled) if per_clip else chunk)
    try:
        for c, g in zip(shuffled, _encode(h, shuffled, taps=False, device=device)):
            r = refs[c["name"]]
            assert g["mp3"] == r["mp3"] and g["hide_str_offset"] == r["hide_str_offset"], (c["name"], chunk, device)
    finally:
        h.close()


def test_single_pair_through_the_mixed_entry(handle, clips, refs):
    group = encgen.by_rate(clips[0])[(48000, 192)]
    l0 = handle.launches
    single = _encode(handle, group, mixed=False)
    l1 = handle.launches
    mixed = _encode(handle, group, mixed=True)
    l2 = handle.launches
    assert l2 - l1 == l1 - l0
    for c, a, b in zip(group, single, mixed):
        assert a["mp3"] == b["mp3"] == refs[c["name"]]["mp3"], c["name"]
        assert a["hide_str_offset"] == b["hide_str_offset"] == refs[c["name"]]["hide_str_offset"], c["name"]
        assert np.array_equal(a["info"], b["info"]) and np.array_equal(a["ix"], b["ix"]), c["name"]


def test_overrun_among_other_rates(built, oracle, clips, refs):
    from mp3stego_b200 import _lib
    corpus, overrun = clips
    h = _lib.Handle(0)
    try:
        for n, c in enumerate(overrun):
            r = oracle.encode(c["pcm"], c["sr"], c["br"], c["bits"], taps=False)
            assert r["status"] == -3
            good = [g for g in corpus if (g["sr"], g["br"]) != (c["sr"], c["br"])][7 * n::53][:8]
            assert len({g["sr"] for g in good}) >= 2
            k = 3 + n % 4
            with pytest.raises(IndexError, match=f"clip {k} frame {r['n_frames']}: .*{_lib.STEP_TABLE_OVERRUN}"):
                _encode(h, good[:k] + [c] + good[k:], taps=False)
            for g, out in zip(good, _encode(h, good)):
                rg = refs[g["name"]]
                assert out["mp3"] == rg["mp3"] and out["hide_str_offset"] == rg["hide_str_offset"], g["name"]
                assert np.array_equal(out["info"][..., :16], rg["info"][..., :16]), g["name"]
    finally:
        h.close()


@pytest.mark.parametrize("bad", [(22050, 128), (44100, 330)], ids=["sr22050", "br330"])
def test_unsupported_rate_names_the_clip(handle, clips, bad):
    from mp3stego_b200 import _lib
    group = [c for c in clips[0] if c["pcm"].shape[0] == 1152][:5]
    k = 3
    sr = [c["sr"] for c in group]
    br = [c["br"] for c in group]
    sr[k], br[k] = bad
    pcm = np.concatenate([c["pcm"].reshape(-1) for c in group]).astype(np.int16)
    l0 = handle.launches
    with pytest.raises(_lib.M3SError, match=f"m3s_encode_mixed failed \\(-2\\): encode: clip {k}: "):
        handle.encode(pcm, [1152] * len(group), sr, br)
    assert handle.launches == l0
    assert ("sample rate 22050" if bad[0] == 22050 else "bitrate 330") in handle._L.m3s_last_error(handle._h).decode()


def _composite_corpus(oracle):
    specs = [(44100, 128, 9), (48000, 320, 14), (32000, 64, 5), (44100, 256, 21), (48000, 96, 7), (32000, 192, 11),
             (44100, 32, 4), (48000, 128, 12), (32000, 320, 6)]
    blobs = [oracle.encode(synth_wav(70 + i, n, sr=sr), sr, br, "", taps=False)["mp3"] for i, (sr, br, n) in enumerate(specs)]
    tag = b"ID3\x04\x00\x00" + bytes([0, 0, 0, 40]) + bytes(40)
    blobs[4] = tag + blobs[4]
    return blobs


def _oracle_chain(oracle, blob, bits):
    dec = oracle.decode(blob, oracle.id3_offset(blob), taps=False)
    pcm = np.asarray(dec["pcm16"], np.int16).reshape(-1, 2)
    return oracle.encode(pcm, dec["sampling_rate"], dec["bit_rate"] // 1000, bits, taps=False)


def test_hide_and_clear_batches_make_one_encode_call(handle, oracle, monkeypatch):
    from mp3stego_b200 import _lib, batch
    from mp3stego_b200.steganography import str_to_binary_str
    blobs = _composite_corpus(oracle)
    calls = []
    orig = _lib.Handle.encode

    def counted(self, *a, **k):
        calls.append(a[2] if len(a) > 2 else k.get("sample_rate"))
        return orig(self, *a, **k)

    monkeypatch.setattr(_lib.Handle, "encode", counted)
    msgs = ["mixed %d" % i if i % 3 else "y" * 250 for i in range(len(blobs))]
    hid, too_long = batch.hide_batch(handle, blobs, msgs)
    assert len(calls) == 1 and sorted(set(np.asarray(calls[0]).tolist())) == [32000, 44100, 48000]
    cleared = batch.clear_batch(handle, blobs)
    assert len(calls) == 2
    for i, (b, m) in enumerate(zip(blobs, msgs)):
        bits = str_to_binary_str(str(len(m)) + "#" + m)
        ref = _oracle_chain(oracle, b, bits)
        assert hid[i] == ref["mp3"], i
        assert too_long[i] == (ref["hide_str_offset"] < len(bits) - 1), i
        assert cleared[i] == _oracle_chain(oracle, b, "")["mp3"], i
    assert any(too_long) and not all(too_long)


def test_encode_files_with_per_file_bitrates(handle, oracle, tmp_path):
    from mp3stego_b200 import files
    from mp3stego_b200.steganography import str_to_binary_str
    from mp3stego_b200.wavio import write_wav
    specs = [(44100, 320, 5), (48000, 64, 9), (32000, 128, 3), (48000, 320, 4), (32000, 40, 8), (44100, 96, 6)]
    wavs, outs, pcms = [], [], []
    for i, (sr, br, n) in enumerate(specs):
        pcm = synth_wav(90 + i, n, sr=sr)
        p = str(tmp_path / f"in{i}.wav")
        write_wav(p, sr, pcm)
        wavs.append(p)
        outs.append(str(tmp_path / f"out{i}.mp3"))
        pcms.append(pcm)
    msgs = ["", "z" * 200, "abc", "hello there", "", "q" * 40]
    too_long = files.encode_files(handle, wavs, outs, bitrate=[br for _, br, _ in specs], messages=msgs)
    for i, ((sr, br, _), m) in enumerate(zip(specs, msgs)):
        bits = str_to_binary_str(str(len(m)) + "#" + m) if m else ""
        ref = oracle.encode(pcms[i], sr, br, bits, taps=False)
        assert open(outs[i], "rb").read() == ref["mp3"], i
        assert too_long[i] == (ref["hide_str_offset"] < len(bits) - 1), i
    assert any(too_long) and not all(too_long)
