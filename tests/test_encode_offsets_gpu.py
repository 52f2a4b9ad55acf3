"""GPU: m3s_encode_offsets -- hide_str_offset of many candidate payloads per clip against one analysis + probe pass -- held to the
encoder and the oracle, and the capacity composites built on it (batch.capacity_batch, batch.hide_batch_fit).

- The whole edge corpus of tests/encgen.py (42 rate pairs, stale-address and slow granules, 1..300 frames), every clip with all
  prefixes of a message that runs past its capacity (printable ASCII, or 2/3/4-byte UTF-8 characters) plus arbitrary-bit heads:
  in ONE offsets call every candidate's offset equals m3s_encode_mixed's hide_str_offset for that clip and payload.
- The same through 37- and 64-frame chunks, from host and from device PCM.
- n = 0, n*, n* + 1 and the longest prefix of every clip against the oracle.
- Overrunning clips among good clips: IndexError naming the clip, the candidate and the frame; the handle stays usable.
- Bad arguments fail with M3S_ERR_ARG naming the clip and candidate, and launch nothing.
- An offsets call launches neither the emit nor the pack kernel, and m3s_encode_taps fails after it.
- capacity_batch / hide_batch_fit on tests/golden/test.mp3, tone+noise files at three sample rates and the stereo writer /
  fuzz / edge streams: hide_batch of message[:n*] fits, of message[:n* + 1] does not, and hide_batch_fit gives hide_batch's bytes."""
import numpy as np
import pytest

import encgen
from conftest import golden_path, synth_wav

pytestmark = pytest.mark.gpu

MULTIBYTE = "aé€\U0001F600中ßx\U0001F3B5"   # 1-, 2-, 3- and 4-byte UTF-8 characters


def _ascii(rng, n):
    return "".join(chr(c) for c in rng.integers(32, 127, n))


def _bits(head, body, bl):
    return "".join(format(b, "08b") for b in head + body[:bl])


@pytest.fixture(scope="module")
def clips():
    return encgen.extreme_clips(0)


@pytest.fixture(scope="module")
def cases(clips):
    """Per clip of the corpus (shuffled so that neighbours differ in rate): its body and candidates."""
    from mp3stego_b200.batch import capacity_candidates
    corpus = clips[0]
    rng = np.random.default_rng(23)
    out = []
    for i in rng.permutation(len(corpus)):
        c = corpus[i]
        n_chars = 12 * (c["pcm"].shape[0] // 1152) // 8 + 6   # more bits than 3 per granule-channel: past any capacity
        m = "".join(rng.choice(list(MULTIBYTE), size=n_chars)) if i % 5 == 2 else _ascii(rng, n_chars)
        body, cands = capacity_candidates(m)
        cands += [(rng.integers(0, 256, int(rng.integers(1, 33)), dtype=np.uint8).tobytes(), 0) for _ in range(2)]
        out.append(dict(clip=c, msg=m, body=body, cands=cands))
    return out


def _offsets(h, cases, device=False):
    pcm = np.concatenate([k["clip"]["pcm"].reshape(-1) for k in cases]).astype(np.int16)
    if device:
        import torch
        pcm = torch.from_numpy(pcm).cuda()
    return h.encode_offsets(pcm, [k["clip"]["pcm"].shape[0] for k in cases], [k["clip"]["sr"] for k in cases],
                            [k["clip"]["br"] for k in cases], [k["body"] for k in cases], [k["cands"] for k in cases])


@pytest.fixture(scope="module")
def expected(built, cases):
    """m3s_encode_mixed's hide_str_offset of every (clip, candidate): one call over per-candidate copies of the clips (they share
    the clip's PCM through pcm_off)."""
    import torch
    from mp3stego_b200 import _lib
    pcm = np.concatenate([k["clip"]["pcm"].reshape(-1) for k in cases]).astype(np.int16)
    base = np.concatenate([[0], np.cumsum([k["clip"]["pcm"].size for k in cases])])
    po, ns, sr, br, pay, owner = [], [], [], [], [], []
    for i, k in enumerate(cases):
        for head, bl in k["cands"]:
            po.append(base[i]); ns.append(k["clip"]["pcm"].shape[0]); sr.append(k["clip"]["sr"]); br.append(k["clip"]["br"])
            pay.append(_bits(head, k["body"], bl)); owner.append(i)
    h = _lib.Handle(0)
    try:
        res = h.encode(torch.from_numpy(pcm).cuda(), ns, sr, br, payloads=pay, pcm_off=po)
    finally:
        h.close()
    hoff, owner = res["hide_str_offset"], np.asarray(owner)
    return [hoff[owner == i] for i in range(len(cases))]


def _handle(monkeypatch, chunk=None):
    from mp3stego_b200 import _lib
    if chunk is not None:
        monkeypatch.setenv("M3S_ENC_CHUNK_FRAMES", str(chunk))
    return _lib.Handle(0)


def _assert_equal(got, expected, cases, what):
    bad = [(k["clip"]["name"], j, int(g[j]), int(e[j])) for k, g, e in zip(cases, got, expected) for j in np.nonzero(g != e)[0][:3]]
    assert not bad, f"{what}: {len(bad)} clips differ, first (clip, candidate, got, encoder): {bad[:8]}"


def test_corpus_equals_the_encoder_in_one_call(built, monkeypatch, cases, expected):
    assert len({(k["clip"]["sr"], k["clip"]["br"]) for k in cases}) == 42
    assert sum(len(k["cands"]) for k in cases) > 5000
    # every clip's candidates run from "0#" past what the clip can carry, so the longest prefix cannot fit
    assert all(8 * (len(k["cands"][-3][0]) + k["cands"][-3][1]) > 12 * k["clip"]["pcm"].shape[0] // 1152 + 1 for k in cases)
    h = _handle(monkeypatch, 1 << 22)
    try:
        got = _offsets(h, cases)
    finally:
        h.close()
    assert [len(g) for g in got] == [len(k["cands"]) for k in cases]
    _assert_equal(got, expected, cases, "one chunk")


@pytest.mark.parametrize("device", [False, True], ids=["host", "device"])
@pytest.mark.parametrize("chunk", [64, 37])
def test_corpus_equals_the_encoder_in_chunks(built, monkeypatch, cases, expected, chunk, device):
    h = _handle(monkeypatch, chunk)
    try:
        _assert_equal(_offsets(h, cases, device=device), expected, cases, f"{chunk}-frame chunks, {'device' if device else 'host'}")
    finally:
        h.close()


def test_prefixes_against_the_oracle(oracle, cases, expected):
    checked = 0
    for k, e in zip(cases, expected):
        c, cands = k["clip"], k["cands"][:-2]   # the message's prefixes (the last two are arbitrary heads)
        fits = [n for n, ((head, bl), o) in enumerate(zip(cands, e)) if o >= 8 * (len(head) + bl) - 1]
        n_star = max(fits) if fits else -1
        for n in sorted({0, max(n_star, 0), min(n_star + 1, len(cands) - 1), len(cands) - 1}):
            head, bl = cands[n]
            r = oracle.encode(c["pcm"], c["sr"], c["br"], _bits(head, k["body"], bl), taps=False)
            assert r["hide_str_offset"] == e[n], (c["name"], n)
            checked += 1
    assert checked > 2 * len(cases)


def test_overrun_names_clip_candidate_and_frame(built, oracle, clips, cases, expected):
    from mp3stego_b200 import _lib
    idx = list(range(0, len(cases), 97))[:6]
    good = [cases[i] for i in idx]
    h = _lib.Handle(0)
    try:
        for n, c in enumerate(clips[1]):
            cands = [(b"", 0), (b"01#", 2), (b"\xff", 0)]
            if c["bits"] and len(c["bits"]) % 8 == 0:   # the clip's own payload, where it is whole bytes
                cands.append((int(c["bits"], 2).to_bytes(len(c["bits"]) // 8, "big"), 0))
            bad = dict(clip=c, body=b"xy", cands=cands)
            k = 1 + n % 5
            group = good[:k] + [bad] + good[k:]
            first = sum(len(g["cands"]) for g in group[:k])
            want = None
            for j, (head, bl) in enumerate(bad["cands"]):
                r = oracle.encode(c["pcm"], c["sr"], c["br"], _bits(head, bad["body"], bl), taps=False)
                if r["status"] == -3:
                    want = (first + j, r["n_frames"])
                    break
            assert want is not None, c["name"]
            with pytest.raises(IndexError, match=f"clip {k} candidate {want[0]} frame {want[1]}: .*{_lib.STEP_TABLE_OVERRUN}"):
                _offsets(h, group)
            _assert_equal(_offsets(h, good), [expected[i] for i in idx], good, "after an overrun")
    finally:
        h.close()


def _small(cases):
    """Indices of the first five one-frame clips."""
    return [i for i, k in enumerate(cases) if k["clip"]["pcm"].shape[0] == 1152][:5]


def test_bad_arguments_name_clip_and_candidate(handle, cases):
    from mp3stego_b200 import _lib
    group = [cases[i] for i in _small(cases)]
    first2 = sum(len(k["cands"]) for k in group[:2])
    l0 = handle.launches
    g = [dict(k) for k in group]
    g[2] = dict(g[2], cands=g[2]["cands"] + [(bytes(33), 0)])
    with pytest.raises(_lib.M3SError, match=f"\\(-2\\): encode_offsets: clip 2 candidate {first2 + len(group[2]['cands'])}: head of 33 bytes"):
        _offsets(handle, g)
    g = [dict(k) for k in group]
    g[2] = dict(g[2], cands=[(b"1#", len(g[2]["body"]) + 1)] + g[2]["cands"])
    with pytest.raises(_lib.M3SError, match=f"\\(-2\\): encode_offsets: clip 2 candidate {first2}: body_len"):
        _offsets(handle, g)
    pcm = np.concatenate([k["clip"]["pcm"].reshape(-1) for k in group]).astype(np.int16)
    sr = [k["clip"]["sr"] for k in group]
    sr[3] = 22050
    with pytest.raises(_lib.M3SError, match="\\(-2\\): encode: clip 3: sample rate 22050"):
        handle.encode_offsets(pcm, [1152] * 5, sr, [k["clip"]["br"] for k in group], [k["body"] for k in group],
                              [k["cands"] for k in group])
    assert handle.launches == l0


def test_kernel_set_and_taps(handle, cases, expected):
    from mp3stego_b200 import _lib
    group = cases[:40]
    pcm = np.concatenate([k["clip"]["pcm"].reshape(-1) for k in group]).astype(np.int16)
    handle.timing_enable(True)
    try:
        handle.encode(pcm, [k["clip"]["pcm"].shape[0] for k in group], [k["clip"]["sr"] for k in group],
                      [k["clip"]["br"] for k in group])
        t_enc = handle.timing()
        handle.timing_enable(True)   # resets the counts
        got = _offsets(handle, group)
        t = handle.timing()
    finally:
        handle.timing_enable(False)
    _assert_equal(got, expected[:40], group, "timed call")
    assert "k_enc_offsets" in t and "k_enc_analysis" in t and "k_enc_rate" in t
    assert "k_enc_resolve" not in t and "k_enc_pack" not in t, t
    # the emit kernel's timing id also counts the one frame -> clip map kernel of a call: an encode launches one emit per chunk
    # (as many as packs) on top of it, an offsets call none
    n_emit = t_enc["k_enc_emit"][1] - t_enc["k_enc_pack"][1]
    assert n_emit == 1 and t["k_enc_emit"][1] == n_emit, (t_enc, t)
    assert handle._L.m3s_encode_taps(handle._h, None, None, None, None) == -3   # M3S_ERR_STATE
    assert _lib.M3S_K_COUNT == 13 and handle._L.m3s_kernel_name(12) == b"k_enc_offsets" and handle._L.m3s_version() == 400


def test_a_clip_without_candidates_and_empty_payloads(handle, oracle, cases, expected):
    i0, i1, i2 = _small(cases)[:3]
    g = [dict(cases[i0], cands=[]), dict(cases[i1], cands=[(b"", 0)] + cases[i1]["cands"]), cases[i2]]
    got = _offsets(handle, g)
    assert len(got[0]) == 0
    c = g[1]["clip"]
    assert got[1][0] == oracle.encode(c["pcm"], c["sr"], c["br"], "", taps=False)["hide_str_offset"]
    assert np.array_equal(got[1][1:], expected[i1]) and np.array_equal(got[2], expected[i2])


# ---------------------------------------------------------------------------------------------------------- capacity composites
def _files(oracle):
    import glob
    import os
    from conftest import GOLDEN
    blobs = [open(golden_path("test.mp3"), "rb").read()]
    specs = [(32000, 64, 40), (32000, 192, 25), (44100, 128, 60), (44100, 320, 30), (48000, 96, 45), (48000, 256, 20)]
    blobs += [oracle.encode(synth_wav(120 + i, n, sr=sr), sr, br, "", taps=False)["mp3"] for i, (sr, br, n) in enumerate(specs)]
    n_tone = len(blobs)
    for p in sorted(glob.glob(os.path.join(GOLDEN, "stream_*.mp3")) + glob.glob(os.path.join(GOLDEN, "fuzz_*.mp3")) +
                    glob.glob(os.path.join(GOLDEN, "edge_*.mp3"))):
        blob = open(p, "rb").read()
        dec = oracle.decode(blob, oracle.id3_offset(blob), taps=False)
        if dec["channels"] == 2 and dec["n_frames"] > 0:
            blobs.append(blob)
    return blobs, n_tone


def test_capacity_of_the_golden_file(handle):
    from mp3stego_b200 import batch
    blob = open(golden_path("test.mp3"), "rb").read()
    assert batch.capacity_batch(handle, [blob], ["d" * 300]) == [48]
    out, best = batch.hide_batch_fit(handle, [blob], ["d" * 300])
    assert best == [48] and batch.reveal_batch(handle, out) == ["d" * 48]


def test_capacity_batch_and_hide_batch_fit(handle, oracle):
    from mp3stego_b200 import batch
    from mp3stego_b200.steganography import str_to_binary_str
    blobs, n_tone = _files(oracle)
    assert len(blobs) >= n_tone + 20
    rng = np.random.default_rng(31)
    msgs = [_ascii(rng, 400) if i % 4 else "".join(rng.choice(list(MULTIBYTE), size=300)) for i in range(len(blobs))]
    msgs[0] = "d" * 300
    best = batch.capacity_batch(handle, blobs, msgs)
    assert best[0] == 48 and all(-1 <= b < len(m) for b, m in zip(best, msgs))
    fit = [m[:max(b, 0)] for m, b in zip(msgs, best)]
    hid, too_long = batch.hide_batch(handle, blobs, fit)
    assert not any(tl for tl, b in zip(too_long, best) if b >= 0)
    _, too_long1 = batch.hide_batch(handle, blobs, [m[:b + 1] for m, b in zip(msgs, best)])
    assert all(tl for tl, b, m in zip(too_long1, best, msgs) if b < len(m)), [i for i, tl in enumerate(too_long1) if not tl]
    assert sum(b < len(m) for b, m in zip(best, msgs)) >= n_tone + 10
    out, best2 = batch.hide_batch_fit(handle, blobs, msgs)
    assert best2 == best and out == hid
    revealed = batch.reveal_batch(handle, out)
    # reveal_batch gives what the oracle reveals from the same bytes ...
    assert revealed == [oracle.reveal_parse(oracle.decode(o, 0, taps=False)["bits"]) for o in out]
    # ... and that is the message itself where every bit went in, the message is ASCII (the reveal reads the length prefix as a byte
    # count and decodes byte by byte) and the file is at 44.1 or 48 kHz.  The reference's hide -> reveal round trip is not an identity
    # beyond that: the facade also accepts an offset of len(bits) - 1, whose last bit is whatever the next table id carries, and on
    # the 32 kHz / 192 kbps tone file "1#" + one character goes in whole (offset 24 of 24 bits) yet the reference's own reveal of
    # its own output is '' -- as is the writer streams' (stale region addresses, A.E6)
    bits = [str_to_binary_str(str(len(f)) + "#" + f) for f in fit]
    _, hoff, _ = batch._transcode(handle, blobs, bits)
    sr = [oracle.decode(b, oracle.id3_offset(b), taps=False)["sampling_rate"] for b in blobs[:n_tone]]
    whole = [i for i in range(n_tone) if hoff[i] >= len(bits[i]) and fit[i].isascii() and sr[i] != 32000]
    assert len(whole) >= 4 and all(revealed[i] == fit[i] for i in whole), [(i, revealed[i][:40], fit[i][:40]) for i in whole]
