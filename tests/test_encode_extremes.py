"""CPU: the encode edge corpus (tests/encgen.py) against the oracle.

- The oracle encodes every clip of the corpus and refuses exactly the clips whose step search runs past the end of the step
  table (status -3, no bytes; SURVEY A.E13).
- The corpus reaches the edges of the rate loop and the bit writer, asserted from the oracle's taps: every table id the encoder
  can write, big_values 288, big_values 0 with count1 > 0, both count1 tables, part2_3_length 4095 through the stuffing spread,
  the 13-linbits books, the quantize() > 8192 cut-off deciding the step, the double-precision quantiser branch, the top of the
  global_gain range, and payloads that run out 1, 2 and 3 bits into a granule.
- m3s_encode_size (host only) equals the oracle's byte count for every sample rate and bitrate.
- The CPU model of the parallel rate loop (tests/model/rate_variants_model.c) reproduces the oracle on the whole corpus."""
import os
import re
import subprocess

import numpy as np
import pytest

import encgen
from conftest import ROOT

PROBE_CACHE = 24   # csrc/m3s_encode.cu: distinct steps k_enc_probe caches per granule


@pytest.fixture(scope="module")
def clips():
    return encgen.extreme_clips(0)


@pytest.fixture(scope="module")
def encoded(oracle, clips):
    return [oracle.encode(c["pcm"], c["sr"], c["br"], c["bits"]) for c in clips[0]]


def export_tables():
    from mp3stego_b200 import _lib
    L = _lib.load()
    hdr = open(os.path.join(ROOT, "include", "mp3stego_b200.h")).read()
    enum = re.search(r"enum\s*\{\s*(M3S_TAB_HUFF_PACKED.*?)M3S_TAB_COUNT", hdr, re.S).group(1)
    ids = {t.strip(): i for i, t in enumerate(t for t in enum.replace("= 0", "").split(",") if t.strip())}

    def ex(name, cap=20000):
        buf = np.zeros(cap, np.float64)
        n = L.m3s_table_export(ids[name], buf.ctypes.data, cap)
        assert 0 < n <= cap
        return buf[:n]
    return dict(steptabi=ex("M3S_TAB_ENC_STEPTABI").astype(np.int64), steptab=ex("M3S_TAB_ENC_STEPTAB"),
                pair=ex("M3S_TAB_STEGO_PAIR").astype(np.int64).reshape(32, 2))


def quantize(xabs, step, T):
    """quantize() of MP3_Encoder.py:374-415 for |xr| values at one step: (ix, ln >= 10000 mask)."""
    xabs = np.asarray(xabs, np.int64)
    ln = (xabs * int(T["steptabi"][step + 127]) + (1 << 31)) >> 32
    big = ln >= 10000
    i = np.arange(10000, dtype=np.float64)
    int2idx = (np.sqrt(np.sqrt(i) * i) - 0.0946 + 0.5).astype(np.int64)
    ix = int2idx[np.minimum(ln, 9999)]
    dbl = xabs.astype(np.float64) * T["steptab"][step + 127] * 4.656612875e-10
    return np.where(big, np.sqrt(np.sqrt(dbl) * dbl).astype(np.int64), ix), big


def test_oracle_refuses_exactly_the_overrun_clips(oracle, clips, encoded):
    corpus, overrun = clips
    assert sum(c["pcm"].shape[0] for c in corpus) // 1152 >= 2800
    for c, r in zip(corpus, encoded):
        assert r["status"] == 0 and len(r["mp3"]) > 0, c["name"]
    for c in overrun:
        r = oracle.encode(c["pcm"], c["sr"], c["br"], c["bits"])
        assert r["status"] == -3 and r["mp3"] == b"", (c["name"], r["status"])
        assert 0 <= r["n_frames"] < c["pcm"].shape[0] // 1152


def test_corpus_reaches_the_rate_loop_edges(built, clips, encoded):
    T = export_tables()
    corpus = clips[0]
    info = np.concatenate([r["info"] for r in encoded])     # [frame][gr][ch][16]
    ix = np.concatenate([r["ix"] for r in encoded])         # [frame][ch][gr][576]
    mdct = np.concatenate([r["mdct"] for r in encoded])
    xabs = np.abs(mdct.astype(np.int64)).transpose(0, 2, 1, 3)    # -> [frame][gr][ch][576] like info
    ixa = np.abs(ix).transpose(0, 2, 1, 3)
    live = xabs.max(axis=-1) > 0                             # granules the rate loop ran on

    # every table id the reference can write, and the swap partners of each
    ts = set(np.unique(info[..., 4:7]).tolist())
    can = {0, 13, 15} | set(range(16, 32))
    assert set(T["pair"][sorted(can)].ravel().tolist()) <= can
    assert ts == can, sorted(can - ts)
    # run lengths, count1 tables
    bv, c1 = info[..., 1], info[..., 2]
    assert bv.max() == 288
    assert ((bv == 0) & (c1 > 0)).any()
    assert set(np.unique(info[..., 9][c1 > 0]).tolist()) == {0, 1}
    # part2_3_length 4095 outside granule (gr0, ch0): only the stuffing spread of resv_frame_end writes that
    p23 = info[..., 0]
    assert p23.max() == 4095
    assert (p23[:, 0, 1] == 4095).any() or (p23[:, 1, :] == 4095).any()
    # the 13-linbits books: ix - 15 > 4095
    assert ixa.max() > 4110
    assert {23, 31} & ts
    # the quantize() > 8192 cut-off decides the step (one step finer overflows) close to its edge, and the double-precision branch
    step = info[..., 13]
    cut = 0
    dbl = 0
    near = 0
    for f, g, c in zip(*np.nonzero(live)):
        s = int(step[f, g, c])
        q, big = quantize(xabs[f, g, c], s, T)
        assert np.array_equal(q, ixa[f, g, c]), (f, g, c)
        dbl += int(big.sum())
        if s > -120 and quantize([xabs[f, g, c].max()], s - 1, T)[0][0] > 8192:
            cut += 1
            near += int(q.max() >= 4096)
    assert cut > 0 and near > 0 and dbl > 0, (cut, near, dbl)
    # global_gain: step -1 (209) occurs, one below the end of the step table; loud Nyquist squares at 32 kbps jump from it
    # straight past step 0 (the overrun list).  The bottom seen stays above the bin search's floor (step -120)
    gg = info[..., 3][live]
    assert gg.max() == 209
    assert 90 <= gg.min() <= 120, gg.min()
    print(f"corpus: global_gain {gg.min()}..{gg.max()}, cut-off decided the step in {cut} granules ({near} with max ix >= 4096), "
          f"{dbl} values through the double-precision branch")
    # granules that meet the end of the payload with 1, 2 and 3 bits left (the probe's 2-, 1- and 3-bit variants there);
    # payloads longer than the capacity
    ends = set()
    longer = 0
    for c, r in zip(corpus, encoded):
        L = len(c["bits"])
        off = 0
        for fi in range(r["info"].shape[0]):
            for ch in range(2):
                for gr in range(2):
                    cnt = int((r["info"][fi, gr, ch, 4:7] > 0).sum())
                    if 1 <= L - off <= 3 and cnt > 0:
                        ends.add(L - off)
                    off += cnt
            assert off == r["info"][fi, 0, 0, 15]
        assert off == r["hide_str_offset"]
        longer += L > 0 and off < L - 1
    assert ends == {1, 2, 3}
    assert longer > 0


def test_encode_size_matches_oracle(built, oracle):
    from mp3stego_b200 import _lib
    L = _lib.load()
    for sr in encgen.SAMPLE_RATES:
        for br in encgen.BITRATES:
            for nf in (1, 2, 7, 37):
                pcm = np.zeros((nf * 1152, 2), np.int16)
                r = oracle.encode(pcm, sr, br, "", taps=False)
                assert L.m3s_encode_size(nf * 1152, sr, br) == len(r["mp3"]), (sr, br, nf)
            assert L.m3s_encode_size(1151, sr, br) == -1


@pytest.fixture(scope="module")
def model(tmp_path_factory):
    d = tmp_path_factory.mktemp("rate_model_extremes")
    exe = str(d / "rate_variants_model")
    subprocess.check_call(["gcc", "-O2", "-w", "-o", exe, os.path.join(ROOT, "tests", "model", "rate_variants_model.c"), "-lm"])
    return d, exe


def test_rate_model_reproduces_the_oracle_on_the_corpus(model, clips):
    d, exe = model
    slow = {sr: 0 for sr in encgen.SAMPLE_RATES}
    maxsteps = 0
    for i, c in enumerate(clips[0]):
        raw, pay = str(d / "clip.raw"), str(d / "clip.txt")
        np.ascontiguousarray(c["pcm"], dtype=np.int16).tofile(raw)
        open(pay, "w").write(c["bits"])
        out = subprocess.run([exe, raw, str(c["pcm"].shape[0] // 1152), str(c["br"]), pay, "-1", str(c["sr"])],
                             capture_output=True, text=True, check=True).stdout
        m = re.search(r"granules (\d+) silent (\d+) slow (\d+) bad (\d+) maxsteps (\d+)", out)
        assert m, (c["name"], out)
        g, _, sl, bad, ms = map(int, m.groups())
        assert bad == 0, (c["name"], out)
        slow[c["sr"]] += sl
        maxsteps = max(maxsteps, ms)
    # the stale-address path (A.E6) is reached at every sample rate
    assert all(v > 0 for v in slow.values()), slow
    # the active variants of one granule probe far fewer distinct steps than k_enc_probe caches, so its cache-full fallback
    # is not reached by this corpus
    assert maxsteps < PROBE_CACHE, maxsteps
    print(f"rate model: slow granules per sample rate {slow}, most distinct steps of one granule {maxsteps}")
