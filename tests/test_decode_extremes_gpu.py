"""GPU: the decoder at the edges of its domain -- the extreme corpus of tests/streamgen.py (|x| up to 8206 through the computed
|x|^(4/3) branch, global_gain 0..255, subblock_gain 0..7, big_values 288, count1 to the stop at 572, part2_3_length near 4095,
PCM far past int16 and past int32) -- against the oracle's float64 decode, for every entry point.

  integer stages   spectra (= the writer's), table ids and reveal bits equal
  float64 (exact)  int16 PCM sample-exact on the goldens; on the extreme corpus wherever v = ref * 32767 is more than
                   C64 * s_f * 32767 from every integer (C64 = 1e-12, the oracle's own pinning to the reference), which
                   includes every out-of-int32 sample: 0x80000000 -> 0 (A.D8)
  FP32 float tap   |got - ref| <= C * s_f, s_f = max(peak of frame f, peak of frame f - 1, 1/32767) of the oracle's PCM
  FP32 int16       with e_f = C * s_f * 32767: wherever v is more than e_f away from every integer and from +-2^31 the
                   sample equals the reference's; elsewhere any truncation of a value in [v - e_f, v + e_f] is accepted

C = 1e-5.  The fractions of samples that fall under an allowance depend only on the oracle's PCM: 23.0 % of the goldens'
in-int32 samples (FP32), 96.1 % of the extreme corpus's (its frames mostly peak far above full scale, where FP32 cannot
resolve integers) and 18.5 % of them in float64.  Measured on one B200 (1000 W power limit): worst float-tap ratio
|got - ref| / (C * s_f) 0.94 on the extreme corpus and 0.46 on the goldens (k_hybrid_fast); on the goldens the FP32 int16
samples of k_hybrid_fast obey the rule even with C = 1e-6.
Found here and fixed: the kernels saturated v >= 2^31 to 0x7FFFFFFF (int16 -1) where x86 gives 0x80000000 (int16 0).
"""
import numpy as np
import pytest

from test_parity_decode import _all_golden_blobs
from test_stream_writer import extreme_corpus, extreme_oracle

pytestmark = pytest.mark.gpu

C = 1e-5
TWO31 = 2.0 ** 31
MAX_FLOAT_RATIO = 1.0      # worst |got - ref| / (C * s_f) accepted from the FP32 float tap
MAX_TOLERATED = 0.30       # fraction of in-int32 FP32 int16 samples allowed to fall under the e_f allowance (goldens)
MAX_TOLERATED_LOUD = 0.98  # the same on the extreme corpus, whose frames mostly peak far above full scale
C64 = 1e-12                # float64 allowance on the extreme corpus: the oracle itself is pinned to the reference at 1e-12
MAX_TOLERATED_F64 = 0.25   # fraction of in-int32 float64 int16 samples of the extreme corpus under the C64 allowance


def _split(sc, pcm, sp=None, ids=None, bits=None):
    fb = np.concatenate([[0], np.cumsum(sc["n_frames"])])
    eb = np.concatenate([[0], np.cumsum(sc["pcm_rows"] * np.maximum(sc["channels"], 1))])
    out = []
    for i in range(len(sc["n_frames"])):
        ch = max(int(sc["channels"][i]), 1)
        out.append(dict(n_frames=int(sc["n_frames"][i]), channels=int(sc["channels"][i]),
                        pcm=pcm[eb[i]:eb[i + 1]].reshape(-1, ch),
                        spectra=None if sp is None else sp[fb[i]:fb[i + 1]].astype(np.int32),
                        ids=None if ids is None else ids[fb[i]:fb[i + 1]], bits=None if bits is None else bits[i]))
    return out


def _decode(h, blobs, starts=None, exact=False, as_float=False, spectra=False):
    data = np.frombuffer(b"".join(blobs), np.uint8)
    off = np.concatenate([[0], np.cumsum([len(b) for b in blobs])])
    sc = h.decode_scan(data, off, starts)
    ids, bits = h.decode_reveal()
    pcm, sp = h.decode_run(spectra=spectra, as_float=as_float, exact=exact)
    return _split(sc, pcm, sp, ids, bits)


def _to_int16(v):
    """x86 numpy astype(int16) of float64 v: truncate to int32 (0x80000000 outside it or NaN), keep the low 16 bits."""
    t = np.where((v >= -TWO31) & (v < TWO31), np.trunc(np.nan_to_num(v)), -TWO31).astype(np.int64)
    return (t & 0xFFFF).astype(np.uint16).view(np.int16)


def _frame_scale(ref_pcm):
    """s_f per row of the oracle's PCM [rows, ch]: max(peak of frame f, peak of frame f - 1, 1/32767)."""
    rows = ref_pcm.shape[0]
    nf = -(-rows // 1152)
    peak = np.zeros(nf)
    a = np.abs(ref_pcm)
    for f in range(nf):
        peak[f] = a[f * 1152:(f + 1) * 1152].max() if a.size else 0.0
    s = np.maximum(peak, np.concatenate([[0.0], peak[:-1]]))
    s = np.maximum(s, 1.0 / 32767)
    return np.repeat(s, 1152)[:rows, None]


def _float_ratio(got, ref_pcm):
    """Worst |got - ref| / (C * s_f) of one file's float tap."""
    if ref_pcm.size == 0:
        return 0.0
    assert got.shape == ref_pcm.shape
    return float((np.abs(got.astype(np.float64) - ref_pcm) / (C * _frame_scale(ref_pcm))).max())


def _int16_rule(got, ref_pcm, c=C):
    """int16 samples vs the reference's conversion of the oracle's float64 PCM, allowance e_f = c * s_f * 32767.
    Returns (violations, tolerated, in-int32)."""
    if ref_pcm.size == 0:
        return 0, 0, 0
    assert got.shape == ref_pcm.shape
    v = ref_pcm * 32767.0
    eps = c * _frame_scale(ref_pcm) * 32767.0
    ref16 = _to_int16(v).astype(np.int64)
    g = got.astype(np.int64)
    near_edge = np.abs(np.abs(v) - TWO31) <= eps
    inside = (v >= -TWO31) & (v < TWO31)
    near_int = inside & (np.abs(v - np.round(v)) <= eps)
    loose = near_int | near_edge
    bad = ~loose & (g != ref16)
    # loose samples: any outcome of v' in [v - eps, v + eps], i.e. a truncation in [lo, hi] modulo 2^16 (or 0x80000000 -> 0 past the edge)
    lo = np.trunc(np.clip(v - eps, -TWO31, TWO31 - 1)).astype(np.int64)
    hi = np.trunc(np.clip(v + eps, -TWO31, TWO31 - 1)).astype(np.int64)
    ok = ((g - lo) % 65536 <= hi - lo) | (hi - lo >= 65535) | (near_edge & (g == 0))
    bad |= loose & ~ok
    return int(bad.sum()), int((loose & inside).sum()), int(inside.sum())


def _check_exact(got, ref, what):
    assert got["pcm"].shape == ref["pcm16"].shape, what
    d = got["pcm"] != ref["pcm16"]
    if d.any():
        v = ref["pcm"][d] * 32767.0
        pytest.fail(f"{what}: {int(d.sum())} int16 samples differ, {int((v >= TWO31).sum())} of them at v >= 2^31, "
                    f"{int((v < -TWO31).sum())} at v < -2^31")


def _check_exact_loud(got, ref, what):
    """float64 int16 PCM of the extreme corpus: equal to the reference's except within C64 * s_f * 32767 of an integer."""
    assert got["pcm"].shape == ref["pcm16"].shape, what
    b, t, n = _int16_rule(got["pcm"], ref["pcm"], C64)
    if b:
        _check_exact(got, ref, what + f" ({b} outside the float64 allowance)")
    return t, n


def _check_all(h, blobs, refs, starts=None, tag="", max_tolerated=MAX_TOLERATED, loud=False):
    """float64 (sample-exact, or by the C64 rule on loud material), FP32 float tap and FP32 int16 rule over one batch."""
    tol64 = n64 = 0
    for i, (g, r) in enumerate(zip(_decode(h, blobs, starts, exact=True), refs)):
        assert g["n_frames"] == r["n_frames"], (tag, i)
        if loud:
            t, n = _check_exact_loud(g, r, f"{tag} exact file {i}")
            tol64, n64 = tol64 + t, n64 + n
        else:
            _check_exact(g, r, f"{tag} exact file {i}")
    assert tol64 <= MAX_TOLERATED_F64 * max(n64, 1), (tag, tol64, n64)
    worst = 0.0
    for i, (g, r) in enumerate(zip(_decode(h, blobs, starts, as_float=True), refs)):
        ratio = _float_ratio(g["pcm"], r["pcm"])
        assert ratio <= MAX_FLOAT_RATIO, (tag, i, ratio)
        worst = max(worst, ratio)
    bad = tol = inside = 0
    for i, (g, r) in enumerate(zip(_decode(h, blobs, starts), refs)):
        b, t, n = _int16_rule(g["pcm"], r["pcm"])
        assert b == 0, f"{tag} FP32 int16 file {i}: {b} samples break the rule"
        tol, inside = tol + t, inside + n
    frac = tol / max(inside, 1)
    print(f"[{tag}] float64 int16 tolerated {tol64} of {n64}; worst float-tap ratio {worst:.4f}, FP32 int16 tolerated {tol} of "
          f"{inside} in-int32 samples ({100 * frac:.3f} %)")
    assert frac <= max_tolerated, frac
    return worst, frac


@pytest.fixture(scope="module")
def corpus(built):
    return [d for d, _, _ in extreme_corpus()], [s for _, s, _ in extreme_corpus()], extreme_oracle()


def test_integer_stages(handle, corpus):
    """Huffman stage, table ids and reveal bits of the extreme corpus: equal to the oracle's, and the spectra to the writer's."""
    blobs, wspec, refs = corpus
    got = _decode(handle, blobs, spectra=True)
    for i, (g, w, r) in enumerate(zip(got, wspec, refs)):
        ch = max(r["channels"], 1)
        assert g["n_frames"] == r["n_frames"] == w.shape[0], i
        assert np.array_equal(g["spectra"][:, :, :ch], r["spectra"][:, :, :ch]), i
        assert np.array_equal(g["spectra"][:, :, :ch], w[:, :, :ch]), i
        assert np.array_equal(g["ids"], r["tables"]), i
        assert g["bits"] == r["bits"], i


def test_extremes_vs_oracle(handle, corpus):
    blobs, _, refs = corpus
    _check_all(handle, blobs, refs, tag="extreme", max_tolerated=MAX_TOLERATED_LOUD, loud=True)


def test_goldens_vs_oracle_int16_rule(handle, oracle):
    """The same three checks over every committed golden stream (encoder-made files, writer / fuzz / edge streams)."""
    blobs = _all_golden_blobs()
    starts = [oracle.id3_offset(b) for b in blobs]
    refs = [oracle.decode(b, s) for b, s in zip(blobs, starts)]
    _check_all(handle, blobs, refs, starts, tag="goldens")


def test_frame_ranges_vs_whole_file(handle, corpus):
    """m3s_decode_run_range at seeded random cuts of the reservoir-using extreme streams: the joined ranges follow the oracle's
    whole-file decode (float64 sample-exact, FP32 by the int16 rule)."""
    blobs, _, refs = corpus
    pick = [i for i, r in enumerate(refs) if (r["main_data_begin"] > 0).any()]
    assert len(pick) >= 30
    sel = [blobs[i] for i in pick]
    data = np.frombuffer(b"".join(sel), np.uint8)
    off = np.concatenate([[0], np.cumsum([len(b) for b in sel])])
    sc = handle.decode_scan(data, off)
    rng = np.random.default_rng(4242)
    for j, i in enumerate(pick):
        nf, ch, ref = int(sc["n_frames"][j]), max(int(sc["channels"][j]), 1), refs[i]
        cuts = np.unique(np.concatenate([[0, nf], rng.integers(1, nf, size=int(rng.integers(1, 5)))]))
        for exact in (True, False):
            parts = []
            for a, b in zip(cuts[:-1], cuts[1:]):
                pcm, rows = handle.decode_run_range(j, int(a), int(b - a), exact=exact)
                parts.append(pcm[:rows * ch].reshape(-1, ch))
            got = np.concatenate(parts)
            if exact:
                _check_exact_loud(dict(pcm=got), ref, f"ranges {cuts.tolist()} of extreme stream {i}")
            else:
                assert _int16_rule(got, ref["pcm"])[0] == 0, (i, cuts.tolist())


@pytest.mark.parametrize("device", [False, True])
def test_pipelined_call_exact(built, corpus, monkeypatch, device):
    """m3s_decode (the one-call pipelined decode) over the extreme corpus in waves of ~30 kB, float64: sample-exact, with host
    buffers and with device-resident input and output."""
    import torch
    from mp3stego_b200 import _lib
    monkeypatch.setenv("M3S_DEC_WAVE_BYTES", "30000")
    h = _lib.Handle(0)
    try:
        blobs, _, refs = corpus
        host = np.frombuffer(b"".join(blobs), np.uint8)
        off = np.concatenate([[0], np.cumsum([len(b) for b in blobs])])
        if device:
            nfr = sum(r["n_frames"] for r in refs) + 8
            pcm = torch.zeros(nfr * 1152 * 2, dtype=torch.int16, device="cuda")
            res = h.decode(torch.from_numpy(host.copy()).cuda(), off, pcm=pcm, frames_bound=nfr, exact=True)
            for k in ("pcm", "table_ids", "reveal_bits"):
                res[k] = res[k].cpu().numpy()
        else:
            res = h.decode(host, off, exact=True)
        strings = h.reveal_strings(res)
        fb = np.concatenate([[0], np.cumsum(res["n_frames"])])
        for i, r in enumerate(refs):
            assert int(res["n_frames"][i]) == r["n_frames"] and strings[i] == r["bits"], i
            assert np.array_equal(np.asarray(res["table_ids"][12 * fb[i]:12 * fb[i + 1]]).reshape(-1, 12), r["tables"]), i
            got = np.asarray(res["pcm"][res["pcm_off"][i]:res["pcm_off"][i + 1]]).reshape(r["pcm16"].shape)
            _check_exact_loud(dict(pcm=got), r, f"m3s_decode extreme stream {i}")
    finally:
        h.close()
