"""CPU: the in-repo stream writer (tests/streamgen.py).  With its new options off it regenerates the 24 committed writer streams
byte for byte; the extreme corpus it writes decodes, through the oracle, to the spectra the writer put in, and reaches the
edges of the decoder's domain the committed streams never reach (|x| >= 256 up to 8206, global_gain 0 / 255, subblock_gain 7,
big_values 288, count1 up to the stop at 572, part2_3_length near 4095, PCM past int16 and past int32)."""
import functools

import numpy as np
import pytest

import streamgen as S
from conftest import golden_path


@functools.lru_cache(maxsize=None)
def extreme_corpus():
    """[(bytes, writer spectra [frame][gr][ch][576], config)] of the N_EXTREME extreme streams (written once per session)."""
    out = []
    for k in range(S.N_EXTREME):
        kw = S.extreme_config(k)
        data, spec, _ = S.make_stream(**kw, spectra=True)
        out.append((data, spec, kw))
    return out


@functools.lru_cache(maxsize=None)
def extreme_oracle():
    from oracle import oracle as O
    return [O.decode(d) for d, _, _ in extreme_corpus()]


@pytest.mark.parametrize("name", sorted(S.STREAMS))
def test_writer_streams_regenerate(built, name):
    assert S.make_stream(**S.STREAMS[name]) == open(golden_path(f"stream_{name}.mp3"), "rb").read()


def test_fuzz_streams_regenerate(built):
    for k in range(S.N_FUZZ):
        assert S.make_stream(**S.fuzz_config(k)) == open(golden_path("fuzz_%02d.mp3" % k), "rb").read(), k


def test_table_sources_agree(built):
    """The library's exported tables and the oracle's header give the writer the same code books."""
    a, b = S._from_export(), S._from_oracle_header()
    assert a.big_value_max == b.big_value_max and a.big_value_linbit == b.big_value_linbit
    assert a.pair == b.pair and a.quad == b.quad and a.sfb_long == b.sfb_long and a.slen == b.slen


def test_extreme_corpus_spectra_vs_oracle(built, oracle):
    """The oracle's Huffman stage returns, for every granule of every extreme stream, the integer spectrum the writer wrote."""
    corpus, refs = extreme_corpus(), extreme_oracle()
    assert 120 <= len(corpus) and 2500 <= sum(len(s) for _, s, _ in corpus)
    for k, ((data, spec, kw), ref) in enumerate(zip(corpus, refs)):
        nch = 1 if kw["mode"] == 3 else 2
        assert ref["status"] == 0 and ref["channels"] == nch and ref["n_frames"] == spec.shape[0], k
        assert ref["sampling_rate"] == kw["sr"], k
        assert np.array_equal(ref["spectra"], spec), k


def test_extreme_corpus_coverage(built, oracle):
    """What the extreme corpus must keep reaching, read from the oracle's decode (not from the writer's intentions)."""
    corpus, refs = extreme_corpus(), extreme_oracle()
    sp = np.concatenate([r["spectra"].reshape(-1, 576) for r in refs])
    side = np.concatenate([r["side"].reshape(-1, r["side"].shape[-1]) for r in refs])
    ax = np.abs(sp)
    for v in (255, 256, 257, 8206):
        assert (ax == v).any(), v
    assert ((ax >= 256).any(axis=1)).sum() >= 50                     # granules that take the computed |x|^(4/3) branch
    assert (side[:, 1] == 288).any()                                   # big_values
    assert (side[:, 2] == 0).any() and (side[:, 2] == 255).any()       # global_gain
    ws = side[:, 4] == 1
    assert (side[ws][:, 10:13] == 7).any()                             # subblock_gain
    assert (side[:, 0] >= 4000).sum() >= 10                            # part2_3_length near the 12-bit limit
    # count1 quads at the end of the spectrum: a non-zero sample at 568..573 outside the big-values region
    c1 = [(sp[i, 568:574] != 0).any() for i in np.nonzero(2 * side[:, 1] <= 568)[0]]
    assert sum(c1) >= 10
    v = np.concatenate([r["pcm"].ravel() for r in refs]) * 32767.0
    assert (np.abs(v) >= 32768).sum() > 1000                           # int16 wrap
    assert (v >= 2.0 ** 31).sum() > 100 and (v < -(2.0 ** 31)).sum() > 100   # past int32: 0x80000000 -> 0 (A.D8)
    inside = np.abs(v) < 2.0 ** 31
    assert inside.mean() > 0.5                                          # most samples still go through the ordinary conversion
    # the writer's configurations: mono / stereo / joint stereo with every mode extension, CRC, VBR, mixed blocks, reservoir
    kws = [kw for _, _, kw in corpus]
    assert {kw["mode"] for kw in kws} == {0, 1, 3}
    assert {kw["mode_ext"] for kw in kws if kw["mode"] == 1} == {0, 1, 2, 3}
    assert any(kw["crc"] for kw in kws) and any("vbr" in kw for kw in kws) and any(kw["reservoir"] for kw in kws)
    assert ((side[:, 5] == 2) & (side[:, 6] == 1)).any() and (side[:, 5] == 1).any() and (side[:, 5] == 3).any()
    assert any((r["main_data_begin"] > 0).any() for r in refs)
