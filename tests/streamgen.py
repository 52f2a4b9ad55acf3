"""Seeded MPEG-1 Layer III stream writer: random integer spectra written with the reference's code books and bit layout
(ISO 11172-3 as FrameSideInformation.py:39-137 and Frame.py:365-559 parse it).

The writer of tests/golden/make_streams.py, made self-contained: the code books, linbits, book dimensions, long-block band
edges and slen pairs come from the library's host-only m3s_table_export (tests/test_tables.py pins every one of them to the
reference's digests), or from oracle/oracle_tables.h when the library is not built.  With every option at its default the
random draws are the original's, so make_stream(**STREAMS[k]) and make_stream(**fuzz_config(k)) give the committed
tests/golden/stream_<k>.mp3 and fuzz_NN.mp3 byte for byte.

Options beyond the original (each off by default, and drawing nothing from the generator while off):
  big_lin       probability per big-values pair in a linbits book of magnitudes over the book's whole range (up to
                15 + 8191 = 8206), with 254..258 -- the requantiser's table / computed boundary -- drawn often
  gain_edge     probability per granule of global_gain 0 or 255 (gain_lo / gain_hi set the ordinary range, up to 0..256)
  sbg_hi        subblock_gain drawn from 0..sbg_hi-1 (default 4; 8 for the whole field)
  bv_full       probability per granule of big_values = 288 (max_bv sets the ordinary bound, up to 288)
  quads_end     probability per granule that count1 quads run until the reference's stop at sample 572 (A.D5)
  fill          probability per granule (of those whose quads ran to the stop) of ignored bits after the stop, up to a
                part2_3_length of 4000..4095; needs 320 kbps at 32 kHz and the reservoir to fit
With the new options on, big values stop early (big_values shrinks) when the granule's 4095-bit budget runs out.

make_stream(..., spectra=True) also returns the integer spectra written, [frame][granule][channel][576] -- what a decoder's
Huffman stage must produce, with the reference's quirks the writer relies on: books 0 / 4 / 14 decode to zeros without bits,
count1 stops at sample + 4 >= 576.
"""
import os
import re

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BITRATES = [0, 32, 40, 48, 56, 64, 80, 96, 112, 128, 160, 192, 224, 256, 320]
SR_CODE = {44100: 0, 48000: 1, 32000: 2}


class _Tables:
    """big_value_max / big_value_linbit / pair books / count1 table A / long band edges / slen, as the writer needs them."""

    def __init__(self, dim, linbits, pair, quad, sfb_long, slen):
        self.big_value_max = dim          # [t] book dimension (0 for 0 / 4 / 14)
        self.big_value_linbit = linbits   # [t]
        self.pair = pair                  # [t] -> flat [(code right-aligned, length)], index x * dim + y
        self.quad = quad                  # count1 table A: [8v + 4w + 2x + y] -> (code, length)
        self.sfb_long = sfb_long          # sample rate -> 23 band edges
        self.slen = slen                  # [scalefac_compress] -> (slen1, slen2)


def _from_export():
    import sys
    pkg = os.path.join(ROOT, "mp3-steganography-lib_b200")
    if pkg not in sys.path:
        sys.path.insert(0, pkg)
    from mp3stego_b200 import _lib
    L = _lib.load()
    hdr = open(os.path.join(ROOT, "include", "mp3stego_b200.h")).read()
    enum = re.search(r"enum\s*\{\s*(M3S_TAB_HUFF_PACKED.*?)M3S_TAB_COUNT", hdr, re.S).group(1)
    ids = {t.strip(): i for i, t in enumerate(t for t in enum.replace("= 0", "").split(",") if t.strip())}

    def ex(name, cap=4096):
        buf = np.zeros(cap, np.float64)
        n = L.m3s_table_export(ids[name], buf.ctypes.data, cap)
        assert 0 < n <= cap
        return [int(v) for v in buf[:n]]
    packed, off, dim = ex("M3S_TAB_HUFF_PACKED"), ex("M3S_TAB_HUFF_BOOK_OFF"), ex("M3S_TAB_HUFF_DIM")
    linbits, sfb, slen = ex("M3S_TAB_HUFF_LINBITS"), ex("M3S_TAB_SFB_LONG"), ex("M3S_TAB_SLEN")
    pair = [[(r >> 8, r & 0xFF) for r in packed[off[t]:off[t] + dim[t] * dim[t]]] for t in range(32)]
    quad = [(r >> 8, r & 0xFF) for r in packed[off[32]:off[32] + 16]]
    sfb_long = {sr: sfb[23 * k:23 * k + 23] for sr, k in SR_CODE.items()}
    return _Tables(dim[:32], linbits[:32], pair, quad, sfb_long, [(slen[2 * i], slen[2 * i + 1]) for i in range(16)])


def _from_oracle_header():
    src = open(os.path.join(ROOT, "oracle", "oracle_tables.h")).read()

    def arr(name):
        body = re.search(r"\b%s\s*\[[^\]]*\]\s*=\s*\{(.*?)\};" % name, src, re.S).group(1)
        return [int(v.rstrip("uU"), 0) for v in re.findall(r"0x[0-9a-fA-F]+u?|-?\d+", body)]
    code, ln, off, mx, lb = (arr(n) for n in ("ORA_HUFF_CODE_L", "ORA_HUFF_LEN", "ORA_HUFF_OFF", "ORA_HUFF_MAX", "ORA_HUFF_LINBITS"))
    qc, ql, sfb, slen = arr("ORA_QUAD_CODE_L"), arr("ORA_QUAD_LEN"), arr("ORA_SFB_LONG"), arr("ORA_SLEN")
    pair = [[(code[off[t] + i] >> (32 - ln[off[t] + i]), ln[off[t] + i]) for i in range(mx[t] * mx[t])] for t in range(32)]
    quad = [(qc[e] >> (32 - ql[e]), ql[e]) for e in range(16)]
    sfb_long = {sr: sfb[23 * k:23 * k + 23] for sr, k in SR_CODE.items()}
    return _Tables(mx[:32], lb[:32], pair, quad, sfb_long, [(slen[2 * i], slen[2 * i + 1]) for i in range(16)])


_T = None


def tables():
    global _T
    if _T is None:
        try:
            _T = _from_export()
        except Exception:
            _T = _from_oracle_header()
    return _T


class Bits:
    def __init__(self):
        self.parts = []
        self.n = 0

    def put(self, v, n):
        if n:
            self.parts.append(format(int(v) & ((1 << n) - 1), "0%db" % n))
            self.n += n

    def extend(self, other):
        self.parts += other.parts
        self.n += other.n

    def __len__(self):
        return self.n

    def tobytes(self):
        s = "".join(self.parts)
        s += "0" * (-len(s) % 8)
        return int(s, 2).to_bytes(len(s) // 8, "big") if s else b""


def huff_pair(w, t, x, y):
    """One big-values pair with table t (1..31, not 4/14)."""
    T = tables()
    dim = T.big_value_max[t]
    lin = T.big_value_linbit[t]
    ax, ay = abs(x), abs(y)
    cx, cy = min(ax, dim - 1), min(ay, dim - 1)
    code, ln = T.pair[t][dim * cx + cy]
    w.put(code, ln)
    for a, c, v in ((ax, cx, x), (ay, cy, y)):
        if lin and c == dim - 1:
            w.put(a - c, lin)
        if c > 0:
            w.put(1 if v < 0 else 0, 1)


def huff_quad(w, sel, q):
    a = [abs(v) for v in q]
    if sel == 1:
        w.put(((1 - a[0]) << 3) | ((1 - a[1]) << 2) | ((1 - a[2]) << 1) | (1 - a[3]), 4)
    else:
        w.put(*tables().quad[8 * a[0] + 4 * a[1] + 2 * a[2] + a[3]])
    for v in q:
        if v:
            w.put(1 if v < 0 else 0, 1)


def table_limit(t):
    T = tables()
    if t in (0, 4, 14):
        return 0
    return T.big_value_max[t] - 1 + ((1 << T.big_value_linbit[t]) - 1 if T.big_value_linbit[t] else 0)


def _big_magnitude(rng, lim):
    """|x| for the big_lin option: the requantiser's table / computed boundary, the book's maximum, or anything in between."""
    r = rng.random()
    if r < 0.4 and lim >= 258:
        m = int(rng.integers(254, 259))
    elif r < 0.55:
        m = lim
    else:
        m = int(rng.integers(0, lim + 1))
    return -m if rng.random() < 0.5 else m


def make_granule(rng, sr, gr, ch, opts, scfsi):
    """Random side info + spectra for one granule-channel; returns (side dict, main-data Bits, integer spectrum[576])."""
    T = tables()
    long_win = T.sfb_long[sr]
    si = dict(scalefac_compress=int(rng.integers(0, 16)) if opts.get("scalefac", True) else 0,
              global_gain=int(rng.integers(opts.get("gain_lo", 135), opts.get("gain_hi", 168))),
              preflag=int(rng.integers(0, 2)) if opts.get("scalefac", True) else 0,
              scalefac_scale=int(rng.integers(0, 2)) if opts.get("scalefac", True) else 0,
              count1table_select=int(rng.integers(0, 2)))
    if opts.get("gain_edge") and rng.random() < opts["gain_edge"]:
        si["global_gain"] = 255 if rng.random() < 0.5 else 0
    ws = 1 if opts.get("switching") and rng.random() < 0.7 else 0
    si["window_switching"] = ws
    tabs_pool = opts.get("tables", [t for t in range(1, 32) if t not in (4, 14)])
    pick = lambda: int(rng.choice(tabs_pool)) if rng.random() > 0.08 else int(rng.choice([0, 4, 14]))  # noqa: E731
    if ws:
        bt = int(rng.choice(opts.get("block_types", [1, 2, 3])))
        si["block_type"] = bt
        si["mixed_block_flag"] = int(rng.integers(0, 2)) if bt == 2 and opts.get("mixed", True) else 0
        si["table_select"] = [pick(), pick()]
        si["subblock_gain"] = [int(rng.integers(0, opts.get("sbg_hi", 4))) for _ in range(3)]
        r0 = 8 if bt == 2 else 7
        r1 = 20 - r0
        if bt == 2:
            bounds = (36, 576)
        else:
            bounds = (long_win[r0 + 1], long_win[min(r0 + r1 + 2, 22)])
    else:
        si["block_type"] = 0
        si["mixed_block_flag"] = 0
        si["table_select"] = [pick(), pick(), pick()]
        r0 = int(rng.integers(0, 16))
        r1 = int(rng.integers(0, 8))
        while r0 + r1 + 2 > 22:
            r0 = int(rng.integers(0, 16))
            r1 = int(rng.integers(0, 8))
        si["region0_count"], si["region1_count"] = r0, r1
        bounds = (long_win[r0 + 1], long_win[r0 + r1 + 2])
    w = Bits()
    spec = np.zeros(576, np.int32)
    # ---- part2: scalefactors (Frame.py:365-441)
    sl1, sl2 = T.slen[si["scalefac_compress"]]
    rnd = lambda n: int(rng.integers(0, 1 << n)) if n else 0  # noqa: E731
    if ws and si["block_type"] == 2:
        if si["mixed_block_flag"]:
            for _ in range(8):
                w.put(rnd(sl1), sl1)
            for _ in range(3, 6):
                for _w in range(3):
                    w.put(rnd(sl1), sl1)
        else:
            for _ in range(6):
                for _w in range(3):
                    w.put(rnd(sl1), sl1)
        for _ in range(6, 12):
            for _w in range(3):
                w.put(rnd(sl2), sl2)
    elif gr == 0:
        for _ in range(11):
            w.put(rnd(sl1), sl1)
        for _ in range(10):
            w.put(rnd(sl2), sl2)
    else:
        for i, (lo, hi) in enumerate(((0, 6), (6, 11), (11, 16), (16, 21))):
            if not scfsi[ch][i]:
                for _ in range(lo, hi):
                    w.put(rnd(sl1 if i < 2 else sl2), sl1 if i < 2 else sl2)
    # ---- part3: big values + count1 (Frame.py:443-559)
    extreme = bool(opts.get("big_lin") or opts.get("quads_end") or opts.get("fill") or opts.get("bv_full"))
    max_bv = opts.get("max_bv", 200)
    bv = int(rng.integers(0, max_bv + 1))
    if opts.get("bv_full") and rng.random() < opts["bv_full"]:
        bv = 288
    amp = opts.get("amp", 12)
    for p in range(bv):
        s = 2 * p
        t = si["table_select"][0] if s < bounds[0] else (si["table_select"][1] if s < bounds[1] else
                                                          (si["table_select"][2] if len(si["table_select"]) > 2 else opts["_stale_t2"]))
        lim = table_limit(t)
        if lim == 0:
            continue   # table 0 / 4 / 14: zeros, no bits
        lin = T.big_value_linbit[t]
        if extreme and len(w) + 19 + 2 * lin + 2 > 3600:
            bv = p     # the granule's bit budget is spent: big values end here
            break
        if lin and opts.get("big_lin") and rng.random() < opts["big_lin"]:
            x, y = _big_magnitude(rng, lim), _big_magnitude(rng, lim)
        else:
            hi = min(lim, amp if s < 60 else max(2, amp // 3))
            if lin and rng.random() < 0.05:
                hi = min(lim, 15 + (1 << min(lin, 6)))
            x = int(rng.integers(-hi, hi + 1))
            y = int(rng.integers(-hi, hi + 1))
        huff_pair(w, t, x, y)
        spec[s], spec[s + 1] = x, y
    si["big_values"] = bv
    to_end = bool(opts.get("quads_end") and rng.random() < opts["quads_end"])
    if to_end:
        nq = max(0, (572 - 2 * bv + 3) // 4)         # quads while sample + 4 < 576: the last one may cover 572, 573 (A.D5)
    else:
        nq_max = max(0, (572 - 2 * bv) // 4)        # the reference stops at sample + 4 < 576 (A.D5)
        nq = int(rng.integers(0, min(nq_max, opts.get("max_quads", 60)) + 1))
    for k in range(nq):
        if extreme and len(w) + 10 > 4095:
            to_end = False
            break
        q = [int(v) for v in rng.integers(-1, 2, size=4)]
        huff_quad(w, si["count1table_select"], q)
        spec[2 * bv + 4 * k:2 * bv + 4 * k + 4] = q
    if to_end and opts.get("fill") and rng.random() < opts["fill"]:
        target = int(rng.integers(4000, 4096))
        while len(w) < target:                       # past the stop: bits the decoder must skip
            n = min(30, target - len(w))
            w.put(int(rng.integers(0, 1 << n)), n)
    elif opts.get("stuff_ones") and si["count1table_select"] == 0 and rng.random() < 0.5:
        for _ in range(int(rng.integers(1, 9))):
            w.put(1, 1)                              # table A '1' = zero quad: stuffing as the reference encoder writes it
    si["part2_3_length"] = len(w)
    assert len(w) < 4096
    return si, w, spec


def side_info_bits(frame, nch):
    w = Bits()
    w.put(frame["main_data_begin"], 9)
    w.put(0, 3 if nch == 2 else 5)
    for ch in range(nch):
        for b in range(4):
            w.put(frame["scfsi"][ch][b], 1)
    for gr in range(2):
        for ch in range(nch):
            s = frame["gr"][gr][ch]
            w.put(s["part2_3_length"], 12)
            w.put(s["big_values"], 9)
            w.put(s["global_gain"], 8)
            w.put(s["scalefac_compress"], 4)
            w.put(s["window_switching"], 1)
            if s["window_switching"]:
                w.put(s["block_type"], 2)
                w.put(s["mixed_block_flag"], 1)
                for t in s["table_select"]:
                    w.put(t, 5)
                for g in s["subblock_gain"]:
                    w.put(g, 3)
            else:
                for t in s["table_select"]:
                    w.put(t, 5)
                w.put(s["region0_count"], 4)
                w.put(s["region1_count"], 3)
            w.put(s["preflag"], 1)
            w.put(s["scalefac_scale"], 1)
            w.put(s["count1table_select"], 1)
    assert len(w) == (256 if nch == 2 else 136), len(w)
    return w.tobytes()


def make_stream(seed, n_frames, sr=44100, bitrate=128, mode=0, mode_ext=0, crc=False, opts=None, vbr=None, reservoir=False,
                spectra=False):
    """mode: 0 stereo, 1 joint stereo, 3 mono.  Returns the stream bytes, or (bytes, integer spectra [frame][gr][ch][576],
    side info [frame][gr][ch] dicts) with spectra=True."""
    opts = dict(opts or {})
    rng = np.random.default_rng(seed)
    nch = 1 if mode == 3 else 2
    hdr_len = 4 + (2 if crc else 0) + (32 if nch == 2 else 17)
    frames = []
    spec = np.zeros((n_frames, 2, 2, 576), np.int32)
    stale_t2 = [[0, 0], [0, 0]]   # table_select[gr][ch][2] as the reference's persistent side-info object holds it (A.D3)
    R = 0                         # bytes of reservoir in front of the next frame (its main_data_begin)
    payload = []
    for f in range(n_frames):
        br = int(rng.choice(vbr)) if vbr else bitrate
        pad = int(rng.integers(0, 2)) if opts.get("padding") else 0
        size = 144000 * br // sr + pad
        cap = size - hdr_len
        scfsi = [[int(rng.integers(0, 2)) if opts.get("scfsi", True) else 0 for _ in range(4)] for _ in range(nch)]
        o = dict(opts)
        while True:   # shrink the granules until the frame's main data fits the reservoir + its own payload area
            grs = [[None] * nch for _ in range(2)]
            md = Bits()
            st = [row[:] for row in stale_t2]
            for gr in range(2):
                for ch in range(nch):
                    o["_stale_t2"] = st[gr][ch]
                    si, w, sp = make_granule(rng, sr, gr, ch, o, scfsi)
                    if not si["window_switching"]:
                        st[gr][ch] = si["table_select"][2]
                    grs[gr][ch] = si
                    md.extend(w)
                    spec[f, gr, ch] = sp
            mdb = md.tobytes()
            if len(mdb) <= R + cap:
                break
            o["max_bv"] = max(4, int(o.get("max_bv", 200) * 0.8))
            o["max_quads"] = max(2, int(o.get("max_quads", 60) * 0.8))
            for k in ("bv_full", "quads_end", "fill"):
                if o.get(k):
                    o[k] *= 0.5
        stale_t2 = st
        M = len(mdb)
        if reservoir:
            extra = max(0, R + cap - 511 - M)
            if rng.random() < 0.25:   # sometimes drain the reservoir completely
                extra = R + cap - M
        else:
            extra = R + cap - M
        frames.append(dict(bitrate=br, pad=pad, size=size, scfsi=scfsi, gr=grs, cap=cap, main_data_begin=R))
        payload.append(mdb + b"\x00" * extra)   # ancillary / padding bytes after the last granule: ignored by the decoder
        R = R + cap - M - extra
        assert 0 <= R <= 511
    payload = b"".join(payload)
    out = []
    pos = 0
    for fr in frames:
        h = Bits()
        h.put(0x7FF, 11)
        h.put(3, 2)
        h.put(1, 2)
        h.put(0 if crc else 1, 1)
        h.put(BITRATES.index(fr["bitrate"]), 4)
        h.put(SR_CODE[sr], 2)
        h.put(fr["pad"], 1)
        h.put(0, 1)
        h.put(mode, 2)
        h.put(mode_ext, 2)
        h.put(0, 1)
        h.put(1, 1)
        h.put(0, 2)
        out.append(h.tobytes() + (b"\xAB\xCD" if crc else b"") + side_info_bits(fr, nch))
        chunk = payload[pos:pos + fr["cap"]]
        out.append(chunk + b"\x00" * (fr["cap"] - len(chunk)))
        pos += fr["cap"]
    out = b"".join(out)
    if spectra:
        return out, spec, [fr["gr"] for fr in frames]
    return out


STREAMS = {
    # name: kwargs
    "long_alltables": dict(seed=1, n_frames=8, bitrate=192, opts=dict(max_bv=140, stuff_ones=True)),
    "reservoir": dict(seed=2, n_frames=12, bitrate=128, reservoir=True, opts=dict(max_bv=110, max_quads=40)),
    "short_mixed": dict(seed=3, n_frames=10, bitrate=192, opts=dict(switching=True, max_bv=130)),
    "ms_stereo": dict(seed=4, n_frames=8, bitrate=160, mode=1, mode_ext=3, reservoir=True, opts=dict(switching=True, max_bv=110)),
    "is_only_bit": dict(seed=5, n_frames=4, bitrate=160, mode=1, mode_ext=1, opts=dict(max_bv=110)),
    "mono_crc_48k": dict(seed=6, n_frames=8, sr=48000, bitrate=96, mode=3, crc=True, reservoir=True, opts=dict(switching=True, max_bv=120)),
    "vbr_32k_pad": dict(seed=7, n_frames=10, sr=32000, vbr=[96, 128, 160, 320], reservoir=True, opts=dict(padding=True, max_bv=90, switching=True)),
    "loud_wrap": dict(seed=8, n_frames=4, bitrate=320, opts=dict(max_bv=200, amp=15, gain_lo=175, gain_hi=190, scalefac=False)),
}


def fuzz_config(seed):
    """A random combination of everything the writer can vary (BASELINE configs[3] as a corpus rather than eight hand-picked
    streams): sample rate, CBR / VBR, padding, mono / stereo / joint stereo with either mode-extension bit, CRC, bit reservoir,
    window switching with short / mixed / start / stop blocks, scalefactors + scfsi, loud spectra."""
    rng = np.random.default_rng(1000 + seed)
    sr = int(rng.choice([44100, 48000, 32000]))
    mode = 3 if seed % 5 == 2 else int(rng.choice([0, 0, 1, 1]))   # every fifth stream is mono (17-byte side info)
    kw = dict(seed=seed, n_frames=int(rng.integers(16, 29)), sr=sr, mode=mode, mode_ext=int(rng.integers(0, 4)) if mode == 1 else 0,
              crc=bool(rng.integers(0, 2)), reservoir=bool(rng.integers(0, 2)))
    rates = [64, 96, 128, 160, 192, 256, 320] if mode != 3 else [48, 64, 96, 128, 160]
    if rng.random() < 0.3:
        kw["vbr"] = [int(v) for v in rng.choice(rates, size=3, replace=False)]
    else:
        kw["bitrate"] = int(rng.choice(rates))
    lo = min(kw.get("vbr", [kw.get("bitrate", 128)]))
    opts = dict(switching=bool(rng.random() < 0.7), padding=bool(rng.integers(0, 2)), scfsi=bool(rng.random() < 0.8),
                stuff_ones=bool(rng.integers(0, 2)), max_bv=int(min(200, 40 + lo * (2 if mode == 3 else 1) // 2)),
                max_quads=int(rng.integers(10, 61)))
    if rng.random() < 0.2:
        opts.update(amp=15, gain_lo=170, gain_hi=186)
    kw["opts"] = opts
    return kw


N_FUZZ = 16

# books with linbits >= 8 reach |x| >= 256 (21-23, 28-31); 23 and 31 (13 linbits) reach 8206
_LOUD_BOOKS = [21, 22, 23, 23, 28, 29, 30, 31, 31, 16, 24, 13, 15, 7, 1]


def extreme_config(seed):
    """fuzz_config's variety plus the edges of the decoder's domain: linbits magnitudes up to 8206 (254..258 often), global_gain
    over 0..255 with both ends drawn on purpose, subblock_gain 0..7, big_values up to 288, count1 running to the stop at 572, and
    -- at 320 kbps / 32 kHz -- granules with part2_3_length near 4095."""
    rng = np.random.default_rng(50000 + seed)
    fill = seed % 4 == 0                                             # every fourth stream: 320 kbps at 32 kHz, long granules
    sr = 32000 if fill else int(rng.choice([44100, 48000, 32000]))
    mode = 3 if seed % 5 == 2 else int(rng.choice([0, 1, 1]))
    kw = dict(seed=70000 + seed, n_frames=int(rng.integers(12, 29)), sr=sr, mode=mode,
              mode_ext=int(rng.integers(0, 4)) if mode == 1 else 0, crc=bool(rng.integers(0, 2)),
              reservoir=bool(fill or rng.integers(0, 2)))
    rates = [96, 128, 160, 192, 256, 320] if mode != 3 else [64, 96, 128, 160, 320]
    if fill:
        kw["bitrate"] = 320
    elif rng.random() < 0.3:
        kw["vbr"] = [int(v) for v in rng.choice(rates, size=3, replace=False)]
    else:
        kw["bitrate"] = int(rng.choice(rates))
    gains = [(0, 256), (0, 256), (90, 200), (120, 175)][int(rng.integers(0, 4))]
    opts = dict(switching=bool(rng.random() < 0.7), padding=bool(rng.integers(0, 2)), scfsi=bool(rng.random() < 0.8),
                stuff_ones=bool(rng.integers(0, 2)), max_bv=288, max_quads=int(rng.integers(20, 144)),
                tables=_LOUD_BOOKS, gain_lo=gains[0], gain_hi=gains[1], gain_edge=0.04, sbg_hi=8,
                big_lin=float(rng.choice([0.02, 0.08, 0.3])), bv_full=0.15, quads_end=0.35, amp=int(rng.choice([6, 12, 15])),
                scalefac=bool(rng.random() < 0.8))
    if fill:
        opts.update(quads_end=0.8, fill=0.7 if mode == 3 else 0.35)
    kw["opts"] = opts
    return kw


N_EXTREME = 150
