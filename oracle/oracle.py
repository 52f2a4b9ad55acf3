"""ctypes binding of the CPU oracle (oracle/mp3stego_oracle.c).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
--impl reference legs.  The product package never imports this module.
"""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libmp3stego_oracle.so")


class _DecResult(ctypes.Structure):
    _fields_ = [("n_frames", ctypes.c_int64), ("n_pcm_rows", ctypes.c_int64),
                ("channels", ctypes.c_int), ("sampling_rate", ctypes.c_int), ("bit_rate", ctypes.c_int),
                ("status", ctypes.c_int),
                ("pcm", ctypes.POINTER(ctypes.c_double)), ("spectra", ctypes.POINTER(ctypes.c_int32)),
                ("tables", ctypes.POINTER(ctypes.c_uint8)), ("bits", ctypes.c_char_p), ("n_bits", ctypes.c_int64),
                ("side", ctypes.POINTER(ctypes.c_int32)), ("frame_off", ctypes.POINTER(ctypes.c_int64)),
                ("frame_mdb", ctypes.POINTER(ctypes.c_int32)), ("xr", ctypes.POINTER(ctypes.c_double))]


class _EncResult(ctypes.Structure):
    _fields_ = [("data", ctypes.POINTER(ctypes.c_uint8)), ("n_bytes", ctypes.c_int64), ("n_frames", ctypes.c_int64),
                ("hide_str_offset", ctypes.c_int64),
                ("mdct", ctypes.POINTER(ctypes.c_int32)), ("ix", ctypes.POINTER(ctypes.c_int32)),
                ("info", ctypes.POINTER(ctypes.c_int32)), ("scfsi", ctypes.POINTER(ctypes.c_int32)),
                ("status", ctypes.c_int)]


def build(force=False):
    if force or not os.path.exists(_LIB_PATH) or \
            os.path.getmtime(_LIB_PATH) < os.path.getmtime(os.path.join(_HERE, "mp3stego_oracle.c")):
        subprocess.check_call(["make", "-C", _HERE, "-s"])
    return _LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = ctypes.CDLL(_LIB_PATH)
        L.ora_decode.restype = ctypes.POINTER(_DecResult)
        L.ora_decode.argtypes = [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64, ctypes.c_int]
        L.ora_dec_free.argtypes = [ctypes.POINTER(_DecResult)]
        L.ora_encode.restype = ctypes.POINTER(_EncResult)
        L.ora_encode.argtypes = [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64, ctypes.c_int, ctypes.c_int,
                                 ctypes.c_int, ctypes.c_char_p, ctypes.c_int64, ctypes.c_int]
        L.ora_enc_free.argtypes = [ctypes.POINTER(_EncResult)]
        L.ora_pcm_to_int16.argtypes = [ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p]
        L.ora_side_fields.restype = ctypes.c_int
        L.ora_enc_fields.restype = ctypes.c_int
        _lib = L
    return _lib


def id3_offset(data: bytes) -> int:
    """Audio start as Decoder.__init__ computes it (decoder/decoder.py:29-33, ID3_Parser.py:106-125)."""
    if len(data) >= 10 and data[0:3] == b"ID3":
        # ID3_Parser.py:129-135: the low four flag bits must be clear, else the tag is ignored (offset 0);
        # offset = 10 + synchsafe size (+10 more with a footer, flag bit 0x10)
        if data[5] & 0x0F:
            return 0
        size = 0
        for i in range(4):
            size = (size << 7) + data[6 + i]
        off = size + 10
        if data[5] & 0x10:
            off += 10
        return off
    return 0


def _arr(ptr, shape, dtype):
    n = int(np.prod(shape))
    if n == 0 or not ptr:
        return np.zeros(shape, dtype=dtype)
    return np.ctypeslib.as_array(ptr, shape=(n,)).astype(dtype, copy=True).reshape(shape)


def decode(data: bytes, offset: int = 0, taps: bool = True) -> dict:
    """Decode one MP3 byte string the way MP3Parser.parse_file does (MP3_Parser.py:57-85)."""
    L = lib()
    buf = (ctypes.c_uint8 * max(len(data), 1)).from_buffer_copy(data if len(data) else b"\0")
    rp = L.ora_decode(ctypes.addressof(buf), len(data), offset, 1 if taps else 0)
    r = rp.contents
    nf, rows, ch = r.n_frames, r.n_pcm_rows, max(r.channels, 1)
    out = dict(n_frames=nf, channels=r.channels, sampling_rate=r.sampling_rate, bit_rate=r.bit_rate,
               status=r.status,
               pcm=_arr(r.pcm, (rows, ch), np.float64),
               tables=_arr(r.tables, (nf, 12), np.uint8),
               bits=(r.bits or b"").decode("ascii"),
               frame_off=_arr(r.frame_off, (nf,), np.int64),
               main_data_begin=_arr(r.frame_mdb, (nf,), np.int32))
    if taps:
        out["spectra"] = _arr(r.spectra, (nf, 2, 2, 576), np.int32)
        out["side"] = _arr(r.side, (nf, 2, 2, L.ora_side_fields()), np.int32)
        out["xr"] = _arr(r.xr, (nf, 2, 2, 576), np.float64)
    pcm16 = np.zeros(out["pcm"].shape, dtype=np.int16)
    if out["pcm"].size:
        src = np.ascontiguousarray(out["pcm"])
        L.ora_pcm_to_int16(src.ctypes.data, src.size, pcm16.ctypes.data)
    out["pcm16"] = pcm16
    L.ora_dec_free(rp)
    return out


def encode(pcm: np.ndarray, samplerate: int = 44100, bitrate: int = 320, hide_bits: str = "",
           taps: bool = True) -> dict:
    """Encode interleaved int16 stereo PCM [n, 2] the way MP3Encoder.encode does (MP3_Encoder.py:596-621).
    status -3: a granule's step search ran past the step table (SURVEY A.E13); no bytes, n_frames = the frame it happened in."""
    L = lib()
    pcm = np.ascontiguousarray(pcm, dtype=np.int16)
    nch = pcm.shape[1] if pcm.ndim == 2 else 1
    n = pcm.shape[0]
    hb = hide_bits.encode("ascii")
    rp = L.ora_encode(pcm.ctypes.data, pcm.size, n, nch, samplerate, bitrate, hb, len(hb), 1 if taps else 0)
    r = rp.contents
    nf = r.n_frames
    out = dict(status=r.status, n_frames=nf, hide_str_offset=r.hide_str_offset,
               mp3=_arr(r.data, (r.n_bytes,), np.uint8).tobytes())
    if taps and r.status == 0:
        out["mdct"] = _arr(r.mdct, (nf, 2, 2, 576), np.int32)   # [frame][ch][gr]
        out["ix"] = _arr(r.ix, (nf, 2, 2, 576), np.int32)       # [frame][ch][gr]
        out["info"] = _arr(r.info, (nf, 2, 2, L.ora_enc_fields()), np.int32)  # [frame][gr][ch]
        out["scfsi"] = _arr(r.scfsi, (nf, 2, 4), np.int32)
    L.ora_enc_free(rp)
    return out


def str_to_bits(s: str) -> str:
    """steganography.py:10-24: utf-8 bytes, MSB first."""
    return "".join(format(b, "08b") for b in s.encode("utf-8"))


def reveal_parse(bits: str) -> str:
    """decoder/decoder.py:86-105 restated: 8-bit groups -> chars, '<len>#' prefix, slice."""
    s = "".join(chr(int(bits[i:i + 8], 2)) for i in range(0, len(bits) - len(bits) % 8, 8))
    ln = ""
    for c in s:
        if c == "#":
            break
        ln += c
    try:
        n = int(ln)
    except Exception:
        n = 0
        ln = ""
    if len(ln) + 1 + n > len(s):
        return s[len(ln) + 1:]
    return s[len(ln) + 1: len(ln) + 1 + n]
