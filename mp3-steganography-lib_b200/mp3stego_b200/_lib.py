"""ctypes binding of libmp3stego_b200.so (include/mp3stego_b200.h) plus the batch entry points.

There is no CPU fallback: importing this module without the built library, or creating a handle
without an sm_100 GPU, raises.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("M3S_LIB_PATH") or os.path.join(os.path.dirname(_HERE), "lib", "libmp3stego_b200.so")   # (override: A/B builds)

M3S_MEM_HOST, M3S_MEM_DEVICE = 0, 1
M3S_FILE_NO_SYNC, M3S_FILE_UNSUPPORTED, M3S_FILE_TRAILING_JUNK, M3S_FILE_STATE_CARRY = 1, 2, 4, 8
M3S_FILE_CHANNEL_SWITCH, M3S_FILE_BAD_SIDEINFO = 16, 32


def raise_for_status(status: int, what: str = "file"):
    """Re-raise what the reference raises for a file the scan flagged (MP3Parser / Frame): IndexError for headers or side info
    outside its tables, ValueError for a channel-count change inside one file.  NO_SYNC is the caller's business (the reference
    parser is then merely 'not valid' and parses nothing)."""
    if status & M3S_FILE_UNSUPPORTED:
        raise IndexError(f"{what}: frame header outside MPEG-1 Layer III (the reference raises while parsing it)")
    if status & M3S_FILE_BAD_SIDEINFO:
        raise IndexError(f"{what}: big_values / region counts outside the band tables (Frame.py:461-478 raises IndexError)")
    if status & M3S_FILE_CHANNEL_SWITCH:
        raise ValueError(f"{what}: mono and stereo frames in one file (MP3_Parser.py:83: setting an array element with a sequence)")
M3S_ERR_ARG = -2
STEP_TABLE_OVERRUN = "runs past the end of the step table"   # in m3s_encode's error text for such a clip
M3S_DEC_PCM_FLOAT = 1
M3S_DEC_EXACT = 2

_c_i64p = ctypes.POINTER(ctypes.c_int64)
_c_i32p = ctypes.POINTER(ctypes.c_int32)

# every symbol include/mp3stego_b200.h declares: (name, restype, argtypes)
SYMBOLS = [
    ("m3s_create", ctypes.c_int, [ctypes.c_int, ctypes.POINTER(ctypes.c_void_p)]),
    ("m3s_destroy", ctypes.c_int, [ctypes.c_void_p]),
    ("m3s_last_error", ctypes.c_char_p, [ctypes.c_void_p]),
    ("m3s_set_stream", ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p]),
    ("m3s_synchronize", ctypes.c_int, [ctypes.c_void_p]),
    ("m3s_launch_count", ctypes.c_int64, [ctypes.c_void_p]),
    ("m3s_version", ctypes.c_int, []),
    ("m3s_decode_scan", ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, _c_i64p, _c_i64p, ctypes.c_int32,
                                       _c_i64p, _c_i64p, _c_i32p, _c_i32p, _c_i32p, _c_i32p]),
    ("m3s_decode_frame_pos", ctypes.c_int, [ctypes.c_void_p, _c_i64p]),
    ("m3s_decode_reveal", ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, _c_i64p]),
    ("m3s_decode_run", ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, _c_i64p, ctypes.c_void_p,
                                      ctypes.c_uint32]),
    ("m3s_decode_run_range", ctypes.c_int, [ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int,
                                            _c_i64p, ctypes.c_uint32]),
    ("m3s_decode", ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, _c_i64p, _c_i64p, ctypes.c_int32, ctypes.c_void_p,
                                  ctypes.c_int64, _c_i64p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, _c_i64p, _c_i64p, _c_i32p,
                                  _c_i32p, _c_i32p, _c_i32p, ctypes.c_uint32]),
    ("m3s_decode_bound", ctypes.c_int64, [ctypes.c_void_p, _c_i64p, _c_i64p, ctypes.c_int32, _c_i64p]),
    ("m3s_encode_bound", ctypes.c_int64, [ctypes.c_int64, ctypes.c_int32, ctypes.c_int32]),
    ("m3s_encode_size", ctypes.c_int64, [ctypes.c_int64, ctypes.c_int32, ctypes.c_int32]),
    ("m3s_encode", ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, _c_i64p, _c_i64p, ctypes.c_int32,
                                  ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p, _c_i64p, ctypes.c_void_p, _c_i64p,
                                  _c_i64p, _c_i64p, _c_i64p]),
    ("m3s_encode_mixed", ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, _c_i64p, _c_i64p, ctypes.c_int32,
                                        _c_i32p, _c_i32p, ctypes.c_void_p, _c_i64p, ctypes.c_void_p, _c_i64p,
                                        _c_i64p, _c_i64p, _c_i64p]),
    ("m3s_encode_offsets", ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, _c_i64p, _c_i64p, ctypes.c_int32,
                                          _c_i32p, _c_i32p, ctypes.c_void_p, _c_i64p, _c_i64p, ctypes.c_void_p, _c_i64p, _c_i64p,
                                          _c_i64p]),
    ("m3s_encode_taps", ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                       ctypes.c_void_p]),
    ("m3s_table_export", ctypes.c_int64, [ctypes.c_int, ctypes.c_void_p, ctypes.c_int64]),
    ("m3s_timing_enable", ctypes.c_int, [ctypes.c_void_p, ctypes.c_int]),
    ("m3s_timing_get", ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(ctypes.c_double), _c_i64p]),
    ("m3s_kernel_name", ctypes.c_char_p, [ctypes.c_int]),
]
M3S_K_COUNT = 13

_lib = None


class M3SError(RuntimeError):
    pass


def load():
    """Load the shared library (once).  Raises M3SError when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise M3SError(f"{LIB_PATH} is missing: build it with `python __graft_entry__.py` "
                           "(nvcc, sm_100a). There is no CPU fallback.")
        L = ctypes.CDLL(LIB_PATH)
        for name, res, args in SYMBOLS:
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def _i64(a):
    a = np.ascontiguousarray(a, dtype=np.int64)
    return a, a.ctypes.data_as(_c_i64p)


def _ptr(x):
    """Raw address of a numpy array / torch tensor / int / None."""
    if x is None:
        return None
    if isinstance(x, int):
        return ctypes.c_void_p(x)
    if isinstance(x, np.ndarray):
        return ctypes.c_void_p(x.ctypes.data)
    if hasattr(x, "data_ptr"):
        return ctypes.c_void_p(x.data_ptr())
    raise TypeError(type(x))


def _ready(*xs):
    """The library works on its own CUDA stream and does not know the caller's: make sure whatever torch queued on ITS current
    stream for these device tensors (the kernel that produced an input, the fill of a freshly allocated output) has finished
    before the library touches them.  Host arrays and None pass through."""
    done = set()
    for x in xs:
        if x is not None and getattr(x, "is_cuda", False) and x.device not in done:
            import torch
            torch.cuda.current_stream(x.device).synchronize()
            done.add(x.device)


def _mem_of(x):
    if hasattr(x, "is_cuda"):
        return M3S_MEM_DEVICE if x.is_cuda else M3S_MEM_HOST
    return M3S_MEM_HOST


class Handle:
    """One CUDA stream + grow-only device workspaces (m3s_handle_t)."""

    def __init__(self, device: int = 0):
        self._L = load()
        h = ctypes.c_void_p()
        rc = self._L.m3s_create(device, ctypes.byref(h))
        if rc != 0:
            raise M3SError(f"m3s_create(device={device}) failed with {rc}: no sm_100 CUDA device "
                           "(this library has no CPU fallback)")
        self._h = h
        self.device = device

    def close(self):
        if getattr(self, "_h", None):
            self._L.m3s_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            raise M3SError(f"{what} failed ({rc}): {self._L.m3s_last_error(self._h).decode()}")

    def set_stream(self, stream_ptr):
        self._check(self._L.m3s_set_stream(self._h, ctypes.c_void_p(stream_ptr) if stream_ptr else None), "m3s_set_stream")

    def synchronize(self):
        self._check(self._L.m3s_synchronize(self._h), "m3s_synchronize")

    @property
    def launches(self) -> int:
        return int(self._L.m3s_launch_count(self._h))

    def timing_enable(self, on=True):
        self._check(self._L.m3s_timing_enable(self._h, 1 if on else 0), "m3s_timing_enable")

    def timing(self):
        """{kernel name: (device ms accumulated, launches)} since the last timing_enable()."""
        out = {}
        for k in range(M3S_K_COUNT):
            ms, n = ctypes.c_double(0), ctypes.c_int64(0)
            self._check(self._L.m3s_timing_get(self._h, k, ctypes.byref(ms), ctypes.byref(n)), "m3s_timing_get")
            if n.value:
                out[self._L.m3s_kernel_name(k).decode()] = (ms.value, n.value)
        return out

    # ------------------------------------------------------------------ decode
    def decode_scan(self, data, file_off, audio_start=None):
        """D0 + D4 over a batch.  `data`: uint8 numpy array / torch tensor (host or cuda) of all files end to end."""
        n = len(file_off) - 1
        fo, fo_p = _i64(file_off)
        if audio_start is not None:
            au, au_p = _i64(audio_start)
        else:
            au, au_p = None, None
        out = dict(n_frames=np.zeros(n, np.int64), pcm_rows=np.zeros(n, np.int64), sample_rate=np.zeros(n, np.int32),
                   channels=np.zeros(n, np.int32), bitrate=np.zeros(n, np.int32), status=np.zeros(n, np.int32))
        self._keep = (data, fo, au)
        _ready(data)
        rc = self._L.m3s_decode_scan(self._h, _ptr(data), _mem_of(data), fo_p, au_p, n,
                                     out["n_frames"].ctypes.data_as(_c_i64p), out["pcm_rows"].ctypes.data_as(_c_i64p),
                                     out["sample_rate"].ctypes.data_as(_c_i32p), out["channels"].ctypes.data_as(_c_i32p),
                                     out["bitrate"].ctypes.data_as(_c_i32p), out["status"].ctypes.data_as(_c_i32p))
        self._check(rc, "m3s_decode_scan")
        self._scan = out
        return out

    def decode_frame_pos(self):
        """File-relative byte position of every frame of the last scan (all files' frames back to back)."""
        total = int(self._scan["n_frames"].sum())
        pos = np.zeros(max(total, 1), np.int64)
        self._check(self._L.m3s_decode_frame_pos(self._h, pos.ctypes.data_as(_c_i64p)), "m3s_decode_frame_pos")
        return pos[:total]

    def decode_reveal(self):
        """Table ids [frames, 12] and the per-file reveal bit strings of the last scan."""
        sc = self._scan
        total = int(sc["n_frames"].sum())
        ids = np.zeros((max(total, 1), 12), np.uint8)
        bits = np.zeros(max(total, 1) * 12, np.uint8)
        ln = np.zeros(len(sc["n_frames"]), np.int64)
        rc = self._L.m3s_decode_reveal(self._h, _ptr(ids), _ptr(bits), M3S_MEM_HOST, ln.ctypes.data_as(_c_i64p))
        self._check(rc, "m3s_decode_reveal")
        base = np.concatenate([[0], np.cumsum(sc["n_frames"])])
        strings = [bits[12 * base[i]: 12 * base[i] + ln[i]].tobytes().decode("ascii") for i in range(len(ln))]
        return ids[:total], strings

    def decode_reveal_into(self, table_ids, reveal_bits):
        """Like decode_reveal but into caller buffers (numpy / torch, host or cuda; either may be None).
        Returns the per-file reveal string lengths; file i's chars start at 12 * (frames of files < i)."""
        ln = np.zeros(len(self._scan["n_frames"]), np.int64)
        mem = _mem_of(table_ids if table_ids is not None else reveal_bits)
        _ready(table_ids, reveal_bits)
        rc = self._L.m3s_decode_reveal(self._h, _ptr(table_ids), _ptr(reveal_bits), mem, ln.ctypes.data_as(_c_i64p))
        self._check(rc, "m3s_decode_reveal")
        return ln

    def decode_run(self, pcm=None, pcm_off=None, spectra=False, as_float=False, exact=False):
        """D1-D3 of the last scan.  With pcm=None a host numpy buffer is allocated and returned."""
        sc = self._scan
        elems = sc["pcm_rows"] * np.maximum(sc["channels"], 1)
        total = int(elems.sum())
        total_frames = int(sc["n_frames"].sum())
        if pcm is None:
            pcm = np.zeros(max(total, 1), np.float32 if as_float else np.int16)
        po, po_p = (None, None) if pcm_off is None else _i64(pcm_off)
        sp = None
        if spectra is True:
            sp = np.zeros((max(total_frames, 1), 2, 2, 576), np.int16)
        elif spectra is not False and spectra is not None:
            sp = spectra
        _ready(pcm, sp)
        rc = self._L.m3s_decode_run(self._h, _ptr(pcm), _mem_of(pcm), po_p, _ptr(sp),
                                    (M3S_DEC_PCM_FLOAT if as_float else 0) | (M3S_DEC_EXACT if exact else 0))
        self._check(rc, "m3s_decode_run")
        return pcm, sp

    def decode_run_range(self, file_index, first, count, pcm=None, as_float=False, exact=False):
        """D1-D3 of frames [first, first + count) of one file of the last scan (m3s_decode_run_range).  Returns (pcm, rows)."""
        ch = max(int(self._scan["channels"][file_index]), 1)
        if pcm is None:
            pcm = np.zeros((count + 1) * 1152 * ch, np.float32 if as_float else np.int16)
        rows = ctypes.c_int64(0)
        _ready(pcm)
        rc = self._L.m3s_decode_run_range(self._h, file_index, first, count, _ptr(pcm), _mem_of(pcm), ctypes.byref(rows),
                                          (M3S_DEC_PCM_FLOAT if as_float else 0) | (M3S_DEC_EXACT if exact else 0))
        self._check(rc, "m3s_decode_run_range")
        return pcm, int(rows.value)

    def decode(self, data, file_off, audio_start=None, pcm=None, table_ids=None, reveal_bits=None, as_float=False, exact=False,
               frames_bound=None):
        """m3s_decode: decode + reveal of a whole batch in ONE self-pipelining call (MP3Parser.parse_file + write_to_wav's int16
        conversion for every file).  `data`: uint8 numpy / torch tensor (host or cuda) of all files end to end.  Output buffers
        (numpy or torch, same side as `data`) are allocated when None -- for host input sized by m3s_decode_bound, for device
        input `pcm` / `frames_bound` must be given.  Returns a dict: per-file arrays n_frames, pcm_rows, sample_rate, channels,
        bitrate, status, reveal_len, pcm_off [n+1] (elements) and the buffers pcm, table_ids, reveal_bits."""
        n = len(file_off) - 1
        fo, fo_p = _i64(file_off)
        au, au_p = (None, None) if audio_start is None else _i64(audio_start)
        mem = _mem_of(data)
        if frames_bound is None:
            if mem == M3S_MEM_DEVICE:
                raise M3SError("decode: device-resident input needs frames_bound (and pcm)")
            fb = ctypes.c_int64(0)
            if self._L.m3s_decode_bound(_ptr(data), fo_p, au_p, n, ctypes.byref(fb)) < 0:
                raise M3SError("m3s_decode_bound failed")
            frames_bound = int(fb.value)
        frames_bound = max(int(frames_bound), 1)
        if mem == M3S_MEM_DEVICE:
            import torch
            mk = lambda cnt, dt: torch.empty(cnt, dtype=dt, device=data.device)   # noqa: E731
            u8, pdt = torch.uint8, (torch.float32 if as_float else torch.int16)
        else:
            mk = lambda cnt, dt: np.empty(cnt, dt)   # noqa: E731
            u8, pdt = np.uint8, (np.float32 if as_float else np.int16)
        if pcm is None:
            pcm = mk(frames_bound * 1152 * 2, pdt)
        if table_ids is None:
            table_ids = mk(frames_bound * 12, u8)
        if reveal_bits is None:
            reveal_bits = mk(frames_bound * 12, u8)
        cap = int(pcm.numel() if hasattr(pcm, "numel") else pcm.size)
        fcap = min(int(t.numel() if hasattr(t, "numel") else t.size) for t in (table_ids, reveal_bits)) // 12
        out = dict(n_frames=np.zeros(n, np.int64), sample_rate=np.zeros(n, np.int32), channels=np.zeros(n, np.int32),
                   bitrate=np.zeros(n, np.int32), status=np.zeros(n, np.int32), reveal_len=np.zeros(n, np.int64),
                   pcm_off=np.zeros(n + 1, np.int64))
        self._keep = (data, fo, au)
        _ready(data, pcm, table_ids, reveal_bits)
        rc = self._L.m3s_decode(self._h, _ptr(data), mem, fo_p, au_p, n, _ptr(pcm), cap, out["pcm_off"].ctypes.data_as(_c_i64p),
                                _ptr(table_ids), _ptr(reveal_bits), fcap, out["reveal_len"].ctypes.data_as(_c_i64p),
                                out["n_frames"].ctypes.data_as(_c_i64p), out["sample_rate"].ctypes.data_as(_c_i32p),
                                out["channels"].ctypes.data_as(_c_i32p), out["bitrate"].ctypes.data_as(_c_i32p),
                                out["status"].ctypes.data_as(_c_i32p), (M3S_DEC_PCM_FLOAT if as_float else 0) | (M3S_DEC_EXACT if exact else 0))
        self._check(rc, "m3s_decode")
        out["pcm_rows"] = np.diff(out["pcm_off"]) // np.maximum(out["channels"], 1)
        out.update(pcm=pcm, table_ids=table_ids, reveal_bits=reveal_bits)
        return out

    def reveal_strings(self, res):
        """Per-file reveal bit strings ('0'/'1') of a decode() result with host buffers."""
        base = np.concatenate([[0], np.cumsum(res["n_frames"])])
        bits = res["reveal_bits"]
        return [bytes(bits[12 * base[i]: 12 * base[i] + int(res["reveal_len"][i])]).decode("ascii") for i in range(len(res["n_frames"]))]

    # ------------------------------------------------------------------ encode
    def encode(self, pcm, n_samples, sample_rate, bitrate_kbps, payloads=None, pcm_off=None, mp3_out=None, taps=False,
               compact=False, payload_packed=None):
        """E1-E3 over a batch of int16 stereo clips laid end to end in `pcm` (numpy or torch, host or cuda).
        sample_rate and bitrate_kbps are ints (one rate pair for the batch, m3s_encode) or sequences with one entry per clip
        (m3s_encode_mixed: clips of different rates in one call).
        compact=True lays the MP3s back to back at their exact sizes (m3s_encode_size at each clip's pair), so that
        (mp3, mp3_off + [end]) can be fed straight to decode_scan.  payload_packed = (uint8 array of '0'/'1' chars, offsets[n+1])
        avoids re-joining.  Raises IndexError, for the whole batch, when a clip drives the rate loop past the end of the step table."""
        L = self._L
        n = len(n_samples)
        ns, ns_p = _i64(n_samples)
        if pcm_off is None:
            pcm_off = np.concatenate([[0], np.cumsum(ns * 2)])[:-1]
        po, po_p = _i64(pcm_off)
        mixed = not (np.isscalar(sample_rate) and np.isscalar(bitrate_kbps))
        if mixed:
            srs = np.ascontiguousarray(np.broadcast_to(np.asarray(sample_rate, np.int32), (n,)))
            brs = np.ascontiguousarray(np.broadcast_to(np.asarray(bitrate_kbps, np.int32), (n,)))
            keys = list(zip(ns.tolist(), srs.tolist(), brs.tolist()))
        else:
            keys = [(int(s), sample_rate, bitrate_kbps) for s in ns]
        size_fn = L.m3s_encode_size if compact else L.m3s_encode_bound
        uniq = {k: size_fn(*k) for k in set(keys)}
        bounds = np.array([uniq[k] for k in keys], np.int64)
        if (bounds < 0).any():
            raise M3SError(f"encode: clip {int(np.argmax(bounds < 0))}: unsupported sample count / sample rate / bitrate")
        mo, mo_p = _i64(np.concatenate([[0], np.cumsum(bounds)])[:-1])
        mc, mc_p = _i64(bounds)
        mem = _mem_of(pcm)
        if mp3_out is None:
            if mem == M3S_MEM_DEVICE:
                import torch
                mp3_out = torch.zeros(int(bounds.sum()) + 16, dtype=torch.uint8, device=pcm.device)   # (its fill is awaited below)
            else:
                mp3_out = np.zeros(int(bounds.sum()) + 16, np.uint8)
        if payload_packed is not None:
            pl = payload_packed[0]
            ploff, ploff_p = _i64(payload_packed[1])
            pl_p = _ptr(pl)
        elif payloads is not None and any(len(p) for p in payloads):
            pl = np.frombuffer("".join(payloads).encode("ascii"), dtype=np.uint8).copy()
            ploff, ploff_p = _i64(np.concatenate([[0], np.cumsum([len(p) for p in payloads])]))
            pl_p = _ptr(pl)
        else:
            pl, ploff, ploff_p, pl_p = None, None, None, None
        out_len = np.zeros(n, np.int64)
        hoff = np.zeros(n, np.int64)
        _ready(pcm, mp3_out)
        if mixed:
            rc = L.m3s_encode_mixed(self._h, _ptr(pcm), mem, po_p, ns_p, n, srs.ctypes.data_as(_c_i32p), brs.ctypes.data_as(_c_i32p),
                                    pl_p, ploff_p, _ptr(mp3_out), mo_p, mc_p, out_len.ctypes.data_as(_c_i64p),
                                    hoff.ctypes.data_as(_c_i64p))
        else:
            rc = L.m3s_encode(self._h, _ptr(pcm), mem, po_p, ns_p, n, sample_rate, bitrate_kbps, pl_p, ploff_p, _ptr(mp3_out),
                              mo_p, mc_p, out_len.ctypes.data_as(_c_i64p), hoff.ctypes.data_as(_c_i64p))
        if rc == M3S_ERR_ARG:
            msg = L.m3s_last_error(self._h).decode()
            if STEP_TABLE_OVERRUN in msg:
                # the reference's quantize() indexes its step table past the end for this input (SURVEY A.E13): no output
                raise IndexError(f"index out of bounds: {msg}")
        self._check(rc, "m3s_encode_mixed" if mixed else "m3s_encode")
        res = dict(mp3=mp3_out, mp3_off=mo, out_len=out_len, hide_str_offset=hoff)
        if taps:
            nf = int((ns // 1152).sum())
            res["mdct"] = np.zeros((nf, 2, 2, 576), np.int32)
            res["ix"] = np.zeros((nf, 2, 2, 576), np.int32)
            res["info"] = np.zeros((nf, 2, 2, 16), np.int32)
            res["scfsi"] = np.zeros((nf, 2, 4), np.int32)
            self._check(L.m3s_encode_taps(self._h, _ptr(res["mdct"]), _ptr(res["ix"]), _ptr(res["info"]), _ptr(res["scfsi"])),
                        "m3s_encode_taps")
        return res

    def encode_offsets(self, pcm, n_samples, sample_rate, bitrate_kbps, bodies, candidates, pcm_off=None):
        """m3s_encode_offsets: hide_str_offset of many candidate payloads per clip, from one analysis + probe pass per clip and
        without writing MP3 bytes.  `pcm`, `n_samples`, `pcm_off` as encode(); sample_rate and bitrate_kbps are ints or one entry
        per clip.  bodies[i] is the bytes of clip i; candidates[i] is a list of (head: bytes, body_len: int), each hiding the
        MSB-first bits of head + bodies[i][:body_len].  Returns one int64 array of offsets per clip, in candidate order.
        Raises IndexError, for the whole call, when a candidate drives the rate loop past the end of the step table."""
        L = self._L
        n = len(n_samples)
        if len(bodies) != n or len(candidates) != n:
            raise ValueError("encode_offsets: one body and one candidate list per clip")
        ns, ns_p = _i64(n_samples)
        if pcm_off is None:
            pcm_off = np.concatenate([[0], np.cumsum(ns * 2)])[:-1]
        po, po_p = _i64(pcm_off)
        srs = np.ascontiguousarray(np.broadcast_to(np.asarray(sample_rate, np.int32), (n,)))
        brs = np.ascontiguousarray(np.broadcast_to(np.asarray(bitrate_kbps, np.int32), (n,)))
        body = np.frombuffer(b"".join(bodies) + b"\0", np.uint8)
        bo, bo_p = _i64(np.concatenate([[0], np.cumsum([len(b) for b in bodies])]))
        co, co_p = _i64(np.concatenate([[0], np.cumsum([len(c) for c in candidates])]))
        heads = [hd for cs in candidates for hd, _ in cs]
        head = np.frombuffer(b"".join(heads) + b"\0", np.uint8)
        ho, ho_p = _i64(np.concatenate([[0], np.cumsum([len(hd) for hd in heads])]))
        bl, bl_p = _i64([b for cs in candidates for _, b in cs] or [0])
        out = np.zeros(max(int(co[-1]), 1), np.int64)
        _ready(pcm)
        rc = L.m3s_encode_offsets(self._h, _ptr(pcm), _mem_of(pcm), po_p, ns_p, n, srs.ctypes.data_as(_c_i32p),
                                  brs.ctypes.data_as(_c_i32p), _ptr(body), bo_p, co_p, _ptr(head), ho_p, bl_p,
                                  out.ctypes.data_as(_c_i64p))
        if rc == M3S_ERR_ARG:
            msg = L.m3s_last_error(self._h).decode()
            if STEP_TABLE_OVERRUN in msg:
                raise IndexError(f"index out of bounds: {msg}")
        self._check(rc, "m3s_encode_offsets")
        return [out[co[i]:co[i + 1]].copy() for i in range(n)]


_default = {}


def default_handle(device: int = 0) -> Handle:
    """Process-wide handle used by the single-file classes (MP3Parser / MP3Encoder)."""
    if device not in _default:
        _default[device] = Handle(device)
    return _default[device]
