"""Batch entry points over the C ABI: what the facade's five methods do (steganography.py:80-182), for many files per
call and without leaving the GPU between the decode and the encode half of the composites (SURVEY.md 8f rows 1 and 3).

  reveal_batch   reveal_massage for N files: frame walk + side-info scan + reveal bits only (D0 + D4, ~36 B/frame of traffic);
                 no Huffman decode, no synthesis, no temp WAV
  hide_batch     hide_message for N files: decode (float64 instantiation, so the int16 PCM equals the reference's WAV sample
                 for sample) -> encode + hide at each file's own sample rate and bitrate, all files in one encode call; the PCM
                 stays in HBM
  clear_batch    clear_file: the same with no payload
The semantics per file are the facade's: message framing '<len>#<message>' as utf-8 bits (steganography.py:10-24,88-90),
bitrate of the last frame (MP3_Parser.py:93-97), too_long = hide_str_offset < len(bits) - 1 (encoder.py:49-51),
ID3v2 skip (decoder.py:29-33).  torch is used for the device buffers only."""
import os
import sys
import time
from typing import List, Sequence, Tuple

import numpy as np

from mp3stego_b200 import _lib
from mp3stego_b200.decoder import id3_offset, parse_reveal
from mp3stego_b200.steganography import str_to_binary_str


def _concat(blobs: Sequence[bytes]):
    data = np.frombuffer(b"".join(blobs), np.uint8)
    off = np.concatenate([[0], np.cumsum([len(b) for b in blobs])]).astype(np.int64)
    audio = [id3_offset(np.frombuffer(b[:10], np.uint8)) if len(b) >= 10 else 0 for b in blobs]
    return data, off, audio


def reveal_batch(handle: "_lib.Handle", blobs: Sequence[bytes]) -> List[str]:
    """Hidden strings of N MP3 files ('' where there is none), from the side info alone."""
    if not blobs:
        return []
    data, off, audio = _concat(blobs)
    sc = handle.decode_scan(data, off, audio)
    for i in range(len(blobs)):   # the reference facade exits / raises on these; a batch must not turn them into ''
        _lib.raise_for_status(int(sc["status"][i]), f"file {i}")
        if sc["status"][i] & _lib.M3S_FILE_NO_SYNC:
            raise ValueError(f"file {i}: no MPEG sync word at the audio start (MP3Parser is not valid, MP3_Parser.py:36-44)")
    _, bits = handle.decode_reveal()
    return [parse_reveal(b) for b in bits]


def _pinned(handle, name: str, nbytes: int):
    """Grow-only pinned staging buffer kept on the handle (pinning costs ~0.1 s per GB: once, not per call)."""
    import torch
    cache = handle.__dict__.setdefault("_batch_pinned", {})
    buf = cache.get(name)
    if buf is None or buf.numel() < nbytes:
        buf = cache[name] = torch.empty(max(int(nbytes * 1.25), 1 << 20), dtype=torch.uint8, pin_memory=True)
    return buf


def _transcode(handle, blobs, payloads) -> Tuple[List[bytes], List[int], List[int]]:
    """decode (exact) -> encode for N files, bytes in -> bytes out.  The host side moves every byte exactly twice: the files are
    gathered straight into a pinned buffer (one pass) that crosses PCIe in one asynchronous copy, and the MP3s come back into a
    pinned buffer from which the per-file `bytes` are cut (one pass); everything in between stays in HBM."""
    import torch
    trace = os.environ.get("M3S_TRACE") is not None   # host wall clock of the stages (diagnostic)
    t_last = [time.perf_counter()]

    def mark(tag):
        if trace:
            torch.cuda.synchronize()
            t = time.perf_counter()
            print("[m3s batch] %-14s +%.1f ms" % (tag, 1e3 * (t - t_last[0])), file=sys.stderr)
            t_last[0] = t
    n = len(blobs)
    sizes = np.fromiter((len(b) for b in blobs), np.int64, n)
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    total = int(off[-1])
    audio = [id3_offset(np.frombuffer(b[:10], np.uint8)) if len(b) >= 10 else 0 for b in blobs]
    dev = torch.device("cuda", handle.device)
    stage = _pinned(handle, "in", total + 16)
    sv = stage.numpy()
    for b, o in zip(blobs, off):
        sv[o:o + len(b)] = np.frombuffer(b, np.uint8)
    mark("gather")
    d_data = torch.empty(total + 16, dtype=torch.uint8, device=dev)
    d_data[:total].copy_(stage[:total], non_blocking=True)   # overlaps the host-side bound computation below
    L = _lib.load()
    fb = np.zeros(1, np.int64)
    au, au_p = _lib._i64(audio)
    elems = int(L.m3s_decode_bound(_lib._ptr(sv), off.ctypes.data_as(_lib._c_i64p), au_p, n, fb.ctypes.data_as(_lib._c_i64p)))
    pcm = torch.empty(max(elems, 2) + 2, dtype=torch.int16, device=dev)
    mark("upload+bound")
    try:     # one self-pipelining call: scan of wave k+1 under the float64 synthesis of wave k, nothing leaves the device
        sc = handle.decode(d_data, off, audio, pcm=pcm, frames_bound=int(fb[0]) + 1, exact=True)
    except _lib.M3SError as e:
        if "hold" not in str(e):
            raise
        s0 = handle.decode_scan(d_data, off, audio)   # VBR input: size from an exact scan
        pcm = torch.empty(int((s0["pcm_rows"] * np.maximum(s0["channels"], 1)).sum()) + 2, dtype=torch.int16, device=dev)
        sc = handle.decode(d_data, off, audio, pcm=pcm, frames_bound=int(s0["n_frames"].sum()) + 1, exact=True)
    mark("decode")
    status, nfr, nchan = sc["status"], sc["n_frames"], sc["channels"]
    for i in np.nonzero((status != 0) | (nfr == 0) | (nchan != 2))[0]:
        _lib.raise_for_status(int(status[i]), f"file {i}")
        if status[i] & _lib.M3S_FILE_NO_SYNC or nfr[i] == 0:
            raise ValueError(f"file {i}: not an MPEG-1 Layer III stream the reference can decode")
        if nchan[i] != 2:
            raise IndexError(f"file {i}: the reference encoder only handles stereo input (WAV_Reader / MP3_Encoder.py:611-614)")
    rows = sc["pcm_rows"].astype(np.int64)
    pcm_off = sc["pcm_off"]
    kbps = sc["bitrate"].astype(np.int64) // 1000
    # one encode call for the whole batch, every file at its own sample rate and last-frame bitrate
    res = handle.encode(pcm, rows, sc["sample_rate"], kbps, payloads=list(payloads), pcm_off=pcm_off[:n], compact=True)
    mark("encode")
    nbytes = int(res["mp3_off"][-1] + res["out_len"][-1])
    back = _pinned(handle, "out", nbytes)
    back[:nbytes].copy_(res["mp3"][:nbytes], non_blocking=True)
    torch.cuda.current_stream(dev).synchronize()
    mark("download")
    mv = memoryview(back.numpy())
    out = [bytes(mv[o:o + ln]) for o, ln in zip(res["mp3_off"].tolist(), res["out_len"].tolist())]
    hoff = res["hide_str_offset"].tolist()
    mark("cut")
    return out, hoff, kbps.tolist()


def hide_batch(handle: "_lib.Handle", blobs: Sequence[bytes], messages: Sequence[str]) -> Tuple[List[bytes], List[bool]]:
    """hide_message for N (mp3 bytes, message) pairs -> (new mp3 bytes, too_long flags)."""
    if len(blobs) != len(messages):
        raise ValueError("one message per file")
    if not blobs:
        return [], []
    bits = [str_to_binary_str(str(len(m)) + "#" + m) for m in messages]
    out, hoff, _ = _transcode(handle, blobs, bits)
    return out, [hoff[i] < len(bits[i]) - 1 for i in range(len(blobs))]


def clear_batch(handle: "_lib.Handle", blobs: Sequence[bytes]) -> List[bytes]:
    """clear_file for N files: decode and re-encode at the file's own bitrate with no payload."""
    if not blobs:
        return []
    return _transcode(handle, blobs, [""] * len(blobs))[0]
