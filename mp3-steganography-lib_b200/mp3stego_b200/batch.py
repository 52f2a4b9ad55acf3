"""Batch entry points over the C ABI: what the facade's five methods do (steganography.py:80-182), for many files per
call and without leaving the GPU between the decode and the encode half of the composites (SURVEY.md 8f rows 1 and 3).

  reveal_batch   reveal_massage for N files: frame walk + side-info scan + reveal bits only (D0 + D4, ~36 B/frame of traffic);
                 no Huffman decode, no synthesis, no temp WAV
  hide_batch     hide_message for N files: decode (float64 instantiation, so the int16 PCM equals the reference's WAV sample
                 for sample) -> encode + hide at each file's own sample rate and bitrate, all files in one encode call; the PCM
                 stays in HBM
  clear_batch    clear_file: the same with no payload
  capacity_batch   the longest prefix of each message that hide_message would hide whole (every prefix resolved in ONE
                   m3s_encode_offsets call against one analysis + probe pass per file)
  hide_batch_fit   hide_batch of those prefixes, from the same decode
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


def _marker():
    """mark(tag): host wall clock of the batch stages on stderr when M3S_TRACE is set (diagnostic)."""
    import torch
    trace = os.environ.get("M3S_TRACE") is not None
    t_last = [time.perf_counter()]

    def mark(tag):
        if trace:
            torch.cuda.synchronize()
            t = time.perf_counter()
            print("[m3s batch] %-14s +%.1f ms" % (tag, 1e3 * (t - t_last[0])), file=sys.stderr)
            t_last[0] = t
    return mark


def _decode_exact(handle, blobs, mark):
    """The decode half of the composites: N files -> int16 PCM in HBM (float64 instantiation, so that it equals the reference's
    WAV sample for sample).  The files are gathered straight into a pinned buffer that crosses PCIe in one asynchronous copy.
    Returns dict(pcm, rows, pcm_off, sample_rate, kbps): what the encode calls take, every file at its own sample rate and
    last-frame bitrate."""
    import torch
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
    return dict(pcm=pcm, rows=sc["pcm_rows"].astype(np.int64), pcm_off=sc["pcm_off"][:n], sample_rate=sc["sample_rate"],
                kbps=sc["bitrate"].astype(np.int64) // 1000)


def _encode_cut(handle, dec, payloads, mark) -> Tuple[List[bytes], List[int], List[int]]:
    """The encode half: one encode call for the whole batch, then the MP3s come back into a pinned buffer from which the per-file
    `bytes` are cut (one pass)."""
    import torch
    dev = torch.device("cuda", handle.device)
    kbps = dec["kbps"]
    res = handle.encode(dec["pcm"], dec["rows"], dec["sample_rate"], kbps, payloads=list(payloads), pcm_off=dec["pcm_off"], compact=True)
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


def _transcode(handle, blobs, payloads) -> Tuple[List[bytes], List[int], List[int]]:
    """decode (exact) -> encode for N files, bytes in -> bytes out.  The host side moves every byte exactly twice (gather, cut);
    everything in between stays in HBM."""
    mark = _marker()
    return _encode_cut(handle, _decode_exact(handle, blobs, mark), payloads, mark)


def hide_batch(handle: "_lib.Handle", blobs: Sequence[bytes], messages: Sequence[str]) -> Tuple[List[bytes], List[bool]]:
    """hide_message for N (mp3 bytes, message) pairs -> (new mp3 bytes, too_long flags)."""
    if len(blobs) != len(messages):
        raise ValueError("one message per file")
    if not blobs:
        return [], []
    bits = [str_to_binary_str(str(len(m)) + "#" + m) for m in messages]
    out, hoff, _ = _transcode(handle, blobs, bits)
    return out, [hoff[i] < len(bits[i]) - 1 for i in range(len(blobs))]


def capacity_candidates(message: str, max_bits: int = None) -> Tuple[bytes, List[Tuple[bytes, int]]]:
    """The candidates of one message for m3s_encode_offsets: the body is the message's utf-8 bytes, and candidate n (n = 0 ..
    len(message)) is (head f"{n}#", the utf-8 length of message[:n]), whose bits are str_to_binary_str(f"{n}#{message[:n]}"), the
    framing hide_message gives message[:n].  The framed length grows with n, so the list stops before the first prefix of more
    than max_bits bits (None: no limit); candidate n is the list's entry n.  Returns (body, [(head, body_len), ...])."""
    body = message.encode("utf-8")
    ends = np.cumsum([0] + [len(ch.encode("utf-8")) for ch in message]).tolist()
    cands = []
    for n, bl in enumerate(ends):
        head = b"%d#" % n
        if max_bits is not None and 8 * (len(head) + bl) > max_bits:
            break
        cands.append((head, bl))
    return body, cands


def _capacity(handle, dec, messages) -> List[int]:
    # hide_str_offset is at most 3 per granule of a channel (the three regions' tables) and a payload fits when the offset reaches
    # its length - 1: a longer candidate cannot fit and is not evaluated
    limits = [12 * (int(r) // 1152) + 1 for r in dec["rows"]]
    bodies, cands = zip(*[capacity_candidates(m, lim) for m, lim in zip(messages, limits)])
    offs = handle.encode_offsets(dec["pcm"], dec["rows"], dec["sample_rate"], dec["kbps"], list(bodies), list(cands),
                                 pcm_off=dec["pcm_off"])
    best = []
    for cs, off in zip(cands, offs):
        fit = [n for n, ((head, bl), o) in enumerate(zip(cs, off.tolist())) if o >= 8 * (len(head) + bl) - 1]
        best.append(max(fit) if fit else -1)
    return best


def capacity_batch(handle: "_lib.Handle", blobs: Sequence[bytes], messages: Sequence[str]) -> List[int]:
    """For each file the largest n in [0, len(message)] for which hide_message(file, message[:n]) would not report too_long, i.e.
    its hide_str_offset reaches len(bits) - 1 under the framing f"{n}#{message[:n]}"; -1 when not even "0#" fits.  Every n is
    evaluated, so the answer is exact where fitting is not monotone in n (the stego swap steers quantisation).  One exact decode
    and one m3s_encode_offsets call for the batch."""
    if len(blobs) != len(messages):
        raise ValueError("one message per file")
    if not blobs:
        return []
    return _capacity(handle, _decode_exact(handle, blobs, _marker()), messages)


def hide_batch_fit(handle: "_lib.Handle", blobs: Sequence[bytes], messages: Sequence[str]) -> Tuple[List[bytes], List[int]]:
    """hide_batch of message[:n*] for each file, n* = capacity_batch(...): the longest prefix that is hidden whole.  Where n* is -1
    the file gets hide_batch's output for the empty message.  The files are decoded once; the PCM feeds both the offsets call and
    the encode.  Returns (new mp3 bytes, n*)."""
    if len(blobs) != len(messages):
        raise ValueError("one message per file")
    if not blobs:
        return [], []
    mark = _marker()
    dec = _decode_exact(handle, blobs, mark)
    best = _capacity(handle, dec, messages)
    mark("offsets")
    fit = [m[:max(n, 0)] for m, n in zip(messages, best)]
    out, _, _ = _encode_cut(handle, dec, [str_to_binary_str(str(len(m)) + "#" + m) for m in fit], mark)
    return out, best


def clear_batch(handle: "_lib.Handle", blobs: Sequence[bytes]) -> List[bytes]:
    """clear_file for N files: decode and re-encode at the file's own bitrate with no payload."""
    if not blobs:
        return []
    return _transcode(handle, blobs, [""] * len(blobs))[0]
