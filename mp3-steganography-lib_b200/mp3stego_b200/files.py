"""Batched file-level I/O edge of the hot path (SURVEY.md 8f row 2): paths in -> files out, many files per call.

  decode_files   MP3 files -> WAV files (+ revealed strings): what Decoder.decode does per file (decoder.py:19-110: read the file,
                 ID3v2 skip, parse, write_to_wav via scipy's layout, optional reveal text), with the reads on a thread pool into
                 ONE pinned buffer, one self-pipelining m3s_decode call for the whole batch, and the WAV writes on the pool again
  encode_files   WAV files -> MP3 files (optionally hiding one message per file): what Encoder.encode does per file
                 (encoder.py:22-51, WAV_Reader.py:30-110), same structure around one m3s_encode_mixed call for all files, each
                 at its own sample rate and bitrate

torch is used for pinned host memory only.  Per-file failures follow the reference: sys.exit messages for missing files / bad
WAV headers, IndexError for input the reference's encoder cannot read (mono, length not a multiple of 1152, a clip that drives the rate loop past the step table)."""
import os
import struct
import sys
from concurrent.futures import ThreadPoolExecutor
from typing import List, Optional, Sequence, Union

import numpy as np

from mp3stego_b200 import _lib
from mp3stego_b200.decoder import id3_offset, parse_reveal
from mp3stego_b200.steganography import str_to_binary_str
from mp3stego_b200.wavio import MPEG1_L3_BITRATES, WavReader


def _pinned(nbytes: int):
    import torch
    return torch.empty(max(nbytes, 16), dtype=torch.uint8, pin_memory=True)


def _wav_header(sample_rate: int, nch: int, nbytes: int) -> bytes:
    return b"RIFF" + struct.pack("<I", 36 + nbytes) + b"WAVE" + b"fmt " + struct.pack(
        "<IHHIIHH", 16, 1, nch, sample_rate, sample_rate * nch * 2, nch * 2, 16) + b"data" + struct.pack("<I", nbytes)


def decode_files(handle: "_lib.Handle", mp3_paths: Sequence[str], wav_paths: Optional[Sequence[str]] = None, reveal: bool = False,
                 threads: int = 8, exact: bool = True) -> List[dict]:
    """Decode N MP3 files to WAV files (wav_paths[i]; None = the reference's default input[:-4] + '.wav'; pass wav_paths=False to
    write nothing) and return per file dict(n_frames, bitrate (kbps), sample_rate, channels, status, message) -- `message` is the
    revealed string when reveal=True.  exact=True runs the float64 instantiation (the WAV then equals the reference's sample for
    sample, which hide / clear round trips need); exact=False is the FP32 path (<= 1 LSB)."""
    n = len(mp3_paths)
    if n == 0:
        return []
    for p in mp3_paths:
        if not os.path.exists(p):
            sys.exit(f"File {p} not found.")
    sizes = [os.path.getsize(p) for p in mp3_paths]
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    buf = _pinned(int(off[-1]))
    view = buf.numpy()

    def read(i):
        with open(mp3_paths[i], "rb") as f:
            got = f.readinto(memoryview(view[off[i]:off[i + 1]]))
        if got != sizes[i]:
            raise IOError(f"{mp3_paths[i]}: short read")
        return id3_offset(view[off[i]:off[i] + 10]) if sizes[i] >= 10 else 0

    with ThreadPoolExecutor(max(1, threads)) as pool:
        audio = list(pool.map(read, range(n)))
        L = _lib.load()
        fb = np.zeros(1, np.int64)
        au, au_p = _lib._i64(audio)
        elems = int(L.m3s_decode_bound(_lib._ptr(view), off.ctypes.data_as(_lib._c_i64p), au_p, n, fb.ctypes.data_as(_lib._c_i64p)))
        import torch
        pcm = torch.empty(max(elems, 2), dtype=torch.int16, pin_memory=True)
        try:
            res = handle.decode(buf[: int(off[-1])] if off[-1] else buf[:0], off, audio, pcm=pcm, frames_bound=int(fb[0]), exact=exact)
        except _lib.M3SError as e:
            if "pcm holds" not in str(e) and "hold" not in str(e):
                raise
            # a VBR file decoded to more frames than its first header promised: size from an exact scan and go again
            sc = handle.decode_scan(buf[: int(off[-1])], off, audio)
            total = int((sc["pcm_rows"] * np.maximum(sc["channels"], 1)).sum())
            pcm = torch.empty(max(total, 2), dtype=torch.int16, pin_memory=True)
            res = handle.decode(buf[: int(off[-1])], off, audio, pcm=pcm, frames_bound=int(sc["n_frames"].sum()) + 1, exact=exact)
        strings = handle.reveal_strings(res) if reveal else [""] * n
        pv = pcm.numpy()
        out = []
        for i in range(n):
            st = int(res["status"][i])
            _lib.raise_for_status(st, mp3_paths[i])
            out.append(dict(n_frames=int(res["n_frames"][i]), bitrate=int(res["bitrate"][i]) // 1000, sample_rate=int(res["sample_rate"][i]),
                            channels=int(res["channels"][i]), status=st, message=parse_reveal(strings[i]) if reveal else None))

        def write(i):
            if wav_paths is False or out[i]["n_frames"] == 0:
                return
            path = mp3_paths[i][:-4] + ".wav" if wav_paths is None else wav_paths[i]
            a, b = int(res["pcm_off"][i]), int(res["pcm_off"][i + 1])
            with open(path, "wb") as f:
                f.write(_wav_header(out[i]["sample_rate"], max(out[i]["channels"], 1), 2 * (b - a)))
                f.write(memoryview(pv[a:b]).cast("B"))

        list(pool.map(write, range(n)))
    return out


def encode_files(handle: "_lib.Handle", wav_paths: Sequence[str], mp3_paths: Sequence[str], bitrate: Union[int, Sequence[int]] = 320,
                 messages: Optional[Sequence[str]] = None, threads: int = 8) -> List[bool]:
    """Encode N WAV files to MP3 files at `bitrate` kbps -- one int for every file, or one entry per file (the reference's
    Encoder(file, out, bitrate=...) sets it per file) -- hiding messages[i] ('' or None = plain encode) in file i with the facade's
    '<len>#<message>' framing (steganography.py:44-47).  All files go through one encode call whatever their sample rates and
    bitrates.  Returns the too_long flags (encoder.py:49-51)."""
    n = len(wav_paths)
    if n == 0:
        return []
    if len(mp3_paths) != n or (messages is not None and len(messages) != n):
        raise ValueError("one output path (and one message) per input file")
    rates = [bitrate] * n if isinstance(bitrate, (int, np.integer)) else list(bitrate)
    if len(rates) != n:
        raise ValueError("one bitrate per input file")
    for p in wav_paths:
        if not os.path.exists(p):
            sys.exit(f"File {p} not found.")
    for b in rates:
        if b not in MPEG1_L3_BITRATES:
            sys.exit("Unsupported bitrate configuration.")
    with ThreadPoolExecutor(max(1, threads)) as pool:
        readers = list(pool.map(WavReader, wav_paths, rates))   # header checks + sample buffer, reference semantics
        for w in readers:
            if w.num_of_channels != 2:
                raise IndexError("index out of bounds: the reference encoder only works on 16-bit stereo input")
            if w.num_of_samples % 1152 or len(w.buffer) < 2 * w.num_of_samples:
                raise IndexError("index out of bounds: sample count is not a multiple of 1152")
        bits = [str_to_binary_str(str(len(m)) + "#" + m) if m else "" for m in (messages or [""] * n)]
        ns = [w.num_of_samples for w in readers]
        po = np.concatenate([[0], np.cumsum([2 * s for s in ns])]).astype(np.int64)
        stage = _pinned(2 * int(po[-1])).view(dtype=__import__("torch").int16)
        sv = stage.numpy()

        def fill(i):
            sv[po[i]:po[i + 1]] = readers[i].buffer[: 2 * ns[i]]

        list(pool.map(fill, range(n)))
        res = handle.encode(stage[: int(po[-1])], ns, [w.samplerate for w in readers], rates, payloads=bits, pcm_off=po[:-1],
                            compact=True)
        mp3 = res["mp3"]

        def write(i):
            o, ln = int(res["mp3_off"][i]), int(res["out_len"][i])
            with open(mp3_paths[i], "wb") as f:
                f.write(memoryview(np.ascontiguousarray(mp3[o:o + ln])).cast("B"))

        list(pool.map(write, range(n)))
    return [int(res["hide_str_offset"][i]) < len(bits[i]) - 1 for i in range(n)]
