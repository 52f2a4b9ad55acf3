"""What a capacity query costs: m3s_encode_offsets against m3s_encode_mixed, and capacity_batch against hide_batch.

    python tools/offsets_bench.py [--clips 1000] [--frames 689] [--reps 3] [--files 256] [--out DIR]

1. Device-resident tone+noise clips (bench.py's generator, 44.1 kHz / 128 kbps) with bench.py's random payload cut to whole
   bytes, one candidate per clip: m3s_encode_offsets and m3s_encode_mixed alternate `reps` times after one warm-up each (host
   clock around the synchronous calls).  The offsets must equal the encoder's hide_str_offsets.
2. The same clips, each with every prefix of a random ASCII message of ~1.25 x the clip's capacity (from 1.): call time,
   candidate count and the per-kernel device times of a separate timed call (m3s_timing_get).  The probe's time here, where
   the shortest candidate ("0#", 16 bits) keeps all 15 payload variants active after its fifth granule, against its time in 1.
   (one long payload: 8 variants until the payload's last granules) says what the pruning costs.
3. `--files` MP3s of the same clips from host bytes: capacity_batch (decode + one offsets call) against one hide_batch
   (decode + encode) of the same messages, alternating `reps` times after one warm-up each.

Prints the card's name and power limit with the numbers and writes everything to <out>/offsets_bench.json (default: a directory
in the temporary directory, so that the tree stays untouched)."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "mp3-steganography-lib_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                       text=True)
    return q.stdout.strip()


def timed(fn):
    t0 = time.perf_counter()
    r = fn()
    return 1e3 * (time.perf_counter() - t0), r


def kernel_times(h, fn):
    h.timing_enable(True)
    try:
        fn()
        return {k: round(ms, 2) for k, (ms, _) in h.timing().items()}
    finally:
        h.timing_enable(False)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--clips", type=int, default=1000)
    ap.add_argument("--frames", type=int, default=689)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--files", type=int, default=256)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import bench
    from mp3stego_b200 import _lib, batch
    out_dir = a.out or tempfile.mkdtemp(prefix="offsets_bench_")
    os.makedirs(out_dir, exist_ok=True)
    res = dict(card=card(), clips=a.clips, frames=a.frames)
    print("card (name, power limit):", res["card"], flush=True)
    h = _lib.Handle(0)
    dev = torch.device("cuda", 0)
    C, F = a.clips, a.frames
    pcm = bench.synth_pcm_device(torch, C, F, 11, dev).reshape(-1)
    torch.cuda.synchronize()
    ns, srs, brs = [F * 1152] * C, [44100] * C, [128] * C
    nbits = bench.PAYLOAD_BITS_PER_FRAME * F // 8 * 8
    pay, poff = bench.random_payload_bits(C, nbits, 7)
    bodies = [np.packbits(pay[i * nbits:(i + 1) * nbits] - ord("0")).tobytes() for i in range(C)]
    one = [[(b"", len(b))] for b in bodies]
    mp3 = torch.empty(C * int(h._L.m3s_encode_bound(F * 1152, 44100, 128)) + 16, dtype=torch.uint8, device=dev)

    # ---- 1. one candidate per clip: offsets vs encode
    enc = lambda: h.encode(pcm, ns, srs, brs, payload_packed=(pay, poff), mp3_out=mp3)   # noqa: E731
    offs = lambda: h.encode_offsets(pcm, ns, srs, brs, bodies, one)                     # noqa: E731
    enc()
    offs()
    t_enc, t_off = [], []
    for _ in range(a.reps):
        ms, r_enc = timed(enc)
        t_enc.append(ms)
        ms, r_off = timed(offs)
        t_off.append(ms)
    got = np.array([o[0] for o in r_off])
    assert np.array_equal(got, r_enc["hide_str_offset"]), "offsets differ from the encoder"
    res["one_candidate"] = dict(encode_mixed_ms=[round(x, 1) for x in t_enc], encode_offsets_ms=[round(x, 1) for x in t_off],
                                kernels_encode=kernel_times(h, enc), kernels_offsets=kernel_times(h, offs),
                                mean_offset_bits=float(got.mean()))
    print("1. one candidate per clip:", json.dumps(res["one_candidate"]), flush=True)

    # ---- 2. every prefix of a message at ~1.25 x capacity
    rng = np.random.default_rng(3)
    msgs = ["".join(chr(c) for c in rng.integers(32, 127, max(1, int(1.25 * o / 8)))) for o in got]
    bc = [batch.capacity_candidates(m) for m in msgs]
    pre_b, pre_c = [b for b, _ in bc], [c for _, c in bc]
    n_cand = sum(len(c) for c in pre_c)
    many = lambda: h.encode_offsets(pcm, ns, srs, brs, pre_b, pre_c)   # noqa: E731
    many()
    t_many = [round(timed(many)[0], 1) for _ in range(max(1, a.reps - 1))]
    res["all_prefixes"] = dict(candidates=n_cand, call_ms=t_many, kernels=kernel_times(h, many))
    print("2. every prefix:", json.dumps(res["all_prefixes"]), flush=True)

    # ---- 3. capacity_batch vs hide_batch from host bytes
    nf = min(a.files, C)
    r = h.encode(pcm[: nf * F * 2304], ns[:nf], 44100, 128, compact=True)
    raw = r["mp3"][: int(r["mp3_off"][-1] + r["out_len"][-1])].cpu().numpy()
    blobs = [raw[o:o + n].tobytes() for o, n in zip(r["mp3_off"].tolist(), r["out_len"].tolist())]
    cap = lambda: batch.capacity_batch(h, blobs, msgs[:nf])   # noqa: E731
    hide = lambda: batch.hide_batch(h, blobs, msgs[:nf])       # noqa: E731
    cap()
    hide()
    t_cap, t_hide = [], []
    for _ in range(a.reps):
        ms, best = timed(cap)
        t_cap.append(round(ms, 1))
        t_hide.append(round(timed(hide)[0], 1))
    res["files"] = dict(files=nf, capacity_batch_ms=t_cap, hide_batch_ms=t_hide, mean_n_star=float(np.mean(best)),
                        mean_message_chars=float(np.mean([len(m) for m in msgs[:nf]])))
    print("3. files:", json.dumps(res["files"]), flush=True)
    h.close()
    with open(os.path.join(out_dir, "offsets_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", os.path.join(out_dir, "offsets_bench.json"))


if __name__ == "__main__":
    main()
