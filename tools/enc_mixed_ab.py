"""What encoding a mixed-rate corpus in one call buys: m3s_encode_mixed against one m3s_encode call per (sample rate, bitrate)
group, and the hide_batch / clear_batch composites of this tree against an older tree.

    python tools/enc_mixed_ab.py [--clips 1000] [--frames 689] [--reps 2] [--parent lib/alt/parent] [--out DIR]

1. A seeded corpus of tone+noise clips spread over {44.1, 48, 32} kHz x {128, 192, 256, 320} kbps, with payloads, encoded per
   group (one Handle.encode per pair) and in one mixed call, from device-resident and from pinned host buffers.  The two forms
   alternate `reps` times after one warm-up each; host clock around synchronous calls; the bytes and hide_str_offsets must be equal.
2. hide_batch and clear_batch over MP3s of the same corpus, in this tree and in `--parent` (a checkout of an older commit built
   in place with `python __graft_entry__.py`), each tree in a process of its own, alternating.  Outputs are compared by digest.
3. bench.py --no-extras (encode+hide ms per step) of this tree and of the parent, alternating twice.

Prints the card's name and power limit with the numbers and writes everything to <out>/enc_mixed_ab.json (default: a directory
in the temporary directory, so that the tree stays untouched)."""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RATES = (44100, 48000, 32000)
KBPS = (128, 192, 256, 320)


def _use_tree(tree):
    pkg = os.path.join(tree, "mp3-steganography-lib_b200")
    sys.path.insert(0, pkg)


def _cache(n_clips, n_frames, seed):
    return os.path.join(tempfile.gettempdir(), f"enc_mixed_ab_{os.getuid()}_{n_clips}_{n_frames}_{seed}")


def corpus(n_clips, n_frames, seed=7):
    """Interleaved int16 stereo PCM of n_clips tone+noise clips, their rate pairs and payloads ('0'/'1').  Cached in the temporary
    directory: every process of a run reads the same corpus."""
    path = _cache(n_clips, n_frames, seed)
    if os.path.exists(path + ".json"):
        meta = json.load(open(path + ".json"))
        return np.load(path + ".npy"), np.array(meta["sr"], np.int32), np.array(meta["br"], np.int32), meta["bits"]
    rng = np.random.default_rng(seed)
    n = n_frames * 1152
    bank = (0.05 * 32767 * rng.standard_normal((4 * n, 2))).astype(np.float32)   # noise shared by all clips at random offsets
    pcm = np.empty((n_clips, n, 2), np.int16)
    t = np.arange(n, dtype=np.float32)
    srs = np.array([RATES[i % 3] for i in range(n_clips)], np.int32)
    brs = np.array([KBPS[(i // 3) % 4] for i in range(n_clips)], np.int32)
    perm = rng.permutation(n_clips)
    srs, brs = srs[perm], brs[perm]
    for i in range(n_clips):
        f = rng.uniform(100, 5000, size=2).astype(np.float32)
        o = int(rng.integers(0, 3 * n))
        x = 0.4 * 32767 * np.sin((2 * np.pi / srs[i]) * f[None, :] * t[:, None]) + bank[o:o + n]
        pcm[i] = np.clip(x, -32768, 32767).astype(np.int16)
    bits = [(rng.integers(0, 2, size=int(rng.integers(100, 12 * n_frames))) + 48).astype(np.uint8).tobytes().decode() for _ in range(n_clips)]
    np.save(path + ".npy", pcm)
    with open(path + ".json", "w") as f:
        json.dump(dict(sr=srs.tolist(), br=brs.tolist(), bits=bits), f)
    return pcm, srs, brs, bits


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def _cut(res, n, device):
    mp3 = res["mp3"].cpu().numpy() if device else res["mp3"]
    return [bytes(mp3[int(o):int(o) + int(ln)]) for o, ln in zip(res["mp3_off"][:n], res["out_len"][:n])]


def encode_ab(args):
    _use_tree(ROOT)
    import torch
    from mp3stego_b200 import _lib
    pcm, srs, brs, bits = corpus(args.clips, args.frames)
    n = args.clips
    ns = np.full(n, args.frames * 1152, np.int64)
    po = np.arange(n, dtype=np.int64) * 2 * args.frames * 1152
    h = _lib.Handle(0)
    groups = {}
    for i in range(n):
        groups.setdefault((int(srs[i]), int(brs[i])), []).append(i)
    out = {}
    for where in ("device", "host"):
        flat = torch.from_numpy(pcm.reshape(-1))
        x = flat.cuda() if where == "device" else flat.pin_memory()
        dev = where == "device"

        def per_group():
            got = [None] * n
            hoff = [0] * n
            for (sr, br), idx in groups.items():
                r = h.encode(x, ns[idx], sr, br, payloads=[bits[i] for i in idx], pcm_off=po[idx])
                for i, b, o in zip(idx, _cut(r, len(idx), dev), r["hide_str_offset"]):
                    got[i], hoff[i] = b, int(o)
            return got, hoff

        def mixed():
            r = h.encode(x, ns, srs, brs, payloads=bits, pcm_off=po)
            return _cut(r, n, dev), [int(o) for o in r["hide_str_offset"]]

        ref = per_group()
        assert mixed() == ref, f"{where}: the mixed call's bytes differ from the per-group calls'"
        times = {"per_group": [], "mixed": []}
        for _ in range(args.reps):
            for name, fn in (("per_group", per_group), ("mixed", mixed)):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                got = fn()
                torch.cuda.synchronize()
                times[name].append(1e3 * (time.perf_counter() - t0))
                assert got == ref, f"{where} {name}: bytes differ"
        out[where] = dict(ms=times, calls_per_group=len(groups))
        print(f"[1] {where:6s} per-group ({len(groups)} calls) ms {['%.1f' % v for v in times['per_group']]}   "
              f"mixed (1 call) ms {['%.1f' % v for v in times['mixed']]}", flush=True)
    h.close()
    return out


def composite(tree, clips, frames, reps):
    """Child process: time hide_batch / clear_batch of `tree` on MP3s of the corpus (made with that tree's per-pair encode)."""
    _use_tree(tree)
    import torch
    from mp3stego_b200 import _lib, batch
    pcm, srs, brs, _ = corpus(clips, frames)
    h = _lib.Handle(0)
    blobs = [None] * clips
    for sr in RATES:
        for br in KBPS:
            idx = np.nonzero((srs == sr) & (brs == br))[0]
            if idx.size == 0:
                continue
            r = h.encode(pcm[idx].reshape(-1), np.full(idx.size, frames * 1152), sr, br)
            for i, b in zip(idx, _cut(r, idx.size, False)):
                blobs[i] = b
    rng = np.random.default_rng(3)
    msgs = ["".join(chr(int(c)) for c in rng.integers(32, 127, size=int(rng.integers(10, 400)))) for _ in range(clips)]
    res = {}
    for name, fn in (("hide_batch", lambda: batch.hide_batch(h, blobs, msgs)), ("clear_batch", lambda: batch.clear_batch(h, blobs))):
        fn()   # warm-up
        ms = []
        for _ in range(reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            got = fn()
            torch.cuda.synchronize()
            ms.append(1e3 * (time.perf_counter() - t0))
        outs = got[0] if name == "hide_batch" else got
        dig = hashlib.sha256(b"".join(outs) + (json.dumps(got[1]).encode() if name == "hide_batch" else b"")).hexdigest()
        res[name] = dict(ms=ms, sha256=dig)
    h.close()
    print(json.dumps(res))


def run_child(tree, args):
    cmd = [sys.executable, os.path.abspath(__file__), "--composite-of", tree, "--clips", str(args.clips), "--frames", str(args.frames),
           "--reps", str(args.reps)]
    p = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT)
    if p.returncode != 0:
        raise RuntimeError(f"composite in {tree} failed:\n{p.stderr[-3000:]}")
    return json.loads(p.stdout.strip().splitlines()[-1])


def bench(tree):
    p = subprocess.run([sys.executable, "bench.py", "--gpus", "1", "--steps", "5", "--warmup", "2", "--no-extras"], capture_output=True,
                       text=True, cwd=tree)
    if p.returncode != 0:
        raise RuntimeError(f"bench.py in {tree} failed:\n{p.stderr[-3000:]}")
    d = json.loads(p.stdout.strip().splitlines()[-1])
    return d["encode_hide"]["ms_per_step"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--clips", type=int, default=1000)
    ap.add_argument("--frames", type=int, default=689)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--parent", default=os.path.join(ROOT, "lib", "alt", "parent"))
    ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "enc_mixed_ab"))
    ap.add_argument("--composite-of", help=argparse.SUPPRESS)
    ap.add_argument("--skip", default="", help="comma list of parts to skip: encode,composite,bench")
    args = ap.parse_args()
    if args.composite_of:
        return composite(args.composite_of, args.clips, args.frames, args.reps)
    skip = set(filter(None, args.skip.split(",")))
    rep = dict(card=card(), clips=args.clips, frames=args.frames, reps=args.reps)
    print("card, power limit:", rep["card"], flush=True)
    if "encode" not in skip:
        rep["encode"] = encode_ab(args)
    if "composite" not in skip:
        rep["composite"] = {"this": [], "parent": []}
        for _ in range(2):
            for arm, tree in (("parent", args.parent), ("this", ROOT)):
                r = run_child(tree, args)
                rep["composite"][arm].append(r)
                print(f"[2] {arm:6s} hide_batch ms {['%.1f' % v for v in r['hide_batch']['ms']]}  clear_batch ms "
                      f"{['%.1f' % v for v in r['clear_batch']['ms']]}", flush=True)
        c = rep["composite"]
        rep["composite_outputs_equal"] = all(a[k]["sha256"] == b[k]["sha256"] for a, b in zip(c["this"], c["parent"])
                                             for k in ("hide_batch", "clear_batch"))
        print("[2] outputs equal:", rep["composite_outputs_equal"], flush=True)
    if "bench" not in skip:
        rep["bench_encode_hide_ms"] = {"parent": [], "this": []}
        for _ in range(2):
            for arm, tree in (("parent", args.parent), ("this", ROOT)):
                rep["bench_encode_hide_ms"][arm].append(bench(tree))
                print(f"[3] {arm:6s} bench encode+hide ms/step {rep['bench_encode_hide_ms'][arm][-1]:.1f}", flush=True)
    for ext in (".npy", ".json"):
        if os.path.exists(_cache(args.clips, args.frames, 7) + ext):
            os.remove(_cache(args.clips, args.frames, 7) + ext)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "enc_mixed_ab.json"), "w") as f:
        json.dump(rep, f, indent=1)


if __name__ == "__main__":
    main()
