#!/usr/bin/env python3
"""bench.py -- throughput of the mp3stego hot path on B200 (contract: task brief; DESIGN.md "Measurement").

  python bench.py [--gpus N] [--steps K] [--warmup W]            product arm (CUDA path through the C ABI)
  python bench.py --impl reference [...]                          CPU arm: the oracle port on all host cores
  torchrun --nproc-per-node N ... bench.py --gpus N ...           one rank per GPU, files sharded by rank (weak scaling)
  python bench.py ... --dump-outputs DIR                          also save what the timed legs returned (write_dump)

Corpus (per GPU, synthetic): `--files` tone+noise 44.1 kHz stereo WAVs of `--frames` frames (SURVEY.md 8d), generated
on the device; the decode corpus is those WAVs encoded to 320 kbps by the product's own encoder (bit-exact with the
reference encoder -- tests/test_parity_encode.py), one MP3 per file.

A step is ONE pass over the whole per-GPU corpus, processed in waves of `--wave` files:
  decode+reveal (the JSON line's metric; BASELINE.json configs[1]: 1,000 x 3-minute 320 kbps files = 6.89 M frames)
      value        frames/s with the MP3 bytes resident in HBM (device pointers through the C ABI)
      e2e          the same through the C ABI with HOST buffers: H2D of MP3 bytes, D2H of PCM + table ids + reveal bits
      roofline     dominant kernel: algorithmic bytes (5,652.9 B/frame, SURVEY.md 8d) over its mean device time
      cpu_baseline the oracle port on one host core over a bounded sample of the same corpus
  encode+hide  (key "encode_hide"; configs[2]: the same WAVs -> 128 kbps hiding a random payload beyond capacity)
      the same five figures for the encoder.
The oracle is used ONLY by the cpu_baseline / --impl reference legs.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "mp3-steganography-lib_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

DEC_BYTES_PER_FRAME = 1044.9 + 4608.0   # SURVEY.md 8(d): compressed frame @320k + int16 stereo PCM
ENC_BYTES_PER_FRAME = 4608.0 + 417.96   # int16 stereo PCM + compressed frame @128k
FRAMES_PER_FILE = 6890                  # 3 minutes at 44.1 kHz (7,937,280 samples)
PAYLOAD_BITS_PER_FRAME = 14             # measured capacity is 11-12 bits/frame: the payload always exceeds it


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# ------------------------------------------------------------------------------------------------
# synthetic corpus
# ------------------------------------------------------------------------------------------------
def synth_pcm_host(n_frames, seed):
    """SURVEY.md 8(d) tone+noise clip on the host (cpu / reference legs): int16 [n, 2]."""
    rng = np.random.default_rng(seed)
    n = n_frames * 1152
    t = np.arange(n) / 44100.0
    f = rng.uniform(100, 5000, size=2)
    x = np.stack([0.4 * np.sin(2 * np.pi * f[c] * t) + 0.05 * rng.standard_normal(n) for c in range(2)], axis=1)
    return (x * 32767).astype(np.int16)


def synth_pcm_device(torch, n_files, n_frames, seed, device):
    """The same recipe on the device (setup only; torch is plumbing): int16 [n_files, 2 * n] interleaved stereo."""
    n = n_frames * 1152
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    f = torch.rand((n_files, 1, 2), generator=g, device=device, dtype=torch.float64) * 4900.0 + 100.0
    out = torch.empty((n_files, n, 2), dtype=torch.int16, device=device)
    step = max(1, (1 << 26) // max(n, 1))
    idx = torch.arange(n, device=device, dtype=torch.float64).reshape(1, n, 1)
    for lo in range(0, n_files, step):
        hi = min(n_files, lo + step)
        ph = torch.remainder(f[lo:hi] * (idx / 44100.0), 1.0).float()        # phase in turns, reduced in float64
        x = 0.4 * torch.sin(ph * (2 * np.pi))
        x += 0.05 * torch.randn((hi - lo, n, 2), generator=g, device=device)
        out[lo:hi] = (x * 32767.0).to(torch.int16)
    return out.reshape(n_files, n * 2)


def random_payload_bits(n_files, bits_per_file, seed):
    """Random 7-bit ASCII (rng.integers(32, 127)) as '0'/'1' chars, all files end to end + offsets."""
    rng = np.random.default_rng(seed)
    nbytes = (bits_per_file + 7) // 8
    chars = rng.integers(32, 127, size=(n_files, nbytes), dtype=np.uint8)
    bits = np.unpackbits(chars, axis=1)[:, :bits_per_file]
    packed = (bits + ord("0")).astype(np.uint8).reshape(-1)
    off = np.arange(n_files + 1, dtype=np.int64) * bits_per_file
    return packed, off


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,timestamp")

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100"], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            pass

    def stop(self, t0=None, t1=None):
        """Summary of the samples taken in the wall-clock window [t0, t1] (all samples when the window is not given, or when
        nvidia-smi -- slow to start, more so with eight ranks spawning it at once -- delivered none inside it)."""
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name).read().strip().splitlines() if r.strip()]
        os.unlink(self.f.name)
        if t0 is not None and t1 is not None:
            import datetime
            inside = []
            for r in rows:
                try:
                    ts = datetime.datetime.strptime(r[7].strip(), "%Y/%m/%d %H:%M:%S.%f").timestamp()
                except (ValueError, IndexError):
                    continue
                if t0 - 0.05 <= ts <= t1 + 0.05:
                    inside.append(r)
            out["window"] = ("first device-resident timed step .. last e2e timed step" if inside
                             else "whole leg incl. warm-up (no sample fell inside the timed regions)")
            rows = inside or rows
        sm, power, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[0]))
                out["sm_max_mhz"] = float(r[1])
                power.append(float(r[2]))
                for k, nme in enumerate(names):
                    if r[3 + k].strip().lower().startswith("active"):
                        reasons.add(nme)
            except (ValueError, IndexError):
                continue
        if sm:
            hi = [v for v, p in zip(sm, power) if p >= 0.6 * max(power)] or sm   # samples under load
            out["sm_mhz"] = float(np.median(hi))
            out["samples"] = len(sm)
            out["power_w_max"] = max(power)
        out["reasons"] = sorted(reasons)
        return out


# ------------------------------------------------------------------------------------------------
# reference / cpu arm (the oracle port + the Python reference; the ONLY code in this file that touches oracle/ or baseline/)
# ------------------------------------------------------------------------------------------------
_CPU_INPUTS = {}


def _cpu_init():
    from oracle import oracle as O
    O.lib()


def _cpu_decode_worker(i):
    from oracle import oracle as O
    r = O.decode(_CPU_INPUTS["mp3"][i], 0, taps=False)
    return int(r["n_frames"]), len(r["bits"])


def _cpu_encode_worker(args):
    from oracle import oracle as O
    i, bitrate, hide = args
    r = O.encode(_CPU_INPUTS["pcm"][i], 44100, bitrate, _CPU_INPUTS["bits"][i] if hide else "", taps=False)
    return int(r["n_frames"]), (r["mp3"] if not hide else None)


class CpuPort:
    """The oracle port (oracle/mp3stego_oracle.c) on `procs` host processes over `n_clips` tone+noise clips of `n_frames` frames.
    The worker pool is created ONCE and the inputs live in the workers (inherited at fork): a timed step only ships clip
    indices out and frame counts back, so neither pool start-up nor pickling of PCM sits inside the timed region."""

    def __init__(self, n_frames, procs, n_clips):
        from oracle import oracle as O
        O.build()
        O.lib()       # loaded in the parent too (the workers inherit it at fork; the driver's record of loaded libraries sees it here)
        self.n_frames, self.procs, self.n = n_frames, procs, n_clips
        _CPU_INPUTS["pcm"] = [synth_pcm_host(n_frames, 4242 + i) for i in range(n_clips)]
        packed, off = random_payload_bits(n_clips, PAYLOAD_BITS_PER_FRAME * n_frames, 7)
        _CPU_INPUTS["bits"] = [packed[off[i]:off[i + 1]].tobytes().decode("ascii") for i in range(n_clips)]
        self.pool = None
        if procs > 1:
            import multiprocessing as mp
            self.pool = mp.get_context("fork").Pool(procs, initializer=_cpu_init)
        # decode inputs: the clips at 320 kbps (untimed); the pool is re-forked afterwards so that the workers inherit them too
        _CPU_INPUTS["mp3"] = [m for _, m in self._map(_cpu_encode_worker, [(i, 320, False) for i in range(n_clips)])]
        if self.pool is not None:
            self.pool.close()
            self.pool.join()
            import multiprocessing as mp
            self.pool = mp.get_context("fork").Pool(procs, initializer=_cpu_init)
            self.pool.map(_cpu_decode_worker, [0] * procs, chunksize=1)      # every worker up, library loaded

    def _map(self, fn, items):
        if self.pool is None:
            return [fn(i) for i in items]
        return self.pool.map(fn, items, chunksize=1)

    def step(self):
        """One timed pass: encode+hide @128k then decode+reveal @320k of every clip.  {"decode": (frames, s), "encode": (frames, s)}"""
        t0 = time.perf_counter()
        res = self._map(_cpu_encode_worker, [(i, 128, True) for i in range(self.n)])
        t_enc = time.perf_counter() - t0
        f_enc = sum(r[0] for r in res)
        t0 = time.perf_counter()
        res = self._map(_cpu_decode_worker, list(range(self.n)))
        t_dec = time.perf_counter() - t0
        return {"decode": (sum(r[0] for r in res), t_dec), "encode": (f_enc, t_enc)}

    def close(self):
        if self.pool is not None:
            self.pool.close()
            self.pool.join()
            self.pool = None


def python_reference_timing(frames_dec=100, frames_enc=50, timeout=420):
    """The UNMODIFIED Python/numba reference (baseline/_ref) on one core of this host, in a subprocess (baseline/ref_timing.py)."""
    script = os.path.join(ROOT, "baseline", "ref_timing.py")
    try:
        p = subprocess.run([sys.executable, script, "--frames-dec", str(frames_dec), "--frames-enc", str(frames_enc),
                            "--test-mp3", os.path.join(ROOT, "tests", "golden", "test.mp3")],
                           capture_output=True, text=True, timeout=timeout)
        lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
        if p.returncode != 0 or not lines:
            return {"unavailable": f"ref_timing.py rc={p.returncode}: {p.stderr.strip()[-200:]}"}
        return json.loads(lines[-1])
    except Exception as e:
        return {"unavailable": f"{type(e).__name__}: {e}"}


def corpus_config(args):
    return {"workload": f"configs[1]: batch decode+reveal of {args.files} synthetic 320 kbps 44.1 kHz stereo "
                        f"{args.frames * 1152 / 44100.0:.0f}-s MP3s per GPU ({args.files * args.frames} frames); "
                        f"encode_hide = configs[2]: the same WAVs -> 128 kbps hiding random ASCII beyond capacity; "
                        f"cfg5 = configs[4]: 10,000 x 30-s tracks + one long file, strong-scaled over the ranks",
            "files_per_gpu": args.files, "frames_per_file": args.frames,
            "l2": f"inputs larger than L2 (a step streams {args.files * args.frames * 1045 / 1e9:.1f} GB of MP3 and "
                  f"{args.files * args.frames * 4608 / 1e9:.1f} GB of PCM per GPU through the kernels; L2 is 126 MB)",
            "corpus": "tone+noise WAVs (SURVEY 8d) generated on device; MP3s produced from them by the product encoder "
                      "(byte-identical to the reference encoder's output)"}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    n_frames = min(args.frames, FRAMES_PER_FILE)    # whole 3-minute files, one per host core per step
    port = CpuPort(n_frames, cores, cores)
    for _ in range(min(args.warmup, 1)):
        port.step()
    dec_f = dec_t = enc_f = enc_t = 0.0
    steps = max(1, min(args.steps, 5))               # a step is ~5 s of wall clock on every core: bounded
    for _ in range(steps):
        r = port.step()
        dec_f += r["decode"][0]; dec_t += r["decode"][1]
        enc_f += r["encode"][0]; enc_t += r["encode"][1]
    port.close()
    v = dec_f / dec_t
    sample = (f"{cores} files x {n_frames} frames of the tone+noise corpus per step ({steps} steps timed), one oracle process per host "
              f"core, persistent pool, inputs resident in the workers")
    pyref = python_reference_timing()
    line = {"impl": "reference", "metric": "decode+reveal throughput (MP3 frames/s)", "value": v, "unit": "frames/s",
            "n_gpus": args.gpus, "steps": steps, "warmup": min(args.warmup, 1), "ms_per_step": 1e3 * dec_t / steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": corpus_config(args),
            "cpu_baseline": {"value": v, "unit": "frames/s", "cores": cores, "kind": "port", "sample": sample,
                             "python_reference": pyref},
            "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "audio_seconds_per_s": v * 1152 / 44100.0,
            "encode_hide": {"value": enc_f / enc_t, "unit": "frames/s", "ms_per_step": 1e3 * enc_t / steps,
                            "e2e": {"value": enc_f / enc_t, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                            "cpu_baseline": {"value": enc_f / enc_t, "unit": "frames/s", "cores": cores, "kind": "port",
                                             "sample": sample}}}
    emit(line)


# ------------------------------------------------------------------------------------------------
# product arm
# ------------------------------------------------------------------------------------------------
def roofline_of(ktimes, names, frames_total, bytes_per_frame, peak, peak_src, steps, whole_frac):
    ks = {k: v for k, v in ktimes.items() if k in names}
    if not ks:
        return None
    dom, (ms_total, n_l) = max(ks.items(), key=lambda kv: kv[1][0])
    fpl = frames_total / n_l
    ach = bytes_per_frame * fpl / (ms_total / n_l * 1e-3) / 1e9
    traffic, traffic_src = None, None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        t = tj.get(dom, {}).get("bytes_per_frame")
        traffic = None if t is None else t * fpl
        traffic_src = tj.get("_source")
    except Exception:
        pass
    return {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
            "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src, "avg_launch_ms": ms_total / n_l,
            "frames_per_launch": fpl, "algorithmic_bytes_per_frame": bytes_per_frame,
            "kernel_ms_per_step": {k: v[0] / steps for k, v in sorted(ks.items())}, "whole_path_frac": whole_frac}


def pcm_checksum(torch, pcm16, first_sample):
    """Range-additive checksum of interleaved int16 PCM whose first element has global index `first_sample`:
    (sum x, sum x * (1 + i mod 65521)) in int64 -- the checksums of consecutive ranges add up to the whole file's."""
    x = pcm16.to(torch.int64)
    i = torch.arange(first_sample, first_sample + x.numel(), device=x.device, dtype=torch.int64)
    return int(x.sum().item()), int((x * (1 + i % 65521)).sum().item())


# ------------------------------------------------------------------------------------------------
# --dump-outputs: what the timed legs returned in their last step, as .npy files (float32 / float64), so that two builds run
# with the same arguments can be compared output for output.  The whole outputs are tens of GB; the per-file arrays go out
# whole, the buffers as a sample whose positions come from a fixed seed and the arguments only.  NaN marks a sampled
# position the call did not fill (a frame past the file's n_frames, a byte past its reveal_len / out_len).
# ------------------------------------------------------------------------------------------------
DUMP_FRAMES = 2048       # decoded frames sampled: their PCM (2,304 samples each), table ids and reveal-bit bytes (12 each)
DUMP_WINDOWS = 2048      # MP3 byte windows sampled from the encoder's output
DUMP_WINDOW = 418        # bytes per window: one 128 kbps frame at 44.1 kHz
DUMP_LIMIT = 64 << 20


def _gather(torch, buf, idx, valid):
    """buf[idx] as float32 (buf on the device), NaN where not `valid`."""
    valid = np.broadcast_to(valid, idx.shape)
    idx = np.clip(np.where(valid, idx, 0), 0, buf.numel() - 1)
    out = buf[torch.from_numpy(idx.reshape(-1)).to(buf.device)].float().cpu().numpy().reshape(idx.shape)
    out[~valid] = np.nan
    return out


def dump_decode(torch, r, files, frames):
    """m3s_decode's result of the device-resident leg: per-file arrays, and PCM / table ids / reveal bits of sampled frames."""
    rng = np.random.default_rng(20261020)
    n = min(DUMP_FRAMES, files * frames)
    fi, fj = rng.integers(0, files, n), rng.integers(0, frames, n)          # frame fj of file fi
    nfr = r["n_frames"]
    base = np.concatenate([[0], np.cumsum(nfr)])
    k = np.arange(12)
    ok = (fj < nfr[fi])[:, None]
    pcm = _gather(torch, r["pcm"], r["pcm_off"][fi][:, None] + 2304 * fj[:, None] + np.arange(2304), ok)
    ids = _gather(torch, r["table_ids"], 12 * (base[fi] + fj)[:, None] + k, ok)
    bits = _gather(torch, r["reveal_bits"], 12 * (base[fi] + fj)[:, None] + k, 12 * fj[:, None] + k < r["reveal_len"][fi][:, None])
    out = {"decode_sample_frames": np.stack([fi, fj], 1), "decode_pcm": pcm, "decode_table_ids": ids, "decode_reveal_bits": bits}
    for key in ("n_frames", "pcm_off", "reveal_len", "sample_rate", "channels", "bitrate", "status"):
        out["decode_" + key] = r[key]
    return out


def dump_encode(torch, r, files):
    """m3s_encode's result of the device-resident leg: per-clip out_len / hide_str_offset, and sampled windows of the MP3 bytes."""
    rng = np.random.default_rng(20261021)
    ci, u = rng.integers(0, files, DUMP_WINDOWS), rng.random(DUMP_WINDOWS)
    ln = r["out_len"][ci]
    start = (u * np.maximum(ln - DUMP_WINDOW, 0)).astype(np.int64)          # byte offset inside clip ci's MP3
    k = np.arange(DUMP_WINDOW)
    mp3 = _gather(torch, r["mp3"], (r["mp3_off"][ci] + start)[:, None] + k, start[:, None] + k < ln[:, None])
    return {"encode_sample_windows": np.stack([ci, start], 1), "encode_mp3": mp3, "encode_out_len": r["out_len"],
            "encode_hide_str_offset": r["hide_str_offset"]}


def write_dump(out_dir, arrays):
    arrays = {k: (v if v.dtype == np.float32 else v.astype(np.float64)) for k, v in arrays.items()}
    total = sum(v.nbytes for v in arrays.values())
    if total > DUMP_LIMIT:
        raise SystemExit(f"bench.py: --dump-outputs would write {total / 2**20:.1f} MiB (limit {DUMP_LIMIT >> 20} MiB)")
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)
    log(f"dump: {len(arrays)} arrays, {total / 2**20:.1f} MiB -> {out_dir}")


def run_product_arm(args):
    import torch
    import __graft_entry__ as ge
    ge.build()
    from mp3stego_b200 import _lib, batch, hostaffinity, shard

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", world))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product arm has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # host placement BEFORE any pinned allocation: the rank's threads (and first-touched staging pages) on its GPU's NUMA node
    try:
        pr = torch.cuda.get_device_properties(local)
        pci = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
    except Exception:
        pci = ""
    affinity = hostaffinity.bind_to_device(pci, local, local_world)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    h = _lib.Handle(local)
    stream = torch.cuda.Stream(device=dev, priority=-1)   # the library launches on this stream, and so do the timing events
    h.set_stream(stream.cuda_stream)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """`steps` calls of fn between barriers; device time by CUDA events on the library's stream, max over ranks."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        t0 = time.perf_counter()
        n = 0
        for _ in range(steps):
            n += fn()
        e1.record(stream)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        t = torch.tensor([e0.elapsed_time(e1) / 1e3, wall], dtype=torch.float64, device=dev)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        barrier()
        return n, float(t[0].item()), float(t[1].item())

    def mem_available():
        try:
            for ln in open("/proc/meminfo"):
                if ln.startswith("MemAvailable:"):
                    return int(ln.split()[1]) * 1024
        except OSError:
            pass
        return 64 << 30

    avail0 = mem_available()      # before this rank pins anything (all ranks of the box read it at about the same time)
    # ---- corpus: per-rank shard of files (weak scaling: every rank holds `files` files)
    t0 = time.perf_counter()
    n_samp = args.frames * 1152
    pay_bits = PAYLOAD_BITS_PER_FRAME * args.frames
    gen = 500
    pcm_all = torch.empty(args.files * n_samp * 2, dtype=torch.int16, device=dev)
    for w, lo in enumerate(range(0, args.files, gen)):
        hi = min(args.files, lo + gen)
        pcm_all[lo * n_samp * 2: hi * n_samp * 2] = synth_pcm_device(torch, hi - lo, args.frames, 100000 * rank + 1000 + w, dev).reshape(-1)
    torch.cuda.synchronize()
    ns_all = [n_samp] * args.files
    res = h.encode(pcm_all, ns_all, 44100, 320, compact=True)                # decode corpus (setup, untimed)
    off_all = np.concatenate([res["mp3_off"], [res["mp3_off"][-1] + res["out_len"][-1]]]).astype(np.int64)
    mp3_all = res["mp3"]
    mp3_host_all = mp3_all.cpu().pin_memory()
    del res
    pay_all, pay_off_all = random_payload_bits(args.files, pay_bits, 31 * rank + 5)
    total_frames = args.files * args.frames
    mp3_bytes = int(off_all[-1])
    log(f"[rank {rank}] corpus: {args.files} files x {args.frames} frames = {total_frames} frames, "
        f"{mp3_bytes / 1e9:.2f} GB MP3 @320k, {total_frames * 4608 / 1e9:.2f} GB PCM ({time.perf_counter() - t0:.1f}s); host affinity {affinity}")

    file_elems = args.frames * 1152 * 2
    pcm_out_dev = torch.empty(total_frames * 2304 + 64, dtype=torch.int16, device=dev)
    ids_dev = torch.empty(total_frames * 12, dtype=torch.uint8, device=dev)
    bits_dev = torch.empty(total_frames * 12, dtype=torch.uint8, device=dev)
    # ONE pinned arena per rank: the e2e decode leg's PCM output, then the e2e encode leg's PCM input.  Sized to what the box can
    # pin for all its ranks (8 ranks x 31.7 GB does not fit a 251 GB host): the decode leg then runs as several batch calls per
    # step, the encode leg cuts every clip to the frames that fit.
    # what one rank may pin in total: 60 % of the box's available memory shared by its ranks; the MP3 corpus (pinned above), the
    # reveal outputs and configs[4]'s pinned MP3 share come out of it first
    cfg5_reserve = 0 if args.no_extras else int(1.1 * args.cfg5_files * 1148 * 1045 / max(world, 1))
    budget = int(0.6 * avail0 / max(local_world, 1)) - mp3_bytes - 2 * total_frames * 12 - cfg5_reserve
    budget = max(budget, 2 * file_elems * 2)
    if budget < args.files * file_elems * 2:
        budget = 1 << (budget.bit_length() - 1)    # torch's pinned allocator may round a request up to a power of two: ask for one
    arena_files = max(1, min(args.files, (budget - 128) // (file_elems * 2)))
    arena = torch.empty(arena_files * file_elems + 64, dtype=torch.int16, pin_memory=True)
    ids_host = torch.empty(total_frames * 12, dtype=torch.uint8, pin_memory=True)
    bits_host = torch.empty(total_frames * 12, dtype=torch.uint8, pin_memory=True)
    enc_cap = int(_lib.load().m3s_encode_bound(n_samp, 44100, 128)) * args.files + 64
    enc_out_dev = torch.empty(enc_cap, dtype=torch.uint8, device=dev)
    enc_out_host = torch.empty(enc_cap, dtype=torch.uint8, pin_memory=True)
    check = {}

    # ---- host ceiling: what plain cudaMemcpyAsync moves between this host and ALL ranks at once (pinned memory, 1 GiB pieces)
    def host_roof():
        nb = min(arena.numel() * 2, 4 << 30) & ~0xFFFFF
        hb = arena.view(torch.uint8)[:nb]
        db = pcm_out_dev.view(torch.uint8)[:nb]
        hb2 = mp3_host_all[: min(mp3_host_all.numel(), nb // 4)]
        db2 = mp3_all[: hb2.numel()]
        s2 = torch.cuda.Stream(device=dev)
        out = {}

        def run(kind):
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            with torch.cuda.stream(stream):
                if kind in ("d2h", "mix"):
                    hb.copy_(db, non_blocking=True)
                if kind == "h2d":
                    db.copy_(hb, non_blocking=True)
            if kind == "mix":     # the decode leg's mix: PCM down, a quarter as many MP3 bytes up, concurrently
                with torch.cuda.stream(s2):
                    db2.copy_(hb2, non_blocking=True)
                stream.wait_stream(s2)
            e1.record(stream)
            torch.cuda.synchronize()
            t = torch.tensor([e0.elapsed_time(e1) / 1e3], dtype=torch.float64, device=dev)
            if dist is not None:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())

        for kind in ("d2h", "h2d", "mix"):
            run(kind)
            t = min(run(kind) for _ in range(2))
            out[kind + "_gbs"] = world * nb / t / 1e9
        out["bytes_per_rank"] = nb
        out["how"] = ("all ranks at once, one plain pinned cudaMemcpyAsync each, CUDA events, max over ranks, best of 2; "
                      "mix = D2H with a quarter as many bytes H2D alongside (the decode leg's ratio); aggregate GB/s")
        return out

    roof = host_roof()
    log(f"[rank {rank}] host ceiling ({world} ranks at once): D2H {roof['d2h_gbs']:.1f} GB/s, H2D {roof['h2d_gbs']:.1f} GB/s, "
        f"D2H under the decode mix {roof['mix_gbs']:.1f} GB/s")

    last = {}      # the result of each device-resident leg's latest call (for --dump-outputs)

    def dec_device():
        r = h.decode(mp3_all, off_all, pcm=pcm_out_dev, table_ids=ids_dev, reveal_bits=bits_dev, frames_bound=total_frames)
        last["decode"] = r
        check["reveal_bits"] = int(r["reveal_len"].sum())
        return int(r["n_frames"].sum())

    # e2e: ONE m3s_decode call with host buffers per arena-full of files (one call per step when the arena holds the corpus):
    # the library pipelines upload / scan / kernels / download internally, the host thread does nothing else
    def dec_host():
        n = 0
        for lo in range(0, args.files, arena_files):
            hi = min(args.files, lo + arena_files)
            b0, b1 = int(off_all[lo]), int(off_all[hi])
            r = h.decode(mp3_host_all[b0:b1], off_all[lo:hi + 1] - b0, pcm=arena, table_ids=ids_host[12 * lo * args.frames:],
                         reveal_bits=bits_host[12 * lo * args.frames:], frames_bound=(hi - lo) * args.frames)
            n += int(r["n_frames"].sum())
        return n

    # encode+hide: ONE call over all clips (the per-clip offset scan of the rate loop wants every clip's chain in flight together)
    def enc_device():
        r = h.encode(pcm_all, ns_all, 44100, 128, payload_packed=(pay_all, pay_off_all), mp3_out=enc_out_dev)
        last["encode"] = r
        check["hide_off"] = int(r["hide_str_offset"].sum())
        check["enc_bytes"] = int(r["out_len"].sum())
        return total_frames

    enc_e2e = dict(frames=max(1, min(args.frames, (arena.numel() - 64) // (args.files * 2304))))

    def enc_host():
        fe = enc_e2e["frames"]
        h.encode(arena[: args.files * fe * 2304], [fe * 1152] * args.files, 44100, 128, payload_packed=(pay_all, pay_off_all),
                 mp3_out=enc_out_host)
        return args.files * fe

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if "hbm_gbs" in peaks else "B200_PROFILING.md fallback 6650 GB/s (of fallback)"
    DEC_K = ("k_walk", "k_fscan", "k_sideinfo", "k_strip", "k_huff", "k_hybrid")
    ENC_K = ("k_enc_analysis", "k_enc_rate", "k_enc_resolve", "k_enc_emit", "k_enc_pack")

    def measure(dev_fn, host_fn, knames, bpf):
        clocks = ClockSampler(local)   # started in front of the warm-up: nvidia-smi needs a few hundred ms before its first sample
        for _ in range(args.warmup):
            dev_fn()
        h.timing_enable(True)
        l0 = h.launches
        t_w0 = time.time()
        n_dev, t_dev, wall = timed(dev_fn, args.steps)
        t_w1 = time.time()
        launches = h.launches - l0
        kt = h.timing()
        h.timing_enable(False)
        assert n_dev == total_frames * args.steps, (n_dev, total_frames)
        host_fn()
        t_w2 = time.time()
        n_e2e, t_e2e, _ = timed(host_fn, args.steps)
        t_w3 = time.time()
        clk = clocks.stop(t_w0, t_w3)
        clk["timed_windows_s"] = [round(t_w1 - t_w0, 3), round(t_w3 - t_w2, 3)]
        value = world * n_dev / t_dev
        roofl = roofline_of(kt, knames, n_dev, bpf, peak, peak_src, args.steps, value / world * bpf / 1e9 / peak)
        return dict(value=value, ms_per_step=1e3 * t_dev / args.steps, e2e_value=world * n_e2e / t_e2e,
                    e2e_ms=1e3 * t_e2e / args.steps, launches=int(launches), clocks=clk, roofline=roofl, wall=wall)

    if args.only_cfg5:      # diagnostic: configs[4] alone
        c5 = run_cfg5(args, torch, dist, h, stream, dev, rank, world, barrier, timed, pcm_out_dev, arena, ids_dev, bits_dev, ids_host, bits_host)
        if rank == 0:
            emit({"cfg5": c5})
        if dist is not None:
            dist.destroy_process_group()
        return
    D = measure(dec_device, dec_host, DEC_K, DEC_BYTES_PER_FRAME)
    log(f"[rank {rank}] decode+reveal: {D['value']:.4g} frames/s device-resident, {D['e2e_value']:.4g} e2e")
    dump = {}
    if args.dump_outputs and rank == 0:
        dump.update(dump_decode(torch, last["decode"], args.files, args.frames))

    # ---- what the timed decode legs computed, against the oracle (untimed, rank 0): 3 corpus files out of the device-resident
    #      leg's output buffer -- reveal bits equal, int16 PCM within 1 LSB
    parity = {}
    if rank == 0:
        from oracle import oracle as O
        O.build()
        rng = np.random.default_rng(12345)
        pick = sorted(int(i) for i in rng.choice(args.files, size=min(3, args.files), replace=False))
        nf_chk = args.frames                # whole files: the oracle decodes ~3.4 k frames/s
        worst, ok = 0, True
        for i in pick:
            blob = bytes(mp3_host_all[int(off_all[i]):int(off_all[i + 1])].numpy())
            ref = O.decode(blob, 0, taps=False)
            got = pcm_out_dev[i * file_elems: i * file_elems + nf_chk * 2304].cpu().numpy().astype(np.int32)
            d = int(np.abs(got - ref["pcm16"].reshape(-1)[: nf_chk * 2304].astype(np.int32)).max())
            gb = bytes(bits_dev[12 * i * args.frames: 12 * i * args.frames + len(ref["bits"])].cpu().numpy()).decode("ascii")
            worst = max(worst, d)
            ok = ok and d <= 1 and gb == ref["bits"] and ref["n_frames"] == args.frames
        parity["decode"] = dict(files=pick, frames_compared_per_file=nf_chk, max_pcm_lsb=worst, reveal_bits_equal=ok, ok=bool(ok))

    E = None
    if not args.no_encode:
        fe = enc_e2e["frames"]
        arena[: args.files * fe * 2304].view(args.files, fe * 2304).copy_(pcm_all.view(args.files, n_samp * 2)[:, : fe * 2304])
        torch.cuda.synchronize()
        log(f"[rank {rank}] encode e2e leg: {args.files} clips x {fe} frames from pinned host memory ({args.files * fe * 4608 / 1e9:.1f} GB)")
        E = measure(enc_device, enc_host, ENC_K, ENC_BYTES_PER_FRAME)
        log(f"[rank {rank}] encode+hide:   {E['value']:.4g} frames/s device-resident, {E['e2e_value']:.4g} e2e")
        if args.dump_outputs and rank == 0:
            dump.update(dump_encode(torch, last["encode"], args.files))
        if rank == 0:
            from oracle import oracle as O
            rng = np.random.default_rng(777)
            pick = sorted(int(i) for i in rng.choice(args.files, size=min(3, args.files), replace=False))
            nf_chk = min(args.frames, 1500)
            ok = True
            for i in pick:     # a clip's first frames encode identically whatever follows (no look-ahead, reservoir off): A.E7
                wav = pcm_all[i * n_samp * 2: i * n_samp * 2 + nf_chk * 2304].cpu().numpy().reshape(-1, 2)
                bits = pay_all[int(pay_off_all[i]):int(pay_off_all[i + 1])].tobytes().decode("ascii")
                ref = O.encode(wav, 44100, 128, bits, taps=False)
                mo = int(_lib.load().m3s_encode_bound(n_samp, 44100, 128)) * i
                nbytes = (len(ref["mp3"]) // 4 - 1) * 4          # the oracle's last word may be a partial flush (A.E8)
                got = bytes(enc_out_dev[mo: mo + nbytes].cpu().numpy())
                ok = ok and got == ref["mp3"][:nbytes]
            parity["encode"] = dict(clips=pick, frames_compared_per_clip=nf_chk, bytes_equal=bool(ok), ok=bool(ok))
    if dump:
        write_dump(args.dump_outputs, dump)

    # ---- composites (SURVEY 8f row 1): hide_message / clear_file for a batch, decode (float64) -> int16 in HBM -> encode
    comp = None
    if not args.no_extras:
        n_c, f_c = min(args.files, 256), min(args.frames, 689)
        # the first f_c frames of file i: reference-encoder frames are self-contained (main_data_begin = 0), so a file cut at a frame
        # boundary is a valid file; every file of the corpus has the same frame positions (same padding recurrence)
        b1 = int(off_all[1])
        h.decode_scan(mp3_host_all[:b1], [0, b1])
        cut = int(h.decode_frame_pos()[f_c]) if f_c < args.frames else b1
        blobs = [bytes(mp3_host_all[int(off_all[i]): int(off_all[i]) + cut].numpy()) for i in range(n_c)]
        msgs = ["".join(chr(32 + (7 * i + 3 * k) % 95) for k in range(40)) for i in range(n_c)]
        cs = max(1, args.steps)
        batch.hide_batch(h, blobs, msgs)      # warm-up
        barrier()
        t0 = time.perf_counter()
        for _ in range(cs):
            out_h, too = batch.hide_batch(h, blobs, msgs)
        torch.cuda.synchronize()
        t_hide = (time.perf_counter() - t0) / cs
        t0 = time.perf_counter()
        for _ in range(cs):
            out_c = batch.clear_batch(h, out_h)
        torch.cuda.synchronize()
        t_clear = (time.perf_counter() - t0) / cs
        rev = batch.reveal_batch(h, out_h[:8])
        comp = dict(clips=n_c, frames_per_clip=f_c, hide_frames_per_s=n_c * f_c / t_hide, clear_frames_per_s=n_c * f_c / t_clear,
                    unit="frames/s", timing="host wall clock around batch.hide_batch / clear_batch (bytes in -> bytes out, one GPU)",
                    roundtrip_ok=bool(rev == msgs[:8] and not any(too)), cleared_reveal_empty=bool(batch.reveal_batch(h, out_c[:4]) == [""] * 4))

    # ---- configs[4]: 10,000 x 30-s tracks strong-scaled by file over the ranks + one long file split by frame range
    cfg5 = None
    if not args.no_extras:
        cfg5 = run_cfg5(args, torch, dist, h, stream, dev, rank, world, barrier, timed, pcm_out_dev, arena, ids_dev, bits_dev, ids_host, bits_host)

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---- CPU baseline: the oracle port on one host core over a bounded sample of the same kind of corpus, and the Python reference
    port = CpuPort(min(args.frames, 6890), 1, 3 if args.frames >= 2000 else 1)
    cb = port.step()
    ncore = os.cpu_count()
    pyref = python_reference_timing() if not args.no_extras else {"unavailable": "--no-extras"}

    def cpu_obj(key, what, pykey):
        f, t = cb[key]
        o = {"value": f / t, "unit": "frames/s", "cores": 1, "kind": "port",
             "sample": f"{what} of {f} frames (tone+noise clips of {min(args.frames, 6890)} frames), oracle/mp3stego_oracle.c, "
                       f"1 thread of {ncore} host cores, {t:.1f} s"}
        if isinstance(pyref, dict) and pykey in pyref:
            o["python_reference"] = dict(pyref[pykey], kind="reference", cores=1, numba=pyref.get("numba"))
            if "configs0_test_mp3" in pyref and key == "decode":
                o["python_reference_test_mp3"] = dict(pyref["configs0_test_mp3"], kind="reference", cores=1)
        else:
            o["python_reference"] = pyref
        return o

    d2h = int(total_frames * (1152 * 2 * 2 + 24))
    e2e_d2h_gbs = D["e2e_value"] * (1152 * 2 * 2 + 24) / 1e9
    line = {"metric": "decode+reveal throughput (MP3 frames/s)", "value": D["value"], "unit": "frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": D["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": corpus_config(args),
            "audio_seconds_per_s": D["value"] * 1152 / 44100.0,
            "e2e": {"value": D["e2e_value"], "unit": "frames/s", "h2d_bytes_per_step": mp3_bytes,
                    "d2h_bytes_per_step": d2h, "ms_per_step": D["e2e_ms"],
                    "calls_per_step": (args.files + arena_files - 1) // arena_files,
                    "api": "one m3s_decode call (host buffers) per pinned-arena-full of files; pipelined inside the library",
                    "host_roof_gbs": roof, "d2h_gbs": e2e_d2h_gbs, "roof_frac": e2e_d2h_gbs / roof["mix_gbs"], "host_affinity": affinity},
            "gpu_launches": D["launches"] + (E["launches"] if E else 0), "clocks": D["clocks"], "roofline": D["roofline"],
            "cpu_baseline": cpu_obj("decode", "decode+reveal @320k", "decode_reveal"),
            "check": dict(check, parity_sampled=bool(parity and all(v["ok"] for v in parity.values())), parity=parity)}
    if E:
        enc_h2d = int(args.files * enc_e2e["frames"] * 4608 + len(pay_all))
        line["encode_hide"] = {
            "metric": "encode+hide throughput (MP3 frames/s)", "value": E["value"], "unit": "frames/s", "dtype": "int32",
            "ms_per_step": E["ms_per_step"], "audio_seconds_per_s": E["value"] * 1152 / 44100.0,
            "e2e": {"value": E["e2e_value"], "unit": "frames/s", "h2d_bytes_per_step": enc_h2d,
                    "d2h_bytes_per_step": int(check.get("enc_bytes", 0) * enc_e2e["frames"] / args.frames), "ms_per_step": E["e2e_ms"],
                    "clips": args.files, "frames_per_clip": enc_e2e["frames"],
                    "h2d_gbs": E["e2e_value"] * 4608 / 1e9, "roof_frac": E["e2e_value"] * 4608 / 1e9 / roof["h2d_gbs"]},
            "gpu_launches": E["launches"], "clocks": E["clocks"], "roofline": E["roofline"],
            "cpu_baseline": cpu_obj("encode", "encode+hide @128k", "encode_hide")}
    if comp:
        line["composite"] = comp
    if cfg5:
        line["cfg5"] = cfg5
    emit(line)
    if dist is not None:
        dist.destroy_process_group()


def run_cfg5(args, torch, dist, h, stream, dev, rank, world, barrier, timed, pcm_out_dev, arena, ids_dev, bits_dev, ids_host, bits_host):
    """BASELINE configs[4]: a FIXED corpus of `--cfg5-files` tracks of 1,148 frames (30 s) partitioned by file over the ranks
    (shard.partition_files: greedy by size, no communication) plus ONE long file of `--cfg5-long` frames split by frame range
    over the ranks (shard.plan_frame_shard + m3s_decode_run_range: whole-file scan on every rank, one warm-up frame and the <= 9
    frames of bit reservoir cut on the device).  Strong scaling: total work is fixed; value = total frames / max-over-ranks time.
    efficiency = value / (world x the rate rank 0 reaches on its share while the other ranks idle), measured in the same run."""
    from mp3stego_b200 import _lib, shard
    NF = 1148
    n_files = args.cfg5_files
    n_samp = NF * 1152
    size_1 = int(_lib.load().m3s_encode_size(n_samp, 44100, 320))
    mine = shard.partition_files([size_1] * n_files, world)[rank]
    # the rank's tracks, seeded by GLOBAL track index (the corpus does not depend on the number of ranks)
    t0 = time.perf_counter()
    chunks, offs = [], [0]
    gen = 500
    for lo in range(0, len(mine), gen):
        idx = mine[lo:lo + gen]
        pcm = torch.empty(len(idx) * n_samp * 2, dtype=torch.int16, device=dev)
        for k, gi in enumerate(idx):
            pcm[k * n_samp * 2:(k + 1) * n_samp * 2] = synth_pcm_device(torch, 1, NF, 5_000_000 + gi, dev).reshape(-1)
        r = h.encode(pcm, [n_samp] * len(idx), 44100, 320, compact=True)
        end = int(r["mp3_off"][-1] + r["out_len"][-1])      # compact layout: the files lie back to back
        chunks.append(r["mp3"][:end].clone())
        base = offs[-1]
        offs.extend((np.asarray(r["mp3_off"][1:], np.int64) + base).tolist())
        offs.append(base + end)
        del pcm, r
    mp3 = torch.cat(chunks) if chunks else torch.empty(0, dtype=torch.uint8, device=dev)
    off = np.asarray(offs, np.int64)
    del chunks
    frames_mine = len(mine) * NF
    mp3_host = mp3.cpu().pin_memory()
    steps = max(1, args.steps)
    cap_files = max(1, (pcm_out_dev.numel() - 64) // (n_samp * 2))
    cap_host = max(1, (arena.numel() - 64) // (n_samp * 2))

    def dec(mp3_t, out, ids, bits, cap):
        n = 0
        for lo in range(0, len(mine), cap):
            hi = min(len(mine), lo + cap)
            b0, b1 = int(off[lo]), int(off[hi])
            r = h.decode(mp3_t[b0:b1], off[lo:hi + 1] - b0, pcm=out, table_ids=ids, reveal_bits=bits, frames_bound=(hi - lo) * NF)
            n += int(r["n_frames"].sum())
        return n

    dev_fn = lambda: dec(mp3, pcm_out_dev, ids_dev, bits_dev, cap_files)          # noqa: E731
    host_fn = lambda: dec(mp3_host, arena, ids_host, bits_host, cap_host)        # noqa: E731
    dev_fn()
    # solo: rank 0 works on its share alone (the other ranks wait) -> the rate one GPU reaches without neighbours
    solo = torch.zeros(2, dtype=torch.float64, device=dev)
    barrier()
    if rank == 0:
        for k, fn in enumerate((dev_fn, host_fn)):
            fn()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            n = fn()
            e1.record(stream)
            torch.cuda.synchronize()
            solo[k] = n / (e0.elapsed_time(e1) / 1e3)
    if dist is not None:
        dist.broadcast(solo, 0)
    n_dev, t_dev, _ = timed(dev_fn, steps)
    host_fn()
    n_e2e, t_e2e, _ = timed(host_fn, steps)
    tot = torch.tensor([n_dev, n_e2e], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(tot)
    value, e2e_value = float(tot[0]) / t_dev, float(tot[1]) / t_e2e
    # sampled parity of the track corpus against the oracle (rank 0, untimed): 2 tracks of its shard, out of the device output
    parity_tracks = None
    if rank == 0 and len(mine):
        from oracle import oracle as O
        lo_call = (len(mine) - 1) // cap_files * cap_files        # the output buffer holds the LAST call's files
        ok, worst, note = True, 0, None
        for k in (lo_call, len(mine) - 1):
            blob = bytes(mp3_host[int(off[k]):int(off[k + 1])].numpy())
            ref = O.decode(blob, 0, taps=False)
            got = pcm_out_dev[(k - lo_call) * n_samp * 2:(k - lo_call + 1) * n_samp * 2].cpu().numpy().astype(np.int32)
            if ref["n_frames"] != NF:
                ok, note = False, f"oracle parsed {ref['n_frames']} frames of track {k} ({len(blob)} bytes, head {blob[:4].hex()})"
                continue
            d = int(np.abs(got - ref["pcm16"].reshape(-1).astype(np.int32)).max())
            worst = max(worst, d)
            ok = ok and d <= 1
        parity_tracks = dict(tracks=[int(mine[lo_call]), int(mine[-1])], max_pcm_lsb=worst, ok=bool(ok))
        if note:
            parity_tracks["note"] = note
    del mp3, mp3_host

    # ---- the long file: every rank holds the same bytes (generated from the same seed), scans all of it, decodes its range
    LF = args.cfg5_long
    pcm = synth_pcm_device(torch, 1, LF, 9_999_999, dev).reshape(-1)
    r = h.encode(pcm, [LF * 1152], 44100, 320, compact=True)
    blob = r["mp3"][: int(r["out_len"][0])].clone()
    del pcm, r
    plan = shard.plan_frame_shard(LF, 0, rank, world)
    out = pcm_out_dev[: (plan["count"] + 1) * 2304]

    def long_fn():
        part = shard.decode_frame_range(h, blob, rank, world, pcm=out)
        return part["count"]

    long_fn()
    n_l, t_l, _ = timed(long_fn, steps)
    part = shard.decode_frame_range(h, blob, rank, world, pcm=out)
    mysum = pcm_checksum(torch, part["pcm"].reshape(-1), plan["first"] * 2304) + (part["first"], part["count"], len(part["bits"]))
    sums = [mysum]
    if dist is not None:
        sums = [None] * world
        dist.all_gather_object(sums, mysum)
    tl = torch.tensor([n_l], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(tl)
    long_ok, long_oracle = None, None
    if rank == 0:
        sc = h.decode_scan(blob, [0, blob.numel()])
        _, wbits = h.decode_reveal()
        whole = torch.empty(int(sc["pcm_rows"][0]) * 2, dtype=torch.int16, device=dev)
        h.decode_run(pcm=whole)
        long_ok = int(sc["n_frames"][0]) == LF and sum(s[3] for s in sums) == LF and sum(s[4] for s in sums) == len(wbits[0])
        for s_, p_ in zip(sums, [shard.plan_frame_shard(LF, 0, r_, world) for r_ in range(world)]):
            ref = pcm_checksum(torch, whole[p_["first"] * 2304:(p_["first"] + p_["count"]) * 2304], p_["first"] * 2304)
            long_ok = long_ok and ref == (s_[0], s_[1]) and s_[2] == p_["first"] and s_[3] == p_["count"]
        from oracle import oracle as O            # and the whole-file decode itself against the oracle on a 1,200-frame cut in the middle
        pos = h.decode_frame_pos()
        mid = LF // 2
        cut = bytes(blob[int(pos[mid]):int(pos[mid + 1200])].cpu().numpy())
        ref = O.decode(cut, 0, taps=False)
        got = whole[(mid + 1) * 2304:(mid + 1200) * 2304].cpu().numpy().astype(np.int32)     # frame 0 of the cut lacks its history
        long_oracle = int(np.abs(got - ref["pcm16"].reshape(-1)[2304:].astype(np.int32)).max())
        long_ok = bool(long_ok and long_oracle <= 1)
        del whole
    return {"workload": f"configs[4]: {n_files} tracks x {NF} frames partitioned by file over {world} rank(s) + one {LF}-frame file split by frame range",
            "scaling": "strong", "value": value, "unit": "frames/s", "ms_per_step": 1e3 * t_dev / steps, "steps": steps,
            "e2e": {"value": e2e_value, "unit": "frames/s", "ms_per_step": 1e3 * t_e2e / steps},
            "solo_rate_per_gpu": {"value": float(solo[0]), "e2e": float(solo[1])},
            "efficiency": value / (world * float(solo[0])) if float(solo[0]) > 0 else None,
            "e2e_efficiency": e2e_value / (world * float(solo[1])) if float(solo[1]) > 0 else None,
            "files_per_rank": len(mine), "frames_per_rank": frames_mine,
            "long_file": {"frames": LF, "value": float(tl) / t_l, "unit": "frames/s", "ms_per_step": 1e3 * t_l / steps,
                          "what": "per step every rank: whole-file scan (D0 + D4) + Huffman / synthesis of its frame range + 1 warm-up frame, device-resident",
                          "range_checksums_equal_whole_file": long_ok, "whole_file_vs_oracle_max_lsb": long_oracle},
            "parity_tracks": parity_tracks,
            "parity_ok": bool((long_ok if long_ok is not None else True) and (parity_tracks["ok"] if parity_tracks else True))}


_REAL_STDOUT = None


def quiet_stdout():
    """Libraries (NCCL's version banner, the compiler) write to fd 1; the contract is ONE JSON line there.  Everything but
    emit() goes to stderr from here on."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--files", type=int, default=1000, help="files per GPU")
    ap.add_argument("--frames", type=int, default=FRAMES_PER_FILE, help="frames per file")
    ap.add_argument("--no-encode", action="store_true", help="skip the encode+hide half")
    ap.add_argument("--no-extras", action="store_true", help="skip cfg5, the composites and the Python-reference timing")
    ap.add_argument("--only-cfg5", action="store_true", help="diagnostic: run configs[4] alone")
    ap.add_argument("--cfg5-files", type=int, default=10000, help="tracks of the strong-scaled configs[4] corpus (whole job)")
    ap.add_argument("--cfg5-long", type=int, default=60000, help="frames of the long file split by frame range")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the device-resident decode and encode legs returned in "
                    "their last timed step to DIR/<name>.npy (rank 0; a seeded sample of the large buffers, <= 64 MiB)")
    args = ap.parse_args()
    quiet_stdout()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_product_arm(args)


if __name__ == "__main__":
    main()
