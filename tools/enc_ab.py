"""A/B timing of the encoder pipeline variants on one GPU (diagnostic; no JSON contract).
usage: python tools/enc_ab.py [clips] [frames]   -- device-resident encode+hide @128k of the tone+noise corpus under each
environment setting of m3s_encode (M3S_ENC_CHAIN, M3S_ENC_SERIAL / M3S_ENC_OVERLAP, M3S_PROBE_CTAS, M3S_PROBE_CFG), per-kernel device milliseconds."""
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
import __graft_entry__ as ge  # noqa: E402


def main():
    clips = int(sys.argv[1]) if len(sys.argv) > 1 else 1000
    frames = int(sys.argv[2]) if len(sys.argv) > 2 else 1378
    ge.build()
    from mp3stego_b200 import _lib
    dev = torch.device("cuda", 0)
    h = _lib.Handle(0)
    n_samp = frames * 1152
    pcm = torch.empty(clips * n_samp * 2, dtype=torch.int16, device=dev)
    for lo in range(0, clips, 250):
        hi = min(clips, lo + 250)
        pcm[lo * n_samp * 2: hi * n_samp * 2] = bench.synth_pcm_device(torch, hi - lo, frames, 1000 + lo, dev).reshape(-1)
    pay, pay_off = bench.random_payload_bits(clips, bench.PAYLOAD_BITS_PER_FRAME * frames, 5)
    cap = int(_lib.load().m3s_encode_bound(n_samp, 44100, 128)) * clips + 64
    out = torch.empty(cap, dtype=torch.uint8, device=dev)
    ns = [n_samp] * clips
    configs = [("default", {}), ("overlap", {"M3S_ENC_OVERLAP": "1"}), ("probe_ctas=296", {"M3S_PROBE_CTAS": "296"}), ("probe_ctas=444", {"M3S_PROBE_CTAS": "444"}),
               ("serial", {"M3S_ENC_SERIAL": "1"}), ("chain (old rate loop)", {"M3S_ENC_CHAIN": "1"}),
               ("chain serial", {"M3S_ENC_CHAIN": "1", "M3S_ENC_SERIAL": "1"})]
    configs += [(f"cfg{k} serial", {"M3S_PROBE_CFG": str(k), "M3S_ENC_SERIAL": "1"}) for k in range(3)]   # configurations 0..2 exist
    if len(sys.argv) > 3:   # only the named configurations; "env:A=1,B=2" adds an ad-hoc one
        adhoc = [(a[4:], dict(kv.split("=") for kv in a[4:].split(","))) for a in sys.argv[3:] if a.startswith("env:")]
        configs = [c for c in configs if any(c[0].startswith(a) for a in sys.argv[3:])] + adhoc
    ref = None
    for name, env in configs:
        for k in ("M3S_PROBE_CTAS", "M3S_ENC_SERIAL", "M3S_ENC_OVERLAP", "M3S_ENC_CHAIN", "M3S_PROBE_CFG", "M3S_ENC_ANALYSIS_DIRECT", "M3S_ENC_FOLD_CFG"):
            os.environ.pop(k, None)
        os.environ.update(env)
        out.zero_()
        r = h.encode(pcm, ns, 44100, 128, payload_packed=(pay, pay_off), mp3_out=out)   # warm-up
        sig = (int(r["hide_str_offset"].sum()), int(out[: int(r["out_len"].sum())].to(torch.int64).sum().item()))
        if ref is None:
            ref = sig
        h.timing_enable(True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(2):
            h.encode(pcm, ns, 44100, 128, payload_packed=(pay, pay_off), mp3_out=out)
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / 2
        kt = h.timing()
        h.timing_enable(False)
        ks = ", ".join(f"{k} {v[0] / 2:.1f}" for k, v in sorted(kt.items()) if k.startswith("k_enc") and v[1])
        print(f"{name:24s} {dt * 1e3:8.1f} ms/pass = {clips * frames / dt / 1e6:6.2f} M frames/s  same_output={sig == ref}  [{ks}]", flush=True)


if __name__ == "__main__":
    main()
