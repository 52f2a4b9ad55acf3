"""Seeded encode edge corpus: int16 stereo clips that drive the encoder's rate loop and bit writer to their edges.

extreme_clips(seed) -> (corpus, overrun).  Each clip is a dict(name, pcm [n, 2] int16, sr, br, bits) with `bits` the payload
('0'/'1' chars, '' = plain encode).  The corpus spreads these families over all 3 sample rates x 14 bitrates:

  nyq{1,2,4}   Nyquist-rate squares at full (+32767 / -32768), half and quarter scale
  hf           sines at 15..21 kHz (below each rate's Nyquist frequency), random amplitude
  dc / steps   DC at -32768 and +32767, and jumps between the two (INT_MIN and the analysis kernel's correction pass)
  imp / lsb    isolated -32768 impulses in silence; sparse 1-LSB patterns (big_values 0 with count1 > 0)
  noise        full-scale white noise
  gate         granules that alternate loud and silent (stale address1..3, SURVEY A.E6; the scfsi conditions)
  tone         the tone+noise clip of SURVEY 8(d)

with payloads: none, all '0', all '1', short ones that run out inside a granule, and ones longer than the capacity; and
lengths of 1 and 2 frames, a few of several hundred frames, and one (sample rate, bitrate) batch with 320 one-frame clips
(k_enc_resolve runs one warp per clip).  About 3,000 frames in all.

`overrun` holds clips whose step search runs past the end of the reference's step table (SURVEY A.E13): loud
high-frequency input at 32 kbps and 44.1 / 48 kHz.  The encoder has no defined output for them; they are kept apart.
The loud high-frequency families therefore meet 32 kbps only at 32 kHz (tests/test_encode_extremes.py asserts that no
clip of the corpus overruns and every clip of `overrun` does)."""
import numpy as np

SAMPLE_RATES = (32000, 44100, 48000)
BITRATES = (32, 40, 48, 56, 64, 80, 96, 112, 128, 160, 192, 224, 256, 320)
GRANULE = 576
FRAME = 1152


def nyquist(n, hi, lo):
    x = np.where(np.arange(n) % 2 == 0, hi, lo).astype(np.int16)
    return np.stack([x, x], axis=1)


def sine(n, sr, f, amp, phase=0.0):
    t = np.arange(n) / sr
    x = np.clip(np.round(amp * np.sin(2 * np.pi * f * t + phase)), -32768, 32767).astype(np.int16)
    return np.stack([x, -x if amp < 32767 else x], axis=1)


def tone_noise(rng, n, sr):
    t = np.arange(n) / sr
    f = rng.uniform(100, 5000, size=2)
    x = np.stack([0.4 * np.sin(2 * np.pi * f[c] * t) + 0.05 * rng.standard_normal(n) for c in range(2)], axis=1)
    return (x * 32767).astype(np.int16)


def _family(rng, fam, n, sr):
    if fam == "nyq1":
        return nyquist(n, 32767, -32768)
    if fam == "nyq2":
        return nyquist(n, 16384, -16384)
    if fam == "nyq4":
        return nyquist(n, 8192, -8192)
    if fam == "hf":
        f = rng.uniform(15000, min(21000, sr / 2 - 200))
        return sine(n, sr, f, rng.choice([32767, 24000, 16000, 6000]), rng.uniform(0, 6.28))
    if fam == "dc":
        v = -32768 if rng.integers(2) else 32767
        return np.full((n, 2), v, np.int16)
    if fam == "steps":   # runs of -32768 / +32767 of random length (some shorter than a subband slot)
        x = np.empty(n, np.int16)
        i, v = 0, -32768
        while i < n:
            k = int(rng.choice([1, 3, 31, 200, 700]))
            x[i:i + k] = v
            v = 32767 if v < 0 else -32768
            i += k
        return np.stack([x, x[::-1].copy()], axis=1)
    if fam == "imp":
        y = np.zeros((n, 2), np.int16)
        idx = rng.choice(n, size=max(1, n // 900), replace=False)
        y[idx, rng.integers(0, 2, size=idx.size)] = -32768
        return y
    if fam == "lsb":
        y = np.zeros((n, 2), np.int16)
        m = rng.random((n, 2)) < rng.choice([0.002, 0.02, 0.3])
        y[m] = rng.choice(np.array([-1, 1], np.int16), size=int(m.sum()))
        return y
    if fam == "noise":
        return rng.integers(-32768, 32768, size=(n, 2)).astype(np.int16)
    if fam == "gate":   # every granule loud or silent at random, loud ones from a loud family
        base = _family(rng, str(rng.choice(["noise", "tone", "nyq4", "steps"])), n, sr)
        on = np.repeat(rng.random(n // GRANULE + 1) < 0.5, GRANULE)[:n]
        return np.where(on[:, None], base, 0).astype(np.int16)
    if fam == "tone":
        return tone_noise(rng, n, sr)
    raise ValueError(fam)


FAMILIES = ("nyq1", "nyq2", "nyq4", "hf", "dc", "steps", "imp", "lsb", "noise", "gate", "tone")
LOUD_HF = ("nyq1", "nyq2", "hf")   # the families that can overrun the step table at 32 kbps, 44.1 / 48 kHz


def _payload(rng, kind, n_frames):
    if kind == "none":
        return ""
    if kind == "zeros":
        return "0" * (12 * n_frames + 8)
    if kind == "ones":
        return "1" * (12 * n_frames + 8)
    if kind == "short":     # runs out early: the granule that meets the end has 1, 2 or 3 bits left
        return "".join(rng.choice(["0", "1"], size=int(rng.integers(1, 12 * n_frames + 2))))
    if kind == "long":      # more than the 12 table ids a frame can carry
        return "".join(rng.choice(["0", "1"], size=12 * n_frames + 100))
    raise ValueError(kind)


PAYLOADS = ("none", "zeros", "ones", "short", "long")


def extreme_clips(seed=0):
    rng = np.random.default_rng(seed)
    corpus = []

    def add(fam, sr, br, n_frames, pay):
        n = n_frames * FRAME
        corpus.append(dict(name=f"{fam}_{sr}_{br}_{n_frames}f_{pay}_{len(corpus)}", pcm=_family(rng, fam, n, sr), sr=sr, br=br,
                           bits=_payload(rng, pay, n_frames)))

    k = 0
    for sr in SAMPLE_RATES:
        for br in BITRATES:
            fams = [f for f in FAMILIES if not (f in LOUD_HF and br == 32 and sr != 32000)]
            # every family at every rate pair, 1 or 2 frames, the payload kinds in turn
            for f in fams:
                add(f, sr, br, 1 + int(rng.integers(2)), PAYLOADS[k % len(PAYLOADS)])
                k += 1
            # one longer clip of a random family per rate pair
            add(str(rng.choice(fams)), sr, br, int(rng.integers(10, 26)), PAYLOADS[k % len(PAYLOADS)])
            k += 1
    # several hundred frames: quiet / loud changes, and the stuffing spread of full-scale Nyquist at 32 kHz / 320k, over long runs
    for sr, br, fam in ((44100, 128, "gate"), (48000, 320, "tone"), (32000, 64, "lsb"), (32000, 320, "nyq1")):
        add(fam, sr, br, 300, "short" if fam == "tone" else "long")
    # one batch of 320 one-frame clips at one rate pair (one k_enc_resolve warp per clip)
    for i in range(320):
        add(FAMILIES[i % len(FAMILIES)], 44100, 160, 1, PAYLOADS[i % len(PAYLOADS)])

    n6 = 6 * FRAME
    overrun = [
        dict(name="nyq1_44100_32", pcm=nyquist(n6, 32767, -32768), sr=44100, br=32, bits=""),
        dict(name="nyq1_48000_32", pcm=nyquist(n6, 32767, -32768), sr=48000, br=32, bits="01" * 40),
        dict(name="nyq2_44100_32", pcm=nyquist(n6, 16384, -16384), sr=44100, br=32, bits="1" * 30),
        dict(name="nyq2_48000_32", pcm=nyquist(n6, 16384, -16384), sr=48000, br=32, bits=""),
        dict(name="sine20k_48000_32", pcm=sine(n6, 48000, 20000, 32767), sr=48000, br=32, bits="0" * 50),
        dict(name="sine21k_44100_32", pcm=sine(n6, 44100, 21000, 16000), sr=44100, br=32, bits=""),
    ]
    return corpus, overrun


def by_rate(clips):
    """{(sr, br): [clip, ...]} in corpus order."""
    out = {}
    for c in clips:
        out.setdefault((c["sr"], c["br"]), []).append(c)
    return out
