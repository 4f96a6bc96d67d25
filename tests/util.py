import hashlib
import json
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
REFERENCE_DIGESTS = os.path.join(GOLDEN, "reference_digests.json")


def digest(a):
    """SHA-256 (first 128 bits) of an array's dtype, shape and bits, with -0.0 counted as +0.0 like same_bits: two
    arrays have the same digest exactly when they are equal bit for bit up to the sign of zero."""
    a = np.ascontiguousarray(a)
    if a.dtype.kind == "f":
        a = a + a.dtype.type(0)
    return hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).hexdigest()[:32]


def reference_digests():
    """What the compiled, unmodified reference returned for the inputs of the tests that compare with it
    (tests/golden/make_golden.py writes the file)."""
    with open(REFERENCE_DIGESTS) as f:
        return json.load(f)


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.int32)


def same_bits(a, b):
    """float arrays equal bit for bit (distinguishes nothing but +-0, which compare equal by value)."""
    a = np.asarray(a, np.float32)
    b = np.asarray(b, np.float32)
    return a.shape == b.shape and bool(np.all((bits(a) == bits(b)) | ((a == 0) & (b == 0))))


def edge_signals(n_frames=24, scale=1.0):
    """Edge-case single-stream inputs the reference never tests itself (SURVEY.md 8c(3))."""
    T = n_frames * 480
    t = np.arange(T) / 48000.0
    rng = np.random.RandomState(11)
    sig = {}
    sig["zeros"] = np.zeros(T, np.float32)
    imp = np.zeros(T, np.float32); imp[2000] = 0.9
    sig["impulse"] = imp
    sig["sine62"] = (0.8 * np.sin(2 * np.pi * 62.5 * t)).astype(np.float32)    # period 768 = PITCH_MAX_PERIOD
    sig["sine800"] = (0.8 * np.sin(2 * np.pi * 800.0 * t)).astype(np.float32)   # period 60  = PITCH_MIN_PERIOD
    h = np.zeros(T)
    for k, a in ((1, 0.3), (2, 1.0), (3, 0.2), (4, 0.8), (6, 0.5)):            # octave-ambiguous stack (doubling logic)
        h += a * np.sin(2 * np.pi * 110.0 * k * t + 0.3 * k)
    sig["octave"] = (0.25 * h / np.abs(h).max()).astype(np.float32)
    sig["noise"] = (0.1 * rng.randn(T)).astype(np.float32)
    sig["fullscale_sq"] = np.sign(np.sin(2 * np.pi * 150.0 * t)).astype(np.float32) * 0.999
    sw = np.sin(2 * np.pi * (80.0 * t + 160.0 * t * t))                        # chirp 80 -> 400 Hz/s
    sig["chirp"] = (0.5 * sw).astype(np.float32)
    return {k: (v * np.float32(scale)).astype(np.float32) for k, v in sig.items()}


def random_mixtures(n_streams, n_frames, seed=2025, max_log_amp=0.0):
    """Seeded random streams: harmonic stacks + noise + DC + exact-silence gaps + clicks at log-uniform amplitudes
    in [1e-4, 10**max_log_amp] (the same family the CPU property test draws from)."""
    T = n_frames * 480
    t = np.arange(T) / 48000.0
    out = np.empty((n_streams, T), np.float32)
    for s in range(n_streams):
        rng = np.random.RandomState(seed + s)
        f0, noise, dc = 55.0 + 845.0 * rng.rand(), rng.rand(), 0.4 * rng.rand() - 0.2
        x = np.zeros(T)
        for h in range(1, 9):
            x += rng.rand() * np.sin(2 * np.pi * f0 * h * t + rng.rand() * 6.28) / h
        x = x / (np.abs(x).max() + 1e-9) * (1 - noise) + noise * rng.randn(T) * 0.3 + dc
        gap = rng.randint(0, 9)
        if gap:
            g0 = rng.randint(0, n_frames - gap + 1) * 480
            x[g0:g0 + gap * 480] = 0.0
        if rng.rand() < 0.5:
            x[rng.randint(0, T)] += 3.0
        out[s] = (x * 10.0 ** (-4.0 + (4.0 + max_log_amp) * rng.rand())).astype(np.float32)
    return out
