"""numpy restatement of mr_device_permutations (mobrob_b200/csrc/ppo.cu: 6-round Feistel network on the
enclosing power-of-two domain, cycle-walked into [0, n)) -- integer work, so the CUDA kernel must match
it bit for bit.  This is the repo's own algorithm (the reference draws np.random.permutation on the
host; PPO(permutation="sb3") keeps that stream), restated only for the test."""
import numpy as np

M64 = (1 << 64) - 1


def round_keys(seed: int, stream: int):
    x = (seed ^ ((stream * 0xD1342543DE82EF95 + 0x2545F4914F6CDD1D) & M64)) & M64
    ks = []
    for _ in range(3):   # splitmix64, two 32-bit round keys per output
        x = (x + 0x9E3779B97F4A7C15) & M64
        z = x
        z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
        z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
        z ^= z >> 31
        ks += [z & 0xFFFFFFFF, z >> 32]
    return ks


def _round(x, k):
    u = np.uint32
    x = x ^ u(k)
    x = x * u(0x9E3779B1); x ^= x >> u(16)
    x = x * u(0x85EBCA6B); x ^= x >> u(13)
    x = x * u(0xC2B2AE35); x ^= x >> u(16)
    return x


def _feistel(x, ks, bits):
    u = np.uint32
    lb = bits >> 1
    rb = bits - lb
    L, R = x >> u(rb), x & u((1 << rb) - 1)
    wl, wr = lb, rb
    for r in range(6):
        f = _round(R, ks[r]) & u((1 << wl) - 1)
        L, R = R, L ^ f
        wl, wr = wr, wl
    return (L << u(wr)) | R


def device_permutation(seed: int, stream: int, n: int) -> np.ndarray:
    bits = 2
    while (1 << bits) < n:
        bits += 1
    ks = round_keys(seed, stream)
    with np.errstate(over="ignore"):
        x = _feistel(np.arange(n, dtype=np.uint32), ks, bits)
        bad = x >= n
        while bad.any():
            x[bad] = _feistel(x[bad], ks, bits)
            bad = x >= n
    return x.astype(np.int64)
