"""oracle/rng_numpy.py — TEST INFRASTRUCTURE ONLY: numpy restatement of the random stream of seeded sampling
(summertts_b200/csrc/rng.cuh, DESIGN.md §12).

Philox4x32-10 (Salmon et al., SC'11; Random123's round function and constants) keyed by the utterance's 64-bit seed,
and Box-Muller normals from its words in float32:
    u1 = ((x0 >> 8) + 1) 2^-24,  u2 = (x1 >> 8) 2^-24,  r = sqrt(-2 ln u1),  (n0, n1) = (r cos 2 pi u2, r sin 2 pi u2)
and (x2, x3) -> (n2, n3) the same way.  Counters:
    prior  (frame f, channel quad q, 0, 0) -> channels 4q .. 4q+3
    SDP    (token t, 0, 1, 0)              -> words 0 / 1 = eps_0(t) / eps_1(t)
"""
from __future__ import annotations

import numpy as np

M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
W0, W1 = np.uint32(0x9E3779B9), np.uint32(0xBB67AE85)
MASK = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, seed):
    """ctr: [N, 4] uint32 counters; seed: 64-bit key (lo word = key 0). Returns [N, 4] uint32."""
    c = [np.asarray(ctr, np.uint32)[:, i].astype(np.uint64) for i in range(4)]
    seed = int(seed) & (2 ** 64 - 1)
    k0, k1 = np.uint32(seed & 0xFFFFFFFF), np.uint32(seed >> 32)
    for _ in range(10):
        p0, p1 = M0 * c[0], M1 * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ np.uint64(k0), p1 & MASK, (p0 >> np.uint64(32)) ^ c[3] ^ np.uint64(k1), p0 & MASK]
        with np.errstate(over="ignore"):
            k0, k1 = k0 + W0, k1 + W1
    return np.stack(c, axis=1).astype(np.uint32)


def normals(words):
    """[N, 4] uint32 Philox words -> [N, 4] float32 standard normals (Box-Muller on (x0, x1) and (x2, x3))."""
    w = np.asarray(words, np.uint32)
    out = np.empty(w.shape, np.float32)
    for j in (0, 2):
        u1 = ((w[:, j] >> 8) + 1).astype(np.float32) * np.float32(2.0 ** -24)
        u2 = (w[:, j + 1] >> 8).astype(np.float32) * np.float32(2.0 ** -24)
        r = np.sqrt(np.float32(-2.0) * np.log(u1))
        a = np.pi * (np.float32(2.0) * u2).astype(np.float64)
        out[:, j] = r * np.cos(a).astype(np.float32)
        out[:, j + 1] = r * np.sin(a).astype(np.float32)
    return out


def prior_noise(seed, rows, cols):
    """eps of z_p: [rows = frames][cols = channels] float32."""
    nq = (cols + 3) // 4
    f, q = np.meshgrid(np.arange(rows, dtype=np.uint32), np.arange(nq, dtype=np.uint32), indexing="ij")
    ctr = np.zeros((rows * nq, 4), np.uint32)
    ctr[:, 0], ctr[:, 1] = f.ravel(), q.ravel()
    return normals(philox4x32_10(ctr, seed)).reshape(rows, nq * 4)[:, :cols].copy()


def sdp_noise(seed, tokens):
    """eps of the stochastic duration predictor: [tokens][2] float32, column r = eps_r(t)."""
    ctr = np.zeros((tokens, 4), np.uint32)
    ctr[:, 0] = np.arange(tokens, dtype=np.uint32)
    ctr[:, 2] = 1
    return normals(philox4x32_10(ctr, seed))[:, :2].copy()
