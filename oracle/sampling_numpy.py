"""oracle/sampling_numpy.py — TEST INFRASTRUCTURE ONLY: the NN half of synthesis with VITS sampling (DESIGN.md §12), built
from the pinned restatement in oracle/vits_numpy.py and the random stream of oracle/rng_numpy.py.

The reference hard-codes noiseScale = 0 (SynthesizerTrn.cpp:357) and its compiled objects draw from a different generator,
so this restatement is the judge for sampled parity.  With both scales 0 it takes exactly the operations of
vits_numpy.infer (tests/test_sampling.py checks that bit for bit), so the pinning of vits_numpy carries over:
  prior:  z_p = m + eps * exp(logs) * noise_scale on the expanded rows (m = logs = 0 on the padding frame)
  SDP:    z = eps * noise_scale_w in place of the zeros, before nn_flip(z, 0) (durPredType 0 only)
A zero scale skips its term.
"""
from __future__ import annotations

import numpy as np

from oracle import rng_numpy
from oracle import vits_numpy as vn

f32 = np.float32


def stoch_dp(x, D, g=None, z0=None):
    """vits_numpy.stoch_dp (StochasticDurationPredictor.cpp:117-149, flows[0] skipped) started from z0 [2][T] instead of
    zeros; nn_flip(z, 0) swaps its two rows."""
    XX = vn.conv1d(x, D["pre"])
    if g is not None:
        XX = XX + vn.conv1d(g, D["cond"])
    XX = vn.dds_conv(XX, D["convs"])
    XX = vn.conv1d(XX, D["proj"])
    T = XX.shape[0]
    zT = np.zeros((2, T), f32) if z0 is None else np.asarray(z0, f32)[::-1].copy()
    flap = zT.T
    for i in range(D["nFlows"] - 1, 0, -1):
        flap = vn.conv_flow(zT, XX, D["flows"][i])
        flap = flap[:, ::-1]
        zT = flap.T.copy()
    aff = (flap - D["ea"]["m"][None, :]) * np.exp(-D["ea"]["logs"])[None, :]
    return aff[:, :1].astype(f32)


def infer(M, ids, sid=0, length_scale=1.0, forced_w=None, noise_scale=0.0, noise_scale_w=0.0, seed=0):
    """vits_numpy.infer with VITS sampling from the utterance's seed.  Also returns `logs`."""
    ids = np.asarray(ids, np.int64)
    xx, m, logs = vn.text_encoder(ids, M["enc"])
    g = None
    if M["isMS"] == 1:
        if sid < 0 or sid >= M["spkNum"]:
            sid = 0
        g = M["emg"][sid][None, :].astype(f32)
    if M["durPredType"] == 1:
        logw = vn.fix_dp(xx, M["dp"], g)
    else:
        z0 = (rng_numpy.sdp_noise(seed, len(ids)).T * f32(noise_scale_w)).astype(f32) if noise_scale_w != 0 else None
        logw = stoch_dp(xx, M["dp"], g, z0=z0)
    w = np.exp(logw[:, 0]) * f32(length_scale)
    w_ceil = np.ceil(w).astype(f32)
    if forced_w is not None:
        w_ceil = np.asarray(forced_w, f32)
    reps = w_ceil.astype(np.int64)
    F = max(int(w_ceil.sum()), 1)
    z_p = np.zeros((F, m.shape[1]), f32)
    rows = np.repeat(np.arange(len(ids)), reps)
    z_p[:len(rows)] = m[rows]
    if noise_scale != 0:
        logs_p = np.zeros_like(z_p)
        logs_p[:len(rows)] = logs[rows]
        eps = rng_numpy.prior_noise(seed, F, m.shape[1])
        z_p = (z_p + eps * np.exp(logs_p) * f32(noise_scale)).astype(f32)
    z = vn.flow_reverse(z_p, M["flow"], g)
    o = vn.generator(z, M["dec"], g)
    pcm = np.trunc(o * f32(32737)).astype(np.int16)  # (int16_t)(o*32737), SynthesizerTrn.cpp:395
    return dict(xx=xx, m=m, logs=logs, logw=logw[:, 0], w_ceil=w_ceil, z_p=z_p, z=z, o=o, pcm=pcm, F=F)
