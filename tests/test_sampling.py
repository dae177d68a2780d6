"""Seeded stochastic sampling (VITS noise_scale / noise_scale_w; stts_set_sampling, DESIGN.md §12).

CPU: the Philox4x32-10 stream of oracle/rng_numpy.py against Random123's known-answer vectors, the library's host restatement
(stts_debug_noise) against it, the statistics of the normals, and the sampling oracle (oracle/sampling_numpy.py) with zero
scales against the pinned oracle/vits_numpy.py.
GPU: off means off (bit-identical, same launches), parity with the sampling oracle fed the same seed, determinism and invariance
under batching / streaming / the device image, argument errors, and the CLI's per-job seeds."""
import json
import os
import subprocess

import numpy as np
import pytest
from parity_util import GOLDEN, TEST_TXT_IDS, rel_err, synth_ids
from scipy import stats

from oracle import rng_numpy
from summertts_b200 import binfmt, engine

NS, NSW = 0.667, 0.8          # the VITS demo defaults
SEEDS = (0, 1, 2 ** 64 - 1)


def _sdp_hp():
    g = np.load(os.path.join(GOLDEN, "synth_hifigan_sdp_spk.npz"))
    return int(g["seed"]), json.loads(str(g["hp"])), int(g["sid"])


def _model(name):
    """(blob, sid) of seeded random weights: the `fast` / `multi_speakers` architectures or the synth_hifigan_sdp_spk model."""
    if name == "sdp_spk":
        seed, hp, sid = _sdp_hp()
        return binfmt.synthetic_model(seed=seed, **hp), sid
    return binfmt.synthetic_model(seed=11, **binfmt.ARCH[name]), (3 if name == "multi_speakers" else 0)


def _pcm_ok(a, b, max_lsb=2, frac=1e-4):
    assert a.size == b.size
    d = np.abs(a.astype(np.int64) - b.astype(np.int64))
    assert d.max() <= max_lsb, "max LSB diff %d" % d.max()
    assert (d > 1).sum() <= max(1, int(frac * a.size)), "%d samples differ by more than 1 LSB" % (d > 1).sum()


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_philox_known_answers():
    """Random123's kat_vectors for philox4x32_10: (counter; key) -> output."""
    cases = [((0, 0, 0, 0), 0, (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
             ((0xFFFFFFFF,) * 4, 2 ** 64 - 1, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
             ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), 0xA4093822 | (0x299F31D0 << 32),
              (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1))]
    for ctr, key, want in cases:
        got = rng_numpy.philox4x32_10(np.array([ctr], np.uint32), key)[0]
        assert [int(v) for v in got] == list(want)


def test_library_noise_equals_numpy(native_lib):
    """stts_debug_noise (the device's code compiled for the host) == rng_numpy, both streams, >= 1e6 normals."""
    total = 0
    for seed in SEEDS:
        a = engine.debug_noise(seed, 0, 1800, 193)      # 193 channels: a partial last quad
        b = rng_numpy.prior_noise(seed, 1800, 193)
        assert np.abs(a - b).max() <= 2e-6
        c = engine.debug_noise(seed, 1, 70000, 2)
        d = rng_numpy.sdp_noise(seed, 70000)
        assert np.abs(c - d).max() <= 2e-6
        total += a.size + c.size
    assert total >= 1_000_000
    with pytest.raises(engine.SttsError):
        engine.debug_noise(0, 1, 10, 3)
    with pytest.raises(engine.SttsError):
        engine.debug_noise(0, 2, 10, 2)


def test_noise_statistics():
    x = rng_numpy.prior_noise(5, 5300, 192).ravel()[:1_000_000].astype(np.float64)
    assert abs(x.mean()) < 5e-3 and abs(x.std() - 1) < 5e-3
    assert stats.kstest(x, "norm").pvalue > 1e-4
    y = rng_numpy.prior_noise(6, 5300, 192).ravel()[:1_000_000].astype(np.float64)
    s = rng_numpy.sdp_noise(5, 500_000).ravel().astype(np.float64)
    for a, b in ((x, y), (x, s)):
        assert abs(np.corrcoef(a, b)[0, 1]) < 5e-3
    assert abs(np.corrcoef(s[0::2], s[1::2])[0, 1]) < 5e-3


@pytest.mark.parametrize("hp", ["sdp_spk", "fix"])
def test_sampling_oracle_zero_scales_equal_the_pinned_oracle(hp):
    """oracle/sampling_numpy.py with both scales 0 == oracle/vits_numpy.py (pinned to the reference), bit for bit."""
    from oracle import sampling_numpy as sn
    from oracle import vits_numpy as vn

    if hp == "sdp_spk":
        seed, kw, sid = _sdp_hp()
    else:
        seed, kw, sid = 100, dict(decType=1, durPredType=1, isMS=0, nLayers=2, preCh=32), 0
    M = binfmt.parse_model(binfmt.synthetic_model(seed=seed, **kw))
    ids = synth_ids(np.random.default_rng(1), 14)
    a = vn.infer(M, ids, sid=sid)
    b = sn.infer(M, ids, sid=sid, noise_scale=0.0, noise_scale_w=0.0, seed=123)
    for k in ("xx", "m", "logw", "w_ceil", "z_p", "z", "o", "pcm"):
        assert np.array_equal(a[k], b[k]), k
    c = sn.infer(M, ids, sid=sid, noise_scale=NS, noise_scale_w=NSW, seed=123)
    assert not np.array_equal(a["z_p"], c["z_p"])


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["single_speaker_fast", "sdp_spk"])
def test_off_means_off(native_lib, name):
    """All-zero scales: PCM bit-identical to no sampling and the same kernel launches."""
    blob, sid = _model(name)
    E = engine.SynthesizerTrn(blob)
    ids = synth_ids(np.random.default_rng(7), 40)
    n0 = E.kernel_launches()
    want = E.infer_ids(ids, sid)
    n1 = E.kernel_launches()
    E.set_sampling([0.0], [0.0], [99])
    got = E.infer_ids(ids, sid)
    n2 = E.kernel_launches()
    E.set_sampling(None)
    assert np.array_equal(got, want) and n2 - n1 == n1 - n0
    if E._L.stts_header_field(E._h, 2) == 1:       # FixDurationPredictor: no noise input, noise_scale_w changes nothing
        got = E.infer_ids(ids, sid, noise_scale_w=NSW, seed=4)
        assert np.array_equal(got, want) and E.kernel_launches() - n2 == n1 - n0
    E.close()


@pytest.mark.gpu
@pytest.mark.parametrize("path", [0, 1])
@pytest.mark.parametrize("name", ["single_speaker_fast", "multi_speakers", "sdp_spk"])
def test_sampled_parity_vs_oracle(native_lib, name, path):
    from oracle import sampling_numpy as sn

    blob, sid = _model(name)
    M = binfmt.parse_model(blob)
    ids = synth_ids(np.random.default_rng(17), 30)
    want = sn.infer(M, ids, sid=sid, noise_scale=NS, noise_scale_w=NSW, seed=2024)
    E = engine.SynthesizerTrn(blob)
    E.set_tensor_path(path)
    E.debug_enable(True)
    pcm = E.infer_ids(ids, sid, noise_scale=NS, noise_scale_w=NSW, seed=2024)
    assert np.array_equal(E.debug_fetch("w_ceil"), want["w_ceil"])
    assert rel_err(E.debug_fetch("logs"), want["logs"]) < 1e-4
    assert rel_err(E.debug_fetch("z_p"), want["z_p"]) < 1e-4
    assert rel_err(E.debug_fetch("o"), want["o"]) < 1e-3
    _pcm_ok(pcm, want["pcm"])
    E.close()


@pytest.mark.gpu
def test_sampled_padding_frame(native_lib):
    """All-zero durations: the single padding frame has m = logs = 0, so z_p = eps * noise_scale there."""
    from oracle import sampling_numpy as sn

    blob, sid = _model("single_speaker_fast")
    ids = synth_ids(np.random.default_rng(3), 12)
    w = np.zeros(12, np.float32)
    E = engine.SynthesizerTrn(blob)
    E.debug_enable(True)
    E.set_forced_durations(w)
    pcm = E.infer_ids(ids, sid, noise_scale=NS, seed=8)
    zp = E.debug_fetch("z_p")
    inter = zp.shape[1]
    assert zp.shape[0] == 1
    assert np.abs(zp - engine.debug_noise(8, 0, 1, inter) * np.float32(NS)).max() <= 2e-6
    want = sn.infer(binfmt.parse_model(blob), ids, sid=sid, forced_w=w, noise_scale=NS, seed=8)
    assert rel_err(zp, want["z_p"]) < 1e-4
    _pcm_ok(pcm, want["pcm"])
    E.close()


@pytest.mark.gpu
def test_determinism_and_batch_invariance(native_lib):
    blob, sid = _model("sdp_spk")
    E = engine.SynthesizerTrn(blob)
    rng = np.random.default_rng(12)
    utts = [synth_ids(rng, n) for n in (9, 64, 17, 33, 5, 120, 48, 26)]
    ns = np.array([NS, 0.0, 0.3, 1.0, 0.667, 0.0, 2.0, 0.1], np.float32)
    nsw = np.array([NSW, 0.0, 0.0, 1.0, 0.5, 0.0, 0.8, 1.2], np.float32)
    seeds = np.array([1, 2, 3, 4, 5, 6, 2 ** 64 - 1, 10 ** 12], np.uint64)
    sids = [sid] * 8
    a = E.infer_ids(utts[0], sid, noise_scale=NS, noise_scale_w=NSW, seed=1)
    assert np.array_equal(a, E.infer_ids(utts[0], sid, noise_scale=NS, noise_scale_w=NSW, seed=1))
    assert not np.array_equal(a, E.infer_ids(utts[0], sid, noise_scale=NS, noise_scale_w=NSW, seed=2))
    batch = E.infer_batch(utts, sids=sids, noise_scale=ns, noise_scale_w=nsw, seed=seeds)
    for i, u in enumerate(utts):
        one = E.infer_ids(u, sid, noise_scale=float(ns[i]), noise_scale_w=float(nsw[i]), seed=int(seeds[i]))
        assert np.array_equal(batch[i], one), i
        if ns[i] == 0 and nsw[i] == 0:
            assert np.array_equal(batch[i], E.infer_ids(u, sid)), i
    E.close()


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", [48, 257])
def test_stream_sampled_equals_one_shot(native_lib, chunk):
    blob, sid = _model("single_speaker_fast")
    ids = (TEST_TXT_IDS[:-1] * 2) + [1]
    E = engine.SynthesizerTrn(blob)
    whole = E.infer_ids(ids, sid, noise_scale=NS, noise_scale_w=NSW, seed=31)
    chunks, _ = E.infer_stream(ids, sid, chunk_frames=chunk, noise_scale=NS, noise_scale_w=NSW, seed=31)
    assert np.array_equal(np.concatenate(chunks), whole)
    assert not np.array_equal(whole, E.infer_ids(ids, sid))
    E.close()


@pytest.mark.gpu
def test_device_noise_statistics(native_lib):
    """eps recovered from the device's z_p, m, logs and w_ceil on a long utterance == stts_debug_noise, and it is N(0, 1)."""
    blob, sid = _model("single_speaker_fast")
    ids = synth_ids(np.random.default_rng(4), 200)
    E = engine.SynthesizerTrn(blob)
    E.debug_enable(True)
    E.set_forced_durations(np.full(200, 5.0, np.float32))
    ns = 10.0                                     # the noise term dominates z_p: eps is recovered to ~1e-7
    E.infer_ids(ids, sid, noise_scale=ns, seed=77)
    zp, m, logs, w = (E.debug_fetch(k).astype(np.float64) for k in ("z_p", "m", "logs", "w_ceil"))
    rows = np.repeat(np.arange(len(ids)), w.astype(np.int64))
    eps = (zp - m[rows]) / (np.exp(logs[rows]) * ns)
    assert eps.size >= 100_000
    ref = engine.debug_noise(77, 0, zp.shape[0], zp.shape[1])
    assert np.abs(eps - ref).max() <= 1e-5
    x = eps.ravel()
    assert abs(x.mean()) < 5e-3 * np.sqrt(1e6 / x.size) and abs(x.std() - 1) < 5e-3 * np.sqrt(1e6 / x.size)
    assert stats.kstest(x, "norm").pvalue > 1e-4
    E.close()


@pytest.mark.gpu
def test_device_image_samples_identically(native_lib, tmp_path):
    blob, sid = _model("sdp_spk")
    ids = synth_ids(np.random.default_rng(8), 30)
    kw = dict(noise_scale=NS, noise_scale_w=NSW, seed=5)
    A = engine.SynthesizerTrn(blob)
    want = A.infer_ids(ids, sid, **kw)
    A.close()
    img = str(tmp_path / "sdp.stts_image")
    engine.SynthesizerTrn(blob, image_path=img).close()
    B = engine.SynthesizerTrn(blob, image_path=img)
    assert B.from_image
    assert np.array_equal(B.infer_ids(ids, sid, **kw), want)
    B.close()


@pytest.mark.gpu
def test_sampling_argument_errors(native_lib):
    blob, sid = _model("single_speaker_fast")
    E = engine.SynthesizerTrn(blob)
    ids = synth_ids(np.random.default_rng(2), 20)
    want = E.infer_ids(ids, sid, noise_scale=NS, seed=9)
    for ns, nsw in ((np.nan, 0.0), (0.5, np.nan), (-0.1, 0.0), (0.0, -1.0), (10.5, 0.0), (0.0, np.inf)):
        with pytest.raises(engine.SttsError) as ei:
            E.set_sampling([ns], [nsw], [1])
        assert ei.value.code == engine.STTS_E_ARG
    E.set_sampling([NS, NS], [0.0, 0.0], [9, 9])     # n = 2, batch of 1: rejected when staged
    with pytest.raises(engine.SttsError) as ei:
        E.infer_ids(ids, sid)
    assert ei.value.code == engine.STTS_E_ARG
    E.set_sampling(None)
    assert np.array_equal(E.infer_ids(ids, sid, noise_scale=NS, seed=9), want)
    E.close()


@pytest.mark.gpu
def test_cli_sampling_seeds_per_line(native_lib, tmp_path):
    """tts_b200_ids --per-line --noise-scale --noise-scale-w --seed S: line j is synthesised with seed S + j."""
    r = subprocess.run(["make", "-C", os.path.join(os.path.dirname(engine.__file__), "host"), "ids-cli"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    cli = os.path.join(os.path.dirname(engine.__file__), "bin", "tts_b200_ids")
    blob = binfmt.synthetic_model(7)
    model = tmp_path / "synthetic.bin"
    blob.tofile(model)
    rng = np.random.default_rng(3)
    utts = [[0] + [int(v) for v in rng.integers(1, 40, size=n)] + [0, 1] for n in (9, 23, 14)]
    ids = tmp_path / "ids.txt"
    ids.write_text("".join(" ".join(map(str, u)) + "\n" for u in utts))
    out = tmp_path / "o.wav"
    r = subprocess.run([cli, "--ids", "--per-line", "--noise-scale", str(NS), "--noise-scale-w", str(NSW), "--seed", "7", str(ids),
                        str(model), str(out)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    E = engine.SynthesizerTrn(blob)
    for i, u in enumerate(utts):
        raw = (tmp_path / ("o.wav_%04d.wav" % i)).read_bytes()
        pcm = E.infer_ids(u, 0, 1.0, noise_scale=NS, noise_scale_w=NSW, seed=7 + i)
        assert np.array_equal(np.frombuffer(raw[44:], dtype="<i2"), pcm), i
        assert not np.array_equal(pcm, E.infer_ids(u))
    E.close()
