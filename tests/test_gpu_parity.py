"""GPU parity tests (run with -m gpu on a B200).  Everything goes through the C ABI
(include/stts_b200.h via summertts_b200.engine) and is compared with
  * the committed golden vectors produced by the compiled, unmodified reference, and
  * the oracle: the compiled reference itself (oracle/_ref) where it is built, else the numpy restatement
    (oracle/vits_numpy.py).  Where the shipped weights are absent, the tests of a shipped model run seeded random
    weights of the same architecture against the oracle instead of against the goldens.
Tolerances of the default (fp32-accurate) path, the same numbers DESIGN.md §7 states: frame counts / w_ceil exact; float
waveform max|a-b|/max|b| <= 1e-3 (BASELINE.json); int16 PCM never more than 2 LSB and <= 1 LSB except on at most 1e-4
of the samples for `fast` / `multi` / synthetic models (the reference itself moves 1 LSB on ~1% of samples when only its
OpenMP thread count changes, SURVEY.md §8c); `english_fast` on its real 700-id input (377 088 samples) <= 6 LSB, <= 2e-3 of
the samples above 1 LSB (measured 5 LSB / 9.6e-4; our fp32 FFMA tiles land at 4 LSB / 1.4e-3 and an exact-arithmetic
restatement at 4 LSB: that is the reference's own fp32 noise on this input); `mid` <= 20 LSB, <= 3 % of the samples above 1 LSB (its own fp32
noise floor is 7-9 LSB: an exact-arithmetic restatement lands 7-9 LSB from the compiled reference, SURVEY.md §8c);
long-form (x4 `fast`) <= 10 LSB / 0.5 %.  Throughput mode (stts_set_tensor_path(2)) has its own, looser, stated tolerance:
test_throughput_mode_tolerance.
"""
import glob
import json
import os

import numpy as np
import pytest
from parity_util import GOLDEN, TEST_TXT_IDS, find_model, lsb_diff, rel_err, synth_ids

from oracle import ref
from summertts_b200 import binfmt, engine

pytestmark = pytest.mark.gpu


def _pcm_ok(a, b, max_lsb=2, frac=1e-4):
    assert a.size == b.size
    d = np.abs(a.astype(np.int64) - b.astype(np.int64))
    assert d.max() <= max_lsb, "max LSB diff %d" % d.max()
    assert (d > 1).sum() <= max(1, int(frac * a.size)), "%d samples differ by more than 1 LSB" % (d > 1).sum()


@pytest.fixture(scope="module")
def fast_blob():
    b = find_model("single_speaker_fast")
    if b is None:
        b = binfmt.synthetic_model(seed=11)  # same architecture, random weights
    return b


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN, "synth_*.npz"))))
def test_synthetic_models_vs_golden(native_lib, path):
    """All four decoder variants, both duration predictors, speaker conditioning — including
    Generator_Istft / Generator_MBB+PQMF which no shipped model reaches (SURVEY.md §4)."""
    g = np.load(path)
    blob = binfmt.synthetic_model(seed=int(g["seed"]), **json.loads(str(g["hp"])))
    E = engine.SynthesizerTrn(blob)
    E.debug_enable(True)
    for pre, forced in (("a", None), ("b", g["forced"])):
        E.set_forced_durations(forced)
        pcm = E.infer_ids(g["ids"], int(g["sid"]), 1.0)
        assert np.array_equal(E.debug_fetch("w_ceil"), g[pre + "_wceil"])
        assert pcm.size == g[pre + "_pcm"].size
        assert rel_err(E.debug_fetch("z"), g[pre + "_z"]) < 1e-4
        assert rel_err(E.debug_fetch("o"), g[pre + "_o"]) < 1e-4
        _pcm_ok(pcm, g[pre + "_pcm"])
        if pre == "a":
            assert rel_err(E.debug_fetch("xx"), g["a_xx"]) < 1e-4
            assert rel_err(E.debug_fetch("m"), g["a_m"]) < 1e-4
            assert rel_err(E.debug_fetch("logw"), g["a_logw"]) < 1e-4
    E.close()


def _oracle(blob, ids, sid=0, length_scale=1.0, forced_w=None, threads=1):
    """(w_ceil, o, pcm) of the compiled reference (oracle/_ref) where it is built, else of the numpy restatement
    (oracle/vits_numpy.py, which tests/test_oracle.py pins to the reference's golden vectors)."""
    if ref.available():
        ref.set_threads(threads)
        r = ref.RefModel(blob).infer(ids, sid=sid, length_scale=length_scale, forced_w=forced_w, dumps=True)
        return r.w_ceil, r.o, r.pcm
    from oracle import vits_numpy as vn

    o = vn.infer(binfmt.parse_model(blob), ids, sid=sid, length_scale=length_scale, forced_w=forced_w)
    return o["w_ceil"], o["o"], o["pcm"]


def _model(name):
    """(blob, shipped): the shipped weights where present, else seeded random weights of the same architecture."""
    blob = find_model(name)
    if blob is not None:
        return blob, True
    return binfmt.synthetic_model(seed=11, **binfmt.ARCH[name]), False


def _golden_or_oracle(name, blob, shipped):
    """Inputs (ids, sid, length scale) of the golden vectors of `name` and what the reference computes on them:
    the golden (w_ceil, o, pcm) for the shipped weights, the oracle's for any other weights."""
    g = np.load(os.path.join(GOLDEN, "real_%s.npz" % name))
    ids, sid, ls = g["ids"], int(g["sid"]), float(g["ls"])
    want = (g["wceil"], g["o"], g["pcm"]) if shipped else _oracle(blob, ids, sid, ls)
    return (ids, sid, ls), want


@pytest.mark.parametrize("name,max_lsb,frac", [("single_speaker_fast", 2, 1e-4), ("multi_speakers", 2, 1e-4),
                                               ("single_speaker_mid", 20, 3e-2), ("single_speaker_english_fast", 6, 2e-3)])
def test_shipped_models_vs_golden(native_lib, name, max_lsb, frac):
    """BASELINE configs 2-4: shipped weights, reference ids, fp32 parity within 1e-3.  Without the shipped weights:
    seeded random weights of the same architecture on the same ids, against the oracle."""
    blob, shipped = _model(name)
    args, (w_ceil, o, want) = _golden_or_oracle(name, blob, shipped)
    E = engine.SynthesizerTrn(blob)
    E.debug_enable(True)
    pcm = E.infer_ids(*args)
    assert np.array_equal(E.debug_fetch("w_ceil"), w_ceil)
    assert pcm.size == want.size
    assert rel_err(E.debug_fetch("o"), o) < 1e-3
    _pcm_ok(pcm, want, max_lsb, frac)
    E.close()


def test_long_form_vs_compiled_reference(native_lib, fast_blob):
    """Config 3 style long-form: the id sequence repeated x4 as ONE utterance through the oracle."""
    ids = (TEST_TXT_IDS[:-1] * 4) + [1]
    w_ceil, o, want = _oracle(fast_blob, ids)
    E = engine.SynthesizerTrn(fast_blob)
    E.debug_enable(True)
    pcm = E.infer_ids(ids)
    assert np.array_equal(E.debug_fetch("w_ceil"), w_ceil)
    assert rel_err(E.debug_fetch("o"), o) < 1e-3
    _pcm_ok(pcm, want, 10, 5e-3)  # longer utterances accumulate more fp32 noise on both sides
    E.close()


def test_long_form_mid_x16_vs_compiled_reference(native_lib):
    """BASELINE config 3 as SURVEY.md §8d words it: single_speaker_mid, the test.txt id sequence repeated x16 as ONE
    utterance (T = 1201 ids, ~6.1 k frames, ~1.57 M samples) through the ID-level compiled reference.
    Tolerance: frame counts exact, waveform rel-err <= 1e-3 (BASELINE.json), PCM within the model's own fp32 noise
    (<= 20 LSB, <= 3 % of samples above 1 LSB — see the module docstring).  Seeded random weights of the same
    architecture predict shorter durations, so without the shipped weights length_scale 5 keeps the utterance as long."""
    blob, shipped = _model("single_speaker_mid")
    ls = 1.0 if shipped else 5.0
    ids = (TEST_TXT_IDS[:-1] * 16) + [1]
    w_ceil, o, want = _oracle(blob, ids, length_scale=ls, threads=8)
    E = engine.SynthesizerTrn(blob)
    E.debug_enable(True)
    pcm = E.infer_ids(ids, 0, ls)
    assert np.array_equal(E.debug_fetch("w_ceil"), w_ceil)
    assert pcm.size == want.size and pcm.size > 1_400_000
    assert rel_err(E.debug_fetch("o"), o) < 1e-3
    _pcm_ok(pcm, want, 20, 3e-2)
    E.close()


def test_batch_equals_per_utterance_ragged(native_lib, fast_blob):
    """Packed varlen batch == the same utterances one at a time (bit-exact): every conv pads at its own
    utterance's edges, exactly as the batch-1 reference does."""
    rng = np.random.default_rng(5)
    E = engine.SynthesizerTrn(fast_blob)
    lens = [5, 128, 17, 64, 9, 33]
    utts = [synth_ids(rng, n) for n in lens]
    single = [E.infer_ids(u) for u in utts]
    batch = E.infer_batch(utts)
    for a, b in zip(single, batch):
        assert np.array_equal(a, b)
    # permutation invariance
    perm = [3, 0, 5, 1, 4, 2]
    batch2 = E.infer_batch([utts[i] for i in perm])
    for k, i in enumerate(perm):
        assert np.array_equal(batch2[k], single[i])
    # determinism
    assert all(np.array_equal(a, b) for a, b in zip(batch, E.infer_batch(utts)))
    E.close()


def test_full_size_batch_properties(native_lib, fast_blob):
    """BASELINE config-5 shape (64 x 128 ids, forced 5 frames/id): size-independent checks —
    S = 256 * sum(w_ceil) per utterance, identical utterances give identical PCM, and a sampled
    utterance equals its stand-alone run."""
    rng = np.random.default_rng(1234)
    E = engine.SynthesizerTrn(fast_blob)
    base = [synth_ids(rng, 128) for _ in range(8)]
    utts = [base[i % 8] for i in range(64)]
    E.set_forced_durations(np.full(64 * 128, 5.0, np.float32))
    out = E.infer_batch(utts)
    assert all(o.size == 128 * 5 * 256 for o in out)
    for i in range(8, 64):
        assert np.array_equal(out[i], out[i % 8])
    E.set_forced_durations(np.full(128, 5.0, np.float32))
    assert np.array_equal(E.infer_ids(base[3]), out[3])
    E.close()


def test_edge_cases(native_lib, fast_blob):
    E = engine.SynthesizerTrn(fast_blob)
    rng = np.random.default_rng(9)
    # fewer than win+1 = 5 ids: the reference cannot run (multi_head_attention.cpp:140-150) -> STTS_E_ARG
    with pytest.raises(engine.SttsError) as ei:
        E.infer_ids([0, 15, 119, 1])
    assert ei.value.code == -1
    with pytest.raises(engine.SttsError):
        E.infer_ids([0, 15, 5000, 3, 1, 1])  # id outside the vocabulary
    # minimum length works
    assert E.infer_ids(synth_ids(rng, 5)).size % 256 == 0
    # zero-duration tokens (forced) and the all-zero case: frames = max(sum, 1) (nn_clamp_min, SynthesizerTrn.cpp:378)
    ids = synth_ids(rng, 12)
    w = np.array([0, 3, 0, 0, 2, 1, 0, 4, 0, 0, 1, 0], np.float32)
    E.set_forced_durations(w)
    assert E.infer_ids(ids).size == int(w.sum()) * 256
    E.set_forced_durations(np.zeros(12, np.float32))
    assert E.infer_ids(ids).size == 256
    E.set_forced_durations(None)
    E.close()


def test_zero_duration_matches_reference(native_lib):
    blob = binfmt.synthetic_model(seed=100, decType=1, durPredType=1, isMS=0, nLayers=2, preCh=32)
    rng = np.random.default_rng(3)
    ids = synth_ids(rng, 12)
    w = np.array([0, 3, 0, 0, 2, 1, 0, 4, 0, 0, 1, 0], np.float32)
    want = _oracle(blob, ids, forced_w=w)[2]
    E = engine.SynthesizerTrn(blob)
    E.set_forced_durations(w)
    _pcm_ok(E.infer_ids(ids), want)
    E.close()


def test_speaker_id_clamp(native_lib):
    """sid out of range behaves as sid 0 (SynthesizerTrn.cpp:366-369)."""
    blob = binfmt.synthetic_model(seed=104, decType=0, durPredType=1, isMS=1, nLayers=2, preCh=32, spkNum=5, gin=32,
                                  upRates=(4, 2, 2), upK=(8, 4, 4))
    rng = np.random.default_rng(4)
    ids = synth_ids(rng, 20)
    E = engine.SynthesizerTrn(blob)
    assert E.getSpeakerNum() == 5
    a0 = E.infer_ids(ids, sid=0)
    assert np.array_equal(E.infer_ids(ids, sid=99), a0)
    assert np.array_equal(E.infer_ids(ids, sid=-1), a0)
    assert not np.array_equal(E.infer_ids(ids, sid=2), a0)
    E.close()


def test_config5_multi_speakers_batch64(native_lib):
    """BASELINE config 5 as worded: multi_speakers.bin (stochastic duration predictor + spline flows + speaker conditioning +
    HiFi-GAN down to 4 channels), 64 synthetic 128-id utterances in ONE batch, a different speaker per utterance, the model's
    own durations.  Sampled utterances: bit-identical to their stand-alone run, and frame count exact / PCM within the `multi`
    tolerance against the compiled reference run on the same ids and speaker (the oracle, with seeded random weights of the
    same architecture where the shipped weights are absent)."""
    blob, _ = _model("multi_speakers")
    rng = np.random.default_rng(55)
    E = engine.SynthesizerTrn(blob)
    nspk = E.getSpeakerNum()
    utts = [synth_ids(rng, 128) for _ in range(64)]
    sids = [(7 * i + 3) % nspk for i in range(64)]
    out = E.infer_batch(utts, sids=sids)
    assert len(out) == 64 and all(o.size > 0 and o.size % 256 == 0 for o in out)
    for i in (0, 21, 63):
        assert np.array_equal(E.infer_ids(utts[i], sid=sids[i]), out[i])
    assert E.tensor_fallbacks() == 0
    for i in (5, 40):
        want = _oracle(blob, utts[i], sid=sids[i], threads=8)[2]
        assert want.size == out[i].size, (want.size, out[i].size)
        _pcm_ok(out[i], want, 2, 1e-4)
    E.close()


def test_native_kernels_ran(native_lib, fast_blob):
    E = engine.SynthesizerTrn(fast_blob)
    n0 = E.kernel_launches()
    E.infer_ids(TEST_TXT_IDS)
    assert E.kernel_launches() - n0 > 50
    t = E.last_timing()
    assert t["total"] > 0 and t["flow"] > 0 and t["dec"] > 0
    E.close()


def _stft_mag(x, n=512, hop=128):
    x = np.asarray(x, np.float64)
    w = np.hanning(n)
    idx = np.arange(0, x.size - n + 1, hop)[:, None] + np.arange(n)[None, :]
    return np.abs(np.fft.rfft(x[idx] * w, axis=1))


@pytest.mark.parametrize("name", ["single_speaker_fast", "single_speaker_mid", "multi_speakers", "single_speaker_english_fast"])
def test_throughput_mode_tolerance(native_lib, name):
    """stts_set_tensor_path(2): one fp16 MMA per K-step (fp16 operands, fp32 accumulate) in the frame-level tensor-core convs;
    the text encoder and the duration predictor keep the accurate MMAs, so the frame counts stay EXACT.  These networks
    amplify operand rounding ~500x (round 1 measured 1e-6-level accumulator bias moving `mid` by 5e-4), so fp16 operands
    cannot meet the 1e-3 sample-wise criterion; the stated tolerance of this mode is waveform SNR >= 25 dB and spectral
    convergence <= 3e-2 against the compiled reference's golden output (measured: 45 / 30 / 40 / 40 dB, 2e-3 ... 1.2e-2).
    Without the shipped weights: seeded random weights of the same architecture, against the oracle."""
    blob, shipped = _model(name)
    args, (w_ceil, want_o, want_pcm) = _golden_or_oracle(name, blob, shipped)
    E = engine.SynthesizerTrn(blob)
    E.debug_enable(True)
    E.set_tensor_path(2)
    pcm = E.infer_ids(*args)
    assert np.array_equal(E.debug_fetch("w_ceil"), w_ceil)
    assert pcm.size == want_pcm.size
    o, want = E.debug_fetch("o").ravel().astype(np.float64), want_o.ravel().astype(np.float64)
    snr = 10 * np.log10((want ** 2).sum() / ((o - want) ** 2).sum())
    A, B = _stft_mag(o), _stft_mag(want)
    assert snr >= 25.0, snr
    assert np.linalg.norm(A - B) / np.linalg.norm(B) <= 3e-2
    assert E.tensor_fallbacks() == 0
    E.close()


def test_tensor_path_matches_ffma_path(native_lib, fast_blob):
    """The tcgen05 split-fp16 path (planes handed from conv to conv, TMA-fed) and the fp32 FFMA tiles are two
    implementations of the same convs: same sample counts, waveforms within the fp32 noise of the stack."""
    rng = np.random.default_rng(21)
    utts = [synth_ids(rng, n) for n in (40, 7, 96)]
    E = engine.SynthesizerTrn(fast_blob)
    E.set_forced_durations(np.full(sum(len(u) for u in utts), 3.0, np.float32))
    E.set_tensor_path(1)
    a = E.infer_batch(utts)
    E.set_tensor_path(0)
    b = E.infer_batch(utts)
    for x, y in zip(a, b):
        assert x.size == y.size
        assert np.abs(x.astype(np.int64) - y.astype(np.int64)).max() <= 4
    E.close()
