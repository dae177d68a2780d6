"""Batched GRU grapheme-to-phoneme (SURVEY.md §8f rank 3; reference: src/engipa/EnglishText2Id.cpp:270-313, 496-545).

CPU (`-m "not gpu"`): the numpy oracle against the golden vectors of the compiled unmodified reference (and against the
live reference where it travelled, including its unmodified getIPAId); the kernel's per-thread phases, run thread by
thread on the CPU through tests/g2p_host_harness.cpp, against the oracle.
GPU (`-m gpu`): stts_g2p_predict through the C ABI against the oracle — phone ids exact, encoder state / logits to fp32 noise.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess

import numpy as np
import pytest
from parity_util import GOLDEN, MODEL_DIRS, ROOT

from oracle import g2p_numpy as gn
from oracle import ref

G = np.load(os.path.join(GOLDEN, "g2p.npz"))


def _words(prefix):
    L, O = G[prefix + "_letters"].tobytes(), G[prefix + "_offsets"]
    return [L[O[i]:O[i + 1]] for i in range(len(O) - 1)]


def _preds(prefix):
    return [[int(p) for p in row if p >= 0] for row in G[prefix + "_preds"]]


def _synth_section():
    sec = gn.synthetic_section(int(G["synth_seed"]), scale=float(G["synth_scale"]))
    assert hashlib.sha256(sec.tobytes()).hexdigest() == str(G["synth_sha"]), "seeded section drifted from the golden's"
    return sec


def _real_section():
    for d in MODEL_DIRS:
        p = os.path.join(d, "single_speaker_english_fast.g2p.bin") if d else ""
        if p and os.path.exists(p):
            return np.fromfile(p, dtype=np.float32)
        p = os.path.join(d, "single_speaker_english_fast.bin") if d else ""
        if p and os.path.exists(p):
            from summertts_b200 import binfmt

            blob = np.fromfile(p, dtype=np.float32)
            return blob[int(binfmt.parse_model(blob)["nn_end"]):]
    return None


# ------------------------------------------------------------------------------------------------ oracle pins (CPU)
def test_oracle_matches_golden_synthetic():
    m = gn.parse_section(_synth_section())
    words, want = _words("synth"), _preds("synth")
    for i, w in enumerate(words):
        p, h, lg = gn.predict_word(m, w)
        assert p == want[i], (w, p, want[i])
        assert np.abs(h - G["synth_hidden"][i]).max() < 2e-5
        assert np.abs(lg - G["synth_logits0"][i]).max() < 1e-4


def test_tables_reproduce_reference_ipa_ids():
    """preds -> IPA ids through the restated tables == the unmodified getIPAId(word) recorded in the golden."""
    want, off = G["real_ipa_ids"], G["real_ipa_offsets"]
    for i, p in enumerate(_preds("real")):
        assert gn.preds_to_ipa_ids(p) == want[off[i]:off[i + 1]].tolist()


@pytest.mark.skipif(_real_section() is None, reason="shipped English model's GRU section did not travel")
def test_oracle_matches_golden_shipped():
    sec = _real_section()
    assert hashlib.sha256(sec[:gn.parse_section(sec)["consumed"]].tobytes()).hexdigest() == str(G["real_sha"])
    m = gn.parse_section(sec)
    for w, want in zip(_words("real"), _preds("real")):
        assert gn.predict_word(m, w)[0] == want


@pytest.mark.skipif(not ref.available(), reason="compiled reference not built")
def test_oracle_matches_live_reference():
    for sec in (_synth_section(), _real_section()):
        if sec is None:
            continue
        m, R = gn.parse_section(sec), ref.RefG2p(sec)
        assert R.consumed == m["consumed"]
        for w in _words("synth")[:24] + [b"a", b"zz", b"rock'n'roll", "naïveté".encode()]:
            pr, hr, lr = R.word(w)
            pn, hn, ln = gn.predict_word(m, w)
            assert pr == pn and np.abs(hr - hn).max() < 2e-5 and np.abs(lr - ln).max() < 1e-4, w
        R.close()
    sec = _real_section()
    if sec is not None:        # the restated loop is pinned by the reference's own text -> ids for unknown words
        R, m = ref.RefG2p(sec), gn.parse_section(sec)
        for w in _words("real")[:32]:
            assert R.ipa_ids(w.decode()) == gn.preds_to_ipa_ids(gn.predict_word(m, w)[0])
        R.close()


# ------------------------------------------------------------------------------------------------ kernel phases on the CPU
@pytest.fixture(scope="module")
def host_harness(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("g2p") / "g2p_host.so")
    r = subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so, os.path.join(ROOT, "tests", "g2p_host_harness.cpp")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    L = C.CDLL(so)
    L.g2p_host_predict.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.g2p_host_predict_cluster.argtypes = L.g2p_host_predict.argtypes + [C.c_int32]
    return L


def _pack(words):
    letters = np.frombuffer(b"".join(words), np.uint8).copy()
    offs = np.cumsum([0] + [len(w) for w in words]).astype(np.int32)
    return letters, offs


@pytest.mark.parametrize("kernel", ["stream", "cluster1", "cluster3", "cluster18"])
@pytest.mark.parametrize("case", ["synth64", "ragged7", "small_dims"])
def test_kernel_phases_on_cpu(host_harness, case, kernel):
    """Both kernels (W_hh streamed per step / resident in an 8-CTA cluster with the state exchanged through the peers' shared memory),
    the cluster one with 1, 3 and 18 co-resident clusters walking the word groups."""
    if case == "small_dims":      # another hidden / table size: 3H = 96 < 4 * V = 148 (the logits phase sets the thread count)
        sec = gn.synthetic_section(5, hidden=32, emb=24, n_letters=29, n_phones=37, scale=4.0)
        words = [b"abcd", b"zyx", b"q", b"hellothere", b"kernel"]
    else:
        sec = _synth_section()
        words = _words("synth") if case == "synth64" else [b"a", b"supercalifragilistic", b"it's", b"xy", b"\xc3\xa9clair", b"mmmmmmmmmmmmmmmmmmmmmmmmmmmmmmmm", b"q"]
    m = gn.parse_section(sec)
    H, V, n = m["enc_w_hh"].shape[1], m["fc_w"].shape[0], len(words)
    letters, offs = _pack(words)
    preds, cnt = np.full((n, 20), -9, np.int32), np.full(n, -9, np.int32)
    hid, lg = np.zeros((n, H), np.float32), np.zeros((n, V), np.float32)
    args = (sec.ctypes.data, n, letters.ctypes.data, offs.ctypes.data, preds.ctypes.data, cnt.ctypes.data, hid.ctypes.data, lg.ctypes.data)
    if kernel == "stream":
        assert host_harness.g2p_host_predict(*args) == 0
    else:
        assert host_harness.g2p_host_predict_cluster(*args, int(kernel[7:])) == 0
    for i, w in enumerate(words):
        p, h, l0 = gn.predict_word(m, w)
        assert np.abs(hid[i] - h).max() < 2e-5 and np.abs(lg[i] - l0).max() < 1e-4, w
        assert preds[i, :cnt[i]].tolist() == p, (w, preds[i], p)


def test_g2p_fails_loudly_without_gpu(native_lib):
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from summertts_b200 import engine

    with pytest.raises(engine.SttsError):
        engine.G2p(_synth_section())


# ------------------------------------------------------------------------------------------------ GPU parity (C ABI)
KERNELS = [0, 1, 2]   # 0 = g2p_words_kernel (streaming), 1 = g2p_cluster_kernel (cluster-resident weights, DSMEM exchange), 2 = per call (default)


def _make(sec, kernel):
    from summertts_b200 import engine

    old = os.environ.get("STTS_G2P_KERNEL")
    os.environ["STTS_G2P_KERNEL"] = str(kernel)
    try:
        g = engine.G2p(sec, device=0)
    finally:
        if old is None:
            del os.environ["STTS_G2P_KERNEL"]
        else:
            os.environ["STTS_G2P_KERNEL"] = old
    assert g.kernel == kernel, "kernel %d not selected (clusters admitted: %d)" % (kernel, g.clusters)
    return g


def _check_gpu(sec, words, want=None, live=None, kernel=0):
    m = gn.parse_section(sec)
    g = _make(sec, kernel)
    assert g.consumed == m["consumed"] and g.hidden == m["enc_w_hh"].shape[1] and g.phones == m["fc_w"].shape[0]
    got, hid, lg = g.predict(words, debug=True)
    assert g.kernel_launches() == 3      # two table builds at create + ONE launch for the whole batch
    for i, w in enumerate(words):
        p, h, l0 = live.word(w) if live is not None else gn.predict_word(m, w)
        assert np.abs(hid[i] - h).max() < 2e-5 and np.abs(lg[i] - l0).max() < 1e-4, (w, np.abs(hid[i] - h).max(), np.abs(lg[i] - l0).max())
        assert got[i] == p, (w, got[i], p)
        if want is not None:
            assert got[i] == want[i], (w, got[i], want[i])
    assert g.predict(words) == got       # without the debug outputs; same handle, second launch
    g.close()
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", KERNELS)
def test_gpu_g2p_synthetic_vs_golden(native_lib, kernel):
    _check_gpu(_synth_section(), _words("synth"), _preds("synth"), kernel=kernel)


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", KERNELS)
def test_gpu_g2p_ragged_batches(native_lib, kernel):
    """Word counts that do not fill the last CTA / word group, 1-letter and 300-letter words, bytes outside a..z, another GRU size,
    and more word groups than co-resident clusters (every cluster walks several groups)."""
    sec = _synth_section()
    rng = np.random.default_rng(3)
    long_word = bytes(int(c) for c in rng.integers(97, 123, 300))
    for words in ([b"q"], [b"ab", b"it's", b"\xc3\xa9clair"], [long_word, b"a", b"bc", b"def", b"ghij"], _words("synth")[:13] + [long_word]):
        _check_gpu(sec, words, kernel=kernel)
    many = [bytes(int(c) for c in rng.integers(97, 123, int(rng.integers(2, 15)))) for _ in range(8 * 18 * 3 + 5)]
    _check_gpu(sec, many, kernel=kernel)
    if kernel == 2:       # the per-call choice: clusters up to 2048 words, the streaming kernel above; and it is the default
        g = _make(sec, 2)
        big = (many * 5)[:2100]
        assert g.predict(many[:50]) == [gn.predict_word(gn.parse_section(sec), w)[0] for w in many[:50]] and g.last_kernel() == 1
        got = g.predict(big)
        assert g.last_kernel() == 0 and got[:len(many)] == g.predict(many) and g.last_kernel() == 1
        g.close()
        from summertts_b200 import engine

        assert os.environ.get("STTS_G2P_KERNEL") is None
        d = engine.G2p(sec)
        assert d.kernel == 2
        d.close()
    _check_gpu(gn.synthetic_section(5, hidden=32, emb=24, n_letters=29, n_phones=37, scale=4.0), [b"abcd", b"zyx", b"q", b"hellothere", b"kernel"],
               kernel=kernel)


@pytest.mark.gpu
def test_gpu_g2p_kernels_bit_identical(native_lib):
    """Same accumulation order per output in both kernels: encoder states and logits are bit-identical, not just close."""
    sec, words = _synth_section(), _words("synth")
    a, b = _make(sec, 0), _make(sec, 1)
    pa, ha, la = a.predict(words, debug=True)
    pb, hb, lb = b.predict(words, debug=True)
    assert pa == pb and np.array_equal(ha, hb) and np.array_equal(la, lb)
    a.close(); b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", KERNELS)
def test_gpu_g2p_shipped_model(native_lib, kernel):
    """The shipped English model's GRU: phone ids == golden (compiled reference) and, through the frontend's tables, the IPA ids
    of the reference's unmodified getIPAId; against the live reference too where libstts_ref.so is built.  Without the
    shipped model: the same words through the seeded GRU of the golden (the shipped GRU's sizes), against the oracle."""
    sec = _real_section()
    words = _words("real")
    if sec is None:
        _check_gpu(_synth_section(), words, kernel=kernel)
        return
    live = ref.RefG2p(sec) if ref.available() else None
    got = _check_gpu(sec, words, _preds("real"), live, kernel=kernel)
    want, off = G["real_ipa_ids"], G["real_ipa_offsets"]
    for i, p in enumerate(got):
        assert gn.preds_to_ipa_ids(p) == want[off[i]:off[i + 1]].tolist()
    if live is not None:
        live.close()


@pytest.mark.gpu
def test_gpu_g2p_errors(native_lib):
    from summertts_b200 import engine

    sec = _synth_section()
    with pytest.raises(engine.SttsError) as e:
        engine.G2p(sec[:1000])
    assert e.value.code == engine.STTS_E_FORMAT
    bad = sec.copy()
    bad[0] = 7            # letter table with fewer rows than the ids the frontend emits
    with pytest.raises(engine.SttsError):
        engine.G2p(bad)
    g = engine.G2p(sec)
    with pytest.raises(engine.SttsError) as e:
        g.predict([b"ok", b""])
    assert e.value.code == engine.STTS_E_ARG
    with pytest.raises(engine.SttsError):
        g.predict([])
    assert g.predict([b"still", b"works"]) == [gn.predict_word(gn.parse_section(sec), w)[0] for w in (b"still", b"works")]
    g.close()
