"""Host-side mirror of the reference's public interface over the C ABI (include/stts_b200.h).

`SynthesizerTrn` keeps the reference class's names and argument meaning
(/root/reference/include/SynthesizerTrn.h:9-19): ctor(model blob), infer(...), getSpeakerNum().
The reference's infer() takes text; the text frontend is host code that stays unchanged and is out
of scope here (SURVEY.md §2), so this mirror exposes the ID-level entry the frontend feeds
(SynthesizerTrn.cpp:340 / :345-353 -> :357-396): `infer_ids`, plus the batched forms.

All compute goes through libstts_b200.so (hand-written sm_100a kernels).  There is NO fallback:
if the library or a B200 is missing, construction raises.
"""
from __future__ import annotations

import contextlib
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("STTS_B200_LIB") or os.path.join(_HERE, "libstts_b200.so")   # override: instrumented dev builds

# every symbol include/stts_b200.h declares (checked by tests/test_abi.py)
ABI_SYMBOLS = [
    "stts_create", "stts_destroy", "stts_nn_end_offset", "stts_speaker_num", "stts_header_field",
    "stts_infer_ids", "stts_infer_batch", "stts_infer_batch_into", "stts_batch_stage", "stts_batch_run",
    "stts_batch_fetch", "stts_set_forced_durations", "stts_debug_fetch", "stts_debug_enable", "stts_last_timing",
    "stts_kernel_launches", "stts_stream", "stts_set_tensor_path", "stts_free", "stts_last_error",
    "stts_describe_model", "stts_version", "stts_profile_enable", "stts_profile_fetch",
    "stts_test_conv1d", "stts_debug_pack_weights", "stts_test_rbpair", "stts_tensor_fallbacks", "stts_infer_stream", "stts_create_cached",
    "stts_g2p_create", "stts_g2p_destroy", "stts_g2p_dim", "stts_g2p_predict", "stts_g2p_kernel_launches",
    "stts_set_sampling", "stts_debug_noise",
]

STTS_OK, STTS_E_ARG, STTS_E_FORMAT, STTS_E_UNSUPPORTED, STTS_E_CUDA, STTS_E_NOMEM = 0, -1, -2, -3, -4, -5   # include/stts_b200.h

_lib = None


class SttsError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("stts_b200 error %d: %s" % (code, msg))
        self.code = code


def load_library():
    """dlopen libstts_b200.so (built in-tree by summertts_b200.build). Raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError("libstts_b200.so is not built (run `python -m summertts_b200.build` or "
                          "__graft_entry__.build()); there is no CPU fallback")
    L = C.CDLL(LIB_PATH)
    vp, i32, i64, f32 = C.c_void_p, C.c_int32, C.c_int64, C.c_float
    L.stts_create.argtypes = [vp, i64, C.c_int, C.POINTER(vp)]
    L.stts_destroy.argtypes = [vp]
    L.stts_destroy.restype = None
    L.stts_nn_end_offset.argtypes = [vp]
    L.stts_nn_end_offset.restype = i64
    L.stts_speaker_num.argtypes = [vp]
    L.stts_speaker_num.restype = i32
    L.stts_header_field.argtypes = [vp, i32]
    L.stts_header_field.restype = i32
    L.stts_infer_ids.argtypes = [vp, vp, i32, i32, f32, C.POINTER(vp), C.POINTER(i32)]
    L.stts_infer_batch.argtypes = [vp, i32, vp, vp, vp, vp, vp, vp]
    L.stts_infer_batch_into.argtypes = [vp, i32, vp, vp, vp, vp, vp, i64, vp]
    L.stts_batch_stage.argtypes = [vp, i32, vp, vp, vp, vp]
    L.stts_batch_run.argtypes = [vp, C.POINTER(i64)]
    L.stts_batch_fetch.argtypes = [vp, vp, i64, vp]
    L.stts_set_forced_durations.argtypes = [vp, vp, i64]
    L.stts_set_sampling.argtypes = [vp, i32, vp, vp, vp]
    L.stts_debug_noise.argtypes = [C.c_uint64, i32, i64, i32, vp]
    L.stts_debug_fetch.argtypes = [vp, i32, C.POINTER(vp), C.POINTER(i64), C.POINTER(i64)]
    L.stts_debug_enable.argtypes = [vp, i32]
    L.stts_last_timing.argtypes = [vp, vp, i32]
    L.stts_profile_enable.argtypes = [vp, i32]
    L.stts_profile_fetch.argtypes = [vp, vp, vp, vp]
    L.stts_test_conv1d.argtypes = [C.c_int, C.c_int, vp, i64, C.c_int, C.c_int, C.c_int, C.c_int, vp, C.c_int, C.c_int, vp,
                                   C.c_int, f32, C.c_int, C.POINTER(vp), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.stts_debug_pack_weights.argtypes = [vp, i32, i32, i32, i32, vp, C.POINTER(vp), C.POINTER(i64)]
    L.stts_kernel_launches.argtypes = [vp]
    L.stts_kernel_launches.restype = i64
    L.stts_tensor_fallbacks.argtypes = [vp]
    L.stts_tensor_fallbacks.restype = i64
    L.stts_stream.argtypes = [vp]
    L.stts_stream.restype = vp
    L.stts_set_tensor_path.argtypes = [vp, i32]
    L.stts_free.argtypes = [vp]
    L.stts_free.restype = None
    L.stts_last_error.restype = C.c_char_p
    L.stts_describe_model.argtypes = [vp, i64, C.POINTER(vp), C.POINTER(i64)]
    L.stts_version.restype = C.c_char_p
    _lib = L
    return L


def _check(rc):
    if rc != 0:
        raise SttsError(rc, load_library().stts_last_error().decode("utf-8", "replace"))


def describe_model(blob: np.ndarray):
    """Host-only parse of the NN section through the C ABI. Returns (text, nn_end)."""
    L = load_library()
    blob = np.ascontiguousarray(blob, dtype=np.float32)
    txt, end = C.c_void_p(), C.c_int64()
    _check(L.stts_describe_model(blob.ctypes.data, blob.nbytes, C.byref(txt), C.byref(end)))
    s = C.string_at(txt.value).decode()
    L.stts_free(txt)
    return s, end.value


def debug_noise(seed: int, stream: int, rows: int, cols: int = 2) -> np.ndarray:
    """Host-only: the normals the device draws for `seed` (stts_debug_noise); stream 0 = prior [frames][channels],
    1 = stochastic duration predictor [tokens][2]."""
    L = load_library()
    out = np.empty((rows, cols), np.float32)
    _check(L.stts_debug_noise(int(seed) & (2 ** 64 - 1), int(stream), int(rows), int(cols), out.ctypes.data))
    return out


STAGES = {"xx": 0, "m": 1, "logw": 2, "w_ceil": 3, "z_p": 4, "z": 5, "o": 6, "logs": 7}


class SynthesizerTrn:
    """Drop-in mirror of the reference class (include/SynthesizerTrn.h:9-19) at the ID level."""

    def __init__(self, model_data: np.ndarray, model_size: int | None = None, device: int = 0, image_path: str | None = None):
        """image_path: optional pre-packed device image (stts_create_cached); `self.from_image` tells whether it was used."""
        L = load_library()
        blob = np.ascontiguousarray(model_data, dtype=np.float32)
        nbytes = blob.nbytes if model_size is None else int(model_size)
        h = C.c_void_p()
        self.from_image = False
        if image_path:
            used = C.c_int32(0)
            L.stts_create_cached.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_char_p, C.POINTER(C.c_void_p), C.POINTER(C.c_int32)]
            _check(L.stts_create_cached(blob.ctypes.data, nbytes, int(device), image_path.encode(), C.byref(h), C.byref(used)))
            self.from_image = bool(used.value)
        else:
            _check(L.stts_create(blob.ctypes.data, nbytes, int(device), C.byref(h)))
        self._h = h
        self._L = L
        self.lang_type = L.stts_header_field(h, 1)
        self.dec_type = L.stts_header_field(h, 3)
        self.nn_end = int(L.stts_nn_end_offset(h))   # float offset of the frontend tail (SynthesizerTrn.cpp:167)

    # -- reference API ---------------------------------------------------------------------------
    def getSpeakerNum(self) -> int:
        n = self._L.stts_speaker_num(self._h)
        return 1 if n == 0 else n  # SynthesizerTrn.cpp:83-86

    def infer_ids(self, ids, sid: int = 0, length_scale: float = 1.0, noise_scale=0.0, noise_scale_w=0.0, seed=0) -> np.ndarray:
        """NN half of SynthesizerTrn::infer for one utterance; returns int16 PCM.  noise_scale / noise_scale_w / seed: seeded
        sampling (set_sampling); the defaults give the reference's deterministic output."""
        ids = np.ascontiguousarray(ids, dtype=np.int32)
        p, n = C.c_void_p(), C.c_int32()
        with self._sampling(1, noise_scale, noise_scale_w, seed):
            _check(self._L.stts_infer_ids(self._h, ids.ctypes.data, ids.size, int(sid), float(length_scale),
                                          C.byref(p), C.byref(n)))
        out = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_int16)), shape=(max(n.value, 1),))[:n.value].copy()
        self._L.stts_free(p)
        return out

    # -- batched / staged forms ------------------------------------------------------------------
    @staticmethod
    def _pack(id_lists):
        offs = np.zeros(len(id_lists) + 1, dtype=np.int32)
        offs[1:] = np.cumsum([len(x) for x in id_lists])
        ids = np.ascontiguousarray(np.concatenate([np.asarray(x, dtype=np.int32) for x in id_lists]), dtype=np.int32)
        return ids, offs

    def infer_batch(self, id_lists, sids=None, length_scales=None, noise_scale=0.0, noise_scale_w=0.0, seed=0):
        """B utterances -> list of int16 arrays (host buffers in, host buffers out).  noise_scale / noise_scale_w / seed:
        scalars or per-utterance arrays (set_sampling)."""
        ids, offs = self._pack(id_lists)
        B = len(id_lists)
        s = None if sids is None else np.ascontiguousarray(sids, dtype=np.int32)
        ls = None if length_scales is None else np.ascontiguousarray(length_scales, dtype=np.float32)
        ptrs = (C.c_void_p * B)()
        ns = (C.c_int32 * B)()
        with self._sampling(B, noise_scale, noise_scale_w, seed):
            _check(self._L.stts_infer_batch(self._h, B, ids.ctypes.data, offs.ctypes.data,
                                            None if s is None else s.ctypes.data, None if ls is None else ls.ctypes.data,
                                            ptrs, ns))
        outs = []
        for b in range(B):
            a = np.ctypeslib.as_array(C.cast(ptrs[b], C.POINTER(C.c_int16)), shape=(max(ns[b], 1),))[:ns[b]].copy()
            self._L.stts_free(ptrs[b])
            outs.append(a)
        return outs

    def infer_batch_into(self, ids, offs, sids, length_scales, pcm_out: np.ndarray, sample_offsets: np.ndarray):
        """Raw C-ABI call with caller-owned (ideally pinned) buffers; used by bench.py's e2e leg."""
        _check(self._L.stts_infer_batch_into(
            self._h, len(offs) - 1, ids.ctypes.data, offs.ctypes.data,
            None if sids is None else sids.ctypes.data, None if length_scales is None else length_scales.ctypes.data,
            pcm_out.ctypes.data, pcm_out.size, sample_offsets.ctypes.data))

    def stage(self, id_lists, sids=None, length_scales=None, noise_scale=0.0, noise_scale_w=0.0, seed=0):
        ids, offs = self._pack(id_lists)
        s = None if sids is None else np.ascontiguousarray(sids, dtype=np.int32)
        ls = None if length_scales is None else np.ascontiguousarray(length_scales, dtype=np.float32)
        with self._sampling(len(id_lists), noise_scale, noise_scale_w, seed):
            _check(self._L.stts_batch_stage(self._h, len(id_lists), ids.ctypes.data, offs.ctypes.data,
                                            None if s is None else s.ctypes.data, None if ls is None else ls.ctypes.data))

    def run(self) -> int:
        tot = C.c_int64()
        _check(self._L.stts_batch_run(self._h, C.byref(tot)))
        return tot.value

    def fetch(self, total: int, B: int):
        pcm = np.empty(max(total, 1), dtype=np.int16)
        so = np.zeros(B + 1, dtype=np.int64)
        _check(self._L.stts_batch_fetch(self._h, pcm.ctypes.data, pcm.size, so.ctypes.data))
        return pcm[:total], so

    # -- seeded sampling ---------------------------------------------------------------------------
    def set_sampling(self, noise_scales=None, noise_scales_w=None, seeds=None):
        """stts_set_sampling for the next staged batches: per-utterance arrays (their length must equal each later batch's
        size); None for both scales clears (deterministic, the default)."""
        if noise_scales is None and noise_scales_w is None:
            _check(self._L.stts_set_sampling(self._h, 0, None, None, None))
            return
        arrs = [None if a is None else np.ascontiguousarray(np.atleast_1d(a), dtype=dt)
                for a, dt in ((noise_scales, np.float32), (noise_scales_w, np.float32), (seeds, np.uint64))]
        n = max(a.size for a in arrs if a is not None)
        if any(a is not None and a.size != n for a in arrs):
            raise ValueError("noise_scales, noise_scales_w and seeds must have the same length")
        _check(self._L.stts_set_sampling(self._h, n, *[None if a is None else a.ctypes.data for a in arrs]))

    @contextlib.contextmanager
    def _sampling(self, B, noise_scale, noise_scale_w, seed):
        """Per-call sampling of the keyword forms: scalars are broadcast to the B utterances; set before the call and cleared
        after it.  All-zero scales leave the engine's sampling state alone (the deterministic path)."""
        if not (np.any(np.asarray(noise_scale) != 0) or np.any(np.asarray(noise_scale_w) != 0)):
            yield
            return
        seeds = np.broadcast_to(np.asarray(seed, dtype=np.uint64), (B,))
        self.set_sampling(np.broadcast_to(np.asarray(noise_scale, np.float32), (B,)),
                          np.broadcast_to(np.asarray(noise_scale_w, np.float32), (B,)), seeds)
        try:
            yield
        finally:
            self.set_sampling(None)

    # -- test hooks --------------------------------------------------------------------------------
    def set_forced_durations(self, w):
        if w is None:
            _check(self._L.stts_set_forced_durations(self._h, None, 0))
        else:
            w = np.ascontiguousarray(w, dtype=np.float32)
            _check(self._L.stts_set_forced_durations(self._h, w.ctypes.data, w.size))

    def debug_enable(self, on=True):
        _check(self._L.stts_debug_enable(self._h, 1 if on else 0))

    def debug_fetch(self, name: str) -> np.ndarray:
        p, r, c = C.c_void_p(), C.c_int64(), C.c_int64()
        _check(self._L.stts_debug_fetch(self._h, STAGES[name], C.byref(p), C.byref(r), C.byref(c)))
        n = r.value * c.value
        a = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_float)), shape=(max(n, 1),))[:n].copy()
        self._L.stts_free(p)
        return a.reshape(r.value, c.value) if c.value > 1 else a

    def last_timing(self) -> dict:
        ms = (C.c_float * 6)()
        _check(self._L.stts_last_timing(self._h, ms, 6))
        return dict(zip(("enc", "dp", "regulate", "flow", "dec", "total"), [float(v) for v in ms]))

    CLASSES = ("other", "enc", "dp", "flow_io", "wn_in", "wn_rs", "dec_pre", "dec_up", "dec_rb", "dec_tail")

    def profile_enable(self, on=True):
        _check(self._L.stts_profile_enable(self._h, 1 if on else 0))

    def profile_fetch(self) -> dict:
        n = len(self.CLASSES)
        ms, fl, ln = (C.c_double * n)(), (C.c_double * n)(), (C.c_int64 * n)()
        _check(self._L.stts_profile_fetch(self._h, ms, fl, ln))
        return {c: dict(ms=ms[i], flops=fl[i], launches=int(ln[i])) for i, c in enumerate(self.CLASSES)}

    def kernel_launches(self) -> int:
        return int(self._L.stts_kernel_launches(self._h))

    def infer_stream(self, ids, sid=0, length_scale=1.0, chunk_frames=128, noise_scale=0.0, noise_scale_w=0.0, seed=0):
        """Chunked synthesis: returns (list of per-chunk int16 arrays in emission order, GPU ms to the first chunk).  With the
        same seed and scales, the chunks concatenate to the one-shot infer_ids result."""
        ids = np.ascontiguousarray(ids, dtype=np.int32)
        chunks = []
        CB = C.CFUNCTYPE(None, C.POINTER(C.c_int16), C.c_int64, C.c_void_p)

        def on_pcm(ptr, n, _user):
            chunks.append(np.ctypeslib.as_array(ptr, shape=(n,)).copy())

        cb = CB(on_pcm)
        first, total = C.c_float(0), C.c_int64(0)
        self._L.stts_infer_stream.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_float, C.c_int32, CB, C.c_void_p,
                                              C.POINTER(C.c_float), C.POINTER(C.c_int64)]
        with self._sampling(1, noise_scale, noise_scale_w, seed):
            _check(self._L.stts_infer_stream(self._h, ids.ctypes.data, ids.size, int(sid), float(length_scale), int(chunk_frames), cb,
                                             None, C.byref(first), C.byref(total)))
        assert total.value == sum(c.size for c in chunks)
        return chunks, float(first.value)

    def tensor_fallbacks(self) -> int:
        """Batches recomputed on the fp32 FFMA tiles because an activation left the split-fp16 range."""
        return int(self._L.stts_tensor_fallbacks(self._h))

    def stream(self) -> int:
        return int(self._L.stts_stream(self._h) or 0)

    def set_tensor_path(self, mode: int):
        _check(self._L.stts_set_tensor_path(self._h, int(mode)))

    def close(self):
        if getattr(self, "_h", None):
            self._L.stts_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def test_conv1d(rec, x, use_tc=0, transposed=False, stride=1, pad=-1, dil=0, seg_off=None, in_act=0, slope=0.0, epi=0,
                device=0):
    """Op-level hook: one conv record through the FFMA tiles or the tcgen05 path (tests only)."""
    L = load_library()
    rec = np.ascontiguousarray(rec, dtype=np.float32)
    x = np.ascontiguousarray(x, dtype=np.float32)
    so = None if seg_off is None else np.ascontiguousarray(seg_off, dtype=np.int32)
    y, r, c = C.c_void_p(), C.c_int(), C.c_int()
    _check(L.stts_test_conv1d(device, int(use_tc), rec.ctypes.data, rec.size, 1 if transposed else 0, int(stride), int(pad),
                              int(dil), x.ctypes.data, x.shape[0], 0 if so is None else so.size - 1,
                              None if so is None else so.ctypes.data, int(in_act), float(slope), int(epi),
                              C.byref(y), C.byref(r), C.byref(c)))
    n = r.value * c.value
    out = np.ctypeslib.as_array(C.cast(y, C.POINTER(C.c_float)), shape=(n,)).copy().reshape(r.value, c.value)
    L.stts_free(y)
    return out


def test_rbpair(rec1, rec2, x, dil1=1, mode=0, seg_off=None, out_leaky=True, device=0):
    """Op-level hook: one fused ResBlock1 pair (rb_fused.cuh) on x[T][C]; returns (y, flags)."""
    L = load_library()
    L.stts_test_rbpair.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int,
                                   C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_uint32)]
    rec1 = np.ascontiguousarray(rec1, dtype=np.float32)
    rec2 = np.ascontiguousarray(rec2, dtype=np.float32)
    x = np.ascontiguousarray(x, dtype=np.float32)
    so = None if seg_off is None else np.ascontiguousarray(seg_off, dtype=np.int32)
    y, fl = C.c_void_p(), C.c_uint32(0)
    _check(L.stts_test_rbpair(device, int(mode), rec1.ctypes.data, rec1.size, rec2.ctypes.data, rec2.size, int(dil1), x.ctypes.data,
                              x.shape[0], 0 if so is None else so.size - 1, None if so is None else so.ctypes.data,
                              1 if out_leaky else 0, C.byref(y), C.byref(fl)))
    out = np.ctypeslib.as_array(C.cast(y, C.POINTER(C.c_float)), shape=(x.size,)).copy().reshape(x.shape)
    L.stts_free(y)
    return out, int(fl.value)


def debug_pack_weights(w, usteps=0):
    """Host-only hook: tensor-path packing of one conv's weights W[outCh][k][inCh] -> (meta dict, uint16 fp16 bit patterns)."""
    L = load_library()
    w = np.ascontiguousarray(w, dtype=np.float32)
    o, k, c = w.shape
    meta = np.zeros(9, np.int32)
    h, n = C.c_void_p(), C.c_int64()
    _check(L.stts_debug_pack_weights(w.ctypes.data, k, c, o, int(usteps), meta.ctypes.data, C.byref(h), C.byref(n)))
    names = ["eligible", "NC", "nchunks", "KC", "kchunks", "colsplit", "merged", "usteps", "wexp"]
    md = {a: int(b) for a, b in zip(names, meta)}
    if not h.value:
        return md, np.zeros(0, np.uint16)
    out = np.ctypeslib.as_array(C.cast(h, C.POINTER(C.c_uint16)), shape=(n.value,)).copy()
    L.stts_free(h)
    return md, out


def ttsLoadModel(path: str) -> np.ndarray:
    """Mirror of ttsLoadModel (src/utils/utils.cpp:8-32): whole file as float32."""
    return np.fromfile(path, dtype=np.float32)


class G2p:
    """Batched GRU grapheme-to-phoneme on the GPU (stts_g2p_*): the out-of-vocabulary branch of the reference's
    EnglishText2Id::getIPAId (src/engipa/EnglishText2Id.cpp:496-545) for many words in one launch.
    `section` = the English model's floats from stts_nn_end_offset on (the reference constructor's `modelData + offset`)."""

    def __init__(self, section: np.ndarray, device: int = 0):
        self._L = L = load_library()
        vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
        L.stts_g2p_create.argtypes = [vp, i64, C.c_int, C.POINTER(vp), C.POINTER(i64)]
        L.stts_g2p_destroy.argtypes = [vp]
        L.stts_g2p_dim.argtypes = [vp, i32]
        L.stts_g2p_dim.restype = i32
        L.stts_g2p_predict.argtypes = [vp, i32, vp, vp, vp, vp, vp, vp]
        L.stts_g2p_kernel_launches.argtypes = [vp]
        L.stts_g2p_kernel_launches.restype = i64
        sec = np.ascontiguousarray(section, dtype=np.float32)
        h, used = vp(), i64()
        _check(L.stts_g2p_create(sec.ctypes.data, sec.size, int(device), C.byref(h), C.byref(used)))
        self._h = h
        self.consumed = int(used.value)
        self.hidden, self.phones, self.letters, self.emb, self.max_steps = (int(L.stts_g2p_dim(h, k)) for k in range(5))
        self.kernel, self.clusters = int(L.stts_g2p_dim(h, 5)), int(L.stts_g2p_dim(h, 6))   # 0 streaming / 1 cluster-resident / 2 per call; co-resident clusters

    def predict(self, words, debug: bool = False):
        """words: lower-cased str / bytes.  Returns a list of phone-id lists (+ encoder states and first-step logits when debug)."""
        ws = [w.encode("utf-8") if isinstance(w, str) else bytes(w) for w in words]
        n = len(ws)
        letters = np.frombuffer(b"".join(ws) or b"\0", dtype=np.uint8).copy()
        offs = np.zeros(n + 1, np.int32)
        offs[1:] = np.cumsum([len(w) for w in ws])
        preds = np.zeros((max(n, 1), self.max_steps), np.int32)
        cnt = np.zeros(max(n, 1), np.int32)
        hid = np.zeros((max(n, 1), self.hidden), np.float32) if debug else None
        lg = np.zeros((max(n, 1), self.phones), np.float32) if debug else None
        _check(self._L.stts_g2p_predict(self._h, n, letters.ctypes.data, offs.ctypes.data, preds.ctypes.data, cnt.ctypes.data,
                                        hid.ctypes.data if debug else None, lg.ctypes.data if debug else None))
        out = [preds[i, :cnt[i]].tolist() for i in range(n)]
        return (out, hid, lg) if debug else out

    def kernel_launches(self) -> int:
        return int(self._L.stts_g2p_kernel_launches(self._h))

    def last_kernel(self) -> int:
        """Kernel of the last predict: 0 streaming, 1 cluster-resident."""
        return int(self._L.stts_g2p_dim(self._h, 7))

    def close(self):
        if getattr(self, "_h", None):
            self._L.stts_g2p_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
