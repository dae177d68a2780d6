/*
 * stts_b200.h — C ABI of the B200-native VITS acoustic+vocoder engine (libstts_b200.so).
 *
 * This is the drop-in boundary for the hot path of huakunyang/SummerTTS: everything that
 * `SynthesizerTrn::infer` does after the text frontend
 * (reference: src/models/SynthesizerTrn.cpp:357-396) and the NN half of its constructor
 * (src/models/SynthesizerTrn.cpp:101-167).  What crosses the boundary is exactly what the
 * reference passes between its frontend and its NN stack:
 *      int32 phoneme ids[T], int32 sid, float lengthScale   ->   int16 pcm[S], S
 * Plain pointers and sizes only; no C++/torch types.  All functions return 0 on success and a
 * negative STTS_E_* code on failure; stts_last_error() gives the message (thread-local).
 *
 * Ownership mirrors the reference (SURVEY.md §8b): the model blob stays owned by the caller and
 * may be freed after stts_create (weights are repacked into device memory); PCM buffers are
 * malloc()-compatible and are released with stts_free() (reference: tts_free_data,
 * src/utils/utils.cpp:34-37).  An engine handle is bound to ONE GPU and ONE caller thread
 * (the reference's SynthesizerTrn is not re-entrant either: SynthesizerTrn.cpp:338).
 *
 * There is no CPU fallback: every entry point that computes fails with STTS_E_CUDA when no
 * sm_100 device is usable.
 */
#ifndef STTS_B200_H_
#define STTS_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define STTS_OK 0
#define STTS_E_ARG (-1)       /* bad argument (null pointer, n < 5 ids, id out of vocabulary ...) */
#define STTS_E_FORMAT (-2)    /* .bin blob truncated / unknown decoder or duration-predictor type */
#define STTS_E_UNSUPPORTED (-3) /* hyper-parameters outside what the kernels implement */
#define STTS_E_CUDA (-4)      /* CUDA runtime failure or no usable device */
#define STTS_E_NOMEM (-5)

typedef struct stts_engine stts_engine;

/* Replaces: SynthesizerTrn::SynthesizerTrn NN section, src/models/SynthesizerTrn.cpp:91-167.
 * `model_bytes` is what ttsLoadModel returns (src/utils/utils.cpp:8-32).  Parses the NN section,
 * repacks the weights into one device arena on GPU `device`.  The frontend tail of the blob is not
 * touched; its start is reported by stts_nn_end_offset. */
int stts_create(const float* model_blob, int64_t model_bytes, int device, stts_engine** out);

/* Replaces: SynthesizerTrn::~SynthesizerTrn, src/models/SynthesizerTrn.cpp:403-416. */
void stts_destroy(stts_engine* e);

/* Float offset at which the frontend tail starts (end of the NN section),
 * src/models/SynthesizerTrn.cpp:167.  The C++ shim hands the rest to the host text frontend. */
int64_t stts_nn_end_offset(const stts_engine* e);

/* Raw speaker count of the model (0 for single-speaker files); SynthesizerTrn::getSpeakerNum
 * (src/models/SynthesizerTrn.cpp:79-89) maps 0 -> 1 in the C++ shim. */
int32_t stts_speaker_num(const stts_engine* e);

/* Header fields (src/models/SynthesizerTrn.cpp:103-106): 0 isMS, 1 langType, 2 durPredType, 3 decType */
int32_t stts_header_field(const stts_engine* e, int32_t which);

/* Replaces: the NN half of SynthesizerTrn::infer, src/models/SynthesizerTrn.cpp:357-396.
 * ids: the phoneme ids produced by the host frontend (:340 / :345-353).  `length_scale` is used as
 * given (the English 0.83 factor, :354, is applied by the caller/shim).  sid out of range -> 0
 * (:366-369).  *pcm is malloc'd (free with stts_free), *n_samples = dataLen. */
int stts_infer_ids(stts_engine* e, const int32_t* ids, int32_t n_ids, int32_t sid, float length_scale,
                   int16_t** pcm, int32_t* n_samples);

/* Batched form of the same call: B independent utterances, ids concatenated, id_offsets[B+1].
 * The reference has no batching (it would loop stts_infer_ids); results are identical to the
 * per-utterance call.  pcm[b] are malloc'd individually; sids / length_scales may be NULL
 * (0 / 1.0).  Host buffers in, host buffers out: H2D and D2H happen inside the call. */
int stts_infer_batch(stts_engine* e, int32_t B, const int32_t* ids_concat, const int32_t* id_offsets,
                     const int32_t* sids, const float* length_scales, int16_t** pcm, int32_t* n_samples);

/* Same, but the PCM of all utterances is written back-to-back into the caller's buffer
 * `pcm_out` (capacity `cap_samples`, pinned host memory recommended); sample_offsets[B+1]. */
int stts_infer_batch_into(stts_engine* e, int32_t B, const int32_t* ids_concat, const int32_t* id_offsets,
                          const int32_t* sids, const float* length_scales, int16_t* pcm_out,
                          int64_t cap_samples, int64_t* sample_offsets);

/* ---- staged form (bench: inputs resident in HBM before the timed region) ------------------- */
/* H2D of ids/offsets/sids/length scales into the engine's device staging area. */
int stts_batch_stage(stts_engine* e, int32_t B, const int32_t* ids_concat, const int32_t* id_offsets,
                     const int32_t* sids, const float* length_scales);
/* Runs the whole forward on the staged batch; PCM stays in device memory.  (One 4*(B+1)-byte
 * device->host read of the frame counts happens inside: the grid of the frame-rate kernels
 * depends on it, SynthesizerTrn.cpp:376-378.)  Returns total samples in *total_samples. */
int stts_batch_run(stts_engine* e, int64_t* total_samples);
/* D2H of the PCM of the last run into pcm_out (capacity cap_samples); sample_offsets[B+1]. */
int stts_batch_fetch(stts_engine* e, int16_t* pcm_out, int64_t cap_samples, int64_t* sample_offsets);

/* ---- test hooks ---------------------------------------------------------------------------- */
/* Forced per-id frame counts replacing ceil(exp(logw)*lengthScale) for the NEXT calls (concatenated
 * over the batch); NULL clears.  Used for shape-stable benches and downstream-stage parity. */
int stts_set_forced_durations(stts_engine* e, const float* w_ceil, int64_t n);

/* ---- seeded sampling (VITS noise_scale / noise_scale_w) ---------------------------------------------------------------------
 * The reference hard-codes noiseScale = 0 (SynthesizerTrn.cpp:357): the prior is never sampled and the stochastic duration
 * predictor starts from z = 0, so every utterance gets the one "mean" prosody.  VITS inference exposes two knobs:
 *   prior:  z_p = m + eps * exp(logs) * noise_scale   (VITS demo default 0.667)
 *   SDP:    z = eps * noise_scale_w before nn_flip(z, 0), stochastic duration predictor only (demo default 0.8; a model with the
 *           FixDurationPredictor has no noise input and ignores it)
 * eps comes from a counter-based Philox4x32-10 keyed by the utterance's 64-bit seed and indexed by position WITHIN the
 * utterance, so the result does not depend on batching, streaming chunks or the GPU it runs on.  A scale of 0 skips its noise
 * term entirely: an utterance with both scales 0 is bit-identical to the deterministic default.  Semantics and the exact random
 * stream: DESIGN.md §12.
 *
 * Sampling for the NEXT staged batches (stts_infer_ids / _batch / _batch_into / stts_batch_stage / stts_infer_stream): n
 * utterances (must equal B of each later batch, else STTS_E_ARG at stage time); noise_scales / noise_scales_w finite, in
 * [0, 10] (a NULL one = 0 for all); seeds NULL = 0 for all.  n = 0 or both scale arrays NULL clears (deterministic, the
 * default).  The shim SynthesizerTrn (the reference's API) never samples. */
int stts_set_sampling(stts_engine* e, int32_t n, const float* noise_scales, const float* noise_scales_w, const uint64_t* seeds);
/* Host-only (no GPU): the normals the device draws for `seed`; stream 0 = prior [rows = frames][cols = channels],
 * 1 = SDP [rows = tokens][cols = 2] (column r = eps_r).  out has rows * cols floats. */
int stts_debug_noise(uint64_t seed, int32_t stream, int64_t rows, int32_t cols, float* out);

/* stts_create with a pre-packed device image on disk (SURVEY.md §8f rank 4; the reference re-parses and copies every weight at every
 * process start, SynthesizerTrn.cpp:91-167 + utils.cpp:8-32).  A missing / stale / foreign image is ignored and rewritten; a
 * matching one (keyed by a hash of the NN section and the library version) supplies every dense conv's packed device representation.
 * *from_image = 1 when the image was used.  image_path NULL or "" = stts_create. */
int stts_create_cached(const float* model_blob, int64_t model_bytes, int device, const char* image_path, stts_engine** out,
                       int32_t* from_image);

/* Chunked / streaming synthesis of one utterance (SURVEY.md §8f rank 1; the reference feeds whole files as one utterance and returns
 * only at the end, test/main.cpp:90-142).  The token-level half (text encoder, duration predictor, length regulator) runs once;
 * flow + decoder then run over chunks of `chunk_frames` frames with a halo covering their receptive field, and `cb` receives each
 * chunk's PCM (a host buffer valid during the call) in order.  The concatenation is bit-identical to stts_infer_ids.
 * *first_chunk_ms: GPU time from the start of the call to the first chunk's PCM on the host. */
typedef void (*stts_pcm_callback)(const int16_t* pcm, int64_t n, void* user);
int stts_infer_stream(stts_engine* e, const int32_t* ids, int32_t n, int32_t sid, float length_scale, int32_t chunk_frames,
                      stts_pcm_callback cb, void* user, float* first_chunk_ms, int64_t* total_samples);

/* Stage tensors of utterance 0 of the last run, time-major [rows][cols] float32.
 * which: 0 xx[T][hidden]  1 m[T][inter]  2 logw[T]  3 w_ceil[T]  4 z_p[F][inter]  5 z[F][inter]
 *        6 o[S] (raw float waveform)  7 logs[T][inter] (only computed when the batch sampled the prior, see
 *        stts_set_sampling).  Returns a malloc'd buffer in *out (stts_free). */
int stts_debug_fetch(stts_engine* e, int32_t which, float** out, int64_t* rows, int64_t* cols);

/* Enable keeping of stage tensors (off by default; costs memory traffic). */
int stts_debug_enable(stts_engine* e, int32_t on);

/* GPU milliseconds of the last stts_batch_run, from CUDA events on the engine's stream:
 * ms[0] text encoder, [1] duration predictor (+frame-count sync), [2] length regulator,
 * [3] flow, [4] decoder, [5] total.  n = capacity of ms. */
int stts_last_timing(const stts_engine* e, float* ms, int32_t n);

/* Per-kernel-class profiler: when enabled, every dense-conv launch of stts_batch_run is bracketed
 * by CUDA events on the engine's stream; fetch returns, per class, the summed GPU milliseconds, the
 * ALGORITHMIC flops (2*MACs of the un-expanded, un-padded convolution) and the launch count
 * accumulated since the last enable.  Arrays have STTS_NUM_CLS entries. */
#define STTS_NUM_CLS 10
#define STTS_CLS_OTHER 0
#define STTS_CLS_ENC 1       /* text-encoder 1x1 / FFN convs (attention excluded) */
#define STTS_CLS_DP 2        /* duration-predictor convs */
#define STTS_CLS_FLOW_IO 3   /* coupling pre / post 1x1 */
#define STTS_CLS_WN_IN 4     /* WN in_layers k5 C->2C with the gate epilogue */
#define STTS_CLS_WN_RS 5     /* WN res_skip 1x1 */
#define STTS_CLS_DEC_PRE 6   /* conv_pre */
#define STTS_CLS_DEC_UP 7    /* ConvTranspose1d upsamplers */
#define STTS_CLS_DEC_RB 8    /* MRF ResBlock1 convs */
#define STTS_CLS_DEC_TAIL 9  /* conv_post / subband_conv_post */
int stts_profile_enable(stts_engine* e, int32_t on);
int stts_profile_fetch(const stts_engine* e, double* ms, double* flops, int64_t* launches);

/* Number of kernels this library launched since creation (all are ours: no cuBLAS/cuDNN). */
int64_t stts_kernel_launches(const stts_engine* e);

/* The cudaStream_t (as void*) all kernels of this engine are launched on. */
void* stts_stream(const stts_engine* e);

/* Conv path selection: 0 = fp32 CUDA-core tiles everywhere, 1 = tcgen05 tensor-core tiles
 * (split-fp16, fp32-accurate) where a layer is eligible (default when the build has it), 2 = throughput mode: as 1, but
 * the fused ResBlock1-pair kernels issue ONE fp16 MMA per K-step (fp16 operands, fp32 accumulate; the residual stream
 * keeps its split-fp16 precision).  Mode 2 trades the <= 1 LSB PCM parity of mode 1 for speed; tolerance in DESIGN.md. */
int stts_set_tensor_path(stts_engine* e, int32_t mode);

/* Batches that were recomputed on the fp32 FFMA tiles because an activation exceeded the range the split-fp16
 * operands of the tensor path can represent (|x| > ~8000); 0 for every shipped model. */
int64_t stts_tensor_fallbacks(const stts_engine* e);

/* Op-level test hook (tests only): runs ONE conv1d record (file format of nn_conv1d.cpp:25-52, or the
 * ConvTranspose1d record of nn_conv1d_transposed.cpp:25-52 when transposed != 0) on x[T][inCh] through
 * the fp32 FFMA tiles (use_tc = 0) or the tcgen05 path (use_tc = 1).  seg_off[nseg+1] packs several
 * utterances (NULL = one).  in_act: 0 none / 1 leaky(slope); epi: 0 store, 1 relu, 4 WN gate, 6 tanh.
 * Returns y (malloc'd, [rows][cols]). */
int stts_test_conv1d(int device, int use_tc, const float* rec, int64_t rec_floats, int transposed, int stride,
                     int pad_override, int dil_override, const float* x, int T, int nseg, const int* seg_off,
                     int in_act, float slope, int epi, float** y, int* rows, int* cols);

/* Op-level test hook (tests only) of the fused ResBlock1 pair kernel (ResBlock1.cpp:55-69, one loop iteration):
 * y = act(x + conv2(leaky_0.1(conv1(leaky_0.1(x))))) with conv1 = rec1 at dilation dil1 (pad = dil1 (k-1)/2), conv2 = rec2
 * (dilation 1), act = leaky 0.1 when out_leaky else identity; x[T][C], C in {32, 64}; mode 0 accurate / 1 throughput.
 * y is malloc'd [T][C].  *flags_out bit 0: an activation left the split-fp16 range. */
int stts_test_rbpair(int device, int mode, const float* rec1, int64_t n1, const float* rec2, int64_t n2, int dil1, const float* x,
                     int T, int nseg, const int* seg_off, int out_leaky, float** y, uint32_t* flags_out);

/* Host-only test hook: packs one conv's weights W[outCh][k][inCh] (the record order of nn_conv1d.cpp:38-41) the way
 * the tensor-core path stores them (split-fp16 hi/lo stages in UMMA core-matrix order, power-of-two pre-scale) -- no GPU
 * needed; the CPU suite checks it against a numpy restatement of the layout.
 * meta[9] = {eligible, NC, nchunks, KC, kchunks, colsplit, merged, usteps, weight exponent}; *halves is malloc'd. */
int stts_debug_pack_weights(const float* w, int32_t k, int32_t inCh, int32_t outCh, int32_t usteps, int32_t* meta,
                            uint16_t** halves, int64_t* n_halves);

/* ---- batched GRU grapheme-to-phoneme for out-of-vocabulary English words (SURVEY.md §8f rank 3) ----------------------
 * Replaces the Eigen GRU the reference's English frontend runs one word at a time: gru_cell / gru
 * (src/engipa/EnglishText2Id.cpp:270-313) and the encoder + greedy decoder of getIPAId (:496-545).  The frontend's
 * dictionary lookup, the phone -> IPA string tables and the IPA -> id map stay on the host (INTEGRATION.md shows the
 * binding inside getIPAId).
 *
 * stts_g2p_create: gru_section points at the 12 GRU records at the start of the English frontend tail, i.e.
 * model_blob + stts_nn_end_offset(e) for an English `.bin` (the constructor EnglishText2Id(modelData, offset),
 * EnglishText2Id.cpp:61-126); *consumed_floats (optional) = floats read, the `offset` the reference constructor returns. */
typedef struct stts_g2p stts_g2p;
int stts_g2p_create(const float* gru_section, int64_t n_floats, int device, stts_g2p** out, int64_t* consumed_floats);
void stts_g2p_destroy(stts_g2p* g);
/* which: 0 hidden size, 1 phone-table size, 2 letter-table size, 3 embedding size, 4 maximum phones per word (20, :527),
 * 5 kernel choice of the handle: 0 = W_hh streamed from L2 every step, 1 = W_hh resident in the shared memory of 8-CTA clusters,
 * 2 = per call (clusters up to 2048 words, streaming above; the default where the device admits the clusters; environment
 * STTS_G2P_KERNEL overrides), 6 co-resident clusters the device admits, 7 kernel of the last stts_g2p_predict (0 / 1). */
int32_t stts_g2p_dim(const stts_g2p* g, int32_t which);
/* One launch for n_words lower-cased words: letters = the words' bytes concatenated, offsets[n_words + 1] their bounds
 * (the reference maps each BYTE: 'a'..'z' -> 3..28, anything else -> <unk>, :496-511).  phones[n_words][20] receives the
 * predicted phone-table ids (the `preds` of :542), n_phones[n_words] their count.  Optional outputs (NULL to skip):
 * enc_hidden[n_words][hidden] = encoder state after </s> (:519), first_logits[n_words][phones] = logits of the first
 * decoder step (:534).  Host buffers; returns after the results are in them. */
int stts_g2p_predict(stts_g2p* g, int32_t n_words, const char* letters, const int32_t* offsets, int32_t* phones, int32_t* n_phones,
                     float* enc_hidden, float* first_logits);
int64_t stts_g2p_kernel_launches(const stts_g2p* g);

/* Replaces: tts_free_data, src/utils/utils.cpp:34-37. */
void stts_free(void* p);

const char* stts_last_error(void);

/* Host-only: parse the NN section and return a malloc'd text description of the layer graph
 * (one line per record) — no GPU needed.  Used by the CPU test-suite to check the parser against
 * summertts_b200/binfmt.py.  *nn_end receives the float offset of the frontend tail. */
int stts_describe_model(const float* model_blob, int64_t model_bytes, char** text, int64_t* nn_end);

const char* stts_version(void);

#ifdef __cplusplus
}
#endif
#endif /* STTS_B200_H_ */
