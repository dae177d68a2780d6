// engine.cu — host orchestration + C ABI (include/stts_b200.h) of the B200-native VITS engine.
//
// Replaces, behind the C ABI, the NN half of the reference's SynthesizerTrn
// (src/models/SynthesizerTrn.cpp:91-167 ctor, :357-396 infer) and every src/models, src/modules,
// src/nn_op call underneath it.  One engine = one GPU, one stream; a batch of utterances is packed
// along the row dimension (see kernels.cuh).  There is no CPU fallback anywhere in this file.
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>   // header-only; ranges are no-ops unless a profiler (nsys / ncu --nvtx) is attached

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <stdexcept>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/stts_b200.h"
#include "kernels.cuh"
#include "nb_fused.cuh"
#include "model.hpp"
#ifdef STTS_WITH_TC
#include "conv_tc.cuh"
#include "rb_fused.cuh"
#include "pc_fused.cuh"
#endif

namespace stts {

struct CudaError : std::runtime_error {
    using std::runtime_error::runtime_error;
};
struct ArgError : std::runtime_error {
    using std::runtime_error::runtime_error;
};
struct Unsupported : std::runtime_error {
    using std::runtime_error::runtime_error;
};

#define CUDA_CHECK(expr)                                                                                   \
    do {                                                                                                   \
        cudaError_t _e = (expr);                                                                           \
        if (_e != cudaSuccess)                                                                             \
            throw CudaError(std::string(#expr) + " failed: " + cudaGetErrorString(_e) + " (" __FILE__ ":" +  \
                            std::to_string(__LINE__) + ")");                                               \
    } while (0)

static thread_local std::string g_last_error;

struct NvtxRange {           // one range per pipeline stage of run(): text encoder / duration predictor / regulator / flow / decoder
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
};

// ---------------------------------------------------------------------------------------------
// device-side weight records
// ---------------------------------------------------------------------------------------------
struct DConv {
    float* w = nullptr;  // [k][Cin][CoutW]
    float* b = nullptr;  // [Cout] or null
    int Cin = 0, Cout = 0, CoutW = 0, k = 1, dil = 1, padl = 0;
    double macs_row = 0;  // algorithmic MACs per input-rate row (un-expanded taps, live outputs only)
#ifdef STTS_WITH_TC
    TcWeights tc;        // split-fp16 UMMA-layout copy (filled when the layer is tensor-path eligible)
    RbWeights rb;        // merged split-fp16 stages for the fused ResBlock1-pair kernel (rb_fused.cuh), ResBlock1 convs only
    PcWeights pc;        // 64-column chunk stages for the staged-epilogue wide conv (pc_fused.cuh), WN in_layers / res_skip only
#endif
};
struct DLN {
    float *g = nullptr, *b = nullptr;
    int C = 0;
};
struct DDds {
    int n = 0, k = 3, C = 0;
    std::vector<float*> sw, sb;  // depthwise [k][C], bias
    std::vector<int> sdil, spad;
    std::vector<DConv> c11;
    std::vector<DLN> n1, n2;
};
struct DConvFlow {
    float *prew = nullptr, *preb = nullptr;  // 1 -> C
    DDds dds;
    DConv proj;
    float fsqrt = 1.f;
};

struct ConvOpts {
    int in_act = ACT_NONE;
    float in_slope = 0.f;
    int epi = EPI_STORE;
    float div = 1.f;
    const float* res = nullptr; int ldr = 0;
    const float* gvec = nullptr; int ldg = 0;
    float* y2 = nullptr; int ldy2 = 0;
    int split = 0, y2_store = 0;
    bool allow_tc = true;
#ifdef STTS_WITH_TC
    const Planes* in_planes = nullptr;   // input already available as split-fp16 planes (activation applied by its producer)
    Planes* out_planes = nullptr;        // also emit y as planes (through out_act) for the next tensor-core conv
    Planes* out2_planes = nullptr;       // EPI_RESSKIP: planes of the skip destination
    int out_act = ACT_NONE; float out_slope = 0.f;
    bool write_f32 = true;               // false: planes only (the fp32 tensor has no other reader)
    // tile-transposed fp32 tensors (conv_tc.cuh, TcP): private to tensor-core epilogues
    bool y_tt = false, y2_tt = false, res_tt = false, acc_tt = false;
    const float* acc_src = nullptr;      // EPI_ACCUM(_DIV): accumulate onto this tensor instead of y
#endif
};

struct Arena {  // bump allocator over one device allocation
    char* base = nullptr;
    size_t cap = 0, off = 0;
    void reset() { off = 0; }
    template <typename T>
    T* get(size_t n) {
        size_t bytes = (n * sizeof(T) + 255) & ~size_t(255);
        if (off + bytes > cap) throw std::runtime_error("workspace arena overflow (planning bug)");
        T* p = reinterpret_cast<T*>(base + off);
        off += bytes;
        return p;
    }
};

}  // namespace stts

using namespace stts;

struct stts_engine {
    int device = 0;
    cudaStream_t stream = nullptr;
    int64_t launches = 0;
    int tensor_mode = 1;
    bool debug = false;

    // model
    int isMS = 0, langType = 0, durPredType = 1, decType = 1, spkNum = 0, gin = 0;
    int64_t nnEnd = 0;
    int hidden = 192, vocab = 0, inter = 192, nHeads = 2, kc = 96, win = 4, relRows = 9, nEnc = 0;
    int wnHidden = 192;
    std::vector<void*> owned;  // all device weight allocations

    float* emb = nullptr;
    struct EncL {
        DConv qkv, o, f1, f2;
        DLN n1, n2;
        float *ek = nullptr, *ev = nullptr;
    };
    std::vector<EncL> enc;
    DConv encProj, encProjLogs;   // the m / logs halves of TextEncoder's proj
    // fix dp
    DConv dp1, dp2, dpProj, dpCond;
    DLN dpn1, dpn2;
    // stochastic dp
    DConv sdpPre, sdpProj, sdpCond;
    DDds sdpConvs;
    std::vector<DConvFlow> sdpFlows;
    float eaM0 = 0.f, eaLogs0 = 0.f;
    int sdpNFlows = 0;
    // flow
    struct CoupL {
        DConv pre, post, cond;
        std::vector<DConv> in, rs;
        bool hasCond = false;
    };
    std::vector<CoupL> flow;
    int flowN = 0, wnLayers = 0;
    // decoder
    DConv convPre, decCond, convPost, subPost;
    bool decHasCond = false;
    std::vector<DConv> ups;
    std::vector<int> upRates;
    struct RB {
        std::vector<DConv> c1, c2;
        std::vector<std::vector<float>> hw1, hb1, hw2, hb2;   // host copies of narrow (<= 8 channel) pairs: kernel-parameter weights of nb_fused.cuh
    };
    std::vector<RB> rbs;
    int nRbK = 0;
    std::vector<int> stageC;  // channels after each upsample
    float* msW = nullptr;     // [63][4] synthesis FIR (learned or PQMF)
    float* msB = nullptr;
    int subBands = 4;
    float* emg = nullptr;

    // workspace
    Arena ws;
    void* wsAlloc = nullptr;
    int16_t* hostPcm = nullptr;  // pinned staging
    size_t hostPcmCap = 0;
    int* hostInts = nullptr;     // pinned: nframes etc.
    size_t hostIntsCap = 0;

    // staged batch (device)
    int B = 0, Tt = 0, maxT = 0;
    std::vector<int> h_toff, h_foff;
    int* d_ids = nullptr; int* d_toff = nullptr; int* d_sids = nullptr; float* d_ls = nullptr;
    int* d_foff = nullptr; int* d_nfr = nullptr; int* d_bseg = nullptr;
    float* d_forced = nullptr;
    size_t stageCapTok = 0, stageCapB = 0;
    std::vector<float> forced;
    // seeded sampling (stts_set_sampling): per-utterance noise_scale / noise_scale_w / seed for the next staged batches; empty =
    // deterministic.  Staged copies on the device and whether the staged batch samples the prior / the SDP noise at all.
    std::vector<float> smpNs, smpNsw;
    std::vector<uint64_t> smpSeed;
    float* d_ns = nullptr; float* d_nsw = nullptr; unsigned long long* d_seed = nullptr;
    bool samplePrior = false, sampleSdp = false;
    // last-run results
    int Ft = 0, maxF = 0;
    int64_t St = 0;
    std::vector<int64_t> h_soff;
    int16_t* d_pcm = nullptr;
    bool runValid = false;       // the last run() completed: d_pcm / dbg / h_soff describe it
    // chunked / streaming synthesis (stts_infer_stream): run() either stops after the length regulator and keeps z_p
    // (stopAfterRegulate), or skips the token-level half and runs flow + decoder on an injected slice of it (injectZ)
    const float* injectZ = nullptr;
    int injectF = 0;
    bool stopAfterRegulate = false;
    float* streamZ = nullptr;
    size_t streamZCap = 0;
    int streamF = 0;
    struct Dbg {
        float *xx = nullptr, *m = nullptr, *logw = nullptr, *wceil = nullptr, *zp = nullptr, *z = nullptr, *o = nullptr, *logs = nullptr;
    } dbg;
    cudaEvent_t ev[7] = {};
    float lastMs[6] = {};
    // per-kernel-class profiler (CUDA events around each conv launch; off by default)
    struct ProfRec { int cls; cudaEvent_t a, b; double flops; };
    bool profOn = false;
    std::vector<cudaEvent_t> profPool;
    size_t profUsed = 0;
    std::vector<ProfRec> profRecs;
    double profMs[STTS_NUM_CLS] = {}, profFlops[STTS_NUM_CLS] = {};
    int64_t profLaunch[STTS_NUM_CLS] = {};
    int64_t curRowsTotal = 0;  // total live rows of the convs being launched (set by run())
    int curCls = 0;
    cudaEvent_t prof_event() {
        if (profUsed == profPool.size()) {
            cudaEvent_t e;
            CUDA_CHECK(cudaEventCreate(&e));
            profPool.push_back(e);
        }
        return profPool[profUsed++];
    }
    void prof_collect() {
        for (auto& r : profRecs) {
            float ms = 0.f;
            CUDA_CHECK(cudaEventElapsedTime(&ms, r.a, r.b));
            profMs[r.cls] += ms; profFlops[r.cls] += r.flops; profLaunch[r.cls] += 1;
        }
        profRecs.clear();
        profUsed = 0;
    }

    // ---- helpers ---------------------------------------------------------------------------
#ifdef STTS_WITH_TC
    void* planeScratch = nullptr;
    size_t planeScratchCap = 0;
    static size_t planes_rows(int64_t rows_total, int nseg) { return (size_t)rows_total + (size_t)2 * nseg * TC_GAP + 512; }   // slack: a 2 x 128-row tile (+ halos) starting at the last valid row stays in the allocation (bulk tile loads do not clip)
    static size_t planes_bytes(int64_t rows_total, int nseg, int C) { return planes_rows(rows_total, nseg) * (size_t)C * 4; }
    Planes scratch_planes(int64_t rows_total, int nseg, int C) {
        const size_t need = planes_bytes(rows_total, nseg, C);
        if (need > planeScratchCap) {
            CUDA_CHECK(cudaStreamSynchronize(stream));
            if (planeScratch) CUDA_CHECK(cudaFree(planeScratch));
            planeScratchCap = need + need / 2;
            CUDA_CHECK(cudaMalloc(&planeScratch, planeScratchCap));
        }
        Planes pl;
        pl.base = (__half*)planeScratch; pl.C = C; pl.rows_p = (long long)planes_rows(rows_total, nseg);
        return pl;
    }
    Planes arena_planes(int64_t rows_total, int nseg, int C) {
        Planes pl;
        pl.C = C; pl.rows_p = (long long)planes_rows(rows_total, nseg);
        pl.base = ws.get<__half>((size_t)pl.rows_p * C * 2);
        return pl;
    }
    bool tc_layer(const DConv& c) const { return tensor_mode >= 1 && c.tc.ok && (c.k - 1) * c.dil <= TC_GAP && c.padl <= TC_GAP; }
#endif
    template <typename T>
    T* dalloc(size_t n) {
        void* p = nullptr;
        CUDA_CHECK(cudaMalloc(&p, std::max<size_t>(n, 1) * sizeof(T)));
        owned.push_back(p);
        return (T*)p;
    }
    float* upload(const std::vector<float>& v) {
        float* d = dalloc<float>(v.size());
        CUDA_CHECK(cudaMemcpy(d, v.data(), v.size() * sizeof(float), cudaMemcpyHostToDevice));
        return d;
    }
    float* upload(const float* p, size_t n) {
        float* d = dalloc<float>(n);
        CUDA_CHECK(cudaMemcpy(d, p, n * sizeof(float), cudaMemcpyHostToDevice));
        return d;
    }

    int tc_usteps = 4;   // promotion unit (MMA steps) for the layers built next: 4 for token-level layers, 8 from the flow on

    // ---- pre-packed device image (SURVEY.md §8f rank 4) ------------------------------------------------------------------------
    // Every dense conv's device-side representation (fp32 [k][Cin][CoutW], bias, and the packed split-fp16 stages of the three
    // tensor-core kernels) is a DConv + up to five blobs.  In record mode build() appends them to a file in creation order; in
    // replay mode make_conv & co. read the next record instead of transposing / splitting / packing on the host.  The file is
    // keyed by a hash of the NN section, the library version and sizeof(DConv).
    struct Image { int mode = 0; FILE* f = nullptr; int64_t nrec = 0; } img;      // mode 1 record, 2 replay
#ifdef STTS_WITH_TC
    static size_t tc_packed_bytes(const TcWeights& t) { return t.ok ? (size_t)t.nchunks * t.kchunks * t.taps * 2 * t.KC * t.NC * 2 : 0; }
#endif
    void img_put(const void* p, size_t n) { if (fwrite(p, 1, n, img.f) != n) throw std::runtime_error("device image: write failed"); }
    void img_get(void* p, size_t n) { if (fread(p, 1, n, img.f) != n) throw FormatError("device image: truncated"); }
    void img_put_blob(const void* dev, size_t n) {
        const uint64_t n64 = n;
        img_put(&n64, 8);
        if (!n) return;
        std::vector<char> h(n);
        CUDA_CHECK(cudaMemcpy(h.data(), dev, n, cudaMemcpyDeviceToHost));
        img_put(h.data(), n);
    }
    void* img_get_blob(size_t expect) {
        uint64_t n64 = 0;
        img_get(&n64, 8);
        if (n64 != expect) throw FormatError("device image: blob size mismatch");
        if (!n64) return nullptr;
        std::vector<char> h(n64);
        img_get(h.data(), n64);
        void* d = nullptr;
        CUDA_CHECK(cudaMalloc(&d, n64));
        owned.push_back(d);
        CUDA_CHECK(cudaMemcpy(d, h.data(), n64, cudaMemcpyHostToDevice));
        return d;
    }
    void img_record(const DConv& d) {
        if (img.mode != 1) return;
        img_put(&d, sizeof(DConv));
        img_put_blob(d.w, (size_t)d.k * d.Cin * d.CoutW * 4);
        img_put_blob(d.b, d.b ? (size_t)d.Cout * 4 : 0);
#ifdef STTS_WITH_TC
        img_put_blob(d.tc.packed, tc_packed_bytes(d.tc));
        img_put_blob(d.rb.packed, d.rb.ok ? (size_t)d.rb.k * 4 * d.Cin * d.Cin : 0);
        img_put_blob(d.pc.packed, d.pc.ok ? (size_t)d.pc.nchunks * d.pc.nst * PC_STAGE : 0);
#endif
        ++img.nrec;
    }
    // replay: the next record must describe a conv of the expected shape (a stale or foreign image is rejected, not trusted)
    DConv img_replay(int k, int Cin, int Cout) {
        DConv d;
        img_get(&d, sizeof(DConv));
        if (d.k != k || d.Cin != Cin || d.Cout != Cout) throw FormatError("device image: record does not match the model");
        d.w = (float*)img_get_blob((size_t)d.k * d.Cin * d.CoutW * 4);
        const bool hadb = d.b != nullptr;
        d.b = (float*)img_get_blob(hadb ? (size_t)d.Cout * 4 : 0);
#ifdef STTS_WITH_TC
        d.tc.packed = (__half*)img_get_blob(tc_packed_bytes(d.tc));
        d.rb.packed = (__half*)img_get_blob(d.rb.ok ? (size_t)d.rb.k * 4 * d.Cin * d.Cin : 0);
        d.rb.bias = d.b;
        d.pc.packed = (__half*)img_get_blob(d.pc.ok ? (size_t)d.pc.nchunks * d.pc.nst * PC_STAGE : 0);
        d.pc.bias = d.b;
#endif
        ++img.nrec;
        return d;
    }

    // Build a dense conv in device layout [k][Cin'][CoutW'] from a file record W[o][k][c].
    // omap[new_o] = orig_o, cmap[new_c] = orig_c (identity when empty); sign scales w and b.
    DConv make_conv(const ConvRec& r, const std::vector<int>& omap = {}, const std::vector<int>& cmap = {},
                    float sign = 1.f, int padl = -1, bool tc_ok = true, bool rb_pair = false, bool pc_wide = false) {
        if (r.sep) throw Unsupported("depthwise record passed to dense conv builder");
        if (img.mode == 2) return img_replay(r.k, cmap.empty() ? r.inCh : (int)cmap.size(), omap.empty() ? r.outCh : (int)omap.size());
        DConv d;
        d.Cout = omap.empty() ? r.outCh : (int)omap.size();
        d.Cin = cmap.empty() ? r.inCh : (int)cmap.size();
        d.CoutW = (d.Cout + 3) & ~3;
        d.k = r.k; d.dil = r.dil;
        d.padl = padl >= 0 ? padl : r.pad;
        if (padl < 0 && 2 * r.pad != r.dil * (r.k - 1))
            throw Unsupported("conv1d with 2*pad != dil*(k-1) (length-changing conv) is not implemented");
        std::vector<float> w((size_t)d.k * d.Cin * d.CoutW, 0.f);
        for (int o = 0; o < d.Cout; ++o) {
            const int oo = omap.empty() ? o : omap[o];
            for (int kk = 0; kk < d.k; ++kk)
                for (int c = 0; c < d.Cin; ++c) {
                    const int co = cmap.empty() ? c : cmap[c];
                    w[((size_t)kk * d.Cin + c) * d.CoutW + o] = sign * r.w[((size_t)oo * r.k + kk) * r.inCh + co];
                }
        }
        d.w = upload(w);
        d.macs_row = (double)d.Cout * d.Cin * d.k;
        if (r.hasBias == 1) {
            std::vector<float> b(d.Cout);
            for (int o = 0; o < d.Cout; ++o) b[o] = sign * r.b[omap.empty() ? o : omap[o]];
            d.b = upload(b);
        }
#ifdef STTS_WITH_TC
        if (tc_ok) tc_prepare_weights(d.tc, w.data(), d.k, d.Cin, d.Cout, d.CoutW, owned, tc_usteps);
        if (rb_pair && d.Cin == d.Cout) rb_prepare_weights(d.rb, w.data(), d.k, d.Cin, d.CoutW, d.dil, d.padl, d.b, owned);
        if (pc_wide) pc_prepare_weights(d.pc, w.data(), d.k, d.Cin, d.Cout, d.CoutW, d.dil, d.padl, d.b, owned);
#else
        (void)tc_ok; (void)rb_pair; (void)pc_wide;
#endif
        img_record(d);
        return d;
    }

    // ConvTranspose1d -> dense conv with stride*Cout output channels (phase decomposition):
    // y[t*s + r][o] = b[o] + sum_{kk == (r+p) mod s} x[t + (r+p-kk)/s] . W[o][kk][:]
    // (nn_conv1d_transposed.cpp:106-150; requires k - 2p == s so that outLen == s*T, true for every
    // shipped model: Generator_*.cpp "padding = floor((k-u)/2)").
    DConv make_convT(const ConvRec& r) {
        const int s = r.stride, p = r.pad, k = r.k;
        if (r.dil != 1) throw Unsupported("ConvTranspose1d with dilation != 1");
        if (k - 2 * p != s) throw Unsupported("ConvTranspose1d with k - 2*pad != stride");
        if (img.mode == 2) {
            int lo = 1 << 30, hi = -(1 << 30);
            for (int ph = 0; ph < s; ++ph)
                for (int kk = (ph + p) % s; kk < k; kk += s) { lo = std::min(lo, (ph + p - kk) / s); hi = std::max(hi, (ph + p - kk) / s); }
            return img_replay(hi - lo + 1, r.inCh, s * r.outCh);
        }
        int dmin = 1 << 30, dmax = -(1 << 30);
        for (int ph = 0; ph < s; ++ph)
            for (int kk = (ph + p) % s; kk < k; kk += s) {
                const int d = (ph + p - kk) / s;  // exact
                dmin = std::min(dmin, d); dmax = std::max(dmax, d);
            }
        DConv d;
        d.Cin = r.inCh; d.Cout = s * r.outCh; d.CoutW = (d.Cout + 3) & ~3;
        d.k = dmax - dmin + 1; d.dil = 1; d.padl = -dmin;
        std::vector<float> w((size_t)d.k * d.Cin * d.CoutW, 0.f);
        for (int ph = 0; ph < s; ++ph)
            for (int kk = (ph + p) % s; kk < k; kk += s) {
                const int j = (ph + p - kk) / s - dmin;
                for (int o = 0; o < r.outCh; ++o)
                    for (int c = 0; c < r.inCh; ++c)
                        w[((size_t)j * d.Cin + c) * d.CoutW + ph * r.outCh + o] = r.w[((size_t)o * k + kk) * r.inCh + c];
            }
        d.w = upload(w);
        d.macs_row = (double)r.outCh * r.inCh * r.k;  // per INPUT row: every x row meets every tap once
        if (r.hasBias == 1) {
            std::vector<float> b(d.Cout);
            for (int ph = 0; ph < s; ++ph)
                for (int o = 0; o < r.outCh; ++o) b[ph * r.outCh + o] = r.b[o];
            d.b = upload(b);
        }
#ifdef STTS_WITH_TC
        tc_prepare_weights(d.tc, w.data(), d.k, d.Cin, d.Cout, d.CoutW, owned, tc_usteps);
#endif
        img_record(d);
        return d;
    }
    DLN make_ln(const LNormRec& r) {
        DLN d;
        d.C = r.size;
        if (r.size > 1024) throw Unsupported("LayerNorm wider than 1024");
        d.g = upload(r.gamma, r.size);
        d.b = upload(r.beta, r.size);
        return d;
    }
    DDds make_dds(const DdsRec& r) {
        DDds d;
        d.n = r.nLayers; d.k = r.k;
        for (int i = 0; i < r.nLayers; ++i) {
            const ConvRec& s = r.sep[i];
            if (s.inCh != 1) throw Unsupported("DDSConv depthwise record with inCh != 1");
            d.C = s.outCh;
            std::vector<float> w((size_t)s.k * s.outCh);
            for (int c = 0; c < s.outCh; ++c)
                for (int kk = 0; kk < s.k; ++kk) w[(size_t)kk * s.outCh + c] = s.w[(size_t)c * s.k + kk];
            d.sw.push_back(upload(w));
            d.sb.push_back(s.hasBias == 1 ? upload(s.b, s.outCh) : nullptr);
            d.sdil.push_back(s.dil); d.spad.push_back(s.pad);
            d.c11.push_back(make_conv(r.c11[i]));
            d.n1.push_back(make_ln(r.norm1[i]));
            d.n2.push_back(make_ln(r.norm2[i]));
        }
        return d;
    }

    void launch_check() {
        ++launches;
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) throw CudaError(std::string("kernel launch failed: ") + cudaGetErrorString(e));
    }

    // dense conv dispatch ------------------------------------------------------------------
    void conv(const DConv& c, const float* x, int ldx, float* y, int ldy, Seg seg, int nseg, int maxlen,
              const ConvOpts& o = ConvOpts()) {
        if (maxlen <= 0 || nseg <= 0) return;
        if (!profOn) { conv_impl(c, x, ldx, y, ldy, seg, nseg, maxlen, o); return; }
        ProfRec r;
        r.cls = curCls; r.a = prof_event(); r.b = prof_event();
        r.flops = 2.0 * c.macs_row * (double)curRowsTotal;
        CUDA_CHECK(cudaEventRecord(r.a, stream));
        conv_impl(c, x, ldx, y, ldy, seg, nseg, maxlen, o);
        CUDA_CHECK(cudaEventRecord(r.b, stream));
        profRecs.push_back(r);
    }
    void conv_impl(const DConv& c, const float* x, int ldx, float* y, int ldy, Seg seg, int nseg, int maxlen,
                   const ConvOpts& o) {
        ConvP p;
        p.x = x; p.ldx = ldx; p.w = c.w; p.CoutW = c.CoutW; p.bias = c.b; p.y = y; p.ldy = ldy;
        p.y2 = o.y2; p.ldy2 = o.ldy2; p.res = o.res; p.ldr = o.ldr; p.gvec = o.gvec; p.ldg = o.ldg;
        p.seg = seg; p.Cin = c.Cin; p.Cout = c.Cout; p.k = c.k; p.dil = c.dil; p.padl = c.padl;
        p.in_act = o.in_act; p.in_slope = o.in_slope; p.epi = o.epi; p.div = o.div; p.split = o.split;
        p.y2_store = o.y2_store;
#ifdef STTS_WITH_TC
        if (tensor_mode >= 1 && o.allow_tc && tc_eligible(c.tc, p)) {
            Planes in;
            if (o.in_planes && o.in_planes->base) in = *o.in_planes;
            else {   // the producer was not a tensor-core conv: split fp32 rows into planes here
                in = scratch_planes(curRowsTotal, nseg, c.Cin);
                dim3 g(((size_t)(maxlen + 2 * TC_GAP) * (c.Cin / 8) + 255) / 256, nseg);
                split_planes_kernel<<<g, 256, 0, stream>>>(x, ldx, seg, c.Cin, o.in_act, o.in_slope, in);
                launch_check();
            }
            TcOut out;
            if (o.out_planes) out.yp = *o.out_planes;
            if (o.out2_planes) out.y2p = *o.out2_planes;
            out.out_act = o.out_act; out.out_slope = o.out_slope; out.write_f32 = o.write_f32;
            out.y_tt = o.y_tt; out.y2_tt = o.y2_tt; out.res_tt = o.res_tt; out.acc_tt = o.acc_tt; out.acc_src = o.acc_src;
            const int r = tc_conv_launch(c.tc, p, in, out, nseg, maxlen, stream, sms,
                                         // throughput mode covers the frame-level layers only: the text encoder and the duration predictor keep the
                                         // fp32-accurate MMAs, because ceil(exp(logw) * length_scale) must not move (SynthesizerTrn.cpp:376-378)
                                         (tensor_mode == 2 && curCls >= STTS_CLS_FLOW_IO) ? 1 : 0);
            if (r == -2) throw std::runtime_error("tile-transposed tensor with a row stride (planning bug)");
            if (r < 0) throw CudaError("cuTensorMapEncodeTiled failed for an activation plane");
            launches += r;
            cudaError_t e = cudaGetLastError();
            if (e != cudaSuccess) throw CudaError(std::string("tc conv launch failed: ") + cudaGetErrorString(e));
            return;
        }
        if (!o.write_f32 || o.in_planes || o.y_tt || o.y2_tt || o.res_tt || o.acc_src)
            throw std::runtime_error("planes-only / tile-transposed tensor routed to a non-tensor-core conv (planning bug)");
#endif
        const int halo = (c.k - 1) * c.dil;
        if (c.Cout <= 8 && o.epi != EPI_GATE && o.epi != EPI_RESSKIP) {
            dim3 g((maxlen + 127) / 128, nseg, 1);
            size_t sm = (size_t)c.k * c.Cin * 8 * sizeof(float);
            if (sm > 48 * 1024) throw Unsupported("narrow conv weight tile exceeds 48 KB");
            conv_narrow_kernel<8><<<g, 128, sm, stream>>>(p);
        } else if (c.Cout >= 48) {
            constexpr int BM = 64, BN = 64;
            dim3 g((maxlen + BM - 1) / BM, nseg, (c.Cout + BN - 1) / BN);
            size_t sm = ((size_t)16 * ((BM + halo + 4) & ~3) + 2 * 16 * BN) * sizeof(float);
            conv_tile_kernel<BM, BN><<<g, (BM / 4) * (BN / 8), sm, stream>>>(p);
        } else if (c.Cout >= 24) {
            constexpr int BM = 128, BN = 32;
            dim3 g((maxlen + BM - 1) / BM, nseg, (c.Cout + BN - 1) / BN);
            size_t sm = ((size_t)16 * ((BM + halo + 4) & ~3) + 2 * 16 * BN) * sizeof(float);
            conv_tile_kernel<BM, BN><<<g, (BM / 4) * (BN / 8), sm, stream>>>(p);
        } else {
            constexpr int BM = 256, BN = 16;
            dim3 g((maxlen + BM - 1) / BM, nseg, (c.Cout + BN - 1) / BN);
            size_t sm = ((size_t)16 * ((BM + halo + 4) & ~3) + 2 * 16 * BN) * sizeof(float);
            conv_tile_kernel<BM, BN><<<g, (BM / 4) * (BN / 8), sm, stream>>>(p);
        }
        launch_check();
    }
    void add_ln(const float* a, const float* b, const DLN& ln, float* y, int rows, int gelu = 0) {
        if (rows <= 0) return;
        add_ln_kernel<<<(rows + 3) / 4, 128, 0, stream>>>(a, b, ln.g, ln.b, y, rows, ln.C, gelu);
        launch_check();
    }

    // DDSConv::forward, src/modules/DDSConv.cpp:84-111.  x is updated in place; t1,t2 scratch [rows][C].
    void dds_forward(const DDds& d, float* x, float* t1, float* t2, Seg seg, int nseg, int maxlen, int rows) {
        for (int i = 0; i < d.n; ++i) {
            dim3 g(((size_t)maxlen * d.C + 255) / 256, nseg);
            dwconv_kernel<<<g, 256, 0, stream>>>(x, d.sw[i], d.sb[i], t1, seg, d.C, d.k, d.sdil[i], d.spad[i]);
            launch_check();
            add_ln(t1, nullptr, d.n1[i], t1, rows, 1);
            conv(d.c11[i], t1, d.C, t2, d.C, seg, nseg, maxlen);
            add_ln(t2, nullptr, d.n2[i], t2, rows, 1);
            add_kernel<<<((size_t)rows * d.C + 255) / 256, 256, 0, stream>>>(x, t2, x, (size_t)rows * d.C);
            launch_check();
        }
    }

    // Per-DEVICE one-time state (function attributes are per device/context: an engine on GPU 1 of the same process needs its
    // own call), SM count and the overflow flag word.
    int sms = 148;
    unsigned int* d_flags = nullptr;
    unsigned int* h_flags = nullptr;   // pinned
    int64_t fallbacks = 0;       // batches re-run on the fp32 FFMA tiles because an activation left the split-fp16 range
    void device_setup() {
        int n = 0;
        CUDA_CHECK(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, device));
        if (n > 0) sms = n;
        CUDA_CHECK(nb_device_setup());
        CUDA_CHECK(cudaFuncSetAttribute(ms_tail_kernel<512>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
        CUDA_CHECK(cudaFuncSetAttribute(ms_tail_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
        d_flags = dalloc<unsigned int>(4);
        CUDA_CHECK(cudaMemset(d_flags, 0, 16));
        CUDA_CHECK(cudaMallocHost((void**)&h_flags, 16));
        h_flags[0] = 0;
#ifdef STTS_WITH_TC
        CUDA_CHECK(tc_device_setup());
        CUDA_CHECK(rb_device_setup());
        CUDA_CHECK(pc_device_setup());
#endif
    }
#ifdef STTS_WITH_TC
    // Super-tile table of the fused ResBlock1-pair kernel for one segmentation (lens = host copy of the row counts) and
    // tile height ov: built on the device from the same offsets, size computed here.
    const int2* rb_tiles(const Seg& seg, const std::vector<int>& lens, int ov, int& ntiles) {
        ntiles = 0;
        for (int L : lens) ntiles += (L + ov - 1) / ov;
        int2* t = ws.get<int2>((size_t)std::max(ntiles, 1));
        rb_tiles_kernel<<<1, 256, 0, stream>>>(seg, (int)lens.size(), ov, t, ntiles);
        launch_check();
        return t;
    }
#endif
    void prof_begin(ProfRec& r, double flops) {
        r.cls = curCls; r.a = prof_event(); r.b = prof_event(); r.flops = flops;
        CUDA_CHECK(cudaEventRecord(r.a, stream));
    }
    void prof_end(ProfRec& r) {
        CUDA_CHECK(cudaEventRecord(r.b, stream));
        profRecs.push_back(r);
    }
    void build(const Model& M);
    void stage(int B_, const int32_t* ids, const int32_t* offs, const int32_t* sids, const float* ls);
    void run();
    void ensure_ws(size_t bytes);
};

// ---------------------------------------------------------------------------------------------
// model upload
// ---------------------------------------------------------------------------------------------
void stts_engine::build(const Model& M) {
    isMS = M.isMS; langType = M.langType; durPredType = M.durPredType; decType = M.decType;
    spkNum = M.spkNum; gin = M.gin; nnEnd = M.nnEnd;
    // --- text encoder (TextEncoder.cpp:20-48)
    const EncRec& E = M.enc;
    hidden = E.hidden; vocab = E.vocab; nEnc = E.nLayers;
    if (E.embDim != E.hidden) throw Unsupported("embedding width != hidden width");
    emb = upload(E.emb, (size_t)E.vocab * E.embDim);
    for (int i = 0; i < E.nLayers; ++i) {
        const MhaRec& m = E.mha[i];
        if (m.nHeads != 2) throw Unsupported("attention head count != 2 (the reference hard-codes 2, multi_head_attention.cpp:287-289)");
        if (m.winSize <= 0) throw Unsupported("attention without relative window (winSize == 0)");
        if (m.channels != hidden || m.outCh != hidden) throw Unsupported("attention width mismatch");
        nHeads = m.nHeads; kc = m.channels / m.nHeads; win = m.winSize; relRows = m.relRows;
        if (kc % 32 != 0 || kc > 128 || (kc != 96 && kc != 64 && kc != 32 && kc != 128))
            throw Unsupported("per-head width must be one of 32/64/96/128");
        if (relRows != 2 * win + 1 || m.relCols != kc || relRows > 16) throw Unsupported("relative embedding shape");
        for (const ConvRec* c : {&m.q, &m.k, &m.v, &m.o})
            if (c->k != 1 || c->inCh != hidden || c->outCh != hidden) throw Unsupported("attention projections must be 1x1");
        EncL L;
        // fused q|k|v projection: one GEMM with N = 3*hidden
        if (img.mode == 2) L.qkv = img_replay(1, hidden, 3 * hidden);
        else {
            DConv d;
            d.Cin = hidden; d.Cout = 3 * hidden; d.CoutW = d.Cout; d.k = 1; d.dil = 1; d.padl = 0;
            std::vector<float> w((size_t)hidden * d.CoutW), b(d.Cout, 0.f);
            const ConvRec* src[3] = {&m.q, &m.k, &m.v};
            for (int s = 0; s < 3; ++s)
                for (int o = 0; o < hidden; ++o) {
                    for (int c = 0; c < hidden; ++c) w[(size_t)c * d.CoutW + s * hidden + o] = src[s]->w[(size_t)o * hidden + c];
                    b[s * hidden + o] = src[s]->hasBias == 1 ? src[s]->b[o] : 0.f;
                }
            d.w = upload(w); d.b = upload(b);
            d.macs_row = (double)d.Cout * d.Cin;
#ifdef STTS_WITH_TC
            tc_prepare_weights(d.tc, w.data(), 1, d.Cin, d.Cout, d.CoutW, owned, tc_usteps);
#endif
            img_record(d);
            L.qkv = d;
        }
        L.o = make_conv(m.o);
        L.ek = upload(m.embRelK, (size_t)m.relRows * m.relCols);
        L.ev = upload(m.embRelV, (size_t)m.relRows * m.relCols);
        L.n1 = make_ln(E.norm1[i]);
        L.n2 = make_ln(E.norm2[i]);
        const FfnRec& f = E.ffn[i];
        // FFN::same_padding (ffn.cpp:47-62): pad_l = (k-1)/2, pad_r = k/2, on top of the record's own pad
        L.f1 = make_conv(f.c1, {}, {}, 1.f, (f.k - 1) / 2 + f.c1.pad);
        L.f2 = make_conv(f.c2, {}, {}, 1.f, (f.k - 1) / 2 + f.c2.pad);
        if (f.c1.k != f.k || f.c2.k != f.k || f.c1.pad != 0 || f.c2.pad != 0) throw Unsupported("FFN conv shape");
        enc.push_back(L);
    }
    {   // proj: m = the first half; logs = the second half, live only in batches that sample the prior (the reference multiplies
        // it by noiseScale == 0, SynthesizerTrn.cpp:357,383)
        inter = E.proj.outCh / 2;
        std::vector<int> om(inter);
        for (int i = 0; i < inter; ++i) om[i] = i;
        encProj = make_conv(E.proj, om);
        for (int i = 0; i < inter; ++i) om[i] = inter + i;
        encProjLogs = make_conv(E.proj, om);
    }
    // --- duration predictor
    if (durPredType == 1) {
        dp1 = make_conv(M.dp.conv_1); dp2 = make_conv(M.dp.conv_2); dpProj = make_conv(M.dp.proj);
        dpn1 = make_ln(M.dp.norm_1); dpn2 = make_ln(M.dp.norm_2);
        if (M.dp.hasCond) dpCond = make_conv(M.dp.cond);
    } else {
        const DurPredRec& D = M.dp;
        sdpNFlows = D.nFlows;
        sdpPre = make_conv(D.pre); sdpProj = make_conv(D.proj);
        if (D.hasCond) sdpCond = make_conv(D.cond);
        sdpConvs = make_dds(D.convs);
        eaM0 = D.ea.m[0]; eaLogs0 = D.ea.logs[0];
        for (int i = 0; i < D.nFlows; ++i) {
            DConvFlow cf;
            const ConvFlowRec& r = D.flows[i];
            if (r.pre.inCh != 1 || r.pre.k != 1) throw Unsupported("ConvFlow pre must be 1->C 1x1");
            if (r.proj.outCh != 29) throw Unsupported("ConvFlow proj must have 3*10-1 outputs (numBins_ = 10, ConvFlow.cpp:37)");
            cf.prew = upload(r.pre.w, r.pre.outCh);
            cf.preb = r.pre.hasBias == 1 ? upload(r.pre.b, r.pre.outCh) : nullptr;
            cf.dds = make_dds(r.dds);
            cf.proj = make_conv(r.proj);
            cf.fsqrt = std::sqrt((float)r.pre.outCh);
            sdpFlows.push_back(cf);
        }
    }
    // --- flow (ResidualCouplingBlock.cpp:29-39).  The channel flip before every layer
    // (ResidualCouplingBlock.cpp:66, nn_flip.cpp) is folded into the pre/post weights: at odd flip
    // parity logical channel c lives at physical channel C-1-c.
    tc_usteps = 8;       // frame-level layers from here on (conv_tc.cuh, TcWeights::usteps)
    flowN = M.flow.nFlows; wnLayers = M.flow.nLayers;
    const int half = inter / 2;
    for (int i = 0; i < flowN; ++i) {
        const CouplingRec& L = M.flow.layers[i];
        const int parity = (flowN - i) % 2;
        CoupL C;
        wnHidden = L.pre.outCh;
        if (L.pre.inCh != half || L.post.outCh != half || L.pre.k != 1 || L.post.k != 1)
            throw Unsupported("coupling layer pre/post shape");
        std::vector<int> cm(half), om(half);
        for (int q = 0; q < half; ++q) { cm[q] = parity ? half - 1 - q : q; om[q] = parity ? half - 1 - q : q; }
        C.pre = make_conv(L.pre, {}, cm);
        C.post = make_conv(L.post, om, {}, -1.f);  // x1 = x1 - m  ->  accumulate (-m)
        const int H = wnHidden;
        if ((int)L.wn.in_layers.size() != L.wn.nLayers) throw FormatError("WN layer count");
        for (int l = 0; l < L.wn.nLayers; ++l) {
            const ConvRec& in = L.wn.in_layers[l];
            if (in.outCh != 2 * H || in.inCh != H) throw Unsupported("WN in_layer shape");
            std::vector<int> gm(2 * H);  // interleave (tanh_j, sigmoid_j) so one thread owns a gate pair
            for (int j = 0; j < H; ++j) { gm[2 * j] = j; gm[2 * j + 1] = H + j; }
            C.in.push_back(make_conv(in, gm, {}, 1.f, -1, true, false, true));
            const ConvRec& rs = L.wn.res_skip[l];
            const bool last = l == L.wn.nLayers - 1;
            if (rs.inCh != H || rs.outCh != (last ? H : 2 * H) || rs.k != 1) throw Unsupported("WN res_skip shape");
            C.rs.push_back(make_conv(rs, {}, {}, 1.f, -1, true, false, true));
        }
        if (L.wn.hasCond) {
            const ConvRec& cd = L.wn.cond;
            if (cd.outCh != 2 * H * L.wn.nLayers || cd.k != 1) throw Unsupported("WN cond_layer shape");
            std::vector<int> gm(cd.outCh);
            for (int l = 0; l < L.wn.nLayers; ++l)
                for (int j = 0; j < H; ++j) {
                    gm[l * 2 * H + 2 * j] = l * 2 * H + j;
                    gm[l * 2 * H + 2 * j + 1] = l * 2 * H + H + j;
                }
            C.cond = make_conv(cd, gm);
            C.hasCond = true;
        }
        flow.push_back(C);
    }
    // --- decoder
    const GenRec& G = M.dec;
    convPre = make_conv(G.conv_pre);
    if (G.conv_pre.inCh != inter) throw Unsupported("decoder input width != flow width");
    if (G.hasCond) { decCond = make_conv(G.cond); decHasCond = true; }
    upRates = G.upRates;
    nRbK = (int)G.rbK.size();
    int ch = G.conv_pre.outCh;
    for (size_t i = 0; i < G.ups.size(); ++i) {
        if (G.ups[i].inCh != ch) throw Unsupported("upsample input width mismatch");
        ups.push_back(make_convT(G.ups[i]));
        ch = G.ups[i].outCh;
        stageC.push_back(ch);
    }
    for (size_t i = 0; i < G.rbs.size(); ++i) {
        RB rb;
        for (auto& c : G.rbs[i].convs1) rb.c1.push_back(make_conv(c, {}, {}, 1.f, -1, true, true));
        for (auto& c : G.rbs[i].convs2) rb.c2.push_back(make_conv(c, {}, {}, 1.f, -1, true, true));
        if (!rb.c1.empty() && rb.c1[0].Cin <= 8 && rb.c1.size() == rb.c2.size())
            for (size_t q = 0; q < rb.c1.size(); ++q) {          // (read back from the device: also valid when the convs came from the image)
                auto fetch = [&](const float* dptr, size_t n) {
                    std::vector<float> h(n);
                    if (dptr && n) CUDA_CHECK(cudaMemcpy(h.data(), dptr, n * 4, cudaMemcpyDeviceToHost));
                    return h;
                };
                const DConv &a = rb.c1[q], &b = rb.c2[q];
                rb.hw1.push_back(fetch(a.w, (size_t)a.k * a.Cin * a.CoutW)); rb.hb1.push_back(fetch(a.b, a.b ? a.Cout : 0));
                rb.hw2.push_back(fetch(b.w, (size_t)b.k * b.Cin * b.CoutW)); rb.hb2.push_back(fetch(b.b, b.b ? b.Cout : 0));
            }
        rbs.push_back(rb);
    }
    if (decType == 0) {
        convPost = make_conv(G.conv_post);
        if (G.conv_post.outCh != 1) throw Unsupported("conv_post must have one output channel");
    } else {
        subBands = decType == 2 ? 1 : G.subBands;
        if (G.nfft != 16 || G.hop != 4) throw Unsupported("iSTFT is hard-wired to (16,4,16) in the reference (Generator_MS.cpp:129)");
        if (decType != 2 && subBands != 4) throw Unsupported("sub-band count must be 4 (pqmf(4), Generator_MBB.cpp:108)");
        subPost = make_conv(G.subband_post);
        if (G.subband_post.outCh != subBands * 18) throw Unsupported("subband_conv_post width");
        if (decType == 1) {
            const ConvRec& r = G.ms_post;
            if (r.k != 63 || r.inCh != 4 || r.outCh != 1 || r.pad != 31) throw Unsupported("multistream_conv_post shape");
            msW = upload(r.w, 63 * 4);  // file order [o=1][k][c] == [63][4]
            msB = r.hasBias == 1 ? upload(r.b, 1) : nullptr;
        } else if (decType == 3) {
            // PQMF synthesis bank, pqmf.cpp:8-25,39-95 (float32 arithmetic like the reference)
            static const float h[63] = {
                8.36595339e-06f, 2.68017852e-05f, 5.05711124e-05f, 6.13482515e-05f, 2.75281598e-05f, -8.62839965e-05f,
                -2.99268467e-04f, -5.88389492e-04f, -8.67064627e-04f, -9.82905838e-04f, -7.47200209e-04f, 8.04087656e-19f,
                1.30001234e-03f, 2.98798828e-03f, 4.64603942e-03f, 5.63488600e-03f, 5.22586317e-03f, 2.82493436e-03f,
                -1.75650987e-03f, -8.06073440e-03f, -1.48622207e-02f, -2.02404650e-02f, -2.18780344e-02f, -1.75512321e-02f,
                -5.71474631e-03f, 1.39652689e-02f, 4.02848855e-02f, 7.05021626e-02f, 1.00706377e-01f, 1.26503321e-01f,
                1.43873012e-01f, 1.50000000e-01f, 1.43873012e-01f, 1.26503321e-01f, 1.00706377e-01f, 7.05021626e-02f,
                4.02848855e-02f, 1.39652689e-02f, -5.71474631e-03f, -1.75512321e-02f, -2.18780344e-02f, -2.02404650e-02f,
                -1.48622207e-02f, -8.06073440e-03f, -1.75650987e-03f, 2.82493436e-03f, 5.22586317e-03f, 5.63488600e-03f,
                4.64603942e-03f, 2.98798828e-03f, 1.30001234e-03f, 8.04087656e-19f, -7.47200209e-04f, -9.82905838e-04f,
                -8.67064627e-04f, -5.88389492e-04f, -2.99268467e-04f, -8.62839965e-05f, 2.75281598e-05f, 6.13482515e-05f,
                5.05711124e-05f, 2.68017852e-05f, 8.36595339e-06f};
            std::vector<float> w(63 * 4);
            for (int b = 0; b < 4; ++b)
                for (int n = 0; n < 63; ++n) {
                    const float tmp1 = ((float)n - (62.0f - 1.0f) / 2.0f) * (float)(M_PI / (2.0 * 4));
                    const float ph = (float)(std::pow(-1.0, b) * (M_PI / 4));
                    w[n * 4 + b] = h[n] * 2.0f * std::cos(tmp1 * (float)(2 * b + 1) - ph);
                }
            msW = upload(w);
        }
    }
    if (isMS == 1) emg = upload(M.emg, (size_t)spkNum * gin);
    CUDA_CHECK(cudaFuncSetAttribute(relattn_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    CUDA_CHECK(cudaFuncSetAttribute(relattn_kernel<96>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    CUDA_CHECK(cudaFuncSetAttribute(relattn_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    device_setup();
    // constant DFT tables
    float c16[16], s16[16];
    for (int i = 0; i < 16; ++i) { c16[i] = (float)std::cos(2.0 * M_PI * i / 16.0); s16[i] = (float)std::sin(2.0 * M_PI * i / 16.0); }
    CUDA_CHECK(cudaMemcpyToSymbol(c_cos16, c16, sizeof(c16)));
    CUDA_CHECK(cudaMemcpyToSymbol(c_sin16, s16, sizeof(s16)));
}

void stts_engine::ensure_ws(size_t bytes) {
    if (bytes <= ws.cap) return;
    CUDA_CHECK(cudaStreamSynchronize(stream));
    if (wsAlloc) CUDA_CHECK(cudaFree(wsAlloc));
    wsAlloc = nullptr;
    size_t want = bytes + bytes / 4;
    CUDA_CHECK(cudaMalloc(&wsAlloc, want));
    ws.base = (char*)wsAlloc; ws.cap = want; ws.off = 0;
}

// ---------------------------------------------------------------------------------------------
// H2D staging of one batch
// ---------------------------------------------------------------------------------------------
void stts_engine::stage(int B_, const int32_t* ids, const int32_t* offs, const int32_t* sids, const float* ls) {
    if (B_ <= 0 || !ids || !offs) throw ArgError("empty batch or null ids/offsets");
    // a new batch invalidates the results of the previous run (stts_batch_fetch / stts_debug_fetch then report STTS_E_ARG)
    St = 0; d_pcm = nullptr; dbg = Dbg(); h_soff.clear(); runValid = false;
    if (ls)
        for (int u = 0; u < B_; ++u)
            if (!(ls[u] > 0.f) || !std::isfinite(ls[u]) || ls[u] > 1000.f) throw ArgError("length_scale must be finite, positive and <= 1000");
    for (float w : forced)
        if (!(w >= 0.f) || w > 65536.f) throw ArgError("forced durations must be finite, non-negative and <= 65536 frames");
    if (!smpNs.empty() && (int)smpNs.size() != B_)
        throw ArgError("sampling was set for " + std::to_string(smpNs.size()) + " utterances, the batch has " + std::to_string(B_));
    if (offs[0] != 0) throw ArgError("id_offsets[0] must be 0");
    int mt = 0;
    for (int u = 0; u < B_; ++u) {
        const int n = offs[u + 1] - offs[u];
        // get_relative_embeddings never slices (multi_head_attention.cpp:140-150): the reference breaks for T < win+1
        if (n < win + 1) throw ArgError("utterance with fewer than " + std::to_string(win + 1) + " phoneme ids");
        mt = std::max(mt, n);
    }
    const int T = offs[B_];
    for (int i = 0; i < T; ++i)
        if (ids[i] < 0 || ids[i] >= vocab) throw ArgError("phoneme id out of range at position " + std::to_string(i));
    if ((size_t)T > stageCapTok || (size_t)B_ > stageCapB) {
        CUDA_CHECK(cudaStreamSynchronize(stream));
        auto re = [&](auto*& p, size_t n) {      // the pointer is nulled before the new allocation: a failed cudaMalloc leaves no dangling pointer
            if (p) { void* old = p; p = nullptr; CUDA_CHECK(cudaFree(old)); }
            void* q = nullptr;
            CUDA_CHECK(cudaMalloc(&q, n));
            p = (std::remove_reference_t<decltype(p)>)q;
        };
        const size_t capTok = std::max<size_t>(stageCapTok, (size_t)T * 2), capB = std::max<size_t>(stageCapB, (size_t)B_ * 2);
        stageCapTok = 0; stageCapB = 0;          // raised only after every allocation succeeded
        re(d_ids, capTok * 4); re(d_forced, capTok * 4);
        re(d_toff, (capB + 1) * 4); re(d_foff, (capB + 1) * 4); re(d_nfr, capB * 4);
        re(d_sids, capB * 4); re(d_ls, capB * 4); re(d_bseg, 2 * 4);
        re(d_ns, capB * 4); re(d_nsw, capB * 4); re(d_seed, capB * 8);
        stageCapTok = capTok; stageCapB = capB;
    }
    B = B_; Tt = T; maxT = mt;
    h_toff.assign(offs, offs + B + 1);
    std::vector<int> hs(B, 0);
    std::vector<float> hl(B, 1.0f);
    if (sids) for (int u = 0; u < B; ++u) hs[u] = sids[u];
    if (ls) for (int u = 0; u < B; ++u) hl[u] = ls[u];
    const int bseg[2] = {0, B};
    CUDA_CHECK(cudaMemcpyAsync(d_ids, ids, (size_t)T * 4, cudaMemcpyHostToDevice, stream));
    CUDA_CHECK(cudaMemcpyAsync(d_toff, offs, (size_t)(B + 1) * 4, cudaMemcpyHostToDevice, stream));
    CUDA_CHECK(cudaMemcpyAsync(d_sids, hs.data(), (size_t)B * 4, cudaMemcpyHostToDevice, stream));
    CUDA_CHECK(cudaMemcpyAsync(d_ls, hl.data(), (size_t)B * 4, cudaMemcpyHostToDevice, stream));
    CUDA_CHECK(cudaMemcpyAsync(d_bseg, bseg, 8, cudaMemcpyHostToDevice, stream));
    if (!forced.empty()) {
        if ((int64_t)forced.size() != T) throw ArgError("forced durations length != total ids of the batch");
        CUDA_CHECK(cudaMemcpyAsync(d_forced, forced.data(), (size_t)T * 4, cudaMemcpyHostToDevice, stream));
    }
    samplePrior = std::any_of(smpNs.begin(), smpNs.end(), [](float v) { return v != 0.f; });
    sampleSdp = durPredType == 0 && std::any_of(smpNsw.begin(), smpNsw.end(), [](float v) { return v != 0.f; });
    if (samplePrior || sampleSdp) {
        CUDA_CHECK(cudaMemcpyAsync(d_ns, smpNs.data(), (size_t)B * 4, cudaMemcpyHostToDevice, stream));
        CUDA_CHECK(cudaMemcpyAsync(d_nsw, smpNsw.data(), (size_t)B * 4, cudaMemcpyHostToDevice, stream));
        CUDA_CHECK(cudaMemcpyAsync(d_seed, smpSeed.data(), (size_t)B * 8, cudaMemcpyHostToDevice, stream));
    }
    CUDA_CHECK(cudaStreamSynchronize(stream));  // host vectors above go out of scope
}

// ---------------------------------------------------------------------------------------------
// forward pass of the staged batch
// ---------------------------------------------------------------------------------------------
void stts_engine::run() {
    if (B <= 0) throw ArgError("no batch staged");
    runValid = false;
    const int H = hidden;
    const Seg tseg{d_toff, 1, 0};
    const Seg bseg{d_bseg, 1, 0};
    CUDA_CHECK(cudaEventRecord(ev[0], stream));
    nvtxRangePushA(injectZ ? "stts:chunk" : "stts:text_encoder");
    struct PopAll { int n = 1; ~PopAll() { while (n-- > 0) nvtxRangePop(); } } nvtx_guard;   // exception-safe: exactly one range open at any time
    if (tensor_mode >= 1) CUDA_CHECK(cudaMemsetAsync(d_flags, 0, 4, stream));

    // ---- token-level workspace ---------------------------------------------------------------
    size_t ffnW = 0, dpW = 0;
    for (auto& L : enc) ffnW = std::max<size_t>(ffnW, L.f1.Cout);
    dpW = durPredType == 1 ? (size_t)std::max(dp1.Cout, dp2.Cout) : (size_t)H;
    size_t condFloats = 64;      // per-utterance conditioning vectors: speaker embedding + DP / decoder / per-flow WN cond outputs (+ 256 B padding each)
    if (isMS) {
        condFloats += (size_t)gin + 64 + (size_t)H + 64 + (size_t)convPre.Cout + 64;
        for (auto& L : flow) if (L.hasCond) condFloats += (size_t)L.cond.Cout + 64;
    }
    size_t tokFloats = (size_t)Tt * (H * 5 + 3 * H + 2 * ffnW + 2 * inter + 3 * dpW + 64 + 8) + (size_t)B * (condFloats + 2 * 64 * ffnW) + 512 * ffnW + 4096;
    ensure_ws(tokFloats * 4 + (1 << 20));
    ws.reset();
    float* x = ws.get<float>((size_t)Tt * H);
    float* qkv = ws.get<float>((size_t)Tt * 3 * H);
    float* att = ws.get<float>((size_t)Tt * H);
    float* y = ws.get<float>((size_t)Tt * H);
    float* x1 = ws.get<float>((size_t)Tt * H);
    float* fh = ws.get<float>((size_t)Tt * ffnW);
#ifdef STTS_WITH_TC
    Planes encFhP;
    if (tensor_mode >= 1) encFhP = arena_planes(Tt, B, (int)ffnW);
#endif
    float* mbuf = ws.get<float>((size_t)Tt * inter);
    float* logsbuf = samplePrior ? ws.get<float>((size_t)Tt * inter) : nullptr;
    float* logw = ws.get<float>((size_t)Tt);
    float* wceil = ws.get<float>((size_t)Tt);
    int* tokFirst = ws.get<int>((size_t)Tt);
    float* d1 = ws.get<float>((size_t)Tt * dpW);
    float* d2 = ws.get<float>((size_t)Tt * dpW);
    float* d3 = ws.get<float>((size_t)Tt * dpW);
    float* h29 = ws.get<float>((size_t)Tt * 32);
    float* sa = ws.get<float>((size_t)Tt);
    float* sb = ws.get<float>((size_t)Tt);
    float* G = isMS ? ws.get<float>((size_t)B * gin) : nullptr;
    float* gDp = isMS ? ws.get<float>((size_t)B * H) : nullptr;
    float* gDec = (isMS && decHasCond) ? ws.get<float>((size_t)B * convPre.Cout) : nullptr;
    std::vector<float*> gWn(flowN, nullptr);
    if (isMS)
        for (int i = 0; i < flowN; ++i)
            if (flow[i].hasCond) gWn[i] = ws.get<float>((size_t)B * flow[i].cond.Cout);
    const size_t tokEnd = ws.off;

    // ---- speaker conditioning vectors (SynthesizerTrn.cpp:363-372; cond convs of DP / WN / decoder)
    curCls = STTS_CLS_OTHER; curRowsTotal = B;
    if (isMS) {
        spk_gather_kernel<<<(B * gin + 255) / 256, 256, 0, stream>>>(emg, d_sids, G, B, gin, spkNum);
        launch_check();
        ConvOpts o; o.allow_tc = false;
        if (durPredType == 1 && dpCond.w) conv(dpCond, G, gin, gDp, dpCond.Cout, bseg, 1, B, o);
        if (durPredType == 0 && sdpCond.w) conv(sdpCond, G, gin, gDp, sdpCond.Cout, bseg, 1, B, o);
        if (gDec) conv(decCond, G, gin, gDec, decCond.Cout, bseg, 1, B, o);
        for (int i = 0; i < flowN; ++i)
            if (gWn[i]) conv(flow[i].cond, G, gin, gWn[i], flow[i].cond.Cout, bseg, 1, B, o);
    }

    if (!injectZ) {
    // ---- text encoder (TextEncoder.cpp:50-74, attention_encoder.cpp:78-94) ---------------------
    curCls = STTS_CLS_ENC; curRowsTotal = Tt;
    embed_kernel<<<((size_t)Tt * H + 255) / 256, 256, 0, stream>>>(d_ids, emb, x, Tt, H, vocab, std::sqrt((float)H));
    launch_check();
    for (int i = 0; i < nEnc; ++i) {
        EncL& L = enc[i];
        conv(L.qkv, x, H, qkv, 3 * H, tseg, B, maxT);
        {
            dim3 g((maxT + RA_QT - 1) / RA_QT, nHeads, B);
            size_t sm = ((size_t)RA_QT * kc + 2 * 32 * (kc + 4) + 2 * relRows * kc + RA_QT * 16) * sizeof(float);
            if (kc == 96) relattn_kernel<96><<<g, RA_THREADS, sm, stream>>>(qkv, att, L.ek, L.ev, tseg, H, win, relRows);
            else if (kc == 64) relattn_kernel<64><<<g, RA_THREADS, sm, stream>>>(qkv, att, L.ek, L.ev, tseg, H, win, relRows);
            else if (kc == 32) relattn_kernel<32><<<g, RA_THREADS, sm, stream>>>(qkv, att, L.ek, L.ev, tseg, H, win, relRows);
            else relattn_kernel<128><<<g, RA_THREADS, sm, stream>>>(qkv, att, L.ek, L.ev, tseg, H, win, relRows);
            launch_check();
        }
        conv(L.o, att, H, y, H, tseg, B, maxT);
        add_ln(x, y, L.n1, x1, Tt);
        ConvOpts r; r.epi = EPI_RELU;
        ConvOpts r2;
#ifdef STTS_WITH_TC
        Planes fhP;
        if (tc_layer(L.f1) && tc_layer(L.f2)) {   // relu(conv1) goes to conv2 as split-fp16 planes only
            fhP = encFhP;
            r.out_planes = &fhP; r.write_f32 = false; r2.in_planes = &fhP;
        }
#endif
        conv(L.f1, x1, H, fh, L.f1.Cout, tseg, B, maxT, r);
        conv(L.f2, fh, L.f1.Cout, y, H, tseg, B, maxT, r2);
        add_ln(x1, y, L.n2, x, Tt);
    }
    conv(encProj, x, H, mbuf, inter, tseg, B, maxT);
    if (samplePrior) conv(encProjLogs, x, H, logsbuf, inter, tseg, B, maxT);
    CUDA_CHECK(cudaEventRecord(ev[1], stream));
    nvtxRangePop(); nvtxRangePushA("stts:duration_predictor");

    // ---- duration predictor ------------------------------------------------------------------
    curCls = STTS_CLS_DP;
    if (durPredType == 1) {
        // FixDurationPredictor::forward, src/models/FixDurationPredictor.cpp:75-96
        const float* xin = x;
        if (isMS && dpCond.w) {  // XX = XX.rowwise() + gg.row(0)
            dim3 g(((size_t)maxT * H + 255) / 256, B);
            add_rowvec_kernel<<<g, 256, 0, stream>>>(x, gDp, dpCond.Cout, d3, tseg, H);
            launch_check();
            xin = d3;
        }
        ConvOpts r; r.epi = EPI_RELU;
        conv(dp1, xin, H, d1, dp1.Cout, tseg, B, maxT, r);
        add_ln(d1, nullptr, dpn1, d1, Tt);
        conv(dp2, d1, dp1.Cout, d2, dp2.Cout, tseg, B, maxT, r);
        add_ln(d2, nullptr, dpn2, d2, Tt);
        conv(dpProj, d2, dp2.Cout, logw, 1, tseg, B, maxT);
    } else {
        // StochasticDurationPredictor::forward, src/models/StochasticDurationPredictor.cpp:117-149 (noise == 0)
        ConvOpts o;
        if (isMS && sdpCond.w) { o.gvec = gDp; o.ldg = sdpCond.Cout; }
        conv(sdpPre, x, H, d1, H, tseg, B, maxT, o);           // pre (+ cond(g))
        dds_forward(sdpConvs, d1, d2, d3, tseg, B, maxT, Tt);  // convs
        conv(sdpProj, d1, H, d2, H, tseg, B, maxT);            // XX = proj(...)  -> d2
        float* XX = d2;
        if (sampleSdp) {
            sdp_noise_kernel<<<dim3((maxT + 127) / 128, B), 128, 0, stream>>>(sa, sb, d_toff, d_nsw, d_seed);
            launch_check();
        } else {
            CUDA_CHECK(cudaMemsetAsync(sa, 0, (size_t)Tt * 4, stream));
            CUDA_CHECK(cudaMemsetAsync(sb, 0, (size_t)Tt * 4, stream));
        }
        float *a = sa, *b = sb;  // (row0, row1) of flapZ_T
        for (int i = sdpNFlows - 1; i > 0; --i) {
            DConvFlow& cf = sdpFlows[i];
            const int C = cf.dds.C;
            expand1_kernel<<<((size_t)Tt * C + 255) / 256, 256, 0, stream>>>(a, cf.prew, cf.preb, d1, Tt, C);
            launch_check();
            add_kernel<<<((size_t)Tt * C + 255) / 256, 256, 0, stream>>>(d1, XX, d1, (size_t)Tt * C);  // DDSConv.cpp:90-93
            launch_check();
            dds_forward(cf.dds, d1, d3, fh, tseg, B, maxT, Tt);
            conv(cf.proj, d1, C, h29, 32, tseg, B, maxT);
            // (x0, x1) -> flip -> (spline(x1|x0), x0): new a = spline(b), new b = a
            rq_spline_inv_kernel<<<(Tt + 127) / 128, 128, 0, stream>>>(h29, 32, b, b, Tt, cf.fsqrt);
            launch_check();
            std::swap(a, b);
        }
        ea_kernel<<<(Tt + 255) / 256, 256, 0, stream>>>(a, logw, Tt, eaM0, eaLogs0);
        launch_check();
    }
    durations_kernel<<<B, 256, 0, stream>>>(logw, 1, forced.empty() ? nullptr : d_forced, d_ls, d_toff, wceil, tokFirst, d_nfr);
    launch_check();
    if ((size_t)B + 1 > hostIntsCap) {
        if (hostInts) CUDA_CHECK(cudaFreeHost(hostInts));
        hostIntsCap = (size_t)B * 2 + 16;
        CUDA_CHECK(cudaMallocHost((void**)&hostInts, hostIntsCap * 4));
    }
    CUDA_CHECK(cudaMemcpyAsync(hostInts, d_nfr, (size_t)B * 4, cudaMemcpyDeviceToHost, stream));
    CUDA_CHECK(cudaStreamSynchronize(stream));  // frame counts size every grid below (SynthesizerTrn.cpp:376-378)
    }   // !injectZ
    h_foff.assign(B + 1, 0);
    maxF = 0;
    if (injectZ) {
        if (B != 1 || injectF <= 0) throw ArgError("chunk injection needs a single staged utterance");
        h_foff[1] = injectF; maxF = injectF;
    } else
    for (int u = 0; u < B; ++u) {
        h_foff[u + 1] = h_foff[u] + hostInts[u];
        maxF = std::max(maxF, hostInts[u]);
    }
    Ft = h_foff[B];
    if (Ft <= 0 || (int64_t)Ft > (int64_t)16 << 20) throw ArgError("implausible frame count (length_scale / forced durations too large?)");
    CUDA_CHECK(cudaMemcpyAsync(d_foff, h_foff.data(), (size_t)(B + 1) * 4, cudaMemcpyHostToDevice, stream));
    CUDA_CHECK(cudaEventRecord(ev[2], stream));
    nvtxRangePop(); nvtxRangePushA("stts:length_regulator");

    // ---- frame-level workspace -----------------------------------------------------------------
    int R = 1;
    for (int r : upRates) R *= r;
    const int tailMul = decType == 0 ? 1 : (decType == 2 ? 4 : 16);
    St = (int64_t)Ft * R * tailMul;
    size_t need = tokEnd + 4096 + (size_t)(1 << 20);   // (+ super-tile tables of the fused ResBlock1 pairs)
    const int WH = wnHidden;
    need += ((size_t)Ft * (inter * 2 + WH * 3)) * 4 + 8 * 256;
    need += 3 * (planes_bytes(Ft, B, WH) + 256) + 4096;   // split-fp16 planes of h / acts / skip
    {
        size_t rows = Ft;
        need += rows * convPre.Cout * 4 + 256;
        int rr = 1;
        for (size_t i = 0; i < ups.size(); ++i) {
            rr *= upRates[i];
            need += ((size_t)Ft * rr * stageC[i] * 4 + 256) * 5;                                  // xx / t1 / xa / accb / accT
            need += 6 * (planes_bytes((int64_t)Ft * rr, B, stageC[i]) + 256);   // planes xx / t1 / xa, or xx / 2 ping-pong / 3 branch outputs (fused pairs)
        }
        if (decType != 0) {
            const size_t fr = (size_t)Ft * R + B;
            need += fr * (stageC.back() + subBands * 18 + subBands * 16) * 4 + (size_t)Ft * R * 4 * subBands * 4 + 2048;
        }
        need += (size_t)St * 4 + (size_t)St * 2 + 1024;
    }
    if (need > ws.cap) {
        // growing would invalidate the token-level buffers that are still live: re-plan conservatively
        // by allocating a separate, larger arena and copying the live token-level region.
        CUDA_CHECK(cudaStreamSynchronize(stream));
        void* nb = nullptr;
        size_t want = need + need / 4;
        CUDA_CHECK(cudaMalloc(&nb, want));
        CUDA_CHECK(cudaMemcpy(nb, ws.base, tokEnd, cudaMemcpyDeviceToDevice));
        const ptrdiff_t delta = (char*)nb - ws.base;
        auto mv = [&](auto*& p) { if (p) p = (std::remove_reference_t<decltype(p)>)((char*)p + delta); };
        mv(x); mv(mbuf); mv(logsbuf); mv(logw); mv(wceil); mv(tokFirst); mv(G); mv(gDp); mv(gDec);
        for (auto& g : gWn) mv(g);
        CUDA_CHECK(cudaFree(wsAlloc));
        wsAlloc = nb; ws.base = (char*)nb; ws.cap = want;
    }
    ws.off = tokEnd;
    const Seg fseg{d_foff, 1, 0};
    float* z = ws.get<float>((size_t)Ft * inter);
    float* zp_dbg = debug ? ws.get<float>((size_t)Ft * inter) : nullptr;
    float* hbuf = ws.get<float>((size_t)Ft * WH);
    float* acts = ws.get<float>((size_t)Ft * WH);
    float* skip = ws.get<float>((size_t)Ft * WH);
#ifdef STTS_WITH_TC
    Planes hP, actsP, skipP;
    bool flowTc = tensor_mode >= 1 && flowN > 0;
    for (auto& L : flow) {
        flowTc = flowTc && tc_layer(L.pre) && tc_layer(L.post);
        for (auto& c : L.in) flowTc = flowTc && tc_layer(c);
        for (auto& c : L.rs) flowTc = flowTc && tc_layer(c);
    }
    if (flowTc) { hP = arena_planes(Ft, B, WH); actsP = arena_planes(Ft, B, WH); skipP = arena_planes(Ft, B, WH); }
    // WaveNet layers on pc_fused.cuh (activation tile resident per row tile, weights streamed): h and skip live as planes only.
    // STTS_PC_FUSED bit 0: res_skip, bit 1: in_layer (default 3: both).  Measured per launch (1xB200, 64 x 640 frames, accurate
    // mode): res_skip 107 us (conv_tc) -> 45 us, in_layer 142 us (conv_tc column-split tiles) -> 115 us; throughput mode 73 us.
    static const int env_pc = getenv("STTS_PC_FUSED") ? atoi(getenv("STTS_PC_FUSED")) : -1;
    const int pc_bits = env_pc >= 0 ? env_pc : 3;
    bool flowPc = flowTc && pc_bits != 0;
    for (auto& L : flow) {
        for (auto& c : L.in) flowPc = flowPc && pc_eligible(c.pc, PC_EPI_GATE) && c.Cout == 2 * WH && c.Cin == WH;
        for (auto& c : L.rs) flowPc = flowPc && pc_eligible(c.pc, PC_EPI_RS) && c.Cin == WH;
    }
    const int2* ftiles = nullptr; int nftiles = 0;
    if (flowPc) {
        std::vector<int> lens(B);
        for (int u = 0; u < B; ++u) lens[u] = h_foff[u + 1] - h_foff[u];
        ftiles = rb_tiles(Seg{d_foff, 1, 0}, lens, 128, nftiles);
    }
#endif

    // ---- length regulator (expandM, SynthesizerTrn.cpp:304-321, :380-383) -----------------------
    if (injectZ) CUDA_CHECK(cudaMemcpyAsync(z, injectZ, (size_t)Ft * inter * 4, cudaMemcpyDeviceToDevice, stream));
    else {
        dim3 g((maxF + 3) / 4, B);
        if (samplePrior)
            regulate_noise_kernel<<<g, 128, 0, stream>>>(mbuf, logsbuf, inter, tokFirst, wceil, d_toff, d_foff, z, inter, d_ns, d_seed);
        else
            regulate_kernel<<<g, 128, 0, stream>>>(mbuf, inter, tokFirst, wceil, d_toff, d_foff, z, inter);
        launch_check();
        if (debug) CUDA_CHECK(cudaMemcpyAsync(zp_dbg, z, (size_t)Ft * inter * 4, cudaMemcpyDeviceToDevice, stream));
    }
    CUDA_CHECK(cudaEventRecord(ev[3], stream));
    nvtxRangePop(); nvtxRangePushA("stts:flow");
    if (stopAfterRegulate) {      // keep z_p for the chunked flow + decoder passes
        const size_t nb = (size_t)Ft * inter * 4;
        if (nb > streamZCap) {
            if (streamZ) { float* old = streamZ; streamZ = nullptr; CUDA_CHECK(cudaFree(old)); }
            CUDA_CHECK(cudaMalloc((void**)&streamZ, nb + nb / 4));
            streamZCap = nb + nb / 4;
        }
        CUDA_CHECK(cudaMemcpyAsync(streamZ, z, nb, cudaMemcpyDeviceToDevice, stream));
        CUDA_CHECK(cudaStreamSynchronize(stream));
        streamF = Ft;
        return;
    }

    // ---- flow: ResidualCouplingBlock::forward (reverse), ResidualCouplingBlock.cpp:59-71 --------
    const int half = inter / 2;
    for (int i = flowN - 1; i >= 0; --i) {
        CoupL& L = flow[i];
        const int parity = (flowN - i) % 2;
        const float* x0 = z + (parity ? half : 0);
        float* x1p = z + (parity ? 0 : half);
        curRowsTotal = Ft; curCls = STTS_CLS_FLOW_IO;
        {
            ConvOpts po;
#ifdef STTS_WITH_TC
            if (flowTc) { po.out_planes = &hP; po.y_tt = true; }   // h feeds the k5 in-layer as planes; its fp32 copy is
                                                                   // only ever touched by the res_skip epilogues
            if (flowPc) { po.y_tt = false; po.write_f32 = false; } // ... and not at all on the staged-epilogue path
#endif
            conv(L.pre, x0, inter, hbuf, WH, fseg, B, maxF, po);                 // h = pre(x0)
        }
        const int nl = (int)L.in.size();
        for (int l = 0; l < nl; ++l) {                                          // WN::forward, WN.cpp:100-149
            ConvOpts g; g.epi = EPI_GATE;
            if (L.hasCond) { g.gvec = gWn[i] + (size_t)l * 2 * WH; g.ldg = L.cond.Cout; }
            curCls = STTS_CLS_WN_IN;
            ConvOpts r; r.epi = EPI_RESSKIP; r.y2 = skip; r.ldy2 = WH; r.y2_store = (l == 0);
            r.split = (l < nl - 1) ? WH : 0;
#ifdef STTS_WITH_TC
            if (flowTc) {
                g.in_planes = &hP; g.out_planes = &actsP; g.write_f32 = false;   // acts only ever feed res_skip
                r.in_planes = &actsP;
                r.y_tt = true; r.y2_tt = true;           // h / skip fp32: tile-transposed (coalesced read-modify-write)
                if (l < nl - 1) r.out_planes = &hP;      // refreshed h for the next in-layer
                else r.out2_planes = &skipP;             // finished skip sum feeds `post`
            }
#endif
#ifdef STTS_WITH_TC
            if (flowPc) {
                const int pmode = tensor_mode == 2 ? 1 : 0;
                ProfRec pr;
                int rc;
                if (pc_bits & 2) {
                    if (profOn) prof_begin(pr, 2.0 * L.in[l].macs_row * (double)curRowsTotal);
                    rc = pc_launch(PC_EPI_GATE, L.in[l].pc, hP, actsP, actsP, 0, 0, 0, g.gvec, g.ldg, fseg, ftiles, nftiles, pmode, sms, d_flags, stream);
                    if (rc < 0) throw CudaError("WN in_layer launch failed (" + std::to_string(rc) + ")");
                    launch_check();
                    if (profOn) prof_end(pr);
                } else conv(L.in[l], hbuf, WH, acts, WH, fseg, B, maxF, g);      // conv_tc: hP planes -> gate -> actsP planes
                curCls = STTS_CLS_WN_RS;
                if (!(pc_bits & 1)) throw std::runtime_error("STTS_PC_FUSED: the in_layer alone cannot run on the staged-epilogue path");
                if (profOn) prof_begin(pr, 2.0 * L.rs[l].macs_row * (double)curRowsTotal);
                rc = pc_launch(PC_EPI_RS, L.rs[l].pc, actsP, hP, skipP, (l < nl - 1) ? WH : 0, 1, l > 0 ? 1 : 0, nullptr, 0, fseg, ftiles, nftiles, pmode, sms,
                               d_flags, stream);
                if (rc < 0) throw CudaError("WN res_skip launch failed (" + std::to_string(rc) + ")");
                launch_check();
                if (profOn) prof_end(pr);
                continue;
            }
#endif
            conv(L.in[l], hbuf, WH, acts, WH, fseg, B, maxF, g);
            curCls = STTS_CLS_WN_RS;
            conv(L.rs[l], acts, WH, hbuf, WH, fseg, B, maxF, r);
        }
        ConvOpts a; a.epi = EPI_ACCUM;
        curCls = STTS_CLS_FLOW_IO;
#ifdef STTS_WITH_TC
        if (flowTc) a.in_planes = &skipP;
#endif
        conv(L.post, skip, WH, x1p, inter, fseg, B, maxF, a);                   // x1 = x1 - post(h)
    }
    if (flowN % 2 == 1) {
        chan_reverse_kernel<<<((size_t)Ft * (inter / 2) + 255) / 256, 256, 0, stream>>>(z, (size_t)Ft, inter);
        launch_check();
    }
    CUDA_CHECK(cudaEventRecord(ev[4], stream));
    nvtxRangePop(); nvtxRangePushA("stts:decoder");

    // ---- decoder --------------------------------------------------------------------------------
    float* cur = ws.get<float>((size_t)Ft * convPre.Cout);
    {
        ConvOpts o;
        if (gDec) { o.gvec = gDec; o.ldg = decCond.Cout; }
        curCls = STTS_CLS_DEC_PRE; curRowsTotal = Ft;
        conv(convPre, z, inter, cur, convPre.Cout, fseg, B, maxF, o);            // conv_pre (+ cond(g))
    }
    int rate = 1, curC = convPre.Cout;
    for (size_t s = 0; s < ups.size(); ++s) {
        const int C = stageC[s];
        const int rate_in = rate;
        rate *= upRates[s];
        const size_t rows = (size_t)Ft * rate;
        float* xx = ws.get<float>(rows * C);
        float* accb = ws.get<float>(rows * C);
        {   // leaky(0.1) + ConvTranspose1d (phase-expanded): Generator_MS.cpp:172-175
            ConvOpts o; o.in_act = ACT_LEAKY; o.in_slope = 0.1f;
            curCls = STTS_CLS_DEC_UP; curRowsTotal = (int64_t)Ft * rate_in;
            conv(ups[s], cur, curC, xx, upRates[s] * C, Seg{d_foff, rate_in, 0}, B, maxF * rate_in, o);
        }
        const Seg sseg{d_foff, rate, 0};
        curCls = STTS_CLS_DEC_RB; curRowsTotal = (int64_t)Ft * rate;
        const int ml = maxF * rate;
        {   // narrow stages (4 / 8 channels): fused ResBlock1 pairs on the CUDA cores (nb_fused.cuh), fp32, any tensor mode
            static const int env_nb = getenv("STTS_NB_FUSED") ? atoi(getenv("STTS_NB_FUSED")) : 1;
            bool nbOk = env_nb && (C == 4 || C == 8) && nRbK >= 1;
            for (int j = 0; j < nRbK && nbOk; ++j) {
                const RB& rb = rbs[s * nRbK + j];
                nbOk = rb.c1.size() == rb.c2.size() && !rb.c1.empty() && rb.hw1.size() == rb.c1.size();
                for (size_t q = 0; q < rb.c1.size() && nbOk; ++q)
                    nbOk = rb.c1[q].Cin == C && rb.c1[q].Cout == C && rb.c2[q].Cin == C && rb.c2[q].Cout == C && rb.c1[q].CoutW == rb.c2[q].CoutW &&
                           nb_supported(C, rb.c1[q].k, rb.c1[q].dil, rb.c1[q].padl, rb.c2[q].k, rb.c2[q].dil, rb.c2[q].padl);
            }
            if (nbOk) {
                float* pp[2] = {ws.get<float>(rows * C), ws.get<float>(rows * C)};
                for (int j = 0; j < nRbK; ++j) {
                    const RB& rb = rbs[s * nRbK + j];
                    const int nb = (int)rb.c1.size();
                    const float* in = xx;
                    for (int q = 0; q < nb; ++q) {
                        const bool last = q == nb - 1;
                        NbP np;
                        np.x = in; np.y = last ? accb : pp[q & 1]; np.acc = accb; np.seg = sseg; np.d1 = rb.c1[q].dil; np.tr = 0;
                        np.out_mode = !last || j == 0 ? NB_STORE : (j < nRbK - 1 ? NB_ACCUM : NB_ACCUM_DIV);
                        if (last && nRbK == 1) np.out_mode = NB_STORE;
                        np.div = (float)nRbK;
                        ProfRec pr;
                        if (profOn) prof_begin(pr, 2.0 * (rb.c1[q].macs_row + rb.c2[q].macs_row) * (double)curRowsTotal);
                        if (nb_pair_launch(C, rb.c1[q].k, np, rb.hw1[q].data(), rb.hb1[q].empty() ? nullptr : rb.hb1[q].data(), rb.hw2[q].data(),
                                           rb.hb2[q].empty() ? nullptr : rb.hb2[q].data(), rb.c1[q].CoutW, B, ml, stream) < 0)
                            throw std::runtime_error("narrow fused pair: unsupported shape (planning bug)");
                        launch_check();
                        if (profOn) prof_end(pr);
                        in = np.y;
                    }
                }
                cur = accb; curC = C;
                continue;
            }
        }
#ifdef STTS_WITH_TC
        Planes xxP, t1P, xaP;
        bool rbTc = tensor_mode >= 1;
        for (int j = 0; j < nRbK; ++j) {
            for (auto& c : rbs[s * nRbK + j].c1) rbTc = rbTc && tc_layer(c);
            for (auto& c : rbs[s * nRbK + j].c2) rbTc = rbTc && tc_layer(c);
        }
        // fused ResBlock1 pairs (rb_fused.cuh): 32/64-channel stages whose every pair fits the fused kernel
        static const int env_fused = getenv("STTS_RB_FUSED") ? atoi(getenv("STTS_RB_FUSED")) : 1;
        bool rbFused = rbTc && env_fused && (C == 16 || C == 32 || C == 64) && nRbK >= 1 && nRbK <= 3;
        for (int j = 0; j < nRbK && rbFused; ++j) {
            const RB& rb = rbs[s * nRbK + j];
            if (rb.c1.size() != rb.c2.size() || rb.c1.empty()) rbFused = false;
            for (size_t q = 0; q < rb.c1.size() && rbFused; ++q)
                rbFused = rb_pair_eligible(rb.c1[q].rb, rb.c2[q].rb) && rb_plan(C, rb.c1[q].rb, rb.c2[q].rb).smem <= 227 * 1024;
        }
        if (rbTc) {
            xxP = arena_planes(curRowsTotal, B, C);
            // leaky(0.1)(xx) once for the three ResBlock1 branches (ResBlock1.cpp:61)
            dim3 g(((size_t)(ml + 2 * TC_GAP) * (C / 8) + 255) / 256, B);
            split_planes_kernel<<<g, 256, 0, stream>>>(xx, C, sseg, C, ACT_LEAKY, 0.1f, xxP);
            launch_check();
        }
        if (rbFused) {
            // x (planes of leaky(x)) -> pair -> pair -> pair (planes of x') per branch; MRF mean over the branches' planes.
            // No fp32 intermediate exists in HBM (ResBlock1.cpp:55-69, Generator_MS.cpp:177-196).
            Planes pp[2] = {arena_planes(curRowsTotal, B, C), arena_planes(curRowsTotal, B, C)};
            Planes op[3];
            for (int j = 0; j < nRbK; ++j) op[j] = arena_planes(curRowsTotal, B, C);
            for (int q = 0; q < 2 + nRbK; ++q) {
                const Planes& z = q < 2 ? pp[q] : op[q - 2];
                dim3 g((2 * (C / 8) * 2 * TC_GAP + 255) / 256, B);
                planes_gap_zero_kernel<<<g, 256, 0, stream>>>(z, sseg);
                launch_check();
            }
            std::vector<int> lens(B);
            for (int u = 0; u < B; ++u) lens[u] = (h_foff[u + 1] - h_foff[u]) * rate;
            for (int j = 0; j < nRbK; ++j) {
                const RB& rb = rbs[s * nRbK + j];
                const int nb = (int)rb.c1.size();
                const Planes* in = &xxP;
                const int2* tiles = nullptr; int ntiles = 0, tiles_ov = 0;
                for (int q = 0; q < nb; ++q) {
                    const bool last = q == nb - 1;
                    const Planes* out = last ? &op[j] : &pp[q & 1];
                    if (rb_ov(rb.c2[q].rb) != tiles_ov) { tiles_ov = rb_ov(rb.c2[q].rb); tiles = rb_tiles(sseg, lens, tiles_ov, ntiles); }
                    ProfRec pr;
                    if (profOn) prof_begin(pr, 2.0 * (rb.c1[q].macs_row + rb.c2[q].macs_row) * (double)curRowsTotal);
                    const int r = rb_pair_launch(C, rb.c1[q].rb, rb.c2[q].rb, *in, *out, sseg, tiles, ntiles, 0.1f, last ? ACT_NONE : ACT_LEAKY, 0.1f,
                                                 tensor_mode == 2 ? 1 : 0, sms, d_flags, stream);
                    if (r < 0) throw CudaError("fused ResBlock1 pair launch failed (" + std::to_string(r) + ")");
                    launch_check();
                    if (profOn) prof_end(pr);
                    in = out;
                }
            }
            {
                dim3 g(((size_t)ml * (C / 8) + 255) / 256, B);
                mrf_combine_kernel<<<g, 256, 0, stream>>>(op[0], op[nRbK > 1 ? 1 : 0], op[nRbK > 2 ? 2 : 0], nRbK, (float)nRbK, sseg, accb, C, 0.f);
                launch_check();
            }
            cur = accb; curC = C;
            continue;
        }
        float* t1 = ws.get<float>(rows * C);
        float* xa = ws.get<float>(rows * C);
        float* accT = nullptr;                   // tensor path: MRF partial sums, tile-transposed
        if (rbTc) {
            t1P = arena_planes(curRowsTotal, B, C); xaP = arena_planes(curRowsTotal, B, C);
            if (nRbK > 1) accT = ws.get<float>(rows * C);
        }
#else
        float* t1 = ws.get<float>(rows * C);
        float* xa = ws.get<float>(rows * C);
        float* accT = nullptr;
#endif
        for (int j = 0; j < nRbK; ++j) {                                         // MRF: Generator_MS.cpp:177-196
            RB& rb = rbs[s * nRbK + j];
            const int nb = (int)rb.c1.size();
            for (int b = 0; b < nb; ++b) {                                       // ResBlock1::forward, ResBlock1.cpp:55-69
                const float* src = b == 0 ? xx : xa;
                ConvOpts o1; o1.in_act = ACT_LEAKY; o1.in_slope = 0.1f;
                ConvOpts o2; o2.in_act = ACT_LEAKY; o2.in_slope = 0.1f; o2.res = src; o2.ldr = C;
                const bool last = b == nb - 1;
#ifdef STTS_WITH_TC
                if (rbTc) {
                    o1.in_planes = b == 0 ? &xxP : &xaP;                                  // leaky(x) planes
                    o1.out_planes = &t1P; o1.out_act = ACT_LEAKY; o1.out_slope = 0.1f;   // leaky(conv1(...)) planes only
                    o1.write_f32 = false;
                    o2.in_planes = &t1P;
                    if (!last) { o2.out_planes = &xaP; o2.out_act = ACT_LEAKY; o2.out_slope = 0.1f; }
                    // xa (the ResBlock's running x) is only read and written by conv2 epilogues: tile-transposed
                    o2.res_tt = b > 0;
                    o2.y_tt = !last;
                }
#endif
                conv(rb.c1[b], src, C, t1, C, sseg, B, ml, o1);
                float* dst = xa;
                if (last) {
                    dst = accb;
                    if (j == 0) o2.epi = EPI_STORE;
                    else if (j < nRbK - 1) o2.epi = EPI_ACCUM;
                    else { o2.epi = EPI_ACCUM_DIV; o2.div = (float)nRbK; }
#ifdef STTS_WITH_TC
                    if (rbTc && accT) {          // partial sums live tile-transposed in accT; the last branch writes row-major accb
                        if (j < nRbK - 1) { dst = accT; o2.y_tt = true; }
                        else { o2.acc_src = accT; o2.acc_tt = true; }
                    }
#endif
                }
                conv(rb.c2[b], t1, C, dst, C, sseg, B, ml, o2);
            }
        }
        cur = accb; curC = C;
    }
    float* o = ws.get<float>((size_t)std::max<int64_t>(St, 1));
    bool tailDone = false;
    curCls = STTS_CLS_DEC_TAIL; curRowsTotal = (int64_t)Ft * rate + (decType == 0 ? 0 : B);
    if (decType == 0) {
        // leaky(0.01) -> conv_post -> tanh: Generator_hifigan.cpp:176-180
        ConvOpts t; t.in_act = ACT_LEAKY; t.in_slope = 0.01f; t.epi = EPI_TANH; t.allow_tc = false;
        conv(convPost, cur, curC, o, 1, Seg{d_foff, rate, 0}, B, maxF * rate, t);
    } else {
        const Seg sin{d_foff, rate, 0}, sfr{d_foff, rate, 1}, sy{d_foff, rate * 4, 0};
        const size_t frRows = (size_t)Ft * rate + B;
        float* xr = ws.get<float>(frRows * curC);
        float* sp = ws.get<float>(frRows * subPost.Cout);
        float* frames = ws.get<float>(frRows * subBands * 16);
        float* yb = ws.get<float>((size_t)Ft * rate * 4 * subBands);
        {
            dim3 g(((size_t)(maxF * rate + 1) * curC + 255) / 256, B);
            refpad_leaky_kernel<<<g, 256, 0, stream>>>(cur, xr, sin, sfr, curC, 0.01f);
            launch_check();
        }
        conv(subPost, xr, curC, sp, subPost.Cout, sfr, B, maxF * rate + 1);
        static const int env_tail = getenv("STTS_TAIL_FUSED") ? atoi(getenv("STTS_TAIL_FUSED")) : 1;
        if (decType != 2 && subBands == 4 && env_tail) {
            // exp / pi*sin, inverse DFT, overlap-add, synthesis FIR and the PCM cast in ONE launch, intermediates in shared memory
            d_pcm = ws.get<int16_t>((size_t)std::max<int64_t>(St, 1));
            static const int env_ti = getenv("STTS_TAIL_TI") ? atoi(getenv("STTS_TAIL_TI")) : 256;
            const int ti = env_ti == 512 ? 512 : (env_ti == 128 ? 128 : 256);
            dim3 g((maxF * rate * 4 + ti - 1) / ti, B);
            const Seg sso{d_foff, rate * 16, 0};
            if (ti == 512) ms_tail_kernel<512><<<g, 256, ms_tail_smem(512), stream>>>(sp, subPost.Cout, msW, msB, o, d_pcm, sfr, sy, sso);
            else if (ti == 128) ms_tail_kernel<128><<<g, 256, ms_tail_smem(128), stream>>>(sp, subPost.Cout, msW, msB, o, d_pcm, sfr, sy, sso);
            else ms_tail_kernel<256><<<g, 256, ms_tail_smem(256), stream>>>(sp, subPost.Cout, msW, msB, o, d_pcm, sfr, sy, sso);
            launch_check();
            tailDone = true;
        } else {
        istft_frames_kernel<<<(frRows + 6) / 7, 256, 0, stream>>>(sp, subPost.Cout, frames, (int)frRows, subBands);
        launch_check();
        {
            dim3 g(((size_t)maxF * rate * 4 * subBands + 255) / 256, B);
            istft_ola_kernel<<<g, 256, 0, stream>>>(frames, yb, sfr, sy, subBands);
            launch_check();
        }
        if (decType == 2) {
            copy_kernel<<<(St + 255) / 256, 256, 0, stream>>>(yb, o, (size_t)St);
            launch_check();
        } else {
            dim3 g(((size_t)maxF * rate * 16 + 255) / 256, B);
            synth_fir_kernel<<<g, 256, 0, stream>>>(yb, msW, msB, o, sy, Seg{d_foff, rate * 16, 0});
            launch_check();
        }
        }
    }
    if (!tailDone) {
        d_pcm = ws.get<int16_t>((size_t)std::max<int64_t>(St, 1));
        pcm_kernel<<<(St + 255) / 256, 256, 0, stream>>>(o, d_pcm, (size_t)St);
        launch_check();
    }
    CUDA_CHECK(cudaEventRecord(ev[5], stream));
    if (tensor_mode >= 1) CUDA_CHECK(cudaMemcpyAsync(h_flags, d_flags, 4, cudaMemcpyDeviceToHost, stream));
    CUDA_CHECK(cudaStreamSynchronize(stream));
    if (tensor_mode >= 1 && (h_flags[0] & 1u)) {
        // an activation left the range the split-fp16 operands can represent (|x| > ~8000; shipped models peak at 126):
        // the saturated result is discarded and the batch is recomputed on the fp32 FFMA tiles
        const int keep = tensor_mode;
        h_flags[0] = 0;
        ++fallbacks;
        tensor_mode = 0;
        try { run(); } catch (...) { tensor_mode = keep; throw; }
        tensor_mode = keep;
        return;
    }
    for (int i = 0; i < 5; ++i) CUDA_CHECK(cudaEventElapsedTime(&lastMs[i], ev[i], ev[i + 1]));
    CUDA_CHECK(cudaEventElapsedTime(&lastMs[5], ev[0], ev[5]));
    if (profOn) prof_collect();
    const int sMul = R * tailMul;
    h_soff.assign(B + 1, 0);
    for (int u = 0; u <= B; ++u) h_soff[u] = (int64_t)h_foff[u] * sMul;
    if (!injectZ) { dbg.xx = x; dbg.m = mbuf; dbg.logs = logsbuf; dbg.logw = logw; dbg.wceil = wceil; dbg.zp = zp_dbg; }
    dbg.z = z; dbg.o = o;
    runValid = true;
}

// ---------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------
template <typename F>
static int guard(F&& f) {
    try {
        f();
        return STTS_OK;
    } catch (const FormatError& e) { g_last_error = e.what(); return STTS_E_FORMAT;
    } catch (const Unsupported& e) { g_last_error = e.what(); return STTS_E_UNSUPPORTED;
    } catch (const ArgError& e) { g_last_error = e.what(); return STTS_E_ARG;
    } catch (const CudaError& e) { g_last_error = e.what(); return STTS_E_CUDA;
    } catch (const std::bad_alloc&) { g_last_error = "out of host memory"; return STTS_E_NOMEM;
    } catch (const std::exception& e) { g_last_error = e.what(); return STTS_E_CUDA; }
}

extern "C" {

const char* stts_last_error(void) { return g_last_error.c_str(); }
const char* stts_version(void) {
#ifdef STTS_WITH_TC
    return "stts_b200 0.2 (sm_100a; fp32 FFMA tiles + tcgen05 split-fp16 tiles)";
#else
    return "stts_b200 0.2 (sm_100a; fp32 FFMA tiles)";
#endif
}
void stts_free(void* p) { free(p); }

int stts_describe_model(const float* blob, int64_t bytes, char** text, int64_t* nn_end) {
    return guard([&] {
        if (!blob || bytes < 16 || !text) throw ArgError("null blob / text");
        Model M = parse_model(blob, bytes / 4);
        std::string s = describe(M);
        *text = (char*)malloc(s.size() + 1);
        memcpy(*text, s.c_str(), s.size() + 1);
        if (nn_end) *nn_end = M.nnEnd;
    });
}

int stts_create(const float* blob, int64_t bytes, int device, stts_engine** out) {
    if (out) *out = nullptr;
    stts_engine* e = nullptr;
    int rc = guard([&] {
        if (!blob || bytes < 16 || !out) throw ArgError("null blob / out");
        int ndev = 0;
        cudaError_t ce = cudaGetDeviceCount(&ndev);
        if (ce != cudaSuccess || ndev <= 0)
            throw CudaError(std::string("no CUDA device available (there is no CPU fallback): ") + cudaGetErrorString(ce));
        if (device < 0 || device >= ndev) throw ArgError("device index out of range");
        CUDA_CHECK(cudaSetDevice(device));
        cudaDeviceProp prop;
        CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
        if (prop.major != 10) throw CudaError("this library contains sm_100a code only; device is sm_" + std::to_string(prop.major) + std::to_string(prop.minor));
        Model M = parse_model(blob, bytes / 4);
        e = new stts_engine();
        e->device = device;
        CUDA_CHECK(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
        for (auto& ev : e->ev) CUDA_CHECK(cudaEventCreate(&ev));
        e->build(M);
        CUDA_CHECK(cudaDeviceSynchronize());
        *out = e;
    });
    if (rc != STTS_OK && e) { stts_destroy(e); }
    return rc;
}

// stts_create with a pre-packed device image on disk (SURVEY.md §8f rank 4: the reference re-parses and copies every weight at
// every process start, SynthesizerTrn.cpp:91-167 + utils.cpp:8-32).  image_path missing / stale / foreign: the engine is built
// from the blob as usual and the image is (re)written; matching: every dense conv's packed device representation is read from the
// image instead of being transposed, split and packed on the host.  *from_image = 1 when the image was used.
static uint64_t nn_hash(const float* blob, int64_t nfloats) {
    const uint32_t* w = reinterpret_cast<const uint32_t*>(blob);
    uint64_t h = 0x9E3779B97F4A7C15ull ^ (uint64_t)nfloats;
    for (int64_t i = 0; i < nfloats; ++i) { h ^= w[i]; h *= 0x100000001B3ull; h ^= h >> 29; }
    return h;
}
int stts_create_cached(const float* blob, int64_t bytes, int device, const char* image_path, stts_engine** out, int32_t* from_image) {
    if (out) *out = nullptr;
    if (from_image) *from_image = 0;
    if (!image_path || !*image_path) return stts_create(blob, bytes, device, out);
    stts_engine* e = nullptr;
    int rc = guard([&] {
        if (!blob || bytes < 16 || !out) throw ArgError("null blob / out");
        int ndev = 0;
        cudaError_t ce = cudaGetDeviceCount(&ndev);
        if (ce != cudaSuccess || ndev <= 0)
            throw CudaError(std::string("no CUDA device available (there is no CPU fallback): ") + cudaGetErrorString(ce));
        if (device < 0 || device >= ndev) throw ArgError("device index out of range");
        CUDA_CHECK(cudaSetDevice(device));
        Model M = parse_model(blob, bytes / 4);
        struct Hdr { char magic[8]; uint64_t key; uint64_t dconv; int64_t nrec; } want;
        memcpy(want.magic, "STTSIMG2", 8);
        want.key = nn_hash(blob, M.nnEnd) ^ std::hash<std::string>()(stts_version());
        want.dconv = sizeof(DConv);
        want.nrec = 0;
        for (int attempt = 0; attempt < 2 && !e; ++attempt) {
            e = new stts_engine();
            e->device = device;
            CUDA_CHECK(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
            for (auto& ev : e->ev) CUDA_CHECK(cudaEventCreate(&ev));
            FILE* f = attempt == 0 ? fopen(image_path, "rb") : nullptr;
            Hdr got;
            if (f && fread(&got, sizeof(got), 1, f) == 1 && !memcmp(got.magic, want.magic, 8) && got.key == want.key && got.dconv == want.dconv) {
                e->img.mode = 2; e->img.f = f;
                try {
                    e->build(M);
                    if (e->img.nrec != got.nrec) throw FormatError("device image: record count mismatch");
                    fclose(f); e->img.f = nullptr; e->img.mode = 0;
                    if (from_image) *from_image = 1;
                } catch (const FormatError&) {        // stale / truncated image: rebuild from the blob and rewrite it
                    fclose(f); e->img.f = nullptr;
                    stts_destroy(e); e = nullptr;
                }
            } else {
                if (f) fclose(f);
                const std::string tmp = std::string(image_path) + ".tmp";
                FILE* w = fopen(tmp.c_str(), "wb");
                if (w) { e->img.mode = 1; e->img.f = w; fwrite(&want, sizeof(want), 1, w); }
                e->build(M);
                if (w) {
                    want.nrec = e->img.nrec;
                    fseek(w, 0, SEEK_SET);
                    fwrite(&want, sizeof(want), 1, w);
                    fclose(w);
                    e->img.f = nullptr; e->img.mode = 0;
                    rename(tmp.c_str(), image_path);
                }
            }
        }
        if (!e) throw std::runtime_error("device image: rebuild failed");
        CUDA_CHECK(cudaDeviceSynchronize());
        *out = e;
    });
    if (rc != STTS_OK && e) { if (e->img.f) fclose(e->img.f); stts_destroy(e); }
    return rc;
}

void stts_destroy(stts_engine* e) {
    if (!e) return;
    cudaSetDevice(e->device);
    if (e->stream) cudaStreamSynchronize(e->stream);
    for (void* p : e->owned) cudaFree(p);
#ifdef STTS_WITH_TC
    if (e->planeScratch) cudaFree(e->planeScratch);
#endif
    if (e->wsAlloc) cudaFree(e->wsAlloc);
    if (e->streamZ) cudaFree(e->streamZ);
    for (void* p : {(void*)e->d_ids, (void*)e->d_toff, (void*)e->d_sids, (void*)e->d_ls, (void*)e->d_foff, (void*)e->d_nfr,
                    (void*)e->d_bseg, (void*)e->d_forced, (void*)e->d_ns, (void*)e->d_nsw, (void*)e->d_seed})
        if (p) cudaFree(p);
    if (e->hostPcm) cudaFreeHost(e->hostPcm);
    if (e->hostInts) cudaFreeHost(e->hostInts);
    if (e->h_flags) cudaFreeHost(e->h_flags);
    for (auto& ev : e->ev) if (ev) cudaEventDestroy(ev);
    for (auto& ev : e->profPool) cudaEventDestroy(ev);
    if (e->stream) cudaStreamDestroy(e->stream);
    delete e;
}

int64_t stts_nn_end_offset(const stts_engine* e) { return e ? e->nnEnd : -1; }
int32_t stts_speaker_num(const stts_engine* e) { return e ? e->spkNum : -1; }
int32_t stts_header_field(const stts_engine* e, int32_t which) {
    if (!e) return -1;
    switch (which) { case 0: return e->isMS; case 1: return e->langType; case 2: return e->durPredType; case 3: return e->decType; }
    return -1;
}
int64_t stts_kernel_launches(const stts_engine* e) { return e ? e->launches : 0; }
int64_t stts_tensor_fallbacks(const stts_engine* e) { return e ? e->fallbacks : 0; }
void* stts_stream(const stts_engine* e) { return e ? (void*)e->stream : nullptr; }

int stts_set_tensor_path(stts_engine* e, int32_t mode) {
    return guard([&] {
        if (!e) throw ArgError("null engine");
#ifndef STTS_WITH_TC
        if (mode != 0) throw Unsupported("this build has no tensor-core path");
#endif
        e->tensor_mode = mode;
    });
}

int stts_set_forced_durations(stts_engine* e, const float* w, int64_t n) {
    return guard([&] {
        if (!e) throw ArgError("null engine");
        if (!w || n <= 0) e->forced.clear();
        else e->forced.assign(w, w + n);
    });
}
int stts_set_sampling(stts_engine* e, int32_t n, const float* ns, const float* nsw, const uint64_t* seeds) {
    return guard([&] {
        if (!e || n < 0) throw ArgError("null engine or n < 0");
        if (n == 0 || (!ns && !nsw)) {
            e->smpNs.clear(); e->smpNsw.clear(); e->smpSeed.clear();
            return;
        }
        std::vector<float> a(n, 0.f), b(n, 0.f);
        std::vector<uint64_t> s(n, 0);
        for (int i = 0; i < n; ++i) {
            if (ns) a[i] = ns[i];
            if (nsw) b[i] = nsw[i];
            if (seeds) s[i] = seeds[i];
            if (!(a[i] >= 0.f && a[i] <= 10.f) || !(b[i] >= 0.f && b[i] <= 10.f))
                throw ArgError("noise scales must be finite and in [0, 10] (utterance " + std::to_string(i) + ")");
        }
        e->smpNs.swap(a); e->smpNsw.swap(b); e->smpSeed.swap(s);
    });
}
int stts_debug_noise(uint64_t seed, int32_t stream, int64_t rows, int32_t cols, float* out) {
    return guard([&] {
        if (!out || rows < 0 || cols < 1 || (stream == RNG_STREAM_SDP && cols != 2) || (stream != RNG_STREAM_PRIOR && stream != RNG_STREAM_SDP))
            throw ArgError("stream 0 (prior, cols >= 1) or 1 (SDP, cols == 2), rows >= 0, out non-null");
        float e[4];
        for (int64_t r = 0; r < rows; ++r) {
            if (stream == RNG_STREAM_SDP) {
                philox_normals4((uint32_t)r, 0u, 1u, 0u, seed, e);
                out[r * 2] = e[0]; out[r * 2 + 1] = e[1];
                continue;
            }
            for (int q = 0; 4 * q < cols; ++q) {
                philox_normals4((uint32_t)r, (uint32_t)q, 0u, 0u, seed, e);
                for (int j = 0; j < 4 && 4 * q + j < cols; ++j) out[r * cols + 4 * q + j] = e[j];
            }
        }
    });
}
int stts_debug_enable(stts_engine* e, int32_t on) {
    if (!e) return STTS_E_ARG;
    e->debug = on != 0;
    return STTS_OK;
}

int stts_batch_stage(stts_engine* e, int32_t B, const int32_t* ids, const int32_t* offs, const int32_t* sids, const float* ls) {
    return guard([&] {
        if (!e) throw ArgError("null engine");
        CUDA_CHECK(cudaSetDevice(e->device));
        e->stage(B, ids, offs, sids, ls);
    });
}
int stts_batch_run(stts_engine* e, int64_t* total) {
    return guard([&] {
        if (!e) throw ArgError("null engine");
        CUDA_CHECK(cudaSetDevice(e->device));
        e->run();
        if (total) *total = e->St;
    });
}
int stts_batch_fetch(stts_engine* e, int16_t* pcm, int64_t cap, int64_t* soff) {
    return guard([&] {
        if (!e || !pcm) throw ArgError("null engine / buffer");
        if (!e->runValid || !e->d_pcm) throw ArgError("no completed run to fetch from");
        if (e->St > cap) throw ArgError("pcm buffer too small");
        CUDA_CHECK(cudaSetDevice(e->device));
        CUDA_CHECK(cudaMemcpyAsync(pcm, e->d_pcm, (size_t)e->St * 2, cudaMemcpyDeviceToHost, e->stream));
        CUDA_CHECK(cudaStreamSynchronize(e->stream));
        if (soff) for (int u = 0; u <= e->B; ++u) soff[u] = e->h_soff[u];
    });
}

int stts_infer_batch_into(stts_engine* e, int32_t B, const int32_t* ids, const int32_t* offs, const int32_t* sids,
                          const float* ls, int16_t* pcm, int64_t cap, int64_t* soff) {
    int rc = stts_batch_stage(e, B, ids, offs, sids, ls);
    if (rc) return rc;
    rc = stts_batch_run(e, nullptr);
    if (rc) return rc;
    return stts_batch_fetch(e, pcm, cap, soff);
}

int stts_infer_batch(stts_engine* e, int32_t B, const int32_t* ids, const int32_t* offs, const int32_t* sids,
                     const float* ls, int16_t** pcm, int32_t* ns) {
    int rc = stts_batch_stage(e, B, ids, offs, sids, ls);
    if (rc) return rc;
    rc = stts_batch_run(e, nullptr);
    if (rc) return rc;
    return guard([&] {
        if (!pcm || !ns) throw ArgError("null output arrays");
        if ((size_t)e->St > e->hostPcmCap) {
            if (e->hostPcm) CUDA_CHECK(cudaFreeHost(e->hostPcm));
            e->hostPcmCap = (size_t)e->St + (size_t)e->St / 4;
            CUDA_CHECK(cudaMallocHost((void**)&e->hostPcm, e->hostPcmCap * 2));
        }
        CUDA_CHECK(cudaMemcpyAsync(e->hostPcm, e->d_pcm, (size_t)e->St * 2, cudaMemcpyDeviceToHost, e->stream));
        CUDA_CHECK(cudaStreamSynchronize(e->stream));
        for (int u = 0; u < B; ++u) pcm[u] = nullptr;
        for (int u = 0; u < B; ++u) {
            const int64_t n = e->h_soff[u + 1] - e->h_soff[u];
            pcm[u] = (int16_t*)malloc(std::max<int64_t>(n, 1) * 2);   // malloc'd like SynthesizerTrn.cpp:391
            if (!pcm[u]) {
                for (int v = 0; v < u; ++v) { free(pcm[v]); pcm[v] = nullptr; }
                throw std::bad_alloc();
            }
            memcpy(pcm[u], e->hostPcm + e->h_soff[u], (size_t)n * 2);
            ns[u] = (int32_t)n;
        }
    });
}

// Chunked synthesis of one utterance (SURVEY.md §8f rank 1): the token-level half runs once, then flow + decoder run over
// frame chunks with a halo that covers their receptive field; every chunk's PCM is handed to `cb` as soon as it is on the
// host.  The flow and the decoder are purely convolutional (ResidualCouplingBlock.cpp:59-71, Generator_MS.cpp:166-229), so the
// concatenated chunks are bit-identical to the one-shot result.  The reference synthesises the whole text as one utterance
// and returns only at the end (test/main.cpp:90-142).
int stts_infer_stream(stts_engine* e, const int32_t* ids, int32_t n, int32_t sid, float ls, int32_t chunk_frames,
                      stts_pcm_callback cb, void* user, float* first_chunk_ms, int64_t* total_samples) {
    int rc = guard([&] {
        if (!e || !ids || !cb || chunk_frames < 16) throw ArgError("null argument or chunk_frames < 16");
        CUDA_CHECK(cudaSetDevice(e->device));
        cudaEvent_t t0, t1;
        CUDA_CHECK(cudaEventCreate(&t0)); CUDA_CHECK(cudaEventCreate(&t1));
        CUDA_CHECK(cudaEventRecord(t0, e->stream));
        const int32_t offs[2] = {0, n};
        e->stage(1, ids, offs, &sid, &ls);
        e->injectZ = nullptr; e->stopAfterRegulate = true;
        try { e->run(); } catch (...) { e->stopAfterRegulate = false; throw; }
        e->stopAfterRegulate = false;
        const int F = e->streamF;
        // receptive-field halo in frames: flow = sum over coupling layers / WN layers of (k-1)/2; decoder = conv_pre + per stage
        // (transposed conv taps + the deepest ResBlock1 branch) / rate + the tail (subband conv, iSTFT overlap, synthesis FIR)
        int halo = 0;
        for (auto& L : e->flow) for (auto& c : L.in) halo += (c.k - 1) / 2 * c.dil;
        halo += e->convPre.padl + 1;
        int rate = 1;
        for (size_t s = 0; s < e->ups.size(); ++s) {
            halo += (e->ups[s].k + rate - 1) / rate + 1;
            rate *= e->upRates[s];
            int deepest = 0;
            for (int j = 0; j < e->nRbK; ++j) {
                int rows = 0;
                const auto& rb = e->rbs[s * e->nRbK + j];
                for (size_t q = 0; q < rb.c1.size(); ++q) rows += rb.c1[q].padl + rb.c2[q].padl;
                deepest = std::max(deepest, rows);
            }
            halo += (deepest + rate - 1) / rate + 1;
        }
        halo += 4;
        int64_t total = 0;
        bool first = true;
        const int sMul = [&] { int R = 1; for (int r : e->upRates) R *= r; return R * (e->decType == 0 ? 1 : (e->decType == 2 ? 4 : 16)); }();
        for (int c0 = 0; c0 < F; c0 += chunk_frames) {
            const int c1 = std::min(F, c0 + chunk_frames);
            const int s0 = std::max(0, c0 - halo), s1 = std::min(F, c1 + halo);
            e->injectZ = e->streamZ + (size_t)s0 * e->inter; e->injectF = s1 - s0;
            try { e->run(); } catch (...) { e->injectZ = nullptr; throw; }
            e->injectZ = nullptr;
            const int64_t ns = (int64_t)(c1 - c0) * sMul, off = (int64_t)(c0 - s0) * sMul;
            if ((size_t)ns > e->hostPcmCap) {
                if (e->hostPcm) CUDA_CHECK(cudaFreeHost(e->hostPcm));
                e->hostPcm = nullptr; e->hostPcmCap = 0;
                CUDA_CHECK(cudaMallocHost((void**)&e->hostPcm, (size_t)ns * 2 + 4096));
                e->hostPcmCap = (size_t)ns + 2048;
            }
            CUDA_CHECK(cudaMemcpyAsync(e->hostPcm, e->d_pcm + off, (size_t)ns * 2, cudaMemcpyDeviceToHost, e->stream));
            if (first) CUDA_CHECK(cudaEventRecord(t1, e->stream));
            CUDA_CHECK(cudaStreamSynchronize(e->stream));
            if (first && first_chunk_ms) CUDA_CHECK(cudaEventElapsedTime(first_chunk_ms, t0, t1));
            first = false;
            cb(e->hostPcm, ns, user);
            total += ns;
        }
        if (total_samples) *total_samples = total;
        e->runValid = false;          // d_pcm holds only the last chunk
        cudaEventDestroy(t0); cudaEventDestroy(t1);
    });
    return rc;
}

int stts_infer_ids(stts_engine* e, const int32_t* ids, int32_t n, int32_t sid, float ls, int16_t** pcm, int32_t* ns) {
    const int32_t offs[2] = {0, n};
    return stts_infer_batch(e, 1, ids, offs, &sid, &ls, pcm, ns);
}

int stts_debug_fetch(stts_engine* e, int32_t which, float** out, int64_t* rows, int64_t* cols) {
    return guard([&] {
        if (!e || !out || !rows || !cols) throw ArgError("null argument");
        if (e->B <= 0 || !e->runValid || !e->dbg.xx) throw ArgError("no completed run to fetch from");
        const int T0 = e->h_toff[1] - e->h_toff[0], F0 = e->h_foff[1] - e->h_foff[0];
        const float* src = nullptr;
        int64_t r = 0, c = 1;
        switch (which) {
            case 0: src = e->dbg.xx; r = T0; c = e->hidden; break;
            case 1: src = e->dbg.m; r = T0; c = e->inter; break;
            case 2: src = e->dbg.logw; r = T0; break;
            case 3: src = e->dbg.wceil; r = T0; break;
            case 4: src = e->dbg.zp; r = F0; c = e->inter; if (!src) throw ArgError("z_p is only kept when stts_debug_enable(1) was set before the run"); break;
            case 5: src = e->dbg.z; r = F0; c = e->inter; break;
            case 6: src = e->dbg.o; r = e->h_soff[1] - e->h_soff[0]; break;
            case 7: src = e->dbg.logs; r = T0; c = e->inter; if (!src) throw ArgError("logs is only computed when the batch samples the prior"); break;
            default: throw ArgError("unknown stage id");
        }
        *out = (float*)malloc(std::max<int64_t>(r * c, 1) * 4);
        CUDA_CHECK(cudaSetDevice(e->device));
        CUDA_CHECK(cudaMemcpy(*out, src, (size_t)(r * c) * 4, cudaMemcpyDeviceToHost));
        *rows = r; *cols = c;
    });
}

int stts_profile_enable(stts_engine* e, int32_t on) {
    if (!e) return STTS_E_ARG;
    e->profOn = on != 0;
    for (int i = 0; i < STTS_NUM_CLS; ++i) { e->profMs[i] = 0; e->profFlops[i] = 0; e->profLaunch[i] = 0; }
    return STTS_OK;
}
int stts_profile_fetch(const stts_engine* e, double* ms, double* flops, int64_t* launches) {
    if (!e || !ms || !flops || !launches) return STTS_E_ARG;
    for (int i = 0; i < STTS_NUM_CLS; ++i) { ms[i] = e->profMs[i]; flops[i] = e->profFlops[i]; launches[i] = e->profLaunch[i]; }
    return STTS_OK;
}

// Op-level test hook: one conv (or ConvTranspose1d) through the FFMA tiles (use_tc == 0) or the
// tcgen05 path (use_tc == 1) on caller-provided data.  x: [T][Cin] with optional utterance offsets.
int stts_debug_pack_weights(const float* w, int32_t k, int32_t Cin, int32_t Cout, int32_t usteps, int32_t* meta,
                            uint16_t** halves, int64_t* n_halves) {
    return guard([&]() {
#ifdef STTS_WITH_TC
        if (!w || !meta || !halves || !n_halves || k < 1 || Cin < 1 || Cout < 1) throw std::invalid_argument("bad argument");
        // file order W[o][k][c] -> device order [k][Cin][CoutW]
        const int CoutW = (Cout + 3) & ~3;
        std::vector<float> dw((size_t)k * Cin * CoutW, 0.f);
        for (int o = 0; o < Cout; ++o)
            for (int t = 0; t < k; ++t)
                for (int c = 0; c < Cin; ++c) dw[((size_t)t * Cin + c) * CoutW + o] = w[((size_t)o * k + t) * Cin + c];
        TcWeights tw;
        std::vector<__half> buf;
        const bool ok = tc_pack_weights_host(tw, dw.data(), k, Cin, Cout, CoutW, buf, usteps);
        meta[0] = ok ? 1 : 0; meta[1] = tw.NC; meta[2] = tw.nchunks; meta[3] = tw.KC; meta[4] = tw.kchunks;
        meta[5] = tw.colsplit; meta[6] = tw.merge; meta[7] = tw.usteps; meta[8] = tw.wexp;
        *n_halves = (int64_t)buf.size();
        *halves = nullptr;
        if (ok && !buf.empty()) {
            *halves = (uint16_t*)malloc(buf.size() * 2);
            if (!*halves) throw std::bad_alloc();
            memcpy(*halves, buf.data(), buf.size() * 2);
        }
#else
        (void)w; (void)k; (void)Cin; (void)Cout; (void)usteps; (void)meta; (void)halves; (void)n_halves;
        throw Unsupported("built without the tensor-core path");
#endif
    });
}

int stts_test_conv1d(int device, int use_tc, const float* rec, int64_t rec_floats, int transposed, int stride,
                     int pad_override, int dil_override, const float* x, int T, int nseg, const int* seg_off,
                     int in_act, float slope, int epi, float** y, int* rows, int* cols) {
    stts_engine* e = nullptr;
    int rc = guard([&] {
        if (!rec || !x || !y || !rows || !cols) throw ArgError("null argument");
        CUDA_CHECK(cudaSetDevice(device));
        e = new stts_engine();
        e->device = device;
        CUDA_CHECK(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
        e->device_setup();
        Cursor c{rec, rec_floats};
        ConvRec r = transposed ? parse_convT(c) : parse_conv(c);
        if (pad_override >= 0) r.pad = pad_override;
        if (dil_override > 0) r.dil = dil_override;
        if (transposed) r.stride = stride;
        DConv d;
        if (transposed) d = e->make_convT(r);
        else if (epi == EPI_GATE) {
            const int H = r.outCh / 2;
            std::vector<int> gm(2 * H);
            for (int j = 0; j < H; ++j) { gm[2 * j] = j; gm[2 * j + 1] = H + j; }
            d = e->make_conv(r, gm);
        } else d = e->make_conv(r);
        e->tensor_mode = use_tc;
#ifdef STTS_WITH_TC
        if (use_tc && !d.tc.ok) throw Unsupported("layer is not eligible for the tensor-core path");
#else
        if (use_tc) throw Unsupported("this build has no tensor-core path");
#endif
        std::vector<int> so;
        if (seg_off) so.assign(seg_off, seg_off + nseg + 1); else { nseg = 1; so = {0, T}; }
        int maxlen = 0;
        for (int i = 0; i < nseg; ++i) maxlen = std::max(maxlen, so[i + 1] - so[i]);
        int* dso = e->dalloc<int>(so.size());
        CUDA_CHECK(cudaMemcpy(dso, so.data(), so.size() * 4, cudaMemcpyHostToDevice));
        float* dx = e->upload(x, (size_t)T * r.inCh);
        const int outC = epi == EPI_GATE ? d.Cout / 2 : (transposed ? r.outCh : d.Cout);
        const int outRows = transposed ? T * r.stride : T;
        float* dy = e->dalloc<float>((size_t)outRows * outC);
        CUDA_CHECK(cudaMemset(dy, 0, (size_t)outRows * outC * 4));
        ConvOpts o; o.in_act = in_act; o.in_slope = slope; o.epi = epi;
        e->curRowsTotal = T;
        e->conv(d, dx, r.inCh, dy, transposed ? d.Cout : outC, Seg{dso, 1, 0}, nseg, maxlen, o);
        CUDA_CHECK(cudaStreamSynchronize(e->stream));
        *y = (float*)malloc((size_t)outRows * outC * 4);
        CUDA_CHECK(cudaMemcpy(*y, dy, (size_t)outRows * outC * 4, cudaMemcpyDeviceToHost));
        *rows = outRows; *cols = outC;
    });
    if (e) stts_destroy(e);
    return rc;
}

// Op-level test hook of the fused ResBlock1 pair (rb_fused.cuh): x' = act(x + conv2(leaky(conv1(leaky(x))))) on caller data,
// through planes in / planes out exactly as the decoder uses it.  mode 0 accurate, 1 throughput.
int stts_test_rbpair(int device, int mode, const float* rec1, int64_t n1, const float* rec2, int64_t n2, int dil1, const float* x,
                     int T, int nseg, const int* seg_off, int out_leaky, float** y, uint32_t* flags_out) {
    stts_engine* e = nullptr;
    int rc = guard([&] {
#ifdef STTS_WITH_TC
        if (!rec1 || !rec2 || !x || !y) throw ArgError("null argument");
        CUDA_CHECK(cudaSetDevice(device));
        e = new stts_engine();
        e->device = device;
        CUDA_CHECK(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
        e->device_setup();
        Cursor c1{rec1, n1}, c2{rec2, n2};
        ConvRec r1 = parse_conv(c1), r2 = parse_conv(c2);
        if (dil1 > 0) { r1.dil = dil1; r1.pad = dil1 * (r1.k - 1) / 2; }
        e->tc_usteps = 8;
        DConv d1 = e->make_conv(r1, {}, {}, 1.f, -1, true, true), d2 = e->make_conv(r2, {}, {}, 1.f, -1, true, true);
        const int C = r1.inCh;
        if (!rb_pair_eligible(d1.rb, d2.rb)) throw Unsupported("pair is not eligible for the fused kernel");
        std::vector<int> so;
        if (seg_off) so.assign(seg_off, seg_off + nseg + 1); else { nseg = 1; so = {0, T}; }
        int maxlen = 0;
        for (int i = 0; i < nseg; ++i) maxlen = std::max(maxlen, so[i + 1] - so[i]);
        int* dso = e->dalloc<int>(so.size());
        CUDA_CHECK(cudaMemcpy(dso, so.data(), so.size() * 4, cudaMemcpyHostToDevice));
        float* dx = e->upload(x, (size_t)T * C);
        float* dy = e->dalloc<float>((size_t)T * C);
        CUDA_CHECK(cudaMemset(dy, 0, (size_t)T * C * 4));
        e->ensure_ws(3 * stts_engine::planes_bytes(T, nseg, C) + (size_t)T / 16 + (2 << 20));
        e->ws.reset();
        const Seg seg{dso, 1, 0};
        Planes inP = e->arena_planes(T, nseg, C), outP = e->arena_planes(T, nseg, C);
        CUDA_CHECK(cudaMemsetAsync(outP.base, 0xff, (size_t)outP.rows_p * C * 4, e->stream));    // poison: every live row must be written
        {
            dim3 g(((size_t)(maxlen + 2 * TC_GAP) * (C / 8) + 255) / 256, nseg);
            split_planes_kernel<<<g, 256, 0, e->stream>>>(dx, C, seg, C, ACT_LEAKY, 0.1f, inP);
            dim3 g2((2 * (C / 8) * 2 * TC_GAP + 255) / 256, nseg);
            planes_gap_zero_kernel<<<g2, 256, 0, e->stream>>>(outP, seg);
        }
        std::vector<int> lens(nseg);
        for (int i = 0; i < nseg; ++i) lens[i] = so[i + 1] - so[i];
        int ntiles = 0;
        const int2* tiles = e->rb_tiles(seg, lens, rb_ov(d2.rb), ntiles);
        const int r = rb_pair_launch(C, d1.rb, d2.rb, inP, outP, seg, tiles, ntiles, 0.1f, out_leaky ? ACT_LEAKY : ACT_NONE, 0.1f, mode, e->sms,
                                     e->d_flags, e->stream);
        if (r < 0) throw CudaError("fused pair launch failed (" + std::to_string(r) + ")");
        e->launch_check();
        {
            dim3 g(((size_t)maxlen * (C / 8) + 255) / 256, nseg);
            mrf_combine_kernel<<<g, 256, 0, e->stream>>>(outP, outP, outP, 1, 1.f, seg, dy, C, 0.f);   // y = act(x') exactly as stored
        }
        CUDA_CHECK(cudaStreamSynchronize(e->stream));
        e->launch_check();
        *y = (float*)malloc((size_t)T * C * 4);
        CUDA_CHECK(cudaMemcpy(*y, dy, (size_t)T * C * 4, cudaMemcpyDeviceToHost));
        if (flags_out) CUDA_CHECK(cudaMemcpy(flags_out, e->d_flags, 4, cudaMemcpyDeviceToHost));
#else
        throw Unsupported("built without the tensor-core path");
#endif
    });
    if (e) stts_destroy(e);
    return rc;
}

int stts_last_timing(const stts_engine* e, float* ms, int32_t n) {
    if (!e || !ms) return STTS_E_ARG;
    for (int i = 0; i < n && i < 6; ++i) ms[i] = e->lastMs[i];
    return STTS_OK;
}

}  // extern "C"

#include "g2p.cuh"   // batched GRU g2p for out-of-vocabulary English words (SURVEY.md §8f rank 3): stts_g2p_*
