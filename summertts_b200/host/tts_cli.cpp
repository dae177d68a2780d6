// tts_cli.cpp — `tts_b200`: the reference demo's command line (test/main.cpp:75-148) plus what a serving box needs:
// batches, several GPUs, phoneme-id input.
//
//   tts_b200 <text.txt> <model.bin> <out.wav>                      reference behaviour: the whole file is ONE utterance
//                                                                  (lines joined with two spaces, BOM stripped, main.cpp:86-97);
//                                                                  models with > 20 speakers: speakers 10..19 at length scale
//                                                                  1.1 -> <out.wav>_<sid>.wav (main.cpp:108-129), else sid 0 / 1.0
//   tts_b200 --per-line ...                                        every non-empty line is its own utterance -> <out>_%04d.wav
//                                                                  (one batched call per GPU; --concat: one file, in order)
//   tts_b200 --ids <ids.txt> <model.bin> <out.wav>                 lines of phoneme ids instead of text (no frontend needed)
//   options: --gpus N (one engine + one host thread per GPU, longest-first partition), --sid S, --length-scale L,
//            --frontend-threads T (text -> ids on T host threads, one frontend instance each: at batch 64 the 3-4 ms/sentence
//            host frontend, not the GPU, is the serial bottleneck -- SURVEY §8f rank 3), --dump-ids (frontend only: print the
//            phoneme ids of every utterance, one line each, and stop -- no GPU needed; feeds `--ids` elsewhere),
//            --selftest-wav <out.wav> (writes one second of a 440 Hz tone; container check without a GPU),
//            --noise-scale NS, --noise-scale-w NSW, --seed S (VITS sampling, stts_set_sampling; defaults 0 0 0 = the reference's
//            deterministic output): job j of the input -- the j-th non-empty line under --per-line / --ids, the j-th speaker job
//            of the multi-speaker loop -- gets seed S + j, whatever GPU it lands on
//
// Text input needs the host frontend (frontend.hpp; built with -DSTTS_WITH_REF_FRONTEND against the reference's sources by
// `make REF=...`); the ids-only build has no dependency outside this repository.  No CPU fallback: without a usable
// sm_100 device stts_create fails and the tool exits non-zero with the library's message.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <numeric>
#include <sstream>
#include <string>
#include <thread>
#include <vector>

#include "stts_b200.h"
#include "wav.hpp"
#ifdef STTS_WITH_REF_FRONTEND
#include "frontend.hpp"
#endif

namespace {

struct Args {
    std::string input, model, out;
    bool ids = false, per_line = false, concat = false, dump_ids = false;
    int gpus = 1, sid = -1, fe_threads = 0;
    float length_scale = -1.f;
    float noise_scale = 0.f, noise_scale_w = 0.f;
    uint64_t seed = 0;
};

struct Utt {
    std::string text;
    std::vector<int32_t> ids;
    float ls = 1.f;
    int32_t sid = 0;
    uint64_t seed = 0;
    std::string out;
    std::vector<int16_t> pcm;
};

int usage(const char* argv0) {
    fprintf(stderr,
            "usage: %s [--ids] [--per-line] [--concat] [--dump-ids] [--gpus N] [--frontend-threads T] [--sid S] [--length-scale L]\n"
            "          [--noise-scale NS] [--noise-scale-w NSW] [--seed S] <input.txt> <model.bin> <out.wav>\n"
            "       %s --selftest-wav <out.wav>\n", argv0, argv0);
    return 2;
}

bool load_file(const std::string& path, std::vector<char>& buf) {
    std::ifstream f(path, std::ios::binary | std::ios::ate);
    if (!f) return false;
    const std::streamsize n = f.tellg();
    f.seekg(0);
    buf.resize((size_t)n);
    return n == 0 || (bool)f.read(buf.data(), n);
}

std::vector<std::string> read_lines(const std::string& path, bool* ok) {
    std::vector<std::string> out;
    std::ifstream f(path);
    *ok = (bool)f;
    std::string l;
    while (std::getline(f, l)) {
        if (l.size() >= 3 && (unsigned char)l[0] == 0xEF && (unsigned char)l[1] == 0xBB && (unsigned char)l[2] == 0xBF) l = l.substr(3);
        if (!l.empty() && l.back() == '\r') l.pop_back();
        out.push_back(l);
    }
    return out;
}

std::string numbered(const std::string& out, const char* fmt, int i) {
    char b[32];
    snprintf(b, sizeof b, fmt, i);
    return out + b;
}

// one engine per GPU; utterances partitioned longest-first (summertts_b200/shard.py::balanced does the same for Python callers)
int run_device(int dev, const std::vector<char>& model, std::vector<Utt*>& work, float noise_scale, float noise_scale_w, std::string* err) {
    if (work.empty()) return 0;
    stts_engine* e = nullptr;
    if (stts_create(reinterpret_cast<const float*>(model.data()), (int64_t)model.size(), dev, &e) != STTS_OK) {
        *err = std::string("stts_create(device ") + std::to_string(dev) + "): " + stts_last_error();
        return 1;
    }
    const int B = (int)work.size();
    std::vector<int32_t> ids, offs(1, 0), sids(B), ns(B);
    std::vector<float> ls(B);
    std::vector<int16_t*> pcm(B, nullptr);
    for (int b = 0; b < B; ++b) {
        ids.insert(ids.end(), work[b]->ids.begin(), work[b]->ids.end());
        offs.push_back((int32_t)ids.size());
        sids[b] = work[b]->sid; ls[b] = work[b]->ls;
    }
    int rc = STTS_OK;
    if (noise_scale != 0.f || noise_scale_w != 0.f) {
        std::vector<float> nsv(B, noise_scale), nswv(B, noise_scale_w);
        std::vector<uint64_t> seeds(B);
        for (int b = 0; b < B; ++b) seeds[b] = work[b]->seed;
        rc = stts_set_sampling(e, B, nsv.data(), nswv.data(), seeds.data());
        if (rc != STTS_OK) *err = std::string("stts_set_sampling: ") + stts_last_error();
    }
    if (rc == STTS_OK) {
        rc = stts_infer_batch(e, B, ids.data(), offs.data(), sids.data(), ls.data(), pcm.data(), ns.data());
        if (rc != STTS_OK) *err = std::string("stts_infer_batch(device ") + std::to_string(dev) + "): " + stts_last_error();
    }
    if (rc == STTS_OK)
        for (int b = 0; b < B; ++b) {
            work[b]->pcm.assign(pcm[b], pcm[b] + ns[b]);
            stts_free(pcm[b]);
        }
    stts_destroy(e);
    return rc == STTS_OK ? 0 : 1;
}

}  // namespace

int main(int argc, char** argv) {
    Args a;
    std::vector<std::string> pos;
    for (int i = 1; i < argc; ++i) {
        const std::string s = argv[i];
        auto need = [&](const char* name) -> const char* {
            if (i + 1 >= argc) { fprintf(stderr, "%s needs a value\n", name); exit(2); }
            return argv[++i];
        };
        if (s == "--ids") a.ids = true;
        else if (s == "--per-line") a.per_line = true;
        else if (s == "--concat") a.concat = true;
        else if (s == "--dump-ids") a.dump_ids = true;
        else if (s == "--gpus") a.gpus = std::max(1, atoi(need("--gpus")));
        else if (s == "--frontend-threads") a.fe_threads = std::max(1, atoi(need("--frontend-threads")));
        else if (s == "--sid") a.sid = atoi(need("--sid"));
        else if (s == "--length-scale") a.length_scale = (float)atof(need("--length-scale"));
        else if (s == "--noise-scale") a.noise_scale = (float)atof(need("--noise-scale"));
        else if (s == "--noise-scale-w") a.noise_scale_w = (float)atof(need("--noise-scale-w"));
        else if (s == "--seed") a.seed = strtoull(need("--seed"), nullptr, 0);
        else if (s == "--selftest-wav") {
            std::vector<int16_t> tone(stts::kSampleRate);
            for (size_t n = 0; n < tone.size(); ++n) tone[n] = (int16_t)std::lrint(8000.0 * std::sin(2.0 * M_PI * 440.0 * n / stts::kSampleRate));
            const char* path = need("--selftest-wav");
            if (!stts::write_wav(path, tone.data(), tone.size())) { fprintf(stderr, "cannot write %s\n", path); return 1; }
            return 0;
        } else if (s == "-h" || s == "--help") return usage(argv[0]);
        else if (!s.empty() && s[0] == '-' && s.size() > 1 && !isdigit((unsigned char)s[1])) { fprintf(stderr, "unknown option %s\n", s.c_str()); return usage(argv[0]); }
        else pos.push_back(s);
    }
    if (pos.size() != 3) return usage(argv[0]);
    a.input = pos[0]; a.model = pos[1]; a.out = pos[2];

    std::vector<char> model;
    if (!load_file(a.model, model) || model.size() < 16) { fprintf(stderr, "cannot read model %s\n", a.model.c_str()); return 1; }
    bool ok = false;
    std::vector<std::string> lines = read_lines(a.input, &ok);
    if (!ok) { fprintf(stderr, "cannot read %s\n", a.input.c_str()); return 1; }

    // ---- header fields the CLI needs before any GPU work (host-only parse) --------------------------
    const float* hdr = reinterpret_cast<const float*>(model.data());
    const int lang_type = (int)hdr[1];
    int64_t nn_end = 0;
    {
        char* text = nullptr;
        if (stts_describe_model(hdr, (int64_t)model.size(), &text, &nn_end) != STTS_OK) {
            fprintf(stderr, "model rejected: %s\n", stts_last_error());
            return 1;
        }
        stts_free(text);
    }
    (void)lang_type;

    // ---- utterances -------------------------------------------------------------------------------
    std::vector<std::string> texts;
    if (a.ids || a.per_line) {
        for (auto& l : lines)
            if (l.find_first_not_of(" \t") != std::string::npos) texts.push_back(l);
    } else {            // reference behaviour: one utterance, lines joined with two spaces (main.cpp:90-97)
        std::string all;
        for (auto& l : lines) all += l + "  ";
        texts.push_back(all);
    }
    if (texts.empty()) { fprintf(stderr, "no input\n"); return 1; }

#ifndef STTS_WITH_REF_FRONTEND
    if (!a.ids) { fprintf(stderr, "this build has no text frontend: pass --ids <file of phoneme ids> (or build with make REF=...)\n"); return 1; }
#endif

    std::vector<Utt> utts;
    auto add = [&](const std::string& t, int sid, float ls, const std::string& out) -> bool {
        Utt u;
        u.text = t; u.sid = sid; u.ls = ls; u.out = out;
        u.seed = a.seed + utts.size();          // job index in input order: independent of the GPU partition below
        if (a.ids) {
            std::istringstream is(t);
            long v;
            while (is >> v) u.ids.push_back((int32_t)v);
            if (!is.eof()) { fprintf(stderr, "bad id line: %s\n", t.c_str()); return false; }
        }
        utts.push_back(std::move(u));
        return true;
    };

    int spk_num = 0;
    {   // speaker count (selects the reference's multi-speaker demo loop) from the host-only parse: " spk=<n>" in the summary line
        char* text = nullptr;
        int64_t e2 = 0;
        if (stts_describe_model(hdr, (int64_t)model.size(), &text, &e2) == STTS_OK && text) {
            if (const char* p = strstr(text, " spk=")) spk_num = atoi(p + 5);
            stts_free(text);
        }
    }
    const float ls_default = a.length_scale > 0 ? a.length_scale : 1.0f;
    if (!a.per_line && !a.ids && a.sid < 0 && spk_num > 20) {
        for (int sid = 10; sid < 20; ++sid)          // main.cpp:108-129
            if (!add(texts[0], sid, a.length_scale > 0 ? a.length_scale : 1.1f, numbered(a.out, "_%d.wav", sid))) return 1;
    } else {
        const int sid = std::max(0, a.sid);
        for (size_t i = 0; i < texts.size(); ++i) {
            const bool many = texts.size() > 1 && !a.concat;
            if (!add(texts[i], sid, ls_default, many ? numbered(a.out, "_%04d.wav", (int)i) : a.out)) return 1;
        }
    }

    // ---- text -> phoneme ids on the host: T threads, one frontend instance each (an instance is not re-entrant:
    //      SynthesizerTrn.cpp:338 mutates a member per call), utterances handed out through an atomic counter -----------
#ifdef STTS_WITH_REF_FRONTEND
    if (!a.ids) {
        int T = a.fe_threads > 0 ? a.fe_threads : (int)std::min<size_t>(std::max(1u, std::thread::hardware_concurrency()), 8);
        // measured (8-core host, CHS model): building one frontend 1.15 s alone, ~2 s when several build at once; 3.65 ms per
        // sentence -> an extra worker pays for itself from ~400 sentences on
        T = (int)std::max<size_t>(1, std::min<size_t>(T, (utts.size() + 383) / 384));
        std::atomic<size_t> next(0);
        std::atomic<int> failed(0);
        const bool verbose = getenv("STTS_CLI_VERBOSE") != nullptr;
        auto worker = [&] {
            const auto t0 = std::chrono::steady_clock::now();
            stts::Frontend* fe = stts::make_frontend(lang_type, const_cast<float*>(hdr), (int64_t)model.size(), nn_end);
            if (!fe) { failed = 2; return; }
            const auto t1 = std::chrono::steady_clock::now();
            size_t n = 0;
            for (size_t i; (i = next.fetch_add(1)) < utts.size(); ++n)
                if (!fe->text_to_ids(utts[i].text, utts[i].ids, utts[i].ls)) failed = 1;
            const auto t2 = std::chrono::steady_clock::now();
            delete fe;
            if (verbose)
                fprintf(stderr, "frontend worker: init %.2f s, %zu utterances in %.2f s\n", std::chrono::duration<double>(t1 - t0).count(), n,
                        std::chrono::duration<double>(t2 - t1).count());
        };
        std::vector<std::thread> ft;
        for (int t = 1; t < T; ++t) ft.emplace_back(worker);
        worker();
        for (auto& t : ft) t.join();
        if (failed == 2) { fprintf(stderr, "model has no frontend tail\n"); return 1; }
        if (failed) { fprintf(stderr, "frontend produced no ids\n"); return 1; }
    }
#endif
    for (auto& u : utts)
        if (u.ids.size() < 5) { fprintf(stderr, "utterance shorter than 5 ids (relative attention window)\n"); return 1; }
    if (a.dump_ids) {
        for (auto& u : utts) {
            for (size_t i = 0; i < u.ids.size(); ++i) printf(i ? " %d" : "%d", u.ids[i]);
            printf("\n");
        }
        return 0;
    }

    // ---- partition longest-first over the GPUs, one thread each --------------------------------------
    const int G = std::min<int>(a.gpus, (int)utts.size());
    std::vector<size_t> order(utts.size());
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](size_t x, size_t y) { return utts[x].ids.size() > utts[y].ids.size(); });
    std::vector<std::vector<Utt*>> work(G);
    std::vector<size_t> load(G, 0);
    for (size_t i : order) {
        const int g = (int)(std::min_element(load.begin(), load.end()) - load.begin());
        work[g].push_back(&utts[i]);
        load[g] += utts[i].ids.size();
    }
    std::vector<std::string> errs(G);
    std::vector<int> rcs(G, 0);
    std::vector<std::thread> th;
    for (int g = 0; g < G; ++g) th.emplace_back([&, g] { rcs[g] = run_device(g, model, work[g], a.noise_scale, a.noise_scale_w, &errs[g]); });
    for (auto& t : th) t.join();
    for (int g = 0; g < G; ++g)
        if (rcs[g]) { fprintf(stderr, "tts_b200: %s\n", errs[g].c_str()); return 1; }

    // ---- WAV files ---------------------------------------------------------------------------------
    if (a.concat && utts.size() > 1) {
        std::vector<int16_t> all;
        for (auto& u : utts) all.insert(all.end(), u.pcm.begin(), u.pcm.end());
        if (!stts::write_wav(a.out, all.data(), all.size())) { fprintf(stderr, "cannot write %s\n", a.out.c_str()); return 1; }
        printf("%s generated (%zu utterances, %zu samples)\n", a.out.c_str(), utts.size(), all.size());
    } else {
        for (auto& u : utts) {
            if (!stts::write_wav(u.out, u.pcm.data(), u.pcm.size())) { fprintf(stderr, "cannot write %s\n", u.out.c_str()); return 1; }
            printf("%s generated\n", u.out.c_str());
        }
    }
    return 0;
}
