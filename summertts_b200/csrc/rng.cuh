// rng.cuh — the random stream of seeded sampling (DESIGN.md §12): a counter-based Philox4x32-10 (Salmon et al., "Parallel
// random numbers: as easy as 1, 2, 3", SC'11; the round function and constants of the Random123 distribution) and the
// Box-Muller normals drawn from its words.  Host and device share this code: the C ABI restates the device's draws on the
// CPU (stts_debug_noise), and the test suite restates them in numpy.
//
// Key = the utterance's 64-bit seed (lo, hi).  Counters are positions WITHIN the utterance, so a draw does not depend on how
// utterances are batched, chunked or sharded:
//     prior  (VITS z_p = m + eps * exp(logs) * noise_scale):   (frame f, channel quad q, 0, 0) -> channels 4q .. 4q+3
//     SDP    (VITS z = eps * noise_scale_w, before nn_flip):   (token t, 0, 1, 0)              -> words 0 / 1 = eps_0(t) / eps_1(t)
#pragma once
#include <math.h>
#include <stdint.h>

#ifdef __CUDACC__
#define STTS_HD __host__ __device__ __forceinline__
#else
#define STTS_HD inline
#endif

namespace stts {

struct Philox4 { uint32_t v[4]; };

STTS_HD Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint64_t key) {
    uint32_t k0 = (uint32_t)key, k1 = (uint32_t)(key >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        c1 = (uint32_t)p1; c3 = (uint32_t)p0; c0 = n0; c2 = n2;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return Philox4{{c0, c1, c2, c3}};
}

// Two standard normals from two words: u1 = ((a >> 8) + 1) 2^-24 in (0, 1], u2 = (b >> 8) 2^-24 in [0, 1),
// r = sqrt(-2 ln u1), (r cos 2 pi u2, r sin 2 pi u2).  Float32 throughout; the device uses the accurate logf / sincospif.
STTS_HD void box_muller(uint32_t a, uint32_t b, float& n0, float& n1) {
    const float u1 = (float)((a >> 8) + 1u) * 5.9604644775390625e-8f;
    const float u2 = (float)(b >> 8) * 5.9604644775390625e-8f;
    const float r = sqrtf(-2.0f * logf(u1));
    float s, c;
#ifdef __CUDA_ARCH__
    sincospif(2.0f * u2, &s, &c);
#else
    s = (float)sin(3.14159265358979323846 * (double)(2.0f * u2));
    c = (float)cos(3.14159265358979323846 * (double)(2.0f * u2));
#endif
    n0 = r * c;
    n1 = r * s;
}

STTS_HD void philox_normals4(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint64_t key, float n[4]) {
    const Philox4 w = philox4x32_10(c0, c1, c2, c3, key);
    box_muller(w.v[0], w.v[1], n[0], n[1]);
    box_muller(w.v[2], w.v[3], n[2], n[3]);
}

enum { RNG_STREAM_PRIOR = 0, RNG_STREAM_SDP = 1 };

}  // namespace stts
