// tests/native/walk_host.cpp — host build of swift3drenderer_b200/csrc/walk.cuh for the CPU unit test.
// Compares walk_jump() with n true sequential binary32 additions.
#include "../../swift3drenderer_b200/csrc/walk.cuh"
#include <math.h>

extern "C" {

float walk_jump_host(float s, float d, uint32_t n) { return s3r::walk_jump(s, d, n); }

float walk_seq_host(float s, float d, uint32_t n) {
    volatile float w = s;
    for (uint32_t i = 0; i < n; i++) { w = w + d; }
    return w;
}

static uint64_t rng_state = 0x9E3779B97F4A7C15ull;
static uint32_t rnd() {
    rng_state ^= rng_state << 13; rng_state ^= rng_state >> 7; rng_state ^= rng_state << 17;
    return (uint32_t)(rng_state >> 16);
}

// mode 0: barycentric-like (s in [-2,2], |d| ~ 1/extent, extents up to 4000 or, for walks over 4096, 65535); mode 1: random bit patterns with nearby
// exponents; mode 2: ties (d = (k + 1/2) ulp(s)); mode 3: subnormal / tiny; mode 4: binade edges with sparse deltas; returns mismatches.
uint64_t walk_fuzz(uint32_t mode, uint64_t trials, uint32_t max_n, uint64_t seed, float *bad) {
    rng_state = seed * 0x9E3779B97F4A7C15ull + 12345;
    uint64_t mism = 0;
    for (uint64_t t = 0; t < trials; t++) {
        float s, d;
        uint32_t n = 1 + rnd() % max_n;
        if (mode == 0) {
            s = ((int32_t)rnd() / 2147483648.0f) * 2.0f;
            float ext = 1.0f + (rnd() % (max_n > 4096 ? 65535u : 4000u));   // box extents up to the longest walk
            d = ((int32_t)rnd() / 2147483648.0f) * 3.0f / ext;
        } else if (mode == 1) {
            uint32_t e = 100 + rnd() % 56;
            uint32_t bs = (rnd() & 0x807FFFFFu) | (e << 23);
            int32_t de = (int32_t)(rnd() % 40) - 30;
            uint32_t bd = (rnd() & 0x807FFFFFu) | ((uint32_t)((int32_t)e + de) << 23);
            s = s3r::u2f(bs); d = s3r::u2f(bd);
        } else if (mode == 2) {
            uint32_t e = 110 + rnd() % 30;
            uint32_t bs = (rnd() & 0x807FFFFFu) | (e << 23);
            s = s3r::u2f(bs);
            float ulp = ldexpf(1.0f, (int)e - 127 - 23);
            float k = (float)(rnd() % 9);
            d = (k + 0.5f) * ulp * ((rnd() & 1) ? 1.f : -1.f);
            if (rnd() & 1) { d *= 0.5f; }
        } else if (mode == 4) {
            // binade edges and sparse deltas: s within a few ulps of a power of two (either side, either sign), d with
            // few significant bits at every exponent distance down to full absorption (ties in every binade)
            uint32_t e = 90 + rnd() % 60;
            uint32_t edge = (rnd() & 1) ? (rnd() % 5) : (0x7FFFFFu - rnd() % 5);
            uint32_t bs = (rnd() & 0x80000000u) | (e << 23) | edge;
            uint32_t keep = 1 + rnd() % 4;
            uint32_t mask = ~((1u << (23 - keep)) - 1u) & 0x7FFFFFu;
            uint32_t bd = (rnd() & 0x80000000u) | ((e - rnd() % 30) << 23) | (rnd() & mask);
            s = s3r::u2f(bs); d = s3r::u2f(bd);
        } else {
            uint32_t bs = (rnd() & 0x80FFFFFFu) & 0x81FFFFFFu;
            uint32_t bd = (rnd() & 0x807FFFFFu) | ((rnd() % 3) << 23);
            s = s3r::u2f(bs); d = s3r::u2f(bd);
        }
        float a = walk_jump_host(s, d, n), b = walk_seq_host(s, d, n);
        if (s3r::f2u(a) != s3r::f2u(b) && !(a != a && b != b)) {
            if (mism == 0 && bad) { bad[0] = s; bad[1] = d; bad[2] = (float)n; bad[3] = a; bad[4] = b; }
            mism++;
        }
    }
    return mism;
}
}
