// avd_rng.cuh -- counter-based RNG for the platoon hot path (device side).
//
// Replaces the reference's global MT19937 stream (src/util.py:55-70 get_random_val,
// src/replaybuffer.py:54 np.random.choice), which is serial by construction, with Philox4x32-10
// streams addressed by (seed, id, tick, purpose).  The host restatement used by the parity tests is
// oracle/philox_np.py; the two must agree bit for bit, so every floating-point step below is a single
// correctly rounded binary32 operation (__fmul_rn/__fadd_rn/__fdiv_rn/__fsqrt_rn: never contracted
// into FMAs by nvcc).
#pragma once
#include <stdint.h>

#include "../../include/avddpg_b200.h"

namespace avd {

constexpr uint32_t kPhiloxM0 = 0xD2511F53u;
constexpr uint32_t kPhiloxM1 = 0xCD9E8D57u;
constexpr uint32_t kPhiloxW0 = 0x9E3779B9u;
constexpr uint32_t kPhiloxW1 = 0xBB67AE85u;

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(kPhiloxM0, c.x), lo0 = kPhiloxM0 * c.x;
        const uint32_t hi1 = __umulhi(kPhiloxM1, c.z), lo1 = kPhiloxM1 * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += kPhiloxW0;
        k.y += kPhiloxW1;
    }
    return c;
}

__device__ __forceinline__ uint4 rng_words(uint64_t seed, uint64_t id, uint32_t tick, uint32_t purpose) {
    return philox4x32_10(make_uint4((uint32_t)id, (uint32_t)(id >> 32), tick, purpose),
                         make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
}

// Stream key of platoon `p` (with runs: a platoon index of the whole batch) and of replay ring `ring` = m*P + p.
// Without a run table that is (seed, p) and ring id m*P + p; with one, platoon p belongs to run s = p / Pr and the key is
// (runs->seed[s], p mod Pr), ring id m*Pr + p mod Pr: the keys of the stand-alone run with random_seed = seed[s].  `runs` points
// at a kernel parameter the host entry has checked (AVD_REQUIRE_RUNS: P = runs * Pr), so s < runs.  The env kernels evaluate
// it once per platoon, the replay kernels once per Philox block (four samples of a ring).
struct StreamKey {
    uint64_t seed, id;
};

__device__ __forceinline__ StreamKey platoon_key(const avd_runs* runs, uint64_t seed, uint64_t p) {
    if (!runs) return {seed, p};
    const uint64_t pr = (uint64_t)runs->platoons_per_run, s = p / pr;
    return {runs->seed[s], p - s * pr};
}

__device__ __forceinline__ StreamKey ring_key(const avd_runs* runs, uint64_t seed, uint64_t ring) {
    if (!runs) return {seed, ring};
    const uint64_t m = ring / ((uint64_t)runs->runs * (uint64_t)runs->platoons_per_run);
    const StreamKey k = platoon_key(runs, seed, ring - m * ((uint64_t)runs->runs * (uint64_t)runs->platoons_per_run));
    return {k.seed, m * (uint64_t)runs->platoons_per_run + k.id};
}

// uint32 -> (0,1): ((x >> 9) + 0.5) * 2^-23, exact in binary32.
__device__ __forceinline__ float u01(uint32_t x) {
    return __fmul_rn(__fadd_rn(__uint2float_rn(x >> 9), 0.5f), 1.1920928955078125e-07f);
}

// ln(u), u in (0,1]: u = m 2^e, m in [sqrt(.5), sqrt(2)); ln m = 2 atanh((m-1)/(m+1)).
__device__ __forceinline__ float log_f32(float u) {
    const uint32_t bits = __float_as_uint(u);
    int e = (int)((bits >> 23) & 0xFFu) - 127;
    uint32_t mb = (bits & 0x007FFFFFu) | 0x3F800000u;
    if (mb >= 0x3FB504F3u) { mb -= 0x00800000u; e += 1; }
    const float m = __uint_as_float(mb);
    const float s = __fdiv_rn(__fadd_rn(m, -1.0f), __fadd_rn(m, 1.0f));
    const float z = __fmul_rn(s, s);
    float p = (float)(2.0 / 9.0);
    p = __fadd_rn(__fmul_rn(p, z), (float)(2.0 / 7.0));
    p = __fadd_rn(__fmul_rn(p, z), (float)(2.0 / 5.0));
    p = __fadd_rn(__fmul_rn(p, z), (float)(2.0 / 3.0));
    p = __fadd_rn(__fmul_rn(p, z), 2.0f);
    return __fadd_rn(__fmul_rn(__int2float_rn(e), (float)0.6931471805599453), __fmul_rn(s, p));
}

// (sin, cos)(2 pi v), v in (0,1): quadrant reduction is exact, then odd/even polynomials on [-pi/4, pi/4].
__device__ __forceinline__ void sincos_2pi_f32(float v, float& s_out, float& c_out) {
    const float t = __fmul_rn(v, 4.0f);
    const float k = floorf(__fadd_rn(t, 0.5f));
    const float f = __fadd_rn(t, -k);
    const float x = __fmul_rn(f, (float)1.5707963267948966);
    const float z = __fmul_rn(x, x);
    float ps = (float)(1.0 / 362880.0);
    ps = __fadd_rn(__fmul_rn(ps, z), (float)(-1.0 / 5040.0));
    ps = __fadd_rn(__fmul_rn(ps, z), (float)(1.0 / 120.0));
    ps = __fadd_rn(__fmul_rn(ps, z), (float)(-1.0 / 6.0));
    ps = __fadd_rn(__fmul_rn(ps, z), 1.0f);
    const float sx = __fmul_rn(x, ps);
    float pc = (float)(-1.0 / 3628800.0);
    pc = __fadd_rn(__fmul_rn(pc, z), (float)(1.0 / 40320.0));
    pc = __fadd_rn(__fmul_rn(pc, z), (float)(-1.0 / 720.0));
    pc = __fadd_rn(__fmul_rn(pc, z), (float)(1.0 / 24.0));
    pc = __fadd_rn(__fmul_rn(pc, z), -0.5f);
    const float cx = __fadd_rn(__fmul_rn(pc, z), 1.0f);
    const int q = ((int)k) & 3;
    s_out = (q == 0) ? sx : (q == 1) ? cx : (q == 2) ? -sx : -cx;
    c_out = (q == 0) ? cx : (q == 1) ? -sx : (q == 2) ? -cx : sx;
}

// Box-Muller: (z0, z1) = sqrt(-2 ln u1) * (cos, sin)(2 pi u2)
__device__ __forceinline__ void normal_pair(uint32_t wa, uint32_t wb, float& z0, float& z1) {
    const float r = __fsqrt_rn(__fmul_rn(-2.0f, log_f32(u01(wa))));
    float s, c;
    sincos_2pi_f32(u01(wb), s, c);
    z0 = __fmul_rn(r, c);
    z1 = __fmul_rn(r, s);
}

__device__ __forceinline__ float uniform_sym(uint32_t w, float bound) {
    return __fmul_rn(__fadd_rn(__fmul_rn(u01(w), 2.0f), -1.0f), bound);
}

// uniform integer in [0, n): 64-bit multiply-shift
__device__ __forceinline__ int64_t index_from_word(uint32_t w, uint64_t n) {
    return (int64_t)(((uint64_t)w * n) >> 32);
}

// One reset/exog style draw: N(0, bound) or U(-bound, bound) from word pair (wa, wb) (normal uses both).
__device__ __forceinline__ float draw_first(uint32_t wa, uint32_t wb, float bound, bool uniform) {
    if (uniform) return uniform_sym(wa, bound);
    float z0, z1;
    normal_pair(wa, wb, z0, z1);
    return __fmul_rn(z0, bound);
}

}  // namespace avd
