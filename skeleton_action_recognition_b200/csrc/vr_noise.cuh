// Receiver noise (VR_FLAG_NOISE, DESIGN §3i): the complex Gaussian sample xi[n, t] that the forward launches add to the
// baseband z[n, t] once z is complete, before the iq store, the STFT or the fused resize read it.
//
//   Philox4x32-10 (Random123 / cuRAND constants), key (seed lo32, seed hi32), counter (t lo32, t hi32, n lo32, n hi32)
//       -> w0..w3
//   u1 = ((w1 2^32 + w0) >> 11 + 1) 2^-53  in (0, 1]         u2 = ((w3 2^32 + w2) >> 11) 2^-53  in [0, 1)
//   rho = sqrt(-2 log u1), (s, c) = sincospi(2 u2), in float64
//   xi  = (fl32(sigma sqrt(1/2) rho c), fl32(sigma sqrt(1/2) rho s))      E|xi|^2 = sigma^2
//
// A counter-based generator: xi depends on (seed, n, t) only, so it is the same bits whichever job, team, CTA or
// schedule synthesises the step, in the halo two jobs of one sequence share, and on any SM count.
#pragma once
#include <cstdint>

namespace vr {

struct NoiseParams {
    const float* std;                 // N noise standard deviations, one per output (I/Q units), or nullptr: no noise
    const unsigned long long* seed;   // one 64-bit seed, read on the device (a graph replays with the tensor's value)
};

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint32_t k0, uint32_t k1) {
    #pragma unroll
    for (int r = 0; r < 10; ++r) {
        if (r) { k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
        const uint32_t lo0 = 0xD2511F53u * c.x, hi0 = __umulhi(0xD2511F53u, c.x);
        const uint32_t lo1 = 0xCD9E8D57u * c.z, hi1 = __umulhi(0xCD9E8D57u, c.z);
        c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
    }
    return c;
}

// xi[n, t] for noise standard deviation sigma (the definition above)
__device__ __forceinline__ float2 receiver_noise(unsigned long long seed, unsigned long long n, unsigned long long t,
                                                 float sigma) {
    const uint4 w = philox4x32_10(make_uint4((uint32_t)t, (uint32_t)(t >> 32), (uint32_t)n, (uint32_t)(n >> 32)),
                                  (uint32_t)seed, (uint32_t)(seed >> 32));
    const double u1 = (double)(((((unsigned long long)w.y << 32) | w.x) >> 11) + 1) * 0x1p-53;
    const double u2 = (double)((((unsigned long long)w.w << 32) | w.z) >> 11) * 0x1p-53;
    double s, c;
    sincospi(2.0 * u2, &s, &c);
    const double a = (double)sigma * 0.70710678118654752440 * sqrt(-2.0 * log(u1));
    return make_float2(__double2float_rn(a * c), __double2float_rn(a * s));
}

// z[i] += xi[n, lo + i] for i in [0, cnt), i strided over the threads [tid, nthreads) that run the pass.  The caller
// makes the pass uniform over its CTA / team and surrounds it with the barriers that order it against the writes that
// complete z and the reads that follow.
__device__ __noinline__ void add_receiver_noise(float2* z, long long lo, int cnt, long long n, NoiseParams q,
                                                int tid, int nthreads) {
    const float sigma = q.std[n];
    const unsigned long long seed = *q.seed;
    for (int i = tid; i < cnt; i += nthreads) {
        const float2 e = receiver_noise(seed, (unsigned long long)n, (unsigned long long)(lo + i), sigma);
        const float2 v = z[i];
        z[i] = make_float2(v.x + e.x, v.y + e.y);
    }
}

}  // namespace vr
