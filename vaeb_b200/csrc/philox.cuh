// Philox4x32-10 counter-based RNG + Box-Muller: the on-device replacement for the
// reference's host-side `srng.normal(mu.shape)` (VAEB.py:42,158).  The counter layout is
// restated on the CPU in oracle/vaeb_oracle.py:philox_normal (uint32 outputs bit-exact).
#pragma once
#include <cstdint>

#define VAEB_STREAM_TRAIN 0u
#define VAEB_STREAM_EVAL 1u
#define VAEB_STREAM_IS 2u
#define VAEB_STREAM_ZETA 3u
#define VAEB_STREAM_RECON 4u
#define VAEB_STREAM_SAMPLE 5u   // vaeb_sample: z ~ N(0, I) (sample 0) and the draw of x from p(x|z) (sample 1)

__host__ __device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                       uint32_t k0, uint32_t k1, uint32_t out[4]) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint64_t p0 = 0xD2511F53ull * (uint64_t)c0;
    const uint64_t p1 = 0xCD9E8D57ull * (uint64_t)c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
    const uint32_t n1 = (uint32_t)p1;
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    const uint32_t n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// Four N(0,1) draws of group `g` (flat elements 4g..4g+3) of (stream, step, sample).
__device__ __forceinline__ void philox_normal4(uint64_t seed, uint32_t stream, uint32_t step, uint32_t sample,
                                               uint64_t g, float n[4]) {
  uint32_t r[4];
  philox4x32_10((uint32_t)g, ((uint32_t)(g >> 32) & 0x00FFFFFFu) | ((stream & 0xFFu) << 24), sample, step,
                (uint32_t)seed, (uint32_t)(seed >> 32), r);
  const float u0 = ((float)(r[0] >> 8) + 0.5f) * 5.9604644775390625e-8f;  // 2^-24
  const float u1 = ((float)(r[1] >> 8) + 0.5f) * 5.9604644775390625e-8f;
  const float u2 = ((float)(r[2] >> 8) + 0.5f) * 5.9604644775390625e-8f;
  const float u3 = ((float)(r[3] >> 8) + 0.5f) * 5.9604644775390625e-8f;
  const float rad0 = sqrtf(-2.0f * logf(u0));
  const float rad1 = sqrtf(-2.0f * logf(u2));
  float s0, c0, s1, c1;
  sincospif(2.0f * u1, &s0, &c0);   // exact argument reduction: no slow path, small code
  sincospif(2.0f * u3, &s1, &c1);
  n[0] = rad0 * c0; n[1] = rad0 * s0; n[2] = rad1 * c1; n[3] = rad1 * s1;
}

// One U(0,1) draw, flat element e: the uniform philox_normal4 makes of output e % 4 of group e / 4, the same 24-bit
// mapping ((r >> 8) + 0.5) * 2^-24, so never 0 or 1.  Restated on the CPU in tests/sample_oracle.py.
__device__ __forceinline__ float philox_uniform1(uint64_t seed, uint32_t stream, uint32_t step, uint32_t sample,
                                                 uint64_t e) {
  uint32_t r[4];
  const uint64_t g = e >> 2;
  philox4x32_10((uint32_t)g, ((uint32_t)(g >> 32) & 0x00FFFFFFu) | ((stream & 0xFFu) << 24), sample, step,
                (uint32_t)seed, (uint32_t)(seed >> 32), r);
  const uint32_t q = (uint32_t)e & 3u;
  const uint32_t rv = q == 0 ? r[0] : (q == 1 ? r[1] : (q == 2 ? r[2] : r[3]));
  return ((float)(rv >> 8) + 0.5f) * 5.9604644775390625e-8f;  // 2^-24
}

// One draw: flat element e.
__device__ __forceinline__ float philox_normal1(uint64_t seed, uint32_t stream, uint32_t step, uint32_t sample,
                                                uint64_t e) {
  float n[4];
  philox_normal4(seed, stream, step, sample, e >> 2, n);
  const uint32_t q = (uint32_t)e & 3u;
  return q == 0 ? n[0] : (q == 1 ? n[1] : (q == 2 ? n[2] : n[3]));
}

// The same draw as philox_normal1 without the three it does not use (one logarithm, one sincospi).
__device__ __forceinline__ float philox_normal_only(uint64_t seed, uint32_t stream, uint32_t step, uint32_t sample,
                                                    uint64_t e) {
  uint32_t r[4];
  const uint64_t g = e >> 2;
  philox4x32_10((uint32_t)g, ((uint32_t)(g >> 32) & 0x00FFFFFFu) | ((stream & 0xFFu) << 24), sample, step,
                (uint32_t)seed, (uint32_t)(seed >> 32), r);
  const uint32_t q = (uint32_t)e & 3u;
  const uint32_t ra = (q & 2u) ? r[2] : r[0], rb = (q & 2u) ? r[3] : r[1];
  const float ua = ((float)(ra >> 8) + 0.5f) * 5.9604644775390625e-8f;  // 2^-24
  const float ub = ((float)(rb >> 8) + 0.5f) * 5.9604644775390625e-8f;
  const float rad = sqrtf(-2.0f * logf(ua));
  float sn, cs;
  sincospif(2.0f * ub, &sn, &cs);
  return rad * ((q & 1u) ? sn : cs);
}
