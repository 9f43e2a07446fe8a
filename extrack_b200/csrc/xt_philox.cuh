// Counter-based Philox4x32-10 (Salmon, Moraes, Dror, Shaw, "Parallel random numbers: as easy as 1, 2, 3", SC 2011),
// written out so that a host implementation (oracle/sample_oracle.py) reproduces every word.  Known answers (Random123):
//   counter {0, 0, 0, 0}, key {0, 0}                          -> 6627e8d5 e169c58d bc57ac4c 9b00dbd8
//   counter all ones, key all ones                            -> 408f276d 41c83b0e a20bc7c6 6d5451fd
//   counter {243f6a88 85a308d3 13198a2e 03707344}, key {a4093822 299f31d0} -> d16cfe09 94fdcceb 5001e420 24126ea1
#pragma once
#include <stdint.h>

struct XtPhilox4 {
  uint32_t x[4];
};

__host__ __device__ inline XtPhilox4 xt_philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                                      uint32_t k1) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    if (r) {
      k0 += W0;
      k1 += W1;
    }
    const uint64_t p0 = (uint64_t)M0 * c0, p1 = (uint64_t)M1 * c2;
    const uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0, hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
    c0 = hi1 ^ c1 ^ k0;
    c1 = lo1;
    c2 = hi0 ^ c3 ^ k1;
    c3 = lo0;
  }
  return XtPhilox4{{c0, c1, c2, c3}};
}

// Uniform double in [0, 1) from the first two output words: the top 53 bits of (x0 << 32 | x1), times 2^-53
__host__ __device__ inline double xt_philox_u01(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint64_t seed) {
  const XtPhilox4 o = xt_philox4x32_10(c0, c1, c2, c3, (uint32_t)seed, (uint32_t)(seed >> 32));
  return (double)((((uint64_t)o.x[0] << 32) | o.x[1]) >> 11) * 0x1.0p-53;
}
