// Natural logarithm of the all-proposal sweep (kernels.cu, sweep_kernel's addition loop).  A header of its
// own so that the tests can evaluate the same function on the host (tests/emu/sweep_log_host.cpp) and
// compare it with an extended-precision logarithm and with the device's bits.
#pragma once

#include <string.h>

#include "bn_common.cuh"

namespace bn {

// One per proposal; the kernel is bound by instruction issue and libdevice's log is ~100 instructions.
// x = 2^e m with m in [sqrt(1/2), sqrt(2)), log m = 2 atanh(s), s = (m - 1) / (m + 1), |s| <= 0.172, odd
// series to s^19 (truncation 2.4e-17 relative), the reciprocal by __drcp_rn.  ~40 instructions; error below
// 2.5 ulp of the result (the worst input found, x = 0.999059206, gives 2.41 ulp; tests/test_score_precision.py
// checks the bound on 2.2e6 inputs against logq); the sweep's parity bar against the oracle is 1e-9 relative.
// The argument is a positive normal number at the call site (RSS above its floor times a finite scale);
// anything else gives NaN.
// On the host (tests only) the reciprocal is 1.0 / x, which rounds to nearest as __drcp_rn does, so with
// contraction off both builds compute the same bits.
BN_HD double sweep_log(double x) {
#if defined(__CUDA_ARCH__)
  int hi = __double2hiint(x);
  const int lo = __double2loint(x);
  if ((unsigned)(hi - 0x00100000) >= 0x7fe00000u) return __longlong_as_double(0x7ff8000000000000ll);  // (not a positive normal number)
#else
  unsigned long long bits;
  memcpy(&bits, &x, 8);
  int hi = (int)(bits >> 32);
  const int lo = (int)(unsigned)bits;
  if ((unsigned)(hi - 0x00100000) >= 0x7fe00000u) return NAN;  // (not a positive normal number)
#endif
  int e = (hi >> 20) - 1023;
  hi = (hi & 0x000fffff) | 0x3ff00000;
  if (hi >= 0x3ff6a09e) { hi -= 0x00100000; e++; }  // m >= ~sqrt(2): halve
#if defined(__CUDA_ARCH__)
  const double m = __hiloint2double(hi, lo);
  const double f = m - 1.0;
  const double s = f * __drcp_rn(2.0 + f);
#else
  const unsigned long long mb = ((unsigned long long)(unsigned)hi << 32) | (unsigned)lo;
  double m;
  memcpy(&m, &mb, 8);
  const double f = m - 1.0;
  const double s = f * (1.0 / (2.0 + f));
#endif
  const double s2 = s * s;
  double p = 2.0 / 19.0;
  p = fma(p, s2, 2.0 / 17.0);
  p = fma(p, s2, 2.0 / 15.0);
  p = fma(p, s2, 2.0 / 13.0);
  p = fma(p, s2, 2.0 / 11.0);
  p = fma(p, s2, 2.0 / 9.0);
  p = fma(p, s2, 2.0 / 7.0);
  p = fma(p, s2, 2.0 / 5.0);
  p = fma(p, s2, 2.0 / 3.0);
  const double de = (double)e;
  // e ln2 + 2s + s^3 p, ln2 split so that e * ln2_hi is exact
  return fma(de, 6.93147180369123816490e-01, fma(s * s2, p, fma(de, 1.90821492927058770002e-10, 2.0 * s)));
}

}  // namespace bn
