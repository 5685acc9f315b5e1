// TEST-ONLY host build of the sweep's logarithm (bayesnetworks_b200/csrc/sweep_log.cuh) and its error against
// libquadmath's logq.  Built by tests/test_score_precision.py with g++ -ffp-contract=off (as the other host
// builds); never part of libbn_b200.so.
#include <math.h>
#include <quadmath.h>

#include "sweep_log.cuh"

extern "C" void emu_sweep_log(const double* x, double* out, long n) {
  for (long i = 0; i < n; i++) out[i] = bn::sweep_log(x[i]);
}

// |sweep_log(x) - log(x)| in units of the last place of log(x) rounded to double (the spacing of the doubles
// at |log x|); log(x) from logq (113-bit significand).  x must be a positive normal number; log(1) = 0 gives 0
// when sweep_log(1) is exactly 0, else +inf.
extern "C" void emu_sweep_log_ulp_err(const double* x, double* err, long n) {
  for (long i = 0; i < n; i++) {
    const __float128 ref = logq((__float128)x[i]);
    const double got = bn::sweep_log(x[i]);
    if (ref == 0) { err[i] = got == 0.0 ? 0.0 : INFINITY; continue; }
    const double r = (double)ref;
    int e;
    frexp(r, &e);                                   // |r| in [2^(e-1), 2^e)
    const __float128 ulp = ldexpq((__float128)1, e - 53);
    err[i] = (double)(fabsq((__float128)got - ref) / ulp);
  }
}
