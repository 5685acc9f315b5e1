// Per-chain uniform streams, generated a warp-width at a time into a ring
// buffer that the (speculative) chain step consumes by absolute stream
// position, so that rewinding after a window is just moving the read position.
//
//  BN_RNG_WH     Wichmann-Hill AS183 exactly as Bayes-networks/random4f.h:27-40:
//                three LCGs (171 mod 30269, 172 mod 30307, 170 mod 30323; the
//                reference's Schrage form 171*(ix%177) - 2*(ix/177) (+30269 if
//                negative) IS 171*ix mod 30269), combined in FP64 as
//                ix/30269.0 + iy/30307.0 + iz/30323.0 minus its floor.  An LCG
//                can jump ahead: lane l multiplies by a^(l+1) mod m, so one
//                warp instruction sequence yields 32 consecutive uniforms.
//  BN_RNG_RMT    R's default generator (R sources src/main/RNG.c: MT_genrand,
//                fixup): MT19937 + scaling by 2.3283064365386963e-10 + the
//                open-interval fix-up; the 624-word twist is done by the warp
//                in steps of 32 (read, sync, write).
//  BN_RNG_REPLAY uniforms supplied by the caller.
#pragma once

#include "bn_common.cuh"

namespace bn {

enum { RNG_WH = 0, RNG_RMT = 1, RNG_REPLAY = 2 };

constexpr int RNG_CAP = 1024;  // ring capacity (power of two)

struct RngStream {
  int kind;
  // Wichmann-Hill: state after gen_hi draws, and this lane's jump multipliers
  uint32_t x, y, z;
  uint32_t mx, my, mz;
  // R Mersenne-Twister
  uint32_t* mt;  // [624], per chain, global memory
  int mti;
  // replay
  const double* replay;
  int64_t replay_len;
  // ring
  double* ubuf;    // [RNG_CAP]
  int64_t gen_hi;  // stream positions [gen_hi - RNG_CAP, gen_hi) are in the ring
};

BN_HD uint32_t pow_mod(uint32_t a, int e, uint32_t m) {
  uint32_t r = 1;
  for (int i = 0; i < e; i++) r = (r * a) % m;
  return r;
}

BN_HD void rng_init_wh(RngStream& r, int ix, int iy, int iz, double* ubuf) {
  r.kind = RNG_WH;
  r.x = (uint32_t)ix; r.y = (uint32_t)iy; r.z = (uint32_t)iz;
  const int l = Warp::lane();
  r.mx = pow_mod(171u, l + 1, 30269u);
  r.my = pow_mod(172u, l + 1, 30307u);
  r.mz = pow_mod(170u, l + 1, 30323u);
  r.ubuf = ubuf; r.gen_hi = 0;
  r.mt = nullptr; r.mti = 0; r.replay = nullptr; r.replay_len = 0;
}

BN_HD void rng_init_rmt(RngStream& r, uint32_t* mt_state, int mti, double* ubuf) {
  r.kind = RNG_RMT;
  r.mt = mt_state; r.mti = mti;  // set.seed() leaves the position at 624 = regenerate
  r.ubuf = ubuf; r.gen_hi = 0;
  r.x = r.y = r.z = r.mx = r.my = r.mz = 0; r.replay = nullptr; r.replay_len = 0;
}

BN_HD void rng_init_replay(RngStream& r, const double* u, int64_t n, double* ubuf) {
  r.kind = RNG_REPLAY;
  r.replay = u; r.replay_len = n;
  r.ubuf = ubuf; r.gen_hi = 0;
  r.x = r.y = r.z = r.mx = r.my = r.mz = 0; r.mt = nullptr; r.mti = 0;
}

// r = ix/30269.0 + iy/30307.0 + iz/30323.0; return r - floor(r)  (random4f.h:36-40)
BN_HD double wh_combine(uint32_t xs, uint32_t ys, uint32_t zs) {
  const double v = add_rn(add_rn(div_rn((double)xs, 30269.0), div_rn((double)ys, 30307.0)),
                          div_rn((double)zs, 30323.0));
  return sub_rn(v, floor(v));
}

// MT19937 state regeneration by the whole warp.
BN_HD void rmt_twist(uint32_t* mt) {
  const int l = Warp::lane();
  for (int k0 = 0; k0 < 623; k0 += Warp::NL) {
    const int kk = k0 + l;
    uint32_t v = 0;
    if (kk < 623) {
      const uint32_t yv = (mt[kk] & 0x80000000u) | (mt[kk + 1] & 0x7fffffffu);
      const uint32_t far = (kk < 624 - 397) ? mt[kk + 397] : mt[kk + (397 - 624)];
      v = far ^ (yv >> 1) ^ ((yv & 1u) ? 0x9908b0dfu : 0u);
    }
    Warp::sync();
    if (kk < 623) mt[kk] = v;
    Warp::sync();
  }
  if (l == 0) {
    const uint32_t yv = (mt[623] & 0x80000000u) | (mt[0] & 0x7fffffffu);
    mt[623] = mt[396] ^ (yv >> 1) ^ ((yv & 1u) ? 0x9908b0dfu : 0u);
  }
  Warp::sync();
}

// Append up to Warp::NL uniforms at positions gen_hi.. ; returns how many.
BN_HD int rng_fill_chunk(RngStream& r) {
  const int l = Warp::lane();
  if (r.kind == RNG_WH) {
    const uint32_t xs = (r.x * r.mx) % 30269u;
    const uint32_t ys = (r.y * r.my) % 30307u;
    const uint32_t zs = (r.z * r.mz) % 30323u;
    r.ubuf[(r.gen_hi + l) & (RNG_CAP - 1)] = wh_combine(xs, ys, zs);
    r.x = (uint32_t)Warp::shfl((int)xs, Warp::NL - 1);
    r.y = (uint32_t)Warp::shfl((int)ys, Warp::NL - 1);
    r.z = (uint32_t)Warp::shfl((int)zs, Warp::NL - 1);
    r.gen_hi += Warp::NL;
    Warp::sync();
    return Warp::NL;
  } else if (r.kind == RNG_RMT) {
    if (r.mti >= 624) { rmt_twist(r.mt); r.mti = 0; }
    int n = 624 - r.mti;
    if (n > Warp::NL) n = Warp::NL;
    if (l < n) {
      uint32_t yv = r.mt[r.mti + l];
      yv ^= (yv >> 11);
      yv ^= (yv << 7) & 0x9d2c5680u;
      yv ^= (yv << 15) & 0xefc60000u;
      yv ^= (yv >> 18);
      double v = mul_rn((double)yv, 2.3283064365386963e-10);
      const double i2_32m1 = 2.328306437080797e-10;
      if (v <= 0.0) v = 0.5 * i2_32m1;
      else if ((1.0 - v) <= 0.0) v = 1.0 - 0.5 * i2_32m1;
      r.ubuf[(r.gen_hi + l) & (RNG_CAP - 1)] = v;
    }
    r.mti += n;
    r.gen_hi += n;
    Warp::sync();
    return n;
  } else {
    const int64_t pos = r.gen_hi + l;
    r.ubuf[pos & (RNG_CAP - 1)] = (pos < r.replay_len) ? r.replay[pos] : 0.5;
    r.gen_hi += Warp::NL;
    Warp::sync();
    return Warp::NL;
  }
}

// Make the ring cover [read_pos, read_pos + RNG_CAP - NL] at least.
BN_HD void rng_top_up(RngStream& r, int64_t read_pos) {
  while (r.gen_hi + Warp::NL <= read_pos + RNG_CAP) rng_fill_chunk(r);
}

// ---- host bookkeeping of a stream's position (the uniforms themselves come from the device) ----

// Wichmann-Hill state after n_draws uniforms from (ix, iy, iz): x a^n mod m per LCG, itself a valid
// seed triple.  A state that reduces to 0 is written as the modulus (the same residue, and a seed the
// range check accepts).
inline void wh_advance(const int* in, int64_t n_draws, int* out) {
  const uint64_t a[3] = {171u, 172u, 170u}, mod[3] = {30269u, 30307u, 30323u};
  for (int t = 0; t < 3; t++) {
    if (n_draws == 0) { out[t] = in[t]; continue; }
    uint64_t r = 1, b = a[t];
    for (int64_t e = n_draws; e > 0; e >>= 1) {
      if (e & 1) r = r * b % mod[t];
      b = b * b % mod[t];
    }
    r = r * (uint64_t)in[t] % mod[t];
    out[t] = r == 0 ? (int)mod[t] : (int)r;
  }
}

// R's MT_genrand state step (R sources, src/main/RNG.c): advance (mt, mti) by n_draws uniforms.
inline void rmt_advance(uint32_t* mt, int& mti, int64_t n_draws) {
  const int N = 624, M = 397;
  const uint32_t UPPER = 0x80000000u, LOWER = 0x7fffffffu, MAG = 0x9908b0dfu;
  while (n_draws > 0) {
    if (mti >= N) {
      int kk = 0;
      for (; kk < N - M; kk++) {
        const uint32_t y = (mt[kk] & UPPER) | (mt[kk + 1] & LOWER);
        mt[kk] = mt[kk + M] ^ (y >> 1) ^ ((y & 1u) ? MAG : 0u);
      }
      for (; kk < N - 1; kk++) {
        const uint32_t y = (mt[kk] & UPPER) | (mt[kk + 1] & LOWER);
        mt[kk] = mt[kk + (M - N)] ^ (y >> 1) ^ ((y & 1u) ? MAG : 0u);
      }
      const uint32_t y = (mt[N - 1] & UPPER) | (mt[0] & LOWER);
      mt[N - 1] = mt[M - 1] ^ (y >> 1) ^ ((y & 1u) ? MAG : 0u);
      mti = 0;
    }
    const int64_t take = n_draws < (int64_t)(N - mti) ? n_draws : (int64_t)(N - mti);
    mti += (int)take;
    n_draws -= take;
  }
}

}  // namespace bn
