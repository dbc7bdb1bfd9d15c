// philox.cuh -- the counter-based generator of seeded MCMC runs (bart_mcmc_run_seeded): Philox4x64-10
// (Salmon, Moraes, Dror & Shaw 2011) with Random123's round constants and key schedule, the
// generator numpy ships as np.random.Philox (numpy's random_raw(4) with counter c returns the block
// of counter c + 1).  tests/philox_oracle.py restates everything here in numpy.
//
// Every retrieval has its own 128-bit key (bart_mcmc_seed).  One draw is one block; its 256-bit
// counter says what the draw is for:
//   c0 = element | attempt << 32   element: free parameter (support, usnooker), else 0;
//                                  attempt: redraws of a polar-method pair or of i2 == i1
//   c1 = chain (within the retrieval)
//   c2 = global iteration: nold + generations run so far (what MC3's burn-in and the snooker
//        thinning schedule count)
//   c3 = purpose (DrawPurpose)
// so a draw is a pure function of (key, purpose, iteration, chain, element): independent of the
// ensemble size, of the retrieval's place in it, of the rank count and of how a run is cut into
// calls.  Transforms of a 64-bit word x (numpy's conversions):
//   uniform [0, 1)       (x >> 11) 2^-53                                 word 0
//   randint(lo, hi)      lo + umulhi(x, hi - lo), hi exclusive           word 0
//   normal               polar method on u = 2 U(w0) - 1, v = 2 U(w1) - 1: s = u u + v v (separately
//                        rounded, so acceptance is reproducible), accepted when 0 < s < 1, else the
//                        next attempt; z = u sqrt(-2 log s / s)
#pragma once

namespace bart {

enum DrawPurpose {
  DRAW_SUPPORT = 1, DRAW_R1 = 2, DRAW_R2 = 3, DRAW_UNIF = 4, DRAW_UGAMMA = 5,
  DRAW_I1 = 6, DRAW_I2 = 7, DRAW_IZ = 8, DRAW_IC = 9, DRAW_USN = 10
};

struct Philox4 { unsigned long long x[4]; };

__device__ __forceinline__ Philox4 philox4x64_10(Philox4 c, unsigned long long k0, unsigned long long k1) {
  const unsigned long long M0 = 0xD2E7470EE14C6C93ull, M1 = 0xCA5A826395121157ull;
  const unsigned long long W0 = 0x9E3779B97F4A7C15ull, W1 = 0xBB67AE8584CAA73Bull;
#pragma unroll
  for (int r = 0; r < 10; r++) {
    const unsigned long long hi0 = __umul64hi(M0, c.x[0]), lo0 = M0 * c.x[0];
    const unsigned long long hi1 = __umul64hi(M1, c.x[2]), lo1 = M1 * c.x[2];
    Philox4 n;
    n.x[0] = hi1 ^ c.x[1] ^ k0; n.x[1] = lo1;
    n.x[2] = hi0 ^ c.x[3] ^ k1; n.x[3] = lo0;
    c = n;
    k0 += W0; k1 += W1;
  }
  return c;
}

// the block of (purpose, iteration, chain, element, attempt) under key (k0, k1)
__device__ __forceinline__ Philox4 draw_block(unsigned long long k0, unsigned long long k1, int purpose,
                                              long long it, int chain, int element, int attempt) {
  Philox4 c;
  c.x[0] = (unsigned long long)(unsigned)element | (unsigned long long)(unsigned)attempt << 32;
  c.x[1] = (unsigned long long)(unsigned)chain;
  c.x[2] = (unsigned long long)it;
  c.x[3] = (unsigned long long)purpose;
  return philox4x64_10(c, k0, k1);
}

__device__ __forceinline__ double u01(unsigned long long x) { return (double)(x >> 11) * 0x1.0p-53; }
__device__ __forceinline__ int randint(unsigned long long x, long long lo, long long hi) {
  return (int)(lo + (long long)__umul64hi(x, (unsigned long long)(hi - lo)));
}

}  // namespace bart
