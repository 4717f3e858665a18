// Device restatement of the three libm functions behind the reference's score arithmetic
//   util/ctc_loss_util.h:39-40                LogSumExp = max + log1pf(expf(min - max))
//   util/ctc_ext_beam_search_decoder.h:76,78  Eigen::numext::exp / log  (-> expf / logf)
// performing, operation for operation, what glibc 2.39 executes on an FMA-capable x86-64 host
// (Arm Optimized Routines expf/logf in double precision with every product-sum fused; fdlibm
// log1pf in single precision without contraction). All operations use explicit round-to-nearest
// intrinsics so nvcc can neither contract nor re-associate them; the results are bit-identical to
// the host libm, which makes device scores bit-identical to the reference's. tests/test_gpu_exact_math.py
// checks these device functions against glibc on every float of the domains below (and LogSumExp on
// every float difference in [-104, 0]); the double functions further down at every reduction-cell and
// table edge plus 2^27 random arguments each (DESIGN.md "Numerics").
//
// Domains used by the decoder: expf(x <= 0 or -inf), log1pf(0 <= x <= 1), logf(1 <= x < 2^16).
#pragma once
#include <cstdint>

namespace ctcx {

// bits of 2^(i/32) - (i << 47)
static __device__ __constant__ unsigned long long kExp2fTabConst[32] = {
    0x3ff0000000000000ull, 0x3fefd9b0d3158574ull, 0x3fefb5586cf9890full, 0x3fef9301d0125b51ull,
    0x3fef72b83c7d517bull, 0x3fef54873168b9aaull, 0x3fef387a6e756238ull, 0x3fef1e9df51fdee1ull,
    0x3fef06fe0a31b715ull, 0x3feef1a7373aa9cbull, 0x3feedea64c123422ull, 0x3feece086061892dull,
    0x3feebfdad5362a27ull, 0x3feeb42b569d4f82ull, 0x3feeab07dd485429ull, 0x3feea47eb03a5585ull,
    0x3feea09e667f3bcdull, 0x3fee9f75e8ec5f74ull, 0x3feea11473eb0187ull, 0x3feea589994cce13ull,
    0x3feeace5422aa0dbull, 0x3feeb737b0cdc5e5ull, 0x3feec49182a3f090ull, 0x3feed503b23e255dull,
    0x3feee89f995ad3adull, 0x3feeff76f2fb5e47ull, 0x3fef199bdd85529cull, 0x3fef3720dcef9069ull,
    0x3fef5818dcfba487ull, 0x3fef7c97337b9b5full, 0x3fefa4afa2a490daull, 0x3fefd0765b6e4540ull,
};

// (1/c, log c) pairs of the logf table
static __device__ __constant__ unsigned long long kLogfTabConst[32] = {
    0x3ff661ec79f8f3beull, 0xbfd57bf7808caadeull, 0x3ff571ed4aaf883dull, 0xbfd2bef0a7c06ddbull,
    0x3ff49539f0f010b0ull, 0xbfd01eae7f513a67ull, 0x3ff3c995b0b80385ull, 0xbfcb31d8a68224e9ull,
    0x3ff30d190c8864a5ull, 0xbfc6574f0ac07758ull, 0x3ff25e227b0b8ea0ull, 0xbfc1aa2bc79c8100ull,
    0x3ff1bb4a4a1a343full, 0xbfba4e76ce8c0e5eull, 0x3ff12358f08ae5baull, 0xbfb1973c5a611cccull,
    0x3ff0953f419900a7ull, 0xbfa252f438e10c1eull, 0x3ff0000000000000ull, 0x0000000000000000ull,
    0x3fee608cfd9a47acull, 0x3faaa5aa5df25984ull, 0x3feca4b31f026aa0ull, 0x3fbc5e53aa362eb4ull,
    0x3feb2036576afce6ull, 0x3fc526e57720db08ull, 0x3fe9c2d163a1aa2dull, 0x3fcbc2860d224770ull,
    0x3fe886e6037841edull, 0x3fd1058bc8a07ee1ull, 0x3fe767dcf5534862ull, 0x3fd4043057b6ee09ull,
};

// Copies the exp2f table into shared memory (lanes index it with divergent subscripts; constant
// memory would serialise those).
__device__ __forceinline__ void LoadExpTable(unsigned long long* smem_tab32, int tid, int nthreads) {
  for (int i = tid; i < 32; i += nthreads) smem_tab32[i] = kExp2fTabConst[i];
}

// expf for x <= 0 (or -inf). `tab` = the 32-entry table (shared or constant memory).
__device__ __forceinline__ float ExpfExact(float x, const unsigned long long* tab) {
  if (x < __uint_as_float(0xc2cff1b4u)) return 0.0f;  // x < -0x1.9fe368p6f: underflow to 0
  const double kInvLn2N = __longlong_as_double(0x40471547652b82feull);
  const double kShift = __longlong_as_double(0x4338000000000000ull);
  const double kC0 = __longlong_as_double(0x3ebc6af84b912394ull);
  const double kC1 = __longlong_as_double(0x3f2ebfce50fac4f3ull);
  const double kC2 = __longlong_as_double(0x3f962e42ff0c52d6ull);
  const double xd = (double)x;
  double z = __dmul_rn(kInvLn2N, xd);
  double kd = __dadd_rn(z, kShift);
  const unsigned long long ki = (unsigned long long)__double_as_longlong(kd);
  kd = __dsub_rn(kd, kShift);
  const double r = __fma_rn(kInvLn2N, xd, -kd);
  const unsigned long long t = tab[ki & 31ull] + (ki << 47);
  const double s = __longlong_as_double((long long)t);
  z = __fma_rn(kC0, r, kC1);
  const double r2 = __dmul_rn(r, r);
  double y = __fma_rn(kC2, r, 1.0);
  y = __fma_rn(z, r2, y);
  y = __dmul_rn(y, s);
  return __double2float_rn(y);
}

// log1pf for 0 <= x <= 1 (fdlibm float algorithm).
__device__ __forceinline__ float Log1pfExact(float x) {
  const float ln2_hi = __uint_as_float(0x3f317180u), ln2_lo = __uint_as_float(0x3717f7d1u);
  const float Lp1 = __uint_as_float(0x3f2aaaabu), Lp2 = __uint_as_float(0x3ecccccdu),
              Lp3 = __uint_as_float(0x3e924925u), Lp4 = __uint_as_float(0x3e638e29u),
              Lp5 = __uint_as_float(0x3e3a3325u), Lp6 = __uint_as_float(0x3e1cd04fu),
              Lp7 = __uint_as_float(0x3e178897u);
  float f = 0.f, c = 0.f;
  int hx = __float_as_int(x);
  const int ax = hx & 0x7fffffff;
  int k = 1, hu = 0;
  if (hx < 0x3ed413d7) {      // x < 0.41422
    if (ax < 0x31000000) {    // |x| < 2**-29
      if (ax < 0x24800000) return x;
      return __fsub_rn(x, __fmul_rn(__fmul_rn(x, x), 0.5f));
    }
    if (hx > 0 || hx <= (int)0xbe95f61f) {
      k = 0;
      f = x;
      hu = 1;
    }
  }
  if (k != 0) {
    float u = __fadd_rn(1.0f, x);
    hu = __float_as_int(u);
    k = (hu >> 23) - 127;
    c = (k > 0) ? __fsub_rn(1.0f, __fsub_rn(u, x)) : __fsub_rn(x, __fsub_rn(u, 1.0f));
    c = __fdiv_rn(c, u);
    hu &= 0x007fffff;
    if (hu < 0x3504f7) {
      u = __int_as_float(hu | 0x3f800000);
    } else {
      k += 1;
      u = __int_as_float(hu | 0x3f000000);
      hu = (0x00800000 - hu) >> 2;
    }
    f = __fsub_rn(u, 1.0f);
  }
  const float hfsq = __fmul_rn(__fmul_rn(0.5f, f), f);
  const float kf = (float)k;
  if (hu == 0) {  // |f| < 2**-20
    if (f == 0.0f) {
      if (k == 0) return 0.0f;
      c = __fadd_rn(c, __fmul_rn(kf, ln2_lo));
      return __fadd_rn(__fmul_rn(kf, ln2_hi), c);
    }
    const float R0 = __fmul_rn(hfsq, __fsub_rn(1.0f, __fmul_rn(__uint_as_float(0x3f2aaaabu), f)));
    if (k == 0) return __fsub_rn(f, R0);
    return __fsub_rn(__fmul_rn(kf, ln2_hi),
                     __fsub_rn(__fsub_rn(R0, __fadd_rn(__fmul_rn(kf, ln2_lo), c)), f));
  }
  const float s = __fdiv_rn(f, __fadd_rn(2.0f, f));
  const float z = __fmul_rn(s, s);
  float R = __fadd_rn(Lp6, __fmul_rn(z, Lp7));
  R = __fadd_rn(Lp5, __fmul_rn(z, R));
  R = __fadd_rn(Lp4, __fmul_rn(z, R));
  R = __fadd_rn(Lp3, __fmul_rn(z, R));
  R = __fadd_rn(Lp2, __fmul_rn(z, R));
  R = __fadd_rn(Lp1, __fmul_rn(z, R));
  R = __fmul_rn(z, R);
  const float shr = __fmul_rn(s, __fadd_rn(hfsq, R));
  if (k == 0) return __fsub_rn(f, __fsub_rn(hfsq, shr));
  return __fsub_rn(
      __fmul_rn(kf, ln2_hi),
      __fsub_rn(__fsub_rn(hfsq, __fadd_rn(shr, __fadd_rn(__fmul_rn(kf, ln2_lo), c))), f));
}

// logf for 1 <= x < 2^16.
__device__ __forceinline__ float LogfExact(float x) {
  const double kLn2 = __longlong_as_double(0x3fe62e42fefa39efull);
  const double kA0 = __longlong_as_double((long long)0xbfd00ea348b88334ull);
  const double kA1 = __longlong_as_double(0x3fd5575b0be00b6aull);
  const double kA2 = __longlong_as_double((long long)0xbfdffffef20a4123ull);
  const unsigned ix = __float_as_uint(x);
  if (ix == 0x3f800000u) return 0.0f;
  const unsigned tmp = ix - 0x3f330000u;
  const int i = (int)((tmp >> 19) & 15u);
  const int k = (int)tmp >> 23;
  const unsigned iz = ix - (tmp & 0xff800000u);
  const double invc = __longlong_as_double((long long)kLogfTabConst[2 * i]);
  const double logc = __longlong_as_double((long long)kLogfTabConst[2 * i + 1]);
  const double z = (double)__uint_as_float(iz);
  const double r = __fma_rn(z, invc, -1.0);
  const double y0 = __fma_rn((double)k, kLn2, logc);
  const double r2 = __dmul_rn(r, r);
  double y = __fma_rn(kA1, r, kA2);
  y = __fma_rn(kA0, r2, y);
  y = __fma_rn(y, r2, __dadd_rn(y0, r));
  return __double2float_rn(y);
}

// util/ctc_loss_util.h:33-41. The reference evaluates (a > b) ? a + f(b - a) : b + f(a - b); the two
// arms are the same expression max + f(min - max) with the same operands, so it is computed once,
// without a divergent branch around the (long) exp/log1p chain.
__device__ __forceinline__ float LogSumExp(float a, float b, const unsigned long long* exp_tab) {
  const float ninf = __int_as_float(0xff800000);
  if (a == ninf) return b;
  if (b == ninf) return a;
  const bool a_gt = a > b;
  const float hi = a_gt ? a : b;
  const float d = a_gt ? __fsub_rn(b, a) : __fsub_rn(a, b);
  return __fadd_rn(hi, Log1pfExact(ExpfExact(d, exp_tab)));
}


// ---------------------------------------------------------------------------------------------
// Double precision (T = double is registered too, kernels.cc:275): the normaliser then calls exp()
// and log(). Same approach: glibc 2.39's Arm Optimized Routines double algorithms (N = 128), in the
// operation order of __exp_fma / __log_fma (read off the disassembly of this image's libm; CPU twin
// and its 2e9-sample check: oracle/libm_port.h). LogSumExp stays in the float functions even for
// double (util/ctc_loss_util.h:39-40).
// ---------------------------------------------------------------------------------------------
}  // namespace ctcx
#define CTCX_TAB_QUAL static __device__ __constant__
#include "ctcx_libm_f64_tables.h"
#undef CTCX_TAB_QUAL
namespace ctcx {

__device__ __forceinline__ double AsD(unsigned long long u) { return __longlong_as_double((long long)u); }

// exp for -512 < x <= 0; smaller arguments (< 1e-222, never able to change a sum >= 1) and -inf give 0.
// `tab` = the 256-entry table (a shared-memory copy where lanes index it divergently).
__device__ __forceinline__ double ExpExactD(double x, const unsigned long long* tab) {
  const unsigned abstop = (unsigned)((unsigned long long)__double_as_longlong(x) >> 52) & 0x7ffu;
  if (abstop - 0x3c9u >= 0x3fu) {
    if (abstop < 0x3c9u) return __dadd_rn(1.0, x);
    return 0.0;
  }
  const double InvLn2N = AsD(kCtcxExpHdr[0]), Shift = AsD(kCtcxExpHdr[1]);
  const double NegLn2hiN = AsD(kCtcxExpHdr[2]), NegLn2loN = AsD(kCtcxExpHdr[3]);
  const double C2 = AsD(kCtcxExpHdr[4]), C3 = AsD(kCtcxExpHdr[5]), C4 = AsD(kCtcxExpHdr[6]), C5 = AsD(kCtcxExpHdr[7]);
  double kd = __fma_rn(InvLn2N, x, Shift);
  const unsigned long long ki = (unsigned long long)__double_as_longlong(kd);
  kd = __dsub_rn(kd, Shift);
  double r = __fma_rn(kd, NegLn2hiN, x);
  r = __fma_rn(kd, NegLn2loN, r);
  const unsigned idx = 2u * ((unsigned)ki & 127u);
  const double tail = AsD(tab[idx]);
  const unsigned long long sbits = tab[idx + 1] + (ki << 45);
  const double r2 = __dmul_rn(r, r);
  const double p23 = __fma_rn(C3, r, C2);
  const double p45 = __fma_rn(r, C5, C4);
  double tmp = __fma_rn(p23, r2, __dadd_rn(tail, r));
  tmp = __fma_rn(__dmul_rn(r2, r2), p45, tmp);
  const double scale = AsD(sbits);
  return __fma_rn(scale, tmp, scale);
}

// log for finite x >= 1.
__device__ __forceinline__ double LogExactD(double x) {
  const unsigned long long ix = (unsigned long long)__double_as_longlong(x);
  if (ix - 0x3fee000000000000ull < 0x3090000000000ull) {  // near 1: dedicated polynomial
    if (ix == 0x3ff0000000000000ull) return 0.0;
    const double B0 = AsD(kCtcxLogHdr[7]);
    const double r = __dsub_rn(x, 1.0);
    const double r2 = __dmul_rn(r, r);
    const double r3 = __dmul_rn(r, r2);
    const double q1 = __fma_rn(r2, AsD(kCtcxLogHdr[10]), __fma_rn(AsD(kCtcxLogHdr[9]), r, AsD(kCtcxLogHdr[8])));
    const double q4 = __fma_rn(r2, AsD(kCtcxLogHdr[13]), __fma_rn(AsD(kCtcxLogHdr[12]), r, AsD(kCtcxLogHdr[11])));
    double q7 = __fma_rn(r2, AsD(kCtcxLogHdr[16]), __fma_rn(AsD(kCtcxLogHdr[15]), r, AsD(kCtcxLogHdr[14])));
    q7 = __fma_rn(r3, AsD(kCtcxLogHdr[17]), q7);
    double y = __fma_rn(q7, r3, q4);
    y = __fma_rn(y, r3, q1);
    const double two27 = 134217728.0;
    const double rw = __fma_rn(r, two27, r);
    const double rhi = __fma_rn(-two27, r, rw);
    const double rlo = __dsub_rn(r, rhi);
    const double rhi2 = __dmul_rn(rhi, rhi);
    const double hi = __fma_rn(rhi2, B0, r);
    double lo = __fma_rn(rhi2, B0, __dsub_rn(r, hi));
    lo = __fma_rn(__dmul_rn(B0, rlo), __dadd_rn(rhi, r), lo);
    y = __fma_rn(y, r3, lo);
    return __dadd_rn(y, hi);
  }
  const unsigned long long tmp = ix - 0x3fe6000000000000ull;
  const int i = (int)((tmp >> 45) & 127ull);
  const int k = (int)((long long)tmp >> 52);
  const unsigned long long iz = ix - (tmp & (0xfffull << 52));
  const double invc = AsD(kCtcxLogTab[2 * i]), logc = AsD(kCtcxLogTab[2 * i + 1]);
  const double z = AsD(iz);
  const double r = __fma_rn(z, invc, -1.0);
  const double kd = (double)k;
  const double w = __fma_rn(kd, AsD(kCtcxLogHdr[0]), logc);
  const double hi = __dadd_rn(w, r);
  double lo = __dadd_rn(__dsub_rn(w, hi), r);
  lo = __fma_rn(kd, AsD(kCtcxLogHdr[1]), lo);
  const double r2 = __dmul_rn(r, r);
  const double p12 = __fma_rn(AsD(kCtcxLogHdr[4]), r, AsD(kCtcxLogHdr[3]));
  const double p34 = __fma_rn(r, AsD(kCtcxLogHdr[6]), AsD(kCtcxLogHdr[5]));
  lo = __fma_rn(r2, AsD(kCtcxLogHdr[2]), lo);
  const double p = __fma_rn(p34, r2, p12);
  const double y = __fma_rn(__dmul_rn(r, r2), p, lo);
  return __dadd_rn(y, hi);
}

// util/ctc_loss_util.h:33-41 with T = double: the difference is rounded to float, expf / log1pf are
// the float functions, their float result is added to the larger operand in double.
__device__ __forceinline__ double LogSumExp(double a, double b, const unsigned long long* exp_tab) {
  const double ninf = __longlong_as_double((long long)0xfff0000000000000ull);
  if (a == ninf) return b;
  if (b == ninf) return a;
  const bool a_gt = a > b;
  const double hi = a_gt ? a : b;
  const double d = a_gt ? __dsub_rn(b, a) : __dsub_rn(a, b);
  return __dadd_rn(hi, (double)Log1pfExact(ExpfExact(__double2float_rn(d), exp_tab)));
}

}  // namespace ctcx
