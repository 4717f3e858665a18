/* TEST INFRASTRUCTURE ONLY (oracle/). Sweeps libm_port.h against the host libm.
 *   ctcx_port_mismatches(stride): every stride-th float of the three domains; returns the number of
 *   inputs whose results differ in any bit (out[0..2] = per-function counts). stride=1 is the
 *   exhaustive sweep quoted in libm_port.h (about 2 CPU-minutes). */
#include "libm_port.h"

long long ctcx_port_mismatches(unsigned stride, long long* out) {
  if (stride == 0) stride = 1;
  long long be = 0, bl = 0, bg = 0;
  for (uint64_t u = 0x80000000ull; u <= (uint64_t)ctcx_asuint(-200.0f); u += stride) {
    volatile float x = ctcx_asfloat((uint32_t)u);
    if (ctcx_asuint(expf(x)) != ctcx_asuint(ctcx_port_expf(x))) ++be;
  }
  for (uint64_t u = 0; u <= 0x3f800000ull; u += stride) {
    volatile float x = ctcx_asfloat((uint32_t)u);
    if (ctcx_asuint(log1pf(x)) != ctcx_asuint(ctcx_port_log1pf(x))) ++bl;
  }
  for (uint64_t u = 0x3f800000ull; u <= (uint64_t)ctcx_asuint(65536.0f); u += stride) {
    volatile float x = ctcx_asfloat((uint32_t)u);
    if (ctcx_asuint(logf(x)) != ctcx_asuint(ctcx_port_logf(x))) ++bg;
  }
  if (out) {
    out[0] = be;
    out[1] = bl;
    out[2] = bg;
  }
  return be + bl + bg;
}

/* util/ctc_loss_util.h:33-41 with the host libm */
static float ctcx_libm_lse(float a, float b) {
  if (a == -INFINITY) return b;
  if (b == -INFINITY) return a;
  return (a > b) ? a + log1pf(expf(b - a)) : b + log1pf(expf(a - b));
}

/* Compares n results `got` of a device function with the host libm at the inputs whose bit patterns
 * are u0 ... u0+n-1. op 0 expf, 1 log1pf, 2 logf, 3 LogSumExp(x, 0), 4 LogSumExp(0, x) (the ops of
 * ctcx_debug_math_f32). Returns the number of inputs whose results differ in any bit; the first
 * min(count, max_bad) of them go to first_bad. */
long long ctcx_libm_mismatches_f32(int op, uint32_t u0, long long n, const float* got, uint32_t* first_bad,
                                   int max_bad) {
  long long bad = 0;
  for (long long i = 0; i < n; ++i) {
    const uint32_t u = u0 + (uint32_t)i;
    volatile float x = ctcx_asfloat(u);
    float want;
    switch (op) {
      case 0: want = expf(x); break;
      case 1: want = log1pf(x); break;
      case 2: want = logf(x); break;
      case 3: want = ctcx_libm_lse(x, 0.0f); break;
      case 4: want = ctcx_libm_lse(0.0f, x); break;
      default: return -1;
    }
    if (ctcx_asuint(want) != ctcx_asuint(got[i])) {
      if (bad < max_bad) first_bad[bad] = u;
      ++bad;
    }
  }
  return bad;
}

/* element-wise helpers for the Python side of the tests */
void ctcx_port_expf_v(const float* x, float* y, int n) { for (int i = 0; i < n; ++i) y[i] = ctcx_port_expf(x[i]); }
void ctcx_port_log1pf_v(const float* x, float* y, int n) { for (int i = 0; i < n; ++i) y[i] = ctcx_port_log1pf(x[i]); }
void ctcx_port_logf_v(const float* x, float* y, int n) { for (int i = 0; i < n; ++i) y[i] = ctcx_port_logf(x[i]); }
void ctcx_libm_expf_v(const float* x, float* y, int n) { for (int i = 0; i < n; ++i) y[i] = expf(x[i]); }
void ctcx_libm_log1pf_v(const float* x, float* y, int n) { for (int i = 0; i < n; ++i) y[i] = log1pf(x[i]); }
void ctcx_libm_logf_v(const float* x, float* y, int n) { for (int i = 0; i < n; ++i) y[i] = logf(x[i]); }

/* Double-precision ports against libm exp()/log() on n pseudo-random arguments per domain
 * (splitmix64 from `seed`): exp on (-512, 0] drawn uniformly in value and uniformly in bit pattern,
 * log on [1, 65536) uniformly in bit pattern plus the near-1 polynomial range [1, 1.0647).
 * out[0] = exp mismatches, out[1] = log mismatches. */
static uint64_t ctcx_sm64(uint64_t* s) {
  uint64_t z = (*s += 0x9E3779B97F4A7C15ull);
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
long long ctcx_port_mismatches_f64(long long n, unsigned long long seed, long long* out) {
  uint64_t s = seed;
  long long be = 0, bl = 0;
  const uint64_t lo_e = ctcx_asuint64(-0x1p-60), hi_e = ctcx_asuint64(-511.99);  /* bit range of (-512, -2^-60] */
  const uint64_t lo_l = ctcx_asuint64(1.0), hi_l = ctcx_asuint64(65536.0), hi_n = ctcx_asuint64(1.0647);
  for (long long i = 0; i < n; ++i) {
    volatile double x1 = -512.0 * ((double)(ctcx_sm64(&s) >> 11) * 0x1p-53);
    volatile double x2 = ctcx_asdouble(lo_e + ctcx_sm64(&s) % (hi_e - lo_e));
    if (ctcx_asuint64(exp(x1)) != ctcx_asuint64(ctcx_port_exp(x1))) ++be;
    if (x2 > -512.0 && ctcx_asuint64(exp(x2)) != ctcx_asuint64(ctcx_port_exp(x2))) ++be;
    volatile double y1 = ctcx_asdouble(lo_l + ctcx_sm64(&s) % (hi_l - lo_l));
    volatile double y2 = ctcx_asdouble(lo_l + ctcx_sm64(&s) % (hi_n - lo_l));
    if (ctcx_asuint64(log(y1)) != ctcx_asuint64(ctcx_port_log(y1))) ++bl;
    if (ctcx_asuint64(log(y2)) != ctcx_asuint64(ctcx_port_log(y2))) ++bl;
  }
  if (out) {
    out[0] = be;
    out[1] = bl;
  }
  return be + bl;
}
void ctcx_port_exp_v(const double* x, double* y, int n) { for (int i = 0; i < n; ++i) y[i] = ctcx_port_exp(x[i]); }
void ctcx_port_log_v(const double* x, double* y, int n) { for (int i = 0; i < n; ++i) y[i] = ctcx_port_log(x[i]); }
void ctcx_libm_exp_v(const double* x, double* y, int n) { for (int i = 0; i < n; ++i) y[i] = exp(x[i]); }
void ctcx_libm_log_v(const double* x, double* y, int n) { for (int i = 0; i < n; ++i) y[i] = log(x[i]); }
