// Genotype likelihood / posterior arithmetic of MALVA, typed exactly as the
// reference evaluates it (SURVEY 8a "G2 evaluation order"):
//   VB::genotype          var_block.hpp:224-330
//   VB::log_binomial      var_block.hpp:792-797
//   arg-max / GQ          var_block.hpp:367-394
// float-typed terms (priors, error terms) go through a bit-exact port of
// glibc's logf (sysdeps/ieee754/flt-32/e_logf.c, 16-entry table + cubic in
// double; verified against libm over every positive float, with and without
// FMA contraction -- both give identical floats).  No FMA contraction is
// allowed anywhere else: every product/sum below uses explicit *_rn intrinsics.
#pragma once
#include <cmath>
#include <cstdint>
#include <cstring>

#include "xxh3.cuh"

namespace mg {

MG_HD float f32_mul(float a, float b) {
#if defined(__CUDA_ARCH__)
  return __fmul_rn(a, b);
#else
  volatile float r = a * b;
  return r;
#endif
}
MG_HD float f32_sub(float a, float b) {
#if defined(__CUDA_ARCH__)
  return __fsub_rn(a, b);
#else
  volatile float r = a - b;
  return r;
#endif
}
MG_HD float f32_div(float a, float b) {
#if defined(__CUDA_ARCH__)
  return __fdiv_rn(a, b);
#else
  volatile float r = a / b;
  return r;
#endif
}
MG_HD double f64_mul(double a, double b) {
#if defined(__CUDA_ARCH__)
  return __dmul_rn(a, b);
#else
  volatile double r = a * b;
  return r;
#endif
}
MG_HD double f64_add(double a, double b) {
#if defined(__CUDA_ARCH__)
  return __dadd_rn(a, b);
#else
  volatile double r = a + b;
  return r;
#endif
}
MG_HD double f64_sub(double a, double b) {
#if defined(__CUDA_ARCH__)
  return __dsub_rn(a, b);
#else
  volatile double r = a - b;
  return r;
#endif
}

MG_HD uint32_t f2u(float f) {
#if defined(__CUDA_ARCH__)
  return __float_as_uint(f);
#else
  uint32_t u;
  memcpy(&u, &f, 4);
  return u;
#endif
}
MG_HD float u2f(uint32_t u) {
#if defined(__CUDA_ARCH__)
  return __uint_as_float(u);
#else
  float f;
  memcpy(&f, &u, 4);
  return f;
#endif
}
MG_HD double u2d(uint64_t u) {
#if defined(__CUDA_ARCH__)
  return __longlong_as_double((long long)u);
#else
  double d;
  memcpy(&d, &u, 8);
  return d;
#endif
}

// bit patterns of glibc's __logf_data (invc, logc) table, ln2 and the cubic
MG_HD double logf_invc(int i) {
  switch (i) {
    case 0: return 0x1.661ec79f8f3bep+0;
    case 1: return 0x1.571ed4aaf883dp+0;
    case 2: return 0x1.49539f0f010bp+0;
    case 3: return 0x1.3c995b0b80385p+0;
    case 4: return 0x1.30d190c8864a5p+0;
    case 5: return 0x1.25e227b0b8eap+0;
    case 6: return 0x1.1bb4a4a1a343fp+0;
    case 7: return 0x1.12358f08ae5bap+0;
    case 8: return 0x1.0953f419900a7p+0;
    case 9: return 0x1p+0;
    case 10: return 0x1.e608cfd9a47acp-1;
    case 11: return 0x1.ca4b31f026aap-1;
    case 12: return 0x1.b2036576afce6p-1;
    case 13: return 0x1.9c2d163a1aa2dp-1;
    case 14: return 0x1.886e6037841edp-1;
    default: return 0x1.767dcf5534862p-1;
  }
}
MG_HD double logf_logc(int i) {
  switch (i) {
    case 0: return -0x1.57bf7808caadep-2;
    case 1: return -0x1.2bef0a7c06ddbp-2;
    case 2: return -0x1.01eae7f513a67p-2;
    case 3: return -0x1.b31d8a68224e9p-3;
    case 4: return -0x1.6574f0ac07758p-3;
    case 5: return -0x1.1aa2bc79c81p-3;
    case 6: return -0x1.a4e76ce8c0e5ep-4;
    case 7: return -0x1.1973c5a611cccp-4;
    case 8: return -0x1.252f438e10c1ep-5;
    case 9: return 0x0p+0;
    case 10: return 0x1.aa5aa5df25984p-5;
    case 11: return 0x1.c5e53aa362eb4p-4;
    case 12: return 0x1.526e57720db08p-3;
    case 13: return 0x1.bc2860d22477p-3;
    case 14: return 0x1.1058bc8a07ee1p-2;
    default: return 0x1.4043057b6ee09p-2;
  }
}

// glibc logf, bit exact (inputs: any float; negative / NaN -> NaN)
MG_HD float glibc_logf(float x) {
  uint32_t ix = f2u(x);
  if (ix == 0x3f800000u) return 0.0f;
  if (ix - 0x00800000u >= 0x7f800000u - 0x00800000u) {
    if (ix * 2u == 0u) return u2f(0xff800000u);                        // log(0) = -inf
    if (ix == 0x7f800000u) return x;                                    // log(inf) = inf
    if ((ix & 0x80000000u) || ix * 2u >= 0xff000000u) return u2f(0x7fc00000u);
    ix = f2u(f32_mul(x, 0x1p23f));                                      // subnormal: normalise
    ix -= 23u << 23;
  }
  uint32_t tmp = ix - 0x3f330000u;
  int i = (int)((tmp >> 19) & 15u);
  int k = (int32_t)tmp >> 23;
  uint32_t iz = ix - (tmp & 0xff800000u);
  double z = (double)u2f(iz);
  double r = f64_sub(f64_mul(z, logf_invc(i)), 1.0);
  double y0 = f64_add(logf_logc(i), f64_mul((double)k, 0x1.62e42fefa39efp-1));
  double r2 = f64_mul(r, r);
  double y = f64_add(f64_mul(0x1.5575b0be00b6ap-2, r), -0x1.ffffef20a4123p-2);
  y = f64_add(f64_mul(-0x1.00ea348b88334p-2, r2), y);
  y = f64_add(f64_mul(y, r2), f64_add(y0, r));
  return (float)y;
}

// log((double)i) for 0 < i < LOG_TABLE_N as the host's libm computes it (built at mg_create).  CUDA's fp64 log is
// within 1 ulp, glibc's is correctly rounded nearly everywhere, and one ulp of log_binomial decides GT wherever two
// genotypes are mathematically tied (uniform priors, coverages like 2,12,2): with the table the device's log-posterior
// is the reference's bit for bit for every tot < 2^16.  Larger arguments (and the host self-test path, table NULL)
// use the libm at hand.
constexpr int LOG_TABLE_N = 1 << 16;
MG_HD double log_int(int x, const double *log_table) {
  return (log_table && x > 0 && x < LOG_TABLE_N) ? log_table[x] : log((double)x);
}

MG_HD double log_binomial(int n, int k, const double *log_table) {  // var_block.hpp:792-797
  if (n == 0 || n == k || k == 0) return 0.0;
  double a = f64_mul((double)n, log_int(n, log_table));
  double b = f64_mul((double)k, log_int(k, log_table));
  double c = f64_mul((double)(n - k), log_int(n - k, log_table));
  return f64_sub(f64_sub(a, b), c);
}

struct GenoConsts {  // per n_alleles: c1..c4 of SURVEY 8a
  float c1, c2, c3, c4;
};
MG_HD GenoConsts geno_consts(float e, int n) {
  GenoConsts c;
  float one_minus_e = f32_sub(1.0f, e);
  c.c1 = glibc_logf(one_minus_e);
  c.c2 = glibc_logf(f32_div(e, (float)(n - 1)));
  c.c3 = glibc_logf(f32_div(one_minus_e, 2.0f));
  c.c4 = n > 2 ? glibc_logf(f32_div(e, (float)(n - 2))) : 0.0f;
  return c;
}

MG_HD double prob_from_log(double log_prior, double log_post) {
  double lp = f64_add(log_prior, log_post);
  if (isinf(lp)) return 0.0;
#if defined(__CUDA_ARCH__)
  // results below DBL_MIN: CUDA's exp does not return glibc's subnormals there, and when every likelihood of a variant
  // is that small the one glibc keeps decides GT.  exp(lp + 64 ln2_hi) * exp(64 (ln2 - ln2_hi)) * 2^-64 instead:
  // lp + 64 ln2_hi is exact (ln2_hi has 32 significant bits), the factor is a constant, and the scaling rounds into
  // the subnormal range once -- within ~1 ulp of the normal-range result, so 1-ulp-of-lp ties keep glibc's order
  // almost always.
  if (lp < -708.0) return __dmul_rn(__dmul_rn(exp(__dadd_rn(lp, 64.0 * 0x1.62e42feep-1)), 0x1.0000003473de7p+0), 0x1p-64);
#endif
  return exp(lp);
}

// homozygous / haploid genotype g (var_block.hpp:272-285, 296-304)
MG_HD double geno_hom(uint32_t t, uint32_t tot, float f, const GenoConsts &c, const double *log_table) {
  uint32_t er = tot - t;
  double log_prior = (double)f32_mul(2.0f, glibc_logf(f));
  double lb = log_binomial((int)(t + er), (int)t, log_table);
  double log_post = f64_add(f64_add(lb, (double)f32_mul((float)t, c.c1)), (double)f32_mul((float)er, c.c2));
  return prob_from_log(log_prior, log_post);
}
// heterozygous genotype g1<g2 (var_block.hpp:306-318)
MG_HD double geno_het(uint32_t t1, uint32_t t2, uint32_t tot, float f1, float f2, int n, const GenoConsts &c,
                      const double *log_table) {
  uint32_t er = tot - t1 - t2;
  double log_prior = (double)glibc_logf(f32_mul(f32_mul(2.0f, f1), f2));
  double lb1 = log_binomial((int)(t1 + t2 + er), (int)(t1 + t2), log_table);
  double lb2 = log_binomial((int)(t1 + t2), (int)t1, log_table);
  double log_post = f64_add(f64_add(f64_add(lb1, lb2), (double)f32_mul((float)t1, c.c3)),
                            (double)f32_mul((float)t2, c.c3));
  if (n > 2) log_post = f64_add(log_post, (double)f32_mul((float)er, c.c4));
  return prob_from_log(log_prior, log_post);
}

}  // namespace mg
