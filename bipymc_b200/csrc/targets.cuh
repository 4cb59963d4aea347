// Built-in batched log-likelihoods: the reference's test targets restated for the
// device (SURVEY.md section 8a rows L1-L4).  Each follows the arithmetic route of the
// scalar reference (scipy.stats.multivariate_normal: eigh whitening, then
// -0.5 * (rank*log(2pi) + log_pdet + maha); the reference then takes log(exp(.)))
// so values agree with it to ~1e-13.
#pragma once
#include <stdint.h>
#include <math.h>

namespace bpm {

// 2-D frozen multivariate normal, scipy style: maha = |(x - mu) . U|^2.
struct Mvn2 {
  double mu0, mu1;
  double U00, U01, U10, U11;  // row-major prec_U (scipy _PSD.U)
  double c0;                  // rank * log(2 pi) + log_pdet
};
__device__ __forceinline__ double mvn2_logpdf(const Mvn2& g, double x0, double x1) {
  double d0 = __dsub_rn(x0, g.mu0), d1 = __dsub_rn(x1, g.mu1);
  double y0 = __dadd_rn(__dmul_rn(d0, g.U00), __dmul_rn(d1, g.U10));
  double y1 = __dadd_rn(__dmul_rn(d0, g.U01), __dmul_rn(d1, g.U11));
  double maha = __dadd_rn(__dmul_rn(y0, y0), __dmul_rn(y1, y1));
  return -0.5 * __dadd_rn(g.c0, maha);
}

// Host params layout (doubles): [log_of_pdf, a, b, mu0, mu1, U00, U01, U10, U11, c0]
struct BananaParams {
  double log_of_pdf, a, b;
  Mvn2 g;
};
// banana_rv.py:26-37
__device__ __forceinline__ double banana_lnl(const BananaParams& p, double y1, double y2) {
  double x1 = __ddiv_rn(y1, p.a);
  double t = __dadd_rn(__dmul_rn(x1, x1), __dmul_rn(p.a, p.a));
  double x2 = __dmul_rn(__dsub_rn(y2, __dmul_rn(p.b, t)), p.a);
  double lp = mvn2_logpdf(p.g, x1, x2);
  return p.log_of_pdf != 0.0 ? log(exp(lp)) : lp;
}

// Host params layout: [log_of_pdf, w1, w2, mvn2 #1 (7), mvn2 #2 (7)]
struct BimodalParams {
  double log_of_pdf, w1, w2;
  Mvn2 g1, g2;
  double lw1, lw2;            // log(w1), log(w2): taken once on the host (bpm_set_target), not once per chain-step
};
// dblgauss_rv.py:26-32
__device__ __forceinline__ double bimodal_lnl(const BimodalParams& p, double y1, double y2) {
  double l1 = mvn2_logpdf(p.g1, y1, y2), l2 = mvn2_logpdf(p.g2, y1, y2);
  if (p.log_of_pdf != 0.0)
    return log(__dadd_rn(__dmul_rn(p.w1, exp(l1)), __dmul_rn(p.w2, exp(l2))));
  double a = l1 + p.lw1, b = l2 + p.lw2;
  double m = fmax(a, b);
  if (!(m > -INFINITY)) return -INFINITY;
  return m + log(exp(a - m) + exp(b - m));
}

// Gaussian: lnl = -0.5 * (c0 + |(x - mu) . W|^2), optional log(exp(.)) round trip
// (d100_gauss.py:29-35 takes np.log(pdf)).
__device__ __forceinline__ double gauss_finish(double c0, double maha, int log_of_pdf) {
  double lp = -0.5 * __dadd_rn(c0, maha);
  return log_of_pdf ? log(exp(lp)) : lp;
}

// Line fit, examples/ex_para_fit.py:39-55.  data = x[M], y[M], yerr[M] (device).
//   lnL = -0.5 * sum_i [ r_i^2 * inv_i - log(inv_i) ],  inv_i = 1 / (yerr_i^2 + model_i^2 e^{2 lnf}),  r_i = y_i - model_i
// Reference form, one IEEE division and one logarithm per data point (~120 instructions per term, 6 000 of the
// 7 300 instructions of a whole line-fit chain-step: profiles/r2/r2x_fused_small_linefit_ncu_summary.txt).
// Kept as the exact fallback of linefit_lnl, out of line so the rare case stays out of the hot kernels' bodies.
// Measured alternatives of the same form (profiles/r2/r2r_secondary.txt, r2s_*): four interleaved partial sums
// 76 us per generation of 10^5 chains, this form 73 us, four LANES per chain 86 us.
__device__ __noinline__ double linefit_lnl_per_term(const double* x, const double* y, const double* yerr,
                                                    int M, double m, double b, double e2) {
  double s = 0.0;
#pragma unroll 5
  for (int i = 0; i < M; ++i) {
    double model = __dadd_rn(__dmul_rn(m, x[i]), b);
    double inv = __ddiv_rn(1.0, __dadd_rn(__dmul_rn(yerr[i], yerr[i]),
                                          __dmul_rn(__dmul_rn(model, model), e2)));
    double r = __dsub_rn(y[i], model);
    s += __dsub_rn(__dmul_rn(__dmul_rn(r, r), inv), log(inv));
  }
  return 0.0 + -0.5 * s;
}

// linefit_lnl: five data points share ONE reciprocal and ONE logarithm.  With P = den_1 ... den_5 (den_i and r_i
// computed exactly as above): inv_i = (1 / P) * prod_{j != i} den_j from prefix / suffix products, and
// -sum log(inv_i) = log(P).  15 multiplications + 1 reciprocal + 1 logarithm per group instead of 5 divisions +
// 5 logarithms.  inv_i carries ~3 ulp instead of 0.5, log(P) the same absolute error as one of the five
// logarithms it replaces: |lnL - reference| / |lnL| stays ~1e-15 (the RNG-replay gate is 1e-12; tests compare
// it with the oracle's per-term numpy form).  A group whose product leaves [1e-250, 1e250] sends the whole
// evaluation to the exact form.
__device__ __forceinline__ double fast_rcp_target(double v) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(v));
  double e = fma(-v, r, 1.0);
  r = fma(r, e, r);
  e = fma(-v, r, 1.0);
  return fma(r, e, r);
}
__device__ __forceinline__ double linefit_lnl(const double* x, const double* y, const double* yerr,
                                              int M, double m, double b, double lnf) {
  if (!(-5.0 < m && m < 0.5 && 0.0 < b && b < 10.0 && -10.0 < lnf && lnf < 1.0)) return -INFINITY;
  const double e2 = exp(__dmul_rn(2.0, lnf));
  double s = 0.0, lg = 0.0;
  bool ok = true;
  // one group of five points: adds sum r_i^2 inv_i to s, returns P = den_1 ... den_5
  auto group5 = [&](int i) -> double {
    double den[5], rr[5];
#pragma unroll
    for (int q = 0; q < 5; ++q) {
      const double model = __dadd_rn(__dmul_rn(m, x[i + q]), b);
      den[q] = __dadd_rn(__dmul_rn(yerr[i + q], yerr[i + q]), __dmul_rn(__dmul_rn(model, model), e2));
      const double r = __dsub_rn(y[i + q], model);
      rr[q] = __dmul_rn(r, r);
    }
    const double p12 = den[0] * den[1], p123 = p12 * den[2], p1234 = p123 * den[3], P = p1234 * den[4];
    const double s45 = den[3] * den[4], s345 = den[2] * s45, s2345 = den[1] * s345;
    ok = ok && P > 1e-120 && P < 1e120;
    const double ip = fast_rcp_target(P);
    s += rr[0] * (ip * s2345);
    s += rr[1] * (ip * (den[0] * s345));
    s += rr[2] * (ip * (p12 * s45));
    s += rr[3] * (ip * (p123 * den[4]));
    s += rr[4] * (ip * p1234);
    return P;
  };
  int i = 0;
#pragma unroll 1
  for (; i + 10 <= M; i += 10) {               // two groups share one logarithm (|log10 P| < 240 for the pair)
    const double Pa = group5(i);
    const double Pb = group5(i + 5);
    lg += log(Pa * Pb);
  }
  if (i + 5 <= M) {
    lg += log(group5(i));
    i += 5;
  }
  if (!ok) return linefit_lnl_per_term(x, y, yerr, M, m, b, e2);
  for (; i < M; ++i) {                         // M % 5 leftover points, reference form
    const double model = __dadd_rn(__dmul_rn(m, x[i]), b);
    const double inv = __ddiv_rn(1.0, __dadd_rn(__dmul_rn(yerr[i], yerr[i]), __dmul_rn(__dmul_rn(model, model), e2)));
    const double r = __dsub_rn(y[i], model);
    s += __dmul_rn(__dmul_rn(r, r), inv);
    lg -= log(inv);
  }
  return 0.0 + -0.5 * (s + lg);
}

// Exponential-relaxation fit, examples/ex_exp_fit.py:38-121.
//   theta = (tau, c_inf, c_0, leak, sigma);  flat box prior (ex_exp_fit.py:103-121);
//   model(t) = c_inf + c_0 * (-1) * exp(-t / tau) - leak * t          (ex_exp_fit.py:38-43)
//   lnprob   = 0.0 + -0.5 * sum_i [ (model_i - y_i)^2 / sigma - log(1 / sigma) ]   (ex_exp_fit.py:73-101)
__device__ __forceinline__ double expfit_lnl(const double* t, const double* y, int M, double tau, double c_inf,
                                             double c_0, double leak, double sigma) {
  if (!(-5.0 < c_inf && c_inf < 5.0 && 1.0 < tau && tau < 50.0 && -1.0 < c_0 && c_0 < 1.0 && -5.0 < leak &&
        leak < 5.0 && 0.0 < sigma && sigma < 1.0))
    return -INFINITY;
  const double c0v = __dmul_rn(c_0, -1.0);
  const double lg = log(__ddiv_rn(1.0, sigma));
  double s = 0.0;
  for (int i = 0; i < M; ++i) {
    const double ex = exp(__ddiv_rn(-t[i], tau));
    const double m = __dsub_rn(__dadd_rn(c_inf, __dmul_rn(c0v, ex)), __dmul_rn(leak, t[i]));
    const double r = __dsub_rn(m, y[i]);
    s += __dsub_rn(__ddiv_rn(__dmul_rn(r, r), sigma), lg);
  }
  return 0.0 + -0.5 * s;
}

}  // namespace bpm
