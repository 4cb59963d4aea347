"""Run-time compiled CUDA likelihoods (targets.CudaLikelihood), the parts that need no GPU:
NVRTC compiles the user's source together with the library's own d <= 4 chain-step kernel and
the batched row kernel for sm_100a, and bad input is refused on the host.  Compiling the three
sources below also catches header drift: host-only code added to a header the run-time
translation unit includes (kernels_small.cuh, step.cuh, rng.cuh, targets.cuh, the public header)
breaks them.  The sources are shared with test_cuda_likelihood_gpu.py."""
import numpy as np
import pytest

# examples/ex_para_fit.py:39-55 in the reference's per-term form; data = x[M], y[M], yerr[M]
LINEFIT_PER_TERM = r'''
__device__ double ln_like(const double* theta, const double* data) {
  const int M = BPM_NDATA / 3;
  const double* x = data;
  const double* y = data + M;
  const double* yerr = data + 2 * M;
  const double m = theta[0], b = theta[1], lnf = theta[2];
  if (!(-5.0 < m && m < 0.5 && 0.0 < b && b < 10.0 && -10.0 < lnf && lnf < 1.0)) return -INFINITY;
  const double e2 = exp(2.0 * lnf);
  double s = 0.0;
  for (int i = 0; i < M; ++i) {
    const double model = m * x[i] + b;
    const double inv = 1.0 / (yerr[i] * yerr[i] + model * model * e2);
    const double r = y[i] - model;
    s += r * r * inv - log(inv);
  }
  return 0.0 + -0.5 * s;
}
'''

# the built-in line fit's own arithmetic (csrc/targets.cuh), data as above
LINEFIT_SAME = r'''
__device__ double ln_like(const double* theta, const double* data) {
  const int M = BPM_NDATA / 3;
  return bpm::linefit_lnl(data, data + M, data + 2 * M, M, theta[0], theta[1], theta[2]);
}
'''

# the built-in banana; data = Banana_2D.device_target().params (10 doubles)
BANANA_SAME = r'''
__device__ double ln_like(const double* theta, const double* data) {
  bpm::BananaParams p;
  p.log_of_pdf = data[0]; p.a = data[1]; p.b = data[2];
  p.g.mu0 = data[3]; p.g.mu1 = data[4];
  p.g.U00 = data[5]; p.g.U01 = data[6]; p.g.U10 = data[7]; p.g.U11 = data[8];
  p.g.c0 = data[9];
  return bpm::banana_lnl(p, theta[0], theta[1]);
}
'''

# the built-in exp fit at d = 5; data = t[M], y[M]
EXPFIT_SAME = r'''
__device__ double ln_like(const double* theta, const double* data) {
  const int M = BPM_NDATA / 2;
  return bpm::expfit_lnl(data, data + M, M, theta[0], theta[1], theta[2], theta[3], theta[4]);
}
'''


def linefit_data():
    from bipymc_b200 import targets
    f = targets.LineFit()
    return np.concatenate([f.x, f.y, f.yerr])


def banana_data():
    from bipymc_b200 import targets
    return targets.Banana_2D(sigma1=1.0, sigma2=1.0).device_target().params


def expfit_data():
    from bipymc_b200 import targets
    f = targets.ExpFit()
    return np.concatenate([f.t, f.y])


@pytest.mark.parametrize("name", ["linefit_per_term", "banana", "expfit_d5"])
def test_sources_compile_for_sm100a(name):
    from bipymc_b200 import targets
    src, dim, data = {"linefit_per_term": (LINEFIT_PER_TERM, 3, linefit_data()),
                      "banana": (BANANA_SAME, 2, banana_data()),
                      "expfit_d5": (EXPFIT_SAME, 5, expfit_data())}[name]
    lik = targets.CudaLikelihood(src, dim, data, fmad=False)
    lik.compile()
    assert lik.compile() is True          # the second compile of the same source comes from the process cache


def test_fmad_is_part_of_the_cache_key():
    from bipymc_b200 import targets
    src = LINEFIT_SAME + "// fmad key\n"
    assert targets.CudaLikelihood(src, 3, linefit_data(), fmad=True).compile() is False
    assert targets.CudaLikelihood(src, 3, linefit_data(), fmad=False).compile() is False
    assert targets.CudaLikelihood(src, 3, linefit_data(), fmad=False).compile() is True


def test_syntax_error_names_the_user_line():
    from bipymc_b200 import targets
    src = ("__device__ double ln_like(const double* theta, const double* data) {\n"
           "  double a = theta[0];\n"
           "  double b = a * 2.0;\n"
           "  return a + ;\n"
           "}\n")
    with pytest.raises(targets.CudaCompileError) as e:
        targets.CudaLikelihood(src, 2).compile()
    assert "ln_like.cu(4)" in str(e.value)
    assert "ln_like.cu(4)" in e.value.log


def test_source_without_ln_like_is_refused():
    from bipymc_b200 import _lib, targets
    with pytest.raises(_lib.BpmError, match="ln_like"):
        targets.CudaLikelihood("__device__ double lnl(const double* t, const double* d) { return 0.0; }",
                               2).compile()


@pytest.mark.parametrize("kw", [dict(dim=0), dict(dim=-3), dict(dim=2.5), dict(dim=True),
                                dict(data=[0.0, np.nan]), dict(data=[np.inf]), dict(data=np.zeros((2, 3))),
                                dict(data=["a", "b"])])
def test_bad_arguments_raise_value_error(kw):
    from bipymc_b200 import targets
    args = dict(source=LINEFIT_SAME, dim=3, data=None)
    args.update(kw)
    with pytest.raises(ValueError):
        targets.CudaLikelihood(**args)


def test_source_must_be_str():
    from bipymc_b200 import targets
    with pytest.raises(ValueError):
        targets.CudaLikelihood(LINEFIT_SAME.encode(), 3)

