"""Several problems in one sampler (targets.CudaLikelihoodSet), the parts that need no GPU: argument
validation, the multi-problem NVRTC translation unit (its own, with P and n_data in the cache key), compile
errors with the user's line numbers, the problem key rule and the C-ABI refusals that need no device.
The sources are shared with test_problems_gpu.py."""
import ctypes as C

import numpy as np
import pytest

from test_cuda_likelihood_cpu import EXPFIT_SAME, LINEFIT_PER_TERM, expfit_data, linefit_data

# theta = (a, b): y = a + b x with known noise, data = x[M], y[M], sigma[M]; box prior |a|, |b| < 100
LINE_GAUSS = r'''
__device__ double ln_like(const double* theta, const double* data) {
  const int M = BPM_NDATA / 3;
  if (!(fabs(theta[0]) < 100.0 && fabs(theta[1]) < 100.0)) return -INFINITY;
  double s = 0.0;
  for (int i = 0; i < M; ++i) {
    const double r = (data[M + i] - theta[0] - theta[1] * data[i]) / data[2 * M + i];
    s += r * r;
  }
  return -0.5 * s;
}
'''


def linefit_set(P, seed=0):
    """P line-fit datasets: the reference's data with the ordinate shifted and rescaled per problem."""
    base = linefit_data()
    M = base.size // 3
    rs = np.random.RandomState(seed)
    rows = np.tile(base, (P, 1))
    rows[:, M:2 * M] = rows[:, M:2 * M] * (1.0 + 0.05 * rs.randn(P, 1)) + 0.2 * rs.randn(P, 1)
    return rows


def expfit_set(P, seed=0):
    base = expfit_data()
    M = base.size // 2
    rs = np.random.RandomState(seed)
    rows = np.tile(base, (P, 1))
    rows[:, M:] += 0.01 * rs.randn(P, 1)
    return rows


def test_validation():
    from bipymc_b200 import targets
    good = np.ones((3, 4))
    with pytest.raises(ValueError, match="str"):
        targets.CudaLikelihoodSet(b"x", 2, good)
    with pytest.raises(ValueError, match="dim"):
        targets.CudaLikelihoodSet(LINE_GAUSS, 0, good)
    with pytest.raises(ValueError, match="dim"):
        targets.CudaLikelihoodSet(LINE_GAUSS, True, good)
    for bad in (np.ones(4), np.ones((0, 4)), np.ones((3, 0)), np.ones((2, 2, 2))):
        with pytest.raises(ValueError, match="shape"):
            targets.CudaLikelihoodSet(LINE_GAUSS, 2, bad)
    with pytest.raises(ValueError, match="finite"):
        targets.CudaLikelihoodSet(LINE_GAUSS, 2, np.array([[1.0, np.nan]]))
    lik = targets.CudaLikelihoodSet(LINE_GAUSS, 2, good, fmad=False)
    assert lik.n_problems == 3 and lik.dim == 2 and not lik.fmad
    assert lik.data.flags.c_contiguous and lik.data.dtype == np.float64
    # a CudaLikelihood still refuses 2-D data
    with pytest.raises(ValueError, match="1-D"):
        targets.CudaLikelihood(LINE_GAUSS, 2, good)


@pytest.mark.parametrize("name", ["linefit_d3", "expfit_d5", "line_gauss_d2"])
def test_sources_compile_for_sm100a(name):
    from bipymc_b200 import targets
    src, dim, data = {"linefit_d3": (LINEFIT_PER_TERM, 3, linefit_set(7)),
                      "expfit_d5": (EXPFIT_SAME, 5, expfit_set(7)),
                      "line_gauss_d2": (LINE_GAUSS, 2, np.ones((7, 30)))}[name]
    for fmad in (True, False):
        targets.CudaLikelihoodSet(src, dim, data, fmad=fmad).compile()


def test_compile_error_carries_user_line_numbers():
    from bipymc_b200 import targets
    src = "__device__ double ln_like(const double* t, const double* d) {\n  return t[0] +\n  undefined_name;\n}\n"
    with pytest.raises(targets.CudaCompileError) as ei:
        targets.CudaLikelihoodSet(src, 2, np.ones((4, 3))).compile()
    assert "ln_like.cu(3)" in ei.value.log and "undefined_name" in ei.value.log


def test_cache_key_includes_problems_and_data_size():
    from bipymc_b200 import targets
    src = LINE_GAUSS + "// cache key test %d\n" % np.random.randint(1 << 30)
    assert targets.CudaLikelihoodSet(src, 2, np.ones((5, 30))).compile() is False
    assert targets.CudaLikelihoodSet(src, 2, 2.0 * np.ones((5, 30))).compile() is True     # data values: not in the key
    assert targets.CudaLikelihoodSet(src, 2, np.ones((6, 30))).compile() is False          # P
    assert targets.CudaLikelihoodSet(src, 2, np.ones((5, 33))).compile() is False          # n_data
    # the single-problem translation unit is another module: same source, same n_data
    assert targets.CudaLikelihood(src, 2, np.ones(30)).compile() is False


def test_problem_seed_rule():
    from bipymc_b200 import targets
    keys = targets.problem_seeds(12345, 4)
    assert keys[0] == 12345
    assert keys == [(12345 + 0x9E3779B97F4A7C15 * g) % (1 << 64) for g in range(4)]
    assert all(0 <= k < 1 << 64 for k in targets.problem_seeds(2 ** 64 - 1, 9))
    assert targets.problem_seeds([3, 1, 2], 3) == [3, 1, 2]
    with pytest.raises(ValueError, match="3 keys for 2 problems"):
        targets.problem_seeds([3, 1, 2], 2)
    with pytest.raises(ValueError, match="2\\^64"):
        targets.problem_seeds([-1, 1], 2)


def test_entry_points_without_device():
    """bpm_jit_compile_problems refuses bad arguments; the problem entry points refuse a null handle."""
    from bipymc_b200 import _lib
    lib = _lib.load()
    log = C.create_string_buffer(1024)
    assert lib.bpm_jit_compile_problems(LINE_GAUSS.encode(), 2, 0, 3, 1, None, log, 1024) != 0
    assert b"n_data" in lib.bpm_last_error()
    assert lib.bpm_jit_compile_problems(LINE_GAUSS.encode(), 2, 30, 0, 1, None, log, 1024) != 0
    assert b"n_problems" in lib.bpm_last_error()
    keys = (C.c_uint64 * 2)(1, 2)
    assert lib.bpm_set_problems(None, 2, keys) != 0
    assert lib.bpm_get_problem_counters(None, None, None) != 0
    assert lib.bpm_get_problem_cr_state(None, None, None, None) != 0
    assert lib.bpm_set_problem_cr_state(None, None, None, None) != 0


@pytest.mark.parametrize("kw, match", [(dict(subpop_k=5), "subpop_k"), (dict(outlier_gen=10), "outlier_gen"),
                                       (dict(ln_like_batched=lambda t: t[:, 0]), "ln_like_batched"),
                                       (dict(device_init=True), "device_init")])
def test_multi_problem_sampler_refuses(kw, match):
    """Refused in the constructor, before any device is touched."""
    from bipymc_b200 import DeMcMpi, DreamMpi, targets
    lik = targets.CudaLikelihoodSet(LINE_GAUSS, 2, np.ones((3, 30)))
    for cls in (DeMcMpi, DreamMpi):
        with pytest.raises(ValueError, match=match):
            cls(None, np.zeros(2), n_chains=8, ln_like_cuda=lik, **kw)


def test_seed_sequence_needs_a_likelihood_set():
    from bipymc_b200 import DreamMpi, targets
    with pytest.raises(ValueError, match="CudaLikelihoodSet"):
        DreamMpi(None, np.zeros(2), n_chains=8, seed=[1, 2],
                 ln_like_cuda=targets.CudaLikelihood(LINE_GAUSS, 2, np.ones(30)))
    with pytest.raises(ValueError, match="2 keys for 3 problems"):
        DreamMpi(None, np.zeros(2), n_chains=8, seed=[1, 2],
                 ln_like_cuda=targets.CudaLikelihoodSet(LINE_GAUSS, 2, np.ones((3, 30))))


def test_serial_demc_refuses_a_likelihood_set():
    from bipymc_b200 import DeMc, targets
    with pytest.raises(NotImplementedError, match="CudaLikelihoodSet"):
        DeMc(None, n_chains=8, ln_like_cuda=targets.CudaLikelihoodSet(LINE_GAUSS, 2, np.ones((3, 30))))
