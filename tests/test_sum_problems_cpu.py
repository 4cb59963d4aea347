"""Per-observation likelihoods for many datasets in one sampler (targets.CudaSumLikelihoodSet), the parts that
need no GPU: argument validation, the translation unit of its own (P, M, k and the prior in the cache key),
compile errors with the user's line numbers, the C-ABI refusals that need no device and the sampler refusals.
The sources are those of test_cuda_sum_likelihood_cpu.py."""
import ctypes as C

import numpy as np
import pytest

from test_cuda_sum_likelihood_cpu import EXPFIT_PRIOR, EXPFIT_TERM, LINEFIT_PRIOR, LINEFIT_TERM, POLY_TERM


def test_validation():
    from bipymc_b200 import targets
    good = np.ones((3, 40, 2))
    with pytest.raises(ValueError, match="str"):
        targets.CudaSumLikelihoodSet(b"x", 2, good)
    with pytest.raises(ValueError, match="dim"):
        targets.CudaSumLikelihoodSet(POLY_TERM, 0, good)
    for bad in (np.ones(4), np.ones((0, 4)), np.ones((3, 0)), np.ones((3, 4, 0)), np.ones((0, 4, 2)),
                np.ones((2, 2, 2, 2)), np.float64(1.0)):
        with pytest.raises(ValueError, match="shape"):
            targets.CudaSumLikelihoodSet(POLY_TERM, 2, bad)
    with pytest.raises(ValueError, match="finite"):
        targets.CudaSumLikelihoodSet(POLY_TERM, 2, np.array([[[1.0], [np.inf]]]))
    with pytest.raises(ValueError, match="finite"):
        targets.CudaSumLikelihoodSet(POLY_TERM, 2, np.array([[1.0, np.nan]]))
    lik = targets.CudaSumLikelihoodSet(POLY_TERM, 2, good, prior=True, fmad=False)
    assert lik.n_problems == 3 and lik.dim == 2 and lik.prior and not lik.fmad
    assert lik.data.shape == (3, 40, 2) and lik.data.flags.c_contiguous and lik.data.dtype == np.float64
    # (P, M) is k = 1, as a 1-D array is for CudaSumLikelihood
    assert targets.CudaSumLikelihoodSet(POLY_TERM, 2, np.ones((5, 7))).data.shape == (5, 7, 1)
    assert not targets.CudaSumLikelihoodSet(POLY_TERM, 2, good).prior


def test_sizes_of_2_to_the_31_are_refused():
    """The limits are checked on the shape alone (a broadcast view: no memory behind it)."""
    from bipymc_b200 import targets
    for shape in ((2 ** 31, 1, 1), (1, 2 ** 31, 1)):
        with pytest.raises(ValueError, match="2\\^31"):
            targets.CudaSumLikelihoodSet._shaped(np.broadcast_to(np.float64(1.0), shape))


SOURCES = {"linefit": (LINEFIT_TERM, LINEFIT_PRIOR, 3), "expfit": (EXPFIT_TERM, EXPFIT_PRIOR, 5),
           "poly_d2": (POLY_TERM, None, 2), "poly_d3": (POLY_TERM, None, 3), "poly_d5": (POLY_TERM, None, 5)}


@pytest.mark.parametrize("name", sorted(SOURCES))
def test_sources_compile_for_sm100a(name):
    from bipymc_b200 import targets
    term, prior_src, dim = SOURCES[name]
    data = np.random.RandomState(0).rand(4, 300, 3)
    for prior in ((False, True) if prior_src else (False,)):
        for fmad in (True, False):
            src = term + (prior_src if prior else "")
            lik = targets.CudaSumLikelihoodSet(src, dim, data, prior=prior, fmad=fmad)
            lik.compile()
            assert lik.compile() is True      # the second compile comes from the process cache


def test_compile_error_carries_user_line_numbers():
    from bipymc_b200 import targets
    src = ("__device__ double ln_like_term(const double* theta, const double* row) {\n"
           "  double a = theta[0];\n"
           "  return a * row[0] + undefined_name;\n"
           "}\n")
    with pytest.raises(targets.CudaCompileError) as e:
        targets.CudaSumLikelihoodSet(src, 2, np.ones((3, 10))).compile()
    assert "ln_like.cu(3)" in e.value.log and "undefined_name" in e.value.log
    with pytest.raises(targets.CudaCompileError, match="ln_prior"):
        targets.CudaSumLikelihoodSet(LINEFIT_TERM, 3, np.ones((3, 10, 3)), prior=True).compile()


def test_cache_key_has_problems_rows_row_length_and_prior_not_values():
    from bipymc_b200 import targets
    src = LINEFIT_TERM + LINEFIT_PRIOR + "// sum set cache key %d\n" % np.random.randint(1 << 30)
    rows = np.ones((5, 100, 3))

    def fresh(cls=targets.CudaSumLikelihoodSet, **kw):
        args = dict(source=src, dim=3, data=rows, prior=False, fmad=True)
        args.update(kw)
        return cls(**args).compile() is False

    assert fresh()
    assert not fresh()                                        # same key: from the cache
    assert not fresh(data=2.0 * rows)                         # the values are not part of the key
    assert fresh(data=np.ones((6, 100, 3)))                   # P
    assert fresh(data=np.ones((5, 101, 3)))                   # M
    assert fresh(data=np.ones((5, 100, 4)))                   # k
    assert fresh(prior=True)
    assert fresh(fmad=False)
    # the single-problem sum module of the same source and rows is another module
    assert fresh(cls=targets.CudaSumLikelihood, data=rows[0])


def test_entry_points_refuse_bad_sizes_and_a_null_handle():
    from bipymc_b200 import _lib
    lib = _lib.load()
    log = C.create_string_buffer(1024)
    src = POLY_TERM.encode()
    for args, word in (((src, 2, 0, 3, 4), b"n_rows"), ((src, 2, 2 ** 31, 3, 4), b"n_rows"),
                       ((src, 2, 10, 0, 4), b"row_len"), ((src, 2, 10, 3, 0), b"n_problems"),
                       ((src, 0, 10, 3, 4), b"dim"), ((None, 2, 10, 3, 4), b"null source"),
                       ((b"__device__ double f() { return 0.0; }", 2, 10, 3, 4), b"ln_like_term")):
        assert lib.bpm_jit_compile_sum_problems(*(args + (1, None, log, 1024))) != 0, args
        err = lib.bpm_last_error()
        assert word in err and b"CUDA sum likelihood set" in err, (args, err)
    data = np.ones(30)
    assert lib.bpm_set_jit_sum_problems_target(None, src, _lib.dptr(data), 10, 3, 1, None, log, 1024) != 0
    assert b"null handle" in lib.bpm_last_error()


def _set(P=3):
    from bipymc_b200 import targets
    return targets.CudaSumLikelihoodSet(POLY_TERM, 2, np.ones((P, 30, 3)))


@pytest.mark.parametrize("kw, match", [(dict(subpop_k=5), "subpop_k"), (dict(outlier_gen=10), "outlier_gen"),
                                       (dict(ln_like_batched=lambda t: t[:, 0]), "ln_like_batched"),
                                       (dict(device_init=True), "device_init")])
def test_multi_problem_sampler_refuses(kw, match):
    """Refused in the constructor, before any device is touched."""
    from bipymc_b200 import DeMcMpi, DreamMpi
    for cls in (DeMcMpi, DreamMpi):
        with pytest.raises(ValueError, match=match) as e:
            cls(None, np.zeros(2), n_chains=8, ln_like_cuda=_set(), **kw)
        assert "CudaSumLikelihoodSet" in str(e.value)


def test_seed_sequence_rules():
    from bipymc_b200 import DreamMpi, targets
    with pytest.raises(ValueError, match="CudaSumLikelihoodSet"):
        DreamMpi(None, np.zeros(2), n_chains=8, seed=[1, 2],
                 ln_like_cuda=targets.CudaSumLikelihood(POLY_TERM, 2, np.ones((30, 3))))
    with pytest.raises(ValueError, match="2 keys for 3 problems"):
        DreamMpi(None, np.zeros(2), n_chains=8, seed=[1, 2], ln_like_cuda=_set(3))


def test_serial_demc_refuses_a_sum_likelihood_set():
    from bipymc_b200 import DeMc
    with pytest.raises(NotImplementedError, match="CudaSumLikelihoodSet"):
        DeMc(None, n_chains=8, ln_like_cuda=_set())
