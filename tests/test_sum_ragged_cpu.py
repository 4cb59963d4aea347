"""Per-observation likelihoods for datasets of different lengths in one sampler (targets.CudaSumLikelihoodSet given
a list of arrays), the parts that need no GPU: validation, the equal-length list as the rectangular set, the ragged
translation unit (P, k and the prior in the cache key, the row counts not), BPM_NROWS left undefined, the C-ABI
refusals that need no device and the sampler refusals."""
import ctypes as C

import numpy as np
import pytest

from test_cuda_sum_likelihood_cpu import LINEFIT_PRIOR, LINEFIT_TERM, POLY_TERM
from test_sum_problems_cpu import SOURCES


def _rows(lengths, k=3, seed=0):
    rs = np.random.RandomState(seed)
    return [rs.rand(m, k) for m in lengths]


def test_ragged_form():
    from bipymc_b200 import targets
    parts = _rows([5, 300, 1], k=2)
    lik = targets.CudaSumLikelihoodSet(POLY_TERM, 2, parts, prior=True, fmad=False)
    assert lik.n_problems == 3 and lik.dim == 2 and lik.prior and not lik.fmad
    assert lik.data.shape == (306, 2) and lik.data.flags.c_contiguous and lik.data.dtype == np.float64
    np.testing.assert_array_equal(lik.data, np.concatenate(parts))
    assert lik.n_rows.dtype == np.int64 and lik.n_rows.tolist() == [5, 300, 1]
    # 1-D arrays are k = 1, and a tuple is a sequence too
    lik = targets.CudaSumLikelihoodSet(POLY_TERM, 2, (np.ones(4), np.ones(9)))
    assert lik.data.shape == (13, 1) and lik.n_rows.tolist() == [4, 9] and lik.n_problems == 2


def test_equal_lengths_are_the_rectangular_set():
    from bipymc_b200 import targets
    parts = _rows([40, 40, 40])
    src = POLY_TERM + "// equal-length list %d\n" % np.random.randint(1 << 30)
    lik = targets.CudaSumLikelihoodSet(src, 3, parts)
    assert lik.n_rows is None and lik.n_problems == 3
    assert lik.data.shape == (3, 40, 3)
    np.testing.assert_array_equal(lik.data, np.stack(parts))
    assert lik.compile() is False
    assert targets.CudaSumLikelihoodSet(src, 3, np.stack(parts)).compile() is True     # the ndarray's cache entry
    # nested lists that np.asarray takes keep their meaning
    assert targets.CudaSumLikelihoodSet(POLY_TERM, 2, [[1.0, 2.0], [3.0, 4.0]]).data.shape == (2, 2, 1)
    assert targets.CudaSumLikelihoodSet(POLY_TERM, 2, [np.ones(3)]).data.shape == (1, 3, 1)


def test_refusals():
    from bipymc_b200 import targets
    for bad, match in (([], "empty"), ((), "empty"),
                       ([np.ones((3, 2)), np.ones((0, 2))], "data\\[1\\] has 0 rows"),
                       ([np.ones(3), np.ones(0)], "data\\[1\\] has 0 rows"),
                       ([np.ones((3, 2)), np.ones((4, 3))], "same k"),
                       ([np.ones((3, 2)), np.ones((4, 1, 2))], "data\\[1\\] must have shape"),
                       ([np.ones((3, 2)), np.float64(1.0)], "data\\[1\\] must have shape"),
                       ([np.ones((3, 0)), np.ones((4, 0))], "data\\[0\\] must have shape"),
                       ([np.ones((3, 2)), np.array([[1.0, np.nan]])], "finite"),
                       ([np.ones(3), np.array([np.inf, 1.0])], "finite")):
        with pytest.raises(ValueError, match=match):
            targets.CudaSumLikelihoodSet(POLY_TERM, 2, bad)
    with pytest.raises(ValueError, match="str"):
        targets.CudaSumLikelihoodSet(b"x", 2, _rows([3, 4]))
    with pytest.raises(ValueError, match="dim"):
        targets.CudaSumLikelihoodSet(POLY_TERM, 0, _rows([3, 4]))


def test_rows_of_2_to_the_31_are_refused():
    """Checked on the shape alone (a broadcast view: no memory behind it)."""
    from bipymc_b200 import targets
    with pytest.raises(ValueError, match="2\\^31"):
        targets.CudaSumLikelihoodSet(POLY_TERM, 2, [np.ones((3, 1)), np.broadcast_to(np.float64(1.0), (2 ** 31, 1))])


@pytest.mark.parametrize("name", sorted(SOURCES))
def test_sources_compile_for_sm100a(name):
    from bipymc_b200 import targets
    term, prior_src, dim = SOURCES[name]
    parts = _rows([300, 17, 1000, 1])
    for prior in (False, True) if prior_src else (False,):
        for fmad in (True, False):
            src = term + (prior_src if prior else "")
            lik = targets.CudaSumLikelihoodSet(src, dim, parts, prior=prior, fmad=fmad)
            assert lik.n_rows is not None
            lik.compile()
            assert lik.compile() is True      # the second compile comes from the process cache


def test_cache_key_has_problems_row_length_and_prior_not_row_counts_or_values():
    from bipymc_b200 import targets
    src = LINEFIT_TERM + LINEFIT_PRIOR + "// ragged cache key %d\n" % np.random.randint(1 << 30)
    parts = _rows([100, 7, 300])

    def fresh(**kw):
        args = dict(source=src, dim=3, data=parts, prior=False, fmad=True)
        args.update(kw)
        return targets.CudaSumLikelihoodSet(**args).compile() is False

    assert fresh()
    assert not fresh()                                            # same key: from the cache
    assert not fresh(data=[2.0 * a for a in parts])               # the values are not part of the key
    assert not fresh(data=_rows([5, 60000, 1]))                   # nor the row counts
    assert fresh(data=_rows([100, 7, 300, 2]))                    # P
    assert fresh(data=_rows([100, 7, 300], k=4))                  # k
    assert fresh(prior=True)
    assert fresh(fmad=False)
    # the rectangular set of the same source is another module
    assert fresh(data=_rows([100, 100, 100]))


def test_bpm_nrows_is_not_defined():
    from bipymc_b200 import targets
    src = ("__device__ double ln_like_term(const double* theta, const double* row) {\n"
           "  double a = theta[0];\n"
           "  return a * row[0] / BPM_NROWS;\n"
           "}\n")
    with pytest.raises(targets.CudaCompileError) as e:
        targets.CudaSumLikelihoodSet(src, 2, _rows([3, 10])).compile()
    assert "ln_like.cu(3)" in e.value.log and "BPM_NROWS" in e.value.log
    # the macros it does define
    ok = ("__device__ double ln_like_term(const double* theta, const double* row) {\n"
          "  return theta[0] * row[BPM_ROWLEN - 1] + BPM_NPROBLEMS + BPM_DIM;\n"
          "}\n")
    targets.CudaSumLikelihoodSet(ok, 2, _rows([3, 10])).compile()
    # the rectangular set still has it
    targets.CudaSumLikelihoodSet(src, 2, _rows([10, 10])).compile()


def test_entry_points_refuse_bad_sizes_and_a_null_handle():
    from bipymc_b200 import _lib
    lib = _lib.load()
    log = C.create_string_buffer(1024)
    src = POLY_TERM.encode()
    for args, word in (((src, 2, 0, 4), b"row_len"), ((src, 2, (1 << 20) + 1, 4), b"row_len"),
                       ((src, 2, 3, 0), b"n_problems"), ((src, 0, 3, 4), b"dim"), ((None, 2, 3, 4), b"null source"),
                       ((b"__device__ double f() { return 0.0; }", 2, 3, 4), b"ln_like_term")):
        assert lib.bpm_jit_compile_sum_ragged(*(args + (1, None, log, 1024))) != 0, args
        err = lib.bpm_last_error()
        assert word in err and b"CUDA sum likelihood set" in err, (args, err)
    data = np.ones(30)
    rows = np.array([4, 6], dtype=np.int64)
    assert lib.bpm_set_jit_sum_ragged_target(None, src, _lib.dptr(data), rows.ctypes.data_as(C.POINTER(C.c_int64)),
                                             3, 1, None, log, 1024) != 0
    assert b"null handle" in lib.bpm_last_error()


def _set(P=3):
    from bipymc_b200 import targets
    return targets.CudaSumLikelihoodSet(POLY_TERM, 2, _rows([30 + g for g in range(P)]))


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


def test_seed_sequence_and_serial_demc():
    from bipymc_b200 import DeMc, DreamMpi
    with pytest.raises(ValueError, match="2 keys for 3 problems"):
        DreamMpi(None, np.zeros(2), n_chains=8, seed=[1, 2], ln_like_cuda=_set(3))
    with pytest.raises(NotImplementedError, match="CudaSumLikelihoodSet"):
        DeMc(None, n_chains=8, ln_like_cuda=_set())
