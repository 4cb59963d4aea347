"""Run-time compiled likelihoods at the shapes the rest of the suite never runs, the parts that need no GPU.

  * a per-observation term that reads every column and every parameter (+ - * / only), its numpy
    restatement, and its compile for sm_100a at every (d, k, M) that test_jit_shapes_gpu.py uses;
  * sum_plan (csrc/engine.cu) restated in Python, and proof that the GPU cases reach each launch-shape
    branch of the sum kernels on a 148-SM B200;
  * the exact product split behind the high-precision reference of the GPU file.
The sources, cases and restatements here are shared with test_jit_shapes_gpu.py."""
import math

import numpy as np
import pytest

from test_cuda_sum_likelihood_cpu import CHUNK

B200_SMS = 148
STAGE_ROWLEN = 8        # csrc/kernels_sum.cuh: kSumSmemRowLen (longer rows are read from global memory)
WS_DOUBLES = 1 << 22    # csrc/engine.cu: kSumWsDoubles

# model = sum_q theta[q % d] * row[q % k] over q < max(d, k): every parameter and every column is read
ALLCOL_TERM = r'''
__device__ double ln_like_term(const double* theta, const double* row) {
  const int nq = BPM_DIM > BPM_ROWLEN ? BPM_DIM : BPM_ROWLEN;
  double model = 0.0;
  for (int q = 0; q < nq; ++q) model = model + theta[q % BPM_DIM] * row[q % BPM_ROWLEN];
  const double r = (row[BPM_ROWLEN - 1] - model) / 3.0;
  return -0.5 * (r * r);
}
'''
# outside the prior when theta[0] > 5: those chains evaluate no term and get -inf
ALLCOL_PRIOR = r'''
__device__ double ln_prior(const double* theta) { return theta[0] > 5.0 ? -INFINITY : 0.0; }
'''
# one rounding per product and one per difference (or one fused multiply-add): the term of the
# high-precision test, whose exact value is known (two_prod)
LIN_TERM = r'''
__device__ double ln_like_term(const double* theta, const double* row) {
  return theta[0] * row[0] - theta[1] * row[1];
}
'''

# a diagonal Gaussian: data = (mu[d], w[d]), ln L = -0.5 sum_q ((theta_q - mu_q) w_q)^2
GAUSS_DIAG = r'''
__device__ double ln_like(const double* t, const double* data) {
  double s = 0.0;
  for (int q = 0; q < BPM_DIM; ++q) {
    const double r = (t[q] - data[q]) * data[BPM_DIM + q];
    s = s + r * r;
  }
  return -0.5 * s;
}
'''


def gauss_diag_data(d, seed=0):
    rs = np.random.RandomState(100 + seed)
    return np.concatenate([rs.uniform(-1.0, 1.0, d), rs.uniform(0.5, 2.0, d)])


def allcol_terms_np(theta, data):
    """ALLCOL_TERM in numpy, the same operations in the same order (every one rounded: fmad=False)."""
    d, k = len(theta), data.shape[1]
    model = np.zeros(data.shape[0])
    for q in range(max(d, k)):
        model = model + theta[q % d] * data[:, q % k]
    r = (data[:, k - 1] - model) / 3.0
    return -0.5 * (r * r)


def allcol_data(M, k, seed=0):
    return np.random.RandomState(seed + 1000 * k).uniform(-1.0, 1.0, (M, k))


def sum_plan(n, M, n_sms=B200_SMS):
    """csrc/engine.cu: sum_plan for n rows of theta and M observations: (tile, log2_group, n_groups,
    log2_groups)."""
    nch = -(-M // CHUNK)
    lp2 = (nch - 1).bit_length()
    target = 8 * n_sms
    tile = 64
    while tile > 8 and -(-n // tile) * nch < target:
        tile //= 2
    tiles = -(-n // tile)

    def groups(lg):
        return (nch + (1 << lg) - 1) >> lg

    lg = lp2
    while lg > 0 and tiles * groups(lg) < target:
        lg -= 1
    while lg < lp2 and (n * groups(lg) > WS_DOUBLES or groups(lg) > 65535):
        lg += 1
    return tile, lg, groups(lg), lp2 - lg


def stage_chunks(k):
    """csrc/kernels_sum.cuh: sum_stage_chunks."""
    return 4 if k <= 2 else (2 if k <= 4 else 1)


def plan_branches(n, M, k):
    """The launch-shape branches of lnl_sum_kernel / lnl_sum_finish_kernel that (n, M, k) takes."""
    tile, lg, n_groups, lgs = sum_plan(n, M)
    out = {"tile%d" % tile}
    out.add("one_group" if n_groups == 1 else ("groups_le32" if lgs <= 5 else "groups_gt32"))
    if lgs > 5 and n_groups % (1 << (lgs - 5)):
        out.add("finish_partial_lane_block")        # the last lane's block of B = 2^(lgs - 5) leaves is partly filled
    out.add("staged" if k <= STAGE_ROWLEN else "unstaged")
    if k <= STAGE_ROWLEN and (1 << lg) < stage_chunks(k):
        out.add("group_below_stage")                 # G < kSumStageChunks: fewer chunks staged than the stage holds
    return out


# Part A of the GPU file: (k, d, M, batch sizes, prior).  Every row length crosses a staging boundary
# (k = 2 | 4 | 5 | 8 | 9) or is far past it (17); d = 32 / 33 is the register / pointer SumTheta boundary.
SUM_CASES = [
    (1, 1, 100003, (1, 7, 4096), False),
    (2, 4, 3000, (1, 7, 4096), False),
    (4, 32, 5 * CHUNK + 3, (1, 7, 4096), False),
    (5, 33, 40000, (1, 7, 4096), False),
    (8, 100, CHUNK + 1, (1, 7, 80000), False),
    (9, 1, CHUNK, (1, 7, 4096), False),
    (9, 33, 70001, (1, 7, 4096), False),
    (17, 100, 5000, (1, 7, 4096), False),
    (3, 4, 100003, (1, 7, 4096), True),             # -inf prior inside CTA tiles, several groups
]

# Part C: d on both sides of each LPC boundary (csrc/engine.cu: pick_lpc 4 | 8 | 32)
ORACLE_DIMS = [5, 16, 17, 32, 33, 200]
ORACLE_SUM = [(5, 3, 600), (33, 3, 600)]            # (d, k, M) of the CudaSumLikelihood cases

# Part D: chains per problem (a warp spans many problems | 2 and 3 passes of the split scan | 3 CR blocks)
# and d (the fused kernel | LPC 8 | LPC 32, the kept-draws proposal)
D_CHAINS = [4, 5, 129, 257, 4099]
D_DIMS = [2, 20, 40]


def n_problems(n):
    """Problems of a part-D set with n chains each: many small ones, so that one warp spans several."""
    return 17 if n <= 5 else (3 if n < 4096 else 2)


def test_allcol_restatement_is_the_scalar_loop():
    rs = np.random.RandomState(1)
    for d, k in [(1, 1), (4, 9), (33, 5), (3, 17)]:
        theta, data = rs.randn(d), rs.randn(20, k)
        got = allcol_terms_np(theta, data)
        for i, row in enumerate(data):
            model = 0.0
            for q in range(max(d, k)):
                model = model + theta[q % d] * row[q % k]
            r = (row[k - 1] - model) / 3.0
            assert got[i] == -0.5 * (r * r)


@pytest.mark.parametrize("case", range(len(SUM_CASES)))
def test_sum_cases_compile_for_sm100a(case):
    from bipymc_b200 import targets
    k, d, M, _, prior = SUM_CASES[case]
    src = ALLCOL_TERM + (ALLCOL_PRIOR if prior else "")
    targets.CudaSumLikelihood(src, d, allcol_data(M, k), prior=prior, fmad=False).compile()


@pytest.mark.parametrize("d,k,M", ORACLE_SUM + [(2, 2, 100003), (2, 2, 3000)])
def test_oracle_and_precision_sum_sources_compile_for_sm100a(d, k, M):
    from bipymc_b200 import targets
    targets.CudaSumLikelihood(ALLCOL_TERM, d, allcol_data(M, k), fmad=False).compile()
    if d == 2:
        targets.CudaSumLikelihood(LIN_TERM, d, allcol_data(M, k)).compile()


@pytest.mark.parametrize("d", sorted(set(ORACLE_DIMS + D_DIMS)))
def test_gauss_diag_compiles_for_sm100a(d):
    from bipymc_b200 import targets
    data = gauss_diag_data(d)
    targets.CudaLikelihood(GAUSS_DIAG, d, data, fmad=False).compile()
    if d in D_DIMS:
        for n in D_CHAINS:
            targets.CudaLikelihoodSet(GAUSS_DIAG, d, np.stack([data] * n_problems(n)), fmad=False).compile()


def test_plan_restatement_by_hand():
    assert sum_plan(4096, 100003) == (64, 4, 25, 5)       # 391 chunks: 25 groups of 16
    assert sum_plan(1, 100003) == (8, 0, 391, 9)          # one chain: every chunk its own group
    assert sum_plan(80000, CHUNK + 1) == (64, 1, 1, 0)    # 1250 tiles fill the GPU: one group
    assert sum_plan(1, 1) == (8, 0, 1, 0)
    assert sum_plan(10 ** 6, 10 ** 6)[2] * 10 ** 6 <= WS_DOUBLES   # the workspace bound moves to larger groups


def test_gpu_cases_reach_every_plan_branch():
    reached = {}
    for k, d, M, batches, prior in SUM_CASES:
        for n in batches:
            for b in plan_branches(n, M, k):
                reached.setdefault(b, []).append((k, d, M, n))
    want = {"tile64", "tile8", "one_group", "groups_le32", "groups_gt32", "finish_partial_lane_block",
            "staged", "unstaged", "group_below_stage"}
    assert want <= set(reached), sorted(want - set(reached))
    for b in sorted(want):
        print("%-26s %s" % (b, reached[b][:4]))
    # the -inf prior case runs with several groups, and every row length stages 4 | 2 | 1 chunks or none
    k, d, M, batches, prior = SUM_CASES[-1]
    assert prior and sum_plan(max(batches), M)[2] > 1 and sum_plan(max(batches), M)[0] == 64
    assert {stage_chunks(c[0]) for c in SUM_CASES if c[0] <= STAGE_ROWLEN} == {1, 2, 4}
    assert {c[1] for c in SUM_CASES} >= {1, 4, 32, 33, 100}
    assert {c[0] for c in SUM_CASES} >= {1, 2, 4, 5, 8, 9, 17}


def two_prod(a, b):
    """a * b = p + e exactly (Dekker's product with Veltkamp's split; no overflow for |a|, |b| < 2^996)."""
    p = a * b

    def split(x):
        c = 134217729.0 * x          # 2^27 + 1
        hi = c - (c - x)
        return hi, x - hi

    ah, al = split(a)
    bh, bl = split(b)
    e = ((ah * bh - p) + ah * bl + al * bh) + al * bl
    return p, e


def lin_exact_sum(theta, data):
    """sum_i (theta0 x_i0 - theta1 x_i1), correctly rounded: every product is split exactly into two doubles
    and math.fsum adds the 4 M parts exactly, rounding once."""
    p0, e0 = two_prod(np.full(data.shape[0], theta[0]), data[:, 0])
    p1, e1 = two_prod(np.full(data.shape[0], theta[1]), data[:, 1])
    return math.fsum(np.concatenate([p0, e0, -p1, -e1]))


def test_two_prod_is_exact():
    import mpmath
    mpmath.mp.prec = 300
    rs = np.random.RandomState(5)
    a = rs.uniform(-1, 1, 2000) * 10.0 ** rs.uniform(-5, 5, 2000)
    b = rs.uniform(-1, 1, 2000) * 10.0 ** rs.uniform(-5, 5, 2000)
    p, e = two_prod(a, b)
    for i in range(a.size):
        assert mpmath.mpf(p[i]) + mpmath.mpf(e[i]) == mpmath.mpf(a[i]) * mpmath.mpf(b[i])
    data = np.stack([a, b], axis=1)[:700]
    exact = mpmath.fsum(mpmath.mpf(0.3) * mpmath.mpf(x) - mpmath.mpf(-0.7) * mpmath.mpf(y) for x, y in data)
    assert lin_exact_sum(np.array([0.3, -0.7]), data) == float(exact)
