"""Native-stream parity (device step == oracle replay of the dumped draws, 1e-12) for the code paths of the
default fused Gaussian kernel that the golden / headline configurations do not reach:
  * the run-time-general proposal stage (DREAM with del_pairs != 3, DE-MC) at d = 100, several tiles;
  * a target with a non-zero mean (the CENTER instantiation of the tile product).
Runs last (file name) so that a regression here does not mask the main parity suite under `pytest -x`."""
import numpy as np
import pytest
from scipy.stats import multivariate_normal

from oracle import targets as otargets
from test_native_gpu import _native_vs_oracle

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("del_pairs,n_cr", [(1, 3), (2, 5), (5, 2)])
def test_native_dream_gauss100_other_pair_counts(del_pairs, n_cr):
    from bipymc_b200 import DreamMpi, targets
    np.random.seed(11)
    s = DreamMpi(targets.Gauss_100D().ln_like, np.zeros(100), n_chains=150, n_cr_gen=2, burnin_gen=1000,
                 seed=5, fused=1, varepsilon=0.5, del_pairs=del_pairs, n_cr=n_cr)
    _native_vs_oracle(s, otargets.GaussND(dim=100).ln_like, gens=6, k0=2)


def test_native_demc_gauss100_several_tiles():
    from bipymc_b200 import DeMcMpi, targets
    np.random.seed(12)
    s = DeMcMpi(targets.Gauss_100D().ln_like, np.zeros(100), n_chains=150, seed=6, fused=1, varepsilon=0.5)
    _native_vs_oracle(s, otargets.GaussND(dim=100).ln_like, gens=12, k0=5, run_kwargs=dict(epsilon=1e-9))


@pytest.mark.parametrize("dim", [40, 100])
def test_native_dream_gauss_with_nonzero_mean(dim):
    from bipymc_b200 import DreamMpi, targets
    rs = np.random.RandomState(3)
    mean = rs.randn(dim)
    t = targets.Gauss_100D(dim=dim, mean=mean)
    rv = multivariate_normal(mean, t.cov)

    def oracle_lnl(y):
        with np.errstate(divide="ignore"):
            return np.log(rv.pdf(y))

    np.random.seed(13)
    s = DreamMpi(t.ln_like, mean, n_chains=130, n_cr_gen=2, burnin_gen=1000, seed=8, fused=1, varepsilon=0.5)
    _native_vs_oracle(s, oracle_lnl, gens=6, k0=2)


# ---- RNG-replay parity against the second batch of golden vectors (oracle/cases.py: EXTRA_CASES) --------
@pytest.mark.parametrize("fused", [1, 0, 3, 5], ids=["fused", "split", "fused-ws12", "fused-v3"])
@pytest.mark.parametrize("name", sorted(__import__("oracle.cases", fromlist=["EXTRA_CASES"]).EXTRA_CASES))
def test_replay_extra_golden_cases(name, fused):
    """Includes gauss100_dream_tiles: 136 chains at d = 100, i.e. one full 64-chain tile plus a partial tile per
    half-phase of the fused kernel (the other 100-D goldens hold 8-12 chains)."""
    from test_replay_parity_gpu import replay_and_check
    replay_and_check(name, fused)


# ---- d <= 4: the fused one-thread-per-chain kernel against the split path ----------------------------------------
@pytest.mark.parametrize("target,n_chains,algo", [("banana", 1000, "dream"), ("dblgauss", 4099, "dream"),
                                                   ("linefit", 2500, "dream"), ("banana", 777, "demc"),
                                                   ("linefit", 33, "dream"), ("banana", 310000, "dream"),
                                                   ("dblgauss", 2049, "demc"), ("linefit", 1500, "demc")])
def test_small_d_fused_kernel_equals_split_path(target, n_chains, algo):
    """fused=1 (default): one fused_small_kernel launch per half-phase over the chain-ordered packed lists, after
    the split and list-packing kernels.  fused=0 launches split / propose / likelihood / accept / CR reduction per
    generation.  Same seed: identical histories, cached likelihoods, counters, running moments and -- the CR block
    partials are summed in the same order -- bit-identical p_cr.  The populations cover a partly filled single
    warp (33), one chain past a list-packing block (2049), the CR reduction at its cap of 148 blocks (310000) and
    DE-MC on every d <= 4 target."""
    import ctypes as C
    import torch
    from bipymc_b200 import DreamMpi, DeMcMpi, targets, _lib
    tgt = {"banana": targets.Banana_2D, "dblgauss": targets.BimodeGauss_2D, "linefit": targets.LineFit}[target]()
    th0 = [-0.8, 4.5, 0.2] if target == "linefit" else [0.0, 0.0]
    G = 37
    runs = []
    eps = 1e-2 if target == "linefit" else 0.3
    for f in (1, 0):
        np.random.seed(21)
        if algo == "dream":
            s = DreamMpi(tgt.ln_like, th0, n_chains=n_chains, seed=9, varepsilon=eps, n_cr_gen=3, burnin_gen=30,
                         fused=f)
        else:
            s = DeMcMpi(tgt.ln_like, th0, n_chains=n_chains, seed=9, varepsilon=eps, fused=f)
        _lib.check(s._libh.bpm_profile(s._handle, 1))
        s.run_mcmc(n_chains * (G + 1), flip=0.3)
        ms, n = (C.c_double * 8)(), (C.c_int64 * 8)()
        _lib.check(s._libh.bpm_profile_read(s._handle, ms, n))
        runs.append((s, [int(v) for v in n]))
    (a, ka), (b, kb) = runs
    assert ka[4] == 2 * G and ka[1] == 0 and ka[0] == G, ka
    assert kb[4] == 0 and kb[1] == 2 * G and kb[0] == G, kb
    assert torch.equal(a._hist.tensor(), b._hist.tensor())
    assert torch.equal(a._lnl, b._lnl) and torch.equal(a._X, b._X)
    assert torch.equal(a._mean, b._mean) and torch.equal(a._m2, b._m2)
    assert (a.n_accepted, a.n_rejected) == (b.n_accepted, b.n_rejected)
    if algo == "dream":
        assert np.array_equal(a.p_cr, b.p_cr) and np.array_equal(a.delta_m, b.delta_m)
        assert np.array_equal(a.n_cr_updates, b.n_cr_updates) and a.n_cr_updates.sum() > 0
