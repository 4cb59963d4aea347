"""Error conventions and boundary sizes of the drop-in classes (SURVEY.md section 8b):
the reference's assertions / exceptions, the numpy NaN-alpha ValueError, zero-generation
calls, the smallest legal population, odd populations, misspelt kwargs, repeated run_mcmc
calls, and the C-ABI's argument checks."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def test_reference_assertions_and_messages():
    from bipymc_b200 import DeMcMpi, DreamMpi, McmcChain, targets
    t = targets.Banana_2D()
    with pytest.raises(AssertionError):                       # samplers.py:249
        DeMcMpi(t.ln_like, [0.0, 0.0], n_chains=3)
    with pytest.raises(ValueError):
        DreamMpi(t.ln_like, [0.0, 0.0], n_chains=8, del_pairs=9)
    with pytest.raises(ValueError):
        DreamMpi(t.ln_like, [0.0, 0.0], n_chains=8, n_cr=17)
    with pytest.raises(ValueError):                           # target / theta_0 dimension mismatch
        DreamMpi(t.ln_like, [0.0, 0.0, 0.0], n_chains=8)
    c = McmcChain(np.zeros(3), varepsilon=0.0)
    with pytest.raises(AssertionError):                       # chain.py:53 shape check of the setter
        c.chain = np.zeros((4, 2))


@pytest.mark.parametrize("fused", [2, 6])
def test_unknown_fused_mode_is_refused(fused):
    """bpm_set_fused accepts 0, 1, 3 and 5 only (include/bipymc_b200.h: BPM_FUSED_*); any other value raises
    instead of silently running the default kernels."""
    from bipymc_b200 import DreamMpi, targets, _lib
    with pytest.raises(_lib.BpmError, match="bpm_set_fused"):
        DreamMpi(targets.Banana_2D().ln_like, [0.0, 0.0], n_chains=8, seed=1, fused=fused)


def test_nan_alpha_raises_numpy_value_error():
    """lnL(cur) = lnL(prop) = -inf gives alpha = NaN; numpy's choice raises
    ValueError("probabilities contain NaN") at samplers.py:336 -- so does the device path."""
    from bipymc_b200 import DeMcMpi, targets
    t = targets.LineFit()
    np.random.seed(0)
    s = DeMcMpi(t.ln_like, [3.0, 4.5, 0.2], n_chains=8, seed=1, varepsilon=1e-6)   # m = 3 is outside the prior box
    with pytest.raises(ValueError, match="probabilities contain NaN"):
        s.run_mcmc(8 * 3)


def test_minus_inf_proposals_are_rejected_not_errors():
    from bipymc_b200 import DreamMpi, targets
    t = targets.LineFit()
    np.random.seed(0)
    s = DreamMpi(t.ln_like, [0.45, 4.5, 0.2], n_chains=16, seed=1, varepsilon=1e-4)   # hugging the m < 0.5 wall
    s.run_mcmc(16 * 200)
    x = s._X[:, :3].cpu().numpy()
    assert np.all(x[:, 0] < 0.5) and np.all(np.isfinite(s._lnl.cpu().numpy()))


@pytest.mark.parametrize("n_chains", [4, 5, 7])
def test_smallest_and_odd_populations(n_chains):
    from bipymc_b200 import DreamMpi, DeMcMpi, targets
    t = targets.Banana_2D()
    for cls in (DeMcMpi, DreamMpi):
        kw = dict(del_pairs=1) if (cls is DreamMpi and n_chains < 6) else {}
        np.random.seed(1)
        s = cls(t.ln_like, [0.0, 0.0], n_chains=n_chains, seed=2, varepsilon=0.1, **kw)
        s.run_mcmc(n_chains * 51)
        assert s.am_chains[0].chain_len == 51 and len(s.am_chains) == n_chains
        assert s.n_accepted + s.n_rejected == n_chains * 50 + 1
        sc = s.super_chain
        assert sc.shape == (n_chains * 51, 2) and np.all(np.isfinite(sc))


def test_zero_generation_calls_and_repeated_runs():
    from bipymc_b200 import DreamMpi, targets
    t = targets.Banana_2D()
    np.random.seed(3)
    s = DreamMpi(t.ln_like, [0.0, 0.0], n_chains=10, seed=4, varepsilon=0.1, suffle=True)   # misspelt kwarg ignored
    x0 = s._X.clone()
    for n in (0, 5, 10):                                      # n <= n_chains: the reference's loop body never runs
        s.run_mcmc(n)
        assert s.am_chains[0].chain_len == 1 and (s._X == x0).all()
        assert s.n_accepted == 0 and s.n_rejected == 1        # demc.py:19-20 counters of an empty run
    s.run_mcmc(10 * 4)
    s.run_mcmc(10 * 6, shuffle=False, flip=2.0)               # flip clipped to [0, 1] (demc.py:73)
    assert s.am_chains[9].chain_len == 1 + 3 + 5
    assert s.n_accepted + s.n_rejected == 10 * 5 + 1          # counters restart every call
    m, sd, sl = s.param_est(n_burn=20)
    assert sl.shape == (90 - 20, 2)
    assert s.in_burnin is True and s.chain is s.am_chains[0]
    assert np.array_equal(s.current_pos, s.am_chains[0].chain[-1])


def test_c_abi_argument_checks():
    from bipymc_b200 import _lib
    lib = _lib.load()
    h = C.c_void_p()
    cfg = _lib.Config(algo=1, n_chains=3, dim=2, ld=2, del_pairs=3, n_cr=3, burnin_gen=0, n_cr_gen=0,
                      shuffle=1, chain_lo=0, chain_hi=3, device=0, gamma_scale=1.0, flip=0.5, epsilon=0.0,
                      u_epsilon=0.0, gamma=0.0, seed=1)
    assert lib.bpm_create(C.byref(cfg), C.byref(h)) != 0 and b"n_chains" in lib.bpm_last_error()
    cfg.n_chains, cfg.chain_hi, cfg.algo = 8, 8, 7
    assert lib.bpm_create(C.byref(cfg), C.byref(h)) != 0 and b"algo" in lib.bpm_last_error()
    cfg.algo, cfg.chain_lo = 1, 8
    assert lib.bpm_create(C.byref(cfg), C.byref(h)) != 0 and b"shard" in lib.bpm_last_error()
    cfg.chain_lo = 0
    assert lib.bpm_create(C.byref(cfg), C.byref(h)) == 0
    st = _lib.State()
    assert lib.bpm_step_generations(h, C.byref(st), 0, 1, None) != 0           # no X / lnl
    assert lib.bpm_propose(h, C.byref(st), 0, None, None, None) != 0           # outside a generation
    assert lib.bpm_set_peers(h, None, 3) != 0 and lib.bpm_set_peers(h, None, 0) == 0
    bad = (C.c_double * 4)(1.0, 2.0, 3.0, 4.0)
    assert lib.bpm_set_target(h, _lib.TARGET_BANANA, bad, 4) != 0
    assert lib.bpm_set_target(h, 99, bad, 4) != 0
    assert lib.bpm_destroy(h) == 0 and lib.bpm_destroy(None) == 0
