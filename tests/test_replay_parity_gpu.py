"""RNG-replay parity on the GPU: the CUDA generation step, fed the numpy draws the
reference consumed, must reproduce the reference's accept decisions step for step and
its chain states to 1e-12 relative (fp64) -- checked against the committed golden
histories written by the unmodified reference (tests/golden/ref_*.npz) and against the
oracle's per-step trace."""
import os
import warnings

import numpy as np
import pytest

from oracle.cases import ALL_CASES, CASES, oracle_target
from oracle.demc_dream import OracleSampler

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
RTOL = 1e-12        # north_star: chain states within 1e-12 relative


def device_target(name):
    from bipymc_b200 import targets
    if name == "banana":
        return targets.Banana_2D(sigma1=1.0, sigma2=1.0)
    if name == "dblgauss":
        return targets.BimodeGauss_2D()
    if name.startswith("gauss"):
        return targets.Gauss_100D(dim=int(name[5:]))
    if name == "linefit":
        return targets.LineFit()
    raise KeyError(name)


def oracle_traces(name):
    case = ALL_CASES[name]
    fn, kw = oracle_target(case["target"])
    np.random.seed(case["seed"])
    s = OracleSampler(fn, case["theta_0"], n_chains=case["n_chains"], algo=case["algo"],
                      ln_kwargs=kw, **case["ctor_kwargs"])
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        tr = s.run(case["n"], record=True, **case["run_kwargs"])
    return s, tr


def make_sampler(name, mode, fused=True):
    from bipymc_b200 import DeMcMpi, DreamMpi
    case = ALL_CASES[name]
    cls = DreamMpi if case["algo"] == "dream" else DeMcMpi
    np.random.seed(case["seed"])
    kw = dict(case["ctor_kwargs"])
    ln_kwargs = {}
    if mode == "device":
        fn = device_target(case["target"]).ln_like
    elif mode == "scalar":
        fn, ln_kwargs = oracle_target(case["target"])        # plain Python callable
    elif mode == "batched":
        import torch
        tgt = device_target(case["target"])
        fn = tgt.ln_like

        def batched(theta):                                   # torch in, torch out
            host = theta.cpu().numpy()
            return torch.tensor([float(tgt.ln_like(r)) for r in host], dtype=torch.float64,
                                device=theta.device)
        kw["ln_like_batched"] = batched
        fn = lambda th: tgt.ln_like(th)                       # noqa: E731  hides device_target()
    return cls(fn, np.asarray(case["theta_0"], dtype=float), n_chains=case["n_chains"],
               ln_kwargs=ln_kwargs, fused=fused, **kw)


def check_against_reference(name, s, sink, traces, osampler):
    case = ALL_CASES[name]
    g = np.load(os.path.join(GOLD, "ref_%s.npz" % name))
    ref = g["history"]
    hist = s._hist.tensor()[:, :, :s.dim].cpu().numpy()
    assert hist.shape == ref.shape
    # initial states come from the same numpy stream: exact
    assert np.array_equal(hist[0], ref[0])
    # accept decisions: step for step
    n_flip = 0
    for k, (got, tr) in enumerate(zip(sink, traces)):
        n_flip += int(np.count_nonzero(got["accept"] != tr["accept"]))
    assert n_flip == 0, "%d accept decisions differ from the reference" % n_flip
    err = np.abs(hist - ref) / np.maximum(1.0, np.abs(ref))
    assert err.max() <= RTOL, "max relative state error %.3e" % err.max()
    # proposals and their likelihoods, every step
    for got, tr in zip(sink, traces):
        perr = np.abs(got["prop"] - tr["prop"]) / np.maximum(1.0, np.abs(tr["prop"]))
        assert perr.max() <= RTOL
        fin = np.isfinite(tr["lnl_prop"])
        assert np.array_equal(np.isfinite(got["lnl_prop"]), fin) or case["target"] in ("banana", "dblgauss")
        both = fin & np.isfinite(got["lnl_prop"])
        lerr = np.abs(got["lnl_prop"][both] - tr["lnl_prop"][both])
        assert lerr.max() <= 1e-9 * np.maximum(1.0, np.abs(tr["lnl_prop"][both])).max()
    assert s.n_accepted == int(g["n_accepted"])
    assert s.n_rejected == int(g["n_rejected"])
    assert s.acceptance_fraction == float(g["acceptance_fraction"])
    if case["algo"] == "dream":
        np.testing.assert_allclose(s.p_cr, g["p_cr"], rtol=1e-10)
        np.testing.assert_allclose(s.delta_m, g["delta_m"], rtol=1e-10)
        assert np.array_equal(s.n_cr_updates, g["n_cr_updates"])
    mean, std, sl = s.param_est(n_burn=0)
    np.testing.assert_allclose(mean, g["mean"], rtol=1e-11, atol=1e-12)
    np.testing.assert_allclose(std, g["std"], rtol=1e-10, atol=1e-12)
    assert sl.shape == (ref.shape[0] * ref.shape[1], ref.shape[2])
    # McmcChain view = column of the history
    c = s.am_chains[1]
    assert c.global_id == 1 and np.array_equal(c.chain, hist[:, 1, :])
    assert np.array_equal(c.current_pos, hist[-1, 1, :]) and c.chain_len == ref.shape[0]


def launches_by_kind(s):
    """Launch counts the engine recorded since bpm_profile(h, 1): split, propose, likelihood, accept,
    fused half-phase, CR reduction (include/bipymc_b200.h: bpm_profile_read)."""
    import ctypes as C
    from bipymc_b200 import _lib
    ms, n = (C.c_double * 8)(), (C.c_int64 * 8)()
    _lib.check(s._libh.bpm_profile_read(s._handle, ms, n))
    return dict(zip(("split", "propose", "likelihood", "accept", "fused_phase", "cr_reduce"), [int(v) for v in n]))


def replay_and_check(name, fused):
    """Replay the reference's recorded draws through the device step with the full trace sink (accept
    flags, proposal likelihoods AND proposal vectors) and prove WHICH kernels ran: the fused ids must have
    launched one fused half-phase kernel per phase and no split-path kernel, the split id the opposite."""
    from bipymc_b200 import _lib
    osampler, traces = oracle_traces(name)
    s = make_sampler(name, "device", fused=fused)
    _lib.check(s._libh.bpm_profile(s._handle, 1))
    sink = []
    s.run_mcmc(ALL_CASES[name]["n"], _replay=traces, _trace=sink, **ALL_CASES[name]["run_kwargs"])
    k = launches_by_kind(s)
    _lib.check(s._libh.bpm_profile(s._handle, 0))
    gens = len(traces)
    if fused:
        assert k["fused_phase"] == 2 * gens and k["propose"] == 0 and k["accept"] == 0, k
    else:
        assert k["fused_phase"] == 0 and k["propose"] == 2 * gens and k["accept"] == 2 * gens, k
    check_against_reference(name, s, sink, traces, osampler)


@pytest.mark.parametrize("fused", [1, 0, 3, 5], ids=["fused", "split", "fused-ws12", "fused-v3"])
@pytest.mark.parametrize("name", sorted(CASES))
def test_replay_device_target(name, fused):
    replay_and_check(name, fused)


@pytest.mark.parametrize("mode", ["scalar", "batched"])
@pytest.mark.parametrize("name", ["banana_demc", "banana_dream_odd", "gauss7_dream_noshuffle",
                                  "linefit_dream"])
def test_replay_user_likelihoods(name, mode):
    """The reference's scalar ln_like_fn(theta, **kw) plug-in and the new batched torch
    plug-in go through bpm_propose / bpm_accept; with a host likelihood the result is the
    reference's to the last bit of the likelihood, so accept flags and states match."""
    osampler, traces = oracle_traces(name)
    s = make_sampler(name, mode)
    assert s._mode() == mode
    sink = []
    s.run_mcmc(ALL_CASES[name]["n"], _replay=traces, _trace=None, **ALL_CASES[name]["run_kwargs"])
    g = np.load(os.path.join(GOLD, "ref_%s.npz" % name))
    hist = s._hist.tensor()[:, :, :s.dim].cpu().numpy()
    err = np.abs(hist - g["history"]) / np.maximum(1.0, np.abs(g["history"]))
    assert err.max() <= RTOL
    assert s.n_accepted == int(g["n_accepted"]) and s.n_rejected == int(g["n_rejected"])


def test_c_abi_batched_callback_equals_torch_plugin():
    """bpm_set_batched_lnl: a C-ABI device-pointer callback (theta[n][ld], lnl[n], stream) drives
    whole generations inside bpm_step_generations; the chains must equal, bit for bit, those of
    the torch plug-in evaluating the same likelihood through bpm_propose / bpm_accept."""
    import ctypes as C
    import torch
    from bipymc_b200 import DreamMpi, _lib
    d, N, G = 6, 40, 15

    def lnl_torch(theta):                                    # isotropic Gaussian; explicit elementwise ops, so
        acc = theta[:, 0] * theta[:, 0]                      # the value does not depend on which reduction
        for i in range(1, theta.shape[1]):                   # kernel torch would pick
            acc = acc + theta[:, i] * theta[:, i]
        return -0.5 * acc

    np.random.seed(9)
    ref = DreamMpi(lambda th: float(-0.5 * np.sum(th ** 2)), np.zeros(d), n_chains=N, seed=21, varepsilon=1.0,
                   ln_like_batched=lnl_torch, n_cr_gen=3, burnin_gen=1000)
    assert ref._mode() == "batched"
    ref.run_mcmc(N * (G + 1))

    np.random.seed(9)
    s = DreamMpi(lambda th: float(-0.5 * np.sum(th ** 2)), np.zeros(d), n_chains=N, seed=21, varepsilon=1.0,
                 ln_like_batched=lnl_torch, n_cr_gen=3, burnin_gen=1000)
    calls = []

    def cb(theta_ptr, n, dim, ld, lnl_ptr, user, stream):
        class _A(object):
            pass
        a, b = _A(), _A()
        a.__cuda_array_interface__ = dict(shape=(n, ld), typestr="<f8", data=(int(theta_ptr), False), version=2)
        b.__cuda_array_interface__ = dict(shape=(n,), typestr="<f8", data=(int(lnl_ptr), False), version=2)
        th = torch.as_tensor(a, device=s._device)[:, :dim]
        out = torch.as_tensor(b, device=s._device)
        assert int(stream or 0) == torch.cuda.current_stream(s._device).cuda_stream   # the caller's stream
        out.copy_(lnl_torch(th))
        calls.append(n)
        return 0
    fn = _lib.LNL_FN(cb)
    _lib.check(s._libh.bpm_set_batched_lnl(s._handle, fn, None))
    _lib.check(s._libh.bpm_reset_counters(s._handle))
    _lib.check(s._libh.bpm_set_run_params(s._handle, *s._run_params({})))
    s._init_lnl()
    base, avail = s._hist.reserve(G)
    st = s._state(base)
    _lib.check(s._libh.bpm_step_generations(s._handle, C.byref(st), 0, G, s._stream()))
    s._hist.advance(G)
    torch.cuda.synchronize()
    assert len(calls) == 2 * G and sum(calls) == N * G       # one call per half-phase
    hs, hr = s._hist.tensor()[:, :, :d], ref._hist.tensor()[:, :, :d]     # (pad columns are never written)
    assert hs.shape == hr.shape, (hs.shape, hr.shape)
    bad = [(t, int((hs[t] != hr[t]).any(dim=1).sum())) for t in range(hs.shape[0]) if not torch.equal(hs[t], hr[t])]
    assert not bad, "generations with differing chains (t, n_rows): %r" % (bad[:5],)
    assert torch.equal(s._lnl, ref._lnl)
