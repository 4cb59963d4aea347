"""What a handle owns, it releases, and a refused call leaves it as it was.

Every device buffer of a handle is freed with it, however it was grown: the side stream of a multi-generation
call, the host entry, the diagnostics scratch, profiling, a replaced target, a multi-problem handle and the
workspace of a sum likelihood.  And a bpm_set_target that is refused changes nothing the next generations
compute."""
import ctypes as C

import numpy as np
import pytest
import torch

from bipymc_b200 import _lib, targets

pytestmark = pytest.mark.gpu

D, N = 100, 64
SET_SRC = """
__device__ double ln_like(const double* theta, const double* data) {
  double s = 0.0;
  for (int i = 0; i < BPM_DIM; ++i) { const double r = theta[i] - data[i % BPM_NDATA]; s += r * r; }
  return -0.5 * s;
}
"""
SUM_SRC = """
__device__ double ln_like_term(const double* theta, const double* row) {
  const double r = row[0] - theta[0] - theta[1];
  return -0.5 * r * r;
}
"""
SUM_ROWS = 16384          # sum_plan: 64 rows of theta use 4096 workspace doubles, 512 rows 32768


def _create(lib, n, d, seed=7):
    ld = d if d <= 4 else (d + 3) // 4 * 4
    cfg = _lib.Config(algo=_lib.BPM_ALGO_DREAM, n_chains=n, dim=d, ld=ld, del_pairs=3, n_cr=3, burnin_gen=1000,
                      n_cr_gen=1, shuffle=1, chain_lo=0, chain_hi=n, device=0, gamma_scale=1.0, flip=0.5,
                      epsilon=0.0, u_epsilon=0.0, gamma=0.0, seed=seed)
    h = C.c_void_p()
    _lib.check(lib.bpm_create(C.byref(cfg), C.byref(h)))
    return h


class _Pop(object):
    """Device state of one population: X, ln L, running moments and a history of `rows` rows."""

    def __init__(self, n, ld, rows=8):
        dev = torch.device("cuda", 0)
        self.X = torch.empty(n, ld, dtype=torch.float64, device=dev)
        self.lnl = torch.empty(n, dtype=torch.float64, device=dev)
        self.mean = torch.empty_like(self.X)
        self.m2 = torch.empty_like(self.X)
        self.hist = torch.empty(rows, n, ld, dtype=torch.float64, device=dev)

    def start(self, lib, h, X0):
        """Reset to X0 (a device tensor) with its ln L; returns the state block."""
        self.X.copy_(X0)
        self.mean.copy_(X0)
        self.m2.zero_()
        self.hist[0].copy_(X0)
        _lib.check(lib.bpm_eval_lnl(h, self.X.data_ptr(), self.X.shape[0], self.lnl.data_ptr(), None))
        return _lib.State(X=self.X.data_ptr(), lnl=self.lnl.data_ptr(), mean=self.mean.data_ptr(),
                          m2=self.m2.data_ptr(), history=self.hist.data_ptr(), hist_len=1, mom_len=0, pending=0)


def _set(lib, h, dt, n=None):
    return lib.bpm_set_target(h, dt.target_id, _lib.dptr(dt.params), dt.params.size if n is None else n)


@pytest.fixture(scope="module")
def setup():
    lib = _lib.load()
    torch.cuda.set_device(0)
    g = torch.Generator(device="cuda").manual_seed(3)
    data = {
        "gauss": targets.Gauss_100D().device_target(),
        "line": targets.LineFit().device_target(),
        "set": targets.CudaLikelihoodSet(SET_SRC, 3, np.arange(12.0).reshape(4, 3) / 10.0),
        "sum": targets.CudaSumLikelihood(SUM_SRC, 2, np.linspace(-1.0, 1.0, SUM_ROWS)),
        "X0": 0.1 * torch.randn(N, D, dtype=torch.float64, device="cuda", generator=g),
        "X0_set": 0.1 * torch.randn(4 * N, 3, dtype=torch.float64, device="cuda", generator=g),
        "theta_sum": 0.1 * torch.randn(512, 2, dtype=torch.float64, device="cuda", generator=g),
        "pop": _Pop(N, D),
        "pop_set": _Pop(4 * N, 3),
        "lnl_sum": torch.empty(512, dtype=torch.float64, device="cuda"),
    }
    return lib, data


def _cycle(lib, t):
    """Create, exercise and destroy one handle of each kind the test covers."""
    h = _create(lib, N, D)
    _lib.check(_set(lib, h, t["gauss"]))                    # tparams and wfrag
    st = t["pop"].start(lib, h, t["X0"])
    _lib.check(lib.bpm_omega_track(h, 1))
    _lib.check(lib.bpm_cov_track(h, 1))
    _lib.check(lib.bpm_profile(h, 1))
    _lib.check(lib.bpm_step_generations(h, C.byref(st), 0, 3, None))      # the side stream
    ms, launches = (C.c_double * 8)(), (C.c_int64 * 8)()
    _lib.check(lib.bpm_profile_read(h, ms, launches))
    assert launches[0] == 3
    _lib.check(lib.bpm_outlier_reset(h, C.byref(st), None, None, None, None, None))
    _lib.check(lib.bpm_flush(h, C.byref(st), None))
    rhat = np.zeros(D)
    _lib.check(lib.bpm_rhat(h, C.byref(st), 0, rhat.ctypes.data, None))
    assert np.all(np.isfinite(rhat))
    Xh, Lh = t["X0"].cpu().numpy().copy(), np.zeros(N)
    _lib.check(lib.bpm_eval_lnl(h, t["X0"].data_ptr(), N, t["pop"].lnl.data_ptr(), None))
    Lh[:] = t["pop"].lnl.cpu().numpy()
    _lib.check(lib.bpm_generations_host(h, Xh.ctypes.data, Lh.ctypes.data, 3, 4, 2))
    _lib.check(_set(lib, h, t["line"]))                     # the line fit replaces the Gaussian's parameters
    _lib.check(lib.bpm_destroy(h))

    h = _create(lib, N * 4, 3)
    keys = (C.c_uint64 * 4)(11, 12, 13, 14)
    _lib.check(lib.bpm_set_problems(h, 4, keys))
    t["set"]._attach(lib, h)
    st = t["pop_set"].start(lib, h, t["X0_set"])
    _lib.check(lib.bpm_step_generations(h, C.byref(st), 0, 3, None))
    _lib.check(lib.bpm_destroy(h))

    h = _create(lib, N, 2)
    t["sum"]._attach(lib, h)
    for n in (64, 512):                                     # the group workspace grows
        _lib.check(lib.bpm_eval_lnl(h, t["theta_sum"].data_ptr(), n, t["lnl_sum"].data_ptr(), None))
    assert np.all(np.isfinite(t["lnl_sum"].cpu().numpy()))
    _lib.check(lib.bpm_destroy(h))


def test_destroyed_handles_release_their_device_memory(setup):
    lib, t = setup
    _cycle(lib, t)                                          # modules load lazily: warm up first
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    free0 = torch.cuda.mem_get_info()[0]
    for _ in range(5):
        _cycle(lib, t)
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    free1 = torch.cuda.mem_get_info()[0]
    assert free1 >= free0 - 2 * (1 << 20), "5 cycles kept %d bytes" % (free0 - free1)


def test_refused_set_target_changes_nothing(setup):
    lib, t = setup
    out = []
    for refuse in (False, True):
        h = _create(lib, N, D)
        _lib.check(_set(lib, h, t["gauss"]))
        if refuse:
            assert _set(lib, h, t["gauss"], t["gauss"].params.size - 1) != 0
            assert _set(lib, h, t["line"], t["line"].params.size + 1) != 0
        st = t["pop"].start(lib, h, t["X0"])
        _lib.check(lib.bpm_step_generations(h, C.byref(st), 0, 3, None))
        _lib.check(lib.bpm_flush(h, C.byref(st), None))
        torch.cuda.synchronize()
        out.append((t["pop"].X.cpu().numpy().copy(), t["pop"].lnl.cpu().numpy().copy()))
        _lib.check(lib.bpm_destroy(h))
    assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1])
