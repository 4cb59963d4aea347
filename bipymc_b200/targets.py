"""Built-in likelihood targets with a batched device implementation.

Mirrors the reference's test-target classes (same constructor arguments, same ``pdf`` /
``ln_like`` / ``rvs`` surface):

  Banana_2D       bipymc/utils/banana_rv.py:10-61
  BimodeGauss_2D  bipymc/utils/dblgauss_rv.py:10-43
  Gauss_100D      bipymc/utils/d100_gauss.py:10-39
  LineFit         examples/ex_para_fit.py:26-55 (lnprob of the second example)
  ExpFit          examples/ex_exp_fit.py:38-121 (5-parameter relaxation fit)

and ``CudaLikelihood``: any other model as CUDA C++ source, compiled at run time into the same
kernels (``ln_like_cuda=`` of the samplers); ``CudaSumLikelihood``: a model that is a sum over
observations, one CUDA C++ term per observation, summed across the whole GPU.

``ln_like`` stays a scalar host function, so the objects remain valid ``ln_like_fn``
arguments everywhere; when a sampler of this package receives ``obj.ln_like`` it
recognises the owner through ``device_target()`` and evaluates the likelihood inside the
CUDA generation kernels instead (bipymc_b200/csrc/targets.cuh).

Host-side parameter preparation follows scipy.stats.multivariate_normal (which the
reference calls): symmetric eigendecomposition, ``U = V / sqrt(lambda)``,
``maha = |(x - mu) U|^2``, ``logpdf = -0.5 (rank log 2pi + log pdet + maha)``
(scipy/stats/_multivariate.py ``_PSD`` and ``_logpdf``).
"""
import ctypes as C

import numpy as np

from . import _lib

_LOG_2PI = np.log(2 * np.pi)


def psd_whiten(cov):
    """(U, log_pdet, rank) of a covariance, the way scipy's _PSD computes them."""
    cov = np.asarray(cov, dtype=float)
    s, u = np.linalg.eigh(cov)
    eps = 1e6 * np.finfo("d").eps * np.max(np.abs(s))     # scipy's _eigvalsh_to_eps default
    if np.min(s) < -eps:
        raise ValueError("the input matrix must be symmetric positive semidefinite")
    keep = s > eps
    d = s[keep]
    s_pinv = np.array([0.0 if abs(x) <= eps else 1.0 / x for x in s])
    U = np.multiply(u, np.sqrt(s_pinv))
    U = U[:, keep]
    return np.ascontiguousarray(U), float(np.sum(np.log(d))), int(len(d))


class _Mvn(object):
    """Minimal frozen multivariate normal (pdf / logpdf / rvs) on the host."""
    def __init__(self, mean, cov):
        self.mean = np.asarray(mean, dtype=float)
        self.cov = np.asarray(cov, dtype=float)
        self.U, self.log_pdet, self.rank = psd_whiten(self.cov)
        self.c0 = self.rank * _LOG_2PI + self.log_pdet

    def logpdf(self, x):
        dev = np.asarray(x, dtype=float) - self.mean
        maha = np.sum(np.square(np.dot(dev, self.U)), axis=-1)
        return -0.5 * (self.c0 + maha)

    def pdf(self, x):
        return np.exp(self.logpdf(x))

    def rvs(self, size=1):
        return np.random.multivariate_normal(self.mean, self.cov, size=size)

    def packed2(self):
        assert self.mean.shape == (2,) and self.U.shape == (2, 2)
        return [self.mean[0], self.mean[1], self.U[0, 0], self.U[0, 1], self.U[1, 0], self.U[1, 1],
                self.c0]


class DeviceTarget(object):
    """(target id, flat float64 parameter array) handed to bpm_set_target."""
    def __init__(self, target_id, params, dim):
        self.target_id = int(target_id)
        self.params = np.ascontiguousarray(np.asarray(params, dtype=np.float64))
        self.dim = int(dim)


class Banana_2D(object):
    def __init__(self, mu1=0, mu2=0, sigma1=1, sigma2=1, rho=0.9, a=1.15, b=0.5, log_of_pdf=True):
        self.mu1, self.mu2 = mu1, mu2
        self.sigma1, self.sigma2, self.rho = sigma1, sigma2, rho
        self.a, self.b = a, b
        self.log_of_pdf = log_of_pdf
        cov = np.array([[sigma1 ** 2.0, rho * (sigma1 * sigma2)],
                        [rho * (sigma1 * sigma2), sigma2 ** 2.0]])
        self.rv_2d_normal = _Mvn(np.array([mu1, mu2], dtype=float), cov)

    def inv_transform(self, y1, y2):
        x1 = y1 / self.a
        x2 = (y2 - self.b * (x1 ** 2.0 + self.a ** 2.0)) * self.a
        return x1, x2

    def transform(self, x1, x2):
        return self.a * x1, x2 / self.a + self.b * (x1 ** 2.0 + self.a ** 2.0)

    def pdf(self, y1, y2):
        x1, x2 = self.inv_transform(np.asarray(y1, dtype=float), np.asarray(y2, dtype=float))
        return self.rv_2d_normal.pdf(np.stack((x1, x2), axis=-1))

    def ln_like(self, y):
        assert len(y) == 2
        with np.errstate(divide="ignore"):
            return np.log(self.pdf(y[0], y[1]))

    def check_prob_lvl(self, y1, y2, pdf_lvl):
        return pdf_lvl < self.pdf(y1, y2)

    def rvs(self, n_samples):
        s = self.rv_2d_normal.rvs(size=n_samples)
        return self.transform(s[:, 0], s[:, 1])

    def device_target(self):
        p = [1.0 if self.log_of_pdf else 0.0, self.a, self.b] + self.rv_2d_normal.packed2()
        return DeviceTarget(_lib.TARGET_BANANA, p, 2)


class BimodeGauss_2D(object):
    def __init__(self, mu_g1=[0, 0], mu_g2=[2, 2], sigma_g1=[0.25, 0.25], sigma_g2=[0.25, 0.25],
                 rho_g1=0.8, rho_g2=-0.8, w_g1=0.25, w_g2=0.75, log_of_pdf=True):
        self.mu_g1, self.mu_g2 = mu_g1, mu_g2
        self.cov_g1 = np.array([[sigma_g1[0] ** 2.0, rho_g1 * (sigma_g1[0] * sigma_g1[1])],
                                [rho_g1 * (sigma_g1[0] * sigma_g1[1]), sigma_g1[1] ** 2.0]])
        self.cov_g2 = np.array([[sigma_g2[0] ** 2.0, rho_g2 * (sigma_g2[0] * sigma_g2[1])],
                                [rho_g2 * (sigma_g2[0] * sigma_g2[1]), sigma_g2[1] ** 2.0]])
        self.rv_2d_g1 = _Mvn(self.mu_g1, self.cov_g1)
        self.rv_2d_g2 = _Mvn(self.mu_g2, self.cov_g2)
        self.w_g1 = w_g1 / (w_g1 + w_g2)
        self.w_g2 = w_g2 / (w_g1 + w_g2)
        self.log_of_pdf = log_of_pdf

    def pdf(self, y1, y2):
        pos = np.stack((np.asarray(y1, dtype=float), np.asarray(y2, dtype=float)), axis=-1)
        return self.w_g1 * self.rv_2d_g1.pdf(pos) + self.w_g2 * self.rv_2d_g2.pdf(pos)

    def ln_like(self, y):
        assert len(y) == 2
        if not self.log_of_pdf:
            # direct log-density (log-sum-exp): finite far from both modes, where the
            # reference's np.log(pdf) underflows to -inf
            pos = np.asarray(y, dtype=float)
            a = self.rv_2d_g1.logpdf(pos) + np.log(self.w_g1)
            b = self.rv_2d_g2.logpdf(pos) + np.log(self.w_g2)
            m = max(a, b)
            return m + np.log(np.exp(a - m) + np.exp(b - m))
        with np.errstate(divide="ignore"):
            return np.log(self.pdf(y[0], y[1]))

    def rvs(self, n_samples):
        sel = np.random.choice((True, False), p=(self.w_g1, self.w_g2), size=n_samples)
        out = np.zeros((n_samples, 2))
        s1, s2 = self.rv_2d_g1.rvs(size=n_samples), self.rv_2d_g2.rvs(size=n_samples)
        out[sel, :] = s1[sel, :]
        out[~sel, :] = s2[~sel, :]
        return out[:, 0], out[:, 1]

    def device_target(self):
        p = ([1.0 if self.log_of_pdf else 0.0, self.w_g1, self.w_g2] + self.rv_2d_g1.packed2() +
             self.rv_2d_g2.packed2())
        return DeviceTarget(_lib.TARGET_BIMODAL, p, 2)


def gauss_cov(dim, rho=0.5):
    """d100_gauss.py:17-25: var_i = i + 1, pairwise correlation rho."""
    sd = np.sqrt(np.arange(dim) + 1.0)
    cov = np.outer(sd, sd) * rho
    cov[np.diag_indices(dim)] = sd ** 2.0
    return cov


class Gauss_100D(object):
    """Correlated Gaussian of any dimension.  ``log_of_pdf=True`` reproduces the
    reference's ``np.log(pdf)`` (which underflows to -inf beyond d of a few hundred);
    ``log_of_pdf=False`` evaluates the log-density directly and is what dim=1000 needs.
    A general (mean, cov) can be passed instead of the rho rule."""
    def __init__(self, rho=0.5, dim=100, log_of_pdf=None, mean=None, cov=None):
        self.dim = dim
        self.rho = rho
        self.mu = np.zeros(dim) if mean is None else np.asarray(mean, dtype=float)
        self.var = np.sqrt(np.arange(dim) + 1.0)
        self.cov = gauss_cov(dim, rho) if cov is None else np.asarray(cov, dtype=float)
        self.rv_100d = _Mvn(self.mu, self.cov)
        self.log_of_pdf = (dim <= 200) if log_of_pdf is None else bool(log_of_pdf)

    def pdf(self, y):
        return self.rv_100d.pdf(y)

    def ln_like(self, y):
        assert len(y) == self.dim
        if not self.log_of_pdf:
            return self.rv_100d.logpdf(y)
        with np.errstate(divide="ignore"):
            return np.log(self.pdf(y))

    def rvs(self, n_samples):
        return self.rv_100d.rvs(size=n_samples)

    def device_target(self):
        rv = self.rv_100d
        head = [1.0 if self.log_of_pdf else 0.0, rv.c0, float(rv.U.shape[1])]
        return DeviceTarget(_lib.TARGET_GAUSS, np.concatenate([head, rv.mean, rv.U.ravel()]), self.dim)


def linefit_data(seed=42, n=50, m_true=-0.9594, b_true=4.294, f_true=0.534):
    """Synthetic data of examples/ex_para_fit.py:17,26-35."""
    rs = np.random.RandomState(seed)
    x = np.sort(10 * rs.rand(n))
    yerr = 0.1 + 0.5 * rs.rand(n)
    y = m_true * x + b_true
    y += np.abs(f_true * y) * rs.randn(n)
    y += yerr * rs.randn(n)
    return x, y, yerr


class LineFit(object):
    """theta = (m, b, ln f): box prior + heteroscedastic Gaussian likelihood."""
    def __init__(self, x=None, y=None, yerr=None):
        if x is None:
            x, y, yerr = linefit_data()
        self.x, self.y, self.yerr = (np.asarray(v, dtype=float) for v in (x, y, yerr))

    def ln_like(self, theta):
        m, b, lnf = theta
        if not (-5.0 < m < 0.5 and 0.0 < b < 10.0 and -10.0 < lnf < 1.0):
            return -np.inf
        model = m * self.x + b
        inv_sigma2 = 1.0 / (self.yerr ** 2 + model ** 2 * np.exp(2 * lnf))
        return 0.0 + -0.5 * (np.sum((self.y - model) ** 2 * inv_sigma2 - np.log(inv_sigma2)))

    def device_target(self):
        p = np.concatenate([[float(len(self.x))], self.x, self.y, self.yerr])
        return DeviceTarget(_lib.TARGET_LINEFIT, p, 3)


def expfit_data(seed=42, n=60, tau=12.0, c_inf=1.5, c_0=0.6, leak=1e-3, sigma=2e-3):
    """Synthetic relaxation data for the model of examples/ex_exp_fit.py:38-43 (the example
    reads a measured .mat series; a seeded synthetic series of the same shape stands in)."""
    rs = np.random.RandomState(seed)
    t = np.linspace(0.5, 60.0, n)
    y = c_inf + c_0 * -1.0 * np.exp(-t / tau) - leak * t + np.sqrt(sigma) * 0.3 * rs.randn(n)
    return t, y


class ExpFit(object):
    """theta = (tau, c_inf, c_0, leak, sigma): lnprob of examples/ex_exp_fit.py:73-121."""
    def __init__(self, t=None, y=None):
        if t is None:
            t, y = expfit_data()
        self.t, self.y = np.asarray(t, dtype=float), np.asarray(y, dtype=float)

    def ln_like(self, theta):
        tau, c_inf, c_0, leak, sigma = theta
        if not (-5.0 < c_inf < 5.0 and 1.0 < tau < 50.0 and -1.0 < c_0 < 1.0 and -5.0 < leak < 5.0 and
                0.0 < sigma < 1.0):
            return -np.inf
        m = c_inf + c_0 * -1.0 * np.exp(-self.t / tau) - leak * self.t
        return 0.0 + -0.5 * np.sum((m - self.y) ** 2. / sigma - np.log(1.0 / sigma))

    def device_target(self):
        p = np.concatenate([[float(len(self.t))], self.t, self.y])
        return DeviceTarget(_lib.TARGET_EXPFIT, p, 5)


def resolve_device_target(ln_like_fn, ln_kwargs):
    """Return a DeviceTarget when ``ln_like_fn`` is the ``ln_like`` of a built-in target
    (or the object itself) and no extra kwargs are bound; otherwise None."""
    if ln_kwargs:
        return None
    owner = getattr(ln_like_fn, "__self__", None)
    if owner is not None and getattr(ln_like_fn, "__name__", "") == "ln_like" and \
            hasattr(owner, "device_target"):
        return owner.device_target()
    if hasattr(ln_like_fn, "device_target") and not callable(getattr(ln_like_fn, "__call__", None)):
        return ln_like_fn.device_target()
    if isinstance(ln_like_fn, DeviceTarget):
        return ln_like_fn
    return None


class CudaCompileError(_lib.BpmError):
    """NVRTC rejected a CudaLikelihood source; ``log`` is the compiler's log, whose line numbers
    refer to the user's source (``ln_like.cu(line)``)."""
    def __init__(self, msg, log=""):
        super(CudaCompileError, self).__init__(msg + ("\n" + log if log else ""))
        self.log = log


class CudaLikelihood(object):
    """A user likelihood in CUDA C++, compiled at run time (NVRTC, sm_100a) into the sampler's
    own generation kernels -- the fast path of the built-in targets, for any model.

    ``source`` defines ONE device function::

        __device__ double ln_like(const double* theta, const double* data)

    with ``theta[BPM_DIM]`` (the parameters) and ``data[BPM_NDATA]`` (``data`` below, read-only,
    copied to the device once); ``BPM_DIM`` / ``BPM_NDATA`` are macros, and the CUDA math functions
    and the ``bpm::`` helpers of the package's csrc/targets.cuh are in scope.  Return ``-INFINITY``
    outside the prior; a NaN makes ``run_mcmc`` raise ``ValueError("probabilities contain NaN")``
    as the reference does.  ``fmad=False`` rounds every ``+ - * /`` on its own (numpy's results);
    ``fmad=True`` lets the compiler fuse multiply-adds.  The first compile of a source takes up to
    about 2 s; later samplers with the same source, dim, data size and fmad reuse the cubin for the rest
    of the process.

    At d <= 4 the likelihood runs inside the fused one-thread-per-chain half-phase kernel, above that
    in a batched row kernel between the proposal and accept kernels.  Pass it as ``ln_like_cuda=``."""

    _LOG_BYTES = 1 << 16

    def __init__(self, source, dim, data=None, fmad=True):
        if not isinstance(source, str):
            raise ValueError("source must be a str of CUDA C++")
        if isinstance(dim, bool) or int(dim) != dim or int(dim) < 1:
            raise ValueError("dim must be an integer >= 1")
        data = np.zeros(0) if data is None else np.asarray(data, dtype=np.float64)
        if data.ndim != 1:
            raise ValueError("data must be 1-D (concatenate the arrays the source reads)")
        if not np.all(np.isfinite(data)):
            raise ValueError("data must be finite")
        self.source = source
        self.dim = int(dim)
        self.data = np.ascontiguousarray(data)
        self.fmad = bool(fmad)

    @property
    def _flags(self):
        return 1 if self.fmad else 0

    def _call(self, fn, *head):
        log = C.create_string_buffer(self._LOG_BYTES)
        cached = C.c_int32(0)
        rc = fn(*(head + (C.byref(cached), log, self._LOG_BYTES)))
        if rc != 0:
            msg = _lib.load().bpm_last_error().decode()
            text = log.value.decode(errors="replace")
            if text:
                raise CudaCompileError(msg, text)
            raise _lib.BpmError(msg)
        return bool(cached.value)

    def compile(self):
        """Compile for sm_100a (no device needed).  Returns True when the cubin came from the
        process cache; raises CudaCompileError with the NVRTC log."""
        lib = _lib.load()
        return self._call(lib.bpm_jit_compile, self.source.encode(), self.dim, self.data.size, self._flags)

    def _attach(self, lib, handle):
        """Compile (or take the cached cubin), load it on the handle's device and copy the data."""
        return self._call(lib.bpm_set_jit_target, handle, self.source.encode(), _lib.dptr(self.data),
                          self.data.size, self._flags)


class CudaSumLikelihood(CudaLikelihood):
    """A likelihood that is a sum over independent observations, in CUDA C++: the library splits the
    sum across the whole GPU.  ``source`` defines::

        __device__ double ln_like_term(const double* theta, const double* row);   // one observation
        __device__ double ln_prior(const double* theta);                          // only when prior=True

    ``data`` is a finite float64 array of shape ``(M, k)`` (a 1-D array is ``(M, 1)``), ``row`` points at
    the k values of one observation.  ``BPM_DIM``, ``BPM_NROWS`` (M) and ``BPM_ROWLEN`` (k) are macros;
    the scope, ``fmad``, the NaN rule, the compile cache and ``CudaCompileError`` are those of
    ``CudaLikelihood`` (M, k and ``prior`` are part of the cache key).  The value is::

        ln L(theta) = ln_prior(theta) + sum_{i < M} ln_like_term(theta, row_i)

    and ``-inf``, with no term of that chain evaluated, when ``ln_prior`` is ``-inf``.

    The order of the additions depends on M alone, never on the number of chains, the batch size, the
    launch shape or the number of GPUs, so a given theta always gets the same bits: rows are cut into
    chunks of 256 consecutive rows (the last padded with 0.0 terms); inside a chunk a halving pairwise
    tree adds ``a[i] + a[i + w/2]`` for w = 256, 128, ..., 2; the chunk partials, padded with 0.0 to the
    next power of two, are added by an adjacent-pair tree ``p[2i] + p[2i+1]``, level by level; the prior
    is added last.  In numpy::

        a = np.zeros((nc, 256)); a.flat[:M] = terms
        while a.shape[1] > 1: a = a[:, :a.shape[1] // 2] + a[:, a.shape[1] // 2:]
        p = np.zeros(P2); p[:nc] = a[:, 0]
        while p.size > 1: p = p[0::2] + p[1::2]
        lnl = prior + p[0]

    Which form to use: ``CudaLikelihood`` (one ``ln_like`` per chain) for a model that is not a sum over
    observations, or for small data at d <= 4, where it runs fused into the one-thread-per-chain step
    kernel.  ``CudaSumLikelihood`` for many observations or few chains: every chain's sum is spread over
    all SMs, between the proposal and accept kernels at every d.  Pass it as ``ln_like_cuda=``."""

    def __init__(self, source, dim, data, prior=False, fmad=True):
        if not isinstance(source, str):
            raise ValueError("source must be a str of CUDA C++")
        if isinstance(dim, bool) or int(dim) != dim or int(dim) < 1:
            raise ValueError("dim must be an integer >= 1")
        data = np.asarray(data, dtype=np.float64)
        if data.ndim == 1:
            data = data.reshape(-1, 1)
        if data.ndim != 2 or data.shape[0] < 1 or data.shape[1] < 1:
            raise ValueError("data must have shape (M, k) with M >= 1 and k >= 1 (or be 1-D with M >= 1)")
        if data.shape[0] >= 2 ** 31:
            raise ValueError("data must have fewer than 2^31 rows")
        if not np.all(np.isfinite(data)):
            raise ValueError("data must be finite")
        self.source = source
        self.dim = int(dim)
        self.data = np.ascontiguousarray(data)
        self.prior = bool(prior)
        self.fmad = bool(fmad)

    @property
    def _flags(self):
        return (1 if self.fmad else 0) | (2 if self.prior else 0)

    def compile(self):
        """Compile for sm_100a (no device needed).  Returns True when the cubin came from the
        process cache; raises CudaCompileError with the NVRTC log."""
        lib = _lib.load()
        M, k = self.data.shape
        return self._call(lib.bpm_jit_compile_sum, self.source.encode(), self.dim, M, k, self._flags)

    def _attach(self, lib, handle):
        """Compile (or take the cached cubin), load it on the handle's device and copy the data."""
        M, k = self.data.shape
        return self._call(lib.bpm_set_jit_sum_target, handle, self.source.encode(), _lib.dptr(self.data), M, k,
                          self._flags)
