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
observations, one CUDA C++ term per observation, summed across the whole GPU; ``CudaLikelihoodSet``: one
``ln_like`` source fitted to many datasets at once, each an independent problem of the same sampler;
``CudaSumLikelihoodSet``: the same for a per-observation source.

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
        data = self._shaped(data)
        if not np.all(np.isfinite(data)):
            raise ValueError("data must be finite")
        self.source = source
        self.dim = int(dim)
        self.data = np.ascontiguousarray(data)
        self.fmad = bool(fmad)

    @staticmethod
    def _shaped(data):
        """``data`` as the float64 array of the shape this kind takes, or ValueError."""
        data = np.zeros(0) if data is None else np.asarray(data, dtype=np.float64)
        if data.ndim != 1:
            raise ValueError("data must be 1-D (concatenate the arrays the source reads)")
        return data

    def _compile_call(self, lib):
        """This kind's C-ABI compile function and its arguments before ``flags``."""
        return lib.bpm_jit_compile, (self.source.encode(), self.dim, self.data.size)

    def _attach_call(self, lib, handle):
        """This kind's C-ABI attach function and its arguments before ``flags``."""
        return lib.bpm_set_jit_target, (handle, self.source.encode(), _lib.dptr(self.data), self.data.size)

    @property
    def _flags(self):
        return 1 if self.fmad else 0

    def _call(self, fn, *head):
        log = C.create_string_buffer(self._LOG_BYTES)
        cached = C.c_int32(0)
        rc = fn(*(head + (self._flags, C.byref(cached), log, self._LOG_BYTES)))
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
        fn, args = self._compile_call(_lib.load())
        return self._call(fn, *args)

    def _attach(self, lib, handle):
        """Compile (or take the cached cubin), load it on the handle's device and copy the data."""
        fn, args = self._attach_call(lib, handle)
        return self._call(fn, *args)


class CudaLikelihoodSet(CudaLikelihood):
    """One CUDA likelihood fitted to P datasets at once: P independent problems in one sampler.

    ``source`` is the ``ln_like`` of ``CudaLikelihood``; ``data`` is a finite float64 array of shape
    ``(P, n_data)`` with P >= 1 and n_data >= 1, and problem g's ``ln_like`` sees row g (``BPM_NDATA`` is
    n_data, ``BPM_NPROBLEMS`` is P).  Pass it as ``ln_like_cuda=`` to ``DreamMpi`` / ``DeMcMpi``: their
    ``n_chains`` then counts the chains of ONE problem, and problem g steps exactly -- bit for bit -- as a
    single-problem sampler with ``n_chains`` chains, data row g and Philox key ``sampler.problem_seeds[g]``
    would, while all P problems run in the same kernel launches.  Validation, ``fmad``, the NaN rule,
    ``CudaCompileError`` and the compile cache are those of ``CudaLikelihood``; P and n_data are part of the
    cache key, and the kernels are compiled in a translation unit of their own."""

    def __init__(self, source, dim, data, fmad=True):
        super(CudaLikelihoodSet, self).__init__(source, dim, data, fmad)

    @staticmethod
    def _shaped(data):
        data = np.asarray(data, dtype=np.float64)
        if data.ndim != 2 or data.shape[0] < 1 or data.shape[1] < 1:
            raise ValueError("data must have shape (P, n_data) with P >= 1 and n_data >= 1: one row per problem")
        if data.shape[0] >= 2 ** 31:
            raise ValueError("data must have fewer than 2^31 rows")
        return data

    def _compile_call(self, lib):
        P, nd = self.data.shape
        return lib.bpm_jit_compile_problems, (self.source.encode(), self.dim, nd, P)

    def _attach_call(self, lib, handle):
        # the handle must be a multi-problem handle with P problems (bpm_set_problems), which gives P
        return lib.bpm_set_jit_problems_target, (handle, self.source.encode(), _lib.dptr(self.data),
                                                 self.data.shape[1])

    @property
    def n_problems(self):
        return int(self.data.shape[0])


def problem_seeds(seed, n_problems):
    """Philox keys of P problems: ``(seed + 0x9E3779B97F4A7C15 g) mod 2^64`` for an int seed (problem 0
    keeps ``seed``), or a sequence of P ints taken as they are."""
    P = int(n_problems)
    if np.ndim(seed) == 0:
        s = int(seed)
        return [(s + 0x9E3779B97F4A7C15 * g) % (1 << 64) for g in range(P)]
    keys = [int(k) for k in seed]
    if len(keys) != P:
        raise ValueError("seed: %d keys for %d problems" % (len(keys), P))
    if any(not 0 <= k < (1 << 64) for k in keys):
        raise ValueError("seed: every key must be in [0, 2^64)")
    return keys


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
        super(CudaSumLikelihood, self).__init__(source, dim, data, fmad)
        self.prior = bool(prior)

    @staticmethod
    def _shaped(data):
        data = np.asarray(data, dtype=np.float64)
        if data.ndim == 1:
            data = data.reshape(-1, 1)
        if data.ndim != 2 or data.shape[0] < 1 or data.shape[1] < 1:
            raise ValueError("data must have shape (M, k) with M >= 1 and k >= 1 (or be 1-D with M >= 1)")
        if data.shape[0] >= 2 ** 31:
            raise ValueError("data must have fewer than 2^31 rows")
        return data

    def _compile_call(self, lib):
        M, k = self.data.shape
        return lib.bpm_jit_compile_sum, (self.source.encode(), self.dim, M, k)

    def _attach_call(self, lib, handle):
        M, k = self.data.shape
        return lib.bpm_set_jit_sum_target, (handle, self.source.encode(), _lib.dptr(self.data), M, k)

    @property
    def _flags(self):
        return (1 if self.fmad else 0) | (2 if self.prior else 0)


class CudaSumLikelihoodSet(CudaSumLikelihood):
    """One per-observation CUDA likelihood fitted to P datasets at once: P independent problems in one sampler.

    ``source`` and ``prior`` are those of ``CudaSumLikelihood``; ``data`` is a finite float64 array of shape
    ``(P, M, k)`` (a 2-D ``(P, M)`` array is ``(P, M, 1)``): problem g's sum runs over its own M rows
    ``data[g]``.  ``BPM_NROWS`` is M (the rows of ONE problem), ``BPM_ROWLEN`` k and ``BPM_NPROBLEMS`` P.
    Pass it as ``ln_like_cuda=`` to ``DreamMpi`` / ``DeMcMpi``: as with ``CudaLikelihoodSet``, ``n_chains``
    then counts the chains of one problem, and problem g steps exactly -- bit for bit -- as a single-problem
    sampler with ``n_chains`` chains, ``CudaSumLikelihood(source, dim, data[g], prior, fmad)`` and Philox key
    ``sampler.problem_seeds[g]`` would, while all P problems run in the same kernel launches.  Each problem's
    sum is added in the order of ``CudaSumLikelihood`` for M rows and is split over the GPU in tiles of chains
    that never straddle two problems: the form for many datasets of many observations and few chains each.
    P, M, k and ``prior`` are part of the cache key, and the kernels are compiled in a translation unit of their
    own.

    Datasets of different lengths: ``data`` may also be a list or tuple of P arrays, array g of shape ``(M_g, k)``
    (or ``(M_g,)``: k = 1), every M_g in [1, 2^31) and one k for all.  When every M_g is equal this is the
    rectangular set above, ``data`` stacked.  Otherwise ``data`` is the concatenated ``(sum_g M_g, k)`` array and
    ``n_rows`` the int64 ``[P]`` array of the M_g; problem g's sum runs over its own M_g rows in the order of
    ``CudaSumLikelihood`` for M_g rows, so the contract above holds with ``CudaSumLikelihood(source, dim,
    data_g, prior, fmad)``.  The work is that of the sum_g M_g terms, not of P max_g M_g.  ``BPM_ROWLEN`` and
    ``BPM_NPROBLEMS`` are defined but ``BPM_NROWS`` is not: a term that needs its problem's row count reads it
    from a data column.  P, k and ``prior`` are part of the cache key, the M_g are not, so new datasets of other
    lengths reuse the compiled module."""

    def __init__(self, source, dim, data, prior=False, fmad=True):
        self.n_rows = None      # ragged form: the int64 [P] row counts
        if isinstance(data, (list, tuple)):
            data, self.n_rows = self._ragged(data)
            if self.n_rows is not None:
                self._shaped = lambda rows: rows      # (sum M_g, k) as _ragged shaped them
        super(CudaSumLikelihoodSet, self).__init__(source, dim, data, prior, fmad)

    @staticmethod
    def _ragged(arrays):
        """P arrays of shape (M_g, k) or (M_g,): ``(stacked (P, M, k), None)`` when every M_g is equal, else
        ``(concatenated (sum M_g, k), n_rows)``; ValueError on an empty sequence, problem or row, or mixed k."""
        if len(arrays) == 0:
            raise ValueError("data: an empty sequence (one array per problem expected)")
        parts = []
        for g, a in enumerate(arrays):
            a = np.asarray(a, dtype=np.float64)
            if a.ndim == 1:
                a = a.reshape(-1, 1)
            if a.ndim != 2 or a.shape[1] < 1:
                raise ValueError("data[%d] must have shape (M, k) or (M,), not %s" % (g, a.shape))
            if not 1 <= a.shape[0] < 2 ** 31:
                raise ValueError("data[%d] has %d rows: every problem needs M in [1, 2^31)" % (g, a.shape[0]))
            if parts and a.shape[1] != parts[0].shape[1]:
                raise ValueError("data[%d] has rows of %d values, data[0] of %d: every problem needs the same k"
                                 % (g, a.shape[1], parts[0].shape[1]))
            parts.append(a)
        if len(parts) >= 2 ** 31:
            raise ValueError("data: P must be below 2^31")
        n_rows = np.array([a.shape[0] for a in parts], dtype=np.int64)
        if np.all(n_rows == n_rows[0]):
            return np.stack(parts), None
        return np.concatenate(parts), n_rows

    @staticmethod
    def _shaped(data):
        data = np.asarray(data, dtype=np.float64)
        if data.ndim == 2:
            data = data.reshape(data.shape + (1,))
        if data.ndim != 3 or min(data.shape) < 1:
            raise ValueError("data must have shape (P, M, k) with P, M, k >= 1 (or (P, M) with k = 1), not %s"
                             % (data.shape,))
        if data.shape[0] >= 2 ** 31 or data.shape[1] >= 2 ** 31:
            raise ValueError("data shape %s: P and M must each be below 2^31" % (data.shape,))
        return data

    def _compile_call(self, lib):
        if self.n_rows is not None:
            return lib.bpm_jit_compile_sum_ragged, (self.source.encode(), self.dim, self.data.shape[1], self.n_problems)
        P, M, k = self.data.shape
        return lib.bpm_jit_compile_sum_problems, (self.source.encode(), self.dim, M, k, P)

    def _attach_call(self, lib, handle):
        # the handle must be a multi-problem handle with P problems (bpm_set_problems), which gives P
        if self.n_rows is not None:
            return lib.bpm_set_jit_sum_ragged_target, (handle, self.source.encode(), _lib.dptr(self.data),
                                                       self.n_rows.ctypes.data_as(C.POINTER(C.c_int64)),
                                                       self.data.shape[1])
        _, M, k = self.data.shape
        return lib.bpm_set_jit_sum_problems_target, (handle, self.source.encode(), _lib.dptr(self.data), M, k)

    @property
    def n_problems(self):
        return int(self.data.shape[0]) if self.n_rows is None else int(self.n_rows.size)


class CudaGaussLikelihood(CudaLikelihood):
    """A Gaussian likelihood with correlated noise: a model mean in CUDA C++ and a dense data covariance.
    ``source`` defines::

        __device__ double model_mean(const double* theta, const double* row);   // E[y_i | theta] at row x_i
        __device__ double ln_prior(const double* theta);                        // only when prior=True

    ``x`` is a finite float64 array of shape ``(M, k)`` (a 1-D array is ``(M, 1)``), 1 <= M <= 32768, and ``row``
    points at the k values of x_i; ``y`` is finite of shape ``(M,)``; ``cov`` is finite, ``(M, M)``, symmetric
    (max |C - C^T| <= 1e-12 max |C|; its lower triangle is used) and positive definite, as scipy's
    ``multivariate_normal`` requires by default.  ``BPM_DIM``, ``BPM_NROWS`` (M), ``BPM_ROWLEN`` (k) and
    ``BPM_HAS_PRIOR`` are macros; the scope, ``fmad``, the NaN rule and ``CudaCompileError`` are those of
    ``CudaLikelihood``.  The value is::

        ln L(theta) = ln_prior(theta) + (-0.5 (c0 + |(m(theta) - y) . B|^2))

    with C = L L^T the Cholesky factor (numpy, on the host), B = L^-T and c0 = M ln(2 pi) + 2 sum_i ln L_ii: it
    equals ``scipy.stats.multivariate_normal(m(theta), cov).logpdf(y) + ln_prior(theta)`` to rounding.  It is
    exactly ``-inf`` when ``ln_prior`` is ``-inf``, whatever ``model_mean`` returns there.  The order of every
    addition is fixed by M alone, so a given theta gets the same bits whatever the batch or the number of chains.
    Each generation runs the proposal kernel, then the model means of every chain, the quadratic form on the FP64
    tensor pipe (half of it: B is triangular) and a finish kernel, then the accept kernel, at every d.  The source,
    dim, M, k, ``prior`` and ``fmad`` are the cache key: new ``y`` or ``cov`` of the same shape reuse the module.

    Which form to use: ``CudaSumLikelihood`` when the noise is independent (a diagonal covariance) -- it costs O(M)
    per chain against this form's O(M^2).  This form when the errors are correlated: a calibration shared by all
    points, drift, overlapping bins, a covariance shipped with the data.  One problem and one rank only.  Pass it
    as ``ln_like_cuda=``."""

    MAX_ROWS = 32768

    def __init__(self, source, dim, x, y, cov, prior=False, fmad=True):
        super(CudaGaussLikelihood, self).__init__(source, dim, x, fmad)
        M = self.data.shape[0]
        y = np.asarray(y, dtype=np.float64)
        if y.shape != (M,):
            raise ValueError("y must have shape (%d,) (one value per row of x), not %s" % (M, y.shape))
        if not np.all(np.isfinite(y)):
            raise ValueError("y must be finite")
        cov = np.asarray(cov, dtype=np.float64)
        if cov.shape != (M, M):
            raise ValueError("cov must have shape (%d, %d), not %s" % (M, M, cov.shape))
        if not np.all(np.isfinite(cov)):
            raise ValueError("cov must be finite")
        if np.max(np.abs(cov - cov.T)) > 1e-12 * np.max(np.abs(cov)):
            raise ValueError("cov must be symmetric: max |C - C^T| > 1e-12 max |C|")
        self.prior = bool(prior)
        self.y = np.ascontiguousarray(y)
        self.cov = cov
        self.B, self.c0 = self.factor(cov)

    @staticmethod
    def factor(cov):
        """``(B, c0)`` of a symmetric covariance (its lower triangle is used): B = L^-T, upper triangular, and
        c0 = M ln(2 pi) + ln det C.  ValueError unless C is positive definite by scipy's test (``_PSD``: every
        eigenvalue above 1e6 eps max |eigenvalue|)."""
        import scipy.linalg
        M = cov.shape[0]
        low = np.tril(cov) + np.tril(cov, -1).T
        s = np.linalg.eigvalsh(low)
        eps = 1e6 * np.finfo(np.float64).eps * np.max(np.abs(s))
        if np.min(s) <= eps:
            raise ValueError("cov must be positive definite (smallest eigenvalue %.3g, scipy's threshold %.3g)"
                             % (np.min(s), eps))
        try:
            L = np.linalg.cholesky(low)
        except np.linalg.LinAlgError:
            raise ValueError("cov must be positive definite (its Cholesky factorisation failed)")
        Linv = scipy.linalg.solve_triangular(L, np.eye(M), lower=True)
        B = np.ascontiguousarray(np.triu(Linv.T))
        c0 = M * np.log(2.0 * np.pi) + 2.0 * np.sum(np.log(np.diag(L)))
        return B, float(c0)

    @staticmethod
    def _shaped(data):
        data = CudaSumLikelihood._shaped(data)
        if data.shape[0] > CudaGaussLikelihood.MAX_ROWS:
            raise ValueError("x has %d rows: M must be in [1, %d]" % (data.shape[0], CudaGaussLikelihood.MAX_ROWS))
        return data

    @property
    def x(self):
        return self.data

    def _compile_call(self, lib):
        M, k = self.data.shape
        return lib.bpm_jit_compile_gauss, (self.source.encode(), self.dim, M, k)

    def _attach_call(self, lib, handle):
        M, k = self.data.shape
        return lib.bpm_set_jit_gauss_target, (handle, self.source.encode(), _lib.dptr(self.data), M, k,
                                              _lib.dptr(self.y), _lib.dptr(self.B), self.c0)

    @property
    def _flags(self):
        return (1 if self.fmad else 0) | (2 if self.prior else 0)
