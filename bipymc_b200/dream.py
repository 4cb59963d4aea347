"""DreamMpi -- drop-in for bipymc/dream.py:12-144 on a device-resident population.

Adds to DeMcMpi the DREAM proposal (randomised-subspace crossover mask, ``del_pairs``
pair differences, the gamma jump-rate schedule, ``e`` / ``epsilon`` jitter,
dream.py:32-107) and the crossover-probability adaptation (dream.py:109-140), both
evaluated inside the CUDA generation kernels (bipymc_b200/csrc).

Differences from the reference, all deliberate and documented in DESIGN.md:
  * ``p_cr`` is refreshed once per generation from the summed jump statistics of all
    chains, not after every single chain-step (a batched kernel cannot serialise chains;
    the sums -- and hence ``p_cr`` at every generation boundary -- are the same);
  * the per-chain history standard deviation comes from running (Welford) moments, not a
    fresh ``np.std`` over the whole history per step (same value to ~1e-16 relative);
  * with several ranks the CR statistics are all-reduced, so every rank adapts the same
    ``p_cr`` (the reference keeps them per rank, dream.py:113-117).
"""
from __future__ import print_function, division
import ctypes as C

import numpy as np

from . import _lib
from .demc import DeMcMpi


class DreamMpi(DeMcMpi):
    _algo = _lib.BPM_ALGO_DREAM

    def __init__(self, ln_like_fn, theta_0=None, varepsilon=1e-6, n_chains=8,
                 mpi_comm=None, ln_kwargs={}, **kwargs):
        self.gamma_scale = kwargs.get("gamma_scale", 1.0)       # dream.py:20
        self.del_pairs = kwargs.get("del_pairs", 3)             # dream.py:22
        self.burnin_gen = kwargs.get("burnin_gen", 300)         # dream.py:24
        self.p_cr_update_gen = kwargs.get("n_cr_gen", 50)       # dream.py:26
        self.n_cr = kwargs.get("n_cr", 3)                       # dream.py:27
        if not 1 <= self.del_pairs <= _lib.BPM_MAX_PAIRS:
            raise ValueError("del_pairs must be in [1, %d]" % _lib.BPM_MAX_PAIRS)
        if not 1 <= self.n_cr <= _lib.BPM_MAX_CR:
            raise ValueError("n_cr must be in [1, %d]" % _lib.BPM_MAX_CR)
        super(DreamMpi, self).__init__(ln_like_fn, theta_0=theta_0, varepsilon=varepsilon,
                                       n_chains=n_chains, mpi_comm=mpi_comm, ln_kwargs=ln_kwargs,
                                       **kwargs)
        self.CR = (np.array(range(self.n_cr)) + 1) / self.n_cr
        if not getattr(self, "_cr_restored", False):            # a warm start restored it already
            self._init_cr()

    def _dream_cfg(self):
        return dict(del_pairs=int(self.del_pairs), n_cr=int(self.n_cr), burnin_gen=int(self.burnin_gen),
                    n_cr_gen=int(self.p_cr_update_gen), gamma_scale=float(self.gamma_scale))

    def _run_params(self, kwargs):
        flip = float(np.clip(kwargs.get("flip", 0.5), 0.0, 1.0))       # demc.py:73
        shuffle = 1 if kwargs.get("shuffle", True) else 0               # demc.py:74
        epsilon = float(kwargs.get("epsilon", 1e-12))                   # dream.py:40
        u_epsilon = float(kwargs.get("u_epsilon", 1e-2))                # dream.py:41
        return flip, shuffle, epsilon, u_epsilon, 0.0

    # ---- crossover state lives on the device; these read / write it -----------------
    def _init_cr(self):
        """dream.py:109-117."""
        self.CR = (np.array(range(self.n_cr)) + 1) / self.n_cr
        shape = self._cr_shape()
        self._set_cr(np.ones(shape) / self.n_cr, np.zeros(shape), np.zeros(shape))

    def _cr_shape(self):
        """[n_cr], or [P, n_cr] on a multi-problem sampler (one row per problem)."""
        return (self.n_problems, self.n_cr) if self._multi else (self.n_cr,)

    def _set_cr(self, p_cr, delta_m, n_cr_updates):
        a = [np.ascontiguousarray(np.asarray(v, dtype=np.float64).reshape(self._cr_shape()))
             for v in (p_cr, delta_m, n_cr_updates)]
        fn = self._libh.bpm_set_problem_cr_state if self._multi else self._libh.bpm_set_cr_state
        _lib.check(fn(self._handle, _lib.dptr(a[0]), _lib.dptr(a[1]), _lib.dptr(a[2])))

    def _get_cr(self):
        out = [np.zeros(self._cr_shape()) for _ in range(3)]
        fn = self._libh.bpm_get_problem_cr_state if self._multi else self._libh.bpm_get_cr_state
        _lib.check(fn(self._handle, _lib.dptr(out[0]), _lib.dptr(out[1]), _lib.dptr(out[2])))
        return out

    @property
    def p_cr(self):
        return self._get_cr()[0]

    @p_cr.setter
    def p_cr(self, v):
        _, dm, cnt = self._get_cr()
        self._set_cr(v, dm, cnt)

    @property
    def delta_m(self):
        return self._get_cr()[1]

    @property
    def n_cr_updates(self):
        return self._get_cr()[2]

    @property
    def p_cr_update(self):
        return self.p_cr

    def _checkpoint_extra(self):
        e = super(DreamMpi, self)._checkpoint_extra()
        p_cr, dm, cnt = self._get_cr()       # (flat: [P n_cr] on a multi-problem sampler)
        e.update(b200_p_cr=p_cr.ravel(), b200_delta_m=dm.ravel(), b200_n_cr_updates=cnt.ravel())
        return e

    def _restore_extra_late(self, extra):
        if "b200_p_cr" in extra:
            self._set_cr(extra["b200_p_cr"], extra["b200_delta_m"], extra["b200_n_cr_updates"])
            self._cr_restored = True

    def _outlier_active(self, k_gen):
        return self.outlier_gen > 0 and k_gen < self.burnin_gen

    @property
    def in_burnin(self):
        return True                                             # dream.py:142-144
