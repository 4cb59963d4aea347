"""DeMc -- drop-in for the serial DE-MC sampler bipymc/samplers.py:237-324 on the device.

Same constructor and ``run_mcmc(n, theta_0, varepsilon=1e-6, gamma=..., inflate=1e1)``.  The
reference's default ``delayed_accept=True`` schedule -- every chain of a sweep proposes from
the frozen previous states, partners drawn from ALL other chains, the whole sweep appended
afterwards (samplers.py:271-308) -- is one kernel sweep over the population here
(BPM_ALGO_DEMC_SERIAL: no a/b split, no shuffle, no gamma jumps; proposal, likelihood and
accept run as separate launches, so no chain ever sees a partner updated in the same sweep).
``delayed_accept=False`` (chain i is updated before chain i+1 proposes) is inherently
sequential and is not offered on the device.
"""
from __future__ import print_function, division
import ctypes as C

import numpy as np

from . import _lib
from .demc import DeMcMpi, GaussianProposalStub, _SingleComm, _default_comm, _resolve_comm, _torch
from .util import var_ball_batch


class DeMc(DeMcMpi):
    _algo = _lib.BPM_ALGO_DEMC_SERIAL
    _n_phases = 1

    def __init__(self, log_like_fn, n_chains=8, ln_kwargs={}, **proposal_kwargs):
        assert n_chains >= 4                                        # samplers.py:249
        self.n_chains = n_chains
        self.comm = _resolve_comm(proposal_kwargs.get("mpi_comm", None))
        if n_chains % self.comm.size != 0:
            raise ValueError("n_chains (%d) must be divisible by the number of ranks (%d)" % (n_chains, self.comm.size))
        self.am_chains = []                                         # samplers.py:23
        self.log_like_fn = log_like_fn
        self._ln_kwargs = dict(ln_kwargs)
        self._freeze_ln_like_fn(**ln_kwargs)
        self.mcmc_proposal = GaussianProposalStub(self.frozen_ln_like_fn)
        self.n_accepted, self.n_rejected = 1, 0                     # samplers.py:30-31
        self.local_n_accepted, self.local_n_rejected = 0, 0
        self.dim = None
        self.h5_file = proposal_kwargs.get("h5_file", "sampler_checkpoint.h5")
        self.warm_start, self.checkpoint = False, 0
        self._seed = proposal_kwargs.get("seed", None)
        self._history_policy = proposal_kwargs.get("history", "full")
        self._ln_like_batched = proposal_kwargs.get("ln_like_batched", None)
        self._ln_like_cuda = proposal_kwargs.get("ln_like_cuda", None)
        self._device_index = proposal_kwargs.get("device", None)
        self._fused = False                                         # the sweep uses the split launches
        self._chunk_bytes = int(proposal_kwargs.get("history_chunk_bytes", 1 << 30))
        self._reserve_rows = int(proposal_kwargs.get("history_reserve", 0))
        # A sweep is ONE phase in which every chain reads all other chains of the frozen population, so
        # accepted rows must not reach another rank's replica while that rank is still proposing: the
        # in-kernel peer stores of exchange="p2p" would race.  Several ranks therefore always refresh the
        # replicas with an all-gather AFTER the sweep (a collective nobody completes before everyone has
        # finished reading), whatever `exchange` asks for.
        self._exchange = proposal_kwargs.get("exchange", "p2p") if self.comm.size == 1 else "allgather"
        self.subpop_k = 0
        self._peer_ptrs, self._own_X_ptr = [], None
        self._sync_peer_ptrs, self._own_sync_ptr, self._sync_on = [], None, False
        self._peer_sync_wanted = False
        self.outlier_gen, self.n_outlier_resets = 0, 0
        self._setup_device()

    def _init_chains(self, theta_0, varepsilon=1e-6, **kwargs):
        """samplers.py:255-259: chain i starts at theta_0 + N(0, varepsilon * inflate)."""
        torch = _torch()
        theta_0 = np.asarray(theta_0, dtype=float).flatten()
        d = len(theta_0)
        if self._handle is not None and d != self.dim:
            self._release_peer_memory()
            self._libh.bpm_destroy(self._handle)
            self._handle = None
        self.dim = d
        x0 = theta_0[None, :] + var_ball_batch(np.asarray(varepsilon * kwargs.get("inflate", 1e1)), d,
                                               self.n_chains)
        if self._handle is None:
            self._create_handle()
        if self.comm.size > 1:
            import torch.distributed as dist
            x0t = torch.from_numpy(x0).to(self._device)
            dist.broadcast(x0t, src=0)
            x0 = x0t.cpu().numpy()
        self._set_population(x0)

    def run_mcmc(self, n, theta_0, **kwargs):                       # samplers.py:60-66
        self._mcmc_run(n, theta_0, **kwargs)

    def _mcmc_run(self, n, theta_0, varepsilon=1e-6, **kwargs):
        if not kwargs.get("delayed_accept", True):
            raise NotImplementedError("delayed_accept=False updates chains one after the other; "
                                      "the device sampler runs the delayed-accept sweep only")
        torch = _torch()
        self._init_chains(theta_0, varepsilon, **kwargs)
        N = self.n_chains
        gamma = float(kwargs.get("gamma", 0.0) or 0.0)              # samplers.py:264 (0 -> 2.38 / sqrt(2 d))
        eps_sd = float(np.sqrt(varepsilon * 1e-3)) if varepsilon * 1e-3 > 0 else 0.0   # samplers.py:286
        _lib.check(self._libh.bpm_reset_counters(self._handle))
        _lib.check(self._libh.bpm_set_run_params(self._handle, 0.5, 0, eps_sd, 0.0, gamma))
        _lib.check(self._libh.bpm_omega_track(self._handle, 0))
        self._init_lnl()
        G = -(-(n - N) // N) if n > N else 0                        # while j < n - n_chains: j += n_chains
        replay = kwargs.get("_replay", None)
        trace = kwargs.get("_trace", None)
        if replay is not None:
            G = min(G, len(replay))
        k_gen, mode = 0, self._mode()
        while k_gen < G:
            base, avail = self._hist.reserve(G - k_gen)
            avail = min(avail, G - k_gen)
            st = self._state(base)
            if replay is not None:
                self._replay_generation(st, replay[k_gen], k_gen, trace)
                done = 1
            elif mode == "device" and self.comm.size == 1:
                done = avail
                _lib.check(self._libh.bpm_step_generations(self._handle, C.byref(st), k_gen, done,
                                                           self._stream()))
            else:
                self._split_generation(st, k_gen)
                done = 1
            self._hist.advance(done)
            self._mom_len += done
            k_gen += done
        torch.cuda.synchronize(self._device)
        acc, rej, nan = C.c_uint64(), C.c_uint64(), C.c_int32()
        _lib.check(self._libh.bpm_get_counters(self._handle, C.byref(acc), C.byref(rej), C.byref(nan)))
        if nan.value:
            raise ValueError("probabilities contain NaN")           # numpy's message at samplers.py:336
        a, r = int(acc.value), int(rej.value)
        if self.comm.size > 1:
            import torch.distributed as dist
            t = torch.tensor([a, r], dtype=torch.int64, device=self._device)
            dist.all_reduce(t)
            a, r = int(t[0].item()), int(t[1].item())
        self.n_accepted += a                                        # samplers.py:294,297 (never reset)
        self.n_rejected += r

    def param_est(self, n_burn):
        """samplers.py:311-315."""
        chain_slice = self.super_chain[n_burn:, :]
        return np.mean(chain_slice, axis=0), np.std(chain_slice, axis=0), chain_slice
