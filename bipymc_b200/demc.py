"""DeMcMpi -- drop-in for bipymc/demc.py:10-338 on a device-resident population.

Same constructor, ``run_mcmc``, ``param_est``, ``save_state`` / ``load_state``,
``super_chain_mpi``, ``gather_all_chains``, ``iter_*_chains``, ``get_chain`` and
attribute surface as the reference.  What changed underneath:

  * the population (current positions, cached log-likelihoods, running moments and the
    full history) lives in torch CUDA tensors; ``am_chains[i]`` are lazy views;
  * ``_mcmc_run`` (demc.py:63-151) issues a few CUDA kernels per generation through the
    C-ABI (include/bipymc_b200.h) instead of looping over chains in Python;
  * the mpi4py rank-per-chain-group layout (demc.py:39,93,116) becomes one process per
    GPU under ``torch.distributed`` (NCCL): each rank owns the contiguous chain block
    ``np.array_split(range(N), world)[rank]`` and keeps a replica of the whole
    population that is refreshed by an all-gather after each half-phase.

Likelihood plug-ins, fastest first:
  1. ``ln_like_fn`` is ``obj.ln_like`` of a built-in target (bipymc_b200.targets): the
     likelihood is evaluated inside the generation kernels;
  1b. ``ln_like_cuda=targets.CudaLikelihood(source, dim, data)``: the user's own
     ``__device__ double ln_like(const double* theta, const double* data)`` (``theta[BPM_DIM]``,
     ``data[BPM_NDATA]``), compiled at run time with NVRTC into the same kernels -- the fused
     d <= 4 half-phase kernel, or a batched row kernel between propose and accept above that.
     ``-INFINITY`` = outside the prior; NaN raises ``ValueError("probabilities contain NaN")``;
     ``fmad=False`` rounds like numpy.  The first compile takes up to about 2 s, later samplers with the
     same source reuse the cubin.  Takes precedence over a built-in target and over
     ``ln_like_batched``; ``ln_like_fn`` stays the drop-in positional argument and is not called;
  1c. ``ln_like_cuda=targets.CudaSumLikelihood(source, dim, data, prior)``: a likelihood that is a sum
     of ``__device__ double ln_like_term(const double* theta, const double* row)`` over the rows of
     ``data[M][k]`` (plus an optional ``ln_prior``), each chain's sum split over the whole GPU between
     the proposal and accept kernels, in an order fixed by M alone;
  2. ``ln_like_batched=f``: ``f(theta)`` takes a CUDA float64 tensor ``[n, dim]`` and
     returns ``[n]`` log-likelihoods (torch ops on the current stream);
  3. any scalar ``ln_like_fn(theta, **ln_kwargs) -> float`` exactly as in the reference
     (samplers.py:36-43): proposals make a host round trip per half-phase -- correct,
     not fast.

There is no CPU fallback: constructing a sampler without a CUDA device raises.
"""
from __future__ import print_function, division
import ctypes as C
import sys

import numpy as np

from . import _lib
from .chain import McmcChain
from .targets import resolve_device_target
from .util import var_ball_batch


def _torch():
    import torch
    return torch


def _try_h5py():
    """The HDF5 module checkpoints go through: h5py where it imports, else the package's own pure-Python
    HDF5 writer / reader (bipymc_b200/h5lite.py, same File / create_dataset / attrs calls)."""
    from . import h5lite
    return h5lite.get_h5()


def _npz_name(h5_file):
    return h5_file if h5_file.endswith(".npz") else h5_file + ".npz"


def shard_bounds(n_chains, size):
    """[lo, hi) of every rank's block = np.array_split(range(N), size) (demc.py:39): the first
    N % size ranks own one extra chain."""
    q, r = divmod(int(n_chains), int(size))
    out, lo = [], 0
    for k in range(size):
        hi = lo + q + (1 if k < r else 0)
        out.append((lo, hi))
        lo = hi
    return out


class _SingleComm(object):
    """Stand-in for MPI.COMM_WORLD when neither mpi4py nor torch.distributed is in use."""
    size, rank = 1, 0

    def Get_size(self):
        return 1

    def Get_rank(self):
        return 0

    def Barrier(self):
        pass


class _TorchComm(object):
    """rank / size / Barrier facade over an initialised torch.distributed group."""
    def __init__(self, dist):
        self._dist = dist
        self.size = dist.get_world_size()
        self.rank = dist.get_rank()

    def Get_size(self):
        return self.size

    def Get_rank(self):
        return self.rank

    def Barrier(self):
        self._dist.barrier()


def _default_comm():
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            return _TorchComm(dist)
    except Exception:
        pass
    return _SingleComm()


def _resolve_comm(mpi_comm):
    """The communicator the sampler shards over.  Collectives run on torch.distributed (NCCL / gloo);
    an mpi4py communicator is accepted for signature compatibility (demc.py:15) but it must describe the
    SAME world: same size and rank as the initialised torch.distributed group, else the ranks would be
    mis-sharded silently or fail deep inside init_chains."""
    if mpi_comm is None or not hasattr(mpi_comm, "rank"):
        return _default_comm()
    if isinstance(mpi_comm, (_SingleComm, _TorchComm)):
        return mpi_comm
    size = int(mpi_comm.Get_size()) if hasattr(mpi_comm, "Get_size") else int(getattr(mpi_comm, "size", 1))
    rank = int(mpi_comm.Get_rank()) if hasattr(mpi_comm, "Get_rank") else int(mpi_comm.rank)
    if size == 1:
        return mpi_comm
    try:
        import torch.distributed as dist
        ok = dist.is_available() and dist.is_initialized()
    except Exception:
        ok = False
    if not ok:
        raise RuntimeError("mpi_comm has %d ranks but torch.distributed is not initialised: bipymc_b200 runs its "
                           "collectives on torch.distributed (one process per GPU, e.g. under torchrun); call "
                           "torch.distributed.init_process_group first" % size)
    if dist.get_world_size() != size or dist.get_rank() != rank:
        raise RuntimeError("mpi_comm (rank %d of %d) and the torch.distributed group (rank %d of %d) disagree"
                           % (rank, size, dist.get_rank(), dist.get_world_size()))
    return _TorchComm(dist)


class GaussianProposalStub(object):
    """The reference instantiates a GaussianProposal in every sampler ctor
    (samplers.py:27) but never calls it on the DE-MC / DREAM path; keep the attribute."""
    def __init__(self, frozen_ln_like_fn):
        self._frozen_ln_like_fn = frozen_ln_like_fn
        self._cov_init = False
        self._mu = None
        self._cov = None


class HistoryStore(object):
    """Device history ``[T][n_local][ld]`` in growable chunks.

    Flattened to ``(T * n_local, d)`` a chunk *is* the reference's interlaced super
    chain (demc.py:260-268).  ``policy``: "full" keeps every generation (drop-in
    default); "none" keeps only the rows present at construction / load time (running
    moments still see every generation).  ``length`` is the LOGICAL chain length
    (generations + 1, what ``len(chain.chain)`` is in the reference); ``stored`` the
    number of rows physically kept."""
    def __init__(self, n_local, dim, ld, device, policy="full", chunk_bytes=1 << 28, reserve_rows=0):
        import torch
        if policy not in ("full", "none"):
            raise ValueError("history must be 'full' or 'none'")
        self._torch = torch
        self.n_local, self.dim, self.ld, self.device = n_local, dim, ld, device
        self.policy = policy
        self.row_bytes = n_local * ld * 8
        self.chunk_rows = max(1, int(chunk_bytes // self.row_bytes), int(reserve_rows))
        self.reserve_rows = int(reserve_rows)
        self.chunks = []      # list of [rows, n_local, ld] tensors
        self.stored = 0
        self.length = 0
        self._current = None  # [n_local, ld] view of the live population rows
        # the fused kernels leave the newest row pending (bpm_state.pending); the owner sets this to a
        # callable that materialises it, run before anything reads the stored rows
        self._before_read = None

    def will_grow(self):
        """The next reserve() allocates a new chunk."""
        return self.policy == "full" and (not self.chunks or self._used_in_last() == self.chunks[-1].shape[0])

    def flat_base(self):
        """Address row 0 of one flat [T][n_local][ld] array would have so that the rows of the LAST chunk
        sit where they are (what reserve() returned for that chunk); None when nothing is kept."""
        if self.policy != "full" or not self.chunks:
            return None
        return self.chunks[-1].data_ptr() - (self.length - self._used_in_last()) * self.row_bytes

    def _used_in_last(self):
        return self.stored - sum(c.shape[0] for c in self.chunks[:-1]) if self.chunks else 0

    def reserve(self, rows):
        """Room for up to `rows` more generations: returns (base_address, rows_available),
        base_address being where row 0 of one flat [T][n_local][ld] array would sit so
        that row `length` lands on the next free row of the last chunk.  (None, rows)
        when nothing is kept."""
        if self.policy != "full":
            return None, rows
        torch = self._torch
        used = self._used_in_last()
        if not self.chunks or used == self.chunks[-1].shape[0]:
            n = min(self.chunk_rows, max(rows, self.reserve_rows, 1))
            if len(self.chunks) == 1 and self.stored == 1:
                # only the initial row so far: fold it into the new chunk so a single
                # run_mcmc leaves ONE contiguous [T][n_local][ld] block (no later concat)
                first = self.chunks[0]
                blk = torch.empty((n + 1, self.n_local, self.ld), dtype=torch.float64,
                                  device=self.device)
                blk[0].copy_(first[0])
                self.chunks = [blk]
                used = 1
            else:
                self.chunks.append(torch.empty((n, self.n_local, self.ld), dtype=torch.float64,
                                               device=self.device))
                used = 0
        last = self.chunks[-1]
        base = last.data_ptr() - (self.length - used) * self.row_bytes
        return base, last.shape[0] - used

    def reserve_contiguous(self, rows):
        """Like reserve(), but every stored row AND the next `rows` rows sit in ONE block, so the returned base is
        a real array base: replay steps walk the whole stored history of a chain (exact np.std, step.cuh:
        cr_variance) and must not cross a chunk boundary through the synthetic base of reserve()."""
        if self.policy != "full":
            return None, rows
        torch = self._torch
        used = self._used_in_last()
        if len(self.chunks) == 1 and self.chunks[0].shape[0] - used >= 1:
            return self.chunks[0].data_ptr(), self.chunks[0].shape[0] - used
        whole = self.tensor()                                   # coalesced [stored, n_local, ld]
        blk = torch.empty((self.stored + max(rows, self.reserve_rows, 1), self.n_local, self.ld), dtype=torch.float64,
                          device=self.device)
        blk[:self.stored].copy_(whole)
        self.chunks = [blk]
        return blk.data_ptr(), blk.shape[0] - self.stored

    def advance(self, rows):
        self.length += rows
        if self.policy == "full":
            self.stored += rows

    def set_initial(self, state):
        """state: [n_local, ld] device tensor = row 0 of every chain."""
        torch = self._torch
        self.chunks = [torch.empty((1, self.n_local, self.ld), dtype=torch.float64, device=self.device)]
        self.chunks[0][0].copy_(state)
        self.stored = self.length = 1

    def tensor(self):
        """[stored, n_local, ld] (concatenates chunks when there are several)."""
        torch = self._torch
        if self._before_read is not None:
            self._before_read()
        parts, left = [], self.stored
        for c in self.chunks:
            take = min(left, c.shape[0])
            if take > 0:
                parts.append(c[:take])
            left -= take
        if len(parts) > 1:          # coalesce once so later reads are free
            whole = torch.cat(parts, dim=0)
            self.chunks = [whole]
            return whole
        return parts[0]

    def chain_host(self, li):
        return self.tensor()[:, li, :self.dim].cpu().numpy()

    def set_chain_host(self, li, arr):
        t = self.tensor()
        if arr.shape[0] != t.shape[0]:
            raise ValueError("chain length mismatch: use the sampler's load_history() to replace "
                             "histories of a different length")
        t[:, li, :self.dim] = self._torch.from_numpy(np.ascontiguousarray(arr)).to(self.device)

    def current_host(self, li):
        return self._current[li, :self.dim].cpu().numpy()

    def load(self, hist):
        """hist: numpy (T, n_local, dim) -> replaces the stored history."""
        torch = self._torch
        T = hist.shape[0]
        t = torch.zeros((T, self.n_local, self.ld), dtype=torch.float64, device=self.device)
        t[:, :, :self.dim] = torch.from_numpy(np.ascontiguousarray(hist)).to(self.device)
        self.chunks = [t]
        self.stored = self.length = T


class _ChainList(object):
    """``am_chains``: a sequence of lazily created McmcChain views (one per local chain)."""
    def __init__(self, sampler):
        self._s = sampler
        self._cache = {}

    def __len__(self):
        return len(self._s.rank_chain_ids)

    def __bool__(self):
        return len(self) > 0

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [self[j] for j in range(*i.indices(len(self)))]
        if i < 0:
            i += len(self)
        if not 0 <= i < len(self):
            raise IndexError(i)
        ch = self._cache.get(i)
        if ch is None:
            ch = McmcChain(None, global_id=int(self._s.rank_chain_ids[i]), _store=self._s._hist,
                           _local_index=i)
            self._cache[i] = ch
        return ch

    def __iter__(self):
        for i in range(len(self)):
            yield self[i]


class DeMcMpi(object):
    """Parallel DE-MC (emcee-style a/b pools) on B200; mirrors bipymc/demc.py:10."""
    _algo = _lib.BPM_ALGO_DEMC
    _n_phases = 2

    def __init__(self, ln_like_fn, theta_0=None, varepsilon=1e-6, n_chains=8,
                 mpi_comm=None, ln_kwargs={}, **kwargs):
        varepsilon = np.asarray(varepsilon)
        assert n_chains >= 4                                   # samplers.py:249
        self.n_chains = n_chains
        self.comm = _resolve_comm(mpi_comm)
        if n_chains % self.comm.size != 0:
            # the reference counts j per rank (demc.py:79,103-109): ranks with fewer chains run more
            # generations and its fixed-count Allgather (demc.py:93) mismatches -- it hangs.  Say so.
            raise ValueError("n_chains (%d) must be divisible by the number of ranks (%d)"
                             % (n_chains, self.comm.size))
        self.local_n_accepted = 0
        self.local_n_rejected = 1                               # demc.py:19-20
        if theta_0 is not None:
            self.dim = len(np.asarray(theta_0))
        else:
            self.dim = kwargs.get("dim", 1)
        self.h5_file = kwargs.get("h5_file", "sampler_checkpoint.h5")
        self.warm_start = kwargs.get("warm_start", False)
        self.checkpoint = kwargs.get("checkpoint", 0)
        # McmcSampler.__init__ (samplers.py:16-31)
        self.log_like_fn = ln_like_fn
        self._ln_kwargs = dict(ln_kwargs)
        self._freeze_ln_like_fn(**ln_kwargs)
        self.mcmc_proposal = GaussianProposalStub(self.frozen_ln_like_fn)
        self.n_accepted, self.n_rejected = 1, 0
        # B200 extensions (all optional)
        self._seed = kwargs.get("seed", None)
        self._history_policy = kwargs.get("history", "full")
        self._ln_like_batched = kwargs.get("ln_like_batched", None)
        self._ln_like_cuda = kwargs.get("ln_like_cuda", None)
        self._device_index = kwargs.get("device", None)
        self._fused = kwargs.get("fused", True)
        self._chunk_bytes = int(kwargs.get("history_chunk_bytes", 1 << 30))
        self._reserve_rows = int(kwargs.get("history_reserve", 0))   # generations to pre-allocate
        # IQR outlier-chain reset every `outlier_gen` generations (0 = off, the reference's
        # behaviour); DREAM applies it only while k < burnin_gen (Vrugt et al. 2009)
        # multi-GPU exchange of updated chain states: "p2p" = accepted rows are stored into the
        # peer replicas from inside the kernels (CUDA IPC peer memory over NVLink) and only a
        # tiny barrier collective runs between half-phases; "allgather" = NCCL all-gather of
        # every rank's shard after each half-phase (the reference's comm.Allgather, demc.py:93,116)
        self._exchange = kwargs.get("exchange", "p2p")
        if self._exchange not in ("p2p", "allgather"):
            raise ValueError("exchange must be 'p2p' or 'allgather'")
        # sub-population ("island") mode for populations whose full replica does not fit or whose
        # per-generation exchange would dominate (BASELINE config 5): every rank steps ITS chains
        # as a self-contained population -- pairs come from the local opposite half, no replica,
        # no per-generation communication -- and every `subpop_k` generations the chains are
        # re-dealt across the ranks (one all-to-all), so each island receives 1/G of every island.
        # A different sampler than the reference's single population, hence opt-in and stated.
        self.subpop_k = int(kwargs.get("subpop_k", 0))
        self._peer_ptrs, self._own_X_ptr = [], None
        self._sync_peer_ptrs, self._own_sync_ptr, self._sync_on = [], None, False
        # peer_sync=False keeps the round-1 protocol (NCCL all-reduce as the barrier between half-phases)
        self._peer_sync_wanted = bool(kwargs.get("peer_sync", True))
        self.outlier_gen = int(kwargs.get("outlier_gen", 0))
        self.n_outlier_resets = 0
        self._setup_device()
        if not self.warm_start:
            self.init_chains(theta_0, varepsilon, **kwargs)
        else:
            self.init_warmstart_chain(self.h5_file)

    # ------------------------------------------------------------------ plumbing
    def _freeze_ln_like_fn(self, **kwargs):
        self._frozen_ln_like_fn = lambda theta: self.log_like_fn(theta, **kwargs)

    @property
    def frozen_ln_like_fn(self):
        return self._frozen_ln_like_fn

    def _setup_device(self):
        torch = _torch()
        self._libh = _lib.load()                       # raises if the CUDA library is missing
        if not torch.cuda.is_available():
            raise RuntimeError("bipymc_b200 needs a CUDA device (B200); there is no CPU fallback")
        if self._device_index is None:
            self._device_index = torch.cuda.current_device() if self.comm.size == 1 else \
                self.comm.rank % torch.cuda.device_count()
        self._device = torch.device("cuda", self._device_index)
        torch.cuda.set_device(self._device)
        self._handle = None
        self._hist = None

    def _dream_cfg(self):
        return dict(del_pairs=1, n_cr=1, burnin_gen=0, n_cr_gen=0, gamma_scale=1.0)

    @property
    def _subpop(self):
        return self.subpop_k > 0 and self.comm.size > 1

    @property
    def _sharded(self):
        """Several ranks stepping ONE population (replicas + exchange)."""
        return self.comm.size > 1 and not self._subpop

    def _local_range(self):
        """Row range of this rank's chains inside self._X / self._lnl."""
        if self._subpop:
            return 0, len(self.rank_chain_ids)
        return int(self.rank_chain_ids[0]), int(self.rank_chain_ids[-1]) + 1

    def _create_handle(self):
        d = self.dim
        if self._ln_like_cuda is not None:
            from .targets import CudaLikelihood
            if not isinstance(self._ln_like_cuda, CudaLikelihood):
                raise TypeError("ln_like_cuda must be a targets.CudaLikelihood or targets.CudaSumLikelihood")
            if self._ln_like_cuda.dim != d:
                raise ValueError("ln_like_cuda dimension %d != theta_0 dimension %d" % (self._ln_like_cuda.dim, d))
        self._ld = d if d <= 4 else ((d + 3) // 4) * 4
        ids = np.array_split(np.arange(self.n_chains), self.comm.size)[self.comm.rank]
        self.rank_chain_ids = ids                                   # demc.py:39-40
        if self._seed is None:
            # keep np.random.seed(...) meaningful for the native stream as well
            self._seed = int(np.random.randint(0, 2 ** 31 - 1))
            if self.comm.size > 1:
                self._seed = self._bcast_int(self._seed)
        dc = self._dream_cfg()
        if self._subpop:
            # an island is a complete, unsharded population of its own with its own Philox key
            n_eng, c_lo, c_hi = len(ids), 0, len(ids)
            seed = (self._seed + 0x9E3779B97F4A7C15 * (self.comm.rank + 1)) % (1 << 64)
        else:
            n_eng, c_lo, c_hi, seed = self.n_chains, int(ids[0]), int(ids[-1]) + 1, self._seed
        self._n_engine = n_eng
        cfg = _lib.Config(algo=self._algo, n_chains=n_eng, dim=d, ld=self._ld,
                          del_pairs=dc["del_pairs"], n_cr=dc["n_cr"], burnin_gen=dc["burnin_gen"],
                          n_cr_gen=dc["n_cr_gen"], shuffle=1, chain_lo=c_lo,
                          chain_hi=c_hi, device=self._device_index,
                          gamma_scale=dc["gamma_scale"], flip=0.5, epsilon=0.0, u_epsilon=0.0,
                          gamma=0.0, seed=seed)
        h = C.c_void_p()
        _lib.check(self._libh.bpm_create(C.byref(cfg), C.byref(h)))
        self._handle = h
        _lib.check(self._libh.bpm_set_fused(h, int(self._fused)))   # 0 split, 1 fused, 2 fused (two-halves variant)
        if self._ln_like_cuda is not None:
            self._target = self._ln_like_cuda
            self._jit_from_cache = self._target._attach(self._libh, h)     # True: the cubin came from the cache
            return
        self._target = resolve_device_target(self.log_like_fn, self._ln_kwargs)
        if self._target is not None:
            if self._target.dim != d:
                raise ValueError("target dimension %d != theta_0 dimension %d" % (self._target.dim, d))
            p = self._target.params
            _lib.check(self._libh.bpm_set_target(h, self._target.target_id, _lib.dptr(p), p.size))

    def _bcast_int(self, v):
        torch = _torch()
        import torch.distributed as dist
        t = torch.tensor([v], dtype=torch.int64, device=self._device)
        dist.broadcast(t, src=0)
        return int(t.item())

    def __del__(self):
        try:
            self._release_peer_memory()
            if getattr(self, "_handle", None) is not None:
                self._libh.bpm_destroy(self._handle)
                self._handle = None
        except Exception:
            pass

    def close(self):
        """Release the engine handle and (sharded runs) the peer mappings.  Collective when the
        population is sharded over peer memory: every rank must call it, because a rank's
        replica must not disappear while a peer kernel may still store into it."""
        torch = _torch()
        if getattr(self, "_handle", None) is None:
            return
        torch.cuda.synchronize(self._device)
        if self._sharded and self._peer_ptrs:
            import torch.distributed as dist
            dist.barrier()
        self._release_peer_memory()
        self._libh.bpm_destroy(self._handle)
        self._handle = None

    # ------------------------------------------------------------------ peer memory
    def _release_peer_memory(self):
        lib = getattr(self, "_libh", None)
        if lib is None:
            return
        if getattr(self, "_handle", None) is not None and getattr(self, "_peer_ptrs", None):
            lib.bpm_set_peers(self._handle, None, 0)
        for q in getattr(self, "_peer_ptrs", []):
            lib.bpm_ipc_close(self._device_index, C.c_void_p(q))
        self._peer_ptrs = []
        if getattr(self, "_handle", None) is not None and getattr(self, "_sync_on", False):
            lib.bpm_set_sync(self._handle, None, 0, 0)
        self._sync_on = False
        for q in getattr(self, "_sync_peer_ptrs", []):
            lib.bpm_ipc_close(self._device_index, C.c_void_p(q))
        self._sync_peer_ptrs = []
        if getattr(self, "_own_sync_ptr", None):
            lib.bpm_dev_free(self._device_index, C.c_void_p(self._own_sync_ptr))
            self._own_sync_ptr = None
        if getattr(self, "_own_X_ptr", None):
            self._X = None
            lib.bpm_dev_free(self._device_index, C.c_void_p(self._own_X_ptr))
            self._own_X_ptr = None
        if getattr(self, "_ipc", None):
            self._X = self._lnl = self._mean_t = self._m2_t = None
            self._release_ipc()

    def _ipc_alloc(self, name, shape):
        """Sub-population mode: a float64 device array every OTHER island can read (plain cudaMalloc block, IPC
        handle exchanged once): the re-deal pulls chains straight out of the peers' arrays over NVLink.  Returns
        the torch view; self._ipc[name] = (own pointer, {rank: mapped pointer})."""
        torch = _torch()
        import torch.distributed as dist
        lib = self._libh
        nbytes = int(np.prod(shape)) * 8
        ptr = C.c_void_p()
        _lib.check(lib.bpm_dev_alloc(self._device_index, nbytes, C.byref(ptr)))
        t = self._wrap_device(ptr.value, shape)
        t.zero_()
        hbuf = C.create_string_buffer(64)
        _lib.check(lib.bpm_ipc_export(self._device_index, ptr, hbuf))
        handles = [None] * self.comm.size
        dist.all_gather_object(handles, bytes(hbuf.raw))
        peers = {}
        for r, hb in enumerate(handles):
            if r == self.comm.rank:
                continue
            q = C.c_void_p()
            if lib.bpm_ipc_open(self._device_index, C.create_string_buffer(hb, 64), C.byref(q)) != 0:
                self._ipc_ok = False
                break
            peers[r] = q.value
        self._ipc[name] = (ptr.value, peers)
        return t

    def _release_ipc(self):
        lib = getattr(self, "_libh", None)
        for name, (own, peers) in list(getattr(self, "_ipc", {}).items()):
            for q in peers.values():
                lib.bpm_ipc_close(self._device_index, C.c_void_p(q))
            lib.bpm_dev_free(self._device_index, C.c_void_p(own))
        self._ipc = {}

    def _alloc_population(self, N, ld):
        """[N, ld] float64 population replica.  Sharded runs with exchange="p2p" take it from
        bpm_dev_alloc (a plain cudaMalloc block, so its IPC handle can be opened by the peers)
        and register every other rank's replica with the engine (bpm_set_peers)."""
        torch = _torch()
        if self._subpop:
            if getattr(self, "_ipc", None):
                torch.cuda.synchronize(self._device)
                import torch.distributed as dist
                dist.barrier()
                self._X = self._lnl = self._mean_t = self._m2_t = None
                self._release_ipc()
            self._ipc, self._ipc_ok = {}, True
            return self._ipc_alloc("X", (N, ld))
        if not self._sharded or self._exchange != "p2p":
            return torch.zeros((N, ld), dtype=torch.float64, device=self._device)
        import torch.distributed as dist
        lib = self._libh
        if self._peer_ptrs or self._own_X_ptr:
            torch.cuda.synchronize(self._device)
            dist.barrier()
            self._release_peer_memory()
        ptr = C.c_void_p()
        _lib.check(lib.bpm_dev_alloc(self._device_index, N * ld * 8, C.byref(ptr)))
        self._own_X_ptr = ptr.value
        X = self._wrap_device(ptr.value, (N, ld))
        X.zero_()
        hbuf = C.create_string_buffer(64)
        _lib.check(lib.bpm_ipc_export(self._device_index, ptr, hbuf))
        handles = [None] * self.comm.size
        dist.all_gather_object(handles, bytes(hbuf.raw))
        ok = 1
        for r, hb in enumerate(handles):
            if r == self.comm.rank:
                continue
            q = C.c_void_p()
            if lib.bpm_ipc_open(self._device_index, C.create_string_buffer(hb, 64), C.byref(q)) != 0:
                ok = 0
                break
            self._peer_ptrs.append(q.value)
        flag = torch.tensor([ok], dtype=torch.int32, device=self._device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 0:
            # no peer access between some pair of GPUs: every rank falls back to the NCCL gather
            for q in self._peer_ptrs:
                lib.bpm_ipc_close(self._device_index, C.c_void_p(q))
            self._peer_ptrs = []
            self._exchange = "allgather"
            return X
        arr = (C.c_void_p * len(self._peer_ptrs))(*self._peer_ptrs)
        _lib.check(lib.bpm_set_peers(self._handle, arr, len(self._peer_ptrs)))
        self._bar = torch.zeros((1,), dtype=torch.float32, device=self._device)
        self._setup_peer_sync()
        return X

    def _setup_peer_sync(self):
        """Peer-memory barrier (bpm_set_sync): one small IPC-mapped block per rank; with it a sharded
        generation is a plain sequence of kernels on one stream -- no NCCL call per half-phase."""
        torch = _torch()
        import torch.distributed as dist
        lib = self._libh
        nbytes = C.c_uint64()
        _lib.check(lib.bpm_sync_bytes(C.byref(nbytes)))
        ptr = C.c_void_p()
        _lib.check(lib.bpm_dev_alloc(self._device_index, nbytes.value, C.byref(ptr)))
        self._own_sync_ptr = ptr.value
        self._wrap_device(ptr.value, (nbytes.value // 8,)).zero_()
        torch.cuda.synchronize(self._device)
        hbuf = C.create_string_buffer(64)
        _lib.check(lib.bpm_ipc_export(self._device_index, ptr, hbuf))
        handles = [None] * self.comm.size
        dist.all_gather_object(handles, bytes(hbuf.raw))
        blocks, ok = [], 1
        for r, hb in enumerate(handles):
            if r == self.comm.rank:
                blocks.append(ptr.value)
                continue
            q = C.c_void_p()
            if lib.bpm_ipc_open(self._device_index, C.create_string_buffer(hb, 64), C.byref(q)) != 0:
                ok = 0
                break
            self._sync_peer_ptrs.append(q.value)
            blocks.append(q.value)
        flag = torch.tensor([ok], dtype=torch.int32, device=self._device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)      # also: every block is zeroed before anyone signals
        self._sync_on = bool(int(flag.item())) and self._peer_sync_wanted
        if self._sync_on:
            arr = (C.c_void_p * len(blocks))(*blocks)
            _lib.check(lib.bpm_set_sync(self._handle, arr, self.comm.rank, self.comm.size))

    def _phase_exchange(self, last):
        """Make this half-phase's updates visible on every rank before the next one reads them.
        p2p: the rows are already in the peer replicas, only a barrier is needed (the CR
        all-reduce that follows the second half-phase of a DREAM generation is that barrier)."""
        if not self._sharded:
            return
        if self._exchange == "p2p":
            if last and self._algo == _lib.BPM_ALGO_DREAM:
                return
            if self._sync_on:
                _lib.check(self._libh.bpm_peer_barrier(self._handle, self._stream()))
                return
            import torch.distributed as dist
            dist.all_reduce(self._bar)
        else:
            self._allgather_population()

    # ------------------------------------------------------------------ chains
    def init_chains(self, theta_0, varepsilon=1e-6, **kwargs):
        """demc.py:34-44 + chain.py:25-29: chain c starts at theta_0 + N(0, varepsilon).

        The jitter is drawn on the host from numpy's global stream, chain after chain, so
        a seeded run starts from the reference's initial states.  (``inflate`` is accepted
        and ignored, as in the reference.)"""
        torch = _torch()
        theta_0 = np.asarray(theta_0, dtype=float).flatten()
        self.dim = len(theta_0)
        assert np.all(np.asarray(varepsilon) >= 0.0)
        N, d = self.n_chains, self.dim
        if kwargs.get("device_init", False):
            # populations too large to draw on the host (BASELINE config 5: 10^7 x 1000 doubles = 80 GB):
            # theta_0 + sqrt(varepsilon) * randn on the device, seeded from the sampler's seed.  NOT numpy's
            # stream, so such a run does not start from the reference's initial states -- opt-in, stated.
            if self._handle is None:
                self._create_handle()
            g = torch.Generator(device=self._device)
            g.manual_seed((int(self._seed) * 2654435761 + (self.comm.rank + 1 if self._subpop else 0)) % (1 << 62))
            n_here = len(self.rank_chain_ids) if self._subpop else N
            sd = torch.from_numpy(np.sqrt(np.broadcast_to(np.asarray(varepsilon, dtype=float), (d,))).copy()).to(self._device)
            th = torch.from_numpy(theta_0).to(self._device)
            self._set_population(None, x0_dev=(n_here, lambda out: out.copy_(
                torch.randn(out.shape, generator=g, device=self._device, dtype=torch.float64) * sd + th)))
            return
        # every rank draws the jitter of ALL chains so the replicas agree (demc.py seeds
        # every rank identically as well, tests/test_banana.py:17).  This is the FIRST use
        # of numpy's global stream, exactly as in the reference's constructor.
        x0 = theta_0[None, :] + var_ball_batch(varepsilon, d, N)
        if self._handle is None:
            self._create_handle()          # draws the Philox seed AFTER the jitter
        if self.comm.size > 1:
            x0t = torch.from_numpy(x0).to(self._device)
            import torch.distributed as dist
            dist.broadcast(x0t, src=0)
            x0 = x0t.cpu().numpy()
        self._set_population(x0)

    def _set_population(self, x0, history=None, x0_dev=None):
        torch = _torch()
        N, d, ld = self._n_engine, self.dim, self._ld
        lo, hi = self._local_range()
        nl = hi - lo
        self._X = self._alloc_population(N, ld)
        if x0_dev is not None:    # (rows, fill): the initial states are produced on the device, in place
            rows, fill = x0_dev
            assert rows == N
            if ld == d:
                fill(self._X)
            else:
                tmp = torch.empty((N, d), dtype=torch.float64, device=self._device)
                fill(tmp)
                self._X[:, :d] = tmp
                del tmp
        else:
            if self._subpop:          # x0 covers every chain of the job: keep this island's block
                g0, g1 = int(self.rank_chain_ids[0]), int(self.rank_chain_ids[-1]) + 1
                x0 = np.asarray(x0)[g0:g1]
            self._X[:, :d] = torch.from_numpy(np.ascontiguousarray(x0)).to(self._device)
        if self.comm.size > 1:
            import torch.distributed as dist
            torch.cuda.synchronize(self._device)
            dist.barrier()          # nobody steps before every replica holds the initial states
        self._pending = 0
        if self._subpop:       # every array that travels in a re-deal is readable by the other islands
            self._lnl = self._ipc_alloc("lnl", (N,))
            self._mean_t = self._ipc_alloc("mean", (nl, ld))
            self._mean_t.copy_(self._X[lo:hi])
            self._m2_t = self._ipc_alloc("m2", (nl, ld))
        else:
            self._lnl = torch.zeros((N,), dtype=torch.float64, device=self._device)
            self._mean_t = self._X[lo:hi].clone()
            self._m2_t = torch.zeros((nl, ld), dtype=torch.float64, device=self._device)
        self._hist = HistoryStore(nl, d, ld, self._device, policy=self._history_policy,
                                  chunk_bytes=self._chunk_bytes, reserve_rows=self._reserve_rows)
        self._hist._current = self._X[lo:hi]
        self._hist._before_read = self._flush
        if history is None:
            self._hist.set_initial(self._X[lo:hi])
        else:
            self._hist.load(history)
            self._rebuild_moments()
        self.am_chains = _ChainList(self)
        self._lnl_valid = False
        self._mom_len = self._hist.length
        self._gens_since_deal = 0

    def init_warmstart_chain(self, h5_file):
        """demc.py:46-51."""
        self.init_chains(np.zeros(self.dim))
        self.load_state(h5_file)

    def _get_local_chain_state(self):
        """demc.py:53-57."""
        lo, hi = self._local_range()
        return self._X[lo:hi, :self.dim].cpu().numpy()

    # ------------------------------------------------------------------ C-ABI helpers
    def _stream(self):
        torch = _torch()
        return C.c_void_p(torch.cuda.current_stream(self._device).cuda_stream)

    def _state(self, hist_base=None):
        st = _lib.State()
        st.X = self._X.data_ptr()
        st.lnl = self._lnl.data_ptr()
        st.mean = self._mean_t.data_ptr()
        st.m2 = self._m2_t.data_ptr()
        st.history = hist_base
        st.hist_len = self._hist.length
        st.mom_len = self._mom_len
        st.pending = self._pending
        return st

    # The fused 100-D kernel leaves every chain's newest row pending (include/bipymc_b200.h,
    # bpm_state.pending): counted by the lengths, not yet written to the history / folded into the running
    # moments -- the next generation does that from registers.  Anything that READS the history or the
    # moments goes through _flush() first (HistoryStore.tensor(), the _mean / _m2 properties).
    def _flush(self):
        if not getattr(self, "_pending", 0):
            return
        st = self._state(self._hist.flat_base())
        _lib.check(self._libh.bpm_flush(self._handle, C.byref(st), self._stream()))
        self._pending = int(st.pending)

    @property
    def _mean(self):
        self._flush()
        return self._mean_t

    @property
    def _m2(self):
        self._flush()
        return self._m2_t

    def _rebuild_moments(self):
        """Running mean / M2 of every local chain from the stored history."""
        torch = _torch()
        h = self._hist.tensor()
        self._mean_t = torch.zeros_like(h[0])
        self._m2_t = torch.zeros_like(h[0])
        self._mom_len = self._hist.length
        st = self._state(h.data_ptr())
        _lib.check(self._libh.bpm_moments_from_history(self._handle, C.byref(st), self._stream()))

    # -- streaming diagnostics (no history needed) ------------------------------------
    def reset_moments(self):
        """Restart the per-chain running mean / M2 at the current state (e.g. after
        burn-in), so ``rhat()`` and ``moment_estimates()`` cover only what follows.  The
        reference has no counterpart; note DREAM's CR adaptation then sees the standard
        deviation of the post-reset history only."""
        lo, hi = self._local_range()
        self._flush()
        self._mean_t.copy_(self._X[lo:hi])
        self._m2_t.zero_()
        self._mom_len = 1

    def _gathered_moments(self):
        """(mean, m2) of ALL chains, [N, d] each (all-gathered when sharded)."""
        torch = _torch()
        mean, m2 = self._mean[:, :self.dim].contiguous(), self._m2[:, :self.dim].contiguous()
        if self.comm.size > 1:
            import torch.distributed as dist
            pm = [torch.empty_like(mean) for _ in range(self.comm.size)]
            p2 = [torch.empty_like(m2) for _ in range(self.comm.size)]
            dist.all_gather(pm, mean)
            dist.all_gather(p2, m2)
            mean, m2 = torch.cat(pm, dim=0), torch.cat(p2, dim=0)
        return mean, m2

    def rhat(self):
        """Gelman-Rubin R-hat per dimension from the running moments of every chain
        (rows since construction / the last reset_moments()); needs no stored history.
        Single rank: bpm_rhat on the device; sharded: the same formula on the all-gathered
        per-chain moments."""
        torch = _torch()
        T = float(self._mom_len)
        if T < 2:
            raise RuntimeError("rhat() needs at least two rows in the running moments")
        if self.comm.size == 1:
            out = np.zeros(self.dim)
            self._flush()
            st = self._state(None)
            _lib.check(self._libh.bpm_rhat(self._handle, C.byref(st), -1, out.ctypes.data, self._stream()))
            return out
        # sharded: three all-reduced sums per dimension instead of gathering N x d moments (80 GB at config 5)
        import torch.distributed as dist
        mean, m2 = self._mean[:, :self.dim], self._m2[:, :self.dim]
        n_all = float(self.n_chains)
        # shift by a common origin (rank 0's first chain mean) so that sum(mean^2) - N gm^2 does not cancel
        origin = mean[0].clone()
        dist.broadcast(origin, src=0)
        dm = mean - origin[None]
        sums = torch.stack([dm.sum(dim=0), (dm * dm).sum(dim=0), m2.sum(dim=0)])
        dist.all_reduce(sums)
        gm = sums[0] / n_all
        B_over_T = (sums[1] - n_all * gm * gm) / (n_all - 1.0)
        W = sums[2] / (n_all * (T - 1.0))
        return torch.sqrt(((T - 1.0) / T * W + B_over_T) / W).cpu().numpy()

    def rhat_history(self, t0=None):
        """Gelman-Rubin R-hat per dimension over stored history rows [t0, T) of this rank's
        chains (default: the second half of every chain, Vrugt et al. 2009)."""
        if self._hist.policy != "full" or self._hist.stored != self._hist.length:
            raise RuntimeError("rhat_history() needs the full stored history; use rhat()")
        if t0 is None:
            t0 = self._hist.length // 2
        out = np.zeros(self.dim)
        st = self._state(self._hist.tensor().data_ptr())
        _lib.check(self._libh.bpm_rhat(self._handle, C.byref(st), int(t0), out.ctypes.data, self._stream()))
        return out

    def outlier_reset(self):
        """IQR outlier-chain reset on Omega = mean log-density since the last check
        (bpm_outlier_reset).  Returns the number of chains of this rank that were reset."""
        torch = _torch()
        cnt = C.c_int64()
        p = C.c_void_p()
        _lib.check(self._libh.bpm_omega(self._handle, C.byref(p), C.byref(cnt)))
        if not p.value or cnt.value < 1:
            raise RuntimeError("outlier_reset(): no generations tracked yet")
        n_reset = C.c_int32()
        stats = (C.c_double * 4)()
        self._flush()          # a reset overwrites X: the pending row is the pre-reset state
        st = self._state(None)
        if not self._sharded:
            _lib.check(self._libh.bpm_outlier_reset(self._handle, C.byref(st), None, None,
                                                    C.byref(n_reset), stats, self._stream()))
        else:
            import torch.distributed as dist
            lo, hi = self._local_range()
            om = self._wrap_device(p.value, (self.n_chains,)) / float(cnt.value)
            self._allgather_rows(om, lo, hi)
            self._allgather_rows(self._lnl, lo, hi)
            _lib.check(self._libh.bpm_outlier_reset(self._handle, C.byref(st), om.data_ptr(), None,
                                                    C.byref(n_reset), stats, self._stream()))
            self._allgather_population()
        self.last_outlier_stats = dict(threshold=stats[0], q1=stats[1], q3=stats[2], best=int(stats[3]))
        self.n_outlier_resets += int(n_reset.value)
        _lib.check(self._libh.bpm_omega_track(self._handle, 1))      # next window starts here
        return int(n_reset.value)

    def _allgather_rows(self, t, lo, hi):
        """In-place all-gather of a per-chain array whose rows [lo, hi) are local; shards may
        differ by one chain (np.array_split), so gather shard by shard."""
        import torch.distributed as dist
        if self.n_chains % self.comm.size == 0:
            src = t[lo:hi].reshape(-1)
            # NCCL gathers in place (the shard already sits at its slot); gloo needs a copy
            dist.all_gather_into_tensor(t.view(-1), src if t.is_cuda else src.clone())
            return
        for r, (b0, b1) in enumerate(shard_bounds(self.n_chains, self.comm.size)):
            dist.broadcast(t[b0:b1], src=r)

    def _outlier_active(self, k_gen):
        return self.outlier_gen > 0

    def moment_estimates(self):
        """Posterior mean and standard deviation pooled over every chain and every row the
        running moments cover (what param_est(0) computes from the history, without one)."""
        torch = _torch()
        T = float(self._mom_len)
        mean, m2 = self._gathered_moments()
        gm = mean.mean(dim=0)
        var = (m2.sum(dim=0) + T * ((mean - gm[None]) ** 2).sum(dim=0)) / (T * mean.shape[0])
        return gm.cpu().numpy(), torch.sqrt(var).cpu().numpy()

    def track_covariance(self, on=True):
        """Start (and zero) / stop the device-side accumulation of the population's cross moments
        (bpm_cov_track): the posterior covariance without a stored history."""
        _lib.check(self._libh.bpm_cov_track(self._handle, 1 if on else 0))

    def covariance_estimate(self):
        """(mean [d], covariance [d, d]) pooled over every chain and every generation since
        track_covariance(); sharded runs add the ranks' sums."""
        d = self.dim
        s1, s2, g = np.zeros(d), np.zeros((d, d)), C.c_int64()
        _lib.check(self._libh.bpm_cov_read(self._handle, _lib.dptr(s1), _lib.dptr(s2), C.byref(g)))
        n = float(g.value) * len(self.rank_chain_ids)
        if self.comm.size > 1:
            torch = _torch()
            import torch.distributed as dist
            t = torch.from_numpy(np.concatenate([s1, s2.ravel(), [n]])).to(self._device)
            dist.all_reduce(t)
            t = t.cpu().numpy()
            s1, s2, n = t[:d], t[d:d + d * d].reshape(d, d), float(t[-1])
        if n < 2:
            raise RuntimeError("covariance_estimate(): nothing accumulated (track_covariance() first)")
        m = s1 / n
        return m, s2 / n - np.outer(m, m)

    def _mode(self):
        if self._target is not None:
            return "device"
        if self._ln_like_batched is not None:
            return "batched"
        return "scalar"

    def _eval_lnl_rows(self, rows):
        """ln_like of a dense [n, ld] device tensor through the active plug-in."""
        torch = _torch()
        n = rows.shape[0]
        mode = self._mode()
        if mode == "device":
            out = torch.empty((n,), dtype=torch.float64, device=self._device)
            _lib.check(self._libh.bpm_eval_lnl(self._handle, rows.data_ptr(), n, out.data_ptr(),
                                               self._stream()))
            return out
        if mode == "batched":
            out = self._ln_like_batched(rows[:, :self.dim])
            return out.to(torch.float64).reshape(n).contiguous()
        host = rows[:, :self.dim].cpu().numpy()
        vals = np.array([float(self._frozen_ln_like_fn(host[i])) for i in range(n)])
        return torch.from_numpy(vals).to(self._device)

    def _init_lnl(self):
        lo, hi = self._local_range()
        self._lnl[lo:hi] = self._eval_lnl_rows(self._X[lo:hi])
        self._lnl_valid = True

    def _run_params(self, kwargs):
        flip = float(np.clip(kwargs.get("flip", 0.5), 0.0, 1.0))       # demc.py:73
        shuffle = 1 if kwargs.get("shuffle", True) else 0               # demc.py:74
        epsilon = float(kwargs.get("epsilon", 1e-15))                   # demc.py:161
        gamma = float(kwargs.get("gamma", 0.0) or 0.0)                  # demc.py:162
        return flip, shuffle, epsilon, 0.0, gamma

    # ------------------------------------------------------------------ sampling
    def run_mcmc(self, n, **kwargs):
        self._mcmc_run(n, **kwargs)

    def _n_generations(self, n):
        """Generations the reference's `while j < int((n - N) / size)` loop performs
        (demc.py:78-79, j advances by n_local per generation)."""
        limit = int((n - self.n_chains) / self.comm.size)
        n_local = len(self.rank_chain_ids)
        if limit <= 0:
            return 0
        return -(-limit // n_local)

    def _mcmc_run(self, n, **kwargs):
        if not self.am_chains:
            raise RuntimeError("ERROR: chains not initilized")
        torch = _torch()
        self.local_n_accepted = 0
        self.local_n_rejected = 1
        _lib.check(self._libh.bpm_reset_counters(self._handle))
        _lib.check(self._libh.bpm_set_run_params(self._handle, *self._run_params(kwargs)))
        if not self._lnl_valid:
            self._init_lnl()
        G = self._n_generations(n)
        replay = kwargs.get("_replay", None)
        trace = kwargs.get("_trace", None)
        if replay is not None:
            G = min(G, len(replay))
        k_gen = 0
        k_off = int(kwargs.get("_k_gen0", 0))     # testing hook: start the schedule at k_off
        track_outliers = self.outlier_gen > 0 and replay is None
        _lib.check(self._libh.bpm_omega_track(self._handle, 1 if track_outliers else 0))
        mode = self._mode()
        while k_gen < G:
            if self._pending and self._hist.will_grow():
                self._flush()      # the pending row belongs to the chunk that is full now
            if replay is not None:
                base, avail = self._hist.reserve_contiguous(G - k_gen)
            else:
                base, avail = self._hist.reserve(G - k_gen)
            avail = min(avail, G - k_gen)
            if self.checkpoint > 0:
                avail = min(avail, self.checkpoint - (k_gen % self.checkpoint))
            if track_outliers:
                avail = min(avail, self.outlier_gen - (k_gen % self.outlier_gen))
            st = self._state(base)
            if replay is not None:
                self._replay_generation(st, replay[k_gen], k_gen + k_off, trace)
                done = 1
            elif mode == "device" and (not self._sharded or (self._sync_on and self._n_phases == 2)):
                # whole generations inside the library; sharded: barriers / CR exchange over peer memory
                done = avail
                if self._subpop:
                    done = min(done, self.subpop_k - (self._gens_since_deal % self.subpop_k))
                _lib.check(self._libh.bpm_step_generations(self._handle, C.byref(st), k_gen + k_off, done,
                                                           self._stream()))
            else:
                self._split_generation(st, k_gen + k_off)
                done = 1
            self._pending = int(st.pending)
            self._hist.advance(done)
            self._mom_len += done
            k_gen += done
            if self._subpop:
                self._gens_since_deal += done
                if self._gens_since_deal % self.subpop_k == 0:
                    self._redeal()
            if track_outliers and k_gen % self.outlier_gen == 0 and self._outlier_active(k_gen + k_off):
                self.outlier_reset()
            if self.checkpoint > 0 and k_gen % self.checkpoint == 0:        # demc.py:138-140
                self.save_state(self.h5_file)
        torch.cuda.synchronize(self._device)
        if self._sync_on:
            err = C.c_int32()
            _lib.check(self._libh.bpm_sync_error(self._handle, C.byref(err)))
            if err.value:
                raise RuntimeError("peer barrier timed out: a rank did not arrive (bpm_sync_error)")
        self._collect_counters()
        self.comm.Barrier()

    def _collect_counters(self):
        """demc.py:143-150 (and the reference's `local_n_rejected = 1` start)."""
        acc, rej, nan = C.c_uint64(), C.c_uint64(), C.c_int32()
        _lib.check(self._libh.bpm_get_counters(self._handle, C.byref(acc), C.byref(rej), C.byref(nan)))
        if nan.value:
            raise ValueError("probabilities contain NaN")       # numpy's message at samplers.py:336
        self.local_n_accepted = int(acc.value)
        self.local_n_rejected = 1 + int(rej.value)
        if self.comm.size > 1:
            torch = _torch()
            import torch.distributed as dist
            t = torch.tensor([self.local_n_accepted, self.local_n_rejected], dtype=torch.int64,
                             device=self._device)
            dist.all_reduce(t)
            self.n_accepted, self.n_rejected = int(t[0].item()), int(t[1].item())
        else:
            self.n_accepted, self.n_rejected = self.local_n_accepted, self.local_n_rejected

    # -- one generation through the split API (user likelihoods, multi-rank) ---------
    def _split_generation(self, st, k_gen, rp=None):
        torch = _torch()
        s = self._stream()
        lib, h = self._libh, self._handle
        _lib.check(lib.bpm_begin_generation(h, C.byref(st), k_gen, rp, s))
        for phase in range(self._n_phases):
            last = phase == self._n_phases - 1
            if self._mode() == "device":
                # built-in likelihood: the whole half-phase stays inside the library
                _lib.check(lib.bpm_phase(h, C.byref(st), phase, s))
                self._phase_exchange(last=last)
                continue
            prop_p, n_p = C.c_void_p(), C.c_int32()
            _lib.check(lib.bpm_propose(h, C.byref(st), phase, C.byref(prop_p), C.byref(n_p), s))
            n = n_p.value
            rows = self._wrap_rows(prop_p.value, n)
            lnl_prop = self._eval_lnl_rows(rows)
            if self.comm.size > 1:
                # rows of chains owned by other ranks were not proposed here; their
                # likelihood values are ignored by bpm_accept (ownership check in-kernel)
                pass
            _lib.check(lib.bpm_accept(h, C.byref(st), phase, lnl_prop.data_ptr(), None, s))
            self._phase_exchange(last=last)
        _lib.check(lib.bpm_end_generation(h, C.byref(st), s))
        if self._sharded and self._algo == _lib.BPM_ALGO_DREAM:
            self._allreduce_cr()

    def _wrap_device(self, ptr, shape):
        """torch view of library-owned device memory (no copy)."""
        torch = _torch()

        class _Iface(object):
            pass
        o = _Iface()
        o.__cuda_array_interface__ = dict(shape=tuple(shape), typestr="<f8", data=(int(ptr), False),
                                          version=2, strides=None)
        return torch.as_tensor(o, device=self._device)

    def _wrap_rows(self, ptr, n):
        return self._wrap_device(ptr, (n, self._ld))

    def _allgather_population(self):
        """comm.Allgather(current_chain_state) of demc.py:93,116 on the device replica."""
        lo, hi = self._local_range()
        self._allgather_rows(self._X, lo, hi)

    def _redeal(self):
        """Sub-population mode: re-deal the chains across the ranks.  Every rank cuts its chains
        into G contiguous groups and sends group j to rank j (one all-to-all of states, cached
        likelihoods and running moments), so afterwards every island holds 1/G of every island.
        History rows stay with the slot, not with the travelling chain."""
        torch = _torch()
        import torch.distributed as dist
        G, nl = self.comm.size, len(self.rank_chain_ids)
        self._flush()          # moments travel with the chains: fold the pending sample first
        import time as _time
        torch.cuda.synchronize(self._device)
        _t0 = _time.perf_counter()
        cuts = [b1 - b0 for b0, b1 in shard_bounds(nl, G)]
        if len(set(len(np.array_split(np.arange(self.n_chains), G)[r]) for r in range(G))) != 1:
            raise RuntimeError("subpop_k needs n_chains divisible by the number of ranks")
        if getattr(self, "_ipc_ok", False) and nl % G == 0 and all(k in self._ipc for k in ("X", "lnl", "mean", "m2")):
            # pull: chunk i of my new arrays = block `rank` of island i's arrays, copied over NVLink by the copy
            # engines (cudaMemcpyAsync on IPC-mapped peer memory).  Two barriers: everyone has stopped stepping
            # before anyone reads, everyone has finished reading before anyone overwrites.
            lib, cut, r = self._libh, nl // G, self.comm.rank
            dist.barrier()
            outs = []
            for name, t in (("X", self._X), ("mean", self._mean_t), ("m2", self._m2_t), ("lnl", self._lnl)):
                out = torch.empty_like(t)
                row_bytes = (t.shape[1] if t.dim() == 2 else 1) * 8
                own, peers = self._ipc[name]
                for i in range(G):
                    src = (own if i == r else peers[i]) + r * cut * row_bytes
                    _lib.check(lib.bpm_peer_copy(self._device_index, C.c_void_p(out.data_ptr() + i * cut * row_bytes),
                                                 C.c_void_p(src), cut * row_bytes, self._stream()))
                outs.append((t, out))
            torch.cuda.synchronize(self._device)
            dist.barrier()
            for t, out in outs:
                t.copy_(out)
            del outs
            torch.cuda.synchronize(self._device)
            self.redeal_seconds = getattr(self, "redeal_seconds", 0.0) + (_time.perf_counter() - _t0)
            self.n_redeals = getattr(self, "n_redeals", 0) + 1
            return
        for t in (self._X, self._mean, self._m2):
            out = torch.empty_like(t)
            dist.all_to_all_single(out, t.contiguous(), output_split_sizes=cuts, input_split_sizes=cuts)
            t.copy_(out)
        out = torch.empty_like(self._lnl)
        dist.all_to_all_single(out, self._lnl, output_split_sizes=cuts, input_split_sizes=cuts)
        self._lnl.copy_(out)
        torch.cuda.synchronize(self._device)
        self.redeal_seconds = getattr(self, "redeal_seconds", 0.0) + (_time.perf_counter() - _t0)
        self.n_redeals = getattr(self, "n_redeals", 0) + 1

    def _allreduce_cr(self):
        torch = _torch()
        import torch.distributed as dist
        p = C.c_void_p()
        _lib.check(self._libh.bpm_cr_partials(self._handle, C.byref(p)))
        t = self._wrap_device(p.value, (2 * self.n_cr,))
        dist.all_reduce(t)
        _lib.check(self._libh.bpm_apply_cr(self._handle, self._stream()))

    # -- RNG replay (testing hook: `_replay=[trace, ...]` from oracle/demc_dream.py) ---
    def _replay_generation(self, st, tr, k_gen, trace_sink):
        torch = _torch()
        dev = self._device
        keep = []

        def dev_arr(a, dt):
            t = torch.from_numpy(np.ascontiguousarray(np.asarray(a, dtype=dt))).to(dev)
            keep.append(t)
            return t.data_ptr()
        rp = _lib.Replay()
        rp.flip = 1 if tr["flip"] else 0
        rp.shuffle_idx = dev_arr(tr["shuffle_idx"], np.int32)
        rp.pairs = dev_arr(tr["pairs"], np.int32)
        rp.gamma_u = dev_arr(np.nan_to_num(tr["gamma_u"], nan=2.0), np.float64)
        nrm = np.asarray(tr["nrm"], dtype=np.float64)
        rp.nrm = dev_arr(nrm, np.float64)
        rp.accept_u = dev_arr(tr["accept_u"], np.float64)
        if self._algo == _lib.BPM_ALGO_DREAM:
            rp.cr_idx = dev_arr(tr["cr_idx"], np.int32)
            rp.z = dev_arr(tr["z"], np.float64)
            rp.fallback_dim = dev_arr(tr["fallback_dim"], np.int32)
            rp.e = dev_arr(tr["e"], np.float64)
        tro = None
        if trace_sink is not None:
            N, d = self.n_chains, self.dim
            acc = torch.zeros((N,), dtype=torch.int32, device=dev)
            lp = torch.zeros((N,), dtype=torch.float64, device=dev)
            pr = torch.zeros((N, d), dtype=torch.float64, device=dev)
            tro = _lib.TraceOut(acc.data_ptr(), lp.data_ptr(), pr.data_ptr())
        if self._mode() == "device":
            _lib.check(self._libh.bpm_step_generation_replay(
                self._handle, C.byref(st), C.byref(rp), k_gen,
                C.byref(tro) if tro is not None else None, self._stream()))
        else:
            self._split_generation(st, k_gen, rp=C.byref(rp))
        torch.cuda.synchronize(dev)
        if trace_sink is not None:
            trace_sink.append(dict(accept=acc.cpu().numpy(), lnl_prop=lp.cpu().numpy(),
                                   prop=pr.cpu().numpy(), state=self._X[:, :self.dim].cpu().numpy()))

    def _dump_native_draws(self, k_gen):
        """Testing / provenance hook: the draws the native Philox stream WILL use for the
        next generation (absolute index = current chain length), as a trace dict with the
        keys oracle/replay.py consumes."""
        torch = _torch()
        dev, N, d = self._device, self.n_chains, self.dim
        npair = self._dream_cfg()["del_pairs"] if self._algo == _lib.BPM_ALGO_DREAM else 1
        i32 = lambda *s: torch.zeros(s, dtype=torch.int32, device=dev)      # noqa: E731
        f64 = lambda *s: torch.zeros(s, dtype=torch.float64, device=dev)    # noqa: E731
        t = dict(shuffle_idx=i32(N), cr_idx=i32(N), z=f64(N, d), fallback_dim=i32(N),
                 pairs=i32(N, npair, 2), gamma_u=f64(N), e=f64(N, d), nrm=f64(N, d), accept_u=f64(N))
        rp = _lib.Replay()
        for k, v in t.items():
            setattr(rp, k, v.data_ptr())
        flip = C.c_int32()
        st = self._state(None)
        _lib.check(self._libh.bpm_dump_draws(self._handle, C.byref(st), k_gen, C.byref(rp),
                                             C.byref(flip), self._stream()))
        torch.cuda.synchronize(dev)
        out = dict((k, v.cpu().numpy()) for k, v in t.items())
        out["flip"] = bool(flip.value)
        return out

    # ------------------------------------------------------------------ results
    @property
    def chain(self):
        return self.am_chains[0]

    @property
    def current_pos(self):
        return self.chain.current_pos

    @property
    def acceptance_fraction(self):
        """samplers.py:76-80."""
        return self.n_accepted / (self.n_accepted + self.n_rejected)

    def param_est(self, n_burn, collection_rank=0):
        """demc.py:235-248: mean / std over super-chain rows [n_burn:]."""
        self.comm.Barrier()
        chain_slice = self.super_chain_mpi(collection_rank)
        if self.comm.rank == collection_rank:
            chain_slice = chain_slice[n_burn:, :]
            return np.mean(chain_slice, axis=0), np.std(chain_slice, axis=0), chain_slice
        return None, None, None

    def param_est_device(self, n_burn):
        """Same estimate computed on the GPU without moving the history to the host;
        returns (mean, std) as numpy arrays of length dim (rank-local chains when sharded)."""
        h = self._hist.tensor()
        flat = h[:, :, :self.dim].reshape(-1, self.dim)[n_burn:]
        return flat.mean(dim=0).cpu().numpy(), flat.std(dim=0, unbiased=False).cpu().numpy()

    def super_chain_mpi(self, collection_rank=0):
        return self._super_chain(collection_rank)

    @property
    def super_chain(self):
        return self._super_chain()

    def _super_chain(self, collection_rank=0):
        """demc.py:260-270: row t*N + i = chain i at time t."""
        torch = _torch()
        h = self._hist.tensor()[:, :, :self.dim]
        if self.comm.size == 1:
            return h.reshape(-1, self.dim).cpu().numpy()
        import torch.distributed as dist
        parts = [torch.empty_like(h) for _ in range(self.comm.size)]
        dist.all_gather(parts, h.contiguous())
        if self.comm.rank != collection_rank:
            return None
        full = torch.cat(parts, dim=1)
        return full.reshape(-1, self.dim).cpu().numpy()

    def gather_all_chains(self, collection_rank=0):
        return list(self.iter_all_chains(collection_rank))

    def iter_local_chains(self):
        for chain in self.am_chains:
            yield chain

    def iter_all_chains(self, collection_rank=0, verbose=0):
        if verbose:
            print("Iter all chains on rank: ", self.comm.rank)
        sys.stdout.flush()
        for c_id in range(self.n_chains):
            yield self.get_chain(c_id, collection_rank)

    def get_chain(self, c_id, collection_rank=0, verbose=0):
        """demc.py:296-325.  Single rank: the local view.  Multi rank: a free-standing
        host McmcChain on the collection rank, None elsewhere."""
        assert 0 <= c_id < self.n_chains
        if self.comm.size == 1:
            return self.am_chains[c_id]
        sc = self._super_chain(collection_rank)
        if self.comm.rank != collection_rank:
            return None
        ch = McmcChain(np.zeros(self.dim), varepsilon=0.0, global_id=int(c_id))
        ch.chain = sc[c_id::self.n_chains, :]
        return ch

    def get_chain_rank(self, c_id):
        assert 0 <= c_id < self.n_chains
        for r, (b0, b1) in enumerate(shard_bounds(self.n_chains, self.comm.size)):
            if b0 <= c_id < b1:
                return r
        raise RuntimeError("ERROR: c_id not in global chain ids")

    # ------------------------------------------------------------------ checkpoint
    def save_state(self, h5_file=""):
        """demc.py:198-215: one gzip dataset /chains/chain_id_<id> of shape (T, dim) per chain.
        Extension: the sampler state the reference loses on resume -- Philox seed, CR
        adaptation state -- is stored next to the chains (HDF5 attributes of /chains).
        Written through h5py where it imports and through bipymc_b200.h5lite (pure Python, same on-disk
        format) where it does not.  For a name ending in ".npz" the same content goes to a numpy archive."""
        if not h5_file:
            h5_file = self.h5_file
        sc = self._super_chain(0)
        extra = self._checkpoint_extra()
        if self.comm.rank == 0:
            h5py = None if h5_file.endswith(".npz") else _try_h5py()
            if h5py is not None:
                with h5py.File(h5_file, "w") as h5f:
                    for c_id in range(self.n_chains):
                        h5f.create_dataset("/chains/chain_id_" + str(c_id), data=sc[c_id::self.n_chains, :],
                                           compression="gzip")
                    for k, v in extra.items():
                        h5f["/chains"].attrs[k] = v
            else:
                T = sc.shape[0] // self.n_chains
                np.savez_compressed(_npz_name(h5_file), history=sc.reshape(T, self.n_chains, self.dim), **extra)
        self.comm.Barrier()

    def _checkpoint_extra(self):
        return dict(b200_seed=np.uint64(self._seed))

    def _restore_extra(self, extra):
        if "b200_seed" in extra:
            self._seed = int(extra["b200_seed"])

    def load_state(self, h5_file=""):
        """demc.py:217-233."""
        if not h5_file:
            h5_file = self.h5_file
        h5py = None if h5_file.endswith(".npz") else _try_h5py()
        if h5py is not None:
            with h5py.File(h5_file, "r") as h5f:
                names = set(h5f["/chains"].keys())
                if names != set("chain_id_" + str(int(c)) for c in range(self.n_chains)):
                    raise RuntimeError        # another population's file (the .npz branch below rejects it too)
                chains = [h5f["/chains/chain_id_" + str(int(c))][:] for c in range(self.n_chains)]
                extra = dict((k, np.asarray(v)) for k, v in h5f["/chains"].attrs.items())
            k_gen = len(chains[0])
            for ch in chains:
                if len(ch) != k_gen:
                    raise RuntimeError
            hist = np.stack(chains, axis=1)
        else:
            with np.load(_npz_name(h5_file)) as z:
                hist = z["history"]
                extra = dict((k, z[k]) for k in z.files if k != "history")
            if hist.shape[1] != self.n_chains:
                raise RuntimeError
        seed_before = self._seed
        self._restore_extra(extra)
        if self._seed != seed_before:
            # the Philox key is part of the engine configuration: rebuild the handle
            self._release_peer_memory()
            self._libh.bpm_destroy(self._handle)
            self._handle = None
            self._create_handle()
        self.load_history(hist)
        self._restore_extra_late(extra)
        self.comm.Barrier()

    def _restore_extra_late(self, extra):
        pass

    def load_history(self, hist):
        """hist: (T, N, dim) array of every chain's history (what load_state reads)."""
        hist = np.asarray(hist, dtype=float)
        assert hist.shape[1] == self.n_chains and hist.shape[2] == self.dim
        if self._subpop:      # an island's rows inside the job-wide history are its GLOBAL chain ids
            lo, hi = int(self.rank_chain_ids[0]), int(self.rank_chain_ids[-1]) + 1
        else:
            lo, hi = self._local_range()
        self._set_population(hist[-1], history=hist[:, lo:hi, :])
