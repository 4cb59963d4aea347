"""Times the UNMODIFIED reference (wgurecky/bipymc, installed by __graft_entry__.build() into
oracle/_ref with `pip install --target`) on the host cores: the `kind: "reference"` CPU baseline of
bench.py (BASELINE.md section 5 items 1-2).

TEST / BENCH INFRASTRUCTURE ONLY.  The reference imports mpi4py / h5py / matplotlib / corner at module
scope and none is installed, so oracle/shims/ goes on sys.path first; its MPI.ShmComm stands in for
mpirun: P forked ranks, each constructing DreamMpi(..., mpi_comm=ShmComm) exactly as
`mpirun -np P python examples/ex_para_fit.py` would, Allgather / Barrier over shared memory.  Nothing of
the reference is modified or copied; every rank seeds numpy identically, as the reference's own tests do
(tests/test_banana.py:17).
"""
import multiprocessing as mp
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF_DIRS = [os.path.join(ROOT, "oracle", "_ref")]


def reference_dir():
    for d in REF_DIRS:
        if os.path.exists(os.path.join(d, "bipymc", "dream.py")):
            return d
    return None


def _import_reference():
    d = reference_dir()
    if d is None:
        raise ImportError("unmodified reference not found (oracle/_ref is written by __graft_entry__.build())")
    shims = os.path.join(HERE, "shims")
    for p in (d, shims):
        if p in sys.path:
            sys.path.remove(p)
    sys.path.insert(0, d)
    sys.path.insert(0, shims)
    import warnings
    warnings.simplefilter("ignore")
    from mpi4py import MPI
    from bipymc.dream import DreamMpi
    from bipymc.demc import DeMcMpi
    from bipymc.utils import d100_gauss
    return MPI, DreamMpi, DeMcMpi, d100_gauss


def _worker(rank, size, shared, barrier, spec, gens_warm, gens, out_q):
    try:
        # one BLAS thread per rank, as `mpirun -np P` on P cores would run it (the reference's var_ball
        # calls a 100 x 100 SVD per step, util.py:13; P ranks x P BLAS threads would thrash)
        try:
            from threadpoolctl import threadpool_limits
            threadpool_limits(1)
        except Exception:
            pass
        MPI, DreamMpi, DeMcMpi, d100_gauss = _import_reference()
        comm = MPI.ShmComm(rank, size, shared, barrier)
        N, d = spec["n_chains"], spec["dim"]
        tgt = d100_gauss.Gauss_100D(dim=d)
        np.random.seed(spec["seed"])
        cls = DreamMpi if spec["algo"] == "dream" else DeMcMpi
        s = cls(tgt.ln_like, np.zeros(d), n_chains=N, mpi_comm=comm, varepsilon=spec.get("varepsilon", 1e-6),
                **spec["ctor_kwargs"])
        devnull = open(os.devnull, "w")
        sys.stdout = devnull
        # run_mcmc(n): generations = ceil(((n - N) / size) / n_local)   (demc.py:79)
        if gens_warm > 0:
            s.run_mcmc(N * (gens_warm + 1))
        barrier.wait()
        t0 = time.perf_counter()
        s.run_mcmc(N * (gens + 1))
        barrier.wait()
        dt = time.perf_counter() - t0
        sys.stdout = sys.__stdout__
        steps = sum(len(c.chain) for c in s.am_chains) - len(s.am_chains) * (1 + gens_warm)
        out_q.put((rank, dt, int(steps), None))
    except Exception as e:      # pragma: no cover
        import traceback
        out_q.put((rank, 0.0, 0, traceback.format_exc()))
        try:
            barrier.abort()
        except Exception:
            pass


def time_reference(spec, procs, gens, gens_warm=1):
    """`gens` timed generations of the unmodified reference on `procs` processes.
    Returns (seconds, chain_steps) -- chain_steps counted from the chains the reference actually grew."""
    ctx = mp.get_context("fork")
    N, d = spec["n_chains"], spec["dim"]
    assert N % procs == 0, "the reference needs n_chains divisible by the number of ranks"
    shared = ctx.RawArray("d", max(N * d, 4 * procs))
    barrier = ctx.Barrier(procs)
    q = ctx.Queue()
    ps = [ctx.Process(target=_worker, args=(r, procs, shared, barrier, spec, gens_warm, gens, q))
          for r in range(procs)]
    for p in ps:
        p.start()
    res = [q.get() for _ in ps]
    for p in ps:
        p.join()
    bad = [r[3] for r in res if r[3]]
    if bad:
        raise RuntimeError("reference rank failed:\n" + bad[0])
    return max(r[1] for r in res), sum(r[2] for r in res)


if __name__ == "__main__":
    P = int(sys.argv[1]) if len(sys.argv) > 1 else 2
    spec = dict(n_chains=40 * P, dim=100, algo="dream", seed=42, ctor_kwargs=dict(n_cr_gen=50, burnin_gen=2000))
    dt, steps = time_reference(spec, P, gens=int(sys.argv[2]) if len(sys.argv) > 2 else 20, gens_warm=1)
    print("reference: %d ranks, %d chain-steps in %.2f s = %.0f chain-steps/s" % (P, steps, dt, steps / dt))
