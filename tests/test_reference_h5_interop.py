"""Checkpoint files travel between the UNMODIFIED reference and bipymc_b200 (chain.py:59-93, demc.py:198-233).

The reference runs from oracle/_ref (pip-installed by __graft_entry__.build() where its source is present) with
oracle/shims on the path: a single-rank mpi4py, and an `h5py` that is the package's HDF5 implementation
(bipymc_b200/h5lite.py) -- so the reference's own write_chain_h5 / read_chain_h5 / save_state / load_state code
executes, calling exactly the h5py API it was written against.  What this pins: the API slice h5lite offers is the
one the reference uses, and the dataset names / shapes / dtypes / compression each side writes are the ones the
other side reads.  (Byte compatibility with libhdf5 is pinned separately: tests/test_h5lite_cpu.py.)"""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "oracle", "_ref")
SHIMS = os.path.join(ROOT, "oracle", "shims")

pytestmark = pytest.mark.skipif(not os.path.exists(os.path.join(REF, "bipymc", "chain.py")),
                                reason="oracle/_ref (the pip-installed reference) is not present")


@pytest.fixture(scope="module")
def ref():
    """The reference package, imported with the shims in front of it."""
    import warnings
    warnings.simplefilter("ignore")
    saved = list(sys.path)
    for p in (REF, SHIMS):
        if p in sys.path:
            sys.path.remove(p)
    sys.path.insert(0, REF)
    sys.path.insert(0, SHIMS)
    try:
        import bipymc.chain as ref_chain
        import bipymc.dream as ref_dream
        import bipymc.demc as ref_demc
        from bipymc.utils import banana_rv
    finally:
        sys.path[:] = saved
    assert not hasattr(ref_chain.h5py, "version")          # the shim, not a real h5py
    return dict(chain=ref_chain, dream=ref_dream, demc=ref_demc, banana=banana_rv)


def _ref_chain(ref, gid, rows, dim=3):
    np.random.seed(100 + gid)
    c = ref["chain"].McmcChain(np.zeros(dim), varepsilon=1e-2, global_id=gid)
    for _ in range(rows):
        c.append_sample(np.random.randn(dim))
    return c


def test_reference_chain_file_is_read_by_bipymc_b200_and_back(ref, tmp_path, monkeypatch):
    from bipymc_b200 import h5lite
    from bipymc_b200.chain import McmcChain
    monkeypatch.setenv("BIPYMC_B200_H5LITE", "1")
    f = str(tmp_path / "ref_one.h5")
    rc = _ref_chain(ref, 7, 5)
    rc.write_chain_h5(f)                                     # the reference's code, str branch (chain.py:64-71)
    with h5lite.File(f, "r") as h:
        ds = h["/chains/chain_id_7"]
        assert ds.shape == (6, 3) and ds.dtype == np.float64 and ds.compression == "gzip"
    mine = McmcChain(np.zeros(3), varepsilon=0.0, global_id=7)
    mine.read_chain_h5(f)
    assert np.array_equal(mine.chain, rc.chain)
    # the other way: bipymc_b200 writes, the reference reads (chain.py:86-91)
    g = str(tmp_path / "mine_one.h5")
    mine.append_sample(np.arange(3.0))
    mine.write_chain_h5(g)
    back = ref["chain"].McmcChain(np.zeros(3), varepsilon=0.0, global_id=7)
    back.read_chain_h5(g)
    assert np.array_equal(back.chain, mine.chain)


def test_open_file_branch_and_rewrite(ref, tmp_path):
    """chain.py:72-79 / 88-89: an open h5py.File object is accepted (isinstance), an existing dataset is deleted
    and rewritten."""
    h5 = ref["chain"].h5py
    f = str(tmp_path / "ref_many.h5")
    chains = [_ref_chain(ref, i, 3 + i % 2, dim=2) for i in range(12)]
    with h5.File(f, "w") as h:
        for c in chains:
            c.write_chain_h5(h)
        chains[4].append_sample(np.ones(2))
        chains[4].write_chain_h5(h)                          # del + create_dataset
    with h5.File(f, "r") as h:
        for c in chains:
            d = ref["chain"].McmcChain(np.zeros(2), varepsilon=0.0, global_id=c.global_id)
            d.read_chain_h5(h)
            assert np.array_equal(d.chain, c.chain)
    with pytest.raises(RuntimeError):
        chains[0].write_chain_h5(3.14)


def _ref_sampler(ref, n_chains=12, steps=9, **kw):
    np.random.seed(5)
    t = ref["banana"].Banana_2D()
    s = ref["dream"].DreamMpi(t.ln_like, np.array([0.0, 0.0]), n_chains=n_chains, varepsilon=1e-2, n_cr_gen=2,
                              burnin_gen=10, **kw)
    if steps:
        s.run_mcmc(n_chains * steps)
    return s


def test_reference_sampler_checkpoint_layout_and_its_own_reload(ref, tmp_path):
    """DeMcMpi.save_state / load_state of the reference (demc.py:198-233), unmodified, on the h5lite-backed shim."""
    from bipymc_b200 import h5lite
    s = _ref_sampler(ref)
    f = str(tmp_path / "ref_ckpt.h5")
    s.save_state(f)
    T = len(s.am_chains[0].chain)
    with h5lite.File(f, "r") as h:
        assert h["/chains"].keys() == sorted("chain_id_%d" % i for i in range(12))
        for i in range(12):
            ds = h["/chains/chain_id_%d" % i]
            assert ds.shape == (T, 2) and ds.compression == "gzip"
            assert np.array_equal(ds[:], s.am_chains[i].chain)
    r = _ref_sampler(ref, steps=0, warm_start=True, h5_file=f, dim=2)       # demc.py:46-51
    for a, b in zip(r.am_chains, s.am_chains):
        assert np.array_equal(a.chain, b.chain)


@pytest.mark.gpu
def test_bipymc_b200_warm_starts_from_a_reference_checkpoint_and_the_reference_from_ours(ref, tmp_path):
    from bipymc_b200 import DreamMpi, targets
    s = _ref_sampler(ref)
    f = str(tmp_path / "ref_ckpt.h5")
    s.save_state(f)
    T = len(s.am_chains[0].chain)
    np.random.seed(1)
    mine = DreamMpi(targets.Banana_2D().ln_like, [0.0, 0.0], n_chains=12, seed=3, warm_start=True, h5_file=f, dim=2,
                    n_cr_gen=2, burnin_gen=10)
    for i in range(12):
        assert mine.am_chains[i].chain_len == T
        np.testing.assert_array_equal(mine.am_chains[i].chain, s.am_chains[i].chain)
    mine.run_mcmc(12 * 4, _k_gen0=T - 1)                     # and it continues from there: 4 * N samples = 3 generations
    assert mine.am_chains[0].chain_len == T + 3
    g = str(tmp_path / "mine_ckpt.h5")
    mine.save_state(g)
    r = _ref_sampler(ref, steps=0, warm_start=True, h5_file=g, dim=2)
    for i in range(12):
        np.testing.assert_array_equal(r.am_chains[i].chain, mine.am_chains[i].chain)
