#!/usr/bin/env python
"""Headline benchmark: DREAM chain-steps/s on the 100-D correlated Gaussian.

  python bench.py --gpus N --steps K --warmup W            (this framework, N GPUs)
  python bench.py --impl reference --gpus N --steps K --warmup W   (CPU port of the reference)

A "step" is one DREAM generation of the whole population (every chain proposes, evaluates
its likelihood and is accepted / rejected once).  Workload = BASELINE.json configs[1]:
DREAM (del_pairs=3, n_cr=3, n_cr_gen=50, burnin_gen=2000) on Gauss_100D(rho=0.5) with 10^5
chains per GPU (weak scaling), Philox seed 42, chains started over-dispersed
(N(0, diag Sigma)) and advanced 60 untimed generations first so the timed region is the
burn-in steady state with crossover adaptation, running moments and full history ON.
Prints ONE JSON line (rank 0).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

N_PER_GPU = 100000
DIM = 100
SETUP_GENS = 60
DUMP_ROWS = 8192        # chains whose rows --dump-outputs writes: all 10^5 would be 80 MB per generation
DUMP_GENS = 4           # ... and how many of the last timed generations of their history (64 MB cap in all)
METRIC = "DREAM chain-steps/s, 100-D Gaussian"
UNIT = "chain-steps/s"


def csrc_hash():
    """sha256 (first 16 hex digits) over the CUDA sources the library is built from: ties a committed ncu
    capture to the kernels that were actually timed."""
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(ROOT, "bipymc_b200", "csrc")
    for f in sorted(os.listdir(d)):
        if f.endswith((".cu", ".cuh")):
            h.update(f.encode())
            h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


def ncu_traffic(history, adapt):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of the dominant kernel, from the committed
    ncu --set full capture of this same workload (profiles/traffic.json, written by tools/ncu_summary.py
    traffic).  The file records the hash of csrc/ it was captured with; any other build gets None -- a stale
    capture must not pass for a measurement of the kernel that was timed."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(p):
        return None
    j = json.load(open(p))
    if j.get("csrc_sha16") != csrc_hash():
        return None
    return j.get("history=%s,adapt=%s" % (history, "on" if adapt else "off"))


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return float(j["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def cpu_port_spec(n_chains):
    return dict(target="gauss100", theta_0=list(np.zeros(DIM)), n_chains=n_chains, algo="dream",
                seed=42, varepsilon=1e-6, ctor_kwargs=dict(n_cr_gen=50, burnin_gen=2000))


def cpu_arm(n_chains, procs, gens, gens_warm):
    """Time the reference's DREAM on `procs` host processes: the UNMODIFIED reference from oracle/_ref
    (oracle/ref_runner.py: shared-memory stand-in for mpirun) when it is installed there, else the
    oracle port (oracle/mp_port.py).  Returns (seconds, chain_steps, kind)."""
    from oracle import ref_runner
    if ref_runner.reference_dir() is not None:
        spec = dict(n_chains=n_chains, dim=DIM, algo="dream", seed=42, varepsilon=1e-6,
                    ctor_kwargs=dict(n_cr_gen=50, burnin_gen=2000))
        dt, steps = ref_runner.time_reference(spec, procs, gens=gens, gens_warm=gens_warm)
        return dt, steps, "reference"
    from oracle.mp_port import time_port
    dt, steps = time_port(cpu_port_spec(n_chains), procs, gens=gens, gens_warm=gens_warm)
    return dt, steps, "port"


def run_reference(args):
    """The reference's own CPU implementation of the path on the host cores: wgurecky/bipymc DreamMpi,
    unmodified (oracle/_ref), one rank per core over a shared-memory communicator."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    procs = max(1, min(cores, 64))
    n_chains = 200 * procs
    # a step = one generation of the sample population; warm-up generations are untimed
    dt, steps, kind = cpu_arm(n_chains, procs, gens=args.steps, gens_warm=max(args.warmup, 1))
    v = steps / dt
    what = "unmodified reference DreamMpi (oracle/_ref)" if kind == "reference" else "oracle port of DreamMpi"
    sample = "%s, %d ranks, 100-D Gaussian, %d chains (200 per rank), %d timed generations, %.1f s" % (
        what, procs, n_chains, args.steps, dt)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "gpu_launches": 0,
            "config": {"workload": "configs[1]: DREAM, Gauss_100D(rho=0.5), CPU sample of %d chains" % n_chains,
                       "del_pairs": 3, "n_cr": 3, "n_cr_gen": 50, "burnin_gen": 2000},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": procs, "kind": kind, "sample": sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def cpu_baseline_leg():
    cores = os.cpu_count() or 1
    procs = max(1, min(cores, 64))
    n_chains = 40 * procs
    gens = 400            # ~10-20 s of host work: np.std over the growing history is O(T) per step (dream.py:128)
    dt, steps, kind = cpu_arm(n_chains, procs, gens=gens, gens_warm=2)
    what = "unmodified reference DreamMpi (oracle/_ref), shared-memory ranks" if kind == "reference" else \
        "oracle port of DreamMpi (shared-memory ranks)"
    out = {"value": steps / dt, "unit": UNIT, "cores": procs, "kind": kind,
           "sample": "%s, 100-D Gaussian, %d chains, %d generations, %.1f s" % (what, n_chains, gens, dt)}
    if kind == "reference":
        # BASELINE.md section 5 item 1: the same reference on ONE core (its bit-reproducible configuration)
        dt1, steps1, _ = cpu_arm(40, 1, gens=100, gens_warm=2)
        out["one_core"] = {"value": steps1 / dt1, "unit": UNIT, "cores": 1,
                           "sample": "40 chains, 100 generations, %.1f s" % dt1}
    return out


def bind_to_gpu_numa(local_rank):
    """Best effort: run this rank (and first-touch its pinned host buffers) on the NUMA node its GPU hangs
    off, so eight ranks' host copies do not all cross one socket link.  Returns the node or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        hnd = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        bus = pynvml.nvmlDeviceGetPciInfo(hnd).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


def selfcheck_sharded(world, rank, local_rank):
    """N > 1 only (the driver's scaling run has no other multi-GPU correctness test): a small sharded DREAM
    run through the same entry points as the timed one must reproduce, bit for bit, rank 0's single-GPU
    run of the same seed (every draw is a function of (seed, generation, chain), never of the rank;
    adaptation off so no cross-rank sum rounds differently)."""
    from bipymc_b200 import DreamMpi, targets
    from bipymc_b200.demc import _SingleComm
    N, G = 1024 * world, 4
    tgt = targets.Gauss_100D(rho=0.5, dim=DIM)
    np.random.seed(7)
    s = DreamMpi(tgt.ln_like, np.zeros(DIM), n_chains=N, varepsilon=1.0, seed=11, burnin_gen=0, device=local_rank)
    s.run_mcmc(N * (G + 1))
    full = s.super_chain_mpi(0)
    acc = s.n_accepted
    out = None
    if rank == 0:
        np.random.seed(7)
        one = DreamMpi(tgt.ln_like, np.zeros(DIM), n_chains=N, varepsilon=1.0, seed=11, burnin_gen=0,
                       device=local_rank, mpi_comm=_SingleComm())
        one.run_mcmc(N * (G + 1))
        ref = one.super_chain
        same = bool(full.shape == ref.shape and np.array_equal(full, ref) and acc == one.n_accepted)
        out = {"ok": same, "chains": N, "generations": G, "rows_compared": int(ref.shape[0]),
               "accepted": int(acc), "exchange": s._exchange,
               "barrier": "peer-memory flags" if s._sync_on else "nccl all-reduce"}
        one.close()
    s.close()
    return out


def dump_outputs(out_dir, s, k_timed):
    """Write what a caller of run_mcmc holds after the last timed generation, as float64 .npy files:
    for a fixed, seeded sample of chains their indices, current states and (history kept) their history rows of
    the last timed generations; every chain's cached ln-likelihood, DREAM's crossover state and the accepted /
    rejected counts of the timed generations."""
    import torch
    rows = np.sort(np.random.RandomState(0).choice(s.n_chains, min(DUMP_ROWS, s.n_chains), replace=False))
    idx = torch.from_numpy(rows).to(s._X.device)
    out = {"state_sample": s._X[idx, :s.dim].cpu().numpy(),
           "state_sample_rows": rows,
           "lnl": s._lnl.cpu().numpy(),
           "p_cr": s.p_cr,
           "delta_m": s.delta_m,
           "accepted_rejected": [s.n_accepted, s.n_rejected]}
    if s._hist.policy == "full":
        # tensor() first writes the newest row, which the fused kernel leaves pending, into the history
        out["history_sample"] = s._hist.tensor()[-min(k_timed, DUMP_GENS):, idx, :s.dim].cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def run_ours(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torchrun for --gpus > 1")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    from bipymc_b200 import DreamMpi, targets, _lib
    N = N_PER_GPU * world
    tgt = targets.Gauss_100D(rho=0.5, dim=DIM)
    np.random.seed(42)
    K, W = args.steps, args.warmup
    # full history = 80 MB per generation per GPU: keep it while it fits comfortably in HBM
    hist_rows = 2 * K + W + SETUP_GENS + 8      # the timed pass and the per-launch-event pass
    if args.history == "full" and hist_rows * N_PER_GPU * DIM * 8 > 0.5 * torch.cuda.get_device_properties(dev).total_memory:
        args.history = "none"
        history_note = "none (the %d requested generations of history would not fit in HBM)" % hist_rows
    else:
        history_note = args.history
    s = DreamMpi(tgt.ln_like, np.zeros(DIM), n_chains=N, varepsilon=np.arange(DIM) + 1.0, seed=42,
                 n_cr_gen=50, burnin_gen=args.burnin_gen, device=local_rank,
                 history=args.history, history_reserve=hist_rows, fused=args.fused,
                 exchange=args.exchange, subpop_k=args.subpop_k)
    lib, h = s._libh, s._handle
    n_local = len(s.rank_chain_ids)

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    k_done = 0

    def gens(n):
        nonlocal k_done
        s.run_mcmc(N * (n + 1), _k_gen0=k_done)
        k_done += n

    gens(SETUP_GENS)
    gens(W)
    sync_all()
    clocks = ClockSampler(local_rank)
    clocks.start()
    # pass 1 -- the timed region: K generations, nothing but the engine's own launches on the stream
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    e0.record()
    gens(K)
    e1.record()
    sync_all()
    ms = e0.elapsed_time(e1)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, s, K)
    # pass 2 -- the next K generations of the same run with CUDA events around every launch
    # (bpm_profile): per-kernel durations for the roofline.  Two event records per launch cost a few
    # microseconds per generation, so they are kept out of `value`; the pass's own time is reported.
    _lib.check(lib.bpm_profile(h, 1))
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    p0.record()
    gens(K)
    p1.record()
    sync_all()
    ms_prof = p0.elapsed_time(p1)
    ck = clocks.stop()
    ms_kind = (C.c_double * 8)()
    n_kind = (C.c_int64 * 8)()
    _lib.check(lib.bpm_profile_read(h, ms_kind, n_kind))
    _lib.check(lib.bpm_profile(h, 0))
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = N * K / (ms * 1e-3)
    acc_frac = s.acceptance_fraction

    # ---- roofline of the dominant kernel (per GPU) -------------------------------------
    kinds = ["split", "propose", "likelihood", "accept", "fused_phase", "cr_reduce"]
    ms_k = [ms_kind[i] for i in range(6)]
    n_k = [int(n_kind[i]) for i in range(6)]
    dom = int(np.argmax(ms_k))
    d = DIM
    hist_b = 8 * d if args.history == "full" else 0
    # algorithmic bytes per chain-step (DESIGN.md): own row + 6 partner rows + write + lnL r/w,
    # + running moments r/w (mean, M2) during burn-in adaptation, + history append
    adapt_b = 8 * d if args.burnin_gen > SETUP_GENS + W + 2 * K else 0  # M2 read by the CR statistic
    step_bytes = 64 * d + 16 + 24 * d + adapt_b + hist_b
    per_kind_bytes = {"fused_phase": step_bytes,
                      "propose": 8 * d * (1 + 6 + 1 + 1),          # own + partners + M2 read + proposal write
                      "likelihood": 8 * d + 8,                      # proposal read + lnL write
                      "accept": 8 * d * (1 + 1 + 4) + hist_b + 16}  # proposal read, state write, moments r/w
    hbm, peak_src = peaks()
    roof = None
    if n_k[dom] > 0 and kinds[dom] in per_kind_bytes:
        chains_per_launch = n_local / 2.0
        avg_ms = ms_k[dom] / n_k[dom]
        ach = per_kind_bytes[kinds[dom]] * chains_per_launch / (avg_ms * 1e-3) / 1e9
        roof = {"bound": "hbm", "kernel": kinds[dom], "achieved": ach, "peak": hbm, "unit": "GB/s",
                "frac": ach / hbm,
                "traffic": ncu_traffic(args.history, adapt_b > 0) if (kinds[dom] == "fused_phase" and world == 1
                                                                      and args.fused == 1) else None,
                "algorithmic_bytes_per_launch": per_kind_bytes[kinds[dom]] * chains_per_launch,
                "avg_launch_ms": avg_ms,
                "bytes_per_chain_step": per_kind_bytes[kinds[dom]], "peak_source": peak_src,
                # share of the event pass's wall time (the shuffle of generation g+1 runs on a side stream under
                # generation g, so the per-kind times do not add up to the step)
                "share_of_step": ms_k[dom] / max(ms_prof, 1e-12)}
        if kinds[dom] == "likelihood":
            fl = 2.0 * d * d * chains_per_launch / (avg_ms * 1e-3) / 1e12
            roof.update({"fp64_tflops": fl})
    # kernels launched in the timed region: one per record, plus the three list-compaction
    # kernels that ride in the "split" record of a sharded generation
    launches = sum(n_k) + (3 * n_k[0] if world > 1 else 0)

    # ---- end to end through the C-ABI with HOST buffers (rank-local population) --------
    e2e = None
    if world == 1 and not args.no_e2e:
        Xh = torch.empty((N, s._ld), dtype=torch.float64).pin_memory()
        Lh = torch.empty((N,), dtype=torch.float64).pin_memory()
        Xh.copy_(s._X.cpu()); Lh.copy_(s._lnl.cpu())
        ke = max(3, min(K, 20))
        g0 = s._hist.length
        for i in range(2):
            _lib.check(lib.bpm_generations_host(h, Xh.data_ptr(), Lh.data_ptr(), k_done + i, g0 + i, 1))
        torch.cuda.synchronize(dev)
        d2h, b = 0, C.c_uint64()
        t0 = time.perf_counter()
        for i in range(ke):
            _lib.check(lib.bpm_generations_host(h, Xh.data_ptr(), Lh.data_ptr(), k_done + 2 + i, g0 + 2 + i, 1))
            lib.bpm_last_d2h_bytes(h, C.byref(b))
            d2h += b.value
        torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
        nb = N * s._ld * 8 + N * 8
        e2e = {"value": N * ke / dt, "unit": UNIT, "h2d_bytes_per_step": nb, "d2h_bytes_per_step": d2h / ke,
               "steps": ke, "ms_per_step": 1e3 * dt / ke,
               "note": "bpm_generations_host: pinned host population -> H2D (all chains) -> one generation "
                       "(crossover adaptation ON: the entry keeps the chains' running moments on the device "
                       "between calls; the chain history is the caller's), the phase kernels storing every accepted "
                       "row straight into the pinned host array -> cached likelihoods D2H (8 N bytes), every step; "
                       "the host arrays hold the full updated population"}

    if world > 1 and not args.no_e2e and args.subpop_k == 0 and s._sync_on:
        # sharded end-to-end step through the C-ABI (bpm_generations_host_sharded): every rank hands in ITS
        # shard (states + cached likelihoods) in pinned host memory; one kernel reads it over PCIe and stores it into
        # every replica (host copy + all-gather fused), a generation runs, accepted rows are stored back into the
        # host shard by the phase kernels, the cached likelihoods return with one copy.
        numa = bind_to_gpu_numa(local_rank)
        lo, hi = int(s.rank_chain_ids[0]), int(s.rank_chain_ids[-1]) + 1
        Xh = torch.empty((hi - lo, s._ld), dtype=torch.float64).pin_memory()
        Lh = torch.empty((hi - lo,), dtype=torch.float64).pin_memory()
        s._flush()
        Xh.copy_(s._X[lo:hi]); Lh.copy_(s._lnl[lo:hi])
        ke = max(3, min(K, 20))
        st = s._state(None)
        stream = s._stream()
        d2h, b = 0, C.c_uint64()

        def e2e_step(i):
            _lib.check(lib.bpm_generations_host_sharded(h, C.byref(st), Xh.data_ptr(), Lh.data_ptr(), k_done + i, 1,
                                                        stream))
        for i in range(2):
            e2e_step(i)
        sync_all()
        t0 = time.perf_counter()
        for i in range(ke):
            e2e_step(2 + i)
            lib.bpm_last_d2h_bytes(h, C.byref(b))
            d2h += b.value
        sync_all()
        dt_t = torch.tensor([time.perf_counter() - t0, d2h / ke], dtype=torch.float64, device=dev)
        dist.all_reduce(dt_t[0:1], op=dist.ReduceOp.MAX)
        dist.all_reduce(dt_t[1:2], op=dist.ReduceOp.SUM)
        dt, d2h_all = float(dt_t[0].item()), float(dt_t[1].item())
        s._pending, s._mom_len = int(st.pending), int(st.mom_len)
        nb = (N * s._ld * 8 + N * 8)
        e2e = {"value": N * ke / dt, "unit": UNIT, "h2d_bytes_per_step": nb, "d2h_bytes_per_step": d2h_all,
               "steps": ke, "ms_per_step": 1e3 * dt / ke, "host_numa_node": numa,
               "shard_in": "copy engines" if os.environ.get("BIPYMC_B200_SHARD_DMA") == "1" else "one kernel",
               "note": "bpm_generations_host_sharded, per rank: pinned host shard -> read over PCIe (zero-copy) and stored "
                       "into the rank's own and the other %d replicas by one kernel (host copy and all-gather fused; "
                       "BIPYMC_B200_SHARD_DMA=1: chunked copies on the copy engines) -> peer barrier -> one sharded "
                       "generation (adaptation ON) whose phase kernels store accepted rows back into the host shard -> "
                       "cached likelihoods D2H; bytes are summed over ranks" % (world - 1)}

    # ---- second point: the same engine on a population AT STATIONARITY (chains drawn from the target) ---
    # acceptance-dependent traffic (accepted-row stores, peer stores, changed-rows write-back) is then
    # quoted at the sampler's real acceptance rate, not that of generations 65-85 of the burn-in
    stationary = None
    if not args.no_stationary and args.subpop_k == 0:
        Ks = max(10, min(K, 50))
        np.random.seed(43)
        s2 = DreamMpi(tgt.ln_like, np.zeros(DIM), n_chains=N, varepsilon=0.0, seed=43, n_cr_gen=50,
                      burnin_gen=args.burnin_gen, device=local_rank, history=args.history,
                      history_reserve=Ks + 16, fused=args.fused, exchange=args.exchange)
        lo2, hi2 = s2._local_range()
        g = torch.Generator(device=dev)
        g.manual_seed(1234)            # same draw on every rank: the replicas must agree
        z = torch.randn((N, DIM), generator=g, device=dev, dtype=torch.float64)
        Lc = torch.linalg.cholesky(torch.from_numpy(tgt.cov).to(dev))
        s2._X[:, :DIM] = z @ Lc.T
        s2._mean_t.copy_(s2._X[lo2:hi2]); s2._hist.set_initial(s2._X[lo2:hi2]); s2._lnl_valid = False
        del z
        k2 = 0

        def gens2(n):
            nonlocal k2
            s2.run_mcmc(N * (n + 1), _k_gen0=k2)
            k2 += n
        gens2(W + 2)
        sync_all()
        q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        q0.record()
        gens2(Ks)
        q1.record()
        sync_all()
        ms2 = q0.elapsed_time(q1)
        if world > 1:
            t = torch.tensor([ms2], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms2 = float(t.item())
        stationary = {"value": N * Ks / (ms2 * 1e-3), "unit": UNIT, "steps": Ks, "ms_per_step": ms2 / Ks,
                      "acceptance_fraction": s2.acceptance_fraction,
                      "init": "chains drawn from the target N(0, Sigma); %d untimed generations" % (W + 2)}
        s2.close()
        del s2

    check = selfcheck_sharded(world, rank, local_rank) if world > 1 else None
    cpu = cpu_baseline_leg() if (rank == 0 and world == 1 and not args.no_cpu) else None
    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic",
                "config": {"workload": "configs[1]: DREAM on Gauss_100D(rho=0.5), %d chains per GPU" % N_PER_GPU,
                           "n_chains": N, "dim": DIM, "del_pairs": 3, "n_cr": 3, "n_cr_gen": 50,
                           "burnin_gen": args.burnin_gen, "history": history_note,
                           "cr_adaptation": "on" if args.burnin_gen > SETUP_GENS + W + 2 * K else "off",
                           "timing": "value / ms_per_step: K generations with only the engine's launches on the "
                                     "stream; kernel_ms / roofline: the next K generations with CUDA events around "
                                     "every launch (ms_per_step_event_pass); gpu_launches counted in the event "
                                     "pass, the timed pass launches the same kernels; kernel_ms['split'] is measured "
                                     "on the side stream and includes its wait for free SMs under the fused launch",
                           "init": "theta_0 + N(0, diag(Sigma)), %d untimed setup generations" % SETUP_GENS,
                           "rng": "philox4x32-10 seed 42", "parallelism": "chains sharded x%d" % world,
                           "exchange": ("none (1 GPU)" if world == 1 else
                                        "sub-population mode: islands of %d chains, re-dealt every %d generations "
                                        "(all-to-all)" % (N_PER_GPU, args.subpop_k) if args.subpop_k > 0 else
                                        "accepted rows stored into peer replicas in-kernel (NVLink P2P) + barrier"
                                        if s._exchange == "p2p" else "NCCL all-gather of the shard per half-phase"),
                           "l2": "working set per generation (state 80 MB + moments 160 MB + history "
                                 "row 80 MB per GPU) exceeds the 126 MB L2; no explicit flush"},
                "ms_per_step_event_pass": ms_prof / K,
                # one proposal + ONE likelihood evaluation per chain-step (the cached ln_like of the current
                # state replaces the reference's second evaluation, samplers.py:330)
                "proposals_and_lnl_evals_per_s": value,
                "acceptance_fraction": acc_frac, "gpu_launches": launches,
                "kernel_ms": dict(zip(kinds, ms_k)), "kernel_launches": dict(zip(kinds, n_k)),
                "roofline": roof, "cpu_baseline": cpu, "e2e": e2e, "clocks": ck,
                "stationary": stationary, "selfcheck": check}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--history", default="full", choices=["full", "none"])
    ap.add_argument("--fused", type=int, default=1, help="1 fused v3 (default), 3 fused 12-producer variant, 2 two-halves fused kernel, 0 split path")
    ap.add_argument("--burnin-gen", type=int, default=2000, help="DREAM burnin_gen (2000 = tests/test_100dgauss.py:109)")
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "allgather"], help="multi-GPU state exchange")
    ap.add_argument("--subpop-k", type=int, default=0,
                    help="sub-population mode: islands re-dealt every K generations (0 = one population, the default)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer end-to-end leg (profiling runs)")
    ap.add_argument("--no-stationary", action="store_true", help="skip the second (stationary-population) point")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed generations, write their results to DIR/<name>.npy (1 GPU only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.gpus != 1):
        ap.error("--dump-outputs needs --impl ours and --gpus 1")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
