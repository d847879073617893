#!/usr/bin/env python
"""Benchmark of the hot path (contract in the task statement, tier rule 4/5).

N = 1 -- BASELINE.json configs[1], "MPS norm/expectation contraction L=200
chi=1024 fp64 on 1xB200".  A *step* is one full contraction <psi|psi> of a
synthetic random MPS (L=200, bond 1024, d=2, fp64): 400 launches of the
pairwise contraction kernel, 1.55 TFLOP of algorithmic work (sum over sites
of 2 l l d r + 2 l d r r).  `value` is device-resident throughput, `e2e` the
same step through the public API from pinned HOST buffers (H2D of all 200 site
tensors inside the timed region, result read back).  The line also carries
`dmrg` (two-site updates at chi=1024: the "DMRG sweep time" half of the
metric) and `shard_unit` (the N>1 workload below run unsharded on this GPU,
the honest N=1 point of the strong-scaling curve).

N > 1 -- the MPS-norm chain does not shard (SURVEY 8e: replicas only), so the
multi-GPU line strong-scales the chi=1024 unit that does: the **bond-sharded
two-site eigensolve** of BASELINE configs[2] (quimb/tensor/tn1d/dmrg.py:
803-870: TNLinearOperator matvec + Lanczos).  Rank r owns the rows
a' in [lo_r, hi_r) of the left environment L[a', w, a] and of every Krylov
vector; per matvec ONE all-gather of the 32 MiB vector (`config.exchange`
says whether it ran as the fused peer-memory kernel or NCCL) and per
Gram-Schmidt pass one all-reduce of <= 24 inner products.  A *step* is one
eigensolve cycle of K = 24 matvecs (a typical site of a sweep from a random
state spends 30-100) on a = b = 1024, d = 2, w = 5: 24 x 86.7 GFLOP.
`value` = that work / max-over-ranks device time; total work is fixed as N
grows ("scaling": "strong").

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]
                  [--dump-outputs DIR]

`--dump-outputs DIR` writes what the last timed step returned as DIR/<name>.npy
(N = 1: the 1x1 norm environment <psi|psi>; N > 1: the Ritz value and the
gathered Ritz vector), so that two builds can be compared output for output:
the inputs are generated from fixed seeds.  For N = 1 that is one number,
because a caller of the MPS-norm path receives nothing else; it still depends
on every one of the 400 contractions of the step.  The CPU arm
(`--impl reference`) times a sample of the workload and has no outputs to
dump, so the two options are rejected together.

`--impl reference` times the reference's own CPU path for the same config
(the numpy/OpenBLAS restatement in oracle/ -- the reference is pure Python +
numpy and cannot be installed on the GPU box) on a FIXED sample of the
workload, all BLAS threads.
"""

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

L_SITES, CHI, PHYS, WBOND = 200, 1024, 2, 5
METRIC = "contracted-TFLOP/s at chi=1024 (MPS norm L=200, fp64)"
METRIC_SHARD = "contracted-TFLOP/s at chi=1024 (bond-sharded DMRG2 two-site eigensolve, fp64)"
CPU_SAMPLE_SITES = 40      # fixed sample of the N=1 workload for the CPU arm
UNIT_MATVECS = 24          # Krylov steps per step of the sharded unit
CPU_UNIT_MATVECS = 4       # fixed sample of the N>1 workload for the CPU arm
UNIT_L = 24                # chain the chi=1024 environments are built from


def bond_dims(L, chi, d):
    out = [1]
    for i in range(1, L):
        e = min(i, L - i)
        cap = d ** e if e < 40 else chi
        out.append(int(min(cap, chi)))
    out.append(1)
    return out


def step_flops(L, chi, d):
    b = bond_dims(L, chi, d)
    fl = 0
    for i in range(L):
        l, r = b[i], b[i + 1]
        fl += 2 * l * l * d * r + 2 * l * d * r * r
    return fl


def matvec_flops(chi=CHI, d=PHYS, w=WBOND):
    # L.x -> .W12 -> .R  (quimb_b200.dmrg.EffHam2.flops with full-size operands)
    return 2 * (chi * w * chi * d * d * chi + chi * d * chi * w * d * w * d
                + chi * d * chi * w * d * w * d + chi * d * d * chi * w * chi)


def config_n1():
    return {"workload": "MPS norm <psi|psi>, L=200 chi=1024 d=2 fp64 (BASELINE configs[1])",
            "flops_per_step": step_flops(L_SITES, CHI, PHYS),
            "l2": "inputs (3.0 GB) are larger than L2; no flush needed",
            "parallelism": "1 GPU"}


def config_shard(world, exchange="nccl"):
    return {"workload": f"DMRG2 two-site eigensolve, Heisenberg MPO w=5, a=b=1024 d=2 fp64 "
                        f"(BASELINE configs[2] local problem), {UNIT_MATVECS} Lanczos matvecs per step",
            "flops_per_step": UNIT_MATVECS * matvec_flops(),
            "l2": "operands per matvec (L-env 40 MiB, intermediate 168 MiB, R-env 40 MiB, "
                  "24 x 32 MiB basis) exceed L2; no flush needed",
            "parallelism": f"bond-sharded over {world} ranks: rows of L-env and of the Krylov "
                           f"vectors; all-gather of the 32 MiB vector per matvec + all-reduce "
                           f"of <= {UNIT_MATVECS} dots per Gram-Schmidt pass",
            "exchange": exchange}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    def __init__(self, index=0):
        self.index = index
        self.rows = []
        self._stop = threading.Event()
        self._th = None

    def start(self):
        def run():
            q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,"
                 "clocks_event_reasons.sw_thermal_slowdown,"
                 "clocks_event_reasons.sw_power_cap")
            while not self._stop.is_set():
                try:
                    out = subprocess.run(
                        ["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                         "--format=csv,noheader,nounits"],
                        capture_output=True, text=True, timeout=5).stdout.strip()
                    if out:
                        self.rows.append([c.strip() for c in out.split(",")])
                except Exception:
                    pass
                self._stop.wait(0.2)
        self._th = threading.Thread(target=run, daemon=True)
        self._th.start()

    def stop(self):
        self._stop.set()
        if self._th:
            self._th.join(timeout=6)
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                 "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1]))
                for nm, v in zip(names, r[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------- CPU arm ---
def _blas_threads_all():
    """Give numpy's BLAS every host thread (torchrun exports OMP_NUM_THREADS=1)
    and report (threads actually used by numpy's BLAS, vendor string)."""
    try:
        import threadpoolctl
        threadpoolctl.threadpool_limits(limits=os.cpu_count(), user_api="blas")
        pools = [p for p in threadpoolctl.threadpool_info() if p.get("user_api") == "blas"]
        npools = [p for p in pools if "numpy" in (p.get("filepath") or "")] or pools
        if npools:
            p = npools[0]
            return int(p.get("num_threads", 1)), f"{p.get('internal_api')} {p.get('version')}"
    except Exception:
        pass
    return int(os.environ.get("OMP_NUM_THREADS", "1")), "unknown"


def cpu_mps_norm(steps, warmup):
    """The reference's CPU path for configs[1] (numpy tensordot chain on
    OpenBLAS) on a FIXED sample: the first CPU_SAMPLE_SITES bulk chi=1024
    sites of the L=200 chain, every run, every arm."""
    from oracle import dmrg_np as dm
    threads, vendor = _blas_threads_all()
    rng = np.random.default_rng(0)
    A = rng.standard_normal((CHI, PHYS, CHI))
    A /= np.linalg.norm(A) ** 0.5
    n = CPU_SAMPLE_SITES
    sites = [A[:1].copy()] + [A] * (n - 2) + [A[:, :, :1].copy()]
    fl = sum(2 * s.shape[0] ** 2 * PHYS * s.shape[2] + 2 * s.shape[0] * PHYS * s.shape[2] ** 2
             for s in sites)
    times = []
    for i in range(steps + warmup):
        t0 = time.perf_counter()
        dm.mps_norm2(sites)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    tm = float(np.mean(times))
    return {"value": fl / tm / 1e12, "ms_per_step": tm * 1e3, "cores": threads,
            "sample": f"{n} chi={CHI} d={PHYS} sites of the L={L_SITES} chain per step "
                      f"({fl / 1e9:.1f} GFLOP, fixed), numpy tensordot, BLAS = {vendor}, "
                      f"{threads} threads of {os.cpu_count()} host CPUs"}


def cpu_eigensolve_unit(steps, warmup):
    """The reference's CPU path for the sharded unit: CPU_UNIT_MATVECS applications of
    the two-site effective Hamiltonian (numpy tensordot chain, the order quimb's
    TNLinearOperator contracts in) + the Lanczos vector algebra of those steps."""
    from oracle import dmrg_np as dm
    threads, vendor = _blas_threads_all()
    rng = np.random.default_rng(0)
    Le = rng.standard_normal((CHI, WBOND, CHI))
    Re = rng.standard_normal((CHI, WBOND, CHI))
    W = dm.mpo_heis(4)[1]
    H = dm.EffHam2(Le, W, W, Re, (CHI, PHYS, PHYS, CHI))
    v = rng.standard_normal(CHI * PHYS * PHYS * CHI)
    v /= np.linalg.norm(v)
    fl = CPU_UNIT_MATVECS * matvec_flops()
    times = []
    for i in range(steps + warmup):
        t0 = time.perf_counter()
        basis = [v]
        for _ in range(CPU_UNIT_MATVECS):
            w_ = H._matvec(basis[-1])
            for _pass in range(2):
                for b in basis:
                    w_ = w_ - (b @ w_) * b
            basis.append(w_ / np.linalg.norm(w_))
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    tm = float(np.mean(times))
    return {"value": fl / tm / 1e12, "ms_per_step": tm * 1e3, "cores": threads,
            "sample": f"{CPU_UNIT_MATVECS} of the {UNIT_MATVECS} matvecs per step "
                      f"({fl / 1e9:.1f} GFLOP, fixed), numpy tensordot, BLAS = {vendor}, "
                      f"{threads} threads of {os.cpu_count()} host CPUs"}


def run_reference(args, rank, world):
    if rank != 0:
        return
    steps, warmup = max(1, args.steps), max(1, args.warmup)
    if args.gpus > 1:
        r = cpu_eigensolve_unit(steps, warmup)
        metric, config, scaling = METRIC_SHARD, config_shard(args.gpus), "strong"
    else:
        r = cpu_mps_norm(steps, warmup)
        metric, config, scaling = METRIC, config_n1(), "weak"
    line = {
        "impl": "reference", "metric": metric, "value": r["value"], "unit": "TFLOP/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": scaling,
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
        "cpu_baseline": {"value": r["value"], "unit": "TFLOP/s", "cores": r["cores"],
                         "kind": "port", "sample": r["sample"]},
        "e2e": {"value": r["value"], "unit": "TFLOP/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------- profile summaries ---
_UNIT = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}


def profile_traffic(path, kernel_substr=None):
    """dram read + write bytes per launch from a committed `ncu --set full`
    summary (profiles/*.txt as written by tools/summarize_profiles.py)."""
    rd = wr = None
    try:
        for ln in open(path):
            for key in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                if ln.startswith(key + " ["):
                    unit = ln[len(key) + 2:ln.index("]")]
                    vals = [float(x) * _UNIT.get(unit, 1.0)
                            for x in ln.split(":", 1)[1].split("|")]
                    if key.endswith("read.sum"):
                        rd = vals
                    else:
                        wr = vals
        if rd and wr:
            return float(np.mean(rd) + np.mean(wr))
    except Exception:
        pass
    return None


def newest_profile(prefixes):
    pdir = os.path.join(ROOT, "profiles")
    for pre in prefixes:
        p = os.path.join(pdir, pre)
        if os.path.exists(p):
            return p
    return None


# ---------------------------------------------------------------- GPU arm ---
def build_unit_problem(qb, dev):
    """chi=1024 environments of the centre bond of a random L=24 Heisenberg
    chain (same data on every rank): (Lenv, W1, W2, Renv, v0, dims)."""
    from quimb_b200.dmrg import _rand_mps
    from quimb_b200.mps import MovingEnvironment, mpo_lrud
    L = UNIT_L
    ham = [mpo_lrud(qb.asarray(w), "lrdu", i, L) for i, w in enumerate(qb.mpo_ham_heis(L))]
    sites = _rand_mps(L, CHI, PHYS, np.float64, seed=7)
    i = L // 2 - 1
    env = MovingEnvironment(sites, ham, begin="left", bsz=2)
    env.move_to(i)
    Lenv, Renv = env()
    A, B = sites[i], sites[i + 1]
    dims = (A.shape[0], A.shape[1], B.shape[1], B.shape[2])
    v0 = qb.Array(qb.contract_pair(A.t, [0, 1, 9], B.t, [9, 2, 3], [0, 1, 2, 3]))
    assert dims == (CHI, PHYS, PHYS, CHI), dims
    return Lenv, ham[i], ham[i + 1], Renv, v0, dims


def run_unit(qb, shard, prob, steps, warmup, barrier, events=True):
    """Time `steps` eigensolve cycles of UNIT_MATVECS matvecs each."""
    import torch
    from quimb_b200.dmrg import EffHam2, ShardedEffHam2
    Lenv, W1, W2, Renv, v0, dims = prob
    if shard is not None:
        H = ShardedEffHam2(Lenv, W1, W2, Renv, dims, shard)
        x0 = H.local_slab(v0)
    else:
        H = EffHam2(Lenv, W1, W2, Renv, dims)
        x0 = v0.reshape(-1)

    def step():
        return qb.eigh_lanczos(H, x0, which="SA", ncv=UNIT_MATVECS, tol=1e-300, maxiter=1,
                               return_info=True, comm=shard, min_steps=UNIT_MATVECS)

    for _ in range(warmup):
        step()
    barrier()
    n0 = H.nmatvec
    ev0 = torch.cuda.Event(enable_timing=True); ev1 = torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(steps):
        theta, x, info = step()
    ev1.record()
    barrier()
    nmv = (H.nmatvec - n0) / steps
    assert nmv == UNIT_MATVECS, nmv
    if shard is not None:
        shard.check()           # a peer-memory kernel that gave up waiting would show here
    return ev0.elapsed_time(ev1) / steps, theta, x, H


def time_exchange(shard, prob, reps=20):
    """The all-gather of one 32 MiB vector alone (ms, device events)."""
    import torch
    from quimb_b200.dmrg import ShardedEffHam2
    Lenv, W1, W2, Renv, v0, dims = prob
    H = ShardedEffHam2(Lenv, W1, W2, Renv, dims, shard)
    x0 = H.local_slab(v0)
    for _ in range(3):
        H.gather(x0)
    torch.cuda.synchronize()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        H.gather(x0)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def dump_outputs(dirname, arrays):
    """Write each array as DIR/<name>.npy (float32 / float64 only)."""
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(dirname, f"{name}.npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-dmrg", action="store_true")
    ap.add_argument("--exchange", default=os.environ.get("QB_EXCHANGE", "auto"),
                    help="N>1: auto | p2p | nccl")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU path, not --impl reference")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import quimb_b200 as qb
    from quimb_b200 import _lib

    assert torch.cuda.is_available(), "bench.py needs a CUDA device"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    args.warmup = max(args.warmup, 3)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    if world > 1:
        line = bench_sharded(args, qb, _lib, dist, dev, rank, local_rank, world, barrier,
                             max_over_ranks)
    else:
        line = bench_mps_norm(args, qb, _lib, dev, barrier)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def dmma_peak(_lib):
    import ctypes
    tf = ctypes.c_double()
    _lib.load().qb_measure_dmma_peak(ctypes.byref(tf), None)
    return tf.value


def bench_sharded(args, qb, _lib, dist, dev, rank, local_rank, world, barrier, max_over_ranks):
    import torch
    from quimb_b200.dist import BondShard
    shard = BondShard(exchange=args.exchange)
    prob = build_unit_problem(qb, dev)
    flops = UNIT_MATVECS * matvec_flops()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    n0 = _lib.launch_count()
    ms, theta, x, H = run_unit(qb, shard, prob, args.steps, args.warmup, barrier)
    launches = _lib.launch_count() - n0
    if args.dump_outputs:
        x_full = H.gather(x).to_numpy()          # collective: every rank takes part
        if rank == 0:
            dump_outputs(args.dump_outputs, {"eigensolve_theta": np.array([theta]),
                                             "eigensolve_x": x_full})
        del x_full
    clocks = sampler.stop() if rank == 0 else None
    ms_max = max_over_ranks(ms)
    value = flops / (ms_max * 1e-3) / 1e12
    gather_ms = max_over_ranks(time_exchange(shard, prob))
    vec_bytes = CHI * PHYS * PHYS * CHI * 8

    # same unit on ONE GPU of this box (rank 0 alone, the others wait): the
    # N=1 point of the strong-scaling curve, measured next to the N-rank run
    single_ms = None
    if rank == 0:
        single_ms, theta1, _, _ = run_unit(qb, None, prob, max(2, args.steps // 2), 2,
                                        torch.cuda.synchronize)
        assert abs(theta1 - theta) <= 1e-9 * abs(theta), (theta1, theta)
    barrier()

    # ---- end to end: operands start in pinned host memory -------------------
    e2e = None
    if not args.no_e2e:
        Lenv, W1, W2, Renv, v0, dims = prob
        host = [t.to_numpy() for t in (Lenv, W1, W2, Renv, v0)]
        hbuf = [torch.from_numpy(np.ascontiguousarray(h)).pin_memory() for h in host]
        in_bytes = sum(h.numel() * 8 for h in hbuf)
        from quimb_b200.dmrg import ShardedEffHam2

        def e2e_step():
            d = [qb.Array(h.to(dev, non_blocking=True)) for h in hbuf]
            Hs = ShardedEffHam2(d[0], d[1], d[2], d[3], dims, shard)
            th, x, info = qb.eigh_lanczos(Hs, Hs.local_slab(d[4]), which="SA", ncv=UNIT_MATVECS,
                                          tol=1e-300, maxiter=1, return_info=True, comm=shard,
                                          min_steps=UNIT_MATVECS)
            return th          # host float: the Ritz value was read back

        for _ in range(2):
            e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            th = e2e_step()
        torch.cuda.synchronize()
        dt = max_over_ranks((time.perf_counter() - t0) / args.steps)
        assert abs(th - theta) <= 1e-9 * abs(theta)
        e2e = {"value": flops / dt / 1e12, "unit": "TFLOP/s",
               "h2d_bytes_per_step": in_bytes, "d2h_bytes_per_step": 8 * (UNIT_MATVECS + 2),
               "ms_per_step": dt * 1e3,
               "note": "every rank uploads the full operands (replicated input), "
                       "d2h = projected-matrix columns + Ritz value"}
    if rank != 0:
        return None
    peak = dmma_peak(_lib)
    mv_ms = ms_max / UNIT_MATVECS
    roofline = {
        "bound": "tensor", "achieved": value / world, "peak": peak, "unit": "TFLOP/s",
        "frac": value / world / peak if peak else None, "traffic": None,
        "kernel": "contract_f64 family (DMMA fp64) inside the sharded matvec; per-GPU "
                  "achieved = whole-step flops / N / step time (includes the exchange and "
                  "the Lanczos vector algebra)",
        "peak_source": "fp64 DMMA issue-rate microbenchmark measured live on this GPU",
    }
    cpu = None
    line = {
        "metric": METRIC_SHARD, "value": value, "unit": "TFLOP/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_max,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": config_shard(world, shard.exchange_name),
        "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
        "roofline": roofline, "cpu_baseline": cpu,
        "exchange": {"kind": shard.exchange_name, "allgather_bytes_per_matvec": vec_bytes,
                     "allgather_ms": gather_ms,
                     "allgather_busbw_GBps": vec_bytes * (world - 1) / world / (gather_ms * 1e-3) / 1e9,
                     "ms_per_matvec_incl_exchange": mv_ms,
                     "bytes_gathered_total": shard.bytes_gathered},
        "shard_unit": {"n1_ms_per_step": single_ms,
                       "n1_tflops": flops / (single_ms * 1e-3) / 1e12,
                       "speedup_vs_n1_same_box": single_ms / ms_max,
                       "strong_scaling_efficiency": single_ms / ms_max / world},
        "check": {"theta": theta},
    }
    return line


def bench_mps_norm(args, qb, _lib, dev, barrier):
    import torch
    from quimb_b200 import mps as qmps
    rank, world = 0, 1
    bonds = bond_dims(L_SITES, CHI, PHYS)
    flops = step_flops(L_SITES, CHI, PHYS)

    # synthetic MPS, quimb layout (l, r, p); scaled like MPS_rand_state does
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    sites = []
    for i in range(L_SITES):
        x = torch.randn((bonds[i], bonds[i + 1], PHYS), dtype=torch.float64,
                        device=dev, generator=g)
        nd = sum(1 for s in x.shape if s > 1) or 1
        x /= torch.linalg.vector_norm(x) ** (1.5 / nd)
        sites.append(x)
    in_bytes = sum(s.numel() * 8 for s in sites)

    def one_step(record=None):
        n = len(sites)
        E = None
        for i, s in enumerate(sites):
            A = qmps.site_lpr(qb.Array(s), "lrp", i, n)
            if E is None:
                E = qb.ones((1, 1), dtype="float64", device=dev)
            if record is not None:
                e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
                e2 = torch.cuda.Event(enable_timing=True)
                e0.record()
                T = qb.contract_pair(E.t, [3, 0], A.t, [0, 1, 2], [3, 1, 2])
                e1.record()
                E = qb.Array(qb.contract_pair(A.t, [3, 1, 5], T, [3, 1, 2], [5, 2]))
                e2.record()
                l, d, r = A.shape
                record.append((e0, e1, 2 * l * l * d * r, l, r))
                record.append((e1, e2, 2 * l * d * r * r, l, r))
            else:
                E = qmps.norm_step(E, A)
        return E

    # ---- device-resident throughput ------------------------------------
    for _ in range(args.warmup):
        one_step()
    barrier()
    sampler = ClockSampler(dev.index or 0)
    sampler.start()
    n0 = _lib.launch_count()
    records = []
    ev0 = torch.cuda.Event(enable_timing=True); ev1 = torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        out = one_step(records)
    ev1.record()
    barrier()
    launches = _lib.launch_count() - n0
    clocks = sampler.stop()
    ms_max = ev0.elapsed_time(ev1) / args.steps
    value = flops / (ms_max * 1e-3) / 1e12
    norm2 = float(out.reshape(()).item())
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"mps_norm2": out.to_numpy()})

    # dominant kernel: the full-size (chi x chi.d x chi) contraction launches
    big = [(a.elapsed_time(b), fl) for a, b, fl, l, r in records if l == CHI and r == CHI]
    k_ms = float(np.mean([t for t, _ in big]))
    k_fl = float(np.mean([fl for _, fl in big]))
    achieved = k_fl / (k_ms * 1e-3) / 1e12

    # ---- end to end: pinned host buffers -> public API -> host scalar ------
    e2e = None
    if not args.no_e2e:
        host = [s.cpu().pin_memory() for s in sites]
        copy_stream = torch.cuda.Stream(device=dev)

        def e2e_step():
            # double-buffered H2D prefetch on a side stream, contraction on
            # the current stream (this is what qb.mps_norm2 does for host input)
            return qb.mps_norm2(host, shape="lrp", copy_stream=copy_stream)

        for _ in range(2):
            e2e_step().item()
        barrier()
        t0 = time.perf_counter()
        t_issue = 0.0
        for _ in range(args.steps):
            ti = time.perf_counter()
            r_dev = e2e_step()
            t_issue += time.perf_counter() - ti   # host time to enqueue one step
            res = r_dev.item()          # D2H of the result inside the timed region
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / args.steps
        assert abs(res - norm2) <= 1e-9 * abs(norm2)
        # what the link alone allows: the same pinned buffers copied with no
        # compute (the e2e step cannot be faster than this)
        stage = [torch.empty(max(h.numel() for h in host), dtype=host[0].dtype, device=dev)
                 for _ in range(4)]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        with torch.cuda.stream(copy_stream):
            for i, h in enumerate(host):
                stage[i % 4][:h.numel()].view(h.shape).copy_(h, non_blocking=True)
        torch.cuda.synchronize()
        h2d_only = time.perf_counter() - t0
        del stage
        e2e = {"value": flops / dt / 1e12, "unit": "TFLOP/s",
               "h2d_bytes_per_step": in_bytes, "d2h_bytes_per_step": 8,
               "ms_per_step": dt * 1e3,
               "host_issue_ms_per_step": t_issue / args.steps * 1e3,
               "h2d_only_ms_per_step": h2d_only * 1e3,
               "h2d_only_GBps": in_bytes / h2d_only / 1e9}
        del host
    del sites
    torch.cuda.empty_cache()

    # ---- roofline denominators --------------------------------------------
    peak = dmma_peak(_lib)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    prof = newest_profile(["r02_contract_kernel_ncu_full.txt", "r01_contract_kernel_ncu_full.txt"])
    traffic = profile_traffic(prof) if prof else None
    roofline = {
        "bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
        "frac": achieved / peak if peak else None, "traffic": traffic,
        "traffic_source": (os.path.relpath(prof, ROOT) if prof else None),
        "algorithmic_bytes_per_launch": 8 * (CHI * CHI + 2 * CHI * PHYS * CHI),
        "kernel": "contract_f64_streamk_kernel<128,128,32> (DMMA fp64, persistent stream-K)",
        "peak_source": "fp64 DMMA issue-rate microbenchmark measured live on this GPU "
                       "(tcgen05 has no f64 kind; MEASURED_PEAKS.json holds bf16 only)",
        "flops_per_launch": k_fl, "ms_per_launch": k_ms,
        "bf16_peak_measured": peaks.get("bf16_tflops"),
        "frac_of_bf16_measured": (achieved / peaks["bf16_tflops"]) if peaks.get("bf16_tflops") else None,
    }

    # ---- the unit the multi-GPU line shards, unsharded on this GPU -----------
    prob = build_unit_problem(qb, dev)
    unit_ms, theta, _, H = run_unit(qb, None, prob, max(2, args.steps // 2), 2, barrier)
    unit_flops = UNIT_MATVECS * matvec_flops()
    shard_unit = {"workload": config_shard(1)["workload"], "ms_per_step": unit_ms,
                  "tflops": unit_flops / (unit_ms * 1e-3) / 1e12,
                  "ms_per_matvec_incl_lanczos": unit_ms / UNIT_MATVECS, "theta": theta}

    # ---- DMRG2 two-site updates at chi = 1024 (the sweep-time half) ----------
    dmrg = None
    if not args.no_dmrg:
        dmrg = bench_dmrg_updates(qb)

    cpu = None
    if not args.no_cpu_baseline:
        r = cpu_mps_norm(2, 1)
        cpu = {"value": r["value"], "unit": "TFLOP/s", "cores": r["cores"], "kind": "port",
               "sample": r["sample"]}
    cfg = config_n1()
    cfg["input_bytes"] = in_bytes
    return {
        "metric": METRIC, "value": value, "unit": "TFLOP/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_max,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": cfg,
        "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
        "roofline": roofline, "cpu_baseline": cpu, "shard_unit": shard_unit, "dmrg": dmrg,
        "check": {"norm2": norm2},
    }


def bench_dmrg_updates(qb):
    """Three consecutive two-site updates at full chi (a = b = 1024) of a
    right sweep over a random L=24 Heisenberg chain, reference settings
    (local_eig_tol 1e-3, cutoff 0, max_bond 1024, method 'svd'); per-update
    time incl. the environment step, matvec count, and the extrapolation to
    BASELINE configs[2] (L=100: 99 updates, 79 of them at full chi)."""
    import torch
    from quimb_b200.mps import env_left_step
    L = UNIT_L
    d = qb.DMRG2(qb.mpo_ham_heis(L), CHI, cutoffs=0.0, mpo_shape="lrdu", seed=5)
    d.right_canonize()
    d._init_right_envs()
    d.lenv = {0: d._ones_env()}
    first = L // 2 - 2
    times, nmv, energies = [], [], []
    for i in range(first + 3):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if i > 0:
            d.lenv[i] = env_left_step(d.lenv[i - 1], d._k[i - 1], d.ham[i - 1])
            d.lenv.pop(i - 1, None)
        le, te = d._update_local_state(i, "right", max_bond=CHI, cutoff=0.0,
                                       cutoff_mode="sum2", method="svd")
        d.renv.pop(i + 1, None)
        torch.cuda.synchronize()
        if i >= first and d._k[i].shape == (CHI, PHYS, CHI):
            times.append(time.perf_counter() - t0)
            nmv.append(d.nmatvecs[-1])
            energies.append(te)
    if not times:
        return None
    per = float(np.median(times))
    return {"s_per_update_chi1024": per, "updates_timed": len(times),
            "matvecs_per_update": float(np.mean(nmv)),
            "sweep_s_L100_extrapolated": per * 79 + per * 0.25 * 20,
            "note": "first right sweep from a random state (hardest local problems); "
                    "a measured full L=100 sweep is in profiles/",
            "energy_after": energies[-1]}


if __name__ == "__main__":
    main()
