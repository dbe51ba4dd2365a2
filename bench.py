#!/usr/bin/env python
"""bench.py -- learn() with RISE on the BASELINE.json headline workload (C3):
N = 1000 sparse random-graph Ising (4-regular, J = +-0.4, h = 0), 1e7-sample histogram.

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torchrun, one rank/GPU)
    python bench.py --impl reference ...                     (CPU oracle port on the host cores)
    python bench.py --config c0|c1|c2|c4                     (time-only lines for the other BASELINE configs, 1 GPU)
    python bench.py --mode node_sharded|sample_sharded|single_process   (multi-GPU partition; default auto)
    python bench.py --dump-outputs DIR                       (also write the last timed step's matrix to DIR/theta.npy)

A "step" is one full learn(): all node problems solved to the stated tolerance on the resident
histogram (+ symmetrisation; + the row all-gather in node-sharded mode).  metric = node*sample evals/s
= N*K*(n_fg + 0.5*n_f)/t  (SURVEY 8d); ms_per_step is the learn() time.  Prints ONE JSON line (rank 0).
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import pathlib
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))


# ------------------------------------------------------------------------------------------------
# workloads
# ------------------------------------------------------------------------------------------------
def regular_graph(n: int, degree: int, seed: int):
    """Random `degree`-regular simple graph by repeated pairing (seeded, deterministic)."""
    rng = np.random.default_rng(seed)
    while True:
        stubs = np.repeat(np.arange(n), degree)
        rng.shuffle(stubs)
        a, b = stubs[0::2], stubs[1::2]
        if np.any(a == b):
            continue
        lo, hi = np.minimum(a, b), np.maximum(a, b)
        if len(set(zip(lo.tolist(), hi.tolist()))) != len(lo):
            continue
        return lo, hi


def csr_of(truth: np.ndarray):
    n = truth.shape[0]
    row_ptr = np.zeros(n + 1, dtype=np.int32)
    col, val = [], []
    for i in range(n):
        nz = [j for j in np.nonzero(truth[i])[0] if j != i]
        row_ptr[i + 1] = row_ptr[i] + len(nz)
        col += nz
        val += truth[i, nz].tolist()
    return row_ptr, np.array(col, dtype=np.int32), np.array(val, dtype=np.float32)


def c3_model(n: int, seed: int = 1000, degree: int = 4, coupling: float = 0.4):
    lo, hi = regular_graph(n, degree, seed)
    rng = np.random.default_rng(seed + 1)
    sign = rng.choice([-1.0, 1.0], size=len(lo))
    truth = np.zeros((n, n))
    for i, j, s in zip(lo, hi, sign):
        truth[i, j] = truth[j, i] = coupling * s
    row_ptr, col, val = csr_of(truth)
    return row_ptr, col, val, truth


def c2_model(side: int = 10, coupling: float = 0.4, seed: int = 100):
    """10 x 10 open-boundary lattice spin glass, J = +-0.4 (SURVEY 8d)."""
    rng = np.random.default_rng(seed)
    n = side * side
    truth = np.zeros((n, n))
    for r in range(side):
        for c in range(side):
            i = r * side + c
            for j in ([i + 1] if c + 1 < side else []) + ([i + side] if r + 1 < side else []):
                truth[i, j] = truth[j, i] = coupling * rng.choice([-1.0, 1.0])
    return truth


def c1_model(n: int = 16, seed: int = 16):
    """Erdos-Renyi p = 0.25, J = +-U[0.2, 0.6], h ~ U[-0.2, 0.2] on the diagonal (SURVEY 8d)."""
    rng = np.random.default_rng(seed)
    m = np.zeros((n, n))
    for i in range(n):
        for j in range(i + 1, n):
            if rng.random() < 0.25:
                m[i, j] = m[j, i] = rng.choice([-1.0, 1.0]) * rng.uniform(0.2, 0.6)
        m[i, i] = rng.uniform(-0.2, 0.2)
    return m


def c4_terms(n: int = 30, seed: int = 30):
    """ring of pair couplings +-0.3 plus n random triples +-0.4, h = 0 (SURVEY 8d); 1-based keys"""
    rng = np.random.default_rng(seed)
    terms = {}
    for i in range(n):
        a, b = i + 1, (i + 1) % n + 1
        terms[(min(a, b), max(a, b))] = float(rng.choice([-0.3, 0.3]))
    for _ in range(n):
        t = tuple(sorted(int(x) + 1 for x in rng.choice(n, 3, replace=False)))
        terms[t] = float(rng.choice([-0.4, 0.4]))
    return terms


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index: int):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.gpu)],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for name, v in zip(names, out[2:]):
                    if v.strip().lower().startswith("active"):
                        self.reasons.add(name)
            except Exception:
                pass
            self._halt.wait(0.2)

    def stop(self):
        self._halt.set()
        self.join(timeout=5)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


DUMP_BYTES = 64 << 20


def dump_outputs(directory: str, name: str, a: np.ndarray) -> None:
    """--dump-outputs: writes `a` as <directory>/<name>.npy in float64, so that two builds can be compared output for
    output.  Above 64 MB only a fixed, seeded sample of its rows is written, with the row numbers in <name>_rows.npy."""
    out = pathlib.Path(directory)
    out.mkdir(parents=True, exist_ok=True)
    a = np.asarray(a, dtype=np.float64)
    if a.nbytes > DUMP_BYTES:
        row_bytes = a.nbytes // a.shape[0]
        rows = np.sort(np.random.default_rng(0).choice(a.shape[0], size=DUMP_BYTES // (row_bytes + 8), replace=False))
        np.save(out / f"{name}_rows.npy", rows.astype(np.float64))
        a = a[rows]
    np.save(out / f"{name}.npy", a)


def load_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return d.get("bf16_tflops_sustained", 1409.8), d.get("hbm_gbs", 6544.3), "measured (MEASURED_PEAKS.json, sustained bf16; int8 peak unmeasured by the driver)"
    return 1590.0, 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
# CPU baseline: the oracle port (reference = Julia + Ipopt cannot run here)
# ------------------------------------------------------------------------------------------------
def cpu_baseline(spins_sample: np.ndarray, counts_sample: np.ndarray, nodes, lam: float):
    """Times the C oracle (per-node second-order solve, dense Hessian every iteration -- what the
    reference asks Ipopt to do) on a bounded sample: `nodes` node problems x K_s histogram rows."""
    sys.path.insert(0, str(ROOT / "oracle"))
    import c_oracle
    c_oracle.set_threads(os.cpu_count() or 1)      # all host cores, also under torchrun (which exports OMP_NUM_THREADS=1)
    t0 = time.time()
    _, info = c_oracle.learn_pairwise_packed(counts_sample, spins_sample, "RISE", lam, False, "exact", 1e-9,
                                             nodes=nodes, return_info=True)
    dt = time.time() - t0
    n_nodes = nodes[1] - nodes[0]
    ks = spins_sample.shape[1]
    evals = n_nodes * ks * (info["n_fgh"] / n_nodes + 0.5 * info["n_f"] / n_nodes)
    return {"value": evals / dt, "unit": "node*sample evals/s", "cores": c_oracle.num_threads(), "kind": "port",
            "seconds": dt, "passes_fgh_per_node": info["n_fgh"] / n_nodes,
            "sample": f"{n_nodes} of N={spins_sample.shape[0]} node problems x first {ks} histogram rows, "
                      f"exact-L1 prox-Newton (f, grad, dense Hessian per iteration), OpenMP over nodes"}


def run_reference(args):
    """--impl reference: the CPU restatement of the reference's per-node solve on the host cores.
    (Julia + JuMP + Ipopt are not in the image, /root/reference has no compilable sources: oracle port.)"""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = args.nspins
    ks = args.cpu_rows
    row_ptr, col, val, _ = c3_model(n)
    # CPU-side Gibbs sample of the bounded row count (same model, same protocol as the device sampler)
    rng = np.random.default_rng(7)
    s = rng.choice(np.array([-1, 1], dtype=np.int8), size=(n, ks))
    for _ in range(args.sweeps):
        for i in range(n):
            fld = np.zeros(ks, dtype=np.float32)
            for q in range(row_ptr[i], row_ptr[i + 1]):
                fld += val[q] * s[col[q]]
            s[i] = np.where(rng.random(ks) < 1.0 / (1.0 + np.exp(-2.0 * fld)), 1, -1)
    counts = np.ones(ks)
    lam = 0.4 * np.sqrt(np.log(n * n / 0.05) / args.nsamples)
    sys.path.insert(0, str(ROOT / "oracle"))
    import c_oracle
    c_oracle.set_threads(os.cpu_count() or 1)
    nodes = (0, min(n, c_oracle.num_threads() * args.cpu_nodes_per_core))
    times, last = [], None
    for step in range(args.warmup + args.steps):
        last = cpu_baseline(np.ascontiguousarray(s), counts, nodes, lam)
        if step >= args.warmup:
            times.append(last["seconds"])
    value = last["value"] * last["seconds"] / np.mean(times)
    line = {"impl": "reference", "metric": "node_sample_evals_per_s", "value": value, "unit": "node*sample evals/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * float(np.mean(times)),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"C3: learn() RISE(0.4,true), N={n} random 4-regular Ising J=+-0.4, M=K={int(args.nsamples):g} Gibbs samples "
                                   f"({args.sweeps} sweeps/chain) -- CPU arm: bounded sample of this workload, see cpu_baseline.sample",
                       "arithmetic": "float64 per-node prox-Newton (f, gradient, dense Hessian per iteration), OpenMP over nodes"},
            "cpu_baseline": {k: last[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": value, "unit": "node*sample evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    line["cpu_baseline"]["value"] = value
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# parity of the timed solution (outside the timed region): float64 KKT check with the oracle's gradient
# ------------------------------------------------------------------------------------------------
def kkt_parity(rows: np.ndarray, node_ids, counts: np.ndarray, spins: np.ndarray, lam: float, mu_lower: float | None):
    """rows: the UN-symmetrised solution rows of `node_ids` (N x N layout: diagonal = field).  Evaluates the float64
    gradient of the smooth part over the FULL histogram with the CPU oracle (gml_oracle_eval_pairwise, restating
    src/GraphicalModelLearning.jl:169-172) and returns the violation of the optimality conditions of
    min f_u(x) + lambda sum_{j != u} |x_j|:  g_j = -lambda sign(x_j) on the support, |g_j| <= lambda off it, g_field = 0."""
    sys.path.insert(0, str(ROOT / "oracle"))
    import c_oracle
    c_oracle.set_threads(os.cpu_count() or 1)
    n = spins.shape[0]
    x = np.zeros((len(node_ids), n + 1))
    for q, u in enumerate(node_ids):
        x[q, :n] = rows[q]
        x[q, n] = rows[q, u]
        x[q, u] = 0.0
    t0 = time.time()
    f, g = c_oracle.eval_pairwise(counts, spins, "RISE", x, np.asarray(node_ids, dtype=np.int32))
    secs = time.time() - t0
    worst, worst_l2, b_max = 0.0, 0.0, 0.0
    for q, u in enumerate(node_ids):
        r = np.zeros(n + 1)
        for j in range(n):
            if j == u:
                continue
            if x[q, j] != 0.0:
                r[j] = g[q, j] + lam * np.sign(x[q, j])
            else:
                r[j] = max(0.0, abs(g[q, j]) - lam)
        r[n] = g[q, n]
        worst = max(worst, float(np.abs(r).max()))
        worst_l2 = max(worst_l2, float(np.linalg.norm(r)))
        b_max = max(b_max, float(np.abs(x[q]).sum()))
    out = {"nodes": [int(u) for u in node_ids], "rows_checked_over_full_K": int(spins.shape[1]),
           "max_kkt_violation": worst, "max_kkt_violation_l2": worst_l2, "oracle_seconds": secs,
           "objective_f64": [float(v) for v in f]}
    if mu_lower is not None:
        # RISE: Hess f_u = sum_k w_k e^{-t_k} S_k S_k' >= e^{-|x_u|_1} C  (C = the weighted second-moment matrix of the features),
        # so F_u is strongly convex with modulus >= e^{-B} lambda_min(C) and |x - x*|_2 <= |r|_2 / mu  (r = min-norm subgradient)
        mu = float(np.exp(-b_max) * mu_lower)
        out["strong_convexity_lower_bound"] = mu
        out["implied_max_dtheta_bound"] = worst_l2 / mu if mu > 0 else None
    return out


def second_moment_lambda_min(spins_dev, chunk: int = 1_000_000) -> float:
    """lambda_min of C = (1/K) S~' S~ over the features [spins | 1] -- exact integer second moments accumulated with bf16
    matmuls (products of +-1 summed in fp32 are exact below 2^24 terms per chunk).  Checker arithmetic, not the product."""
    import torch
    n, k = spins_dev.shape
    acc = torch.zeros((n + 1, n + 1), dtype=torch.float64, device=spins_dev.device)
    for a in range(0, k, chunk):
        s = spins_dev[:, a:a + chunk].to(torch.bfloat16)
        s = torch.cat([s, torch.ones((1, s.shape[1]), dtype=torch.bfloat16, device=s.device)], dim=0)
        acc += (s @ s.T).double()
    ev = torch.linalg.eigvalsh(acc / k)
    return float(ev[0].item())


# ------------------------------------------------------------------------------------------------
# GPU arm, headline config
# ------------------------------------------------------------------------------------------------
def run_b200(args):
    import torch
    import torch.distributed as dist
    import gml_b200
    from gml_b200 import _lib
    from gml_b200.distributed import (learn_sample_sharded, learn_sharded, sample_slice, shard_bounds, upload_replicated,
                                      upload_sample_sharded)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    dev = torch.device(f"cuda:{local}")
    lib = _lib.load()

    n, k = args.nspins, int(args.nsamples)
    # partition of the multi-GPU solve (SURVEY 8e): sample slices stream K/world rows per rank and pass, node shards stream the
    # whole replicated histogram on every rank; auto = sample slices whenever every rank keeps a GPU-filling number of rows
    mode = args.mode
    if mode == "auto":
        mode = "sample_sharded" if (world > 1 and k // world >= 65536) else "node_sharded"
    if world == 1:
        mode = "single_gpu"
    row_ptr, col, val, truth = c3_model(n)
    # ---- synthetic histogram, generated once on the device (same seed on every rank => identical bytes)
    spins = torch.empty((n, k), dtype=torch.int8, device=dev)
    counts = torch.ones(k, dtype=torch.float64, device=dev)
    t0 = time.time()
    _lib.check(lib.gml_b200_sample_gibbs_device(local, n, row_ptr.ctypes.data, col.ctypes.data, val.ctypes.data, None,
                                                k, args.sweeps, 1000, ctypes.c_void_p(spins.data_ptr()), k, None))
    torch.cuda.synchronize()
    gen_s = time.time() - t0
    form = gml_b200.RISE(0.4, True)
    lam = gml_b200.regularizer_lambda(0.4, n, float(k))
    method = gml_b200.B200(solver=args.solver, tol=args.tol, device=local, profile=True, verbose=args.verbose, multilevel=args.multilevel,
                           coarse_level=not args.no_coarse, warm_start=args.warm_start)
    if mode == "sample_sharded":
        sb, se = sample_slice(k, world, rank)
        my_spins = spins[:, sb:se].contiguous()
        my_counts = counts[sb:se].contiguous()
        sess = gml_b200.Session(local).attach_device(my_counts.data_ptr(), my_spins.data_ptr(), se - sb, n, se - sb)
        sess.comm_init()
        b, e = 0, n
        learn_fn = lambda m, sym=True: learn_sample_sharded(sess, form, m, symmetrize=sym)
    else:
        sess = gml_b200.Session(local).attach_device(counts.data_ptr(), spins.data_ptr(), k, n, k)
        b, e = shard_bounds(n, world, rank)
        learn_fn = lambda m, sym=True: learn_sharded(sess, form, m, symmetrize=sym)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def one_step():
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record()
        full = learn_fn(method)
        ev1.record()
        barrier()
        ms = torch.tensor([ev0.elapsed_time(ev1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), full, dict(method.last_stats)

    for _ in range(args.warmup):
        one_step()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    times, stats, full = [], None, None
    for _ in range(args.steps):
        ms, full, stats = one_step()
        times.append(ms)
    clocks = sampler.stop() if rank == 0 else {}
    ms_step = float(np.mean(times))
    # evals: passes weighted by the fraction of the histogram and of the nodes they sweep, summed over the ranks' parts
    # (node shards: each rank counts its nodes x K; sample slices: each rank counts N x its rows)
    ev = torch.tensor([stats["evals"]], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ev)
    value = float(ev.item()) / (ms_step * 1e-3)
    learned = full.cpu().numpy()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, "theta", learned)      # the symmetrised N x N matrix of the last timed step
    recon_err = float(np.abs(learned - np.diag(np.diag(learned)) - truth).max())
    nnz_row = (learned != 0.0).sum(axis=1)          # symmetrised support (union of the two directed estimates)

    # ---- the un-symmetrised rows of the timed configuration (for the KKT check below), and lambda_min of the feature second moments
    unsym = learn_fn(gml_b200.B200(solver=args.solver, tol=args.tol, device=local, coarse_level=not args.no_coarse, warm_start=args.warm_start), False)
    mu_lower = second_moment_lambda_min(spins) if (args.parity and rank == 0) else None

    # ---- multi-GPU correctness, visible to the driver: every rank must hold the SAME matrix, and a single-rank re-solve of one
    # 64-node tile on the full replicated histogram must reproduce those rows of the multi-GPU solve (both at one precision level,
    # where node problems follow partition-independent paths: src/GraphicalModelLearning.jl:161 has no cross-node dependency)
    multi_gpu_check = None
    if world > 1:
        one_level = gml_b200.B200(solver=args.solver, tol=args.tol, device=local, coarse_level=False, warm_start=False)
        multi = learn_fn(one_level, False)
        ref0 = multi.clone()
        dist.broadcast(ref0, src=0)
        same = torch.tensor([float((ref0 - multi).abs().max().item())], device=dev)
        dist.all_reduce(same, op=dist.ReduceOp.MAX)
        tile_b = 64 * (rank % max(1, n // 64))
        tile_e = min(n, tile_b + 64)
        chk = gml_b200.Session(local).attach_device(counts.data_ptr(), spins.data_ptr(), k, n, k)
        tile_rows = torch.empty((tile_e - tile_b, n), dtype=torch.float64, device=dev)
        chk.solve_pairwise_device(form, gml_b200.B200(solver=args.solver, tol=args.tol, device=local, coarse_level=False, warm_start=False),
                                  tile_rows.data_ptr(), tile_b, tile_e)
        torch.cuda.synchronize()
        tile_err = torch.tensor([float((tile_rows - multi[tile_b:tile_e]).abs().max().item())], device=dev)
        dist.all_reduce(tile_err, op=dist.ReduceOp.MAX)
        two_level = torch.tensor([float((unsym - multi).abs().max().item())], device=dev)
        chk.close()
        del chk, tile_rows, multi, ref0
        multi_gpu_check = {"max_abs_diff_between_ranks": float(same.item()),
                           "max_abs_diff_vs_single_rank_tile_resolve": float(tile_err.item()),
                           "max_abs_diff_two_level_vs_one_level_solve": float(two_level.item()),
                           "tile": "64 nodes per rank (a different tile on every rank), re-solved on ONE GPU from the full histogram; "
                                   "both solves cold and on one precision level (coarse_level=False, warm_start=False)"}
        assert mode == "node_sharded" or same.item() == 0.0, f"ranks disagree: {same.item()}"
        assert tile_err.item() <= 1e-6, f"multi-GPU solve differs from the single-rank re-solve: {tile_err.item()}"

    # ---- roofline of the dominant kernel (per-launch CUDA-event times from the library, this rank)
    nn_local = e - b
    k_local = (sample_slice(k, world, rank)[1] - sample_slice(k, world, rank)[0]) if mode == "sample_sharded" else k
    F = n + 1
    flops_per_launch = 2.0 * k_local * F * nn_local              # algorithmic: 2*K*F per node per contraction
    nfull = max(1, stats["timed_full_passes"])          # launches that swept this rank's whole part (finest level)
    ker = {"tc_energy_pair_kernel(full)": (stats["energy_fg_ms"], nfull),
           "tc_grad_kernel": (stats["grad_ms"], nfull),
           "tc_energy_pair_kernel(objective)": (stats["energy_f_ms"], stats["n_f_passes"])}
    dom = max(ker, key=lambda kk: ker[kk][0])
    peak_tf, peak_gbs, peak_src = load_peaks()
    roof = None
    traffic = None
    for tname in ("r2_traffic.json", "r1_traffic.json"):
        tfile = ROOT / "profiles" / tname
        if tfile.exists() and world == 1 and n == 1000 and k == 10_000_000 and traffic is None:
            traffic = json.loads(tfile.read_text()).get("c3_1gpu", {}).get(dom.split("(")[0])      # from the committed ncu --set full capture
    if ker[dom][0] > 0:
        avg_ms = ker[dom][0] / max(1, ker[dom][1])
        ach = flops_per_launch / (avg_ms * 1e-3) / 1e12
        roof = {"bound": "tensor", "kernel": dom, "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf,
                "traffic": traffic, "avg_launch_ms": avg_ms, "launches": ker[dom][1], "peak_source": peak_src,
                "algorithmic_flops_per_launch": flops_per_launch,
                "kernel_ms_share": {kk: v[0] / stats["solve_ms"] for kk, v in ker.items()},
                "note": "launches over this rank's whole part only (compacted tail passes are not timed, so kernel_ms_share sums to < 1); "
                        "algorithmic flops = 2*K*F*nodes per contraction; the int8 limb split executes 3x (energy) / 2x (gradient) that "
                        "many int8 MACs on the coarse precision level, 4x / 3x on the fine one; the denominator is the measured bf16 peak "
                        "(the driver measures no int8 peak; cuBLASLt int8 reaches ~2x it on these boxes)"}

    # ---- e2e: host (pinned) buffers in, host matrix out, through the same C ABI
    e2e = None
    h_spins = None
    if not args.skip_e2e:
        h_spins = torch.empty((n, k), dtype=torch.int8, pin_memory=True)
        h_spins.copy_(spins)
        h_counts = torch.ones(k, dtype=torch.float64, pin_memory=True)
        sess.close()
        if mode == "sample_sharded":
            del my_spins, my_counts
        del spins
        torch.cuda.empty_cache()
        e2e_method = gml_b200.B200(solver=args.solver, tol=args.tol, device=local, multilevel=args.multilevel, coarse_level=not args.no_coarse,
                                   warm_start=args.warm_start)
        e_times = []
        for it in range(1 + args.e2e_steps):
            barrier()
            t0 = time.perf_counter()
            if mode == "sample_sharded":
                s2 = upload_sample_sharded(gml_b200.Session(local), h_counts, h_spins)   # H2D of this rank's K/world rows + validate + layout
            else:
                s2 = upload_replicated(gml_b200.Session(local), h_counts, h_spins)    # H2D (1/world per rank) + NVLink all-gather + validate + layout
            torch.cuda.synchronize(); t1 = time.perf_counter()
            out = (learn_sample_sharded(s2, form, e2e_method) if mode == "sample_sharded" else learn_sharded(s2, form, e2e_method))
            host = out.cpu()                                                  # D2H of the N x N result
            torch.cuda.synchronize()
            if args.verbose and rank == 0:
                print(f"[bench e2e] upload {t1 - t0:.3f} s, solve+gather+d2h {time.perf_counter() - t1:.3f} s", file=sys.stderr)
            dt = torch.tensor([time.perf_counter() - t0], device=dev)
            if world > 1:
                dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            st2 = dict(e2e_method.last_stats)
            s2.close()
            if it > 0:
                e_times.append(float(dt.item()))
        ev2 = torch.tensor([st2["evals"]], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ev2)
        e_med = float(np.median(e_times))                 # median of the timed end-to-end calls
        h2d = int(n * k + 8 * k) if mode != "sample_sharded" else int(n * k + 8 * k)      # every histogram byte crosses the host link once
        e2e = {"value": float(ev2.item()) / e_med, "unit": "node*sample evals/s",
               "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": int(8 * n * n * world),
               "learn_seconds": e_med, "steps": len(e_times), "all_seconds": e_times,
               "input": "pre-packed pinned host buffers: counts f64[K], spins int8 [N x K]; the reference's own K x (N+1) Float64 matrix "
                        "form is e2e_from_matrix (N = 1) and scripts/bench_matrix_input.py"}

    # ---- parity of the timed solution: float64 KKT check of 8 random rows over the full K (CPU oracle), outside the timed region
    parity = None
    if args.parity and rank == 0:
        if h_spins is None:
            h_spins = spins.cpu()
        node_ids = sorted(np.random.default_rng(5).choice(n, size=min(args.parity_nodes, n), replace=False).tolist())
        rows = unsym[node_ids].cpu().numpy()
        parity = kkt_parity(rows, node_ids, np.ones(k), h_spins.numpy(), lam, mu_lower)
        parity["tolerance_note"] = ("solver stops at max-norm of the prox-gradient mapping <= tol; the KKT residual is that mapping measured with an "
                                    "independent float64 gradient over all K rows")

    # ---- e2e from the reference's own input type (N = 1 only; needs ~100 GB of free host memory): learn() receives a K x (N+1)
    # column-major Float64 matrix (src/GraphicalModelLearning.jl:69-81, test/runtests.jl:71); the call narrows it on the host
    # cores while streaming it to the device (gml_b200_learn_pairwise_matrix), solves, symmetrises and returns the N x N matrix
    e2e_matrix = None
    if rank == 0 and world == 1 and not args.skip_e2e and not args.skip_matrix_e2e and h_spins is not None:
        try:
            import psutil
            need = 8.0 * k * (n + 1)
            if psutil.virtual_memory().available > need + 40e9:
                t_build = time.time()
                mat = np.empty((k, n + 1), dtype=np.float64, order="F")          # Julia-native layout
                mat[:, 0] = 1.0
                hs = h_spins.numpy()
                for i in range(n):
                    mat[:, 1 + i] = hs[i]
                t_build = time.time() - t_build
                m_times, m_ingest = [], []
                for it in range(1 + args.matrix_e2e_steps):
                    mm = gml_b200.B200(solver=args.solver, tol=args.tol, device=local, coarse_level=not args.no_coarse, warm_start=args.warm_start)
                    t0 = time.perf_counter()
                    theta = gml_b200.learn_matrix(mat, form, mm)
                    dt = time.perf_counter() - t0
                    if it:
                        m_times.append(dt); m_ingest.append(mm.last_stats["h2d_ms"] * 1e-3)
                m_med = float(np.median(m_times))
                e2e_matrix = {"value": mm.last_stats["evals"] / m_med, "unit": "node*sample evals/s", "learn_seconds": m_med, "all_seconds": m_times,
                              "ingest_seconds": float(np.median(m_ingest)), "matrix_bytes": int(mat.nbytes), "dtype": "float64",
                              "max_abs_diff_vs_packed_entry": float(np.abs(theta - learned).max()), "host_matrix_build_seconds": t_build,
                              "note": "gml_b200_learn_pairwise_matrix: threaded host narrowing (+-1 validated) overlapped with H2D of the bytes, "
                                      "lambda and num_samples computed by the library, solve, device symmetrisation, D2H"}
                del mat
            else:
                e2e_matrix = {"skipped": "less than %.0f GB of host memory available" % ((need + 40e9) / 1e9)}
        except Exception as err:          # never lose the bench line to the optional measurement
            e2e_matrix = {"skipped": f"{type(err).__name__}: {err}"}

    cpu = None
    if rank == 0 and world == 1 and not args.skip_cpu:      # reported at N=1 only
        sys.path.insert(0, str(ROOT / "oracle"))
        import c_oracle
        c_oracle.set_threads(os.cpu_count() or 1)
        ks = args.cpu_rows
        src = h_spins if h_spins is not None else spins.cpu()
        sample = np.ascontiguousarray(src[:, :ks].numpy())
        nodes = (0, min(n, c_oracle.num_threads() * args.cpu_nodes_per_core))
        cpu = cpu_baseline(sample, np.ones(ks), nodes, lam)
        cpu["learn_seconds_extrapolated"] = (n * k * cpu["passes_fgh_per_node"]) / cpu["value"]

    if rank == 0:
        line = {"metric": "node_sample_evals_per_s", "value": value, "unit": "node*sample evals/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "int8",
                "data": "synthetic",
                "config": {"workload": f"C3: learn() RISE(0.4,true), N={n} random 4-regular Ising J=+-0.4, M=K={k:g} Gibbs samples "
                                       f"({args.sweeps} sweeps/chain), {world} GPU(s), partition: {mode}",
                           "partition": mode,
                           "arithmetic": "int8 tensor-core contractions with s32/s64 accumulation (exact), f32 per-sample epilogue, f64 solver state",
                           "tol": args.tol, "solver": args.solver, "l2_note": "inputs (10 GB int8 + 20-30 GB residual digits) exceed the 126 MB L2",
                           "lambda": lam, "sampler_seconds": gen_s,
                           "warm_start": "library default (mean-field start for cold solves of all nodes; node shards start cold)" if args.warm_start is None else bool(args.warm_start)},
                "learn_seconds": ms_step * 1e-3, "passes": {"fg": stats["n_fg_passes"], "f": stats["n_f_passes"], "iterations": stats["iterations"]},
                "max_abs_coupling_error_vs_truth": recon_err, "max_residual": stats["max_residual"], "n_stalled": stats.get("n_stalled", 0),
                "support": {"mean_nnz_per_row": float(nnz_row.mean()), "max_nnz_per_row": int(nnz_row.max()), "true_degree": 4},
                "gpu_launches": int(stats["kernel_launches"]) * args.steps,
                "roofline": roof, "cpu_baseline": cpu, "e2e": e2e, "e2e_from_matrix": e2e_matrix, "parity": parity, "multi_gpu_check": multi_gpu_check, "clocks": clocks}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------
# the other BASELINE configs: time-only lines (latency-bound, SURVEY 8d), one GPU
# ------------------------------------------------------------------------------------------------
def run_small(args):
    import torch
    import gml_b200
    from gml_b200 import _lib
    sys.path.insert(0, str(ROOT / "oracle"))
    cfg = args.config
    dev = torch.device("cuda:0")
    torch.cuda.set_device(0)
    lib = _lib.load()
    rng = np.random.default_rng(0)
    extra = {}
    if cfg in ("c0", "c1"):
        import gml_oracle as o
        model = np.array([[0, .1, .2], [.1, 0, .3], [.2, .3, 0]]) if cfg == "c0" else c1_model()
        n = model.shape[0]
        hist = o.sample_exact(o.matrix_to_terms(model), n, 100_000, rng)      # exact multinomial over 2^N configurations
        counts, spins = gml_b200.pack_histogram(hist)
        form = gml_b200.RISE(0.4, True)
        name = "C0: README quick-start, 3 spins, M=1e5" if cfg == "c0" else "C1: N=16 random Ising, M=1e5 (exact sampler)"
    elif cfg == "c2":
        truth = c2_model()
        n, k = 100, 1_000_000
        row_ptr, col, val = csr_of(truth)
        d = torch.empty((n, k), dtype=torch.int8, device=dev)
        _lib.check(lib.gml_b200_sample_gibbs_device(0, n, row_ptr.ctypes.data, col.ctypes.data, val.ctypes.data, None, k, 60, 100,
                                                    ctypes.c_void_p(d.data_ptr()), k, None))
        spins, counts = d.cpu().numpy(), np.ones(k)
        form = gml_b200.RISE(0.4, True)
        name = "C2: N=100 10x10 lattice spin glass J=+-0.4, M=K=1e6 Gibbs samples"
    elif cfg == "c4":
        n, k = 30, int(args.nsamples) if args.nsamples != 1e7 else 1_000_000
        terms = c4_terms(n)
        spins = gml_b200.sample_terms_device(terms, n, k, sweeps=80, seed=30).cpu().numpy()
        counts = np.ones(k)
        form = gml_b200.multiRISE(0.4, True, 3)
        name = f"C4: N=30, ring pairs +-0.3 + 30 triples +-0.4, multiRISE(0.4,true,3), M=K={k:g} Gibbs samples"
    else:
        raise SystemExit(f"unknown config {cfg}")
    n, k = spins.shape
    sess = gml_b200.Session(0).upload(counts, np.ascontiguousarray(spins))
    method = gml_b200.B200(tol=args.tol if cfg in ("c2", "c4") else 0.0, profile=True)
    multibody = isinstance(form, gml_b200.multiRISE)

    def solve():
        return sess.solve_multibody(form, method, return_info=True) if multibody else sess.solve_pairwise(form, method, return_info=True)

    for _ in range(args.warmup):
        solve()
    times, e_times = [], []
    for _ in range(args.steps):
        torch.cuda.synchronize(); t0 = time.perf_counter()
        res, info = solve()
        torch.cuda.synchronize(); times.append(time.perf_counter() - t0)
    for _ in range(args.steps):      # end to end: one-shot C entry (create + upload + solve + download + destroy)
        t0 = time.perf_counter()
        gml_b200.learn_packed(counts, np.ascontiguousarray(spins), form, gml_b200.B200(tol=method.tol))
        e_times.append(time.perf_counter() - t0)
    st = method.last_stats
    sec = float(np.mean(times))
    F = int(lib.gml_b200_multibody_num_keys(n, 3)) if multibody else n + 1
    peak_tf, peak_gbs, peak_src = load_peaks()
    passes = st["n_fg_passes"] + st["n_f_passes"]
    hbm_bytes = passes * k * (n + 8.0)                       # one sweep of the int8 histogram + weights per pass (algorithmic)
    if cfg == "c4":
        # parity on the timed solution: three node problems against the oracle need minutes at K = 1e6; the committed test
        # (tests/test_gpu_headline_parity.py::test_multirise_c4_shape_vs_oracle) pins this shape at K = 1e5.  Here: recovery of truth.
        fg = gml_b200.learn_packed(counts, np.ascontiguousarray(spins), form, gml_b200.B200(tol=method.tol))
        extra["max_abs_error_vs_generating_terms"] = float(max(abs(fg[key] - v) for key, v in terms.items()))
        extra["largest_spurious_term"] = float(max((abs(v) for key, v in fg.terms.items() if key not in terms), default=0.0))
    line = {"metric": "learn_seconds", "value": sec, "unit": "s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * sec, "higher_is_better": False, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64" if st["solver_used"] == 1 else "int8", "data": "synthetic",
            "config": {"workload": name, "features_per_node": F, "K": int(k), "solver_used": {1: "newton", 2: "fista_cc", 3: "fista_tc"}[st["solver_used"]]},
            "evals_per_s": st["evals"] / sec, "passes": {"fg": st["n_fg_passes"], "f": st["n_f_passes"], "iterations": st["iterations"]},
            "gpu_launches": int(st["kernel_launches"]) * args.steps,
            "roofline": {"bound": "hbm", "achieved": hbm_bytes / sec / 1e9, "peak": peak_gbs, "unit": "GB/s", "frac": hbm_bytes / sec / 1e9 / peak_gbs,
                         "traffic": None, "note": "latency-bound configuration (whole histogram fits in L2 or a pass is tens of microseconds): "
                                                  "time is the figure of merit, the HBM fraction is reported for honesty (SURVEY 8d)"},
            "e2e": {"value": float(np.median(e_times)), "unit": "s", "h2d_bytes_per_step": int(n * k + 8 * k), "d2h_bytes_per_step": int(8 * n * F),
                    "steps": len(e_times)},
            **extra}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c3", choices=["c0", "c1", "c2", "c3", "c4"])
    ap.add_argument("--mode", default="auto", choices=["auto", "node_sharded", "sample_sharded"])
    ap.add_argument("--nspins", type=int, default=1000)
    ap.add_argument("--nsamples", type=float, default=1e7)
    ap.add_argument("--sweeps", type=int, default=40)
    ap.add_argument("--tol", type=float, default=1e-6)
    ap.add_argument("--solver", default="fista_tc")
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--no-parity", dest="parity", action="store_false")
    ap.add_argument("--parity-nodes", type=int, default=8)
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--skip-matrix-e2e", action="store_true")
    ap.add_argument("--matrix-e2e-steps", type=int, default=3)
    ap.add_argument("--cpu-rows", type=int, default=2048)
    ap.add_argument("--cpu-nodes-per-core", type=int, default=1)
    ap.add_argument("--verbose", type=int, default=0)
    ap.add_argument("--multilevel", action="store_true")
    ap.add_argument("--no-coarse", action="store_true")
    ap.add_argument("--warm-start", dest="warm_start", action="store_true", default=None)
    ap.add_argument("--no-warm-start", dest="warm_start", action="store_false")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the learned matrix of the last timed step to DIR/theta.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.config != "c3"):
        ap.error("--dump-outputs applies to the C3 workload on the GPU")
    if args.impl == "reference":
        run_reference(args)
    elif args.config != "c3":
        run_small(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
