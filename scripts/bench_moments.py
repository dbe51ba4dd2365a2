"""Measures moments (csrc/mcmc_sampler.cu RECORD mode + csrc/moments.cu) and empirical_moments.  Reads the card's name,
power limit and max SM clock in the same call, then prints one JSON line per run (and writes them to
DIR/moments_b200.jsonl with --out DIR).

  sample    on the C3 model of bench.py (N = 1000, random 4-regular, J = +-0.4) with 1e6 draws, for B200Gibbs() and the
            default B200Tempering(): the sample_device call, moments with gm's keys, and moments with "pairwise".
  bitgemm   the pairwise bit-GEMM (pair_sums_kernel) at N = 4096 (fields-only model, 4096 chains, 64 records), as kernel
            time from torch.profiler and the popcount rate N^2/2 * records * warps * 32 / time (32-bit popcounts of
            32 lanes each counted as one).
  data      empirical_moments "pairwise" (the tensor-core pass at x = 0) on a C3-sized histogram: 1e7 B200Gibbs draws of
            the C3 model, resident on the device (Session.attach_device), plus the gm-key list.

Call time: CUDA events around a whole call after a warm-up call.

    python scripts/bench_moments.py [--parts sample,bitgemm,data] [--out DIR]
"""
import argparse
import json
import pathlib
import sys

ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "scripts"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import gml_b200  # noqa: E402
from bench import c3_model  # noqa: E402
from bench_sample_mcmc import card  # noqa: E402
from bench_sample_tempering import timed  # noqa: E402
from gml_b200 import B200Gibbs, B200Tempering, FactorGraph  # noqa: E402


def c3_graph():
    return FactorGraph.from_matrix(c3_model(1000)[3])


def part_sample(emit):
    gm = c3_graph()
    n = 1_000_000
    for sampler in (B200Gibbs(), B200Tempering()):
        name = type(sampler).__name__
        _, t_sample = timed(lambda: gml_b200.sample_device(gm, n, 1, sampler))
        _, t_keys = timed(lambda: gml_b200.moments(gm, sampler, n))
        _, t_pair = timed(lambda: gml_b200.moments(gm, sampler, n, keys="pairwise"))
        emit({"part": "sample", "model": "C3 N=1000", "sampler": name, "draws": n, "keys": len(gm.terms),
              "sample_device_ms": t_sample, "moments_keys_ms": t_keys, "moments_pairwise_ms": t_pair,
              "keys_over_sample": t_keys / t_sample, "pairwise_over_sample": t_pair / t_sample})


def part_bitgemm(emit):
    N, chains, n = 4096, 4096, 4096 * 64
    gm = FactorGraph(1, N, "spin", {(i + 1,): 0.1 for i in range(N)})
    sampler = B200Gibbs(chains=chains, burn_in=1, thin=1)
    gml_b200.moments(gm, sampler, n, keys="pairwise")                     # warm-up
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        _, total = timed(lambda: gml_b200.moments(gm, sampler, n, keys="pairwise"), lambda: None)
    kernels = {}
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            kernels[e.name] = kernels.get(e.name, 0.0) + e.device_time / 1e3
    gemm_ms = sum(v for k, v in kernels.items() if "pair_sums_kernel" in k)
    warps, records = chains // 32, n // chains
    popc = (N * N / 2.0) * records * warps
    emit({"part": "bitgemm", "N": N, "chains": chains, "records": records, "call_ms": total, "pair_sums_ms": gemm_ms,
          "popc_words": popc, "popc_per_s": popc / (gemm_ms / 1e3) if gemm_ms else None,
          "kernels_ms": {k.split("(")[0][-40:]: round(v, 3) for k, v in kernels.items()}})


def part_data(emit):
    gm = c3_graph()
    K = 10_000_000
    counts, spins = gml_b200.sample_device(gm, K, 1, B200Gibbs(seed=1))
    sess = gml_b200.Session().attach_device(counts.data_ptr(), spins.data_ptr(), K, 1000, spins.stride(0))
    _, t_pair = timed(lambda: sess.moments("pairwise"))
    keys = list(gm.terms)
    _, t_keys = timed(lambda: sess.moments(keys))
    emit({"part": "data", "model": "C3 N=1000", "rows": K, "pairwise_ms": t_pair, "keys": len(keys), "keys_ms": t_keys})
    sess.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parts", default="sample,bitgemm,data")
    ap.add_argument("--out", default="", help="directory for moments_b200.jsonl (default: print only)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    gpu = card()
    print(gpu, flush=True)
    lines = []

    def emit(rec):
        lines.append(json.dumps({"card": gpu, **rec}))
        print(lines[-1], flush=True)
    for part in args.parts.split(","):
        {"sample": part_sample, "bitgemm": part_bitgemm, "data": part_data}[part](emit)
    if args.out:
        pathlib.Path(args.out).mkdir(parents=True, exist_ok=True)
        (pathlib.Path(args.out) / "moments_b200.jsonl").write_text("".join(l + "\n" for l in lines))


if __name__ == "__main__":
    main()
