"""Measures the Swendsen-Wang sampler (sample_device with B200SwendsenWang, cluster_kernel in csrc/mcmc_sampler.cu) against
B200Gibbs and B200Tempering, in one process.  Prints the card's name, power limit and max SM clock first, then one JSON
line per run.

  ferro     8 x 8, 32 x 32 and 64 x 64 open ferromagnets at J = 1 and J = 0.44 (about the critical coupling), 1024 chains
            of 40 records at the defaults: B200Gibbs, B200Tempering (default ladder and 32 rungs geometric from 1 to 0.1)
            and B200SwendsenWang: call time, R-hat (energy, magnetisation) and spin updates per second (chains * sweeps *
            N / call time; one cluster update counts N).
  glass     C2 (N = 100, 1e6 draws) and C3 (N = 1000, 1e7 draws) of bench.py at the defaults, B200Gibbs and
            B200SwendsenWang: call time, R-hat and the max error of the RISE(0.4, false) couplings and fields learned from
            the sample.
  schedule  B200SwendsenWang at (burn_in, thin) settings below the defaults on C2 and the 32 x 32 J = 1 and 64 x 64
            J = 0.44 ferromagnets: R-hat, to pick the cheapest default with R-hat <= 1.01 everywhere.

Call time: CUDA events around a whole sample_device call after a warm-up call.  Each item runs once.

    python scripts/bench_sample_cluster.py [--parts ferro,glass,schedule] [--out DIR]
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
from bench import c2_model, c3_model  # noqa: E402
from bench_sample_mcmc import card, learned_error  # noqa: E402
from bench_sample_tempering import LADDER_32, open_ferromagnet, timed  # noqa: E402
from gml_b200 import B200Gibbs, B200SwendsenWang, B200Tempering, FactorGraph  # noqa: E402

CHAINS, RECORDS = 1024, 40


def describe(sampler):
    if isinstance(sampler, B200Tempering):
        return f"B200Tempering({'default' if sampler.betas is None else len(sampler.betas)} rungs)"
    return type(sampler).__name__


def part_ferro():
    for side in (8, 32, 64):
        for J in (1.0, 0.44):
            gm = open_ferromagnet(side, side, J)
            N = side * side
            for sampler in (B200Gibbs(seed=5, chains=CHAINS), B200Tempering(seed=5, chains=CHAINS),
                            B200Tempering(seed=5, chains=CHAINS, betas=LADDER_32), B200SwendsenWang(seed=5, chains=CHAINS)):
                _, ms = timed(lambda: gml_b200.sample_device(gm, RECORDS * CHAINS, sampler=sampler))
                sweeps = sampler.burn_in + RECORDS * sampler.thin
                rungs = 1 if not isinstance(sampler, B200Tempering) else len(sampler.betas or [0] * 16)
                yield {"part": "ferro", "model": f"{side}x{side} J={J}", "sampler": describe(sampler), "draws": RECORDS * CHAINS,
                       "chains": CHAINS, "burn_in": sampler.burn_in, "thin": sampler.thin, "call_ms": round(ms, 2),
                       "rhat_energy": sampler.last_rhat[0][0], "rhat_magnetisation": sampler.last_rhat[0][1],
                       "spin_updates_per_s": CHAINS * rungs * sweeps * N / (ms * 1e-3)}


def part_glass():
    for name, model, draws in (("c2", lambda: c2_model(), 1_000_000), ("c3", lambda: c3_model(1000)[3], 10_000_000)):
        truth = model()
        gm = FactorGraph.from_matrix(truth)
        for sampler in (B200Gibbs(seed=1), B200SwendsenWang(seed=1)):
            (counts, spins), ms = timed(lambda: gml_b200.sample_device(gm, draws, sampler=sampler))
            rec = {"part": "glass", "config": name, "sampler": describe(sampler), "draws": draws, "call_ms": round(ms, 2),
                   "rhat_energy": sampler.last_rhat[0][0], "rhat_magnetisation": sampler.last_rhat[0][1]}
            rec["coupling_err"], rec["field_err"] = learned_error(truth, counts, spins)
            del counts, spins
            torch.cuda.empty_cache()
            yield rec


def part_schedule():
    models = [("c2", FactorGraph.from_matrix(c2_model()), 1_000_000, 0),
              ("32x32 J=1.0", open_ferromagnet(32, 32, 1.0), RECORDS * CHAINS, CHAINS),
              ("64x64 J=0.44", open_ferromagnet(64, 64, 0.44), RECORDS * CHAINS, CHAINS)]
    for burn_in, thin in ((200, 10), (100, 5), (50, 2), (20, 1)):
        for name, gm, draws, chains in models:
            sampler = B200SwendsenWang(seed=2, chains=chains, burn_in=burn_in, thin=thin)
            _, ms = timed(lambda: gml_b200.sample_device(gm, draws, sampler=sampler))
            yield {"part": "schedule", "model": name, "burn_in": burn_in, "thin": thin, "draws": draws, "chains": chains,
                   "call_ms": round(ms, 2), "rhat_energy": sampler.last_rhat[0][0],
                   "rhat_magnetisation": sampler.last_rhat[0][1]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parts", default="ferro,glass,schedule")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    gpu = card()
    print(f"card: {gpu}", flush=True)
    runs = {"ferro": part_ferro, "glass": part_glass, "schedule": part_schedule}
    lines = []
    for part in a.parts.split(","):
        for rec in runs[part]():
            rec["card"] = gpu
            print(json.dumps(rec), flush=True)
            lines.append(rec)
    if a.out:
        pathlib.Path(a.out).mkdir(parents=True, exist_ok=True)
        (pathlib.Path(a.out) / "sample_cluster_b200.jsonl").write_text("".join(json.dumps(r) + "\n" for r in lines))


if __name__ == "__main__":
    main()
