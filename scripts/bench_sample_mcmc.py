"""Times the multi-sample Gibbs sampler (sample_device with B200Gibbs, csrc/mcmc_sampler.cu) on the C2 (10 x 10 lattice,
N = 100, 1e6 draws) and C3 (N = 1000, 1e7 draws) models of bench.py, against the one-draw-per-chain sampler that bench.py
uses for its input (gml_b200_sample_gibbs_device), in one process.

Per config and thin in {1, 2, 5, 10} at the default burn_in: the whole sample_device call (CUDA events, after a warm-up
call), site updates per second, per seed (--seeds) the max error of the RISE couplings and fields learned from the sample against the truth,
and the split-R-hat (energy, magnetisation).  The baseline runs bench.py's settings (C3: 40 sweeps, seed 1000; C2: 60
sweeps, seed 100 as in test_gpu_fullsize).  Prints the card's name and power limit first, then one JSON line per run.

    python scripts/bench_sample_mcmc.py [--configs c2,c3] [--thins 1,2,5,10] [--seeds 1,2,3] [--calls-only] [--out DIR]

--calls-only times the default setting only (no learn, no baseline): with GML_B200_LIB_PATH pointing at a build made with
`build.py -DGML_MCMC_NO_ENERGY --suffix=_noenergy`, it gives the call time without the energy pass of the R-hat diagnostic.
"""
import argparse
import ctypes
import json
import pathlib
import subprocess
import sys

ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import gml_b200  # noqa: E402
from bench import c2_model, c3_model, csr_of  # noqa: E402
from gml_b200 import _lib  # noqa: E402

CONFIGS = {"c2": (lambda: c2_model(), 1_000_000, 60, 100), "c3": (lambda: c3_model(1000)[3], 10_000_000, 40, 1000)}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def timed(fn):
    fn()                                                                      # warm-up: module load, pool growth
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    out = fn()
    t1.record()
    torch.cuda.synchronize()
    return out, t0.elapsed_time(t1)


def learned_error(truth, counts, spins):
    n = truth.shape[0]
    sess = gml_b200.Session(0).attach_device(counts.data_ptr(), spins.data_ptr(), counts.numel(), n, spins.stride(0))
    theta = sess.solve_pairwise(gml_b200.RISE(0.4, False), gml_b200.B200())
    sess.close()
    off = theta - np.diag(np.diag(theta))
    return float(np.abs(off - truth).max()), float(np.abs(np.diag(theta)).max())


def run_mcmc(name, truth, draws, thin, learn, seed=1):
    gm = gml_b200.FactorGraph.from_matrix(truth)
    sampler = gml_b200.B200Gibbs(seed=seed, thin=thin)
    (counts, spins), ms = timed(lambda: gml_b200.sample_device(gm, draws, sampler=sampler))
    chains = min(-(-draws // 32) * 32, 2 ** 17) if sampler.chains == 0 else sampler.chains
    updates = chains * truth.shape[0] * (sampler.burn_in + thin * -(-draws // chains))
    rec = {"config": name, "sampler": "B200Gibbs", "seed": seed, "burn_in": sampler.burn_in, "thin": thin, "chains": chains, "draws": draws,
           "call_ms": round(ms, 2), "site_updates": updates, "site_updates_per_s": updates / (ms / 1e3),
           "rhat_energy": sampler.last_rhat[0][0], "rhat_magnetisation": sampler.last_rhat[0][1]}
    if learn:
        rec["coupling_err"], rec["field_err"] = learned_error(truth, counts, spins)
    del counts, spins
    torch.cuda.empty_cache()
    return rec


def run_baseline(name, truth, draws, sweeps, seed):
    n = truth.shape[0]
    row_ptr, col, val = csr_of(truth)
    spins = torch.empty((n, draws), dtype=torch.int8, device="cuda:0")
    counts = torch.ones(draws, dtype=torch.float64, device="cuda:0")
    lib = _lib.load()

    def call():
        _lib.check(lib.gml_b200_sample_gibbs_device(0, n, row_ptr.ctypes.data, col.ctypes.data, val.ctypes.data, None, draws,
                                                    sweeps, seed, ctypes.c_void_p(spins.data_ptr()), draws, None))

    _, ms = timed(call)
    updates = draws * n * sweeps
    rec = {"config": name, "sampler": "gibbs_device (one draw per chain)", "sweeps": sweeps, "seed": seed, "draws": draws,
           "call_ms": round(ms, 2), "site_updates": updates, "site_updates_per_s": updates / (ms / 1e3)}
    rec["coupling_err"], rec["field_err"] = learned_error(truth, counts, spins)
    del counts, spins
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="c2,c3")
    ap.add_argument("--thins", default="1,2,5,10")
    ap.add_argument("--seeds", default="1", help="B200Gibbs seeds per thin: several give the spread of the learned error")
    ap.add_argument("--calls-only", action="store_true")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    gpu = card()
    print(f"card: {gpu}  library: {_lib.LIB_PATH.name}", flush=True)
    lines = []
    for name in a.configs.split(","):
        model, draws, sweeps, seed = CONFIGS[name]
        truth = model()
        if a.calls_only:
            runs = [lambda: run_mcmc(name, truth, draws, gml_b200.B200Gibbs().thin, False)]
        else:
            runs = [lambda: run_baseline(name, truth, draws, sweeps, seed)]
            runs += [lambda t=t, sd=sd: run_mcmc(name, truth, draws, t, True, sd) for t in map(int, a.thins.split(","))
                     for sd in map(int, a.seeds.split(","))]
        for run in runs:
            rec = {**run(), "card": gpu, "library": _lib.LIB_PATH.name}
            print(json.dumps(rec), flush=True)
            lines.append(rec)
    if a.out:
        pathlib.Path(a.out).mkdir(parents=True, exist_ok=True)
        suffix = "_calls" if a.calls_only else ""
        (pathlib.Path(a.out) / f"bench_sample_mcmc{suffix}_{_lib.LIB_PATH.stem}.jsonl").write_text(
            "".join(json.dumps(r) + "\n" for r in lines))


if __name__ == "__main__":
    main()
