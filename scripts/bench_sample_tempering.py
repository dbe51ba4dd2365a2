"""Measures the replica-exchange sampler (sample_device with B200Tempering, csrc/mcmc_sampler.cu with R > 1 rungs) against
B200Gibbs, in one process.  Prints the card's name, power limit and max SM clock first, then one JSON line per run.

  hard   4 x 5 open ferromagnet, J = 1.5, field 0.05 (N = 20), 32 replicates of 2e5 draws: max |t| of the magnetisations
         and pair correlations against enumeration (threshold at family-wise rate 1e-6), and call time.
  ferro  8 x 8 and 32 x 32 open J = 1 ferromagnets, 1024 chains of 40 records at the defaults: the default ladder, a
         32-rung ladder (geometric from 1 to 0.1) and B200Gibbs: R-hat (energy, magnetisation), swap rates, call time.
  learn  C2 (N = 100, 1e6 draws) and C3 (N = 1000, 1e7 draws) of bench.py at the defaults: call time and the max error of
         the RISE couplings learned from the sample.
  gibbs  B200Gibbs (gml_b200_sample_mcmc_device) at C2 and C3, this build against the build at --compare-lib, each in a
         child process of its own, alternating, --repeats times each.

Call time: CUDA events around a whole sample_device call after a warm-up call (C3 B200Tempering: a warm-up of a tenth of
the draws).

    python scripts/bench_sample_tempering.py [--parts hard,ferro,learn,gibbs] [--compare-lib PATH] [--repeats 3] [--out DIR]
"""
import argparse
import ctypes
import json
import pathlib
import subprocess
import sys

ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "scripts"))
sys.path.insert(0, str(ROOT / "tests"))
sys.path.insert(0, str(ROOT / "oracle"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import gml_b200  # noqa: E402
from bench import c2_model, c3_model  # noqa: E402
from bench_sample_mcmc import card, learned_error  # noqa: E402
from gml_b200 import B200Gibbs, B200Tempering, FactorGraph, _lib  # noqa: E402

LEARN = {"c2": (lambda: c2_model(), 1_000_000), "c3": (lambda: c3_model(1000)[3], 10_000_000)}
LADDER_32 = np.geomspace(1.0, 0.1, 32).tolist()


def timed(fn, warm=None):
    (warm or fn)()                                                            # warm-up: module load, pool growth
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    out = fn()
    t1.record()
    torch.cuda.synchronize()
    return out, t0.elapsed_time(t1)


def open_ferromagnet(rows, cols, J, h=0.0):
    m = np.zeros((rows * cols, rows * cols))
    for r in range(rows):
        for c in range(cols):
            i = r * cols + c
            m[i, i] = h
            for j in ([i + 1] if c + 1 < cols else []) + ([i + cols] if r + 1 < rows else []):
                m[i, j] = m[j, i] = J
    return FactorGraph.from_matrix(m)


def describe(sampler):
    if isinstance(sampler, B200Gibbs):
        return "B200Gibbs"
    return f"B200Tempering({'default' if sampler.betas is None else len(sampler.betas)} rungs)"


def part_hard():
    from test_gpu_tempering_sampler import moments_t
    gm = open_ferromagnet(4, 5, 1.5, 0.05)
    for sampler in (B200Gibbs(seed=7), B200Tempering(seed=7)):
        _, ms = timed(lambda: gml_b200.sample_device(gm, 200_000, 32, sampler))
        t, thr = moments_t(gm, sampler)
        yield {"part": "hard", "model": "4x5 J=1.5 h=0.05", "sampler": describe(sampler), "draws": 200_000, "replicates": 32,
               "call_ms": round(ms, 2), "max_t": round(float(t), 2), "threshold": round(float(thr), 2)}


def part_ferro():
    for side in (8, 32):
        gm = open_ferromagnet(side, side, 1.0)
        for sampler in (B200Gibbs(seed=5, chains=1024), B200Tempering(seed=5, chains=1024),
                        B200Tempering(seed=5, chains=1024, betas=LADDER_32)):
            _, ms = timed(lambda: gml_b200.sample_device(gm, 40 * 1024, sampler=sampler))
            rec = {"part": "ferro", "model": f"{side}x{side} J=1", "sampler": describe(sampler), "draws": 40 * 1024,
                   "chains": 1024, "call_ms": round(ms, 2), "rhat_energy": sampler.last_rhat[0][0],
                   "rhat_magnetisation": sampler.last_rhat[0][1]}
            if isinstance(sampler, B200Tempering):
                rec["swap_rate"] = [round(x, 3) for x in sampler.last_swap_rate[0]]
            yield rec


def part_learn():
    for name, (model, draws) in LEARN.items():
        truth = model()
        gm = FactorGraph.from_matrix(truth)
        for sampler in (B200Gibbs(seed=1), B200Tempering(seed=1)):
            warm = None
            if name == "c3" and isinstance(sampler, B200Tempering):
                warm = lambda: gml_b200.sample_device(gm, draws // 10, sampler=sampler)   # noqa: E731
            (counts, spins), ms = timed(lambda: gml_b200.sample_device(gm, draws, sampler=sampler), warm)
            rec = {"part": "learn", "config": name, "sampler": describe(sampler), "draws": draws, "call_ms": round(ms, 2),
                   "rhat_energy": sampler.last_rhat[0][0], "rhat_magnetisation": sampler.last_rhat[0][1]}
            rec["coupling_err"], rec["field_err"] = learned_error(truth, counts, spins)
            del counts, spins
            torch.cuda.empty_cache()
            yield rec


def gibbs_times(lib_path):
    """B200Gibbs call times at C2 and C3 through gml_b200_sample_mcmc_device of the library at lib_path (bound here, so a
    build without this change's symbols works too), into device buffers."""
    c = ctypes
    lib = c.CDLL(lib_path)
    lib.gml_b200_sample_mcmc_device.argtypes = [c.c_int32, c.c_int32, c.c_int32, c.c_int32, c.c_void_p, c.c_void_p,
                                                c.c_int64, c.c_int32, c.c_int64, c.c_int32, c.c_int32, c.c_uint64, c.c_void_p,
                                                c.c_void_p, c.c_void_p, c.c_void_p, c.c_int64, c.c_void_p]
    out = {}
    for name, (model, draws) in LEARN.items():
        gm = FactorGraph.from_matrix(model())
        order, idx, wts = gml_b200.api._term_arrays(gm)
        N = gm.varible_count
        counts = torch.empty(draws, dtype=torch.float64, device="cuda:0")
        spins = torch.empty((N, draws), dtype=torch.int8, device="cuda:0")
        K, rhat = np.zeros(1, dtype=np.int64), np.zeros(2)
        s = B200Gibbs(seed=1)

        def call():
            rc = lib.gml_b200_sample_mcmc_device(0, N, order, len(gm.terms), idx.ctypes.data, wts.ctypes.data, draws, 1, s.chains,
                                                 s.burn_in, s.thin, s.seed, K.ctypes.data, rhat.ctypes.data, counts.data_ptr(),
                                                 spins.data_ptr(), draws, None)
            assert rc == 0, rc

        _, ms = timed(call)
        out[name] = round(ms, 2)
        del counts, spins
        torch.cuda.empty_cache()
    return out


def part_gibbs(compare_lib, repeats):
    libs = [("this", str(_lib.LIB_PATH)), ("compare", compare_lib)]
    for rep in range(repeats):
        for tag, path in libs:
            res = subprocess.run([sys.executable, __file__, "--gibbs-child", path], capture_output=True, text=True, check=True)
            yield {"part": "gibbs", "library": tag, "path": pathlib.Path(path).name, "repeat": rep,
                   **json.loads(res.stdout.strip().splitlines()[-1])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parts", default="hard,ferro,learn,gibbs")
    ap.add_argument("--compare-lib", default="")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--gibbs-child", default="", help="(internal) time B200Gibbs with the library at this path")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    if a.gibbs_child:
        print(json.dumps(gibbs_times(a.gibbs_child)))
        return
    gpu = card()
    print(f"card: {gpu}  library: {_lib.LIB_PATH.name}", flush=True)
    lines = []
    parts = a.parts.split(",")
    runs = [("hard", part_hard), ("ferro", part_ferro), ("learn", part_learn)]
    gens = [fn() for p, fn in runs if p in parts]
    if "gibbs" in parts:
        if not a.compare_lib:
            raise SystemExit("the gibbs part needs --compare-lib")
        gens.append(part_gibbs(a.compare_lib, a.repeats))
    for gen in gens:
        for rec in gen:
            rec["card"] = gpu
            print(json.dumps(rec), flush=True)
            lines.append(rec)
    if a.out:
        pathlib.Path(a.out).mkdir(parents=True, exist_ok=True)
        (pathlib.Path(a.out) / "bench_sample_tempering.jsonl").write_text("".join(json.dumps(r) + "\n" for r in lines))


if __name__ == "__main__":
    main()
