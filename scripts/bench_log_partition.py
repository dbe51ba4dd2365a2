"""Measures the partition-function estimator (log_partition with B200Tempering, csrc/mcmc_sampler.cu with BRIDGE) and
the B200Tempering sampler that shares its kernel.  Prints the card's name, power limit and max SM clock first, then one
JSON line per run.

  estimate  log_partition at its defaults (32 rungs evenly spaced from 1 to 0, 4096 ladders, burn_in 200, 1000 sweeps)
            on the closed-form cases of tests/test_gpu_log_partition.py -- fields at N = 4096, periodic rings N = 1000
            J = 1 and N = 4096 J = 0.5, Curie-Weiss N = 256 at J = 0.5 and 1.5 -- and on 8 x 8 and 32 x 32 open J = 1
            ferromagnets: log Z, stderr, error against the exact value where there is one, swap rates and call time.
  tempering B200Tempering sampling (gml_b200_sample_tempering_device, default ladder and settings) at C2 (N = 100, 1e6
            draws) and on the 8 x 8 J = 1 ferromagnet (1024 ladders, 40 records each), this build against the build at
            --compare-lib, each in a child process of its own, alternating, --repeats times each.

Call time: CUDA events around a whole call after a warm-up call (estimate: a warm-up of 5 sweeps).

    python scripts/bench_log_partition.py [--parts estimate,tempering] [--compare-lib PATH] [--repeats 3] [--out DIR]
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
from bench import c2_model  # noqa: E402
from bench_sample_mcmc import card  # noqa: E402
from bench_sample_tempering import open_ferromagnet, timed  # noqa: E402
from gml_b200 import B200Tempering, FactorGraph, _lib  # noqa: E402


def cases():
    """(name, model, exact log Z or None)"""
    from test_gpu_log_partition import curie_weiss, curie_weiss_log_z, log_2cosh, ring
    h = np.random.default_rng(1).integers(-64, 65, 4096) / 64.0
    yield "fields N=4096", FactorGraph(1, 4096, "spin", {(i + 1,): float(v) for i, v in enumerate(h)}), float(log_2cosh(h).sum())
    for n, J in ((1000, 1.0), (4096, 0.5)):
        yield f"ring N={n} J={J}", ring(n, J), float(n * log_2cosh(J) + np.log1p(np.tanh(J) ** n))
    for J in (0.5, 1.5):
        yield f"Curie-Weiss N=256 J={J}", curie_weiss(256, J), curie_weiss_log_z(256, J)
    for side in (8, 32):
        yield f"open ferromagnet {side}x{side} J=1", open_ferromagnet(side, side, 1.0), None


def part_estimate():
    for name, gm, exact in cases():
        sampler = B200Tempering(seed=1)
        (log_z, err, info), ms = timed(lambda: gml_b200.log_partition(gm, sampler, return_info=True),
                                       lambda: gml_b200.log_partition(gm, sampler, 5))
        rec = {"part": "estimate", "model": name, "N": gm.varible_count, "terms": len(gm.terms), "ladders": info["ladders"],
               "rungs": len(info["betas"]), "burn_in": sampler.burn_in, "sweeps": info["sweeps"], "log_z": log_z,
               "stderr": err, "exact": exact, "error": None if exact is None else log_z - exact,
               "min_swap_rate": round(min(info["swap_rate"]), 4), "max_pair_stderr": max(info["log_ratio_stderr"]),
               "call_ms": round(ms, 2)}
        yield rec


def tempering_times(lib_path):
    """B200Tempering call times at C2 and on the 8 x 8 ferromagnet through gml_b200_sample_tempering_device of the library at
    lib_path (bound here, so a build without this change's symbols works too), into device buffers."""
    c = ctypes
    lib = c.CDLL(lib_path)
    lib.gml_b200_sample_tempering_device.argtypes = [c.c_int32, c.c_int32, c.c_int32, c.c_int32, c.c_void_p, c.c_void_p,
                                                     c.c_int32, c.c_void_p, c.c_int64, c.c_int32, c.c_int64, c.c_int32,
                                                     c.c_int32, c.c_uint64, c.c_void_p, c.c_void_p, c.c_void_p, c.c_void_p,
                                                     c.c_void_p, c.c_int64, c.c_void_p]
    runs = {"c2": (FactorGraph.from_matrix(c2_model()), 1_000_000, 0),
            "ferro8x8": (open_ferromagnet(8, 8, 1.0), 40 * 1024, 1024)}
    out = {}
    for name, (gm, draws, chains) in runs.items():
        order, idx, wts = gml_b200.api._term_arrays(gm)
        N = gm.varible_count
        ld = min(draws, 1 << N)
        counts = torch.empty(ld, dtype=torch.float64, device="cuda:0")
        spins = torch.empty((N, ld), dtype=torch.int8, device="cuda:0")
        K, rhat, swap = np.zeros(1, dtype=np.int64), np.zeros(2), np.zeros(_lib.TEMPERING_DEFAULT_RUNGS - 1)
        s = B200Tempering(seed=1, chains=chains)

        def call():
            rc = lib.gml_b200_sample_tempering_device(0, N, order, len(gm.terms), idx.ctypes.data, wts.ctypes.data, 0, None,
                                                      draws, 1, s.chains, s.burn_in, s.thin, s.seed, K.ctypes.data,
                                                      rhat.ctypes.data, swap.ctypes.data, counts.data_ptr(), spins.data_ptr(),
                                                      ld, None)
            assert rc == 0, rc

        _, ms = timed(call)
        out[name] = round(ms, 2)
        del counts, spins
        torch.cuda.empty_cache()
    return out


def part_tempering(compare_lib, repeats):
    libs = [("this", str(_lib.LIB_PATH)), ("compare", compare_lib)]
    for rep in range(repeats):
        for tag, path in libs:
            res = subprocess.run([sys.executable, __file__, "--tempering-child", path], capture_output=True, text=True,
                                 check=True)
            yield {"part": "tempering", "library": tag, "path": pathlib.Path(path).name, "repeat": rep,
                   **json.loads(res.stdout.strip().splitlines()[-1])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parts", default="estimate,tempering")
    ap.add_argument("--compare-lib", default="")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--tempering-child", default="", help="(internal) time B200Tempering with the library at this path")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    if a.tempering_child:
        print(json.dumps(tempering_times(a.tempering_child)))
        return
    gpu = card()
    print(f"card: {gpu}  library: {_lib.LIB_PATH.name}", flush=True)
    parts = a.parts.split(",")
    gens = [part_estimate()] if "estimate" in parts else []
    if "tempering" in parts:
        if not a.compare_lib:
            raise SystemExit("the tempering part needs --compare-lib")
        gens.append(part_tempering(a.compare_lib, a.repeats))
    lines = []
    for gen in gens:
        for rec in gen:
            rec["card"] = gpu
            print(json.dumps(rec), flush=True)
            lines.append(rec)
    if a.out:
        pathlib.Path(a.out).mkdir(parents=True, exist_ok=True)
        (pathlib.Path(a.out) / "bench_log_partition.jsonl").write_text("".join(json.dumps(r) + "\n" for r in lines))


if __name__ == "__main__":
    main()
