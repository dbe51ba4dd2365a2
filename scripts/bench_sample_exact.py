"""Times the exact device sampler (gml_b200.sample_device, csrc/exact_sampler.cu) on random Ising models of N = 20..32 spins.

Per N: the device time of each phase (sum of its kernels in a torch.profiler run of one call), the wall time of a whole
call (CUDA events, after a warm-up call), enumerated configurations per second of the partition pass and of the whole call,
and, where the 2^N x N spin table fits in host memory (N <= 24), the time of the numpy enumeration of oracle.sample_exact.
Prints the card's name and power limit first; one JSON line per N.

    python scripts/bench_sample_exact.py [--sizes 20,24,28,32] [--draws 1000000] [--out DIR]
"""
import argparse
import json
import pathlib
import subprocess
import sys
import time

ROOT = pathlib.Path(__file__).resolve().parent.parent
for p in (ROOT, ROOT / "oracle", ROOT / "tests"):
    sys.path.insert(0, str(p))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import gml_b200  # noqa: E402
import gml_oracle as o  # noqa: E402
from helpers import random_ising  # noqa: E402

# kernel name fragment -> phase (numbered as in csrc/exact_sampler.cu)
PHASES = (("exact_partition_kernel", "1_partition"), ("max_kernel", "2_normalise"), ("rescale_kernel", "2_normalise"),
          ("tile_scan_kernel<double>", "2_normalise"), ("tile_add_kernel<double>", "2_normalise"),
          ("count_draws_kernel", "3_draw"), ("scatter_draws_kernel", "3_draw"), ("tile_scan_kernel<unsigned long long>", "3_draw"),
          ("tile_add_kernel<unsigned long long>", "3_draw"), ("exact_resolve_kernel", "4_resolve"), ("exact_emit_kernel", "4_resolve"))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def phase_ms(gm, draws, sampler):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        gml_b200.sample_device(gm, draws, sampler=sampler)
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        phase = next((ph for frag, ph in PHASES if frag in ev.key), None)
        if phase:
            out[phase] = out.get(phase, 0.0) + ev.device_time_total / 1e3
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="20,24,28,32")
    ap.add_argument("--draws", type=int, default=1_000_000)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    gpu = card()
    print(f"card: {gpu}", flush=True)
    lines = []
    for n in map(int, a.sizes.split(",")):
        gm = gml_b200.FactorGraph.from_matrix(random_ising(n, n))
        sampler = gml_b200.B200Exact(seed=1)
        gml_b200.sample_device(gm, a.draws, sampler=sampler)                    # warm-up: module load, pool growth
        torch.cuda.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        counts, _ = gml_b200.sample_device(gm, a.draws, sampler=sampler)
        t1.record()
        torch.cuda.synchronize()
        call_ms = t0.elapsed_time(t1)
        phases = phase_ms(gm, a.draws, sampler)
        rec = {"N": n, "n_terms": len(gm.terms), "draws": a.draws, "K": int(counts.numel()), "call_ms": round(call_ms, 3),
               "phase_ms": {k: round(v, 3) for k, v in sorted(phases.items())},
               "configs_per_s_partition": 2.0 ** n / (phases["1_partition"] / 1e3),
               "configs_per_s_call": 2.0 ** n / (call_ms / 1e3), "oracle_ms": None, "card": gpu}
        if n <= 24:
            t = time.perf_counter()
            o.sample_exact(gm.terms, n, a.draws, np.random.default_rng(1))
            rec["oracle_ms"] = round((time.perf_counter() - t) * 1e3, 1)
        print(json.dumps(rec), flush=True)
        lines.append(rec)
    if a.out:
        pathlib.Path(a.out).mkdir(parents=True, exist_ok=True)
        (pathlib.Path(a.out) / "bench_sample_exact.jsonl").write_text("".join(json.dumps(r) + "\n" for r in lines))


if __name__ == "__main__":
    main()
