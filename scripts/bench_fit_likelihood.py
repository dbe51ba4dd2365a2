"""Measures fit_likelihood with B200Gibbs (csrc/likelihood.cu, the PERSIST mode of csrc/mcmc_sampler.cu) on the C2 (N = 100,
10 x 10 lattice, J = +-0.4) and C3 (N = 1000, random 4-regular, J = +-0.4) models of bench.py.  Reads the card's name,
power limit and max SM clock in the same call, then prints one JSON line per measurement (and writes them to
DIR/fit_likelihood_b200.jsonl with --out DIR).

  fit       data: sample(gm, M, B200Gibbs(seed=1)) (C2 M = 1e6, C3 M = 2e5); start: gm's keys at weight 0.  One fit of
            `steps` steps with B200Gibbs(thin=1) and the default chains (2^17), burn_in (200) and step size: call time from
            CUDA events after a warm-up fit of 20 steps; per_step_ms = call_ms / steps (burn-in and set-up included).
            The final moment residual max_t |m^_t - m_t| comes from an
            independent moments(fit, B200Gibbs(seed=2, thin=1), 1e6) call; coupling_error is max |w - w*| over the pairs.
  fresh     the same gradient loop built from one fresh-chain moments(gm, B200Gibbs(thin=1), 2^17) call per step (200
            burn-in sweeps every step) and a host update, for `fresh_steps` steps only: its per-step time against the
            persistent fit's.
  eta       the final moment residual and coupling error at C2 for step sizes 0.05, 0.1, 0.2 and 0.4 (the default's
            measurement).

    python scripts/bench_fit_likelihood.py [--parts fit,fresh,eta] [--steps 2000] [--out DIR]
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
from bench_sample_mcmc import card  # noqa: E402
from gml_b200 import B200Gibbs, FactorGraph  # noqa: E402


def timed_once(fn):
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    out = fn()
    t1.record()
    torch.cuda.synchronize()
    return out, t0.elapsed_time(t1)


def setup(config):
    truth = c2_model() if config == "C2" else c3_model(1000)[3]
    gm = FactorGraph.from_matrix(truth)
    M = 1_000_000 if config == "C2" else 200_000
    data = gml_b200.sample(gm, M, 1, B200Gibbs(seed=1)).astype(np.int8)
    start = FactorGraph(2, gm.varible_count, "spin", {k: 0.0 for k in gm.terms})
    return truth, gm, data, start


def quality(fg, truth, dm):
    m = np.array(list(gml_b200.moments(fg, B200Gibbs(seed=2, thin=1), 1_000_000)[0].terms.values()))
    coup = max(abs(v - truth[k[0] - 1, k[1] - 1]) for k, v in fg.terms.items() if len(k) == 2)
    return float(np.abs(m - dm).max()), float(coup)


def part_fit(emit, steps, fresh_steps, etas, parts):
    for config in ("C2", "C3"):
        truth, gm, data, start = setup(config)
        if "fit" in parts:
            gml_b200.fit_likelihood(start, data, B200Gibbs(thin=1), steps=20)                # warm-up
            (fg, info), ms = timed_once(lambda: gml_b200.fit_likelihood(start, data, B200Gibbs(thin=1), steps=steps,
                                                                        return_info=True))
            dm = np.array(info["data_moments"])
            res, coup = quality(fg, truth, dm)
            trace = np.array(info["trace"])
            emit({"part": "fit", "model": config, "N": gm.varible_count, "terms": len(gm.terms), "rows": len(data),
                  "steps": steps, "thin": 1, "chains": 1 << 17, "call_ms": ms, "per_step_ms": ms / steps,
                  "moment_residual": res, "coupling_error": coup, "model_moment_residual": float(np.abs(np.array(info["model_moments"]) - dm).max()),
                  "trace_first10": float(trace[:steps // 10].mean()), "trace_last10": float(trace[-steps // 10:].mean())})
        if "fresh" in parts:
            dm = np.array(list(gml_b200.empirical_moments(data, list(gm.terms)).terms.values()))
            w = np.zeros(len(dm))
            keys = list(gm.terms)
            d = np.maximum(1 - dm * dm, 1e-2)

            def loop():
                nonlocal w
                for s in range(fresh_steps):
                    fg = FactorGraph(2, gm.varible_count, "spin", dict(zip(keys, w.tolist())))
                    m = np.array(list(gml_b200.moments(fg, B200Gibbs(seed=s, thin=1), 1 << 17)[0].terms.values()))
                    w = w + 0.1 * (1 + s / 100) ** -0.6 * (dm - m) / d
            loop()
            w = np.zeros(len(dm))
            _, ms = timed_once(loop)
            emit({"part": "fresh", "model": config, "steps": fresh_steps, "per_step_ms": ms / fresh_steps})
        if "eta" in parts and config == "C2":
            for eta in etas:
                fg, info = gml_b200.fit_likelihood(start, data, B200Gibbs(thin=1), steps=steps, step_size=eta, return_info=True)
                res, coup = quality(fg, truth, np.array(info["data_moments"]))
                emit({"part": "eta", "model": config, "step_size": eta, "steps": steps, "moment_residual": res,
                      "coupling_error": coup})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parts", default="fit,fresh,eta")
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--fresh-steps", type=int, default=20)
    ap.add_argument("--out", default="", help="directory for fit_likelihood_b200.jsonl (default: print only)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    gpu = card()
    print(gpu, flush=True)
    lines = []

    def emit(rec):
        lines.append(json.dumps({"card": gpu, **rec}))
        print(lines[-1], flush=True)
    part_fit(emit, args.steps, args.fresh_steps, (0.05, 0.1, 0.2, 0.4), args.parts.split(","))
    if args.out:
        pathlib.Path(args.out).mkdir(parents=True, exist_ok=True)
        (pathlib.Path(args.out) / "fit_likelihood_b200.jsonl").write_text("".join(l + "\n" for l in lines))


if __name__ == "__main__":
    main()
