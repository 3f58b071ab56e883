"""Look-ahead decoder throughput: GenerateCaptionsWithActorCriticLookAhead (beam 5, 16 steps) on the fused engine
(engine.LookAheadEngine) against the reference's loop on the drop-in modules (trainers._look_ahead_modules).

Seeded synthetic weights (oracle.synth, vocabulary 1004) and features; the two paths alternate, `--runs` timed calls each per
batch size after one warm-up call of each, every call from a reset value state.  Captions/s = B / wall time of one call
(host clock around a call that ends in a device synchronise).  Also checks that the five candidates are identical and
reports the largest score difference.  Prints one JSON object and, with --out, writes it to that file:

    python scripts/lookahead_bench.py --batches 128 1024 --runs 3 --out profiles/r04_lookahead.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, nargs="+", default=[128, 1024])
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--seed", type=int, default=11)
    ap.add_argument("--out", default=None, help="also write the JSON object to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("lookahead_bench needs a CUDA device")
    import __graft_entry__ as ge
    ge.build()
    import icrl_b200.trainers as T
    from oracle import synth
    from tests.helpers import make_nets

    A, _, _ = make_nets(a.seed)
    P, Vn = A.policy_network, A.value_network
    paths = {"fused": T.GenerateCaptionsWithActorCriticLookAhead, "modules": T._look_ahead_modules}

    def call(name, f, c):
        Vn.valrnn.init_hidden()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        beams = paths[name](f, c, P, Vn)
        torch.cuda.synchronize()
        return time.perf_counter() - t0, beams

    out = {"card": card(), "seed": a.seed, "beam": 5, "steps": 16, "vocab": synth.VOCAB, "runs": a.runs, "results": {}}
    for B in a.batches:
        f, c = synth.make_inputs(a.seed, B, 17)
        beams = {}
        for name in paths:                                  # warm-up: module loads, workspaces, the chain's warm-up size
            _, beams[name] = call(name, f, c)
        times = {name: [] for name in paths}
        for _ in range(a.runs):
            for name in paths:
                dt, _ = call(name, f, c)
                times[name].append(dt)
        same = all(torch.equal(x[0].cpu(), y[0].cpu()) for x, y in zip(beams["fused"], beams["modules"]))
        err = 0.0
        for (_, s1), (_, s2) in zip(beams["fused"], beams["modules"]):
            d = (s1 - s2).abs()
            d = d[~torch.isnan(d)]
            err = max(err, float(d.max()) if d.numel() else 0.0)
        eng = P._icrl_lookahead
        r = {name: {"seconds": ts, "captions_per_s": [B / t for t in ts]} for name, ts in times.items()}
        r.update(candidates_identical=bool(same), max_score_diff=err,
                 speedup_median=float(np.median(times["modules"]) / np.median(times["fused"])),
                 fused_step_paths=list(eng.step_paths[-16:]), fused_fallbacks=eng.segment_stats["fallbacks"],
                 fused_warm_v=eng.warm["v"])
        out["results"][str(B)] = r
        print(B, json.dumps(r), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(out, fh, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
