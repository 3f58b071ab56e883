"""Cost of the entropy bonus at the benchmark's size: B = 4096 captions, 20 columns (S = 19 sampled steps), one GPU.

Two engines on the same seeded weights (icrl_b200.synth, vocabulary 1004) and inputs, one with entropy_coef = 0 (the
reference's loss: today's kernels) and one with entropy_coef = 0.01, step in alternation: after the warm-up (every
shape loaded, the chain warm-ups settled) `--rounds` rounds of `--steps` checked steps each.  Step time = CUDA events
around one step, which ends in the device-to-host read of its check words.  The weights do not change (no optimizer
step), so every step does the same work.

Then the two new kernels alone, CUDA events around each of `--reps` launches on the engine's own buffers:
icrl_policy_entropy on the logits stash (S*B*V*4 = 312 MB: more than the 126 MB L2) and icrl_softmax_entropy_bwd on a
fresh copy of the logits at the backward's row stride (the copy lies outside the timed pair).  And a torch.profiler
run of two steps of each engine (separate from the timing) gives every kernel's device time, so the dL/dlogits pass
with and without the entropy term can be compared.  Prints one JSON object (card name and power limit included):

    python scripts/entropy_cost.py --out profiles/r05_entropy.json
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

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
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--coef", type=float, default=0.01)
    ap.add_argument("--warmup", type=int, default=6)
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--steps", type=int, default=4, help="timed steps per engine and round")
    ap.add_argument("--reps", type=int, default=50, help="timed launches of each new kernel")
    ap.add_argument("--out", default=None, help="also write the JSON object to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("entropy_cost needs a CUDA device")
    import __graft_entry__ as ge
    ge.build()
    from icrl_b200 import _lib, synth
    from icrl_b200.engine import A2CEngine
    import icrl_b200.models as M

    dev = torch.device("cuda:0")
    w = synth.make_weights(100)
    w2i = synth.word_to_idx()
    P, Vn, R = M.PolicyNetwork(w2i), M.ValueNetwork(w2i), M.RewardNetwork(w2i)
    P.load_state_dict(w["policy"]); Vn.load_state_dict(w["value"]); R.load_state_dict(w["reward"])
    R.requires_grad_(False)
    R.train(False)
    A, R = M.AdvantageActorCriticNetwork(Vn, P).to(dev), R.to(dev)
    B, L = a.batch, 20
    f, c = synth.make_inputs(100, B, L)
    u = synth.make_uniforms(100, L - 1, B)
    engines = {"coef_0": A2CEngine(A, R), "coef_%g" % a.coef: A2CEngine(A, R, entropy_coef=a.coef)}
    preps = {k: e.prepare(f, c, u) for k, e in engines.items()}

    def step(k):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        res = engines[k].step(preps[k])
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), res

    last = {}
    for _ in range(a.warmup):
        for k in engines:
            _, last[k] = step(k)
    for _ in range(16):                      # until no chain warm-up changed in the last three steps
        settled = all(not e.segment_stats["warm_history"] or e.segment_stats["warm_history"][-1][0] + 3 < e.segment_stats["steps"]
                      for e in engines.values())
        if settled:
            break
        for k in engines:
            _, last[k] = step(k)
    times = {k: [] for k in engines}
    for _ in range(a.rounds):
        for k in engines:
            for _ in range(a.steps):
                ms, last[k] = step(k)
                times[k].append(ms)

    k0, k1 = list(engines)
    r0, r1 = last[k0], last[k1]
    same = {n: bool(torch.equal(r0[n], r1[n])) for n in ("tokens", "logp", "values", "rewards")}
    loss_gap = (r1.loss - r0.loss) + a.coef * r1.mean_entropy

    # the two new kernels alone, on the coefficient engine's buffers
    eng = engines[k1]
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    V, S = eng.V, r1["S"]
    logits = eng._bufs["p_logits"][:S * B * V]
    ent = torch.empty(B * S, device=dev)
    ldz = int(_lib.call("icrl_vocab_pad"))
    dz = torch.zeros(S * B, ldz, device=dev)
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    kern = {"policy_entropy": [], "softmax_entropy_bwd": []}
    for i in range(a.reps + 3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _lib.call("icrl_policy_entropy", st, B, S, V, p(logits), V, p(ent), None)
        e1.record()
        dz[:, :V].copy_(logits.view(S * B, V))
        e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e2.record()
        _lib.call("icrl_softmax_entropy_bwd", st, B, S, V, p(dz), ldz, p(r1["tokens"]), p(eng._bufs["dlogp"]), p(ent),
                  a.coef / (B * S), None)
        e3.record()
        torch.cuda.synchronize()
        if i >= 3:
            kern["policy_entropy"].append(e0.elapsed_time(e1) * 1e3)
            kern["softmax_entropy_bwd"].append(e2.elapsed_time(e3) * 1e3)

    # per-kernel device time of two steps of each engine (its own run: tracing slows the host)
    prof = {}
    for k in engines:
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as pr:
            for _ in range(2):
                step(k)
        ev = {}
        for e in pr.key_averages():
            t = getattr(e, "device_time_total", None)
            if t is None:
                t = e.cuda_time_total
            name = next((n for n in ("softmax_bwd_kernel", "policy_entropy_kernel", "a2c_loss_kernel") if n in e.key), None)
            if t and name:
                ev[name] = {"us_per_step": t / 2.0, "calls_per_step": e.count / 2.0}
        prof[k] = ev

    med = {k: float(np.median(v)) for k, v in times.items()}
    rounds = {k: [float(np.median(v[i * a.steps:(i + 1) * a.steps])) for i in range(a.rounds)] for k, v in times.items()}
    out = {"card": card(), "batch": B, "S": S, "vocab": V, "coef": a.coef, "timed_steps_each": len(times[k0]),
           "step_ms_median": med, "step_ms_min": {k: float(min(v)) for k, v in times.items()},
           "step_ms_max": {k: float(max(v)) for k, v in times.items()}, "round_medians_ms": rounds,
           "overhead_pct_of_median": 100.0 * (med[k1] - med[k0]) / med[k0],
           "kernel_us_median": {k: float(np.median(v)) for k, v in kern.items()},
           "kernel_us_min": {k: float(min(v)) for k, v in kern.items()},
           "entropy_pass_bytes": S * B * V * 4,
           "entropy_pass_GBps": S * B * V * 4 / (float(np.median(kern["policy_entropy"])) * 1e-6) / 1e9,
           "profiler_kernels": prof, "outputs_identical": same, "loss_minus_expected": loss_gap,
           "mean_entropy": r1.mean_entropy,
           "reruns": {k: e.segment_stats["reruns"] for k, e in engines.items()},
           "fallbacks": {k: e.segment_stats["fallbacks"] for k, e in engines.items()}}
    s = json.dumps(out, indent=1)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(s + "\n")


if __name__ == "__main__":
    main()
