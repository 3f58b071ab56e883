"""Per-minibatch time of train_policy_network on its two routes: the fused engine (engine.PolicyPretrainEngine +
optim.FlatAdam, the unidirectional default) and the module route (trainers._train_policy_modules: the drop-in modules'
autograd, one CrossEntropyLoss per row, torch.optim.Adam), at B = 512 (the reference's default) and B = 4096, L = 17.

Both routes run the public loop on the same seeded weights (icrl_b200.synth, vocabulary 1004) and the same dataset of
synthetic captions: <START>, words, <END> at a column drawn per row from 1..L-1, <NULL> after it.  The dataset holds
warm-up + timed + 1 full minibatches; torch.manual_seed gives both routes the same torch.randperm draw, so their first
minibatch is the same rows and its loss is compared.  SummaryWriter.add_scalar, which the loop calls once per minibatch
with the loss, is replaced by a recorder that synchronises the device and reads a host clock: the interval between two
calls is one whole minibatch of the loop (the previous optimizer step, the minibatch draw, forward, loss, backward, the
loss read).  The first `--warmup` intervals are dropped; the median and the spread of the next `--timed` are reported.
Checkpoint writes (torch.save on every new best loss, which is nearly every minibatch while the loss falls) are disk
time, the same in both routes, and are replaced by a counter here.

Prints one JSON object (card name and power limit included) and, with --out PREFIX, writes PREFIX.json and PREFIX.md:

    python scripts/pretrain_policy_bench.py --out profiles/r06_pretrain_policy
"""
import argparse
import json
import os
import statistics
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


def dataset(seed, N, L):
    from icrl_b200 import synth
    rs = np.random.RandomState(seed)
    caps = rs.randint(4, synth.VOCAB, size=(N, L)).astype(np.int64)
    caps[:, 0] = synth.START
    ends = rs.randint(1, L, size=N)
    for i, e in enumerate(ends):
        caps[i, e] = synth.END
        caps[i, e + 1:] = 0
    feats = rs.standard_normal((N, 512)).astype(np.float32)
    return {"train_captions": caps, "train_image_idxs": np.arange(N), "train_features": feats,
            "train_urls": np.array(["u"] * N), "word_to_idx": synth.word_to_idx(), "embeddings": None}


def run_route(route, B, L, warmup, timed, seed):
    import icrl_b200.models as M
    import icrl_b200.trainers as T
    from icrl_b200 import synth
    w = synth.make_weights(seed)
    data = dataset(seed, (warmup + timed + 1) * B, L)
    stamps, losses, saves = [], [], [0]

    class Rec:
        def __init__(self, *a, **k):
            pass

        def add_scalar(self, tag, val, step):
            torch.cuda.synchronize()
            stamps.append(time.perf_counter())
            losses.append(float(val.detach()) if torch.is_tensor(val) else float(val))

    def make(*a, **k):
        net = M.PolicyNetwork(*a, **k)
        net.load_state_dict(w["policy"])
        return net

    def no_save(*a, **k):
        saves[0] += 1

    patched = {"PolicyNetwork": T.PolicyNetwork, "SummaryWriter": T.SummaryWriter}
    real_save = torch.save
    T.PolicyNetwork, T.SummaryWriter, torch.save = make, Rec, no_save
    try:
        torch.manual_seed(seed)
        paths = {"policy_network": os.devnull}
        if route == "fused":
            T.train_policy_network(data, paths, "/nonexistent", False, epochs=1, batch_size=B)
        else:
            net = make(data["word_to_idx"]).to(M.device)
            T._train_policy_modules(net, data, paths, Rec(), 1, B)
    finally:
        T.PolicyNetwork, T.SummaryWriter, torch.save = patched["PolicyNetwork"], patched["SummaryWriter"], real_save
    dt = np.diff(np.array(stamps))[warmup:warmup + timed] * 1e3
    return {"median_ms": float(statistics.median(dt)), "min_ms": float(dt.min()), "max_ms": float(dt.max()),
            "minibatches_timed": int(dt.size), "first_loss": losses[0], "last_loss": losses[-1], "checkpoint_calls": saves[0]}


def markdown(res):
    lines = ["# Policy pretraining: fused engine against the module route", "",
             "`scripts/pretrain_policy_bench.py`, one run on %s (name, power limit, max SM clock)." % res["card"], "",
             "Per-minibatch time of `train_policy_network` (median of %d minibatches after %d warm-up ones; each window ends "
             "with a device synchronise; checkpoint writes left out), L = %d, vocabulary 1004, synthetic captions with "
             "<END> at a random column." % (res["timed"], res["warmup"], res["L"]), "",
             "| B | route | median ms | min ms | max ms | speed-up | loss on the shared first minibatch |",
             "|---|---|---|---|---|---|---|"]
    for B, r in res["batches"].items():
        for route in ("modules", "fused"):
            x = r[route]
            sp = "%.1fx" % (r["modules"]["median_ms"] / x["median_ms"]) if route == "fused" else ""
            lines.append("| %s | %s | %.2f | %.2f | %.2f | %s | %.8f |" % (B, route, x["median_ms"], x["min_ms"], x["max_ms"],
                                                                        sp, x["first_loss"]))
        lines.append("")
        lines.append("B = %s: the two routes' losses on the shared minibatch differ by %.2e relative." % (B, r["loss_rel_diff"]))
        lines.append("")
    return "\n".join(lines).rstrip() + "\n"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="512,4096")
    ap.add_argument("--L", type=int, default=17)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--timed", type=int, default=20)
    ap.add_argument("--seed", type=int, default=60)
    ap.add_argument("--out", default=None, help="write PREFIX.json and PREFIX.md")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("pretrain_policy_bench needs a CUDA device")
    import __graft_entry__ as ge
    ge.build()
    res = {"card": card(), "L": a.L, "warmup": a.warmup, "timed": a.timed, "batches": {}}
    for B in [int(x) for x in a.batches.split(",")]:
        r = {route: run_route(route, B, a.L, a.warmup, a.timed, a.seed) for route in ("modules", "fused")}
        r["speedup"] = r["modules"]["median_ms"] / r["fused"]["median_ms"]
        r["loss_rel_diff"] = abs(r["fused"]["first_loss"] - r["modules"]["first_loss"]) / abs(r["modules"]["first_loss"])
        res["batches"][str(B)] = r
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out + ".json", "w") as fh:
            json.dump(res, fh, indent=1)
        with open(a.out + ".md", "w") as fh:
            fh.write(markdown(res))


if __name__ == "__main__":
    main()
