#!/usr/bin/env python
"""A2C caption-training throughput on B200 (BASELINE.json metric) and the CPU reference arm.

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
  python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on host cores

Workload (config.workload): BASELINE.json configs[3] -- the full A2C training step (rollout +
embedding reward + value + loss + backward + gradient all-reduce + Adam), global batch 4096 captions,
max_len 20 (S = 19 sampled steps), rows sharded contiguously over the N ranks (strong scaling).
Synthetic data of that shape and random-init weights of the reference architecture (the
models_pretrained/*.pt blobs are absent from the reference checkout).

One JSON line on rank 0.  `value` = captions/s with the minibatch already in HBM; `e2e` = the same
step driven through the public API from pinned host buffers, including the H2D copies and the D2H
read of the loss.  Timing: CUDA events on the launching stream bracketed by barrier + synchronize,
max over ranks.  The working set per step (activation stash of the serial chains, GBs) is far larger
than the 126 MB L2, so no explicit L2 flush is needed between iterations.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H, L_CAP = 512, 20


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=4096, help="global batch (captions per step)")
    ap.add_argument("--cpu-sample", type=int, default=256, help="rows of the workload per sampled step on the host cores")
    ap.add_argument("--chain-shards", type=int, default=1, choices=[1, 2, 4, 8],
                    help="value/reward recurrences per rank (1 = the reference's single carried-state chain)")
    ap.add_argument("--chain-engine", default="tc", choices=["tc", "simt"],
                    help="tc = chain pieces on tcgen05 (chain_tc.cu, default); simt = CUDA-core segment kernels (chain.cu)")
    ap.add_argument("--chain-pieces", type=int, default=None, help="tc: cap on the lockstep pieces (default: co-resident clusters x 128)")
    ap.add_argument("--chain-segments", type=int, default=32, choices=[1, 2, 4, 8, 16, 32],
                    help="simt: lockstep pieces of the single carried-state chain (1 = serial kernels only, either engine)")
    ap.add_argument("--chain-warmup", type=int, default=256, help="first warm-up of every chain piece (the tc engine adapts it)")
    ap.add_argument("--torch-adam", action="store_true", help="torch.optim.Adam instead of the flat fused Adam kernel")
    ap.add_argument("--sharded-leg", action="store_true", help="also time 8 zero-state row shards per rank")
    ap.add_argument("--no-serial-leg", action="store_true", help="skip the serial-kernel leg (chain_segments = 1)")
    ap.add_argument("--no-extras", action="store_true", help="skip the config 3 (reward throughput) and config 5 (curriculum) objects")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


WORKLOAD = ("configs[3]: full A2C training step (rollout+reward+value+loss+backward+allreduce+Adam), "
            "global batch %d, max_len %d, S=%d")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.stamps, self.proc = index, [], [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            p = [x.strip() for x in line.split(",")]
            if len(p) >= 9 and p[0] == str(self.index):
                self.rows.append(p)
                self.stamps.append(time.time())

    def stop(self, t0=None, t1=None):
        """Samples taken inside [t0, t1] (the timed region).  nvidia-smi needs ~0.5 s to start, so the sampler is
        started before the warm-up steps; if the timed region is shorter than one sampling period the samples of the
        warm-up steps (the same kernels, the same load) are used and `window` says so."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        window = "timed region"
        if t0 is not None:
            inside = [r for r, ts in zip(self.rows, self.stamps) if t0 <= ts <= t1 + 0.05]
            if inside:
                self.rows = inside
            else:
                window = "warm-up + timed region (timed region shorter than the 200 ms sampling period)"
        sm = sorted(float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit())
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        mx = [float(r[2]) for r in self.rows if r[2].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows), "window": window}


def workload(batch):
    from icrl_b200 import synth       # seeded synthetic inputs (product-side helper; oracle/ is not touched here)
    f, c = synth.make_inputs(100, batch, L_CAP)
    u = synth.make_uniforms(100, L_CAP - 1, batch)
    return f, c, u


def make_nets(seed, dev):
    """Drop-in modules with random-init weights of the reference architecture (the .pt blobs are absent)."""
    import icrl_b200.models as M
    from icrl_b200 import synth
    w = synth.make_weights(seed)
    w2i = synth.word_to_idx()
    P, V, R = M.PolicyNetwork(w2i), M.ValueNetwork(w2i), M.RewardNetwork(w2i)
    P.load_state_dict(w["policy"])
    V.load_state_dict(w["value"])
    R.load_state_dict(w["reward"])
    R.requires_grad_(False)
    R.train(False)
    return M.AdvantageActorCriticNetwork(V, P).to(dev), R.to(dev)


DUMP_ROWS = 8192


def dump_outputs(out_dir, per_row, stats, grads):
    """What a caller of the timed training step receives from its last step, as float32 / float64 .npy files: the
    sampled token ids, their log-probabilities, the values and rewards (`per_row`: tokens / logp / values / rewards,
    rows x S), the loss, mean reward and mean advantage (`stats`), and every parameter's gradient (`grads`, written as
    grad.<name>).  The weights after the Adam update are left out: Adam's first step moves an entry by
    ~lr * g / (|g| + eps), so last-bit differences of a near-zero gradient (float atomics) become differences far above
    rounding in the weight, while the gradient itself shows them as what they are.  Batches above DUMP_ROWS rows keep a
    fixed, seeded sample of rows, listed in rows.npy, so that the files stay below 64 MB.  With several GPUs these are
    rank 0's rows."""
    os.makedirs(out_dir, exist_ok=True)
    B = int(per_row["tokens"].shape[0])
    rows = np.arange(B)
    if B > DUMP_ROWS:
        rows = np.sort(np.random.RandomState(0).choice(B, DUMP_ROWS, replace=False))
        np.save(os.path.join(out_dir, "rows.npy"), rows.astype(np.float64))
    out = {k: np.asarray(per_row[k], dtype=np.float32)[rows] for k in ("tokens", "logp", "values", "rewards")}
    out.update(loss=np.float64(stats[0]), mean_reward=np.float64(stats[1]), mean_advantage=np.float64(stats[2]))
    for name, g in grads.items():
        out["grad." + name] = np.asarray(g, dtype=np.float32)
    for name, arr in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), arr)


def cpu_reference(rows_per_step, warm_rows=64):
    """The reference algorithm as executed (oracle/ref_port: per-step prefix re-runs, batch-as-time RNN calls, numpy
    sampling, autograd backward, Adam) on all host cores.  `rows_per_step` lists the rows of each timed step (leading
    rows of the bench workload); one un-timed step of `warm_rows` rows comes first (thread pool, allocator, Adam state).
    Returns (captions/s over the timed steps, cores, [seconds per step], the last step's result)."""
    from oracle import ref_port        # the one place bench.py executes oracle/: the CPU reference being timed
    from icrl_b200 import synth
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    nets = ref_port.Nets(synth.make_weights(0))
    opt = torch.optim.Adam([p for _, p in nets.named_trainable()], lr=1e-4)
    f, c, u = workload(max(list(rows_per_step) + [warm_rows]))
    times = []
    for i, rows in enumerate([warm_rows] + list(rows_per_step)):
        t0 = time.perf_counter()
        res = ref_port.a2c_minibatch(nets, f[:rows], c[:rows], np.ascontiguousarray(u[:, :rows]))
        opt.step()
        if i > 0:
            times.append(time.perf_counter() - t0)
    return sum(rows_per_step) / sum(times), torch.get_num_threads(), times, res


def main_reference(args, rank):
    """Reference arm: rank 0 alone times the reference's CPU implementation of the path on the box's host cores.  The
    first timed step is the FULL workload (every row of the global batch: one carried-state chain over all of them, as
    the reference runs it); the remaining --steps - 1 steps are bounded samples (--cpu-sample leading rows; the cost is
    linear in rows) so that the run ends within minutes; value = rows processed / time over all timed steps."""
    if rank != 0:
        return
    sample = min(args.cpu_sample, args.batch)
    n_sample = args.steps - 1
    rows = [args.batch] + [sample] * n_sample
    cps, cores, times, res = cpu_reference(rows)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, res, (res["loss"], res["mean_reward"], res["mean_adv"]),
                     {k: g.numpy() for k, g in res["grads"].items()})
    desc = ("step 1: all %d captions of the workload (%.1f s); %d further steps of the first %d captions each (%.2f s "
            "mean); 1 un-timed warm-up step of 64 captions; value = captions processed / time over the timed steps" % (
                args.batch, times[0], n_sample, sample, (sum(times[1:]) / n_sample) if n_sample else 0.0))
    print(json.dumps({
        "impl": "reference", "metric": "A2C train captions/sec", "value": cps, "unit": "captions/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": times[0] * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD % (args.batch, L_CAP, L_CAP - 1), "global_batch": args.batch,
                   "steps_timed": len(rows), "full_size_step_s": times[0]},
        "cpu_baseline": {"value": cps, "unit": "captions/s", "cores": cores, "kind": "port", "sample": desc},
        "e2e": {"value": cps, "unit": "captions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# dram__bytes_read.sum + dram__bytes_write.sum per launch of the chain kernels from `ncu --set full` captures of THIS command
# (profiles/r02b_ncu.md); keyed by (kernel, local batch).  A configuration that was not captured reports null.
NCU_TRAFFIC = {("chains_tc_fwd_fused_kernel", 4096): 12.61e9, ("chain_tc_bwd_kernel", 4096): 23.96e9}


def roofline_of(phases, Bl, lay, peaks, clk):
    """Roofline of the dominant kernel of the step (the longest chain launch): tensor pipe.  `achieved` counts the
    ALGORITHMIC flops of the recurrent products once (2 x 512 x G per chain position, G = 2048 LSTM / 1536 GRU; the input
    half of the gates is the packed table): SURVEY 8(d) per-caption figures minus the tabled half.  The kernels execute
    3x that (fp16 hi/lo' split, fp32-grade) on the warm-up positions as well."""
    Tv, Tr = Bl * 190, Bl * 209
    fwd_ms, bwd_ms = phases.get("chains_fwd_fused", 0.0), phases.get("chain_lstm_bwd", 0.0)
    peak = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1400.0)))
    src = "measured (MEASURED_PEAKS.json bf16_tflops_sustained: the kernel is timed inside a long step)" if peaks else "fallback"
    if lay is None:
        return {"kernel": "serial chain kernels (chain.cu)", "bound": "latency", "achieved": None, "peak": peak, "unit": "TFLOP/s",
                "frac": None, "traffic": None, "note": "chains too short to cut or chain_segments=1: latency-bound serial walk"}
    (Pv, seg_v, warm_v), (Pr, seg_r, warm_r) = lay["v"], lay["r"]
    if bwd_ms >= fwd_ms:
        Pv, seg_v, warm_v = lay.get("b") or lay["v"]
        kname, kms = "chain_tc_bwd_kernel", bwd_ms
        alg = Tv * 2.0 * 2048 * 512
        executed = 3.0 * Pv * (seg_v + warm_v) * 2.0 * 2048 * 512
        steps = seg_v + warm_v
        hbm_bytes = Tv * (6 * H * 4 + 4 * H * 4 + 4)          # stash read (gates, c_t, c_{t-1}) + dgates write + take
    else:
        fused = bool(lay.get("fused"))
        kname = ("chains_tc_fwd_fused_kernel (value LSTM + reward GRU side by side, one launch)" if fused else
                 "chain_tc_fwd_kernel<4> + chain_tc_fwd_kernel<3> (value LSTM, reward GRU; two launches)")
        kms = fwd_ms
        alg = Tv * 2.0 * 512 * 2048 + Tr * 2.0 * 512 * 1536
        executed = 3.0 * (Pv * (seg_v + warm_v) * 2.0 * 512 * 2048 + Pr * (seg_r + warm_r) * 2.0 * 512 * 1536)
        steps = max(seg_v + warm_v, seg_r + warm_r) if fused else seg_v + warm_v + seg_r + warm_r
        hbm_bytes = Tv * (4 * H * 4 + 6 * H * 4 + 4) + Tr * (3 * H * 4 + H * 4 + 4)     # table row + stash (+ token)
    ach = alg / (kms * 1e-3) / 1e12 if kms > 0 else 0.0
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    hbm_ach = hbm_bytes / (kms * 1e-3) / 1e9 if kms > 0 else 0.0
    return {"kernel": kname, "bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
            "traffic": NCU_TRAFFIC.get((kname.split(" ")[0], Bl)), "peak_source": src, "ms_per_launch": kms,
            "executed_tflops": executed / (kms * 1e-3) / 1e12 if kms > 0 else 0.0,
            "frac_executed": executed / (kms * 1e-3) / 1e12 / peak if kms > 0 else 0.0,
            "kernel_steps_per_launch": steps, "us_per_kernel_step": kms * 1e3 / steps if steps else None,
            "pieces": {"value": Pv, "reward": Pr}, "warmup": {"value": warm_v, "reward": warm_r},
            "limited_by": "shared-memory bandwidth of the SM during the step GEMM (MMA operand reads + TMA fill at 128 B/clk: model "
                          "within 1 % of the measured cycles) and the number of global row segments gathered / stored in the "
                          "epilogue; the tensor pipe itself needs 12.3 K of a step's 31 K (forward) / 38 K (backward) cycles "
                          "(DESIGN.md 4.0)",
            "hbm": {"achieved": hbm_ach, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_ach / hbm_peak,
                    "note": "algorithmic stash / table bytes of the same launch against the measured copy bandwidth"},
            "note": "one kernel step = [pieces x 512] . W_hh^T on tcgen05 (M = 128 pieces per cluster of 8 CTAs) + cell "
                    "update; `achieved` = algorithmic recurrent flops of the live chain positions, counted once; "
                    "`executed` = x3 (fp16 hi/lo' split) including the discarded warm-up positions and padded rows"}


def main():
    args = parse()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        return main_reference(args, rank)

    import ctypes
    import torch.distributed as dist
    from icrl_b200 import _lib, synth
    from icrl_b200.dp import DataParallelA2C, shard_bounds
    from icrl_b200.engine import A2CEngine
    from icrl_b200.optim import FlatAdam

    torch.cuda.set_device(local)
    dev = "cuda:%d" % local
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(dev))
    A, R = make_nets(0, dev)
    eng = A2CEngine(A, R, chain_shards=args.chain_shards, chain_segments=args.chain_segments, chain_warmup=args.chain_warmup,
                    chain_engine=args.chain_engine, chain_pieces=args.chain_pieces)
    opt = torch.optim.Adam(A.parameters(), lr=1e-4) if args.torch_adam else FlatAdam(eng, lr=1e-4)
    dp = DataParallelA2C(eng, opt)
    B = args.batch
    S = L_CAP - 1
    f, c, u = workload(B)
    lo, hi = shard_bounds(B, rank, world)
    fl, cl, ul = f[lo:hi], c[lo:hi], np.ascontiguousarray(u[:, lo:hi])
    plan = (1, S)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def all_min(flag):
        t = torch.tensor([1 if flag else 0], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return int(t.item()) == 1

    def timed(run_step, steps, warmup, reset=None):
        """Mean ms per step over `steps` steps after `warmup` un-timed ones.  `reset`, if given, runs before every step
        and outside the timed intervals (each step is then timed by its own pair of events)."""
        for _ in range(warmup):
            if reset:
                reset()
            run_step()
        barrier()
        l0 = eng.launches.value
        if reset is None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                run_step()
            e1.record()
            barrier()
            ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        else:
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
            for e0, e1 in ev:
                reset()
                e0.record()
                run_step()
                e1.record()
            barrier()
            ms = torch.tensor([sum(e0.elapsed_time(e1) for e0, e1 in ev)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()) / steps, (eng.launches.value - l0) // steps

    def seg_counters():
        st = eng.segment_stats
        return {"fallbacks_to_serial": st["fallbacks"], "warmup_reruns": st["reruns"], "steps": st["steps"]}

    def seg_delta(c0):
        c1 = seg_counters()
        return {k: c1[k] - c0[k] for k in c0}

    def snapshot():
        st = {"warm": dict(eng.warm), "clean": dict(eng._clean), "hold": dict(eng._hold)}
        if args.torch_adam:
            import copy
            st["params"] = [p.detach().clone() for p in A.parameters()]
            st["opt"] = copy.deepcopy(opt.state_dict())
        else:
            st["flat"] = (opt.flat_param.clone(), opt.exp_avg.clone(), opt.exp_avg_sq.clone(), opt.t)
        return st

    def restore(st, chains=True):
        if chains:
            eng.warm, eng._clean, eng._hold = dict(st["warm"]), dict(st["clean"]), dict(st["hold"])
        if args.torch_adam:
            with torch.no_grad():
                for p, q in zip(A.parameters(), st["params"]):
                    p.copy_(q)
            opt.load_state_dict(st["opt"])
        else:
            opt.flat_param.copy_(st["flat"][0])
            opt.exp_avg.copy_(st["flat"][1])
            opt.exp_avg_sq.copy_(st["flat"][2])
            opt.t = st["flat"][3]

    # Every warm-up and timed step of the two legs starts from the seeded weights and a fresh optimizer state; only the
    # engine's chain warm-ups carry over from step to step.  A step that continued training would start from weights
    # that depend on the rounding of every earlier step's gradients (float atomics), which Adam turns into steps of ~lr
    # on near-zero entries: with the same arguments, the timed steps then compute the same thing from the same inputs
    # on every run.
    init = snapshot()

    def reset():
        restore(init, chains=False)

    # ---- warm-up: W (>= 3) steps, then up to 16 more checked steps while the engine is still re-sizing its chain warm-ups
    # (every step verified; the warm-up of each chain follows the measured contraction rate, engine._adapt_warm)
    prep = eng.prepare(fl, cl, ul, plan=plan)
    clocks = ClockSampler(local)
    clocks.start()
    n_warm = 0
    for _ in range(max(args.warmup, 3)):
        reset()
        dp.step(prep, global_rows=B)
        n_warm += 1
    for _ in range(16):
        settled = len(eng.segment_stats["warm_history"]) == 0 or \
            eng.segment_stats["warm_history"][-1][0] + 3 < eng.segment_stats["steps"]
        if all_min(settled):
            break
        reset()
        dp.step(prep, global_rows=B)
        n_warm += 1
    barrier()
    reset()
    state0 = snapshot()           # the seeded weights with the chain warm-ups the warm-up settled on

    # ---- leg 1: minibatch resident in HBM.  The steps run unchecked (no host read inside the timed region) and are
    # verified together afterwards (the joint-check words are running maxima); a failure re-times with a check per step.
    last = {}

    def step_hbm(check):
        last["res"] = dp.step(prep, global_rows=B, check=check)

    c0 = seg_counters()
    eng.phase_events = []
    t_wall0 = time.time()
    ms_step, launches = timed(lambda: step_hbm(False), args.steps, 0, reset)
    clk = clocks.stop(t_wall0, time.time())
    phases = {k: sum(v) / len(v) for k, v in eng.phase_times_ms().items()}
    eng.phase_events = None
    lay = eng.piece_layout if args.chain_engine == "tc" else None
    seg_layout = eng.segment_layout
    value_checked_per_step = False
    if not all_min(eng.segments_verified()):
        # some rank's joint check failed inside the unchecked loop: those steps are not the reference's numbers.
        # Time again with every step checked (re-runs with longer warm-ups included); every rank takes this branch.
        value_checked_per_step = True
        eng.phase_events = []
        ms_step, launches = timed(lambda: step_hbm(True), args.steps, 2, reset)
        phases = {k: sum(v) / len(v) for k, v in eng.phase_times_ms().items()}
        eng.phase_events = None
        lay = eng.piece_layout if args.chain_engine == "tc" else None
        seg_layout = eng.segment_layout
    value_seg = seg_delta(c0)
    if args.dump_outputs and rank == 0:
        res = last["res"]                                  # before the later legs overwrite the gradients
        dump_outputs(args.dump_outputs, {k: res[k].float().cpu().numpy() for k in ("tokens", "logp", "values", "rewards")},
                     res["stats"].double().cpu().numpy(), {k: p.grad.float().cpu().numpy() for k, p in A.named_parameters()})

    # ---- leg 2: end to end through the public API from pinned host buffers, every step checked, loss read on the host
    e2e = None
    if not args.no_e2e:
        fh = torch.from_numpy(fl).pin_memory()
        uh = torch.from_numpy(ul).pin_memory()
        sink = []

        def step_e2e():
            res = dp.step(fh, cl, uh, global_rows=B, plan=plan)
            sink.append(res.loss)                     # D2H read of the step's result (rides the joint-check read)

        restore(state0)
        c0 = seg_counters()
        ms_e2e, _ = timed(step_e2e, args.steps, 1, reset)   # one un-timed step: first touch of the pinned buffers
        e2e = {"value": B / (ms_e2e * 1e-3), "unit": "captions/s", "ms_per_step": ms_e2e,
               "h2d_bytes_per_step": int(fl.nbytes + (hi - lo) * 4 + ul.nbytes), "d2h_bytes_per_step": 80,
               "chain_checks": seg_delta(c0)}

    # ---- leg 3 (reported separately, never the headline): the serial chain kernels; 8 zero-state shards per rank
    sharded = None
    serial_leg = None
    if seg_layout is not None and not args.no_serial_leg:
        eng1 = A2CEngine(A, R, chain_segments=1)
        dp1 = DataParallelA2C(eng1, None)
        ms1, _ = timed(lambda: dp1.step(prep, global_rows=B, check=False), min(args.steps, 2), 1)
        _lib.call("icrl_chain_check", ctypes.c_void_p(torch.cuda.current_stream().cuda_stream),
                  ctypes.c_void_p(eng1.sync_state.data_ptr()))
        serial_leg = {"value": B / (ms1 * 1e-3), "unit": "captions/s", "ms_per_step": ms1, "steps": min(args.steps, 2),
                      "note": "the same step (without Adam) on the serial chain kernels (chain_segments=1): one CTA group walks "
                              "the whole carried-state chain position by position"}
        del eng1, dp1
        eng._attach_grads()
    if args.chain_shards == 1 and args.sharded_leg and (hi - lo) % 8 == 0:
        eng8 = A2CEngine(A, R, chain_shards=8, chain_segments=1)
        dp8 = DataParallelA2C(eng8, None)
        ms8, _ = timed(lambda: dp8.step(prep, global_rows=B, check=False), args.steps, 2)
        _lib.call("icrl_chain_check", ctypes.c_void_p(torch.cuda.current_stream().cuda_stream),
                  ctypes.c_void_p(eng8.sync_state.data_ptr()))
        sharded = {"chain_shards_per_rank": 8, "value": B / (ms8 * 1e-3), "unit": "captions/s", "ms_per_step": ms8,
                   "note": "value/reward recurrences restart from zero state every local_batch/8 rows and run in lockstep "
                           "(numerically = the reference on 8x%d row shards with averaged gradients, i.e. %d-rank data "
                           "parallel, SURVEY 8e); NOT the single carried-state chain of `value`" % (world, 8 * world)}
        del eng8, dp8
        eng._attach_grads()

    # ---- BASELINE configs 3 and 5 in the same run (side objects, not the headline)
    reward_tp, curriculum = None, None
    if not args.no_extras:
        restore(state0)
        # config 3: RewardNetwork embedding-cosine reward throughput, 8192 captions x 20 tokens, one GPU (rank 0)
        if rank == 0:
            f3, c3 = synth.make_inputs(103, 8192, L_CAP)
            for _ in range(2):
                eng.get_rewards(f3, c3)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 5
            e0.record()
            for _ in range(reps):
                eng.get_rewards(f3, c3)
            e1.record()
            torch.cuda.synchronize()
            ms3 = e0.elapsed_time(e1) / reps
            reward_tp = {"workload": "configs[2]: GetRewards on 8192 captions x %d tokens from zero state (163,840 serial GRU "
                                     "positions), one GPU, host inputs" % L_CAP,
                         "value": 8192 / (ms3 * 1e-3), "unit": "captions/s", "ms_per_call": ms3, "n_gpus": 1,
                         "pieces": None if eng.piece_layout is None else eng.piece_layout["r"][0],
                         "warmup": None if eng.piece_layout is None else eng.piece_layout["r"][2]}
        # config 5: curriculum A2C (partial-prefix rollouts), global batch 8192 sharded over the run's ranks
        B5 = 8192
        f5, c5 = synth.make_inputs(105, B5, L_CAP)
        lo5, hi5 = shard_bounds(B5, rank, world)
        levels = {}
        tot_ms = 0.0
        for level in (3, 6, 9, 12, 15, 16):
            p0 = L_CAP - level
            u5 = np.ascontiguousarray(synth.make_uniforms(105 + level, level, B5)[:, lo5:hi5])
            prep5 = eng.prepare(f5[lo5:hi5], c5[lo5:hi5], u5, plan=(p0, level))
            c0 = seg_counters()
            ms5, _ = timed(lambda: dp.step(prep5, global_rows=B5), 2, 2)
            levels[str(level)] = {"p0": p0, "S": level, "ms_per_step": ms5, "captions_per_s": B5 / (ms5 * 1e-3),
                                  "chain_checks": seg_delta(c0)}
            tot_ms += ms5
        curriculum = {"workload": "configs[4]: curriculum A2C step (ground-truth prefix of L - level columns, `level` sampled "
                                  "steps), global batch %d over %d GPU(s), levels 3..16, every step checked" % (B5, world),
                      "global_batch": B5, "local_batch": hi5 - lo5, "n_gpus": world, "levels": levels,
                      "aggregate_captions_per_s": 6 * B5 / (tot_ms * 1e-3), "unit": "captions/s"}
        eng.prepare(fl, cl, ul, plan=plan)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    # ---- tensor-pipe figure of the persistent decode kernel (policy_decode_kernel: all S steps in one launch).
    # Timed live as the policy_fwd phase (h0 GEMM + h split + the decode kernel; the kernel is >95 % of it).
    Bl = hi - lo
    decode = None
    try:
        us = phases.get("policy_fwd", 0.0) * 1e3
        alg = Bl * (S * 2.0 * 2048 * 512 + S * 2.0 * 1004 * 512)
        rows_pad = ((Bl + 127) // 128) * 128
        executed = 3.0 * rows_pad * (S * 2.0 * 2048 * 512 + S * 2.0 * 1024 * 512)
        tp = float(peaks.get("bf16_tflops", 1590.0))
        decode = {"kernel": "policy_decode_kernel (gate GEMM + cell update + vocab GEMM + softmax + sampling, all %d steps)" % S,
                  "bound": "tensor", "achieved": alg / us / 1e6, "executed_tflops": executed / us / 1e6, "unit": "TFLOP/s",
                  "us_per_launch": us, "rows": Bl, "mma_passes": 3, "peak": tp, "frac": alg / us / 1e6 / tp,
                  "frac_executed": executed / us / 1e6 / tp, "peak_source": "measured" if peaks else "fallback",
                  "note": "achieved counts the algorithmic 2MNK of the recurrent gate GEMM and the vocab GEMM once; the "
                          "tensor pipe executes 3x that (2-part fp16 split) on rows padded to 128 and V padded to 1024"}
    except Exception as exc:                                   # never let the side measurement kill the bench line
        decode = {"error": str(exc)}
    try:
        roofline = roofline_of(phases, Bl, lay, peaks, clk)
    except Exception as exc:
        roofline = {"error": str(exc)}

    st = eng.segment_stats
    chain_cfg = None
    if lay is not None:
        chain_cfg = {"engine": "tc", "forward_launch": "fused (value + reward side by side)" if lay.get("fused") else "two launches",
                     "pieces": {"value": lay["v"][0], "reward": lay["r"][0], "value_backward": (lay.get("b") or lay["v"])[0]},
                     "positions_per_piece": {"value": lay["v"][1], "reward": lay["r"][1]},
                     "warmup": {"value": lay["v"][2], "reward": lay["r"][2], "value_backward": (lay.get("b") or lay["v"])[2]},
                     "tolerance": eng.chain_tol,
                     "checked_max": dict(zip(("value_h", "value_c", "value_h_half", "value_c_half", "reward_h", "-", "reward_h_half",
                                              "--", "bwd_dh", "bwd_dc", "bwd_dh_half", "bwd_dc_half", "dh_take_max", "fp16_overflow"),
                                             st["tc_max_err"][:14])),
                     "warmup_history": st["warm_history"][-12:], "value_leg": dict(value_seg, checked_per_step=value_checked_per_step)}
    elif seg_layout is not None:
        chain_cfg = {"engine": "simt", "pieces": seg_layout[0], "value_segment": seg_layout[1], "reward_segment": seg_layout[2],
                     "warmup": seg_layout[3], "tolerance": eng.chain_tol, "value_leg": value_seg}
    out = {
        "metric": "A2C train captions/sec", "value": B / (ms_step * 1e-3), "unit": "captions/s", "n_gpus": world,
        "steps": args.steps, "warmup": n_warm, "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD % (B, L_CAP, S),
                   "global_batch": B, "local_batch": Bl, "parallelism": "dp%d" % world, "vocab": 1004,
                   "optimizer": "torch.optim.Adam" if args.torch_adam else "FlatAdam (one kernel over the flat bucket)",
                   "chain_shards_per_rank": args.chain_shards, "chain_segments": chain_cfg,
                   "l2_flush": "not needed: per-step working set (chain stash, GBs) >> 126 MB L2",
                   "timed_steps_start": "every warm-up and timed step starts from the seeded weights and a fresh "
                                        "optimizer state (the first training step, replayed); only the chain warm-ups "
                                        "adapt from step to step"},
        "clocks": clk, "gpu_launches": int(launches), "phases_ms": phases, "roofline": roofline,
        "roofline_decode": decode,
    }
    if e2e:
        out["e2e"] = e2e
    if serial_leg:
        out["serial_chain"] = serial_leg
    if sharded:
        out["sharded"] = sharded
    if reward_tp:
        out["reward_throughput"] = reward_tp
    if curriculum:
        out["curriculum"] = curriculum
    if world == 1 and not args.no_cpu_baseline:
        Bs = min(args.cpu_sample, B)
        cps, cores, times, _ = cpu_reference([Bs])
        out["cpu_baseline"] = {"value": cps, "unit": "captions/s", "cores": cores, "kind": "port",
                               "sample": "1 timed step of the first %d of the %d captions (%.1f s) after an un-timed 64-caption "
                                         "step; the reference's cost is linear in rows (serial RNN chains); the reference arm "
                                         "(--impl reference) times all %d rows" % (Bs, B, times[0], B)}
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
