import os, sys
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from icrl_b200 import synth
from icrl_b200.engine import A2CEngine, H
from icrl_b200.optim import FlatAdam
from tests.helpers import make_nets
seed, B, L = 307, 1024, 20
nsteps = int(sys.argv[1]) if len(sys.argv) > 1 else 200
A, R, w = make_nets(seed)
eng = A2CEngine(A, R)
opt = FlatAdam(eng, lr=1e-4)
f, c = synth.make_inputs(seed, B, L)
for i in range(nsteps):
    res = eng.step(f, c, uniforms=synth.make_uniforms(seed + i, L - 1, B))
    opt.step()
print("after", nsteps, "steps: warm", eng.warm, "hist", eng.segment_stats["warm_history"], "reruns", eng.segment_stats["reruns"], flush=True)
u = synth.make_uniforms(seed + 999, L - 1, B)
def grads(e, **kw):
    r = e.step(f, c, uniforms=u, **kw)
    torch.cuda.synchronize()
    return r, e.flat_grad.clone()
out = {}
e1 = A2CEngine(A, R, chain_segments=1); out["serial"] = grads(e1)
ea = A2CEngine(A, R, chain_warmup=eng.warm["v"], chain_adapt=False); ea.warm = dict(eng.warm); out["tc_adapted"] = grads(ea)
eb = A2CEngine(A, R, chain_warmup=1024, chain_adapt=False); out["tc_warm1024"] = grads(eb)
ed = A2CEngine(A, R, chain_pieces=128, chain_warmup=1024, chain_adapt=False); out["tc_128pieces_warm1024"] = grads(ed)
print("layouts", ea.piece_layout, eb.piece_layout, ed.piece_layout)
print("tc errs adapted", ["%.1e" % x for x in ea.segment_stats["tc_max_err"][:14]])
print("tc errs 1024   ", ["%.1e" % x for x in eb.segment_stats["tc_max_err"][:14]])
names = list(out)
gmax = float(out["serial"][1].abs().max())
vmax = float(out["serial"][0]["values"].abs().max())
print("grad max", gmax, "values max", vmax)
for i in range(len(names)):
    for j in range(i + 1, len(names)):
        a, b = out[names[i]], out[names[j]]
        print("%-24s vs %-24s: grads rel-to-max %.2e   values %.2e   rewards %.2e" % (names[i], names[j],
              float((a[1] - b[1]).abs().max()) / gmax, float((a[0]["values"] - b[0]["values"]).abs().max()),
              float((a[0]["rewards"] - b[0]["rewards"]).abs().max())), flush=True)
# per-tensor breakdown serial vs tc_warm1024
off = 0
g1, g2 = out["serial"][1], out["tc_warm1024"][1]
for (k, p), o in zip(A.named_parameters(), eng._flat_offsets):
    a, b = g1[o:o + p.numel()], g2[o:o + p.numel()]
    print("  %-45s max %.3e  diff/max %.2e" % (k, float(a.abs().max()), float((a - b).abs().max() / a.abs().max())))
sc = e1._bufs["v_stash_c"][: (out["serial"][0]["Tv"] + 1) * H]
sg = e1._bufs["v_stash_g"][: out["serial"][0]["Tv"] * 4 * H].view(-1, 4, H)
print("max |c| %.2f  mean forget gate %.4f  frac f>0.99: %.4f" % (float(sc.abs().max()), float(sg[:, 1].mean()), float((sg[:, 1] > 0.99).float().mean())))
