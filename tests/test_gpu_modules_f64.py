"""The module route (models.py's autograd Functions: _PolicyFn, _LstmSeqFn, _ChainLSTMFn, _ChainGRUFn, _ValueHeadFn,
_LinearFn) against a float64 reference at the shapes the supervised pretraining loops and the bidirectional networks
run, forward and backward.

The reference is oracle/ref_port.Nets(dtype=torch.float64), which tests/test_oracle_golden.py pins to the unmodified
reference on CPU.  Each module case runs the drop-in module on CUDA and the reference on CPU with the same weights and
back-propagates sum(out * g) for a seeded standard-normal g over every output of every call, so every row and position
carries gradient; it compares the outputs, every entry of every parameter gradient and the hidden_cell after the calls.
The loop cases run one minibatch of each pretraining loop of icrl_b200.trainers.  Where a loop makes a discrete decision
(the greedy captions of train_value_network, the ReLU active set of the VSE loss) the float64 side takes the CUDA side's
decision, so the comparison measures arithmetic; a separate assertion requires every decision that float64 would make
differently to lie within 1e-5 of its boundary.

Tolerances (the suite's own): outputs within 2e-6 * max(1, max|ref|); the loss within 2e-6 relative; each gradient
within 2e-5 of the tensor's max |entry| and its L2 norm within 2e-5 relative.  The errors of the kernels and of the
float32 port against the same float64 result go to module_f64_errors.json in the directory named by ICRL_ERRORS_DIR,
when that variable is set.

dW_hh of the value chain and of the policy runs on tcgen05 (wgrad_tc.cu) when the module route's fixed workspace
(models._gemm_ws) holds icrl_wgrad_tc_ws_bytes(2048, 512, T, 2) bytes -- T <= 9,009 positions -- and on the fp32 SIMT
GEMM above; each case asserts which side of the switch it is on.
"""
import json
import os

import numpy as np
import pytest
import torch

from oracle import ref_port, synth

pytestmark = pytest.mark.gpu

FTOL = 2e-6          # outputs, relative to max(1, max|ref|)
LTOL = 2e-6          # losses, relative
GTOL = 2e-5          # gradients, of the tensor's max |entry|; L2 norms, relative
DTOL = 1e-5          # a decision that differs from float64's own lies this close to its boundary
PORT_FACTOR = 3      # bound where the float32 port itself misses the tolerance: this multiple of the port's error

ERRORS = {}


def _record(name, **kv):
    """Measured errors (kernel and float32 port vs float64), dumped to $ICRL_ERRORS_DIR/module_f64_errors.json when
    ICRL_ERRORS_DIR is set; nothing is written otherwise."""
    ERRORS.setdefault(name, {}).update({k: (float(v) if isinstance(v, (float, int, np.floating)) else v) for k, v in kv.items()})
    out = os.environ.get("ICRL_ERRORS_DIR")
    if not out:
        return
    try:
        os.makedirs(out, exist_ok=True)
        with open(os.path.join(out, "module_f64_errors.json"), "w") as fh:
            json.dump(ERRORS, fh, indent=1, sort_keys=True)
    except OSError:
        pass


def _np(t):
    return t.detach().double().cpu().numpy()


def _fwd_err(got, ref):
    return float(np.abs(got - ref).max()) / max(1.0, float(np.abs(ref).max()))


def _grad_errs(got, ref):
    """(max |got - ref| / max |ref|, relative error of the L2 norm)."""
    scale = max(float(np.abs(ref).max()), 1e-300)
    nrm, ref_n = float(np.sqrt((got ** 2).sum())), float(np.sqrt((ref ** 2).sum()))
    return float(np.abs(got - ref).max()) / scale, abs(nrm - ref_n) / max(ref_n, 1e-300)


def _errors(got, ref):
    """Per-tensor errors of got against ref: {('out', k): fwd} and {('grad', name): (max error, norm error)}."""
    errs = {}
    for k, (a, b) in enumerate(zip(got["outs"] + got["hidden"], ref["outs"] + ref["hidden"])):
        assert a.shape == b.shape, (k, a.shape, b.shape)
        errs[("out", k)] = (_fwd_err(a, b),)
    assert sorted(got["grads"]) == sorted(ref["grads"])
    for k in ref["grads"]:
        errs[("grad", k)] = _grad_errs(got["grads"][k], ref["grads"][k])
    return errs


def _worst(errs):
    """(worst output error, worst gradient error, worst norm error)."""
    pick = lambda kind, i: max([e[i] for (t, _), e in errs.items() if t == kind] or [0.0])
    return pick("out", 0), pick("grad", 0), pick("grad", 1)


def _check(name, errs, port_errs):
    """Each tensor within the suite's tolerance.  Where the float32 port itself misses that tolerance on the same tensor
    (so no float32 arithmetic of the operation meets it: the cell state after thousands of slow-forgetting steps, a bias
    gradient that is a cancelling sum over 512 rows), the bound is PORT_FACTOR times the port's error instead; those
    tensors are returned so that they are recorded."""
    over = []
    for key, e in errs.items():
        for i, tol in enumerate((FTOL,) if key[0] == "out" else (GTOL, GTOL)):
            bound = tol
            if port_errs[key][i] > tol:
                bound = PORT_FACTOR * port_errs[key][i]
                over.append("%s/%s" % key)
            assert e[i] <= bound, "%s: %s %s error %.3e (bound %.1e; float32 port %.3e)" % (
                name, key[0], key[1], e[i], bound, port_errs[key][i])
    return over


# ---------------------------------------------------------------------------------------------------------------------
# the dW_hh switch of icrl_value_chain_param_grads / policy_rollout_bwd_common

def _gemm_ws_bytes():
    import icrl_b200.models as M
    return M._gemm_ws(torch.device("cuda:0")).numel() * 4


def _tc_fits(T):
    from icrl_b200 import _lib
    _lib.load()
    return _gemm_ws_bytes() >= int(_lib.call("icrl_wgrad_tc_ws_bytes", 2048, 512, T, 2))


def test_wgrad_switch_lies_at_9009_positions():
    """The module route's workspace holds the tcgen05 dW_hh contraction up to T = 9,009 positions exactly, so the
    cases below at B = 529 / 530 x 17 columns (and the policy at 512 / 564 x 16 cells) sit on both sides of it."""
    assert _tc_fits(1) and _tc_fits(9009) and not _tc_fits(9010)


def _dwhh_paths(kind, variant, B, calls):
    """The dW_hh path of every call, from the shape: the value chain contracts T = n*B positions per call, the policy
    n*B cell steps; the reward GRU and the bidirectional policy's sequence backward have no tcgen05 path."""
    if kind == "reward" or (kind == "policy" and variant == "bidir"):
        return ["simt"] * len(calls)
    return ["tcgen05" if _tc_fits(n * B) else "simt" for n in calls]


# ---------------------------------------------------------------------------------------------------------------------
# module cases

def _weights(seed, variant):
    w = synth.make_weights(seed, wordvec_dim=300 if variant == "wemb300" else 512, bidirectional=variant == "bidir")
    if variant == "slow":
        # slow forgetting, as in test_slow_forgetting_weights_degrade_gracefully: value LSTM forget gate and reward GRU
        # update gate pushed towards 'keep' by +1.5
        w["value"]["valrnn.lstm.bias_hh_l0"][512:1024] += 1.5
        w["reward"]["rewrnn.gru.bias_hh_l0"][512:1024] += 1.5
    return w


def _module_net(kind, variant, w):
    import icrl_b200.models as M
    w2i = synth.word_to_idx()
    cls, emb = {"policy": (M.PolicyNetwork, "caption_embedding.weight"),
                "value": (M.ValueNetwork, "valrnn.caption_embedding.weight"),
                "reward": (M.RewardNetwork, "rewrnn.caption_embedding.weight")}[kind]
    pre = w[kind][emb].numpy() if variant == "wemb300" else None
    net = cls(w2i, pretrained_embeddings=pre, bidirectional=variant == "bidir")
    net.load_state_dict(w[kind])
    return net.cuda()


def _run_module(kind, variant, w, f, c, calls, gs):
    net = _module_net(kind, variant, w)
    ft, ct = torch.from_numpy(f).cuda(), torch.from_numpy(c).cuda()
    if kind == "policy":
        outs = [net(ft.unsqueeze(0), ct[:, :calls[0]])]
    elif kind == "value":
        net.valrnn.init_hidden()
        outs = [net(ft, ct[:, :n]) for n in calls]
    else:
        net.rewrnn.init_hidden()
        outs = [o for n in calls for o in net(ft, ct[:, :n])]
    assert len(outs) == len(gs)
    for p in net.parameters():
        p.grad = None
    sum((o * torch.from_numpy(g).cuda()).sum() for o, g in zip(outs, gs)).backward()
    torch.cuda.synchronize()
    hidden = net.valrnn.hidden_cell if kind == "value" else (net.rewrnn.hidden_cell,) if kind == "reward" else ()
    grads = {}
    for k, p in net.named_parameters():
        if p.requires_grad:
            assert p.grad is not None, k
            grads[k] = _np(p.grad)
        else:                                        # a frozen pretrained embedding gets no gradient
            assert variant == "wemb300" and k.endswith("caption_embedding.weight") and p.grad is None, k
    return dict(outs=[_np(o) for o in outs], hidden=[_np(h) for h in hidden], grads=grads)


def _run_reference(kind, nets, f, c, calls, gs):
    dt = nets.dtype
    ft, ct = torch.from_numpy(f).to(dt), torch.from_numpy(c)

    def fn():
        nets.reset_state()
        if kind == "policy":
            outs = [ref_port.policy_logits(nets, ft, ct[:, :calls[0]])]
        elif kind == "value":
            outs = [ref_port.value_call(nets, ft, ct[:, :n]) for n in calls]
        else:
            outs = [o for n in calls for o in ref_port.reward_embed(nets, ft, ct[:, :n])]
        hidden = {"policy": (), "value": nets.v_state, "reward": (nets.r_state,)}[kind]
        loss = sum((o * torch.from_numpy(g).to(dt)).sum() for o, g in zip(outs, gs))
        return loss, outs, [h.detach().clone() for h in hidden]

    (_, outs, hidden), grads = ref_port.network_grads(nets, kind, fn)
    nets.reset_state()
    return dict(outs=[_np(o) for o in outs], hidden=[_np(h) for h in hidden], grads={k: _np(v) for k, v in grads.items()})


# (kind, variant, B, columns of each call, dW_hh path of each call)
TC, SIMT = "tcgen05", "simt"
MODULE_CASES = [
    ("policy", "plain", 1, [1], [TC]),                       # wgrad_tc at T = 1, M = 1 GEMMs
    ("policy", "plain", 129, [16], [TC]),                    # ragged 128-row tiles
    ("policy", "plain", 512, [16], [TC]),                    # train_policy_network's default, n*B = 8,192
    ("policy", "plain", 564, [16], [SIMT]),                  # n*B = 9,024
    ("policy", "wemb300", 129, [16], [TC]),                  # dE null, dW_ih 2048 x 300
    ("policy", "bidir", 129, [16], [SIMT]),                  # _LstmSeqFn both directions, dh0 into both cnn2linear halves
    ("value", "plain", 1, [1, 2, 3], [TC] * 3),              # T = 1 chain, dh0 / dc0 handed across calls
    ("value", "plain", 129, list(range(1, 17)), [TC] * 16),  # the A2C module-route pattern, 17,544 positions
    ("value", "plain", 529, [17], [TC]),                     # T = 8,993
    ("value", "plain", 530, [17], [SIMT]),                   # T = 9,010
    ("value", "wemb300", 129, [1, 2, 3, 4], [TC] * 4),
    ("value", "bidir", 129, [1, 2, 3, 4], [TC] * 4),         # reverse chains, rnn_linear
    ("value", "slow", 512, [17], [TC]),                      # gradient carried back hundreds of positions
    ("reward", "plain", 1, [1, 1], [SIMT] * 2),              # GRU backward at T = 1, dh_init / dh0_out, no init_hidden
    ("reward", "plain", 512, [17], [SIMT]),                  # train_reward_network's default, T = 8,704
    ("reward", "plain", 129, [17, 17], [SIMT] * 2),          # carried GRU state with graph
    ("reward", "plain", 129, [17, 1], [SIMT] * 2),           # the same, second call's gradient reaches the first chain
    ("reward", "wemb300", 129, [17], [SIMT]),
    ("reward", "bidir", 129, [17], [SIMT]),                  # reverse GRU, 1024-wide semantic_embed
    ("reward", "slow", 512, [17], [SIMT]),
]
SEEDS = {"plain": 401, "wemb300": 402, "bidir": 403, "slow": 404}


def _case_id(case):
    kind, variant, B, calls, _ = case
    return "%s-%s-b%d-%s" % (kind, variant, B, "x".join(map(str, calls)) if len(calls) <= 4 else "1to%d" % calls[-1])


@pytest.mark.parametrize("case", MODULE_CASES, ids=[_case_id(c) for c in MODULE_CASES])
def test_module_vs_float64(case):
    kind, variant, B, calls, paths = case
    name = _case_id(case)
    assert _dwhh_paths(kind, variant, B, calls) == paths, name
    seed = SEEDS[variant]
    w = _weights(seed, variant)
    f, c = synth.make_inputs(seed, B, 17)
    rs = np.random.RandomState(seed * 1000 + B)
    V = w["policy"]["linear2vocab.weight"].shape[0]
    shapes = {"policy": [(B, calls[0], V)], "value": [(B, 1)] * len(calls), "reward": [(B, 512), (B, 512)] * len(calls)}
    gs = [rs.standard_normal(s).astype(np.float32) for s in shapes[kind]]
    got = _run_module(kind, variant, w, f, c, calls, gs)
    bidir = variant == "bidir"
    ref = _run_reference(kind, ref_port.Nets(w, dtype=torch.float64, bidirectional=bidir), f, c, calls, gs)
    port = _run_reference(kind, ref_port.Nets(w, bidirectional=bidir), f, c, calls, gs)
    port_errs, errs = _errors(port, ref), _errors(got, ref)
    pf, pg, pn = _worst(port_errs)
    kf, kg, kn = _worst(errs)
    _record(name, port_fwd=pf, port_grad=pg, port_norm=pn, fwd=kf, grad=kg, norm=kn,
            dwhh_path=",".join(sorted(set(paths))), positions=B * sum(calls))
    _record(name, port_bound=_check(name, errs, port_errs))


# ---------------------------------------------------------------------------------------------------------------------
# loop cases: one minibatch of each pretraining loop of icrl_b200.trainers

LOOP_CASES = [("plain", 512, 411), ("bidir", 129, 413)]


def _run_loop(key, variant, B, seed, tmp_path, monkeypatch):
    """One minibatch of train_<key>_network with the patches of test_pretraining_loops_vs_reference_golden.  Returns
    (loss, net, decisions): the VSE loss's ReLU masks, or the greedy captions and the value prefix length."""
    import icrl_b200.models as M
    import icrl_b200.trainers as T
    w = _weights(seed, variant)
    f, c = synth.make_inputs(seed, B, 17)
    data = {"train_captions": c, "train_image_idxs": np.arange(B), "train_features": f,
            "train_urls": np.array(["u"] * B), "word_to_idx": synth.word_to_idx(), "embeddings": None}
    paths = {k: str(tmp_path / (k + ".pt")) for k in ("policy_network", "reward_network", "value_network")}
    torch.save(w["policy"], paths["policy_network"])
    torch.save(w["reward"], paths["reward_network"])

    def factory(cls, sd):
        def make(*a, **k):
            net = cls(*a, **k)
            net.load_state_dict(sd)
            return net
        return make

    losses, seen = [], {}

    class Rec:
        def __init__(self, *a, **k):
            pass

        def add_scalar(self, tag, val, step):
            losses.append(float(val))

    vse, greedy, randint = T.VisualSemanticEmbeddingLoss, T.GenerateCaptionsGreedy, T.random.randint

    def vse_rec(ve, se):
        seen["vse"] = (ve.detach(), se.detach())
        return vse(ve, se)

    def greedy_rec(*a):
        seen["gen"] = greedy(*a)
        return seen["gen"]

    def randint_rec(a, b):
        seen["k"] = randint(a, b)
        return seen["k"]

    monkeypatch.setattr(T, "PolicyNetwork", factory(T.PolicyNetwork, w["policy"]))
    monkeypatch.setattr(T, "ValueNetwork", factory(T.ValueNetwork, w["value"]))
    monkeypatch.setattr(T, "RewardNetwork", factory(T.RewardNetwork, w["reward"]))
    monkeypatch.setattr(T, "SummaryWriter", Rec)
    monkeypatch.setattr(T.torch, "randperm", lambda n: torch.arange(n))
    monkeypatch.setattr(T, "VisualSemanticEmbeddingLoss", vse_rec)
    monkeypatch.setattr(T, "GenerateCaptionsGreedy", greedy_rec)
    monkeypatch.setattr(T.random, "randint", randint_rec)
    T.random.seed(seed)
    fn = {"policy": T.train_policy_network, "reward": T.train_reward_network, "value": T.train_value_network}[key]
    net = fn(data, paths, str(tmp_path), variant == "bidir", epochs=1, batch_size=B)
    assert len(losses) == 1
    dec = {}
    if key == "reward":
        # the active sets of the module's ReLUs: the hinge exactly as VisualSemanticEmbeddingLoss forms it
        ve, se = seen["vse"]
        N = ve.shape[0]
        margin = (0.2 / N) * (1.0 - torch.eye(N, device=ve.device))
        zero = torch.zeros(N, device=ve.device)
        masks = []
        for a, b in ((ve, se), (se, ve)):
            sim = M._LinearFn.apply(a, b, zero)
            masks.append(((sim - torch.diag(sim).unsqueeze(1) + margin) > 0).cpu())
        dec["masks"] = masks
    elif key == "value":
        dec["gen"], dec["k"] = seen["gen"].cpu().long(), seen["k"]
    return losses[0], net, w, f, c, dec


def _loop_reference(key, nets, f, c, dec):
    dt = nets.dtype
    if key == "policy":
        fn = lambda: ref_port.policy_xent_loss(nets, f, c)
    elif key == "reward":
        fn = lambda: ref_port.reward_vse_loss(nets, f, c, masks=[m.to(dt) for m in dec["masks"]])
    else:
        fn = lambda: ref_port.value_mse_loss(nets, f, c, dec["k"], gen=dec["gen"])
    res, grads = ref_port.network_grads(nets, key, fn)
    return res, {k: _np(v) for k, v in grads.items()}


def _check_decisions(key, nets, f, res, dec, name):
    """Every decision of the CUDA side that float64 makes differently lies within DTOL of its boundary."""
    if key == "reward":
        _, ve, se = res
        flips, worst = 0, 0.0
        for m, (a, b) in zip(dec["masks"], ((ve, se), (se, ve))):
            x = ref_port.vse_hinge(a.detach(), b.detach()).numpy()
            diff = (x > 0) != m.numpy()
            flips += int(diff.sum())
            worst = max(worst, float(np.abs(x[diff]).max()) if diff.any() else 0.0)
        _record(name, relu_flips=flips, relu_flip_margin=worst)
        assert worst <= DTOL, (flips, worst)
    elif key == "value":
        gen, ft = dec["gen"], torch.from_numpy(f).to(nets.dtype)
        flips, worst = 0, 0.0
        with torch.no_grad():
            for s in range(gen.shape[1] - 1):                 # the greedy loop re-runs the whole prefix every step
                z = ref_port.policy_logits(nets, ft, gen[:, :s + 1])[:, -1]
                own = z.argmax(dim=1)
                diff = own != gen[:, s + 1]
                if bool(diff.any()):
                    gap = z.max(dim=1).values - z.gather(1, gen[:, s + 1:s + 2])[:, 0]
                    flips += int(diff.sum())
                    worst = max(worst, float(gap[diff].max()))
        _record(name, greedy_flips=flips, greedy_flip_gap=worst)
        assert worst <= DTOL, (flips, worst)


@pytest.mark.parametrize("key", ["policy", "reward", "value"])
@pytest.mark.parametrize("variant,B,seed", LOOP_CASES, ids=[v for v, _, _ in LOOP_CASES])
def test_pretraining_loop_vs_float64(variant, B, seed, key, tmp_path, monkeypatch):
    """train_policy_network / train_reward_network / train_value_network at their default batch_size=512 and a
    bidirectional minibatch of 129 rows: the loss and every gradient against the float64 restatement."""
    name = "loop_%s_%s_b%d" % (key, variant, B)
    loss, net, w, f, c, dec = _run_loop(key, variant, B, seed, tmp_path, monkeypatch)
    bidir = variant == "bidir"
    got = dict(outs=[], hidden=[], grads={k: _np(p.grad) for k, p in net.named_parameters() if p.requires_grad})
    nets = ref_port.Nets(w, dtype=torch.float64, bidirectional=bidir)
    res, grads = _loop_reference(key, nets, f, c, dec)
    _check_decisions(key, nets, f, res, dec, name)
    ref_loss = float(res[0].detach())
    pres, pgrads = _loop_reference(key, ref_port.Nets(w, bidirectional=bidir), f, c, dec)
    ref = dict(outs=[], hidden=[], grads=grads)
    port_errs, errs = _errors(dict(outs=[], hidden=[], grads=pgrads), ref), _errors(got, ref)
    _, pg, pn = _worst(port_errs)
    _, kg, kn = _worst(errs)
    el = abs(loss - ref_loss) / max(abs(ref_loss), 1e-300)
    _record(name, port_loss=abs(float(pres[0].detach()) - ref_loss) / max(abs(ref_loss), 1e-300), port_grad=pg,
            port_norm=pn, loss=el, grad=kg, norm=kn)
    assert el <= LTOL, (loss, ref_loss)
    _record(name, port_bound=_check(name, errs, port_errs))
