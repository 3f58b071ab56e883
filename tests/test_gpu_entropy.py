"""GPU tests of the entropy bonus (loss = reference loss - entropy_coef * mean policy entropy of the sampled steps):
the three kernels through the C ABI against float64, the fused engine against the CPU port of the reference with the
same term (tests/test_entropy_port.a2c_minibatch_entropy), the module route, the data-parallel identity and the public
trainer.

Tolerances are those of test_gpu_parity: token ids bit-exact, loss / mean entropy 2e-6 abs, gradients 2e-5 of each
tensor's largest entry.  Where a check asks for equality of gradients, the value-chain and gate-table gradients are
compared to 1e-6 of the bucket's largest entry: their scatters sum with float atomics, so two runs of the SAME step
already differ in the last bits (test_gpu_parity.test_determinism_and_row_independence_full_size)."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import ref_port, synth
from tests.helpers import check_grads_vs_oracle, make_nets, named_grads
from tests.test_entropy_port import a2c_minibatch_entropy

pytestmark = pytest.mark.gpu

TOL = 2e-6
GTOL = 2e-5
REPRO = 1e-6          # run-to-run reproducibility of the atomically summed gradients, relative to the bucket's max

# decode x policy_bptt x overlap_backward
CONFIGS = [(d, b, o) for d in ("fused", "tc", "simt") for b in ("tc", "simt") for o in (True, False)]
CASES = {"b256_l20": (301, 256, 20, None), "curr_b48_l12_lv5": (302, 48, 12, 5), "ragged_b129": (303, 129, 9, None)}


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


_ORACLE = {}


def _oracle(case, coef):
    """The CPU port with the entropy term on the host cores (cached per case and coefficient)."""
    key = (case, coef)
    if key not in _ORACLE:
        seed, B, L, level = CASES[case]
        w = synth.make_weights(seed)
        f, c = synth.make_inputs(seed, B, L)
        u = synth.make_uniforms(seed, L - 1 if level is None else level, B)
        torch.set_num_threads(max(torch.get_num_threads(), 8))
        _ORACLE[key] = a2c_minibatch_entropy(ref_port.Nets(w), f, c, u, level=level, entropy_coef=coef)
    return _ORACLE[key]


def _run(case, coef, **kw):
    from icrl_b200.engine import A2CEngine
    seed, B, L, level = CASES[case]
    A, R, w = make_nets(seed)
    f, c = synth.make_inputs(seed, B, L)
    u = synth.make_uniforms(seed, L - 1 if level is None else level, B)
    eng = A2CEngine(A, R, entropy_coef=coef, **kw) if coef is not None else A2CEngine(A, R, **kw)
    res = eng.step(f, c, uniforms=u, level=level)
    torch.cuda.synchronize()
    return eng, A, res


def _check_vs_oracle(res, A, ref):
    assert np.array_equal(res["tokens"].cpu().numpy(), ref["tokens"])
    for k in ("values", "rewards", "logp"):
        assert float(np.abs(res[k].cpu().numpy() - ref[k]).max()) <= TOL, k
    assert abs(res.loss - ref["loss"]) <= TOL, (res.loss, ref["loss"])
    assert abs(res.mean_entropy - ref["mean_entropy"]) <= TOL, (res.mean_entropy, ref["mean_entropy"])
    check_grads_vs_oracle(named_grads(A), ref["grads"], GTOL)


# ---------------------------------------------------------------- 1. off means off

def test_coefficient_zero_is_the_default_engine():
    """entropy_coef=0.0 runs exactly today's path: same launches, three stats words, the same outputs bit for bit."""
    outs = []
    for coef in (None, 0.0):
        eng, A, res = _run("b256_l20", coef)
        outs.append((eng.launches.value, res, {k: p.grad.clone() for k, p in A.named_parameters()}))
        assert len(res["stats"]) == 3 and (res.host_stats is None or len(res.host_stats) == 3)
        with pytest.raises(AttributeError):
            res.mean_entropy
    (l0, r0, g0), (l1, r1, g1) = outs
    assert l0 == l1
    for k in ("tokens", "logp", "values", "rewards", "stats"):
        assert torch.equal(r0[k], r1[k]), k
    scale = max(float(g.abs().max()) for g in g0.values())
    for k in g0:
        assert float((g0[k] - g1[k]).abs().max()) <= REPRO * scale, k


# ---------------------------------------------------------------- 2. against the oracle

@pytest.mark.parametrize("coef", [0.01, 1.0])
@pytest.mark.parametrize("decode,bptt,overlap", CONFIGS)
@pytest.mark.parametrize("case", list(CASES))
def test_engine_vs_cpu_port(case, decode, bptt, overlap, coef):
    """Tokens bit-exact, loss and mean entropy within 2e-6, every gradient within 2e-5 of its tensor's max, against
    the CPU port with the same entropy term, at the usual coefficient and at one a hundred times larger."""
    eng, A, res = _run(case, coef, decode=decode, policy_bptt=bptt, overlap_backward=overlap)
    assert len(res["stats"]) == 4
    _check_vs_oracle(res, A, _oracle(case, coef))


@pytest.mark.parametrize("coef", [0.01, 1.0])
def test_odd_vocabulary_vs_cpu_port(coef):
    """V % 4 != 0: the engine takes the per-step decode; the entropy pass and backward see row stride V (and 1024 in
    the tcgen05 backward)."""
    import warnings
    import icrl_b200.models as M
    from icrl_b200.engine import A2CEngine
    seed, B, L, V = 82, 10, 6, 203
    w = synth.make_weights(seed, vocab=V)
    w2i = synth.word_to_idx(V)
    P, Vn, R = M.PolicyNetwork(w2i), M.ValueNetwork(w2i), M.RewardNetwork(w2i)
    P.load_state_dict(w["policy"]); Vn.load_state_dict(w["value"]); R.load_state_dict(w["reward"])
    R.requires_grad_(False)
    A = M.AdvantageActorCriticNetwork(Vn, P).cuda()
    f, c = synth.make_inputs(seed, B, L, vocab=V)
    u = synth.make_uniforms(seed, L - 1, B)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        eng = A2CEngine(A, R.cuda(), entropy_coef=coef)
    assert eng.decode == "simt"
    res = eng.step(f, c, uniforms=u)
    ref = a2c_minibatch_entropy(ref_port.Nets(w), f, c, u, entropy_coef=coef)
    _check_vs_oracle(res, A, ref)


# ---------------------------------------------------------------- 3. the kernels against float64

def _entropy64(z):
    z = z.double()
    return -(torch.softmax(z, -1) * torch.log_softmax(z, -1)).nan_to_num(0.0).sum(-1)


def _logits(S, B, V, ld, seed=7):
    g = torch.Generator().manual_seed(seed)
    z = torch.randn(S, B, V, generator=g) * 4
    z[0, 0, ::3] = -1e4                                 # p underflows to 0
    z[0, 1, 5::7] = -float("inf")
    z[1, 0] = -1e30                                     # one-hot row: H = 0
    z[1, 0, 17] = 3.0
    z[1, 2] = 0.0                                       # uniform row: H = log V
    zp = torch.full((S, B, ld), float("nan"))           # padding columns must not enter the sums
    zp[..., :V] = z
    return z, zp


@pytest.mark.parametrize("ld", [1004, 1024])
def test_policy_entropy_vs_float64(ld):
    from icrl_b200 import _lib
    S, B, V = 3, 37, 1004
    z, zp = _logits(S, B, V, ld)
    ent, zd = torch.empty(B, S, device="cuda"), zp.cuda()
    n = _lib.Launches()
    _lib.call("icrl_policy_entropy", _stream(), B, S, V, _p(zd), ld, _p(ent), n.ref)
    torch.cuda.synchronize()
    ref = _entropy64(z).t()                             # [B][S]
    got = ent.cpu().double()
    assert n.value == 1 and torch.isfinite(got).all()
    assert float(got[0, 1]) == 0.0
    assert abs(float(got[2, 1]) - np.log(V)) <= 1e-6 * np.log(V)
    assert float(((got - ref).abs() / ref.clamp(min=1.0)).max()) <= 1e-6


def test_softmax_entropy_bwd_vs_float64_keeps_padding_zero():
    from icrl_b200 import _lib
    S, B, V, ld = 3, 37, 1004, 1024
    z, _ = _logits(S, B, V, V)
    z[0, 1, 5::7] = -1e4                                # finite logits, as the rollout stashes them
    zp = torch.zeros(S, B, ld)
    zp[..., :V] = z
    g = torch.Generator().manual_seed(3)
    tokens = torch.randint(0, V, (B, S), generator=g)
    dlogp = torch.randn(B, S, generator=g) * 1e-3
    scale = 0.37 / (B * S)
    # device copies held in locals until the kernels have run (a temporary's memory would be handed out again at once)
    zd, ent, td, dd = zp.cuda(), torch.empty(B, S, device="cuda"), tokens.cuda(), dlogp.cuda()
    _lib.call("icrl_policy_entropy", _stream(), B, S, V, _p(zd), ld, _p(ent), None)
    _lib.call("icrl_softmax_entropy_bwd", _stream(), B, S, V, _p(zd), ld, _p(td), _p(dd), _p(ent), scale, None)
    got = zd.cpu()
    assert torch.equal(got[..., V:], torch.zeros(S, B, ld - V))
    # float64: dL/dz of  sum_{b,s} dlogp[b][s] log p[a]  -  (scale) sum_{b,s} H[b][s]
    zz = z.double().requires_grad_(True)
    lp = torch.log_softmax(zz, -1)
    a = tokens.t().unsqueeze(-1)
    loss = (dlogp.t().double() * lp.gather(-1, a).squeeze(-1)).sum() - scale * _entropy64(zz).sum()
    loss.backward()
    ref = zz.grad
    err = float((got[..., :V].double() - ref).abs().max())
    assert err <= 1e-5 * float(ref.abs().max()), err


def test_loss_entry_matches_the_reference_entry():
    """icrl_a2c_loss_entropy_fwd_bwd: dv_sb, dlogp, sum_dv and the reward / advantage words bit-identical to
    icrl_a2c_loss_fwd_bwd; out4[3] = mean entropy; out4[0] = loss - coef * mean entropy."""
    from icrl_b200 import _lib
    B, S, coef = 129, 19, 0.25
    g = torch.Generator().manual_seed(5)
    values, rewards = torch.randn(B, S, generator=g).cuda(), torch.rand(B, S, generator=g).cuda()
    logp = (-torch.rand(B, S, generator=g) * 6).cuda()
    ent = (torch.rand(B, S, generator=g) * 6).cuda()
    inv = 1.0 / (B * S)
    outs = []
    for e in (None, ent):
        out, dv, dl, sd = torch.zeros(4, device="cuda"), torch.empty(S, B, device="cuda"), torch.empty(B, S, device="cuda"), \
            torch.empty(1, device="cuda")
        if e is None:
            _lib.call("icrl_a2c_loss_fwd_bwd", _stream(), B, S, _p(values), _p(rewards), _p(logp), inv, _p(out), _p(dv), _p(dl), _p(sd),
                      None)
        else:
            _lib.call("icrl_a2c_loss_entropy_fwd_bwd", _stream(), B, S, _p(values), _p(rewards), _p(logp), _p(e), coef, inv, _p(out),
                      _p(dv), _p(dl), _p(sd), None)
        outs.append((out.cpu(), dv.cpu(), dl.cpu(), sd.cpu()))
    (o3, dv0, dl0, sd0), (o4, dv1, dl1, sd1) = outs
    assert torch.equal(dv0, dv1) and torch.equal(dl0, dl1) and torch.equal(sd0, sd1)
    assert torch.equal(o3[1:3], o4[1:3]) and float(o3[3]) == 0.0
    me = float(ent.double().mean())
    assert abs(float(o4[3]) - me) <= 1e-6 * me
    assert abs(float(o4[0]) - (float(o3[0]) - coef * me)) <= 1e-6


# ---------------------------------------------------------------- 4. what must not move

@pytest.mark.parametrize("coef", [0.01, 1.0])
def test_bonus_touches_only_the_policy_gradient_and_the_loss(coef):
    e0, A0, r0 = _run("b256_l20", 0.0)
    g0 = {k: p.grad.clone() for k, p in A0.named_parameters()}
    e1, A1, r1 = _run("b256_l20", coef)
    g1 = {k: p.grad.clone() for k, p in A1.named_parameters()}
    for k in ("tokens", "logp", "values", "rewards"):
        assert torch.equal(r0[k], r1[k]), k
    assert torch.equal(r0["stats"][1:3], r1["stats"][1:3])
    assert abs((r1.loss - r0.loss) - (-coef * r1.mean_entropy)) <= 1e-6
    value = [k for k in g0 if k.startswith("value_network.")]
    scale = max(float(g0[k].abs().max()) for k in value)
    for k in value:
        if k.startswith("value_network.linear"):        # value head: no atomics on its way
            assert torch.equal(g0[k], g1[k]), k
        assert float((g0[k] - g1[k]).abs().max()) <= REPRO * scale, k
    moved = [k for k in g0 if k.startswith("policy_network.") and not torch.equal(g0[k], g1[k])]
    assert "policy_network.linear2vocab.weight" in moved
    assert e1.launches.value == e0.launches.value + 1           # the entropy pass; the backward swaps one pass for another


# ---------------------------------------------------------------- 5. module route

def test_module_route_agrees_with_the_engine():
    """The reference-style loop on the drop-in modules with the torch entropy term (trainers._module_route_step) against
    the fused step on the same numpy stream."""
    import icrl_b200.trainers as T
    from icrl_b200.engine import A2CEngine
    seed, B, L, coef = 311, 32, 9, 0.5
    A, R, w = make_nets(seed)
    f, c = synth.make_inputs(seed, B, L)
    np.random.seed(seed)
    A.value_network.valrnn.init_hidden()
    R.rewrnn.init_hidden()
    mr = T._module_route_step(A, R, f, c, None, entropy_coef=coef)
    gm = named_grads(A)
    A.value_network.valrnn.init_hidden()
    R.rewrnn.init_hidden()
    np.random.seed(seed)
    res = A2CEngine(A, R, entropy_coef=coef).step(f, c)
    ge = named_grads(A)
    assert abs(res.loss - mr.loss) <= TOL and abs(res.mean_entropy - mr.mean_entropy) <= TOL
    for k in gm:
        if k.startswith("policy_network."):
            err = float(np.abs(ge[k] - gm[k]).max()) / max(float(np.abs(gm[k]).max()), 1e-12)
            assert err <= GTOL, (k, err)


def test_bidirectional_module_route_vs_cpu_port():
    import icrl_b200.models as M
    import icrl_b200.trainers as T
    seed, B, L, coef = 312, 12, 7, 0.5
    w = synth.make_weights(seed, bidirectional=True)
    w2i = synth.word_to_idx()
    P, V, R = M.PolicyNetwork(w2i, bidirectional=True), M.ValueNetwork(w2i, bidirectional=True), M.RewardNetwork(w2i, bidirectional=True)
    P.load_state_dict(w["policy"]); V.load_state_dict(w["value"]); R.load_state_dict(w["reward"])
    R.requires_grad_(False)
    R.train(False)
    A = M.AdvantageActorCriticNetwork(V, P).cuda()
    R = R.cuda()
    f, c = synth.make_inputs(seed, B, L)
    u = synth.make_uniforms(seed, L - 1, B)
    np.random.seed(seed)
    mr = T._module_route_step(A, R, f, c, None, entropy_coef=coef)
    ref = a2c_minibatch_entropy(ref_port.Nets(w, bidirectional=True), f, c, u, entropy_coef=coef)
    assert abs(mr.loss - ref["loss"]) <= TOL and abs(mr.mean_entropy - ref["mean_entropy"]) <= TOL
    grads = named_grads(A)
    assert len(grads) == 28
    check_grads_vs_oracle(grads, ref["grads"], GTOL)


# ---------------------------------------------------------------- 6. data parallel

@pytest.mark.parametrize("level", [None, 4])
def test_chain_shards_equal_two_half_batch_ranks(level):
    """chain_shards=2 on one GPU = two ranks of B/2 rows each scaling by 1/(B*S): loss, mean entropy (stats words
    summed, as DataParallelA2C all-reduces them) and gradients."""
    from icrl_b200.engine import A2CEngine
    seed, B, L, coef = 321, 32, 9, 0.3
    A, R, w = make_nets(seed)
    f, c = synth.make_inputs(seed, B, L)
    S = (L - 1) if level is None else level
    u = synth.make_uniforms(seed, S, B)
    e1 = A2CEngine(A, R, entropy_coef=coef)
    gsum, ssum = None, None
    for k in range(2):
        sl = slice(k * B // 2, (k + 1) * B // 2)
        r = e1.step(f[sl], c[sl], uniforms=np.ascontiguousarray(u[:, sl]), level=level, global_rows=B)
        gsum = e1.flat_grad.clone() if gsum is None else gsum + e1.flat_grad
        ssum = r["stats"].clone() if ssum is None else ssum + r["stats"]
    ek = A2CEngine(A, R, chain_shards=2, entropy_coef=coef)
    rk = ek.step(f, c, uniforms=u, level=level)
    assert len(ssum) == 4 and len(rk["stats"]) == 4
    assert abs(rk.loss - float(ssum[0])) <= GTOL and abs(rk.mean_entropy - float(ssum[3])) <= GTOL
    assert float((ek.flat_grad - gsum).abs().max() / gsum.abs().max()) <= GTOL


# ---------------------------------------------------------------- 7. public trainer

@pytest.mark.parametrize("coef", [0.0, 0.01])
def test_train_a2c_network_logs_mean_entropy(tmp_path, monkeypatch, coef):
    import icrl_b200.trainers as T
    seed, n, L = 331, 32, 9
    w = synth.make_weights(seed)
    network_paths = {}
    for k in ("policy", "value", "reward"):
        network_paths[k + "_network"] = str(tmp_path / ("%sNetwork.pt" % k))
        torch.save(w[k], network_paths[k + "_network"])
    network_paths["a2c_network"] = str(tmp_path / "a2cNetwork.pt")
    save_paths = {"model_path": str(tmp_path / "log_a2c.pt"), "results_path": str(tmp_path / "results.txt")}
    f, c = synth.make_inputs(seed, n, L)
    data = {"train_captions": c, "train_image_idxs": np.arange(n), "train_features": f, "train_urls": np.array(["u"] * n),
            "word_to_idx": synth.word_to_idx(), "embeddings": None}
    scalars = {}

    class Rec:
        def __init__(self, *a, **k):
            pass

        def add_scalar(self, tag, val, step):
            scalars[tag.split("episodic-")[-1]] = float(val)

    monkeypatch.setattr(T, "SummaryWriter", Rec)
    np.random.seed(seed)
    T.train_a2c_network(data, save_paths, network_paths, str(tmp_path), False, 1, n, entropy_coef=coef)
    expect = {"loss", "mean-rewards", "mean-advantage"} | ({"mean-entropy"} if coef else set())
    assert set(scalars) == expect, scalars
    if coef:
        assert 0.0 < scalars["mean-entropy"] <= np.log(1004) + 1e-5
    import os
    assert os.path.exists(network_paths["a2c_network"]) and os.path.exists(save_paths["model_path"])
