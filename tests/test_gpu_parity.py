"""GPU parity tests: the CUDA path (through the C ABI) against the golden vectors produced by the
unmodified reference and against the CPU oracle.

Tolerances (fp32 path, stated per BASELINE north_star; measured errors are dumped to
gpurun_out/parity_errors.json -- round 1: values 5.5e-7, rewards 1.1e-7, log-probs 4.8e-7, grads 2.0e-6):
  token ids                      bit-exact
  logits / log-probs             2e-6 abs
  values / rewards               2e-6 abs   (the reference's own formulations differ by ~2e-7)
  loss, mean reward / advantage  2e-6 abs
  gradients                      2e-5 of the tensor's max |entry| (sampled entries) and of its L2 norm
"""
import numpy as np
import pytest
import torch

from oracle import ref_port, single_pass, synth
from tests.helpers import (check_grads_vs_golden, check_grads_vs_oracle, load_case, make_nets, named_grads, GOLDEN)
from oracle.gen_golden import grad_sample_index

pytestmark = pytest.mark.gpu

TOL = 2e-6
GTOL = 2e-5


DECODES = ["fused", "tc", "simt"]     # persistent tcgen05 kernel / per-step tcgen05 GEMMs / per-step fp32 SIMT


def _engine(seed, decode="fused"):
    from icrl_b200.engine import A2CEngine
    A, R, w = make_nets(seed)
    return A2CEngine(A, R, decode=decode), A, R, w


ERRORS = {}


def _record(name, **kv):
    """Measured parity errors, dumped to gpurun_out/parity_errors.json (margin vs the tolerances)."""
    import json, os
    ERRORS.setdefault(name, {}).update({k: float(v) for k, v in kv.items()})
    try:
        os.makedirs("gpurun_out", exist_ok=True)
        json.dump(ERRORS, open("gpurun_out/parity_errors.json", "w"), indent=1, sort_keys=True)
    except OSError:
        pass


def _compare_forward(res, g, name="case"):
    toks = res["tokens"].cpu().numpy()
    assert np.array_equal(toks, g["tokens"]), "token ids differ in %d places" % int((toks != g["tokens"]).sum())
    for k in ("values", "rewards", "logp"):
        err = float(np.abs(res[k].cpu().numpy() - g[k]).max())
        _record(name, **{k: err})
        assert err <= TOL, "%s: %.3e" % (k, err)
    assert abs(res.loss - float(g["loss"])) <= TOL
    assert abs(res.mean_reward - float(g["mean_reward"])) <= TOL
    assert abs(res.mean_adv - float(g["mean_adv"])) <= TOL


@pytest.mark.parametrize("trans", [(0, 1), (0, 0), (1, 0), (1, 1)])
@pytest.mark.parametrize("shape", [(37, 1004, 512), (256, 2048, 512), (2048, 512, 4864), (8, 512, 2048)])
def test_gemm_f32(trans, shape):
    import ctypes
    from icrl_b200 import _lib
    ta, tb = trans
    M, N, K = shape
    rs = np.random.RandomState(0)
    A = torch.from_numpy(rs.standard_normal((K, M) if ta else (M, K)).astype(np.float32)).cuda()
    Bm = torch.from_numpy(rs.standard_normal((N, K) if tb else (K, N)).astype(np.float32)).cuda()
    bias = torch.from_numpy(rs.standard_normal(N).astype(np.float32)).cuda()
    C = torch.zeros((M, N), dtype=torch.float32, device="cuda")
    ws = torch.empty(24 * 2048 * 512, dtype=torch.float32, device="cuda")
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    _lib.call("icrl_gemm_f32", ctypes.c_void_p(torch.cuda.current_stream().cuda_stream), ta, tb, M, N, K, p(A),
              A.shape[1], p(Bm), Bm.shape[1], p(C), N, p(bias), 0.0, p(ws), ws.numel() * 4, None)
    ref = (A.double().t() if ta else A.double()) @ (Bm.double().t() if tb else Bm.double()) + bias.double()
    err = float((C.double() - ref).abs().max() / ref.abs().max())
    assert err < 2e-6, err


@pytest.mark.parametrize("shape", [(128, 256, 512), (4096, 2048, 512), (300, 1004, 512), (8, 2048, 512), (256, 1004, 64)])
def test_gemm_bf16x3_tcgen05(shape):
    """tcgen05 split-bf16 GEMM vs float64: fp32-grade (measured 3.6e-7 of max|C| at K=512, torch fp32 matmul
    8.7e-7) once the full-magnitude term and the correction terms use separate TMEM accumulators
    (gemm_tc.cu header; one shared accumulator gave 3.9e-6 through the tensor core's truncating adds)."""
    import ctypes
    from icrl_b200 import _lib
    M, N, K = shape
    rs = np.random.RandomState(1)
    A = torch.from_numpy(rs.standard_normal((M, K)).astype(np.float32)).cuda()
    Bm = torch.from_numpy((rs.standard_normal((N, K)) / np.sqrt(K)).astype(np.float32)).cuda()
    bias = torch.from_numpy(rs.standard_normal(N).astype(np.float32)).cuda()
    C = torch.full((M, N), float("nan"), dtype=torch.float32, device="cuda")
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    parts = []
    for x in (A, Bm):
        pr = torch.empty((3,) + tuple(x.shape), dtype=torch.bfloat16, device="cuda")
        _lib.call("icrl_split_bf16x3", st, x.numel(), p(x), p(pr), None)
        assert float((x - pr.float().sum(0)).abs().max()) <= 2.0 ** -22 * float(x.abs().max())
        parts.append(pr)
    _lib.call("icrl_gemm_bf16x3", st, M, N, K, p(parts[0]), p(parts[1]), p(C), N, p(bias), None)
    torch.cuda.synchronize()
    ref = A.double() @ Bm.double().t() + bias.double()
    assert torch.isfinite(C).all()
    err = float((C.double() - ref).abs().max() / ref.abs().max())
    _record("gemm_bf16x3_%dx%dx%d" % shape, rel_err=err)
    assert err < 1e-6, err


def test_greedy_config1():
    """BASELINE config 1: greedy decode, B=32, 16 steps."""
    import icrl_b200.trainers as T
    g = np.load(GOLDEN + "/greedy_b32.npz")
    A, R, w = make_nets(0)
    f, _ = synth.make_inputs(0, 32, 17)
    toks = T.GenerateCaptionsGreedy(f, np.ones((32, 17), dtype=np.int64), A.policy_network)
    assert tuple(toks.shape) == (32, 17) and toks.dtype == torch.int64
    assert np.array_equal(toks.cpu().numpy(), g["tokens"])
    _, last = A.policy_network._icrl_greedy.greedy_decode(f, np.ones(32), 16)
    assert float(np.abs(last.cpu().numpy() - g["last_logits"]).max()) <= TOL


@pytest.mark.parametrize("decode", DECODES)
@pytest.mark.parametrize("name", ["a2c_b8_l6", "a2c_b32_l9", "curr_b16_l10_lv4", "curr_b24_l20_lv6"])
def test_a2c_step_vs_reference_golden(name, decode):
    g, seed, f, c, u, level = load_case(name)
    eng, A, R, w = _engine(seed, decode)
    res = eng.step(f, c, uniforms=u, level=level)
    _compare_forward(res, g, name + "_" + decode)
    _record(name + "_" + decode, grad_worst=check_grads_vs_golden(named_grads(A), g, GTOL))


@pytest.mark.parametrize("decode", DECODES)
def test_a2c_config2_vs_reference_golden(decode):
    """BASELINE config 2: B=256, L=20, S=19, fixed uniforms."""
    g, seed, f, c, u, level = load_case("a2c_b256_l20")
    eng, A, R, w = _engine(seed, decode)
    res = eng.step(f, c, uniforms=u, backward=False)
    _compare_forward(res, g, "a2c_b256_l20_" + decode)
    last = eng._bufs["p_logits"][18 * 256 * 1004:19 * 256 * 1004].view(256, 1004).cpu().numpy()
    assert float(np.abs(last[g["last_logits_rows"]] - g["last_logits"]).max()) <= TOL
    res = eng.step(f, c, uniforms=u)
    _compare_forward(res, g, "a2c_b256_l20")
    _record("a2c_b256_l20", grad_worst=check_grads_vs_golden(named_grads(A), g, GTOL))


def test_sampling_from_global_numpy_stream():
    """uniforms=None consumes np.random's global stream like np.random.choice (trainers.py:447-450)."""
    g, seed, f, c, u, level = load_case("a2c_b8_l6")
    eng, A, R, w = _engine(seed)
    np.random.seed(seed)
    res = eng.step(f, c, backward=False)
    assert np.array_equal(res["tokens"].cpu().numpy(), g["tokens"])


def test_step_vs_oracle_fresh_case():
    """A case no fixture covers, checked against the CPU oracle on this box (B=48, L=12, level 5)."""
    seed, B, L, level = 21, 48, 12, 5
    eng, A, R, w = _engine(seed)
    f, c = synth.make_inputs(seed, B, L)
    u = synth.make_uniforms(seed, level, B)
    ref = single_pass.a2c_minibatch(w, f, c, u, level=level, lib=True)
    res = eng.step(f, c, uniforms=u, level=level)
    assert np.array_equal(res["tokens"].cpu().numpy(), ref["tokens"])
    for k in ("values", "rewards", "logp"):
        assert float(np.abs(res[k].cpu().numpy() - ref[k]).max()) <= TOL, k
    assert abs(res.loss - ref["loss"]) <= TOL
    check_grads_vs_oracle(named_grads(A), ref["grads"], GTOL)


def test_curriculum_level_too_long_is_skipped():
    eng, A, R, w = _engine(1)
    f, c = synth.make_inputs(1, 8, 6)
    assert eng.step(f, c, level=6) is None          # caplen - level < 1 (trainers.py:550)


def test_get_rewards_config3_shape():
    import icrl_b200.trainers as T
    g = np.load(GOLDEN + "/rewards_b64_l20.npz")
    eng, A, R, w = _engine(6)
    f, c = synth.make_inputs(6, 64, 20)
    r = eng.get_rewards(f, c)
    assert float(np.abs(r.cpu().numpy() - g["rewards"]).max()) <= TOL
    # module path (carried state, reset by init_hidden) gives the same numbers
    R.rewrnn.init_hidden()
    r2 = T.GetRewards(torch.from_numpy(f).cuda(), torch.from_numpy(c).cuda(), R)
    assert float(np.abs(r2.cpu().numpy() - g["rewards"]).max()) <= TOL


def test_module_forward_semantics_vs_port():
    """Per-call module API: growing prefix, hidden state carried across calls until init_hidden()."""
    seed, B = 9, 12
    A, R, w = make_nets(seed)
    nets = ref_port.Nets(w, requires_grad=False)
    f, c = synth.make_inputs(seed, B, 7)
    ft, ct = torch.from_numpy(f), torch.from_numpy(c)
    A.value_network.valrnn.init_hidden()
    R.rewrnn.init_hidden()
    with torch.no_grad():
        for n in (1, 2, 4):
            v_ref = ref_port.value_call(nets, ft, ct[:, :n]).numpy()
            r_ref = ref_port.reward_call(nets, ft, ct[:, :n + 1]).numpy()
            z_ref = ref_port.policy_logits(nets, ft, ct[:, :n]).numpy()
            v, z = A(ft.cuda(), ct[:, :n].cuda())
            import icrl_b200.trainers as T
            r = T.GetRewards(ft.cuda(), ct[:, :n + 1].cuda(), R)
            assert tuple(v.shape) == (B, 1) and tuple(z.shape) == (B, 1, 1004)
            assert float(np.abs(v.cpu().numpy() - v_ref).max()) <= TOL
            assert float(np.abs(r.cpu().numpy() - r_ref).max()) <= TOL
            assert float(np.abs(z.cpu().numpy()[:, 0] - z_ref[:, -1]).max()) <= TOL
        full = A.policy_network(ft.cuda().unsqueeze(0), ct[:, :5].cuda())
        assert tuple(full.shape) == (B, 5, 1004)
        assert float(np.abs(full.cpu().numpy() - ref_port.policy_logits(nets, ft, ct[:, :5]).numpy()).max()) <= TOL


def test_determinism_and_row_independence_full_size():
    """Size-independent properties at a BASELINE-scale batch (B=1024, L=20): two runs agree bit for
    bit on tokens / values / rewards, rewards lie in [-1,1], and the policy's tokens for a row shard
    equal the same rows of the full batch (rows are independent in the policy; SURVEY 8e)."""
    seed, B, L = 31, 1024, 20
    eng, A, R, w = _engine(seed)
    f, c = synth.make_inputs(seed, B, L)
    u = synth.make_uniforms(seed, L - 1, B)
    r1 = eng.step(f, c, uniforms=u)
    t1, v1, w1 = r1["tokens"].clone(), r1["values"].clone(), r1["rewards"].clone()
    g1 = eng.flat_grad.clone()
    r2 = eng.step(f, c, uniforms=u)
    assert torch.equal(t1, r2["tokens"]) and torch.equal(v1, r2["values"]) and torch.equal(w1, r2["rewards"])
    assert float((g1 - eng.flat_grad).abs().max()) <= 1e-6 * float(g1.abs().max())   # atomics reorder only
    assert float(w1.abs().max()) <= 1.0 + 1e-6
    assert torch.isfinite(eng.flat_grad).all()
    r3 = eng.step(f[256:512], c[256:512], uniforms=u[:, 256:512], backward=False)
    assert torch.equal(r3["tokens"], t1[256:512])


def test_decode_paths_agree_large_batch():
    """B=2048 (16 clusters of the persistent kernel, ragged last tile at B=2000): the fused tcgen05 kernel and
    the fp32 SIMT path sample the same tokens from the same uniforms, greedy and forced modes included."""
    seed, B, L = 41, 2000, 20
    f, c = synth.make_inputs(seed, B, L)
    u = synth.make_uniforms(seed, L - 1, B)
    ef, A, R, w = _engine(seed, "fused")
    from icrl_b200.engine import A2CEngine
    es = A2CEngine(A, R, decode="simt")
    rf = ef.step(f, c, uniforms=u, backward=False)
    rs = es.step(f, c, uniforms=u, backward=False)
    nflip = int((rf["tokens"] != rs["tokens"]).sum())
    _record("decode_agree_b2000", flips=nflip, logp=float((rf["logp"] - rs["logp"]).abs().max()))
    assert nflip == 0
    assert float((rf["logp"] - rs["logp"]).abs().max()) <= TOL
    gf = ef.step(f, c, greedy=True, backward=False)
    gs = es.step(f, c, greedy=True, backward=False)
    assert torch.equal(gf["tokens"], gs["tokens"])
    forced = rs["tokens"].cpu().numpy()
    ff = ef.step(f, c, forced_tokens=forced, backward=False)
    assert torch.equal(ff["tokens"], rs["tokens"])
    assert float((ff["logp"] - rs["logp"]).abs().max()) <= TOL


@pytest.mark.parametrize("name", ["a2c_b8_l6", "curr_b16_l10_lv4"])
def test_reference_rollout_loop_trains_dropin_modules(name):
    """The reference's own loop body (trainers.py:428-480 / 544-594, restated verbatim below) run on the drop-in
    modules with torch autograd: module outputs carry autograd history (SURVEY 8b / H8), the value RNN's
    hidden_cell keeps its graph from call to call, and loss.backward() reaches all 18 parameters with the
    gradients of the unmodified reference (golden fixtures)."""
    import icrl_b200.trainers as T
    from torch.nn import functional as F
    g, seed, f, c, u, level = load_case(name)
    A, R, w = make_nets(seed)
    R.requires_grad_(False)
    features = torch.tensor(f, device="cuda").float()
    captions = torch.tensor(c, device="cuda").long()
    caplen = int(np.nonzero(c == 2)[1].max() + 1)
    if level is None:
        captions_in, steps = captions[:, :1], caplen - 1
    else:
        captions_in, steps = captions[:, :caplen - level], level
    np.random.seed(seed)
    A.value_network.valrnn.init_hidden()
    R.rewrnn.init_hidden()
    values, rewards, log_probs = [], [], []
    for step in range(steps):
        value, probs = A(features, captions_in)
        probs = F.softmax(probs, dim=2)
        dist = probs.cpu().detach().numpy()[:, 0]
        actions = [np.random.choice(probs.shape[-1], p=dist[i]) for i in range(captions.shape[0])]
        gen_cap = torch.from_numpy(np.array(actions)).unsqueeze(-1).to(captions_in.device)
        captions_in = torch.cat((captions_in, gen_cap), axis=1)
        log_prob = torch.log(probs[:, 0, :].gather(1, gen_cap))
        reward = T.GetRewards(features, captions_in, R)
        values.append(value)
        rewards.append(reward)
        log_probs.append(log_prob)
    values = torch.stack(values, axis=1).squeeze()
    rewards = torch.stack(rewards, axis=1).squeeze()
    log_probs = torch.stack(log_probs, axis=1).squeeze()
    advantage = values - rewards
    loss = (-log_probs * advantage).mean() + 0.5 * advantage.pow(2).mean()
    for p in A.parameters():
        p.grad = None
    loss.mean().backward(retain_graph=True)
    p0 = captions_in.shape[1] - steps
    assert np.array_equal(captions_in[:, p0:].cpu().numpy(), g["tokens"])
    assert float(np.abs(values.detach().cpu().numpy() - g["values"]).max()) <= TOL
    assert float(np.abs(rewards.detach().cpu().numpy() - g["rewards"]).max()) <= TOL
    assert abs(float(loss) - float(g["loss"])) <= TOL
    assert all(p.grad is not None for p in A.parameters())
    _record(name + "_autograd_loop", grad_worst=check_grads_vs_golden(named_grads(A), g, GTOL))


@pytest.mark.parametrize("shards", [2, 4, 8])
@pytest.mark.parametrize("level", [None, 4])
def test_chain_shards_equal_independent_shard_runs(shards, level):
    """chain_shards=K (K value/reward recurrences in lockstep, each from zero state) must equal K independent
    single-chain runs on the row shards with the global loss normalisation and summed gradients -- the N-rank
    data-parallel oracle of SURVEY 8e, which tests/test_oracle_golden.py pins to the reference on CPU."""
    from icrl_b200.engine import A2CEngine
    seed, B, L = 51, 32, 9
    A, R, w = make_nets(seed)
    f, c = synth.make_inputs(seed, B, L)
    S = (L - 1) if level is None else level
    u = synth.make_uniforms(seed, S, B)
    e1 = A2CEngine(A, R, chain_shards=1)
    Bs = B // shards
    gsum, vals, rews, toks = None, [], [], []
    for k in range(shards):
        sl = slice(k * Bs, (k + 1) * Bs)
        r = e1.step(f[sl], c[sl], uniforms=np.ascontiguousarray(u[:, sl]), level=level, global_rows=B)
        vals.append(r["values"].clone()); rews.append(r["rewards"].clone()); toks.append(r["tokens"].clone())
        gsum = e1.flat_grad.clone() if gsum is None else gsum + e1.flat_grad
    ek = A2CEngine(A, R, chain_shards=shards)
    rk = ek.step(f, c, uniforms=u, level=level)
    assert torch.equal(rk["tokens"], torch.cat(toks))
    assert float((rk["values"] - torch.cat(vals)).abs().max()) <= TOL
    assert float((rk["rewards"] - torch.cat(rews)).abs().max()) <= TOL
    err = float((ek.flat_grad - gsum).abs().max() / gsum.abs().max())
    _record("chain_shards_%d_%s" % (shards, level), grad_rel=err)
    assert err <= GTOL


def test_lookahead_beam_vs_reference_golden():
    """SURVEY 8f row 1: value-guided beam look-ahead (trainers.py:73-105) on the drop-in modules vs the unmodified
    reference: all 5 final candidate caption batches identical, scores within 2e-5 (16 steps of accumulated
    0.6 V + 0.4 log(logit); the value RNN state is carried through all ~400 calls)."""
    import icrl_b200.trainers as T
    g = np.load(GOLDEN + "/lookahead_b6.npz")
    seed, B, beam = int(g["seed"]), int(g["B"]), int(g["beam"])
    A, R, w = make_nets(seed)
    f, _ = synth.make_inputs(seed, B, 17)
    A.value_network.valrnn.init_hidden()
    cands = T.GenerateCaptionsWithActorCriticLookAhead(f, np.ones((B, 17), dtype=np.int64), A.policy_network,
                                                       A.value_network, beamSize=beam, most_likely=False)
    assert len(cands) == beam
    for k, (cap, score) in enumerate(cands):
        assert np.array_equal(cap.cpu().numpy(), g["captions"][k]), "candidate %d differs" % k
        ref = g["scores"][k]
        got = score.cpu().numpy().reshape(-1)
        assert np.array_equal(np.isnan(got), np.isnan(ref))
        ok = ~np.isnan(ref)
        assert float(np.abs(got[ok] - ref[ok]).max()) <= 2e-5
    best = T.GenerateCaptionsWithActorCriticLookAhead(f, np.ones((B, 17), dtype=np.int64), A.policy_network,
                                                      A.value_network, most_likely=True)
    assert tuple(best.shape) == (B, 17)


@pytest.mark.parametrize("B,L,level", [(37, 7, None), (130, 6, 3), (5, 20, None)])
def test_ragged_batch_sizes_vs_oracle(B, L, level):
    """Batch sizes that fill no tile exactly (the decode kernel pads rows to 128 per cluster, the chains are
    serial in B): tokens bit-exact and values / rewards / log-probs / gradients within tolerance of the CPU oracle."""
    seed = 60 + B
    eng, A, R, w = _engine(seed)
    f, c = synth.make_inputs(seed, B, L)
    S = (L - 1) if level is None else level
    u = synth.make_uniforms(seed, S, B)
    ref = single_pass.a2c_minibatch(w, f, c, u, level=level, lib=True)
    res = eng.step(f, c, uniforms=u, level=level)
    assert np.array_equal(res["tokens"].cpu().numpy(), ref["tokens"])
    for k in ("values", "rewards", "logp"):
        assert float(np.abs(res[k].cpu().numpy() - ref[k]).max()) <= TOL, k
    check_grads_vs_oracle(named_grads(A), ref["grads"], GTOL)


def test_config3_rewards_full_size_properties():
    """BASELINE config 3 at full size (8192 captions x 20 tokens = 163,840 serial GRU steps): deterministic,
    finite, inside [-1, 1]; and the first rows agree with a run on a batch that shares the first column block
    only up to the point where the streams diverge (the chain is causal in stream order)."""
    import time
    seed, B, L = 71, 8192, 20
    eng, A, R, w = _engine(seed)
    f, c = synth.make_inputs(seed, B, L)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r1 = eng.get_rewards(f, c)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    r2 = eng.get_rewards(f, c)
    assert torch.equal(r1, r2)
    assert torch.isfinite(r1).all() and float(r1.abs().max()) <= 1.0 + 1e-6
    _record("config3_rewards_b8192", seconds=dt, captions_per_s=B / dt)
    # causality: a single-column batch is a prefix of the stream of any batch that starts with the same column
    r_a = eng.get_rewards(f[:64], c[:64, :1])
    r_b = eng.get_rewards(f[:64], np.concatenate([c[:64, :1], c[:64, 1:2]], axis=1))
    assert tuple(r_a.shape) == (64, 1) and tuple(r_b.shape) == (64, 1)


def test_curriculum_full_size_properties():
    """BASELINE config 5 local shape (1024 rows per rank, L=20) at two curriculum levels: finite gradients,
    deterministic tokens, loss equals mean(-logp*adv) + 0.5*mean(adv^2) recomputed from the returned tensors."""
    seed, B, L = 73, 1024, 20
    eng, A, R, w = _engine(seed)
    f, c = synth.make_inputs(seed, B, L)
    for level in (3, 12):
        u = synth.make_uniforms(seed + level, level, B)
        r = eng.step(f, c, uniforms=u, level=level)
        assert r["tokens"].shape == (B, level)
        adv = (r["values"] - r["rewards"]).double()
        loss = float((-r["logp"].double() * adv).mean() + 0.5 * (adv ** 2).mean())
        assert abs(loss - r.loss) <= 1e-6
        assert torch.isfinite(eng.flat_grad).all()
        r2 = eng.step(f, c, uniforms=u, level=level, backward=False)
        assert torch.equal(r["tokens"], r2["tokens"])


def _pretrain_case():
    g = np.load(GOLDEN + "/pretrain_b12.npz")
    seed, B = int(g["seed"]), int(g["B"])
    w = synth.make_weights(seed)
    f, c = synth.make_inputs(seed, B, 17)
    data = {"train_captions": c, "train_image_idxs": np.arange(B), "train_features": f,
            "train_urls": np.array(["u"] * B), "word_to_idx": synth.word_to_idx(), "embeddings": None}
    return g, seed, B, w, data


def _check_pretrain_grads(net, g, key, tol=GTOL):
    worst = 0.0
    for k, p_ in net.named_parameters():
        assert p_.grad is not None, k
        flat = p_.grad.detach().float().cpu().numpy().reshape(-1)
        ref = g["%s/gsamp/%s" % (key, k)]
        got = flat[grad_sample_index(flat.size)]
        err = float(np.abs(got - ref).max()) / max(float(np.abs(ref).max()), 1e-12)
        worst = max(worst, err)
        assert err <= tol, "%s %s: %.3e" % (key, k, err)
        nrm = float(np.sqrt((flat.astype(np.float64) ** 2).sum()))
        assert abs(nrm - float(g["%s/gnorm/%s" % (key, k)])) <= tol * max(float(g["%s/gnorm/%s" % (key, k)]), 1e-12), k
    return worst


@pytest.mark.parametrize("key", ["policy", "reward", "value"])
def test_pretraining_loops_vs_reference_golden(key, tmp_path, monkeypatch):
    """SURVEY 8f row 2: one minibatch of train_policy_network / train_reward_network / train_value_network on the
    drop-in modules (autograd through the CUDA kernels, GRU BPTT included) against the unmodified reference: loss and
    all gradients.  As in the golden generator, the loops' own network constructors are wrapped to load the
    synthetic weights."""
    import random
    import icrl_b200.trainers as T
    g, seed, B, w, data = _pretrain_case()
    paths = {k: str(tmp_path / (k + ".pt")) for k in ("policy_network", "reward_network", "value_network")}
    torch.save(w["policy"], paths["policy_network"])
    torch.save(w["reward"], paths["reward_network"])

    def factory(cls, sd):
        def make(*a, **k):
            net = cls(*a, **k)
            net.load_state_dict(sd)
            return net
        return make

    losses = []

    class Rec:
        def __init__(self, *a, **k):
            pass

        def add_scalar(self, tag, val, step):
            losses.append(float(val))

    monkeypatch.setattr(T, "PolicyNetwork", factory(T.PolicyNetwork, w["policy"]))
    monkeypatch.setattr(T, "ValueNetwork", factory(T.ValueNetwork, w["value"]))
    monkeypatch.setattr(T, "RewardNetwork", factory(T.RewardNetwork, w["reward"]))
    monkeypatch.setattr(T, "SummaryWriter", Rec)
    monkeypatch.setattr(T.torch, "randperm", lambda n: torch.arange(n))
    random.seed(seed)
    fn = {"policy": T.train_policy_network, "reward": T.train_reward_network, "value": T.train_value_network}[key]
    net = fn(data, paths, str(tmp_path), False, epochs=1, batch_size=B)
    ref_loss = float(g[key + "_loss"])
    assert abs(losses[0] - ref_loss) <= 2e-6 * max(1.0, abs(ref_loss)), (losses[0], ref_loss)
    # gradients survive the optimizer step (zero_grad precedes backward in the loops)
    _record("pretrain_" + key, loss=losses[0], grad_worst=_check_pretrain_grads(net, g, key))


def test_frozen_pretrained_embeddings_variant_vs_reference_golden():
    """SURVEY 8f row 3 (first half): `pretrained_embeddings` given -> frozen 300-d word vectors, 300-wide LSTM / GRU
    inputs (models.py:61-63, 113-115, 208-210).  One A2C minibatch through the fused engine against the unmodified
    reference: tokens bit-exact, values / rewards / log-probs / loss within tolerance, the 16 trainable gradients
    match and the frozen tables get none."""
    import icrl_b200.models as M
    from icrl_b200.engine import A2CEngine
    g = np.load(GOLDEN + "/a2c_b16_l8_wemb300.npz")
    seed, B, L, D = int(g["seed"]), int(g["B"]), int(g["L"]), int(g["wordvec_dim"])
    w = synth.make_weights(seed, wordvec_dim=D)
    w2i = synth.word_to_idx()
    P = M.PolicyNetwork(w2i, pretrained_embeddings=w["policy"]["caption_embedding.weight"].numpy())
    V = M.ValueNetwork(w2i, pretrained_embeddings=w["value"]["valrnn.caption_embedding.weight"].numpy())
    R = M.RewardNetwork(w2i, pretrained_embeddings=w["reward"]["rewrnn.caption_embedding.weight"].numpy())
    P.load_state_dict(w["policy"]); V.load_state_dict(w["value"]); R.load_state_dict(w["reward"])
    assert P.lstm.weight_ih_l0.shape == (2048, D) and not P.caption_embedding.weight.requires_grad
    R.requires_grad_(False)
    A = M.AdvantageActorCriticNetwork(V, P).cuda()
    R = R.cuda()
    f, c = synth.make_inputs(seed, B, L)
    u = synth.make_uniforms(seed, L - 1, B)
    eng = A2CEngine(A, R)
    res = eng.step(f, c, uniforms=u)
    _compare_forward(res, g, "a2c_b16_l8_wemb300")
    grads = {k: p.grad.detach().float().cpu().numpy() for k, p in A.named_parameters() if p.requires_grad}
    assert len(grads) == 16 and A.policy_network.caption_embedding.weight.grad is None
    _record("a2c_b16_l8_wemb300", grad_worst=check_grads_vs_golden(grads, g, GTOL))


def test_odd_vocabulary_falls_back_to_per_step_decode():
    """A vocabulary the persistent decode kernel cannot hold (V % 4 != 0) still trains: the engine switches to the
    per-step kernels (with a warning) and matches the CPU oracle."""
    import warnings
    import icrl_b200.models as M
    from icrl_b200.engine import A2CEngine
    seed, B, L, V = 81, 10, 6, 203
    w = synth.make_weights(seed, vocab=V)
    w2i = synth.word_to_idx(V)
    P, Vn, R = M.PolicyNetwork(w2i), M.ValueNetwork(w2i), M.RewardNetwork(w2i)
    P.load_state_dict(w["policy"]); Vn.load_state_dict(w["value"]); R.load_state_dict(w["reward"])
    R.requires_grad_(False)
    A = M.AdvantageActorCriticNetwork(Vn, P).cuda()
    f, c = synth.make_inputs(seed, B, L, vocab=V)
    u = synth.make_uniforms(seed, L - 1, B)
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter("always")
        eng = A2CEngine(A, R.cuda())
    assert eng.decode == "simt" and any("fused decode" in str(x.message) for x in rec)
    ref = single_pass.a2c_minibatch(w, f, c, u, lib=True)
    res = eng.step(f, c, uniforms=u)
    assert np.array_equal(res["tokens"].cpu().numpy(), ref["tokens"])
    for k in ("values", "rewards", "logp"):
        assert float(np.abs(res[k].cpu().numpy() - ref[k]).max()) <= TOL, k
    check_grads_vs_oracle(named_grads(A), ref["grads"], GTOL)


def test_bidirectional_variant_vs_reference_golden(tmp_path, monkeypatch):
    """SURVEY 8f row 3 (second half): bidirectional=True networks (models.py:59-78, 120-128, 163-172, 215-221, 247-251)
    on the module route.  One A2C minibatch driven by icrl_b200.trainers.a2c_training -- which switches to the
    reference-style loop for bidirectional networks -- against the unmodified reference: loss, mean reward / advantage
    and all 28 gradients (reverse-direction RNN weights, rnn_linear, 1024-wide cnn2linear / linear2vocab included)."""
    import icrl_b200.models as M
    import icrl_b200.trainers as T
    g = np.load(GOLDEN + "/a2c_b12_l7_bidir.npz")
    seed, B, L = int(g["seed"]), int(g["B"]), int(g["L"])
    w = synth.make_weights(seed, bidirectional=True)
    w2i = synth.word_to_idx()
    P, V, R = M.PolicyNetwork(w2i, bidirectional=True), M.ValueNetwork(w2i, bidirectional=True), M.RewardNetwork(w2i, bidirectional=True)
    P.load_state_dict(w["policy"]); V.load_state_dict(w["value"]); R.load_state_dict(w["reward"])
    assert V.valrnn.hidden_cell[0].shape == (2, 1, 512) and P.linear2vocab.weight.shape == (1004, 1024)
    R.requires_grad_(False)
    R.train(False)
    A = M.AdvantageActorCriticNetwork(V, P).cuda()
    R = R.cuda()
    f, c = synth.make_inputs(seed, B, L)
    data = {"train_captions": c, "train_image_idxs": np.arange(B), "train_features": f, "train_urls": np.array(["u"] * B)}
    scalars = {}

    class Rec:
        def __init__(self, *a, **k):
            pass

        def add_scalar(self, tag, val, step):
            scalars[tag.split("episodic-")[-1]] = float(val)

    monkeypatch.setattr(T, "SummaryWriter", Rec)
    monkeypatch.setattr(T.torch, "randperm", lambda n: torch.arange(n))
    opt = torch.optim.SGD(A.parameters(), lr=0.0)                   # keeps the weights, gradients stay in .grad
    np.random.seed(seed)
    T.a2c_training(data, A, R, opt, str(tmp_path), [str(tmp_path / "a.pt")], B, 1)
    assert abs(scalars["loss"] - float(g["loss"])) <= TOL, scalars
    assert abs(scalars["mean-rewards"] - float(g["mean_reward"])) <= TOL
    assert abs(scalars["mean-advantage"] - float(g["mean_adv"])) <= TOL
    grads = named_grads(A)
    assert len(grads) == 28
    _record("a2c_b12_l7_bidir", grad_worst=check_grads_vs_golden(grads, g, GTOL))
    # greedy decode of a bidirectional policy goes through the module route too
    toks = T.GenerateCaptionsGreedy(f, np.ones((B, 17), dtype=np.int64), A.policy_network)
    assert tuple(toks.shape) == (B, 17)


def test_three_optimizer_steps_track_the_cpu_port():
    """Training trajectory: three A2C minibatches with Adam between them (weights change, derived operands -- gate
    tables, fp16 weight splits, collapsed value head -- must be rebuilt every step) against the as-executed CPU port
    with the same optimizer: token ids bit-exact at every step, losses within 1e-5.  Final weights: Adam turns a
    gradient entry into a step of ~lr whatever its size, so an entry whose true gradient is below the fp32 noise
    floor may step the other way on the two sides; hence the check is that at most 1 % of a tensor's entries differ
    by more than 1e-5 and none by more than the 3-step Adam budget."""
    seed, B, L = 91, 8, 6
    eng, A, R, w = _engine(seed)
    nets = ref_port.Nets(w)
    opt_g = torch.optim.Adam(A.parameters(), lr=1e-3)
    opt_c = torch.optim.Adam([p for _, p in nets.named_trainable()], lr=1e-3)
    for it in range(3):
        f, c = synth.make_inputs(seed + it, B, L)
        u = synth.make_uniforms(seed + it, L - 1, B)
        ref = ref_port.a2c_minibatch(nets, f, c, u)
        opt_c.step()
        res = eng.step(f, c, uniforms=u)
        opt_g.step()
        assert np.array_equal(res["tokens"].cpu().numpy(), ref["tokens"]), "step %d" % it
        assert abs(res.loss - ref["loss"]) <= 1e-5, (it, res.loss, ref["loss"])
    cpu = dict(nets.named_trainable())
    for k, p in A.named_parameters():
        d = (p.detach().cpu() - cpu[k].detach()).abs()
        assert float(d.max()) <= 3.5e-3, (k, float(d.max()))
        assert float((d > 1e-5).float().mean()) <= 0.01, (k, float((d > 1e-5).float().mean()))


@pytest.mark.parametrize("T", [64, 1000, 48640])
def test_wgrad_tcgen05_vs_float64(T):
    """tcgen05 weight-gradient contraction dW = A^T B (time-major fp32 operands, per-column scaling, fp16-split MMAs,
    TMEM flushed to registers every 512 K elements) against float64, with gradient-like magnitudes (columns of A span
    ten orders of magnitude)."""
    import ctypes
    from icrl_b200 import _lib
    M, N = 2048, 512
    rs = np.random.RandomState(T)
    colscale = 10.0 ** rs.uniform(-12, -3, size=M)
    A = torch.from_numpy((rs.standard_normal((T, M)) * colscale).astype(np.float32)).cuda()
    B = torch.from_numpy(np.tanh(rs.standard_normal((T, N))).astype(np.float32)).cuda()
    C = torch.full((M, N), float("nan"), device="cuda")
    nbytes = int(_lib.call("icrl_wgrad_tc_ws_bytes", M, N, T, 2))
    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    _lib.call("icrl_wgrad_tc", ctypes.c_void_p(torch.cuda.current_stream().cuda_stream), M, N, T, p(A), M, p(B), N, p(C), N,
              p(ws), nbytes, 2, None)
    torch.cuda.synchronize()
    ref = A.double().t() @ B.double()
    assert torch.isfinite(C).all()
    # every ROW (gate index) is checked against its own scale: the per-column scaling must keep tiny rows accurate
    err = ((C.double() - ref).abs().max(dim=1).values / ref.abs().max(dim=1).values.clamp_min(1e-300)).max().item()
    _record("wgrad_tc_T%d" % T, rel_err_per_row=err)
    assert err < 2e-6, err


def test_flat_adam_matches_torch():
    """SURVEY 8f row 4: the one-kernel Adam over the flat buckets against torch.optim.Adam (the reference's optimizer,
    trainers.py:378) over three training steps from identical gradients."""
    from icrl_b200.engine import A2CEngine
    from icrl_b200.optim import FlatAdam
    seed, B, L = 95, 8, 6
    A1, R1, w = make_nets(seed)
    A2, R2, _ = make_nets(seed)
    e1, e2 = A2CEngine(A1, R1), A2CEngine(A2, R2)
    o1 = torch.optim.Adam(A1.parameters(), lr=1e-3)
    o2 = FlatAdam(e2, lr=1e-3)
    for it in range(3):
        f, c = synth.make_inputs(seed + it, B, L)
        u = synth.make_uniforms(seed + it, L - 1, B)
        e1.step(f, c, uniforms=u)
        e2.flat_grad.copy_(e1.flat_grad)            # identical gradients: this test isolates the optimizer
        o1.step()
        o2.step()
        for (k, p1), (_, p2) in zip(A1.named_parameters(), A2.named_parameters()):
            d = float((p1 - p2).abs().max())
            assert d <= 5e-7, (it, k, d)            # one float ulp of the largest weights (|w| < 4)
            p2.data.copy_(p1.data)                  # keep both sides on the same trajectory
    assert A2.policy_network.linear2vocab.weight.data_ptr() >= o2.flat_param.data_ptr()      # parameters live in the flat buffer
    # the kernels must run on parameters that live inside the flat buffer (16-byte accesses: every tensor, including
    # the ones behind the 1-element linear2.bias, starts on a 256-byte boundary of the bucket)
    assert all(p.data_ptr() % 256 == 0 for p in A2.parameters())
    f, c = synth.make_inputs(seed + 7, B, L)
    u = synth.make_uniforms(seed + 7, L - 1, B)
    r1, r2 = e1.step(f, c, uniforms=u), e2.step(f, c, uniforms=u)
    assert torch.equal(r1["tokens"], r2["tokens"]) and abs(r1.loss - r2.loss) <= TOL
    assert float((e1.flat_grad - e2.flat_grad).abs().max() / e1.flat_grad.abs().max()) <= 1e-6


def test_config4_full_size_properties():
    """BASELINE config 4 at its full single-GPU size (4096 rows, L=20: 778,240 + 856,064 serial steps): the loss equals
    the reference's formula recomputed from the returned tensors, gradients are finite, rewards lie in [-1, 1], and --
    rows being independent in the policy -- the tokens of a 512-row data-parallel shard equal those rows of the full batch."""
    seed, B, L = 97, 4096, 20
    eng, A, R, w = _engine(seed)
    f, c = synth.make_inputs(seed, B, L)
    u = synth.make_uniforms(seed, L - 1, B)
    r = eng.step(f, c, uniforms=u)
    adv = (r["values"] - r["rewards"]).double()
    loss = float((-r["logp"].double() * adv).mean() + 0.5 * (adv ** 2).mean())
    assert abs(loss - r.loss) <= 1e-6
    assert torch.isfinite(eng.flat_grad).all() and float(eng.flat_grad.abs().max()) > 0
    assert float(r["rewards"].abs().max()) <= 1.0 + 1e-6
    toks = r["tokens"].clone()
    rs = eng.step(f[1024:1536], c[1024:1536], uniforms=np.ascontiguousarray(u[:, 1024:1536]), backward=False)
    assert torch.equal(rs["tokens"], toks[1024:1536])


# ---------------------------------------------------------------------------------------------------------------
# chain pieces: the single carried-state chain advanced as lockstep pieces on tcgen05 (chain_tc.cu) with a discarded,
# verified warm-up.

def _seg_engines(seed, segments, warm, tol=1e-5, **kw):
    from icrl_b200.engine import A2CEngine
    A, R, w = make_nets(seed)
    return (A2CEngine(A, R, chain_segments=1),
            A2CEngine(A, R, chain_segments=segments, chain_warmup=warm, chain_tol=tol, **kw), A)


@pytest.mark.parametrize("name", ["a2c_b32_l9", "curr_b24_l20_lv6", "a2c_b256_l20"])
def test_chain_pieces_vs_reference_golden(name):
    """The unmodified reference's numbers (one carried-state chain over the whole batch) reproduced by the default
    engine: the chains cut into tcgen05 pieces (a 64-position first warm-up, lengthened by the joint check where a
    chain needs more): same tolerances as the serial kernels, no fall-back to them."""
    from icrl_b200.engine import A2CEngine
    g, seed, f, c, u, level = load_case(name)
    A, R, w = make_nets(seed)
    eng = A2CEngine(A, R, chain_warmup=64)
    res = eng.step(f, c, uniforms=u, level=level)
    st = eng.segment_stats
    assert eng.piece_layout is not None and st["segmented_steps"] >= 1 and st["fallbacks"] == 0, (eng.piece_layout, st)
    _compare_forward(res, g, name + "_pieces")
    _record(name + "_pieces", grad_worst=check_grads_vs_golden(named_grads(A), g, GTOL), reruns=st["reruns"],
            pieces_v=eng.piece_layout["v"][0], warm_v=eng.piece_layout["v"][2], warm_r=eng.piece_layout["r"][2])


@pytest.mark.parametrize("pieces,B,L,level,warm", [(None, 64, 10, None, 96), (7, 64, 8, None, 96), (2, 48, 7, None, 96),
                                                    (130, 96, 14, 5, 160), (300, 512, 12, None, 160), (None, 256, 20, 7, 160)])
def test_chain_pieces_equal_the_serial_chain(pieces, B, L, level, warm):
    """tcgen05 pieces and serial kernels on the same inputs: identical tokens, values / rewards within 2e-6, gradients
    within 2e-5 of the bucket's largest entry -- for piece counts that do not fill a cluster (7, 2), that straddle
    clusters (130, 300) and for the automatic layout."""
    seed = 131 + (pieces or 0)
    e1, ek, A = _seg_engines(seed, 32, warm, chain_pieces=pieces)
    f, c = synth.make_inputs(seed, B, L)
    S = (L - 1) if level is None else level
    u = synth.make_uniforms(seed, S, B)
    r1 = e1.step(f, c, uniforms=u, level=level)
    v1, w1, g1 = r1["values"].clone(), r1["rewards"].clone(), e1.flat_grad.clone()
    assert e1.segment_stats["segmented_steps"] == 0
    rk = ek.step(f, c, uniforms=u, level=level)
    st = ek.segment_stats
    assert ek.piece_layout is not None and st["fallbacks"] == 0, (ek.piece_layout, st)
    if pieces is not None:
        assert ek.piece_layout["v"][0] <= pieces and ek.piece_layout["r"][0] <= pieces
    assert torch.equal(rk["tokens"], r1["tokens"])
    ev, er = float((rk["values"] - v1).abs().max()), float((rk["rewards"] - w1).abs().max())
    eg = float((ek.flat_grad - g1).abs().max() / g1.abs().max())
    _record("chain_pieces_%s_b%d" % (pieces, B), values=ev, rewards=er, grad_rel=eg, reruns=st["reruns"],
            **{"err%d" % i: e for i, e in enumerate(st["tc_max_err"][:14])})
    assert ev <= TOL and er <= TOL and eg <= GTOL, (ev, er, eg)
    assert abs(rk.loss - r1.loss) <= TOL


def test_chain_pieces_short_warmup_is_caught_and_rerun():
    """A warm-up too short to forget the initial state (4 positions) must be caught by the joint check: the chains are
    re-run with a longer warm-up (or, after three attempts, on the serial kernels) before anything leaves the engine,
    a warning is raised, and the step comes out within the serial kernels' tolerances."""
    seed, B, L = 141, 64, 10
    e1, ek, A = _seg_engines(seed, 32, 4)
    f, c = synth.make_inputs(seed, B, L)
    u = synth.make_uniforms(seed, L - 1, B)
    r1 = e1.step(f, c, uniforms=u)
    v1, w1, g1 = r1["values"].clone(), r1["rewards"].clone(), e1.flat_grad.clone()
    with pytest.warns(UserWarning, match="chain segments did not converge"):
        rk = ek.step(f, c, uniforms=u)
    assert ek.segment_stats["reruns"] >= 1 and ek.warm["v"] > 4 and ek.warm["r"] > 4
    assert float((rk["values"] - v1).abs().max()) <= TOL and float((rk["rewards"] - w1).abs().max()) <= TOL
    assert float((ek.flat_grad - g1).abs().max() / g1.abs().max()) <= GTOL
    # unverified steps (check=False) are reported by segments_verified()
    ek.warm = {"v": 4, "r": 4, "b": 4}
    ek.step(f, c, uniforms=u, check=False)
    with pytest.warns(UserWarning):
        assert ek.segments_verified() is False
    assert ek.segments_verified() is True


def test_chain_pieces_fall_back_to_the_serial_kernels():
    """A step whose joint checks fail on every tcgen05 attempt (chain_tol far below the float rounding of the joints)
    ends on the serial kernels: one fall-back is counted, and values and rewards are those of the serial engine bit for
    bit."""
    seed, B, L = 141, 64, 10
    e1, ek, A = _seg_engines(seed, 32, 64, tol=1e-12)
    f, c = synth.make_inputs(seed, B, L)
    u = synth.make_uniforms(seed, L - 1, B)
    r1 = e1.step(f, c, uniforms=u)
    v1, w1, g1 = r1["values"].clone(), r1["rewards"].clone(), e1.flat_grad.clone()
    with pytest.warns(UserWarning, match="chain segments did not converge"):
        rk = ek.step(f, c, uniforms=u)
    st = ek.segment_stats
    assert st["fallbacks"] == 1 and ek.piece_layout is None, st
    assert torch.equal(rk["values"], v1) and torch.equal(rk["rewards"], w1)
    assert float((ek.flat_grad - g1).abs().max() / g1.abs().max()) <= 1e-6      # atomics in the table scatter reorder sums


def test_get_rewards_pieces_equal_the_serial_chain():
    from icrl_b200.engine import A2CEngine
    seed, B, L = 151, 512, 12
    A, R, w = make_nets(seed)
    f, c = synth.make_inputs(seed, B, L)
    r1 = A2CEngine(A, R, chain_segments=1).get_rewards(f, c)
    ek = A2CEngine(A, R, chain_warmup=160)
    rk = ek.get_rewards(f, c)
    assert ek.piece_layout is not None and ek.piece_layout["v"] is None and ek.segment_stats["fallbacks"] == 0
    assert float((rk - r1).abs().max()) <= TOL


def test_config4_pieces_full_size():
    """BASELINE config 4 at full single-GPU size with the default engine: the joint checks pass without a serial
    fall-back, and values / rewards / gradients agree with the serial chain at the tolerances of the golden tests."""
    from icrl_b200.engine import A2CEngine
    seed, B, L = 97, 4096, 20
    A, R, w = make_nets(seed)
    f, c = synth.make_inputs(seed, B, L)
    u = synth.make_uniforms(seed, L - 1, B)
    ek = A2CEngine(A, R)
    rk = ek.step(f, c, uniforms=u)
    assert ek.piece_layout is not None and ek.segment_stats["fallbacks"] == 0, ek.segment_stats
    vk, wk, gk = rk["values"].clone(), rk["rewards"].clone(), ek.flat_grad.clone()
    e1 = A2CEngine(A, R, chain_segments=1)
    r1 = e1.step(f, c, uniforms=u)
    assert torch.equal(rk["tokens"], r1["tokens"])
    ev, er = float((vk - r1["values"]).abs().max()), float((wk - r1["rewards"]).abs().max())
    eg = float((gk - e1.flat_grad).abs().max() / e1.flat_grad.abs().max())
    _record("config4_pieces", values=ev, rewards=er, grad_rel=eg, pieces=ek.piece_layout["v"][0],
            **{"err%d" % i: e for i, e in enumerate(ek.segment_stats["tc_max_err"][:14])})
    assert ev <= TOL and er <= TOL and eg <= GTOL, (ev, er, eg)


# ---- full-size parity against the CPU port of the reference computed on the GPU box (not against our own kernels)

def test_full_step_b1024_vs_cpu_port():
    """One complete A2C minibatch at B = 1024, L = 20 (config 4's per-rank size at 4 GPUs: 194,560 + 214,016 serial chain
    positions) on the default engine against oracle/ref_port executing the reference's algorithm on the host cores:
    token ids bit-exact, values / rewards / log-probs within 2e-6, loss within 2e-6, all 18 gradients within 2e-5 of
    each tensor's largest entry."""
    from icrl_b200.engine import A2CEngine
    seed, B, L = 211, 1024, 20
    A, R, w = make_nets(seed)
    f, c = synth.make_inputs(seed, B, L)
    u = synth.make_uniforms(seed, L - 1, B)
    eng = A2CEngine(A, R)
    res = eng.step(f, c, uniforms=u)
    assert eng.piece_layout is not None and eng.segment_stats["fallbacks"] == 0, eng.segment_stats
    torch.set_num_threads(max(torch.get_num_threads(), 8))
    ref = ref_port.a2c_minibatch(ref_port.Nets(w), f, c, u)
    assert np.array_equal(res["tokens"].cpu().numpy(), ref["tokens"])
    errs = {k: float(np.abs(res[k].cpu().numpy() - ref[k]).max()) for k in ("values", "rewards", "logp")}
    errs["loss"] = abs(res.loss - ref["loss"])
    grads = named_grads(A)
    worst = 0.0
    for k, gr in grads.items():
        r = ref["grads"][k].numpy()
        worst = max(worst, float(np.abs(gr - r).max()) / max(float(np.abs(r).max()), 1e-12))
    _record("full_step_b1024_vs_port", grad_worst=worst, **errs)
    assert all(v <= TOL for v in errs.values()), errs
    assert worst <= GTOL, worst


def test_get_rewards_config3_full_size_vs_cpu_port():
    """BASELINE config 3 at full size (8192 captions x 20 tokens, one GetRewards from zero state = 163,840 serial GRU
    positions) against the CPU port of the reference computed here: within 2e-6."""
    from icrl_b200.engine import A2CEngine
    seed, B, L = 223, 8192, 20
    A, R, w = make_nets(seed)
    f, c = synth.make_inputs(seed, B, L)
    eng = A2CEngine(A, R)
    got = eng.get_rewards(f, c).cpu().numpy()
    assert eng.piece_layout is not None and eng.segment_stats["fallbacks"] == 0
    ref = ref_port.get_rewards(ref_port.Nets(w), f, c)
    err = float(np.abs(got - ref).max())
    _record("rewards_b8192_vs_port", rewards=err, pieces=eng.piece_layout["r"][0], warm=eng.piece_layout["r"][2])
    assert got.shape == (B, 1) and err <= TOL, err


# ---- the warm-up survives training

def test_pieces_survive_200_adam_steps():
    """200 optimizer steps at B = 1024 on the default engine (the weights move, so does the forgetting length of the two
    chains): the warm-up adapts (it may grow and shrink), no step falls back to the serial kernels, re-runs stay rare,
    and the last step agrees with the serial kernels run on the same weights."""
    from icrl_b200.engine import A2CEngine
    from icrl_b200.optim import FlatAdam
    seed, B, L = 307, 1024, 20
    A, R, w = make_nets(seed)
    eng = A2CEngine(A, R)
    opt = FlatAdam(eng, lr=1e-4)
    f, c = synth.make_inputs(seed, B, L)
    for i in range(200):
        res = eng.step(f, c, uniforms=synth.make_uniforms(seed + i, L - 1, B))
        assert np.isfinite(res.loss)
        opt.step()
    st = eng.segment_stats
    _record("pieces_200_steps", reruns=st["reruns"], fallbacks=st["fallbacks"], warm_v=eng.warm["v"], warm_r=eng.warm["r"],
            changes=len(st["warm_history"]))
    assert st["fallbacks"] == 0 and st["reruns"] <= 4, st
    assert st["segmented_steps"] >= 200
    u = synth.make_uniforms(seed + 999, L - 1, B)
    rk = eng.step(f, c, uniforms=u)
    gk = eng.flat_grad.clone()
    e1 = A2CEngine(A, R, chain_segments=1)
    r1 = e1.step(f, c, uniforms=u)
    eng._attach_grads()
    assert torch.equal(rk["tokens"], r1["tokens"])
    # 200 steps of this unbounded loss (advantage = values - rewards, trainers.py:471) have driven |values| to ~10: the
    # tolerance is relative to their magnitude (2e-6 of 8 is two float ulps)
    vscale = max(1.0, float(r1["values"].abs().max()))
    ev = float((rk["values"] - r1["values"]).abs().max())
    _record("pieces_200_steps", values_rel=ev / vscale, vscale=vscale)
    assert ev <= TOL * vscale, (ev, vscale)
    assert float((rk["rewards"] - r1["rewards"]).abs().max()) <= TOL
    # Gradients: by now the critic has learned the mean of its target, so the value-side gradients are sums that cancel
    # (linear2.bias = sum of dL/dvalues ~ 0) and amplify any difference in the values.  The tensor-core kernels
    # (truncating accumulation, compensated in the mean: chain_tc.cu g_tc_bias) agree with the serial chain to ~1e-4
    # here; the policy-side gradients stay at 2e-6.  Tolerance for this regime: 3e-4 of max.
    eg = float((gk - e1.flat_grad).abs().max() / e1.flat_grad.abs().max())
    _record("pieces_200_steps", grad_rel=eg)
    assert eg <= 3e-4, eg


def test_slow_forgetting_weights_degrade_gracefully():
    """Weights whose gates forget slowly (forget-gate bias of the value LSTM +1.5, update gate of the reward GRU pushed
    towards 'keep'; +4 would make the recurrence itself non-contractive -- the reference's own gradients overflow there):
    the joint check notices, the warm-up grows (or the step ends on the serial kernels) and the numbers still match the
    serial chain -- slower, never wrong."""
    from icrl_b200.engine import A2CEngine
    seed, B, L = 311, 512, 12
    A, R, w = make_nets(seed)
    with torch.no_grad():
        A.value_network.valrnn.lstm.bias_hh_l0[512:1024] += 1.5
        R.rewrnn.gru.bias_hh_l0[512:1024] += 1.5
    f, c = synth.make_inputs(seed, B, L)
    u = synth.make_uniforms(seed, L - 1, B)
    e1 = A2CEngine(A, R, chain_segments=1)
    r1 = e1.step(f, c, uniforms=u)
    v1, w1, g1 = r1["values"].clone(), r1["rewards"].clone(), e1.flat_grad.clone()
    assert torch.isfinite(g1).all()
    ek = A2CEngine(A, R, chain_warmup=32)
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        rk = ek.step(f, c, uniforms=u)
        first = dict(ek.segment_stats)
        rk2 = ek.step(f, c, uniforms=u)               # the second step starts from the warm-up the first one learned
    st = ek.segment_stats
    _record("slow_forgetting", reruns=st["reruns"], fallbacks=st["fallbacks"], warm_v=ek.warm["v"], warm_r=ek.warm["r"])
    assert first["reruns"] + first["fallbacks"] >= 1, "a 32-position warm-up cannot be enough for these weights"
    assert max(ek.warm.values()) > 32
    for r in (rk, rk2):
        assert float((r["values"] - v1).abs().max()) <= TOL and float((r["rewards"] - w1).abs().max()) <= TOL
    assert float((ek.flat_grad - g1).abs().max() / g1.abs().max()) <= GTOL


@pytest.mark.parametrize("switch", ["tma_store", "separate_forward_launches", "no_backward_overlap", "simt_policy_bptt"])
def test_chain_engine_switches_agree(switch):
    """The alternative code paths kept behind switches compute the same step as the default engine: the forward stash
    through TMA tensor stores, value / reward forward chains as two launches instead of the fused one, the policy
    backward on the main stream instead of a second one, and the per-step SIMT policy BPTT."""
    from icrl_b200 import _lib
    from icrl_b200.engine import A2CEngine
    seed, B, L = 173, 384, 14
    A, R, w = make_nets(seed)
    f, c = synth.make_inputs(seed, B, L)
    u = synth.make_uniforms(seed, L - 1, B)
    e0 = A2CEngine(A, R, chain_warmup=160)
    r0 = e0.step(f, c, uniforms=u)
    v0, w0, g0 = r0["values"].clone(), r0["rewards"].clone(), e0.flat_grad.clone()
    assert e0.piece_layout is not None and e0.piece_layout["fused"]
    kw = {"separate_forward_launches": dict(chain_fuse_fwd=False), "no_backward_overlap": dict(overlap_backward=False),
          "simt_policy_bptt": dict(policy_bptt="simt")}.get(switch, {})
    if switch == "tma_store":
        _lib.call("icrl_chain_tc_set_tma_store", 1)
    try:
        e1 = A2CEngine(A, R, chain_warmup=160, **kw)
        r1 = e1.step(f, c, uniforms=u)
        torch.cuda.synchronize()
    finally:
        _lib.call("icrl_chain_tc_set_tma_store", 0)
    assert e1.piece_layout is not None and e1.segment_stats["fallbacks"] == 0
    if switch == "separate_forward_launches":
        assert not e1.piece_layout["fused"]
    assert torch.equal(r1["tokens"], r0["tokens"])
    assert float((r1["values"] - v0).abs().max()) <= TOL and float((r1["rewards"] - w0).abs().max()) <= TOL
    assert float((e1.flat_grad - g0).abs().max() / g0.abs().max()) <= GTOL


@pytest.mark.parametrize("B,p0,S", [(96, 1, 7), (64, 5, 4), (130, 1, 19)])
def test_value_param_grads_stream_scatter_matches_generic(B, p0, S):
    """icrl_value_chain_param_grads with the stream's shape (positions that consumed the same token summed before one
    vector reduction, column maxima handed to the contraction) against the same call without it (one reduction per
    position, maxima from a pre-pass) and against float64 for the gate-table gradient."""
    import ctypes
    from icrl_b200 import _lib
    V, D, G = 211, 512, 2048
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
    rs = np.random.RandomState(B + S)
    T = int(_lib.call("icrl_stream_len", B, p0, S, 0))
    tokcm = torch.from_numpy(rs.randint(0, V, size=((p0 + S) * B,)).astype(np.int32)).cuda()
    stream = torch.zeros(T + 1, dtype=torch.int32, device="cuda")
    take = torch.zeros(T + 1, dtype=torch.int32, device="cuda")
    pos = torch.zeros(S * B, dtype=torch.int32, device="cuda")
    _lib.call("icrl_build_stream", st, B, p0, S, 0, p(tokcm), p(stream), p(take), p(pos), None)
    colscale = 10.0 ** rs.uniform(-9, -3, size=G)
    dgates = torch.from_numpy((rs.standard_normal((T, G)) * colscale).astype(np.float32)).cuda()
    stash_h = torch.from_numpy(np.tanh(rs.standard_normal((T + 1, 512))).astype(np.float32)).cuda()
    E = torch.from_numpy(rs.standard_normal((V, D)).astype(np.float32)).cuda()
    W_ih = torch.from_numpy((rs.standard_normal((G, D)) * 0.05).astype(np.float32)).cuda()
    cs = int(_lib.call("icrl_colsum_ws_floats", max(T, V), G))
    wsb = int(_lib.call("icrl_wgrad_tc_ws_bytes", G, 512, T, 2))
    out = {}
    for tag, shape in (("stream", (B, p0, S)), ("generic", (0, 0, 0))):
        dtable = torch.full((V, G), float("nan"), device="cuda")
        csws = torch.zeros(cs, device="cuda")
        ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
        dE, dWih = torch.empty((V, D), device="cuda"), torch.empty((G, D), device="cuda")
        dWhh, dbi, dbh = torch.empty((G, 512), device="cuda"), torch.empty(G, device="cuda"), torch.empty(G, device="cuda")
        _lib.call("icrl_value_chain_param_grads", st, T, V, D, p(stream), p(dgates), p(stash_h), p(E), p(W_ih), p(dtable),
                  p(csws), p(ws), wsb, p(dE), p(dWih), p(dWhh), p(dbi), p(dbh), *shape, 0, None)
        torch.cuda.synchronize()
        out[tag] = dict(dtable=dtable, dE=dE, dWih=dWih, dWhh=dWhh, dbi=dbi, dbh=dbh)
    ref = torch.zeros((V, G), dtype=torch.float64, device="cuda")
    ref.index_add_(0, stream[:T].long(), dgates.double())
    rowscale = ref.abs().max(dim=0).values.clamp_min(1e-300)
    for tag in out:
        err = ((out[tag]["dtable"].double() - ref).abs() / rowscale).max().item()
        assert err < 2e-6, (tag, err)
    worst = 0.0
    for k in out["stream"]:
        a, b = out["stream"][k].double(), out["generic"][k].double()
        assert torch.isfinite(a).all(), k
        rel = ((a - b).abs().max() / b.abs().max().clamp_min(1e-300)).item()
        worst = max(worst, rel)
        assert rel < 2e-6, (k, rel)
    _record("value_param_grads_stream_b%d_s%d" % (B, S), rel_vs_generic=worst)
