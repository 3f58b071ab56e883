"""Pins the oracle: ref_port and single_pass against the golden vectors that
oracle/gen_golden.py produced by executing the unmodified reference (SURVEY.md §8c).
Tolerances: token ids bit-exact; values/rewards/logp 2e-6 abs (the reference's own two
formulations differ by 1.5e-7..5e-7, Appendix A.3); gradients 5e-6 of the tensor's max."""
import os

import numpy as np
import pytest
import torch

from oracle import ref_port, single_pass, synth
from oracle.gen_golden import THREADS, grad_sample_index

A2C_CASES = ["a2c_b8_l6", "a2c_b32_l9", "curr_b16_l10_lv4", "curr_b24_l20_lv6"]


@pytest.fixture(autouse=True)
def _golden_thread_count():
    """ref_port matches the fixtures bit for bit only with the intra-op thread count they were generated with, whatever
    the host's core count."""
    n = torch.get_num_threads()
    torch.set_num_threads(THREADS)
    yield
    torch.set_num_threads(n)


def _load(golden_dir, name):
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    seed, B, L = int(g["seed"]), int(g["B"]), int(g["L"])
    level = int(g["level"])
    level = None if level < 0 else level
    w = synth.make_weights(seed)
    f, c = synth.make_inputs(seed, B, L)
    S = (L - 1) if level is None else level
    return g, w, f, c, synth.make_uniforms(seed, S, B), level


def _check(res, g, tol_val, tol_grad):
    assert np.array_equal(res["tokens"], g["tokens"])
    for k in ("values", "rewards", "logp"):
        assert np.abs(res[k] - g[k]).max() <= tol_val, k
    assert abs(res["loss"] - float(g["loss"])) <= tol_val
    assert abs(res["mean_reward"] - float(g["mean_reward"])) <= tol_val
    assert abs(res["mean_adv"] - float(g["mean_adv"])) <= tol_val
    for k, grad in res["grads"].items():
        flat = grad.detach().numpy().reshape(-1)
        ref = g["gsamp/" + k]
        got = flat[grad_sample_index(flat.size)]
        scale = max(float(np.abs(ref).max()), 1e-12)
        assert np.abs(got - ref).max() <= tol_grad * scale, k
        nrm = float(np.sqrt((flat.astype(np.float64) ** 2).sum()))
        assert abs(nrm - float(g["gnorm/" + k])) <= 1e-5 * max(float(g["gnorm/" + k]), 1e-12), k


@pytest.mark.parametrize("name", A2C_CASES)
def test_ref_port_matches_reference(golden_dir, name):
    g, w, f, c, u, level = _load(golden_dir, name)
    res = ref_port.a2c_minibatch(ref_port.Nets(w), f, c, u, level=level)
    _check(res, g, 1e-7, 1e-6)          # same library calls in the same order: ~bitwise


def _variant_case(golden_dir, name):
    """a2c_b12_l7_bidir / a2c_b16_l8_wemb300 with the weight layout they were generated with."""
    g, _, f, c, u, level = _load(golden_dir, name)
    w = synth.make_weights(int(g["seed"]), wordvec_dim=int(g["wordvec_dim"]), bidirectional=name.endswith("bidir"))
    return g, w, f, c, u, level


@pytest.mark.parametrize("dtype,tol_val,tol_grad", [(torch.float32, 1e-7, 1e-6), (torch.float64, 2e-6, 5e-6)])
@pytest.mark.parametrize("name", ["a2c_b12_l7_bidir", "a2c_b16_l8_wemb300"])
def test_ref_port_variants_match_reference(golden_dir, name, dtype, tol_val, tol_grad):
    """The bidirectional networks and the frozen 300-d word vectors, in float32 (the as-executed port: ~bitwise) and in
    float64 (the reference the module-route kernels are checked against: tokens equal, the rest to fp32 rounding)."""
    g, w, f, c, u, level = _variant_case(golden_dir, name)
    nets = ref_port.Nets(w, dtype=dtype, bidirectional=name.endswith("bidir"))
    res = ref_port.a2c_minibatch(nets, f, c, u, level=level)
    _check(res, g, tol_val, tol_grad)
    assert nets.v_state[0].dtype == dtype and nets.v_state[0].shape == (1 + nets.bidirectional, 1, 512)
    if name.endswith("wemb300"):
        assert nets.p_rnn.weight_ih_l0.shape == (2048, 300) and not nets.p_emb.weight.requires_grad
        assert len(res["grads"]) == 16


@pytest.mark.parametrize("dtype,tol_val,tol_grad", [(torch.float32, 1e-7, 1e-6), (torch.float64, 2e-6, 5e-6)])
def test_ref_port_pretraining_losses_match_reference(golden_dir, dtype, tol_val, tol_grad):
    """The three supervised pretraining losses (weighted cross-entropy, VisualSemanticEmbeddingLoss, MSE on the greedy
    captions' rewards) and all 27 gradients, against one minibatch of each of the reference's loops."""
    g = np.load(os.path.join(golden_dir, "pretrain_b12.npz"))
    seed, B = int(g["seed"]), int(g["B"])
    w = synth.make_weights(seed)
    f, c = synth.make_inputs(seed, B, 17)
    nets = ref_port.Nets(w, dtype=dtype)
    k = int(g["value_prefix_len"])
    runs = {"policy": lambda: ref_port.policy_xent_loss(nets, f, c),
            "reward": lambda: ref_port.reward_vse_loss(nets, f, c),
            "value": lambda: ref_port.value_mse_loss(nets, f, c, k)}
    ngrads = 0
    for key, fn in runs.items():
        res, grads = ref_port.network_grads(nets, key, fn)
        ref_loss = float(g[key + "_loss"])
        loss = float(res[0].detach())
        assert abs(loss - ref_loss) <= tol_val * max(1.0, abs(ref_loss)), (key, loss, ref_loss)
        for name, grad in grads.items():
            flat = grad.numpy().reshape(-1)
            ref = g["%s/gsamp/%s" % (key, name)]
            scale = max(float(np.abs(ref).max()), 1e-12)
            assert np.abs(flat[grad_sample_index(flat.size)] - ref).max() <= tol_grad * scale, (key, name)
            nrm, ref_n = float(np.sqrt((flat.astype(np.float64) ** 2).sum())), float(g["%s/gnorm/%s" % (key, name)])
            assert abs(nrm - ref_n) <= 1e-5 * max(ref_n, 1e-12), (key, name)
            ngrads += 1
    assert ngrads == 27


@pytest.mark.parametrize("name", A2C_CASES)
@pytest.mark.parametrize("lib", [False, True])
def test_single_pass_matches_reference(golden_dir, name, lib):
    g, w, f, c, u, level = _load(golden_dir, name)
    res = single_pass.a2c_minibatch(w, f, c, u, level=level, lib=lib)
    _check(res, g, 2e-6, 5e-6)


@pytest.mark.slow
def test_single_pass_config2(golden_dir):
    """BASELINE config 2 (B=256, L=20): forward quantities only (the gradient check at
    this size lives in the GPU suite where the kernels are compared to the fixture)."""
    g, w, f, c, u, level = _load(golden_dir, "a2c_b256_l20")
    res = single_pass.a2c_minibatch(w, f, c, u, backward=False, lib=True)
    assert np.array_equal(res["tokens"], g["tokens"])
    for k in ("values", "rewards", "logp"):
        assert np.abs(res[k] - g[k]).max() <= 5e-6, k


def test_greedy_config1(golden_dir):
    g = np.load(os.path.join(golden_dir, "greedy_b32.npz"))
    w = synth.make_weights(0)
    f, _ = synth.make_inputs(0, 32, 17)
    for toks, logits in (single_pass.greedy_decode(w, f, np.ones(32)),
                         ref_port.greedy_decode(ref_port.Nets(w), f, np.ones(32))):
        assert np.array_equal(toks, g["tokens"])
        assert np.abs(logits - g["last_logits"]).max() <= 1e-5


def test_get_rewards_config3_shape(golden_dir):
    g = np.load(os.path.join(golden_dir, "rewards_b64_l20.npz"))
    w = synth.make_weights(6)
    f, c = synth.make_inputs(6, 64, 20)
    assert np.abs(single_pass.get_rewards(w["reward"], f, c) - g["rewards"]).max() <= 1e-6
    assert np.abs(ref_port.get_rewards(ref_port.Nets(w), f, c) - g["rewards"]).max() <= 1e-7


def test_sampling_is_numpy_choice():
    """np.random.choice(V, p=row) consumes one double and equals the explicit inverse CDF
    (trainers.py:449): the contract the sampling kernel implements."""
    rs = np.random.RandomState(7)
    p = torch.softmax(torch.from_numpy(rs.standard_normal((16, 1004)).astype(np.float32)), dim=1).numpy()
    np.random.seed(11)
    got = [np.random.choice(1004, p=p[i]) for i in range(16)]
    u = synth.make_uniforms(11, 1, 16)[0]
    assert got == [single_pass.sample_inverse_cdf(p[i], u[i]) for i in range(16)]


def test_dp_shard_oracle_is_sum_of_shards(golden_dir):
    """SURVEY §8e: an N-rank run == N independent runs on contiguous row shards with the
    gradient seeds scaled by 1/(B_global*S); policy tokens are shard-invariant."""
    g, w, f, c, u, level = _load(golden_dir, "a2c_b8_l6")
    full = single_pass.a2c_minibatch(w, f, c, u)
    halves = [single_pass.a2c_minibatch(w, f[i:i + 4], c[i:i + 4], u[:, i:i + 4], loss_scale_rows=8)
              for i in (0, 4)]
    assert np.array_equal(np.concatenate([h["tokens"] for h in halves]), full["tokens"])
    k = "policy_network.linear2vocab.bias"
    assert halves[0]["grads"][k].shape == full["grads"][k].shape


def test_chain_segment_formulation_on_cpu():
    """The chain-segment formulation of DESIGN 4.1, restated with the oracle's cells on the CPU: cut ONE carried-state
    LSTM chain into K pieces, let every later piece start from zero state `warm` positions early (forward) and every
    earlier piece start its backward recurrence `warm` positions late with zero dh / dc (backward), discard the warm-up
    steps -- hidden states and gate-table gradients must equal the serial chain's to float rounding.  Same geometry as
    the kernels: piece k covers positions [k*seg, (k+1)*seg + warm), seg = ceil((T - warm) / K)."""
    torch.manual_seed(0)
    w = synth.make_weights(7)["value"]
    E, w_ih, w_hh = w["valrnn.caption_embedding.weight"], w["valrnn.lstm.weight_ih_l0"], w["valrnn.lstm.weight_hh_l0"]
    bias = w["valrnn.lstm.bias_ih_l0"] + w["valrnn.lstm.bias_hh_l0"]
    T, K, warm = 700, 4, 64
    seg = (T - warm + K - 1) // K
    rs = np.random.RandomState(5)
    stream = torch.from_numpy(rs.randint(0, synth.VOCAB, T))
    inject = torch.zeros(T, single_pass.HID)
    take = rs.rand(T) < 0.3                                    # positions whose hidden state feeds the loss
    inject[torch.from_numpy(take)] = torch.from_numpy(rs.standard_normal((int(take.sum()), single_pass.HID)).astype(np.float32)) * 1e-3

    def run(lo, hi, h, c, xg):
        hs = []
        for t in range(lo, hi):
            h, c = single_pass.lstm_cell(xg[t - lo], h, c, w_hh)
            hs.append(h)
        return torch.stack(hs), h, c

    zero = torch.zeros(single_pass.HID)
    xg_all = (E[stream] @ w_ih.t() + bias).detach()
    # serial chain with autograd
    xg = xg_all.clone().requires_grad_(True)
    hs, _, _ = run(0, T, zero, zero, xg)
    (hs * inject).sum().backward()
    h_serial, g_serial = hs.detach(), xg.grad.clone()

    h_seg, g_seg = torch.zeros_like(h_serial), torch.zeros_like(g_serial)
    for k in range(K):
        lo, hi = k * seg, min((k + 1) * seg + warm, T)
        # forward: later pieces start from ZERO state and discard their first `warm` steps
        with torch.no_grad():
            hk, _, _ = run(lo, hi, zero, zero, xg_all[lo:hi])
        live = lo + (warm if k > 0 else 0)
        h_seg[live:hi] = hk[live - lo:]
        # backward: the piece runs [lo, hi) from the TRUE state at lo (the stash) and its recurrence starts at hi - 1
        # with zero dh / dc, i.e. nothing flows in from positions >= hi; the gradients of its last `warm` positions
        # are discarded unless it is the last piece
        h0 = h_serial[lo - 1] if lo > 0 else zero
        with torch.no_grad():
            c0 = zero
            if lo > 0:
                _, _, c0 = run(0, lo, zero, zero, xg_all[:lo])
        xk = xg_all[lo:hi].clone().requires_grad_(True)
        hk, _, _ = run(lo, hi, h0, c0, xk)
        (hk * inject[lo:hi]).sum().backward()
        keep_hi = hi if k == K - 1 else (k + 1) * seg
        g_seg[lo:keep_hi] = xk.grad[:keep_hi - lo]
    assert float((h_seg - h_serial).abs().max()) <= 1e-6
    scale = float(g_serial.abs().max())
    assert float((g_seg - g_serial).abs().max()) <= 1e-5 * scale
    # and a warm-up that is too short IS visible (what the run-time check is for)
    with torch.no_grad():
        lo = seg
        hk, _, _ = run(lo, lo + 4, zero, zero, xg_all[lo:lo + 4])
    assert float((hk[-1] - h_serial[lo + 3]).abs().max()) > 1e-3
