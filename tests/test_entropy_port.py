"""The CPU port of the reference's A2C minibatch with the entropy bonus the engine offers (entropy_coef), and its checks.

The reference's loss has no entropy term, so the as-executed port (oracle/ref_port.a2c_minibatch) has none either.
`a2c_minibatch_entropy` is that function step for step -- the same library layers of oracle/ref_port, called in the same
order -- with the bonus added to the loss before backward():

    loss = mean(-logp * adv) + 0.5 * mean(adv^2) - entropy_coef * mean_{b,s} H[b][s],
    H = -sum_j softmax(z)_j log_softmax(z)_j  over the logits z each sampled step drew from.

tests/test_gpu_entropy.py compares the fused engine with it.  The tests here pin it to ref_port at entropy_coef = 0 and
check the term's gradient in float64."""
import numpy as np
import torch
import torch.nn.functional as F

from oracle import ref_port, synth


def a2c_minibatch_entropy(nets, features, captions, uniforms, level=None, entropy_coef=0.0):
    """ref_port.a2c_minibatch (trainers.py:428-496 / 540-612) with the entropy bonus.  Returns its dict plus
    ``mean_entropy``."""
    feats = torch.as_tensor(features).to(nets.dtype)
    caps = torch.as_tensor(captions).long()
    B = caps.shape[0]
    caplen = int((caps == 2).nonzero()[:, 1].max()) + 1
    if level is None:
        p0, S = 1, caplen - 1
    else:
        p0, S = caplen - level, level
        if p0 < 1:
            return None
    nets.reset_state()
    prefix = caps[:, :p0]
    vals, rews, lps, toks, ents = [], [], [], [], []
    for s in range(S):
        value = ref_port.value_call(nets, feats, prefix)
        z = ref_port.policy_logits(nets, feats, prefix)[:, -1:, :]
        probs = F.softmax(z, dim=2)
        ents.append(-(probs[:, 0, :] * F.log_softmax(z[:, 0, :], dim=1)).sum(dim=1))
        acts = ref_port.sample_rows(probs.detach().numpy()[:, 0], uniforms[s])
        a = torch.from_numpy(acts).view(B, 1)
        prefix = torch.cat((prefix, a), dim=1)
        lps.append(torch.log(probs[:, 0, :].gather(1, a)))
        rews.append(ref_port.reward_call(nets, feats, prefix))
        vals.append(value)
        toks.append(acts)
    values = torch.stack(vals, dim=1).reshape(B, S)
    rewards = torch.stack(rews, dim=1).reshape(B, S)
    logp = torch.stack(lps, dim=1).reshape(B, S)
    adv = values - rewards
    loss = (-logp * adv).mean() + 0.5 * adv.pow(2).mean()
    mean_entropy = torch.stack(ents, dim=1).mean()
    if entropy_coef:
        loss = loss - entropy_coef * mean_entropy
    named = nets.named_trainable()
    for _, p in named:
        p.grad = None
    loss.backward()
    grads = {k: (p.grad.detach().clone() if p.grad is not None else torch.zeros_like(p)) for k, p in named}
    nets.reset_state()
    return dict(tokens=np.stack(toks, axis=1), values=values.detach().numpy(), rewards=rewards.detach().numpy(),
                logp=logp.detach().numpy(), loss=float(loss.detach()), mean_reward=float(rewards.detach().mean()),
                mean_adv=float(adv.detach().mean()), mean_entropy=float(mean_entropy.detach()), grads=grads, p0=p0, S=S)


def _case(seed=3, B=6, L=5, vocab=64):
    w = synth.make_weights(seed, vocab=vocab)
    f, c = synth.make_inputs(seed, B, L, vocab=vocab)
    return w, f, c, synth.make_uniforms(seed, L - 1, B)


def test_coefficient_zero_is_ref_port():
    """At entropy_coef = 0 the port computes what ref_port computes, bit for bit."""
    w, f, c, u = _case()
    ref = ref_port.a2c_minibatch(ref_port.Nets(w), f, c, u)
    got = a2c_minibatch_entropy(ref_port.Nets(w), f, c, u)
    assert np.array_equal(got["tokens"], ref["tokens"])
    for k in ("values", "rewards", "logp"):
        assert np.array_equal(got[k], ref[k]), k
    assert got["loss"] == ref["loss"]
    for k in ref["grads"]:
        assert torch.equal(got["grads"][k], ref["grads"][k]), k


def test_entropy_term_gradient_in_float64():
    """The bonus moves the loss by -coef * mean entropy and the policy's gradients by the gradient of that term alone:
    coef * d(mean H)/d(theta), here for linear2vocab through autograd in float64 (the value network does not move)."""
    w, f, c, u = _case()
    coef = 0.7
    n0, n1 = ref_port.Nets(w, dtype=torch.float64), ref_port.Nets(w, dtype=torch.float64)
    r0 = a2c_minibatch_entropy(n0, f, c, u)
    r1 = a2c_minibatch_entropy(n1, f, c, u, entropy_coef=coef)
    assert np.array_equal(r0["tokens"], r1["tokens"])
    assert abs((r1["loss"] - r0["loss"]) + coef * r1["mean_entropy"]) <= 1e-12
    for k in r0["grads"]:
        if k.startswith("value_network."):
            assert torch.equal(r0["grads"][k], r1["grads"][k]), k
    # the term's own gradient w.r.t. the vocabulary projection: the teacher-forced logits of the sampled prefix
    caps = np.concatenate((c[:, :1], r1["tokens"]), axis=1)
    nets = ref_port.Nets(w, dtype=torch.float64)
    z = ref_port.policy_logits(nets, torch.as_tensor(f).double(), torch.as_tensor(caps[:, :-1]).long())
    H = -(F.softmax(z, -1) * F.log_softmax(z, -1)).sum(-1)
    (gw,) = torch.autograd.grad(H.mean(), nets.p_out.weight)
    k = "policy_network.linear2vocab.weight"
    diff = r0["grads"][k] - r1["grads"][k]
    assert float((diff - coef * gw).abs().max()) <= 1e-10 * max(1.0, float(gw.abs().max()))
