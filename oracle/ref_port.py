"""The reference algorithm AS EXECUTED, on torch CPU library layers.

TEST INFRASTRUCTURE (see oracle/__init__).  This is the CPU baseline bench.py times
(``cpu_baseline.kind = "port"`` and ``--impl reference``) and the first-level checker
for the single-pass restatement.  It keeps every cost the reference pays:

* the policy LSTM is re-run over the whole prefix at every rollout step
  (``models.py:286`` called from ``trainers.py:441-443``),
* the value / reward RNNs are fed the batch axis as the time axis, one library
  call per caption column, with the hidden state carried between calls and reset
  once per minibatch (``models.py:130-135, 166-169, 223-228, 253-255``;
  ``trainers.py:495-496``),
* sampling is numpy's inverse-CDF in float64 (``trainers.py:447-450``); here the
  uniforms are injected so a run is reproducible (``np.random.choice(V, p=row)``
  == ``searchsorted(cumsum(p)/cumsum(p)[-1], u, 'right')``, SURVEY.md Appendix A.3).

Third-party arithmetic: torch ``nn.LSTM / nn.GRU / nn.Linear / nn.Embedding /
softmax / normalize`` (the reference does not pin a torch version; the oracle runs
on the container's torch 2.11.0) and numpy ``cumsum / searchsorted`` (2.3.x).
"""
import numpy as np
import torch
from torch import nn
import torch.nn.functional as F

HID = 512


def _load(module, sd, prefix):
    with torch.no_grad():
        for name, p in module.named_parameters():
            p.copy_(sd[prefix + name])
    return module


class Nets:
    """Library layers holding one set of weights (policy, value, reward).

    ``dtype`` builds every layer in that precision (torch.float64 gives the high-precision reference the module-route
    tests compare the kernels with; the float32 default is the as-executed port).  ``bidirectional`` builds the
    reference's bidirectional variant (models.py:58-69, 114-120, 160-164, 209-215, 247-251): bidirectional RNNs, a
    1024-wide cnn2linear / linear2vocab / semantic_embed and the value network's rnn_linear.  Weights whose embeddings
    are not 512 wide are the frozen pretrained word vectors (models.py:61-63), built as
    ``gen_golden.build_reference_nets`` builds them: the tables get no gradient."""

    def __init__(self, weights, requires_grad=True, dtype=torch.float32, bidirectional=False):
        p, v, r = weights["policy"], weights["value"], weights["reward"]
        vocab, D = p["caption_embedding.weight"].shape
        self.vocab, self.dtype, self.bidirectional = vocab, dtype, bidirectional
        self.frozen_emb = D != HID
        nd = 2 if bidirectional else 1
        # policy (models.py:65-69)
        self.p_emb = _load(nn.Embedding(vocab, D), p, "caption_embedding.")
        self.p_init = _load(nn.Linear(HID, nd * HID), p, "cnn2linear.")
        self.p_rnn = _load(nn.LSTM(D, HID, batch_first=True, bidirectional=bidirectional), p, "lstm.")
        self.p_out = _load(nn.Linear(nd * HID, vocab), p, "linear2vocab.")
        # value (models.py:117-120, 160-164)
        self.v_emb = _load(nn.Embedding(vocab, D), v, "valrnn.caption_embedding.")
        self.v_rnn = _load(nn.LSTM(D, HID, bidirectional=bidirectional), v, "valrnn.lstm.")
        self.v_rl = _load(nn.Linear(2 * HID, HID), v, "rnn_linear.") if bidirectional else None
        self.v_l1 = _load(nn.Linear(2 * HID, HID), v, "linear1.")
        self.v_l2 = _load(nn.Linear(HID, 1), v, "linear2.")
        # reward (models.py:212-215, 250-251) -- frozen (trainers.py:372-373)
        self.r_emb = _load(nn.Embedding(vocab, D), r, "rewrnn.caption_embedding.")
        self.r_rnn = _load(nn.GRU(D, HID, bidirectional=bidirectional), r, "rewrnn.gru.")
        self.r_vis = _load(nn.Linear(HID, HID), r, "visual_embed.")
        self.r_sem = _load(nn.Linear(nd * HID, HID), r, "semantic_embed.")
        for m in (self.p_emb, self.p_init, self.p_rnn, self.p_out, self.v_emb, self.v_rnn, self.v_rl, self.v_l1, self.v_l2,
                  self.r_emb, self.r_rnn, self.r_vis, self.r_sem):
            if m is not None:
                m.to(dtype)
        for m in (self.r_emb, self.r_rnn, self.r_vis, self.r_sem):
            m.requires_grad_(False)
        if not requires_grad:
            for _, m in self.trainable_modules():
                m.requires_grad_(False)
        if self.frozen_emb:
            for m in (self.p_emb, self.v_emb, self.r_emb):
                m.requires_grad_(False)
        self.reset_state()

    def network_modules(self, key):
        """(state_dict prefix, module) of one network, in the reference's named_parameters() order."""
        mods = {"policy": [("caption_embedding.", self.p_emb), ("cnn2linear.", self.p_init), ("lstm.", self.p_rnn),
                           ("linear2vocab.", self.p_out)],
                "value": [("valrnn.caption_embedding.", self.v_emb), ("valrnn.lstm.", self.v_rnn), ("linear1.", self.v_l1),
                          ("linear2.", self.v_l2)] + ([("rnn_linear.", self.v_rl)] if self.bidirectional else []),
                "reward": [("rewrnn.caption_embedding.", self.r_emb), ("rewrnn.gru.", self.r_rnn),
                           ("visual_embed.", self.r_vis), ("semantic_embed.", self.r_sem)]}[key]
        return [(k, m) for k, m in mods if not (self.frozen_emb and isinstance(m, nn.Embedding))]

    def network_params(self, key):
        """(name, parameter) of one network as its named_parameters() lists them (frozen embeddings left out)."""
        return [(prefix + name, p) for prefix, m in self.network_modules(key) for name, p in m.named_parameters()]

    def trainable_modules(self):
        # a2c.parameters() order: value_network then policy_network (models.py:279-280)
        return ([("value_network." + k, m) for k, m in self.network_modules("value")] +
                [("policy_network." + k, m) for k, m in self.network_modules("policy")])

    def named_trainable(self):
        out = []
        for prefix, m in self.trainable_modules():
            for name, p in m.named_parameters():
                out.append((prefix + name, p))
        return out

    def reset_state(self):
        """init_hidden() of both RNNs (models.py:122-128, 217-221)."""
        z = lambda: torch.zeros(2 if self.bidirectional else 1, 1, HID, dtype=self.dtype)
        self.v_state = (z(), z())
        self.r_state = z()


def policy_logits(nets, features, prefix):
    """PolicyNetwork.forward, models.py:71-84.  features (B,512), prefix (B,n) -> (B,n,V).  Bidirectional: cnn2linear
    gives both initial states, the first half the forward direction's."""
    h0 = nets.p_init(features.unsqueeze(0))
    if nets.bidirectional:
        h0 = torch.cat((h0[..., :HID], h0[..., HID:]), dim=0)
    out, _ = nets.p_rnn(nets.p_emb(prefix), (h0, torch.zeros_like(h0)))
    return nets.p_out(out)


def value_call(nets, features, prefix):
    """ValueNetwork.forward, models.py:166-180: one seq=B,batch=1 LSTM call per column,
    carried state; head = linear2(linear1(cat(features, h))), h through rnn_linear when bidirectional."""
    for t in range(prefix.shape[1]):
        x = nets.v_emb(prefix[:, t]).view(prefix.shape[0], 1, -1)
        out, nets.v_state = nets.v_rnn(x, nets.v_state)
    h = out.squeeze(1)
    if nets.bidirectional:
        h = nets.v_rl(h)
    return nets.v_l2(nets.v_l1(torch.cat((features, h), dim=1)))


def reward_embed(nets, features, prefix):
    """RewardNetwork.forward, models.py:253-262: (visual embedding, semantic embedding), carried GRU state."""
    for t in range(prefix.shape[1]):
        x = nets.r_emb(prefix[:, t]).view(prefix.shape[0], 1, -1)
        out, nets.r_state = nets.r_rnn(x, nets.r_state)
    return nets.r_vis(features), nets.r_sem(out.squeeze(1))


def reward_call(nets, features, prefix):
    """RewardNetwork.forward + GetRewards: models.py:253-262, trainers.py:108-121."""
    ve, se = reward_embed(nets, features, prefix)
    se = F.normalize(se, p=2, dim=1)
    ve = F.normalize(ve, p=2, dim=1)
    return (ve * se).sum(dim=1, keepdim=True)


def sample_rows(probs_f32, u_row):
    """np.random.choice(V, p=row) with the consumed double given (trainers.py:447-450)."""
    acts = np.empty(len(u_row), dtype=np.int64)
    for i in range(len(u_row)):
        cdf = np.cumsum(probs_f32[i].astype(np.float64))
        cdf /= cdf[-1]
        acts[i] = np.searchsorted(cdf, u_row[i], side="right")
    return acts


def greedy_decode(nets, features, first_col, steps=16):
    """GenerateCaptionsGreedy, trainers.py:57-70 (MAX_SEQ_LEN-1 = 16 steps, no early stop).
    Returns (tokens (B,steps+1) int64, last-step logits (B,V))."""
    feats = torch.as_tensor(features).to(nets.dtype)
    caps = torch.as_tensor(first_col).long().view(-1, 1)
    with torch.no_grad():
        for _ in range(steps):
            logits = policy_logits(nets, feats, caps)[:, -1, :]
            caps = torch.cat((caps, logits.argmax(dim=1, keepdim=True)), dim=1)
    return caps.numpy(), logits.numpy()


def a2c_minibatch(nets, features, captions, uniforms, level=None, backward=True, greedy=False):
    """One minibatch of a2c_training (trainers.py:428-496) or, with ``level``, of
    a2c_curriculum_training (trainers.py:540-612).  ``uniforms`` is (S,B) float64.
    Returns dict(tokens, values, rewards, logp, loss, mean_reward, mean_adv, grads, p0, S)."""
    feats = torch.as_tensor(features).to(nets.dtype)
    caps = torch.as_tensor(captions).long()
    B = caps.shape[0]
    caplen = int((caps == 2).nonzero()[:, 1].max()) + 1           # trainers.py:436
    if level is None:
        p0, S = 1, caplen - 1
    else:
        p0, S = caplen - level, level                             # trainers.py:548-554
        if p0 < 1:
            return None
    nets.reset_state()
    prefix = caps[:, :p0]
    vals, rews, lps, toks = [], [], [], []
    for s in range(S):
        value = value_call(nets, feats, prefix)                                  # models.py:284
        probs = F.softmax(policy_logits(nets, feats, prefix)[:, -1:, :], dim=2)  # :286, trainers.py:444
        dist = probs.detach().numpy()[:, 0]
        if greedy:
            acts = dist.argmax(axis=1).astype(np.int64)
        else:
            acts = sample_rows(dist, uniforms[s])
        a = torch.from_numpy(acts).view(B, 1)
        prefix = torch.cat((prefix, a), dim=1)
        lps.append(torch.log(probs[:, 0, :].gather(1, a)))                       # trainers.py:458
        rews.append(reward_call(nets, feats, prefix))                            # trainers.py:459
        vals.append(value)
        toks.append(acts)
    values = torch.stack(vals, dim=1).reshape(B, S)
    rewards = torch.stack(rews, dim=1).reshape(B, S)
    logp = torch.stack(lps, dim=1).reshape(B, S)
    adv = values - rewards                                                       # trainers.py:471
    loss = (-logp * adv).mean() + 0.5 * adv.pow(2).mean()                        # :472-475
    grads = None
    if backward:
        named = nets.named_trainable()
        for _, p in named:
            p.grad = None
        loss.backward()
        grads = {k: (p.grad.detach().clone() if p.grad is not None else torch.zeros_like(p))
                 for k, p in named}
    nets.reset_state()
    return dict(tokens=np.stack(toks, axis=1), values=values.detach().numpy(),
                rewards=rewards.detach().numpy(), logp=logp.detach().numpy(),
                loss=float(loss.detach()), mean_reward=float(rewards.detach().mean()),
                mean_adv=float(adv.detach().mean()),
                grads=grads, p0=p0, S=S)


def policy_xent_loss(nets, features, captions):
    """train_policy_network's loss (trainers.py:202-257): teacher-forced logits of captions[:, :-1] against
    captions[:, 1:]; row i adds (caplen_i / B) times its mean cross-entropy over its first caplen_i positions.
    Returns (loss, logits)."""
    feats = torch.as_tensor(features).to(nets.dtype)
    caps = torch.as_tensor(captions).long()
    out = policy_logits(nets, feats, caps[:, :-1])
    target = caps[:, 1:]
    B = caps.shape[0]
    loss = 0
    for i in range(B):
        caplen = int(np.nonzero(caps[i].numpy() == 2)[0][0]) + 1
        loss = loss + (caplen / B) * F.cross_entropy(out[i][:caplen], target[i][:caplen])
    return loss, out


def vse_hinge(a, b):
    """The argument of one side's ReLU in VisualSemanticEmbeddingLoss (trainers.py:23-54), beta = 0.2:
    S - diag(S)[:, None] + (beta / N)(1 - I) for S = a b^T."""
    N = a.shape[0]
    sim = a @ b.t()
    return sim - torch.diag(sim).unsqueeze(1) + (0.2 / N) * (1.0 - torch.eye(N, dtype=a.dtype))


def vse_loss(ve, se, masks=None):
    """VisualSemanticEmbeddingLoss (trainers.py:23-54): sum(relu(hinge)) / N for (ve, se) and for (se, ve).  ``masks``
    (two 0/1 tensors) replaces each ReLU's own active set by a given one, so that a high-precision restatement can take
    the decisions of a lower-precision run and measure its arithmetic alone."""
    N = ve.shape[0]
    loss = 0
    for k, (a, b) in enumerate(((ve, se), (se, ve))):
        x = vse_hinge(a, b)
        loss = loss + (F.relu(x) if masks is None else x * masks[k]).sum() / N
    return loss


def reward_vse_loss(nets, features, captions, masks=None):
    """train_reward_network's loss (trainers.py:260-309) from zero state.  Returns (loss, ve, se)."""
    nets.reset_state()
    ve, se = reward_embed(nets, torch.as_tensor(features).to(nets.dtype), torch.as_tensor(captions).long())
    nets.reset_state()
    return vse_loss(ve, se, masks), ve, se


def value_mse_loss(nets, features, captions, prefix_len, gen=None):
    """train_value_network's loss (trainers.py:125-199) from zero states: greedy captions of the policy (or the given
    ``gen``), their rewards under the reward network, MSE of the values of gen[:, :prefix_len] against them.
    Returns (loss, gen, values, rewards)."""
    feats = torch.as_tensor(features).to(nets.dtype)
    if gen is None:
        gen, _ = greedy_decode(nets, feats, np.asarray(captions)[:, 0])
    gen = torch.as_tensor(gen).long()
    nets.reset_state()
    with torch.no_grad():
        rewards = reward_call(nets, feats, gen)
    values = value_call(nets, feats, gen[:, :prefix_len])
    nets.reset_state()
    return F.mse_loss(values, rewards), gen, values, rewards


def network_grads(nets, key, loss_fn):
    """Gradients of loss_fn()[0] w.r.t. one network's parameters, made trainable for the call (the reward network is
    frozen in the A2C step).  Returns (loss_fn's result, {name: grad})."""
    named = nets.network_params(key)
    flags = [p.requires_grad for _, p in named]
    for _, p in named:
        p.requires_grad_(True)
        p.grad = None
    try:
        res = loss_fn()
        res[0].backward()
        grads = {k: p.grad.detach().clone() for k, p in named}
    finally:
        for (_, p), f in zip(named, flags):
            p.requires_grad_(f)
            p.grad = None
    return res, grads


def get_rewards(nets, features, captions):
    """GetRewards from zero state on whole captions (config 3), trainers.py:108-121."""
    nets.reset_state()
    with torch.no_grad():
        r = reward_call(nets, torch.as_tensor(features).to(nets.dtype), torch.as_tensor(captions).long())
    nets.reset_state()
    return r.numpy()
