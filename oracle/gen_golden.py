"""Generate tests/golden/*.npz by executing the UNMODIFIED reference (build container only).

TEST INFRASTRUCTURE (see oracle/__init__).  Usage:  python -m oracle.gen_golden [--only NAME]

The reference modules are imported from oracle.reference_dir() (oracle/_ref/ or the checkout); the three
packages it imports but this image lacks (h5py, gensim, pycocoevalcap) are stubbed in
sys.modules -- none of them is touched on the A2C path.  Inputs and weights come from
oracle.synth (seeded, portable), so only OUTPUTS are stored.  Gradients are stored as
per-tensor L2 norm + sum + 512 sampled entries (fixed index set), not in full.

What is captured, and how, without editing the reference:
  tokens   np.random.choice wrapped (records each returned index; trainers.py:449/561)
  rewards  trainers.GetRewards wrapped (trainers.py:459/568)
  values   forward hook on a2c_network.value_network (models.py:284)
  logits   forward hook on a2c_network.policy_network, last position (models.py:286)
  loss &c  trainers.SummaryWriter replaced by a recorder (trainers.py:489-491/598-603)
  grads    .grad of a2c_network.parameters() after the call (1 epoch, 1 minibatch)
"""
import argparse
import os
import sys
import tempfile
import types

import numpy as np
import torch

from . import reference_dir, synth

REF = reference_dir() or ""
OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
GRAD_SAMPLES = 512
LOGIT_ROWS = 64
# torch's CPU kernels split some reductions by the intra-op thread count, so the fixtures are reproducible bit for bit
# only with the count they were generated with
THREADS = 8


def import_reference():
    """Stub the absent third-party imports and import the reference's trainers module."""
    if "trainers" in sys.modules and getattr(sys.modules["trainers"], "__file__", "").startswith(REF):
        return sys.modules["trainers"]

    def mod(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m
        return m

    mod("h5py")
    g = mod("gensim")
    g.downloader = mod("gensim.downloader")
    g.models = mod("gensim.models", KeyedVectors=object)
    mod("gensim.models.keyedvectors", BaseKeyedVectors=object)
    g.utils = mod("gensim.utils", simple_preprocess=lambda s: s.split())
    mod("pycocoevalcap")
    for pkg, cls in (("bleu", "Bleu"), ("rouge", "Rouge"), ("cider", "Cider"), ("meteor", "Meteor")):
        mod("pycocoevalcap.%s" % pkg)
        mod("pycocoevalcap.%s.%s" % (pkg, pkg), **{cls: object})
    sys.path.insert(0, REF)
    import trainers  # noqa: the reference's own module
    return trainers


class _Recorder:
    scalars = []

    def __init__(self, *a, **k):
        pass

    def add_scalar(self, tag, val, step):
        _Recorder.scalars.append((tag, float(val)))


def grad_sample_index(numel):
    n = min(numel, GRAD_SAMPLES)
    return np.sort(np.random.RandomState(numel % 100003).choice(numel, n, replace=False))


def summarize_grads(named_grads):
    out = {}
    for k, g in named_grads.items():
        g = np.asarray(g, dtype=np.float32).reshape(-1)
        out["gnorm/" + k] = np.float64(np.sqrt((g.astype(np.float64) ** 2).sum()))
        out["gsum/" + k] = np.float64(g.astype(np.float64).sum())
        out["gsamp/" + k] = g[grad_sample_index(g.size)]
    return out


def build_reference_nets(T, weights, pretrained=False, bidirectional=False):
    w2i = synth.word_to_idx(weights["policy"]["caption_embedding.weight"].shape[0])
    if bidirectional:
        P, V, R = (T.PolicyNetwork(w2i, bidirectional=True), T.ValueNetwork(w2i, bidirectional=True),
                   T.RewardNetwork(w2i, bidirectional=True))
    elif pretrained:          # frozen pretrained word vectors (models.py:61-63): every net gets its own table
        P = T.PolicyNetwork(w2i, pretrained_embeddings=weights["policy"]["caption_embedding.weight"].numpy())
        V = T.ValueNetwork(w2i, pretrained_embeddings=weights["value"]["valrnn.caption_embedding.weight"].numpy())
        R = T.RewardNetwork(w2i, pretrained_embeddings=weights["reward"]["rewrnn.caption_embedding.weight"].numpy())
    else:
        P, V, R = T.PolicyNetwork(w2i), T.ValueNetwork(w2i), T.RewardNetwork(w2i)
    P.load_state_dict(weights["policy"])
    V.load_state_dict(weights["value"])
    R.load_state_dict(weights["reward"])
    R.requires_grad_(False)
    R.train(False)
    A = T.AdvantageActorCriticNetwork(V, P)
    return P, V, R, A


def run_reference_a2c(weights, features, captions, seed, level=None, pretrained=False, bidirectional=False):
    T = import_reference()
    import utilities
    P, V, R, A = build_reference_nets(T, weights, pretrained, bidirectional)
    opt = T.optim.Adam(A.parameters(), lr=1e-4)
    B = captions.shape[0]
    data = {"train_captions": captions, "train_image_idxs": np.arange(B),
            "train_features": features, "train_urls": np.array(["u"] * B)}
    rec = dict(tokens=[], rewards=[], values=[], logits=[])
    orig_choice, orig_rew, orig_sw, orig_perm = np.random.choice, T.GetRewards, T.SummaryWriter, utilities.torch.randperm

    def choice(n, p=None):
        a = orig_choice(n, p=p)
        rec["tokens"].append(int(a))
        return a

    def rewards(f, c, net):
        r = orig_rew(f, c, net)
        rec["rewards"].append(r.detach().numpy()[:, 0].copy())
        return r

    hv = V.register_forward_hook(lambda m, i, o: rec["values"].append(o.detach().numpy()[:, 0].copy()))
    hp = P.register_forward_hook(lambda m, i, o: rec["logits"].append(o.detach().numpy()[:, -1].copy()))
    _Recorder.scalars = []
    np.random.choice, T.GetRewards, T.SummaryWriter = choice, rewards, _Recorder
    utilities.torch.randperm = lambda n: torch.arange(n)
    tmp = tempfile.mkdtemp()
    try:
        np.random.seed(seed)
        if level is None:
            T.a2c_training(data, A, R, opt, tmp, [os.path.join(tmp, "a.pt")], B, 1)
        else:
            T.a2c_curriculum_training(data, A, R, opt, tmp, [os.path.join(tmp, "a.pt")], B, 1, [level])
    finally:
        np.random.choice, T.GetRewards, T.SummaryWriter = orig_choice, orig_rew, orig_sw
        utilities.torch.randperm = orig_perm
        hv.remove()
        hp.remove()
    S = len(rec["values"])
    tokens = np.array(rec["tokens"], dtype=np.int64).reshape(S, B).T
    logits = np.stack(rec["logits"], axis=1)                       # (B,S,V)
    z = torch.from_numpy(logits)
    logp = torch.log(torch.softmax(z, dim=2).gather(2, torch.from_numpy(tokens).unsqueeze(2)))[:, :, 0].numpy()
    grads = {k: p.grad.detach().numpy() for k, p in A.named_parameters() if p.grad is not None}
    sc = dict(_Recorder.scalars)
    loss = [v for k, v in _Recorder.scalars if k.endswith("loss")][0]
    mr = [v for k, v in _Recorder.scalars if k.endswith("mean-rewards")][0]
    ma = [v for k, v in _Recorder.scalars if k.endswith("mean-advantage")][0]
    out = dict(tokens=tokens, values=np.stack(rec["values"], axis=1), rewards=np.stack(rec["rewards"], axis=1),
               logp=logp, last_logits=logits[:, -1], loss=np.float64(loss), mean_reward=np.float64(mr),
               mean_adv=np.float64(ma))
    out.update(summarize_grads(grads))
    return out


def case_a2c(name, seed, B, L, level=None, wordvec_dim=512, bidirectional=False):
    w = synth.make_weights(seed, wordvec_dim=wordvec_dim, bidirectional=bidirectional)
    f, c = synth.make_inputs(seed, B, L)
    out = run_reference_a2c(w, f, c, seed, level, pretrained=wordvec_dim != 512, bidirectional=bidirectional)
    out.update(seed=seed, B=B, L=L, level=-1 if level is None else level, wordvec_dim=wordvec_dim)
    if B > LOGIT_ROWS:          # a fixed, seeded sample of rows of the last step's logits keeps the fixture below 1 MB
        rows = np.sort(np.random.RandomState(0).choice(B, LOGIT_ROWS, replace=False))
        out.update(last_logits=out["last_logits"][rows], last_logits_rows=rows)
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
    print(name, "loss", out["loss"], "tokens", out["tokens"].shape)


def case_greedy(name, seed, B):
    T = import_reference()
    w = synth.make_weights(seed)
    f, _ = synth.make_inputs(seed, B, 17)
    P, _, _, _ = build_reference_nets(T, w)
    caps = np.ones((B, 17), dtype=np.int64)
    last = []
    h = P.register_forward_hook(lambda m, i, o: last.append(o.detach().numpy()[:, -1].copy()))
    with torch.no_grad():
        toks = T.GenerateCaptionsGreedy(f, caps, P).numpy()
    h.remove()
    np.savez_compressed(os.path.join(OUT, name + ".npz"), tokens=toks, last_logits=last[-1], seed=seed, B=B)
    print(name, toks.shape)


def case_rewards(name, seed, B, L):
    T = import_reference()
    w = synth.make_weights(seed)
    f, c = synth.make_inputs(seed, B, L)
    _, _, R, _ = build_reference_nets(T, w)
    with torch.no_grad():
        r = T.GetRewards(torch.from_numpy(f), torch.from_numpy(c), R).numpy()
    np.savez_compressed(os.path.join(OUT, name + ".npz"), rewards=r, seed=seed, B=B, L=L)
    print(name, r.shape, float(r.mean()))


def case_lookahead(name, seed, B, beam=5):
    """Value-guided beam look-ahead (trainers.py:73-105), all `beam` final candidates and their scores."""
    T = import_reference()
    w = synth.make_weights(seed)
    f, _ = synth.make_inputs(seed, B, 17)
    P, V, _, _ = build_reference_nets(T, w)
    caps = np.ones((B, 17), dtype=np.int64)
    V.valrnn.init_hidden()
    with torch.no_grad():
        cands = T.GenerateCaptionsWithActorCriticLookAhead(f, caps, P, V, beamSize=beam, most_likely=False)
    np.savez_compressed(os.path.join(OUT, name + ".npz"), seed=seed, B=B, beam=beam,
                        captions=np.stack([c.numpy() for c, _ in cands]),
                        scores=np.stack([s.numpy().reshape(-1) for _, s in cands]))
    print(name, [float(s.mean()) for _, s in cands])


def case_pretrain(name, seed, B):
    """One minibatch of each supervised pretraining loop of the reference (train_policy_network :202-257,
    train_reward_network :260-309, train_value_network :125-199; SURVEY 8f row 2): loss and gradients.
    The loops construct their networks themselves, so the class names inside the reference's trainers module are
    wrapped by factories that load the synthetic weights right after construction (no source is modified)."""
    import random
    T = import_reference()
    import utilities
    w = synth.make_weights(seed)
    f, c = synth.make_inputs(seed, B, 17)
    data = {"train_captions": c, "train_image_idxs": np.arange(B), "train_features": f,
            "train_urls": np.array(["u"] * B), "word_to_idx": synth.word_to_idx(), "embeddings": None}
    tmp = tempfile.mkdtemp()
    paths = {k: os.path.join(tmp, k + ".pt") for k in ("policy_network", "reward_network", "value_network")}
    torch.save(w["policy"], paths["policy_network"])
    torch.save(w["reward"], paths["reward_network"])
    orig = dict(P=T.PolicyNetwork, V=T.ValueNetwork, R=T.RewardNetwork, sw=T.SummaryWriter, perm=utilities.torch.randperm,
                tqdm=T.tqdm, ri=random.randint)

    def factory(cls, sd):
        def make(*a, **k):
            net = cls(*a, **k)
            net.load_state_dict(sd)
            return net
        return make

    picked = []

    def randint(a, b):
        v = orig["ri"](a, b)
        picked.append(v)
        return v

    T.PolicyNetwork, T.ValueNetwork, T.RewardNetwork = factory(orig["P"], w["policy"]), factory(orig["V"], w["value"]), factory(orig["R"], w["reward"])
    T.SummaryWriter = _Recorder
    utilities.torch.randperm = lambda n: torch.arange(n)
    T.tqdm = lambda it, **k: _Quiet(it)
    random.randint = randint
    out = dict(seed=seed, B=B)
    try:
        for key, fn in (("policy", T.train_policy_network), ("reward", T.train_reward_network), ("value", T.train_value_network)):
            _Recorder.scalars = []
            random.seed(seed)
            net = fn(data, paths, tmp, False, epochs=1, batch_size=B)
            out[key + "_loss"] = np.float64(_Recorder.scalars[0][1])
            grads = {k: p.grad.detach().numpy() for k, p in net.named_parameters()}
            out.update({key + "/" + k: v for k, v in summarize_grads(grads).items()})
            print(name, key, "loss", out[key + "_loss"])
        out["value_prefix_len"] = np.int64(picked[-1])
    finally:
        T.PolicyNetwork, T.ValueNetwork, T.RewardNetwork = orig["P"], orig["V"], orig["R"]
        T.SummaryWriter, utilities.torch.randperm, T.tqdm, random.randint = orig["sw"], orig["perm"], orig["tqdm"], orig["ri"]
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)


class _Quiet:
    """tqdm stand-in: iterable with the two methods the loops call on the progress bar."""

    def __init__(self, it):
        self.it = it

    def __iter__(self):
        return iter(self.it)

    def set_description_str(self, *a, **k):
        pass


CASES = {
    "a2c_b16_l8_wemb300": lambda: case_a2c("a2c_b16_l8_wemb300", 9, 16, 8, wordvec_dim=300),   # SURVEY 8f row 3 (frozen 300-d vectors)
    "a2c_b12_l7_bidir": lambda: case_a2c("a2c_b12_l7_bidir", 10, 12, 7, bidirectional=True),   # SURVEY 8f row 3 (bidirectional RNNs)
    "pretrain_b12": lambda: case_pretrain("pretrain_b12", 8, 12),              # SURVEY 8f row 2
    "lookahead_b6": lambda: case_lookahead("lookahead_b6", 7, 6),              # SURVEY 8f row 1
    "greedy_b32": lambda: case_greedy("greedy_b32", 0, 32),                    # BASELINE config 1
    "a2c_b8_l6": lambda: case_a2c("a2c_b8_l6", 1, 8, 6),
    "a2c_b32_l9": lambda: case_a2c("a2c_b32_l9", 2, 32, 9),
    "a2c_b256_l20": lambda: case_a2c("a2c_b256_l20", 3, 256, 20),              # BASELINE config 2
    "curr_b16_l10_lv4": lambda: case_a2c("curr_b16_l10_lv4", 4, 16, 10, level=4),
    "curr_b24_l20_lv6": lambda: case_a2c("curr_b24_l20_lv6", 5, 24, 20, level=6),
    "rewards_b64_l20": lambda: case_rewards("rewards_b64_l20", 6, 64, 20),     # config 3 shape, small B
}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default=None)
    args = ap.parse_args()
    if not REF or not os.path.isdir(REF):
        raise SystemExit("gen_golden needs the reference sources in oracle/_ref/ or ICRL_REFERENCE_DIR (default /root/reference)")
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(THREADS)
    for name, fn in CASES.items():
        if args.only in (None, name):
            fn()


if __name__ == "__main__":
    main()
