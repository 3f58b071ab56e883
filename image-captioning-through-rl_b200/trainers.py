"""The reference's A2C call sites (``trainers.py``) on the fused B200 engine.

Same function names, argument order and return values as the reference
(``GetRewards :108``, ``GenerateCaptionsGreedy :57``, ``a2c_training :402``,
``a2c_curriculum_training :503``, ``train_a2c_network :312``); the per-step Python loop
(``:441-480``) is replaced by one ``A2CEngine.step`` per minibatch.  Sampling consumes numpy's
global MT19937 stream exactly like the reference's ``np.random.choice`` calls (one double per row
per step, step-major), so ``np.random.seed(s)`` reproduces the reference's token ids.

``GenerateCaptionsWithActorCriticLookAhead`` / ``test_a2c_network`` (``:73-105``, ``:619-665``; SURVEY 8f row 1) run
the reference's beam look-ahead on ``engine.LookAheadEngine`` (one tcgen05 value-chain launch per beam step from the
carried value state), bidirectional networks on the drop-in modules.

The supervised pretraining loops (``train_policy_network :202``, ``train_reward_network :260``,
``train_value_network :125``, ``VisualSemanticEmbeddingLoss :23``; SURVEY 8f row 2): ``train_policy_network`` with a
unidirectional policy runs on ``engine.PolicyPretrainEngine`` (teacher-forced fused decode, fused masked cross entropy
and tcgen05 BPTT in one ``xent_step`` per minibatch, ``optim.FlatAdam``).  The bidirectional policy and the reward and
value loops run on the drop-in modules through their autograd wrappers: the recurrent forwards / backwards are the CUDA
kernels, the loss arithmetic on the module outputs (cross entropy, MSE, hinge) is torch host code exactly as in the
reference.  As in the reference, a missing pretrained file makes ``train_a2c_network`` pretrain that network.
"""
import math
import os
import random

import numpy as np
import torch
import torch.optim as optim

from .engine import A2CEngine, PolicyOnlyEngine, PolicyPretrainEngine
from .models import *          # noqa: F401,F403  (torch, nn, F, np, device, MAX_SEQ_LEN, classes)
from .models import AdvantageActorCriticNetwork, PolicyNetwork, RewardNetwork, ValueNetwork, device, MAX_SEQ_LEN

try:                            # tensorboard is optional plumbing (trainers.py:19)
    from torch.utils.tensorboard import SummaryWriter
except Exception:               # pragma: no cover
    class SummaryWriter:        # type: ignore
        def __init__(self, *a, **k):
            pass

        def add_scalar(self, *a, **k):
            pass


def _engine_for(a2c_network, reward_network, entropy_coef=0.0):
    eng = getattr(a2c_network, "_icrl_engine", None)
    if eng is None or eng.reward is not reward_network:
        eng = A2CEngine(a2c_network, reward_network, entropy_coef=entropy_coef)
        object.__setattr__(a2c_network, "_icrl_engine", eng)
    # the cached engine is kept (its flat gradient bucket is the one FlatAdam steps); only the coefficient follows the call
    eng.entropy_coef = float(entropy_coef)
    return eng


def get_coco_minibatches(data, batch_size=100, split="train"):
    """Random-permutation minibatch generator with the reference's tuple contract
    (captions (B,L) int, features (B,512) f32, urls), utilities.py:160-178."""
    n = data["%s_captions" % split].shape[0]
    perm = torch.randperm(n)
    for i in range(0, n, batch_size):
        mask = perm[i:i + batch_size].numpy()
        idxs = data["%s_image_idxs" % split][mask]
        yield data["%s_captions" % split][mask], data["%s_features" % split][idxs], data["%s_urls" % split][idxs]


def global_minibatch_number(epoch, batch_id, batch_size):
    return epoch * batch_size + batch_id            # utilities.py:204-212 (sic)


def save_a2c_model(model, save_paths):
    """Plain state_dict files, one per path (utilities.py:286-296)."""
    for path in ([save_paths] if isinstance(save_paths, str) else list(save_paths)):
        torch.save(model.state_dict(), path)


def load_a2c_models(model_path, train_data, network_paths, bidirectional):
    """Rebuild an A2C network from its checkpoints (utilities.py:299-323): policy and value state dicts first, then the
    a2cNetwork*.pt file over them, all with strict=False; both sub-networks in eval mode."""
    nets = {}
    for key, cls in (("policy_network", PolicyNetwork), ("value_network", ValueNetwork)):
        net = cls(train_data["word_to_idx"], pretrained_embeddings=train_data.get("embeddings"),
                  bidirectional=bidirectional).to(device)
        net.load_state_dict(torch.load(network_paths[key], map_location=device), strict=False)
        nets[key] = net
    a2c_network = AdvantageActorCriticNetwork(nets["value_network"], nets["policy_network"]).to(device)
    a2c_network.load_state_dict(torch.load(model_path, map_location=device), strict=False)
    a2c_network.policy_network.train(mode=False)
    a2c_network.value_network.train(mode=False)
    return a2c_network


def get_filename(base_name, bidirectional, curriculum=None):
    """Checkpoint naming of the reference (utilities.py:326-338): `_bidirectional`, then `_curriculum`, before the extension."""
    name, ext = os.path.splitext(base_name)
    if bidirectional:
        name += "_bidirectional"
    if curriculum:
        name += "_curriculum"
    return name + ext


def GetRewards(features, captions, reward_network):
    """Cosine similarity of the visual and semantic embeddings, (B,1) (trainers.py:108-121).
    Uses and advances ``reward_network.rewrnn.hidden_cell`` like the reference."""
    ve, se = reward_network(features, captions)
    dev = ve.device
    out = torch.empty((ve.shape[0], 1), dtype=torch.float32, device=dev)
    from . import _lib
    import ctypes
    with torch.cuda.device(dev):
        _lib.call("icrl_reward_cosine_fwd", ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream), ve.shape[0], 1,
                  ctypes.c_void_p(ve.data_ptr()), ctypes.c_void_p(se.data_ptr()), ctypes.c_void_p(out.data_ptr()), None)
    return out


def _np(x):
    return x.detach().cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)


def GenerateCaptionsGreedy(features, captions, policy_network):
    """MAX_SEQ_LEN-1 greedy steps from column 0, no early stop: (B,17) int64 (trainers.py:57-70)."""
    features, captions = _np(features), _np(captions)
    if getattr(policy_network, "bidirectional", False):
        # module route (the fused decode kernel is unidirectional): the reference's loop, trainers.py:65-69
        dev = policy_network.linear2vocab.weight.device
        feats = torch.as_tensor(features, device=dev).float().unsqueeze(0)
        gen = torch.as_tensor(captions[:, 0:1], device=dev).long()
        with torch.no_grad():
            for _ in range(MAX_SEQ_LEN - 1):
                gen = torch.cat((gen, policy_network(feats, gen)[:, -1:, :].argmax(dim=2)), dim=1)
        return gen
    eng = getattr(policy_network, "_icrl_greedy", None)
    if eng is None:
        eng = PolicyOnlyEngine(policy_network)
        object.__setattr__(policy_network, "_icrl_greedy", eng)
    tokens, _ = eng.greedy_decode(np.asarray(features, dtype=np.float32), np.asarray(captions)[:, 0], MAX_SEQ_LEN - 1)
    return tokens


def GenerateCaptionsWithActorCriticLookAhead(features, captions, policy_network, value_network, beamSize=5,
                                             most_likely=False):
    """Value-guided beam search of the reference's evaluation path (trainers.py:73-105; SURVEY 8f row 1).

    Keeps `beamSize` candidate caption BATCHES.  Each of the MAX_SEQ_LEN-1 steps expands every candidate with
    the policy's top-`beamSize` words of the last position, scores an expansion as
    ``score - (0.6 * V(features, caption) + 0.4 * log(top-k logit))`` (the reference takes the log of the raw
    top-k logit, a NaN where it is negative -- reproduced, the ordering key is the batch MEAN of the score), and
    keeps the `beamSize` expansions with the smallest mean.  The value network's hidden_cell is carried through
    every call and never reset inside (Q1), exactly as in the reference; callers reset it per batch
    (trainers.py:661).

    Unidirectional networks on CUDA with beamSize <= 16 run on engine.LookAheadEngine: one policy beam step and ONE
    value-chain launch per step (cached on the policy network, like GenerateCaptionsGreedy's engine).  Every other case
    runs the reference's loop on the drop-in modules (_look_ahead_modules)."""
    dev = policy_network.linear2vocab.weight.device
    if (dev.type == "cuda" and 1 <= beamSize <= 16 and not getattr(policy_network, "bidirectional", False)
            and not getattr(value_network, "bidirectional", False)):
        eng = getattr(policy_network, "_icrl_lookahead", None)
        if eng is None or eng.value is not value_network:
            from .engine import LookAheadEngine
            eng = LookAheadEngine(policy_network, value_network)
            object.__setattr__(policy_network, "_icrl_lookahead", eng)
        beam = eng.look_ahead(features, np.asarray(captions)[:, 0], beam=beamSize, steps=MAX_SEQ_LEN - 1)
        return beam[0][0] if most_likely else beam
    return _look_ahead_modules(features, captions, policy_network, value_network, beamSize, most_likely)


def _look_ahead_modules(features, captions, policy_network, value_network, beamSize=5, most_likely=False):
    """GenerateCaptionsWithActorCriticLookAhead as the reference's loop over the drop-in modules (bidirectional networks,
    beamSize > 16, and the reference of the fused path's tests).  Policy and value forwards run on the CUDA kernels;
    top-k, log and the sort are torch plumbing on (B,1,beam) tensors."""
    dev = policy_network.linear2vocab.weight.device
    feats = torch.as_tensor(np.asarray(features), device=dev).float().unsqueeze(0)
    start = torch.as_tensor(np.asarray(captions)[:, 0:1], device=dev).long()
    beam = [(start, 0)]
    with torch.no_grad():
        for _ in range(MAX_SEQ_LEN - 1):
            grown = []
            for cap, score in beam:
                logits = policy_network(feats, cap)[:, -1:, :]
                top, words = torch.topk(logits, beamSize)
                for i in range(beamSize):
                    longer = torch.cat((cap, words[:, :, i]), dim=1)
                    value = value_network(feats.squeeze(0), longer).detach()
                    grown.append((longer, score - (0.6 * value + 0.4 * torch.log(top[:, :, i]))))
            grown.sort(key=lambda cs: cs[1].mean())
            beam = grown[:beamSize]
    return beam[0][0] if most_likely else beam


def decode_captions(captions, idx_to_word):
    """ids -> sentences, stopping at <END> and skipping <NULL> (utilities.py:116-140)."""
    caps = np.asarray(captions.cpu() if isinstance(captions, torch.Tensor) else captions)
    single = caps.ndim == 1
    caps = caps[None] if single else caps
    out = []
    for row in caps:
        words = []
        for t in row:
            w = idx_to_word[int(t)]
            if w != "<NULL>":
                words.append(w)
            if w == "<END>":
                break
        out.append(" ".join(words))
    return out[0] if single else out


def test_a2c_network(a2c_network, test_data, image_caption_data, data_size, validation_batch_size=128):
    """Validation-set caption dump with the look-ahead decoder (trainers.py:619-665): appends real captions,
    generated captions and urls to the three files, resetting the value RNN state after every batch.  The
    reference slices `i : i + validation_batch_size - 1` (one row of every batch is skipped) -- kept."""
    a2c_network.train(False)
    n = min(int(data_size), test_data["val_captions"].shape[0])
    mask = np.random.choice(test_data["val_captions"].shape[0], n)            # get_coco_batch, utilities.py:143-157
    caps_all = test_data["val_captions"][mask]
    idxs = test_data["val_image_idxs"][mask]
    feats_all, urls_all = test_data["val_features"][idxs], test_data["val_urls"][idxs]
    with open(image_caption_data["real_captions_path"], "a") as f_real, \
            open(image_caption_data["generated_captions_path"], "a") as f_gen, \
            open(image_caption_data["image_urls_path"], "a") as f_url:
        for i in range(0, len(caps_all), validation_batch_size):
            sl = slice(i, i + validation_batch_size - 1)
            if len(caps_all[sl]) == 0:
                continue
            gen = GenerateCaptionsWithActorCriticLookAhead(feats_all[sl], caps_all[sl], a2c_network.policy_network,
                                                           a2c_network.value_network, most_likely=True)
            f_real.write("\n".join(decode_captions(caps_all[sl], test_data["idx_to_word"])))
            f_gen.write("\n".join(decode_captions(gen, test_data["idx_to_word"])))
            f_url.write("\n".join(str(u) for u in urls_all[sl]))
            a2c_network.value_network.valrnn.init_hidden()


def VisualSemanticEmbeddingLoss(visuals, semantics):
    """Bidirectional hinge ranking loss of the reward pretraining (trainers.py:23-54), beta = 0.2:
    sum(relu(S - diag(S)[:,None] + (beta/N)(1 - I))) / N for S = V S^T and for its transpose."""
    from .models import _LinearFn
    N = visuals.shape[0]
    margin = (0.2 / N) * (1.0 - torch.eye(N, device=visuals.device))
    zero = torch.zeros(N, device=visuals.device)

    def side(a, b):
        sim = _LinearFn.apply(a, b, zero)                      # a b^T on the library GEMM (with autograd)
        return torch.relu(sim - torch.diag(sim).unsqueeze(1) + margin).sum() / N

    return side(visuals, semantics) + side(semantics, visuals)


def _minibatches(train_data, batch_size):
    return get_coco_minibatches(train_data, batch_size=batch_size, split="train")


def train_policy_network(train_data, network_paths, plot_dir, bidirectional, epochs=100, batch_size=512):
    """Cross-entropy pretraining of the policy (trainers.py:202-257): teacher-forced logits of captions[:, :-1]
    against captions[:, 1:], each row weighted by caplen/B and averaged over its first caplen positions.

    The unidirectional policy runs on engine.PolicyPretrainEngine: features resident in HBM (get_coco_minibatches_device,
    the same torch.randperm draw), one xent_step per minibatch (teacher-forced fused decode, fused cross entropy, policy
    BPTT) and Adam(lr=1e-3) as optim.FlatAdam.  The bidirectional policy runs the reference's loop on the drop-in modules
    (_train_policy_modules)."""
    policy_network = PolicyNetwork(train_data["word_to_idx"], pretrained_embeddings=train_data.get("embeddings"),
                                   bidirectional=bidirectional).to(device)
    writer = SummaryWriter(log_dir=os.path.join(plot_dir, "runs"))
    if bidirectional:
        return _train_policy_modules(policy_network, train_data, network_paths, writer, epochs, batch_size)
    from .optim import FlatAdam
    eng = PolicyPretrainEngine(policy_network)
    optimizer = FlatAdam(eng, lr=0.001)
    best = float("inf")
    for epoch in range(epochs):
        for minibatch_id, (captions, features, _) in enumerate(get_coco_minibatches_device(train_data, eng, batch_size)):
            loss = eng.xent_step(features, captions)
            if loss < best:
                best = loss           # saved before the step: the checkpoint holds the parameters that gave this loss
                torch.save(policy_network.state_dict(), network_paths["policy_network"])
            writer.add_scalar("Policy Network-loss", loss, global_minibatch_number(epoch, minibatch_id, batch_size))
            optimizer.step()
    return policy_network


def _train_policy_modules(policy_network, train_data, network_paths, writer, epochs, batch_size):
    """train_policy_network as the reference's loop over the drop-in modules (bidirectional policy, and the reference of
    the fused route's tests): autograd through the policy's CUDA forward / backward, one CrossEntropyLoss per row."""
    criterion = nn.CrossEntropyLoss().to(device)
    optimizer = optim.Adam(policy_network.parameters(), lr=0.001)
    best = float("inf")
    for epoch in range(epochs):
        for minibatch_id, (captions, features, _) in enumerate(_minibatches(train_data, batch_size)):
            feats = torch.as_tensor(np.asarray(features), device=device).float().unsqueeze(0)
            caps_in = torch.as_tensor(captions[:, :-1], device=device).long()
            caps_out = torch.as_tensor(captions[:, 1:], device=device).long()
            output = policy_network(feats, caps_in)
            loss = 0
            for i in range(captions.shape[0]):
                caplen = int(np.nonzero(captions[i] == 2)[0][0]) + 1          # <END> = 2 marks the caption length
                loss = loss + (caplen / captions.shape[0]) * criterion(output[i][:caplen], caps_out[i][:caplen])
            if loss.item() < best:
                best = loss.item()
                torch.save(policy_network.state_dict(), network_paths["policy_network"])
            writer.add_scalar("Policy Network-loss", loss, global_minibatch_number(epoch, minibatch_id, batch_size))
            optimizer.zero_grad()
            loss.backward()
            optimizer.step()
    return policy_network


def train_reward_network(train_data, network_paths, plot_dir, bidirectional, epochs=50, batch_size=512):
    """Visual-semantic-embedding pretraining of the reward network (trainers.py:260-309)."""
    writer = SummaryWriter(log_dir=os.path.join(plot_dir, "runs"))
    reward_network = RewardNetwork(train_data["word_to_idx"], pretrained_embeddings=train_data.get("embeddings"),
                                   bidirectional=bidirectional).to(device)
    optimizer = optim.Adam(reward_network.parameters(), lr=0.0001)
    best = float("inf")
    for epoch in range(epochs):
        for minibatch_id, (captions, features, _) in enumerate(_minibatches(train_data, batch_size)):
            feats = torch.as_tensor(np.asarray(features), device=device).float()
            caps = torch.as_tensor(captions, device=device).long()
            ve, se = reward_network(feats, caps)
            loss = VisualSemanticEmbeddingLoss(ve, se)
            if loss.item() < best:
                best = loss.item()
                torch.save(reward_network.state_dict(), network_paths["reward_network"])
            writer.add_scalar("Reward Network-loss", loss, global_minibatch_number(epoch, minibatch_id, batch_size))
            optimizer.zero_grad()
            loss.backward(retain_graph=True)
            optimizer.step()
            reward_network.rewrnn.init_hidden()
    return reward_network


def train_value_network(train_data, network_paths, plot_dir, bidirectional, epochs=50, batch_size=512):
    """MSE pretraining of the value network (trainers.py:125-199): greedy captions of the frozen policy, their
    reward under the frozen reward network, and the value of a random-length prefix regressed onto it."""
    writer = SummaryWriter(log_dir=os.path.join(plot_dir, "runs"))
    frozen = {}
    for key, cls in (("reward_network", RewardNetwork), ("policy_network", PolicyNetwork)):
        net = cls(train_data["word_to_idx"], pretrained_embeddings=train_data.get("embeddings"),
                  bidirectional=bidirectional).to(device)
        net.load_state_dict(torch.load(network_paths[key], map_location=device), strict=False)
        net.train(False)
        net.requires_grad_(False)
        frozen[key] = net
    reward_network, policy_network = frozen["reward_network"], frozen["policy_network"]
    value_network = ValueNetwork(train_data["word_to_idx"], pretrained_embeddings=train_data.get("embeddings"),
                                 bidirectional=bidirectional).to(device)
    criterion = nn.MSELoss().to(device)
    optimizer = optim.Adam(value_network.parameters(), lr=0.001)
    value_network.train(mode=True)
    best = float("inf")
    for epoch in range(epochs):
        for minibatch_id, (captions, features, _) in enumerate(_minibatches(train_data, batch_size)):
            feats = torch.as_tensor(np.asarray(features), device=device).float()
            gen = GenerateCaptionsGreedy(feats, captions, policy_network)
            rewards = GetRewards(feats, gen, reward_network)
            values = value_network(feats, gen[:, :random.randint(1, MAX_SEQ_LEN)])
            loss = criterion(values, rewards)
            if loss.item() < best:
                best = loss.item()
                torch.save(value_network.state_dict(), network_paths["value_network"])
            writer.add_scalar("Value Network-loss", loss, global_minibatch_number(epoch, minibatch_id, batch_size))
            optimizer.zero_grad()
            loss.backward(retain_graph=True)
            optimizer.step()
            value_network.valrnn.init_hidden()
            reward_network.rewrnn.init_hidden()
    return value_network


class _ModuleRouteResult:
    def __init__(self, loss, mean_reward, mean_adv, mean_entropy=None):
        self.loss, self.mean_reward, self.mean_adv, self.mean_entropy = loss, mean_reward, mean_adv, mean_entropy


def _module_route_step(a2c_network, reward_network, features, captions, level, entropy_coef=0.0):
    """One minibatch through the modules' autograd instead of the fused engine (used for the bidirectional variant):
    the reference's loop body, trainers.py:428-479 / 544-593.  Leaves the gradients in .grad; returns None when the
    curriculum level does not fit (trainers.py:550).  entropy_coef != 0 subtracts entropy_coef times the mean entropy
    of the sampled steps' softmax from the loss (A2CEngine's entropy bonus); autograd carries it into the policy."""
    from .engine import plan_rollout
    p0, S = plan_rollout(captions, level)
    if p0 < 1:
        return None
    dev = a2c_network.policy_network.linear2vocab.weight.device
    feats = torch.as_tensor(np.asarray(features), device=dev).float()
    caps_in = torch.as_tensor(np.asarray(captions)[:, :p0], device=dev).long()
    values, rewards, log_probs, entropies = [], [], [], []
    for _ in range(S):
        value, logits = a2c_network(feats, caps_in)
        if entropy_coef:
            z = logits[:, 0, :]
            entropies.append(-(F.softmax(z, dim=1) * F.log_softmax(z, dim=1)).sum(dim=1))
        probs = F.softmax(logits, dim=2)
        dist = probs.detach().cpu().numpy()[:, 0]
        acts = [np.random.choice(probs.shape[-1], p=dist[i]) for i in range(dist.shape[0])]     # trainers.py:447-450
        gen = torch.from_numpy(np.array(acts)).unsqueeze(-1).to(dev)
        caps_in = torch.cat((caps_in, gen), dim=1)
        log_probs.append(torch.log(probs[:, 0, :].gather(1, gen)))
        rewards.append(GetRewards(feats, caps_in, reward_network))
        values.append(value)
    values = torch.stack(values, dim=1).squeeze()
    rewards = torch.stack(rewards, dim=1).squeeze()
    log_probs = torch.stack(log_probs, dim=1).squeeze()
    advantage = values - rewards
    loss = (-log_probs * advantage).mean() + 0.5 * advantage.pow(2).mean()
    mean_entropy = None
    if entropy_coef:
        mean_entropy = torch.stack(entropies, dim=1).mean()
        loss = loss - entropy_coef * mean_entropy
        mean_entropy = float(mean_entropy.detach())
    for p in a2c_network.parameters():
        p.grad = None
    loss.backward()
    return _ModuleRouteResult(float(loss), float(rewards.mean()), float(advantage.mean()), mean_entropy)


def get_coco_minibatches_device(data, eng, batch_size=100, split="train"):
    """get_coco_minibatches (utilities.py:160-178) with the feature matrix resident in HBM (SURVEY 8f row 4): it is uploaded
    once per (split, device); every minibatch draws the same torch.randperm slice as the reference, sends only the B image
    indices to the device and gathers the B feature rows there (icrl_gather_rows).  Yields the reference's tuple with the
    features as a (B,512) CUDA tensor, which A2CEngine.step / prepare take without a host->device copy."""
    cache = data.setdefault("_icrl_device_features", {})
    key = (split, str(eng.device))
    if key not in cache:
        cache[key] = torch.as_tensor(np.ascontiguousarray(data["%s_features" % split]), dtype=torch.float32).to(eng.device).contiguous()
    feats = cache[key]
    n = data["%s_captions" % split].shape[0]
    perm = torch.randperm(n)
    for i in range(0, n, batch_size):
        mask = perm[i:i + batch_size].numpy()
        idxs = data["%s_image_idxs" % split][mask]
        yield data["%s_captions" % split][mask], eng.gather_rows(feats, idxs), data["%s_urls" % split][idxs]


def _run_minibatches(train_data, a2c_network, reward_network, optimizer, writer, batch_size, epoch, level, tag, best,
                     entropy_coef=0.0):
    bidir = getattr(a2c_network.policy_network, "bidirectional", False)
    eng = None if bidir else _engine_for(a2c_network, reward_network, entropy_coef)
    batches = get_coco_minibatches(train_data, batch_size=batch_size) if bidir else \
        get_coco_minibatches_device(train_data, eng, batch_size=batch_size)
    for minibatch_id, (captions, features, _) in enumerate(batches):
        res = (_module_route_step(a2c_network, reward_network, features, captions, level, entropy_coef) if bidir
               else eng.step(features, captions, level=level))
        if res is not None:                           # curriculum: prefix shorter than 1 => skipped (trainers.py:550)
            optimizer.step()                          # gradients already sit in .grad (flat bucket)
            loss = res.loss
            best = min(best, loss)
            n = global_minibatch_number(epoch, minibatch_id, batch_size)
            writer.add_scalar(tag + "loss", loss, n)
            writer.add_scalar(tag + "mean-rewards", res.mean_reward, n)
            writer.add_scalar(tag + "mean-advantage", res.mean_adv, n)
            if entropy_coef:
                writer.add_scalar(tag + "mean-entropy", res.mean_entropy, n)
        # trainers.py:495-496 / :611-612 -- the engine always starts its chains from zero state;
        # the module-level carried state is reset too so mixed use stays consistent
        reward_network.rewrnn.init_hidden()
        a2c_network.value_network.valrnn.init_hidden()
    return best


def a2c_training(train_data, a2c_network, reward_network, optimizer, plot_dir, save_paths, batch_size, epochs,
                 entropy_coef=0.0):
    """trainers.py:402-500.  entropy_coef: weight of the entropy bonus (A2CEngine); 0 is the reference's loss."""
    writer = SummaryWriter(log_dir=os.path.join(plot_dir, "runs"))
    best = float("inf")
    for epoch in range(epochs):
        best = _run_minibatches(train_data, a2c_network, reward_network, optimizer, writer, batch_size, epoch, None,
                                "A2C Network-episodic-", best, entropy_coef)
        save_a2c_model(a2c_network, save_paths)
    return a2c_network


def a2c_curriculum_training(train_data, a2c_network, reward_network, optimizer, plot_dir, save_paths, batch_size,
                            epochs, curriculum, entropy_coef=0.0):
    """trainers.py:503-616: for each level, rollouts start from the ground-truth prefix
    captions[:, :caplen-level] and sample `level` tokens (the entropy bonus, when set, over those `level` steps)."""
    writer = SummaryWriter(log_dir=os.path.join(plot_dir, "runs"))
    for level in curriculum:
        best = float("inf")
        for epoch in range(epochs):
            best = _run_minibatches(train_data, a2c_network, reward_network, optimizer, writer, batch_size, epoch,
                                    level, "A2C Curriculum Level-%s-" % level, best, entropy_coef)
            save_a2c_model(a2c_network, save_paths)
    return a2c_network


def train_a2c_network(train_data, save_paths, network_paths, plot_dir, bidirectional, epochs, batch_size,
                      retrain_all=False, curriculum=None, entropy_coef=0.0):
    """trainers.py:312-399: build the three networks, load the pretrained state dicts
    (``torch.load(path, map_location=device)`` + ``load_state_dict(strict=False)``), freeze the
    reward network, wrap, Adam(lr=1e-4), dispatch.  entropy_coef > 0 adds the entropy bonus
    ``- entropy_coef * mean policy entropy`` to the A2C loss and logs ``<tag>mean-entropy``; the default 0 is the
    reference's loss."""
    w2i, emb = train_data["word_to_idx"], train_data.get("embeddings")
    trainers_ = {"reward_network": train_reward_network, "policy_network": train_policy_network,
                 "value_network": train_value_network}
    nets = {}
    for key, cls in (("reward_network", RewardNetwork), ("policy_network", PolicyNetwork), ("value_network", ValueNetwork)):
        if retrain_all or not os.path.exists(network_paths[key]):
            # trainers.py:330-370: retrain everything, or fall back to pretraining the network whose file is missing
            nets[key] = trainers_[key](train_data, network_paths, plot_dir, bidirectional, batch_size=batch_size)
            continue
        net = cls(w2i, pretrained_embeddings=emb, bidirectional=bidirectional).to(device)
        net.load_state_dict(torch.load(network_paths[key], map_location=device), strict=False)
        nets[key] = net
    reward_network = nets["reward_network"]
    reward_network.requires_grad_(False)
    reward_network.train(False)
    a2c_network = AdvantageActorCriticNetwork(nets["value_network"], nets["policy_network"]).to(device)
    a2c_network.train(True)
    if bidirectional:
        optimizer = optim.Adam(a2c_network.parameters(), lr=0.0001)          # module route: torch's own Adam (trainers.py:378)
    else:
        # fused route: the same Adam(lr=1e-4) as ONE kernel over the flat gradient bucket the engine fills (optim.FlatAdam;
        # torch's update operation by operation, <= 2e-7 from torch.optim.Adam over 3 steps)
        from .optim import FlatAdam
        optimizer = FlatAdam(_engine_for(a2c_network, reward_network, entropy_coef), lr=0.0001)
    paths = [save_paths["model_path"], network_paths["a2c_network"]]
    if curriculum is None:
        a2c_network = a2c_training(train_data, a2c_network, reward_network, optimizer, plot_dir, paths, batch_size, epochs,
                                   entropy_coef)
    else:
        if 16 not in curriculum:
            curriculum.append(16)                    # trainers.py:389-390
        a2c_network = a2c_curriculum_training(train_data, a2c_network, reward_network, optimizer, plot_dir, paths,
                                              batch_size, epochs, curriculum, entropy_coef)
    with open(save_paths["results_path"], "a") as fh:
        fh.write("\n" + "-" * 10 + " network " + "-" * 10 + "\n" + str(a2c_network) + "\n" + "-" * 10 + " network "
                 + "-" * 10 + "\n")
    return a2c_network
