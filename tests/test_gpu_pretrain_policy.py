"""The policy's cross-entropy pretraining on the fused engine (engine.PolicyPretrainEngine, the unidirectional route of
trainers.train_policy_network) against the float64 restatement of the reference's loss (oracle/ref_port.policy_xent_loss
on ref_port.Nets(dtype=float64)) and against the module route (trainers._train_policy_modules).

Tolerances are the suite's: the loss within 2e-6 relative; each gradient within 2e-5 of the tensor's max |entry| and its
L2 norm within 2e-5 relative.  Where the float32 port itself misses that on a tensor, the bound is 3x the port's error,
as in tests/test_gpu_modules_f64.py."""
import numpy as np
import pytest
import torch

from oracle import ref_port, synth

pytestmark = pytest.mark.gpu

LTOL, GTOL, PORT_FACTOR = 2e-6, 2e-5, 3


def _policy(w, vocab=synth.VOCAB):
    import icrl_b200.models as M
    E = w["policy"]["caption_embedding.weight"]
    net = M.PolicyNetwork(synth.word_to_idx(vocab), pretrained_embeddings=E.numpy() if E.shape[1] != 512 else None)
    net.load_state_dict(w["policy"])
    return net.cuda()


def _captions(seed, B, L=17, vocab=synth.VOCAB):
    """Rows in four kinds, in turn: <END> at column 1, mid-row, a stray <END> mid-row before another in the last column,
    and <END> in the last column only.  <NULL> (0) follows the first <END> except in the stray kind."""
    rs = np.random.RandomState(500 + seed)
    caps = rs.randint(4, vocab, size=(B, L)).astype(np.int64)
    caps[:, 0] = 1
    for b in range(B):
        kind = b % 4
        if kind == 0:
            e = 1
        elif kind == 1:
            e = int(rs.randint(2, L - 1))
        elif kind == 2:
            caps[b, int(rs.randint(2, L - 1))] = 2
            caps[b, L - 1] = 2
            continue
        else:
            e = L - 1
        caps[b, e] = 2
        caps[b, e + 1:] = 0
    return caps


def _features(seed, B):
    return np.random.RandomState(700 + seed).standard_normal((B, 512)).astype(np.float32)


def _reference(w, f, caps, dtype=torch.float64):
    nets = ref_port.Nets(w, dtype=dtype)
    res, grads = ref_port.network_grads(nets, "policy", lambda: ref_port.policy_xent_loss(nets, f, caps))
    return float(res[0].detach()), {k: v.double().numpy() for k, v in grads.items()}


def _grad_errs(got, ref):
    scale = max(float(np.abs(ref).max()), 1e-300)
    nrm, ref_n = float(np.sqrt((got ** 2).sum())), float(np.sqrt((ref ** 2).sum()))
    return float(np.abs(got - ref).max()) / scale, abs(nrm - ref_n) / max(ref_n, 1e-300)


def _check_vs_float64(net, loss, w, f, caps):
    ref_loss, ref = _reference(w, f, caps)
    assert abs(loss - ref_loss) <= LTOL * abs(ref_loss), (loss, ref_loss)
    got = {k: p.grad.detach().double().cpu().numpy() for k, p in net.named_parameters() if p.requires_grad}
    assert sorted(got) == sorted(ref)
    port = None
    for k in ref:
        errs = _grad_errs(got[k], ref[k])
        if max(errs) <= GTOL:
            continue
        if port is None:                       # the float32 port, only when a tensor misses the suite's tolerance
            port = _reference(w, f, caps, torch.float32)[1]
        perr = _grad_errs(port[k].astype(np.float64), ref[k])
        for e, pe in zip(errs, perr):
            assert e <= max(GTOL, PORT_FACTOR * pe), "%s: error %.3e (float32 port %.3e)" % (k, e, pe)
    return got


def _engine(net, **kw):
    from icrl_b200.engine import PolicyPretrainEngine
    return PolicyPretrainEngine(net, **kw)


@pytest.mark.parametrize("B", [512, 2048])
def test_variable_length_captions_vs_float64(B):
    w = synth.make_weights(31)
    net = _policy(w)
    f, caps = _features(31, B), _captions(31, B)
    eng = _engine(net)
    assert eng.decode == "fused"
    loss = eng.xent_step(f, caps)
    _check_vs_float64(net, loss, w, f, caps)


def test_short_rows_only_run_the_steps_they_need():
    """Every row ends by column 5: the decode runs 6 steps, and the loss and gradients are still the reference's."""
    w = synth.make_weights(32)
    net = _policy(w)
    B = 256
    f, caps = _features(32, B), _captions(32, B)
    ends = np.random.RandomState(32).randint(1, 6, size=B)
    ends[0] = 5
    for b, e in enumerate(ends):
        caps[b, e], caps[b, e + 1:] = 2, 0
        caps[b, 1:e] = np.where(caps[b, 1:e] == 2, 7, caps[b, 1:e])
    from icrl_b200.engine import plan_xent
    assert plan_xent(caps)[2] == 6
    eng = _engine(net)
    loss = eng.xent_step(f, caps)
    _check_vs_float64(net, loss, w, f, caps)


def test_frozen_300d_embeddings_vs_float64():
    w = synth.make_weights(33, wordvec_dim=300)
    net = _policy(w)
    assert not net.caption_embedding.weight.requires_grad
    B = 512
    f, caps = _features(33, B), _captions(33, B)
    loss = _engine(net).xent_step(f, caps)
    got = _check_vs_float64(net, loss, w, f, caps)
    assert len(got) == 8 and net.caption_embedding.weight.grad is None


def test_vocabulary_off_the_fused_decode_vs_float64():
    V = 1001
    w = synth.make_weights(34, vocab=V)
    net = _policy(w, V)
    B = 256
    f, caps = _features(34, B), _captions(34, B, vocab=V)
    eng = _engine(net)
    assert eng.decode == "simt"
    loss = eng.xent_step(f, caps)
    _check_vs_float64(net, loss, w, f, caps)


def test_fp32_bptt_gives_the_same_gradients():
    w = synth.make_weights(35)
    B = 512
    f, caps = _features(35, B), _captions(35, B)
    grads, losses = [], []
    for bptt in ("tc", "simt"):
        net = _policy(w)
        eng = _engine(net, policy_bptt=bptt)
        losses.append(eng.xent_step(f, caps))
        assert eng.bptt_reruns == 0
        grads.append(_check_vs_float64(net, losses[-1], w, f, caps))
    assert losses[0] == losses[1]                  # the same decode and loss kernels
    for k in grads[0]:
        assert _grad_errs(grads[0][k], grads[1][k])[0] <= GTOL, k


def test_batch_size_changes_between_minibatches():
    """Consecutive steps of different B and S on one engine (buffers sized for the first step are reused)."""
    w = synth.make_weights(36)
    net = _policy(w)
    eng = _engine(net)
    for B, L, seed in ((384, 17, 36), (100, 17, 37), (513, 9, 38)):
        f, caps = _features(seed, B), _captions(seed, B, L)
        loss = eng.xent_step(f, caps)
        _check_vs_float64(net, loss, w, f, caps)


def test_row_without_end_raises_before_any_launch():
    w = synth.make_weights(37)
    net = _policy(w)
    eng = _engine(net)
    caps = _captions(37, 8)
    caps[3] = 5
    n0 = eng.launches.value
    with pytest.raises(ValueError, match="row 3"):
        eng.xent_step(_features(37, 8), caps)
    assert eng.launches.value == n0


def test_five_epochs_match_the_module_route(tmp_path, monkeypatch):
    """train_policy_network's fused route (FlatAdam) against the module route (torch.optim.Adam) from the same weights and
    torch.randperm draws, five epochs of a 700-row dataset at batch 256 (minibatches of 256, 256 and 188 rows): the logged
    losses and the final parameters agree, and the best-loss checkpoint holds the parameters that produced that loss."""
    import icrl_b200.models as M
    import icrl_b200.trainers as T
    w = synth.make_weights(40)
    N, batch, epochs = 700, 256, 5
    data = {"train_captions": _captions(40, N), "train_image_idxs": np.arange(N), "train_features": _features(40, N),
            "train_urls": np.array(["u"] * N), "word_to_idx": synth.word_to_idx(), "embeddings": None}
    made, logged = [], {"fused": [], "modules": []}
    snaps = []

    def make(*a, **k):
        net = M.PolicyNetwork(*a, **k)
        net.load_state_dict(w["policy"])
        made.append(net)
        return net

    route = ["fused"]

    class Rec:
        def __init__(self, *a, **k):
            pass

        def add_scalar(self, tag, val, step):
            assert tag == "Policy Network-loss"
            logged[route[0]].append(float(val.detach()) if torch.is_tensor(val) else float(val))
            if route[0] == "fused":            # logged after the checkpoint and before the optimizer step
                snaps.append({k: v.detach().clone() for k, v in made[-1].state_dict().items()})

    monkeypatch.setattr(T, "PolicyNetwork", make)
    monkeypatch.setattr(T, "SummaryWriter", Rec)
    paths = {"policy_network": str(tmp_path / "policy.pt")}
    torch.manual_seed(123)
    fused = T.train_policy_network(data, paths, str(tmp_path), False, epochs=epochs, batch_size=batch)
    from icrl_b200.engine import A2CEngine
    assert not any(isinstance(v, A2CEngine) for v in vars(fused).values())        # no engine left on the network
    assert len(logged["fused"]) == epochs * 3

    best = int(np.argmin(logged["fused"]))
    fresh = M.PolicyNetwork(synth.word_to_idx()).cuda()
    fresh.load_state_dict(torch.load(paths["policy_network"], map_location="cuda"))
    for k, v in fresh.state_dict().items():
        assert torch.equal(v, snaps[best][k]), k

    route[0] = "modules"
    torch.manual_seed(123)
    ref = make(synth.word_to_idx()).cuda()
    T._train_policy_modules(ref, data, {"policy_network": str(tmp_path / "modules.pt")}, Rec(), epochs, batch)
    a, b = np.array(logged["fused"]), np.array(logged["modules"])
    assert a.shape == b.shape
    assert float(np.abs(a - b).max() / np.abs(b).max()) <= 1e-5, (a, b)
    assert b[-1] < b[0]                            # it trains
    init = {k: v.cuda() for k, v in w["policy"].items()}
    for (k, p), q in zip(fused.state_dict().items(), ref.state_dict().values()):
        moved = float((q - init[k]).norm())
        assert float((p - q).norm()) <= 1e-3 * moved + 1e-7, (k, float((p - q).norm()), moved)
