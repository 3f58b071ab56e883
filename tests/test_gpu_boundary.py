"""GPU tests of the drop-in boundary itself (SURVEY.md 8b): network construction / checkpoint loading
(`train_a2c_network`, trainers.py:312-399), the UNMODIFIED reference training loop running on the drop-in `models`
module (north_star: "keeps the trainers.py call sites"), and engine caches that must follow parameter changes."""
import importlib.util
import os
import sys
import types

import numpy as np
import pytest
import torch

from oracle import reference_dir, synth
from tests.helpers import check_grads_vs_golden, load_case, make_nets, named_grads

pytestmark = pytest.mark.gpu

TOL, GTOL = 2e-6, 2e-5


def _train_data(seed, n, L):
    f, c = synth.make_inputs(seed, n, L)
    return {"train_captions": c, "train_image_idxs": np.arange(n), "train_features": f,
            "train_urls": np.array(["u"] * n), "word_to_idx": synth.word_to_idx(), "embeddings": None}


def test_train_a2c_network_loads_checkpoints_and_trains(tmp_path):
    """train_a2c_network (trainers.py:312-399): three bare state_dict files written by the reference's key names are
    loaded (torch.load + load_state_dict(strict=False)), the reward network is frozen, Adam(lr=1e-4) drives
    a2c_curriculum_training with `[16]` appended to the curriculum (:389-390), the result is saved to both paths
    (utilities.py:286-296) and appended to results_path.  The first minibatch is checked against a fresh engine."""
    import icrl_b200.trainers as T
    from icrl_b200.engine import A2CEngine
    seed, n, L = 401, 48, 20
    w = synth.make_weights(seed)
    paths = {k: str(tmp_path / ("%sNetwork.pt" % k)) for k in ("policy", "value", "reward")}
    for k in ("policy", "value", "reward"):
        torch.save(w[k], paths[k])
    network_paths = {"policy_network": paths["policy"], "value_network": paths["value"], "reward_network": paths["reward"],
                     "a2c_network": str(tmp_path / "a2cNetwork_curriculum.pt")}
    save_paths = {"model_path": str(tmp_path / "log_a2c.pt"), "results_path": str(tmp_path / "results.txt")}
    data = _train_data(seed, n, L)
    # expected first minibatch: level 3 on the whole (identity-permuted) data set
    A0, R0, _ = make_nets(seed)
    e0 = A2CEngine(A0, R0)
    np.random.seed(5)
    r0 = e0.step(data["train_features"], data["train_captions"], level=3)
    first_loss = r0.loss
    before = {k: v.clone() for k, v in A0.state_dict().items()}

    calls = []
    orig_step, orig_perm = A2CEngine.step, T.torch.randperm

    def spy(self, *a, **k):
        res = orig_step(self, *a, **k)
        calls.append((k.get("level"), None if res is None else res.loss))
        return res

    A2CEngine.step, T.torch.randperm = spy, (lambda m: torch.arange(m))
    try:
        np.random.seed(5)
        curriculum = [3]
        net = T.train_a2c_network(data, save_paths, network_paths, str(tmp_path), False, 1, n, curriculum=curriculum)
    finally:
        A2CEngine.step, T.torch.randperm = orig_step, orig_perm
    assert curriculum == [3, 16]                                   # trainers.py:389-390
    assert [lv for lv, _ in calls] == [3, 16]
    assert abs(calls[0][1] - first_loss) <= TOL                    # same weights, same uniforms as the fresh engine
    sd = torch.load(network_paths["a2c_network"], map_location="cpu")
    sd2 = torch.load(save_paths["model_path"], map_location="cpu")
    assert set(sd) == set(before) and all(torch.equal(sd[k], sd2[k]) for k in sd)
    moved = sum(float((sd[k] - before[k].cpu()).abs().max()) > 0 for k in sd)
    assert moved == len(sd), "every one of the 18 tensors must have been updated by Adam"
    assert max(float((sd[k] - before[k].cpu()).abs().max()) for k in sd) <= 2.1e-4    # two Adam steps of lr 1e-4
    assert "AdvantageActorCriticNetwork" in open(save_paths["results_path"]).read()


def _import_reference_trainers(ref_dir):
    """The reference's own trainers.py / utilities.py / metrics.py, unmodified, with `models` resolved to the drop-in
    module (INTEGRATION.md section 1) and the three absent third-party packages stubbed (SURVEY.md 8c)."""
    import icrl_b200.models as drop_in

    def mod(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m
        return m

    saved = {k: sys.modules.get(k) for k in ("models", "trainers", "utilities", "metrics")}
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
    sys.modules["models"] = drop_in
    loaded = {}
    for name in ("metrics", "utilities", "trainers"):
        spec = importlib.util.spec_from_file_location(name, os.path.join(ref_dir, name + ".py"))
        m = importlib.util.module_from_spec(spec)
        sys.modules[name] = m
        spec.loader.exec_module(m)
        loaded[name] = m

    def restore():
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v

    return loaded["trainers"], loaded["utilities"], restore


@pytest.mark.parametrize("name", ["a2c_b8_l6", "curr_b16_l10_lv4"])
def test_unmodified_reference_loop_runs_on_dropin_models(name, tmp_path):
    """`sys.modules["models"] = icrl_b200.models`, then the reference's OWN a2c_training / a2c_curriculum_training
    (imported from its source file, not restated) trains the drop-in networks: sampled tokens, the three logged scalars
    and all 18 gradients equal the golden fixtures the unmodified reference produced on its own models.
    Needs the reference sources: the copy __graft_entry__.build() installs in oracle/_ref/, or the checkout itself
    (ICRL_REFERENCE_DIR, by default /root/reference); skipped where neither exists."""
    ref_dir = reference_dir()
    if ref_dir is None:
        pytest.skip("reference sources not found in oracle/_ref/ or ICRL_REFERENCE_DIR (default /root/reference)")
    g, seed, f, c, u, level = load_case(name)
    A, R, w = make_nets(seed)
    T, U, restore = _import_reference_trainers(ref_dir)
    scalars, tokens = [], []

    class Writer:
        def __init__(self, *a, **k):
            pass

        def add_scalar(self, tag, value, step):
            scalars.append((tag, float(value)))

        def close(self):
            pass

    orig_choice, orig_perm = np.random.choice, U.torch.randperm

    def choice(n, p=None):
        a = orig_choice(n, p=p)
        tokens.append(int(a))
        return a

    B = c.shape[0]
    data = {"train_captions": c, "train_image_idxs": np.arange(B), "train_features": f, "train_urls": np.array(["u"] * B)}
    opt = torch.optim.Adam(A.parameters(), lr=1e-4)
    step_calls = []
    opt_step = opt.step
    opt.step = lambda *a, **k: step_calls.append(1)                 # keep the gradients of the single minibatch readable
    T.SummaryWriter, np.random.choice = Writer, choice
    U.torch.randperm = lambda m: torch.arange(m)
    try:
        np.random.seed(seed)
        if level is None:
            T.a2c_training(data, A, R, opt, str(tmp_path), [str(tmp_path / "a.pt")], B, 1)
        else:
            T.a2c_curriculum_training(data, A, R, opt, str(tmp_path), [str(tmp_path / "a.pt")], B, 1, [level])
    finally:
        np.random.choice = orig_choice
        U.torch.randperm = orig_perm
        restore()
    S = g["tokens"].shape[1]
    assert step_calls == [1]
    assert np.array_equal(np.array(tokens, dtype=np.int64).reshape(S, B).T, g["tokens"])
    loss = [v for k, v in scalars if k.endswith("loss")][0]
    mr = [v for k, v in scalars if k.endswith("mean-rewards")][0]
    ma = [v for k, v in scalars if k.endswith("mean-advantage")][0]
    assert abs(loss - float(g["loss"])) <= TOL and abs(mr - float(g["mean_reward"])) <= TOL and abs(ma - float(g["mean_adv"])) <= TOL
    check_grads_vs_golden(named_grads(A), g, GTOL)
    assert os.path.exists(str(tmp_path / "a.pt"))                   # save_a2c_model of the reference wrote the drop-in's state_dict


def test_reward_operands_follow_in_place_weight_changes():
    """The engine packs the frozen reward network's derived operands (gate table, fp16 split of W_hh) once.  If the
    reward parameters are then changed in place (load_state_dict, more reward pretraining on the same object), the next
    call must repack: rewards equal those of a fresh engine on the new weights, not a mix of stale and fresh operands."""
    from icrl_b200.engine import A2CEngine
    seed, B, L = 421, 256, 12
    A, R, w = make_nets(seed)
    f, c = synth.make_inputs(seed, B, L)
    eng = A2CEngine(A, R)
    r_old = eng.get_rewards(f, c).clone()
    w2 = synth.make_weights(seed + 1)
    R.load_state_dict(w2["reward"])
    r_new = eng.get_rewards(f, c)
    A2, R2, _ = make_nets(seed + 1)
    r_fresh = A2CEngine(A2, R2).get_rewards(f, c)
    assert float((r_new - r_fresh).abs().max()) <= TOL
    assert float((r_new - r_old).abs().max()) > 1e-3
    u = synth.make_uniforms(seed, L - 1, B)
    res = eng.step(f, c, uniforms=u, backward=False)
    R.load_state_dict(w["reward"])
    res2 = eng.step(f, c, uniforms=u, backward=False)
    A3, R3, _ = make_nets(seed)
    ref = A2CEngine(A3, R3).step(f, c, uniforms=u, backward=False)
    assert float((res2["rewards"] - ref["rewards"]).abs().max()) <= TOL
    assert float((res["rewards"] - ref["rewards"]).abs().max()) > 1e-3
