"""The value-guided look-ahead decoder on the fused engine (GenerateCaptionsWithActorCriticLookAhead, trainers.py:73-105):
the tcgen05 chain pieces from a carried state against the serial chain, the policy beam step against torch.topk and
PolicyNetwork.forward, and the whole decoder against the reference's loop on the drop-in modules (_look_ahead_modules)."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import synth
from tests.helpers import make_nets

pytestmark = pytest.mark.gpu

TOL = 2e-6
H = 512


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _st():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _value_operands(A):
    from icrl_b200 import _lib
    rnn = A.value_network.valrnn
    E, lstm = rnn.caption_embedding.weight, rnn.lstm
    V = E.shape[0]
    table = torch.empty(V * 4 * H, device="cuda")
    _lib.call("icrl_pack_gate_table", _st(), V, 4 * H, 4 * H, E.shape[1], _p(E), _p(lstm.weight_ih_l0), _p(lstm.bias_ih_l0),
              _p(lstm.bias_hh_l0), _p(table), None)
    packed = torch.empty(int(_lib.call("icrl_chain_tc_weight_halves", 0)), dtype=torch.float16, device="cuda")
    _lib.call("icrl_pack_chain_tc_weights", _st(), 0, _p(lstm.weight_hh_l0), _p(packed), None)
    return table, packed, lstm.weight_hh_l0


def _serial(tokens, table, W_hh, h0, c0):
    from icrl_b200 import _lib
    T = tokens.numel()
    sh, sc = torch.empty((T + 1, H), device="cuda"), torch.empty((T + 1, H), device="cuda")
    sync = torch.zeros(int(_lib.call("icrl_chain_sync_bytes")), dtype=torch.uint8, device="cuda")
    _lib.call("icrl_chain_lstm_fwd", _st(), _p(tokens), T, _p(table), _p(W_hh), _p(h0), _p(c0), _p(sh), _p(sc), None, None, None,
              _p(sync), None)
    _lib.call("icrl_chain_check", _st(), _p(sync))
    return sh, sc


def _pieces(tokens, table, packed, h0, c0, P, warm, stash_g=False, entry="icrl_chain_tc_lstm_fwd_from"):
    """One tcgen05 launch over `tokens`; returns the stash rows 0..T, the gate stash and the joint-check words."""
    from icrl_b200 import _lib
    T = tokens.numel()
    seg = -(-(T - warm) // P)
    n = P * seg + warm
    stream = torch.zeros(n, dtype=torch.int32, device="cuda")
    stream[:T] = tokens
    sh, sc = torch.empty((n + 1, H), device="cuda"), torch.empty((n + 1, H), device="cuda")
    sg = torch.empty((n, 4 * H), device="cuda") if stash_g else None
    ws = torch.empty((int(_lib.call("icrl_chain_tc_ws_bytes", P)) + 3) // 4, device="cuda")
    cp = torch.empty(int(_lib.call("icrl_chain_tc_cp_floats", P)), device="cuda")
    err = torch.zeros(16, device="cuda")
    if entry == "icrl_chain_tc_fwd":
        _lib.call(entry, _st(), 0, P, seg, warm, _p(stream), _p(table), _p(packed), None, _p(sh), _p(sc), _p(sg), _p(ws), _p(cp),
                  _p(err), None)
    else:
        _lib.call(entry, _st(), P, seg, warm, _p(stream), _p(table), _p(packed), _p(h0), _p(c0), _p(sh), _p(sc), _p(sg), _p(ws),
                  _p(cp), _p(err), None)
    torch.cuda.synchronize()
    return sh[:T + 1], sc[:T + 1], sg, err


def _state(seed):
    g = torch.Generator().manual_seed(seed)
    return (0.5 * torch.randn(H, generator=g)).cuda(), torch.randn(H, generator=g).cuda()


def _stream(seed, T):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(0, synth.VOCAB, (T,), generator=g, dtype=torch.int32).cuda()


def _close(sh, sc, rh, rc):
    eh = float((sh - rh).abs().max())
    ec = float(((sc - rc).abs() / rc.abs().clamp(min=1.0)).max())
    assert eh <= TOL and ec <= TOL, (eh, ec)


def test_chain_pieces_from_a_carried_state_match_the_serial_chain():
    A, _, _ = make_nets(81)
    table, packed, W_hh = _value_operands(A)
    h0, c0 = _state(1)
    tokens = _stream(2, 60000)
    rh, rc = _serial(tokens, table, W_hh, h0, c0)
    sh, sc, _, err = _pieces(tokens, table, packed, h0, c0, P=256, warm=256)
    assert float(err[:2].max()) <= 1e-5
    assert torch.equal(sh[0], h0) and torch.equal(sc[0], c0)
    _close(sh, sc, rh, rc)


def test_two_launches_from_carried_state_match_one_launch_over_the_joined_stream():
    A, _, _ = make_nets(82)
    table, packed, _ = _value_operands(A)
    h0, c0 = _state(3)
    tokens = _stream(4, 50000)
    T1 = 21000
    jh, jc, _, _ = _pieces(tokens, table, packed, h0, c0, P=256, warm=256)
    ah, ac, _, _ = _pieces(tokens[:T1], table, packed, h0, c0, P=128, warm=256)
    bh, bc, _, err = _pieces(tokens[T1:], table, packed, ah[T1].contiguous(), ac[T1].contiguous(), P=128, warm=256)
    assert float(err[:2].max()) <= 1e-5
    _close(torch.cat((ah, bh[1:])), torch.cat((ac, bc[1:])), jh, jc)


def test_chain_pieces_without_a_state_are_bit_identical_to_the_zero_state_launch():
    A, _, _ = make_nets(83)
    table, packed, _ = _value_operands(A)
    tokens = _stream(5, 20000)
    a = _pieces(tokens, table, packed, None, None, P=128, warm=128, stash_g=True)
    b = _pieces(tokens, table, packed, None, None, P=128, warm=128, stash_g=True, entry="icrl_chain_tc_fwd")
    for x, y in zip(a, b):
        assert torch.equal(x, y)


@pytest.mark.parametrize("k", [1, 5, 16])
def test_policy_beam_step_top_k_and_logits(k):
    """First step (R = B rows from the features) and a later step (R = 3B rows gathered from random parents): top-k equal
    to torch.topk of the step's own logits, logits within 1e-5 of PolicyNetwork.forward on the same prefixes."""
    from icrl_b200 import _lib
    from icrl_b200.engine import LookAheadEngine
    A, _, _ = make_nets(84 + k)
    P = A.policy_network
    eng = LookAheadEngine(P, A.value_network)
    eng.pack_weights()
    B, V = 48, synth.VOCAB
    f, _ = synth.make_inputs(84 + k, B, 17)
    fd = torch.from_numpy(f).cuda()
    g = torch.Generator().manual_seed(k)
    first = torch.randint(3, V, (B,), generator=g, dtype=torch.int32).cuda()
    b = eng._bufs

    def step(R, is_first, parent, h_in, c_in, tok):
        h, c, lg = torch.empty((R, H), device="cuda"), torch.empty((R, H), device="cuda"), torch.empty((R, V), device="cuda")
        tv, ti = torch.empty((R, k), device="cuda"), torch.empty((R, k), dtype=torch.int32, device="cuda")
        ws = torch.empty((R * (46 * H + 4 * V) + 3) // 4, device="cuda")
        _lib.call("icrl_lookahead_policy_step", _st(), R, V, k, int(is_first), _p(fd), _p(P.cnn2linear.weight), _p(P.cnn2linear.bias),
                  _p(b["p_table"]), _p(parent), _p(h_in), _p(c_in), _p(tok), _p(b["p_whh_parts"]), _p(b["p_wv_parts"]),
                  _p(P.linear2vocab.bias), _p(h), _p(c), _p(lg), _p(tv), _p(ti), _p(ws), None)
        ref_v, ref_i = torch.topk(lg, k)
        assert torch.equal(ti.long(), ref_i) and torch.equal(tv, ref_v)
        return h, c, lg

    h1, c1, lg1 = step(B, True, None, None, None, first)
    caps = first.long().unsqueeze(1)
    with torch.no_grad():
        ref = P(fd.unsqueeze(0), caps)[:, -1]
    assert float((lg1 - ref).abs().max()) <= 1e-5
    R = 3 * B
    parent = torch.randint(0, B, (R,), generator=g, dtype=torch.int32).cuda()
    tok = torch.randint(3, V, (R,), generator=g, dtype=torch.int32).cuda()
    _, _, lg2 = step(R, False, parent, h1, c1, tok)
    caps2 = torch.stack((first.long()[parent.long()], tok.long()), dim=1)
    with torch.no_grad():
        ref2 = P(fd[parent.long()].unsqueeze(0), caps2)[:, -1]
    assert float((lg2 - ref2).abs().max()) <= 1e-5


def _same_beams(got, ref, tol=2e-5):
    assert len(got) == len(ref)
    for j, ((gc, gs), (rc, rs)) in enumerate(zip(got, ref)):
        assert torch.equal(gc.cpu(), rc.cpu()), "candidate %d differs" % j
        a, r = gs.cpu().numpy().reshape(-1), rs.cpu().numpy().reshape(-1)
        assert np.array_equal(np.isnan(a), np.isnan(r))
        ok = ~np.isnan(r)
        assert not ok.any() or float(np.abs(a[ok] - r[ok]).max()) <= tol


def test_fused_look_ahead_matches_the_module_loop_and_carries_the_value_state():
    import icrl_b200.trainers as T
    A, _, _ = make_nets(91)
    P, Vn = A.policy_network, A.value_network
    B = 64                                        # first step: 5 x 2 x 64 = 640 positions, long enough to cut
    f, c = synth.make_inputs(91, B, 17)
    Vn.valrnn.init_hidden()
    ref1 = T._look_ahead_modules(f, c, P, Vn)
    ref2 = T._look_ahead_modules(f, c, P, Vn)    # from the state the first call left
    ref_hc = [x.clone() for x in Vn.valrnn.hidden_cell]
    Vn.valrnn.init_hidden()
    got1 = T.GenerateCaptionsWithActorCriticLookAhead(f, c, P, Vn)
    eng = P._icrl_lookahead
    assert eng.step_paths.count("pieces") >= 1
    got2 = T.GenerateCaptionsWithActorCriticLookAhead(f, c, P, Vn)
    _same_beams(got1, ref1)
    _same_beams(got2, ref2)
    for x, y in zip(Vn.valrnn.hidden_cell, ref_hc):
        assert float((x.reshape(-1) - y.reshape(-1)).abs().max()) <= TOL
    assert eng.segment_stats["fallbacks"] == 0
    best = T.GenerateCaptionsWithActorCriticLookAhead(f, c, P, Vn, most_likely=True)
    assert tuple(best.shape) == (B, 17) and best.dtype == torch.int64


def test_failed_joint_checks_fall_back_to_the_serial_chain():
    import icrl_b200.trainers as T
    from icrl_b200.engine import LookAheadEngine
    A, _, _ = make_nets(92)
    P, Vn = A.policy_network, A.value_network
    B = 64
    f, c = synth.make_inputs(92, B, 17)
    Vn.valrnn.init_hidden()
    ref = T._look_ahead_modules(f, c, P, Vn)
    Vn.valrnn.init_hidden()
    eng = LookAheadEngine(P, Vn, chain_tol=1e-30)        # far below the joints' rounding: every piece launch fails
    with pytest.warns(UserWarning):
        got = eng.look_ahead(f, c[:, 0])
    _same_beams(got, ref)
    assert len(eng.step_paths) == 16 and "pieces" not in eng.step_paths
    assert eng.segment_stats["fallbacks"] == eng.step_paths.count("fallback") >= 1


def test_bidirectional_networks_and_wide_beams_take_the_module_route(monkeypatch):
    import icrl_b200.models as M
    import icrl_b200.trainers as T
    monkeypatch.setattr(T, "_look_ahead_modules", lambda *a, **k: "modules")
    f, c = synth.make_inputs(93, 4, 17)
    w2i = synth.word_to_idx()
    torch.manual_seed(93)
    P, Vn = M.PolicyNetwork(w2i, bidirectional=True).cuda(), M.ValueNetwork(w2i, bidirectional=True).cuda()
    assert T.GenerateCaptionsWithActorCriticLookAhead(f, c, P, Vn) == "modules"
    A, _, _ = make_nets(93)
    P, Vn = A.policy_network, A.value_network
    assert T.GenerateCaptionsWithActorCriticLookAhead(f, c, P, Vn, beamSize=17) == "modules"
    assert not hasattr(P, "_icrl_lookahead")


def test_a2c_network_caption_dump_matches_the_module_route(tmp_path, monkeypatch):
    import icrl_b200.trainers as T
    A, _, _ = make_nets(94)
    n_img = 30
    f, c = synth.make_inputs(94, n_img, 17)
    data = {"val_captions": c, "val_image_idxs": np.arange(n_img), "val_features": f,
            "val_urls": np.array(["http://img/%d" % i for i in range(n_img)]),
            "idx_to_word": {i: w for w, i in synth.word_to_idx().items()}}

    def run(tag):
        paths = {k: str(tmp_path / (tag + k)) for k in ("real_captions_path", "generated_captions_path", "image_urls_path")}
        np.random.seed(5)
        A.value_network.valrnn.init_hidden()
        T.test_a2c_network(A, data, paths, 24, validation_batch_size=12)
        return [open(paths[k]).read() for k in sorted(paths)]

    fused = run("fused_")
    assert hasattr(A.policy_network, "_icrl_lookahead")
    monkeypatch.setattr(T, "GenerateCaptionsWithActorCriticLookAhead",
                        lambda *a, **k: T._look_ahead_modules(*a, **k))
    assert fused == run("modules_")
    assert all(len(x) > 0 for x in fused)
