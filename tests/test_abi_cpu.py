"""CPU-side checks of the boundary: the shared library builds, loads, and exports every symbol the
header declares with the argument count the ctypes binding uses; the product path refuses to run
without CUDA (no CPU fallback); the host-side planning logic matches the reference's rules."""
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from icrl_b200 import _lib
    return _lib


def _header_decls():
    txt = open(os.path.join(ROOT, "include", "icrl_b200.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    decls = {}
    for m in re.finditer(r"\b(icrl_\w+)\s*\(([^;{]*?)\)\s*;", txt, flags=re.S):
        args = m.group(2).strip()
        n = 0 if args in ("", "void") else len([a for a in args.split(",") if a.strip()])
        decls[m.group(1)] = n
    return decls


def test_library_exports_every_declared_symbol(lib):
    handle = lib.load()
    decls = _header_decls()
    assert len(decls) >= 20
    for name, nargs in decls.items():
        assert hasattr(handle, name), "missing export " + name
        assert name in lib.SIGNATURES, "no ctypes signature for " + name
        assert len(lib.SIGNATURES[name]) == nargs, "%s: header has %d args, binding %d" % (name, nargs, len(lib.SIGNATURES[name]))
    assert handle.icrl_version() >= 100


def test_host_helpers_without_gpu(lib):
    # pure host arithmetic of the ABI (no device work)
    assert lib.call("icrl_stream_len", 256, 1, 19, 0) == 256 * 190          # value chain, config 2
    assert lib.call("icrl_stream_len", 256, 1, 19, 1) == 256 * 209          # reward chain
    assert lib.call("icrl_stream_len", 8192, 20, 1, 0) == 8192 * 20         # GetRewards config 3
    assert lib.call("icrl_chain_sync_bytes") >= 64 + 8 * 2 * 512


def test_no_cpu_fallback(lib):
    import icrl_b200.models as M
    from icrl_b200.engine import A2CEngine
    from oracle import synth
    w2i = synth.word_to_idx(64)
    P, V, R = M.PolicyNetwork(w2i), M.ValueNetwork(w2i), M.RewardNetwork(w2i)
    A = M.AdvantageActorCriticNetwork(V, P)
    with pytest.raises(lib.IcrlError):
        A2CEngine(A, R)
    with pytest.raises(lib.IcrlError):
        P(torch.zeros(1, 2, 512), torch.ones(2, 3, dtype=torch.long))
    with pytest.raises(lib.IcrlError):
        R(torch.zeros(2, 512), torch.ones(2, 3, dtype=torch.long))


def test_state_dict_layout_matches_reference_keys():
    """SURVEY 8b: key names / shapes of policyNetwork.pt, valueNetwork.pt, rewardNetwork.pt, a2cNetwork.pt."""
    import icrl_b200.models as M
    from oracle import synth
    w = synth.make_weights(0)
    w2i = synth.word_to_idx()
    P, V, R = M.PolicyNetwork(w2i), M.ValueNetwork(w2i), M.RewardNetwork(w2i)
    for mod, sd in ((P, w["policy"]), (V, w["value"]), (R, w["reward"])):
        own = mod.state_dict()
        assert set(own) == set(sd)
        for k in sd:
            assert tuple(own[k].shape) == tuple(sd[k].shape), k
        mod.load_state_dict(sd)                       # strict
    A = M.AdvantageActorCriticNetwork(V, P)
    assert list(A.state_dict().keys()) == list(synth.a2c_state_dict(w).keys())
    assert sum(p.numel() for p in A.parameters()) == 6533613
    assert V.valrnn.hidden_cell[0].shape == (1, 1, 512) and R.rewrnn.hidden_cell.shape == (1, 1, 512)
    # bidirectional variant: the reference's extra keys exist (models.py:68, 120, 163-164, 215, 251)
    wb = synth.make_weights(0, bidirectional=True)
    Pb, Vb, Rb = M.PolicyNetwork(w2i, bidirectional=True), M.ValueNetwork(w2i, bidirectional=True), M.RewardNetwork(w2i, bidirectional=True)
    for mod, sd in ((Pb, wb["policy"]), (Vb, wb["value"]), (Rb, wb["reward"])):
        assert set(mod.state_dict()) == set(sd)
        mod.load_state_dict(sd)
    assert Vb.valrnn.hidden_cell[0].shape == (2, 1, 512) and Rb.rewrnn.hidden_cell.shape == (2, 1, 512)


def test_plan_rollout_rules():
    from icrl_b200.engine import plan_rollout
    caps = np.full((4, 20), 7, dtype=np.int64)
    caps[:, 0] = 1
    caps[:, 19] = 2
    caps[2, 11] = 2
    assert plan_rollout(caps) == (1, 19)              # trainers.py:436-441
    assert plan_rollout(caps, 6) == (14, 6)           # trainers.py:548-554
    assert plan_rollout(caps, 16) == (4, 16)
    assert plan_rollout(caps, 20)[0] < 1              # skipped by the caller (trainers.py:550)
    with pytest.raises(ValueError):
        plan_rollout(np.ones((2, 5), dtype=np.int64))


def test_checkpoint_helpers_roundtrip(tmp_path):
    """save_a2c_model / load_a2c_models / get_filename keep the reference's plain-state_dict format and naming
    (utilities.py:286-338): a checkpoint written from one set of modules loads into freshly built ones on CPU."""
    import icrl_b200.models as M
    import icrl_b200.trainers as T
    from oracle import synth
    w = synth.make_weights(3)
    w2i = synth.word_to_idx()
    P, V = M.PolicyNetwork(w2i), M.ValueNetwork(w2i)
    P.load_state_dict(w["policy"])
    V.load_state_dict(w["value"])
    A = M.AdvantageActorCriticNetwork(V, P)
    paths = {"policy_network": str(tmp_path / "p.pt"), "value_network": str(tmp_path / "v.pt")}
    torch.save(P.state_dict(), paths["policy_network"])
    torch.save(V.state_dict(), paths["value_network"])
    a2c_path = str(tmp_path / T.get_filename("a2cNetwork.pt", False, True))
    assert a2c_path.endswith("a2cNetwork_curriculum.pt")
    assert T.get_filename("x.pt", True, None) == "x_bidirectional.pt"
    T.save_a2c_model(A, [a2c_path])
    B = T.load_a2c_models(a2c_path, {"word_to_idx": w2i, "embeddings": None}, paths, False)
    for (k, a), (_, b) in zip(A.state_dict().items(), B.state_dict().items()):
        assert torch.equal(a.cpu(), b.cpu()), k
    assert not B.policy_network.training and not B.value_network.training


def test_bench_reference_arm_json_contract():
    """`bench.py --impl reference` (the CPU arm the driver runs beside the GPU arm) prints ONE JSON line with the keys of
    the bench contract; it times oracle/ref_port on the host cores and needs no GPU."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "0",
                          "--cpu-sample", "4", "--batch", "16"], capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "A2C train captions/sec" and d["unit"] == "captions/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["n_gpus"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"] and "model" not in d["config"]
    # the first timed step is the whole global batch (same workload string as the GPU arm), the rest bounded samples
    assert d["config"]["workload"].startswith("configs[3]: full A2C training step") and "global batch 16" in d["config"]["workload"]
    assert d["config"]["steps_timed"] == 2 and "all 16 captions" in d["cpu_baseline"]["sample"]


def test_bench_clock_sampler_window():
    """bench.ClockSampler.stop(t0, t1): samples inside the timed region are used; when the region is shorter than one
    sampling period the warm-up samples (same kernels, same load) are used and the window says so; throttle reasons are
    collected from the rows that are used."""
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    import bench

    class _Proc:
        def terminate(self):
            pass

    def sampler(rows, stamps):
        s = bench.ClockSampler(0)
        s.proc, s.rows, s.stamps = _Proc(), list(rows), list(stamps)
        return s

    idle = ["0", "1200", "1965", "300", "0x0", "Not Active", "Not Active", "Not Active", "Not Active"]
    busy = ["0", "1965", "1965", "900", "0x4", "Not Active", "Not Active", "Not Active", "Active"]
    out = sampler([idle, busy, busy, busy], [10.0, 10.2, 10.4, 10.6]).stop(10.1, 10.5)
    assert out["samples"] == 2 and out["sm_mhz"] == 1965.0 and out["window"] == "timed region"
    assert out["reasons"] == ["sw_power_cap"] and out["sm_max_mhz"] == 1965.0
    out = sampler([busy, busy], [10.0, 10.2]).stop(10.25, 10.30)              # timed region between two samples
    assert out["samples"] == 2 and out["window"].startswith("warm-up")
    assert bench.ClockSampler(0).stop()["reasons"] == ["nvidia-smi unavailable"]


def test_stream_length_and_take_positions_match_the_oracle(lib):
    """icrl_stream_len (host arithmetic of the C ABI) against the oracle's stream builder for random shapes: the value
    chain holds B * sum_s (p0 + s) positions, the reward chain one more column per block, and the take positions are
    the last B positions of every block (models.py:168-169, 254-255: one RNN call per column, state carried)."""
    from hypothesis import given, settings, strategies as st
    from oracle import single_pass

    @settings(max_examples=40, deadline=None)
    @given(B=st.integers(1, 9), p0=st.integers(1, 6), S=st.integers(1, 7), extra=st.integers(0, 1))
    def check(B, p0, S, extra):
        tokens = np.arange(B * (p0 + S + 1), dtype=np.int64).reshape(B, p0 + S + 1)
        stream, take = single_pass.stream_tokens(tokens, p0, S, extra)
        assert int(lib.call("icrl_stream_len", B, p0, S, extra)) == len(stream) == B * sum(p0 + s + extra for s in range(S))
        off = 0
        for s in range(S):
            off += (p0 + s + extra) * B
            assert list(take[s]) == list(range(off - B, off))
            # block s is the column-major prefix of length p0 + s + extra
            blk = stream[off - (p0 + s + extra) * B: off].reshape(p0 + s + extra, B)
            assert np.array_equal(blk, tokens[:, :p0 + s + extra].T)

    check()


def test_stream_positions_of_a_token_closed_form():
    """The gate-table scatter (scatter_add_stream_kernel, policy.cu) sums, for every (column, row) of the token matrix, the
    stream positions B * (s (p0 + extra) + s (s - 1) / 2 + col) + b of the blocks s >= max(0, col - p0 - extra + 1) and
    reduces once into the row of the token at the first of them.  Checked against the oracle's stream builder: those
    positions are exactly the positions that consumed that token, every position is covered once."""
    from hypothesis import given, settings, strategies as st
    from oracle import single_pass

    @settings(max_examples=60, deadline=None)
    @given(B=st.integers(1, 9), p0=st.integers(1, 6), S=st.integers(1, 8), extra=st.integers(0, 1))
    def check(B, p0, S, extra):
        n_col = p0 + S - 1 + extra
        tokens = np.arange(B * (n_col + 1), dtype=np.int64).reshape(B, n_col + 1)       # every (row, column) its own token
        stream, _ = single_pass.stream_tokens(tokens, p0, S, extra)
        seen = np.zeros(len(stream), dtype=np.int64)
        for col in range(n_col):
            for b in range(B):
                s0 = max(0, col - p0 - extra + 1)
                pos = [B * (s * (p0 + extra) + s * (s - 1) // 2 + col) + b for s in range(s0, S)]
                assert pos and all(0 <= q < len(stream) for q in pos)
                assert all(stream[q] == tokens[b, col] for q in pos)
                assert sorted(np.nonzero(stream == tokens[b, col])[0].tolist()) == pos
                seen[pos] += 1
        assert (seen == 1).all()

    check()
