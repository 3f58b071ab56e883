"""The value chain's parameter gradients from the gate-gradient pairs that the tcgen05 chain backward writes (fp16 hi/lo'
planes, one power-of-two scale per launch, columns in the chain backward's store order) instead of fp32 dgates."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import synth
from tests.helpers import make_nets, named_grads

H, G = 512, 2048


def stored_col(n):
    """Column of natural gate column n = a * 512 + u in the pair planes (icrl_gate_pair_col, common.cuh)."""
    a, u = n // H, n % H
    return 128 * (u >> 5) + 16 * ((u >> 2) & 7) + 4 * a + (u & 3)


def make_pairs(dg, rows):
    """[T][2048] fp32 -> ([2][rows][2048] fp16 planes in stored column order, inverse scale, decoded fp32 values) with the
    chain backward's scale: max |dg| * s in [8, 16)."""
    T = dg.shape[0]
    ex = int(np.frexp(float(dg.abs().max()))[1])
    s = 2.0 ** (4 - ex)
    v = dg * s
    hi = v.half()
    lo = ((v - hi.float()) * 2048.0).half()
    perm = torch.tensor([stored_col(n) for n in range(G)], device=dg.device)
    assert torch.equal(perm.sort().values, torch.arange(G, device=dg.device))
    planes = torch.zeros((2, rows, G), dtype=torch.float16, device=dg.device)
    planes[0, :T, perm] = hi
    planes[1, :T, perm] = lo
    planes[:, T:] = float("nan")            # rows past T must not be read
    decoded = (hi.double() + lo.double() / 2048.0) / s
    return planes, torch.tensor([1.0 / s], device=dg.device), decoded


@pytest.mark.gpu
@pytest.mark.parametrize("B,p0,S", [(96, 1, 7), (130, 1, 19)])
def test_value_param_grads_from_pairs_vs_float64(B, p0, S):
    """icrl_value_chain_param_grads_pairs against float64: the gate-table gradient (and through it dW_ih, db) and dW_hh,
    with the stored column order undone.  Rows whose gradients keep all 22 bits of the pair (at or above 2^-17 of the
    largest) are checked against their own scale, everything against its tensor's maximum."""
    from icrl_b200 import _lib
    V, D = 211, 512
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
    stash_h = torch.from_numpy(np.tanh(rs.standard_normal((T + 1, H))).astype(np.float32)).cuda()
    E = torch.from_numpy(rs.standard_normal((V, D)).astype(np.float32)).cuda()
    W_ih = torch.from_numpy((rs.standard_normal((G, D)) * 0.05).astype(np.float32)).cuda()
    planes, inv_scale, dec = make_pairs(dgates, T + 37)
    cs = int(_lib.call("icrl_colsum_ws_floats", max(T, V), G))
    wsb = int(_lib.call("icrl_wgrad_tc_ws_bytes", G, H, T, 2))
    dtable = torch.full((V, G), float("nan"), device="cuda")
    csws = torch.zeros(cs, device="cuda")
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    dE, dWih = torch.empty((V, D), device="cuda"), torch.empty((G, D), device="cuda")
    dWhh, dbi, dbh = torch.empty((G, H), device="cuda"), torch.empty(G, device="cuda"), torch.empty(G, device="cuda")
    _lib.call("icrl_value_chain_param_grads_pairs", st, T, V, D, p(stream), p(planes), T + 37, p(inv_scale), p(stash_h), p(E),
              p(W_ih), p(dtable), p(csws), p(ws), wsb, p(dE), p(dWih), p(dWhh), p(dbi), p(dbh), B, p0, S, 0, None)
    torch.cuda.synchronize()

    exact = dgates.double()
    full_bits = exact.abs().max(dim=0).values >= exact.abs().max() * 2.0 ** -17       # per gate column
    assert full_bits.any() and not full_bits.all()
    ref_table = torch.zeros((V, G), dtype=torch.float64, device="cuda").index_add_(0, stream[:T].long(), exact)
    ref_table_dec = torch.zeros((V, G), dtype=torch.float64, device="cuda").index_add_(0, stream[:T].long(), dec)
    ref_whh = exact.t() @ stash_h[:T].double()
    ref_whh_dec = dec.t() @ stash_h[:T].double()
    refs = {"dtable": ref_table, "dWhh": ref_whh, "dWih": ref_table.t() @ E.double(), "dE": ref_table @ W_ih.double(),
            "dbi": ref_table.sum(0), "dbh": ref_table.sum(0)}
    got = {"dtable": dtable, "dWhh": dWhh, "dWih": dWih, "dE": dE, "dbi": dbi, "dbh": dbh}
    for k, ref in refs.items():
        assert torch.isfinite(got[k]).all(), k
        err = ((got[k].double() - ref).abs().max() / ref.abs().max()).item()
        assert err < 2e-6, (k, err)
    # against the decoded pairs, per gate column (dtable) / row (dW_hh) of full precision
    col = ((dtable.double() - ref_table_dec).abs().max(dim=0).values / ref_table_dec.abs().max(dim=0).values.clamp_min(1e-300))
    assert col[full_bits].max().item() < 2e-6, col[full_bits].max().item()
    row = ((dWhh.double() - ref_whh_dec).abs().max(dim=1).values / ref_whh_dec.abs().max(dim=1).values.clamp_min(1e-300))
    assert row[full_bits].max().item() < 2e-6, row[full_bits].max().item()


@pytest.mark.gpu
def test_engine_pairs_match_serial_chain_gradients():
    """The default engine (chain pieces on tcgen05, parameter gradients from the gate-gradient pairs) against the serial
    kernels' fp32 gate gradients (chain_segments = 1) on the same weights and batch: every value-network gradient within
    2e-6 of its tensor's maximum."""
    from icrl_b200.engine import A2CEngine
    seed, B, L = 11, 1024, 20
    A, R, _ = make_nets(seed, "cuda:0")
    f, c = synth.make_inputs(seed, B, L)
    u = synth.make_uniforms(seed, L - 1, B)
    e_serial = A2CEngine(A, R, chain_segments=1)
    r0 = e_serial.step(f, c, uniforms=u)
    torch.cuda.synchronize()
    g0 = named_grads(A)
    e_tc = A2CEngine(A, R)
    r1 = e_tc.step(f, c, uniforms=u)
    torch.cuda.synchronize()
    g1 = named_grads(A)
    assert e_tc.piece_layout is not None and e_tc.segment_stats["fallbacks"] == 0, "the tcgen05 chain pieces did not run"
    assert torch.equal(r0["tokens"], r1["tokens"])
    worst = {}
    for k in g0:
        if not k.startswith("value"):
            continue
        scale = float(np.abs(g0[k]).max())
        worst[k] = float(np.abs(g1[k] - g0[k]).max()) / scale
        assert worst[k] <= 2e-6, (k, worst[k])
    k_hh = [k for k in g0 if k.startswith("value") and k.endswith("weight_hh_l0")]
    assert len(k_hh) == 1
    a, b = g1[k_hh[0]].astype(np.float64), g0[k_hh[0]].astype(np.float64)
    per_row = np.abs(a - b).max(axis=1) / np.maximum(np.abs(b).max(axis=1), 1e-300)
    print("value gradients vs serial (max error / tensor max): %s; dW_hh worst per-row error %.3g"
          % (", ".join("%s %.2g" % kv for kv in sorted(worst.items())), float(per_row.max())))
