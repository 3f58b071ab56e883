"""Fused A2C minibatch on the GPU: one call replaces the body of the reference's training loop
(``trainers.py:432-480`` / ``:544-594``): rollout -> rewards -> values -> loss -> backward.

Host code is PyTorch plumbing only (device memory, streams); all arithmetic runs in the CUDA
kernels behind ``include/icrl_b200.h``.  There is no CPU fallback.

Single-pass formulation (verified against the unmodified reference, SURVEY.md section 8c):
  policy   one incremental LSTM pass with sampling (instead of re-running the prefix every step)
  value    ONE serial LSTM chain over the column-major token stream, h taken at the last B
           positions of each step block; head evaluated in collapsed form.  By default the chain
           is advanced as hundreds of consecutive pieces in lockstep on the tensor cores, each with
           a discarded warm-up that is verified against the previous piece on every step (chain
           pieces, DESIGN 4.1)
  reward   ONE serial GRU chain, semantic/visual embeds batched over all steps, fused cosine
  loss     advantage = values - rewards, gradient seeds for both networks
  backward policy BPTT (batched GEMMs + S serial cell steps), value-chain BPTT kernel, weight
           gradients as contractions over all steps; gradients land in one flat bucket that the
           parameters' ``.grad`` tensors alias (ready for a single all-reduce).
"""
import ctypes

import numpy as np
import torch

from . import _lib

H = 512
END_TOKEN = 2       # trainers.py:436


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


class StepResult(dict):
    """Device tensors of one minibatch; ``loss`` / ``mean_reward`` / ``mean_adv`` (and ``mean_entropy`` when the engine
    has an entropy bonus) sync lazily."""

    host_stats = None       # (loss, mean reward, mean advantage[, mean entropy]) when the step's check brought them over

    def _stat(self, i):
        if self.host_stats is not None:
            return float(self.host_stats[i])
        return float(self["stats"][i].item())

    @property
    def loss(self):
        return self._stat(0)

    @property
    def mean_reward(self):
        return self._stat(1)

    @property
    def mean_adv(self):
        return self._stat(2)

    @property
    def mean_entropy(self):
        """Mean policy entropy of the sampled steps; only steps of an engine with entropy_coef != 0 track it."""
        if len(self["stats"]) < 4:
            raise AttributeError("the step ran without an entropy bonus (entropy_coef = 0): no entropy was computed")
        return self._stat(3)


class Prepared:
    """A minibatch already resident in HBM (A2CEngine.prepare): features (B,512) f32, the prefix
    columns int32 [p0][B], uniforms (S,B) f64 or None, and the rollout plan."""

    def __init__(self, f, prefix_cm, u, B, p0, S):
        self.f, self.prefix_cm, self.u, self.B, self.p0, self.S = f, prefix_cm, u, B, p0, S


def plan_rollout(captions, level=None):
    """(p0, S) as the reference derives them: caplen = max <END> column + 1 (trainers.py:436);
    non-curriculum p0 = 1, S = caplen - 1 (:438-441); curriculum p0 = caplen - level, S = level
    (:548-554).  Raises like the reference when no row holds <END>."""
    caps = np.asarray(captions)
    cols = np.nonzero(caps == END_TOKEN)[1]
    if cols.size == 0:
        raise ValueError("no <END> (=2) token in the caption batch (trainers.py:436 would fail on max())")
    caplen = int(cols.max()) + 1
    if level is None:
        return 1, caplen - 1
    return caplen - int(level), int(level)


def plan_xent(captions):
    """Row plan of the policy's cross-entropy pretraining (trainers.py:202-257), as the reference derives it: caplen_b =
    column of the FIRST <END> of row b + 1; the row counts its first n_b = min(caplen_b, L-1) teacher-forced positions
    (the last counted one predicts the token after <END>) with weight w_b = caplen_b / (B * n_b) -- the reference's
    (caplen/B) * mean, with the unclamped caplen.  Returns (n [B] int, w [B] float64, S = max n_b): positions at or past
    every row's n_b add nothing, so the decode runs S steps only.  Raises ValueError for a row without <END> (the
    reference fails there with an IndexError)."""
    caps = np.asarray(captions)
    if caps.ndim != 2 or caps.shape[0] < 1 or caps.shape[1] < 2:
        raise ValueError("captions must be (B, L) with B >= 1 and L >= 2, got %s" % (caps.shape,))
    B, L = caps.shape
    end = caps == END_TOKEN
    missing = np.nonzero(~end.any(axis=1))[0]
    if missing.size:
        raise ValueError("caption row %d has no <END> (=2) token (the reference's loop raises IndexError there)" % missing[0])
    caplen = end.argmax(axis=1) + 1
    n = np.minimum(caplen, L - 1)
    return n, caplen / (float(B) * n), int(n.max())


class A2CEngine:
    DECODE_MODES = ("fused", "tc", "simt")
    entropy_coef = 0.0            # engines that skip __init__ (look-ahead, greedy decode) have no entropy bonus

    def __init__(self, a2c_network, reward_network, use_tc=None, decode="fused", chain_shards=1, wgrad="tc",
                 chain_segments=32, chain_warmup=256, chain_tol=1e-5, chain_engine="tc",
                 chain_pieces=None, chain_adapt=True, chain_warmup_min=32, policy_bptt="tc", chain_fuse_fwd=True, overlap_backward=True,
                 entropy_coef=0.0):
        # entropy_coef: weight of the entropy bonus, loss = reference loss - entropy_coef * mean policy entropy over the
        # sampled steps (the A3C regulariser; positive values favour exploration).  0 is the reference's loss, computed
        # by exactly the kernels it always was.
        self.entropy_coef = float(entropy_coef)
        self.policy = a2c_network.policy_network
        self.value = a2c_network.value_network
        self.reward = reward_network
        self.a2c = a2c_network
        if any(getattr(m, "bidirectional", False) for m in (self.policy, self.value, self.reward)):
            raise NotImplementedError("the fused engine is built for the unidirectional networks; bidirectional=True runs "
                                      "on the module (autograd) route -- icrl_b200.trainers switches to it by itself")
        dev = self.policy.linear2vocab.weight.device
        if dev.type != "cuda":
            raise _lib.IcrlError("A2CEngine needs the networks on a CUDA device (no CPU fallback)")
        _lib.load()
        self.device = dev
        self.V = self.policy.linear2vocab.weight.shape[0]
        self._bufs = {}
        self.launches = _lib.Launches()
        self.phase_events = None          # set to [] to record (name, start, end) CUDA events per phase
        # policy decode path: "fused" = the persistent cluster kernel (decode.cu: tcgen05 GEMMs with the cell
        # update / softmax / sampling in their epilogues, one launch per rollout); "tc" = per-step kernels with
        # the two GEMMs on tcgen05 (gemm_tc.cu); "simt" = per-step kernels, fp32 CUDA-core GEMMs.
        if use_tc is not None:
            decode = "tc" if use_tc else "simt"
        if decode not in self.DECODE_MODES:
            raise ValueError("decode must be one of %s" % (self.DECODE_MODES,))
        if decode == "fused" and (self.V > 1024 or self.V % 4):
            # the persistent kernel keeps one row of logits inside a cluster (8 x 128 columns, float4 stash)
            import warnings
            warnings.warn("vocabulary of %d words does not fit the fused decode kernel (V <= 1024, V %% 4 == 0): "
                          "using the per-step kernels" % self.V)
            decode = "simt"
        self.decode = decode
        self.use_tc = decode == "tc"
        # chain_shards = K > 1 cuts the (local) batch into K contiguous row shards whose value / reward recurrences
        # each start from zero state -- the reference run on K minibatches of B/K rows with averaged gradients,
        # i.e. exactly what K data-parallel ranks compute (SURVEY.md 8e/H6).  K = 1 is the reference's single
        # carried-state chain over the whole batch.  The K chains advance in lockstep on the same CTAs.
        # wgrad: "tc" = the K = T weight-gradient contraction of the value chain on tcgen05 (wgrad_tc.cu; needs a
        # workspace of ~10 KB per serial step), "simt" = fp32 CUDA-core GEMM with split-K.  Steps whose value chain ran
        # as tcgen05 pieces contract on tcgen05 either way: their gate gradients exist only as its fp16 pairs.
        if wgrad not in ("tc", "simt"):
            raise ValueError("wgrad must be 'tc' or 'simt'")
        self.wgrad = wgrad
        if chain_shards not in (1, 2, 4, 8):
            raise ValueError("chain_shards must be 1, 2, 4 or 8")
        self.chain_shards = int(chain_shards)
        # chain_segments = 1 runs the reference's ONE carried-state chain on the serial kernels; any other value cuts it
        # into tcgen05 pieces (chain_engine below).
        if chain_segments not in (1, 2, 4, 8, 16, 32):
            raise ValueError("chain_segments must be 1, 2, 4, 8, 16 or 32")
        self.chain_segments = 1 if self.chain_shards > 1 else int(chain_segments)
        self.chain_warmup = int(chain_warmup)
        self.chain_tol = float(chain_tol)
        if self.chain_warmup < 1:
            raise ValueError("chain_warmup must be positive")
        # chain_engine "tc" = chain pieces on tcgen05 (chain_tc.cu): hundreds of lockstep pieces, 128 per cluster of 8 CTAs,
        # one kernel step = H_prev [pieces x 512] . W_hh^T on the tensor cores.  Piece k >= 1 starts from zero state a
        # warm-up early and throws those steps away: a gated recurrence forgets its initial state, so the piece then
        # carries the single chain's state up to float rounding, which the joint check verifies on every step.  The
        # warm-up is sized PER CHAIN (value LSTM forward + backward, reward GRU) from the contraction rate measured on
        # every step (errors half-way through and at the end of the warm-up): it grows before the check can fail and
        # shrinks again after `_SHRINK_AFTER` clean steps; a failed check re-runs the chains with a longer warm-up, and
        # after _TC_ATTEMPTS failures, or for a chain too short to cut, the step runs on the serial kernels.
        if chain_engine != "tc":
            raise ValueError("chain_engine must be 'tc': the CUDA-core chain-segment engine ('simt') was removed; "
                             "chain_segments=1 runs the serial kernels")
        self.chain_pieces = None if chain_pieces is None else int(chain_pieces)
        if self.chain_pieces is not None and self.chain_pieces < 2:
            raise ValueError("chain_pieces must be at least 2")
        # policy_bptt: "tc" = the policy's serial cell-backward steps on the tcgen05 chain-backward kernel (one launch),
        # "simt" = one pointwise kernel + one fp32 CUDA-core GEMM per cell step
        if policy_bptt not in ("tc", "simt"):
            raise ValueError("policy_bptt must be 'tc' or 'simt'")
        self.policy_bptt = policy_bptt
        # overlap_backward: the policy's backward on a second stream beside the value-chain backward (separate workspaces)
        self.overlap_backward = bool(overlap_backward)
        self._side_stream = None
        self._n_cell_max = 1
        self.chain_fuse_fwd = bool(chain_fuse_fwd)     # value + reward forward chains in one launch when that is faster
        self.chain_adapt = bool(chain_adapt)
        self.chain_warmup_min = int(chain_warmup_min)
        # current warm-up per recurrence (tc engine): value forward, reward forward, value backward -- each follows its own
        # measured contraction (the forward cell state is the slowest to converge; the backward need not pay for it)
        self.warm = {"v": self.chain_warmup, "r": self.chain_warmup, "b": self.chain_warmup}
        self._clean = {"v": 0, "r": 0, "b": 0}
        self._hold = {"v": 0, "r": 0, "b": 0}
        self._tc = None                   # {"v": (P, seg, warm) | None, "r": (P, seg, warm)} of the current step
        self.segment_stats = {"steps": 0, "segmented_steps": 0, "fallbacks": 0, "reruns": 0, "tc_max_err": [0.0] * 16,
                              "warm_history": []}
        self._seg_unverified = False
        with torch.cuda.device(dev):
            self.sync_state = torch.zeros(int(_lib.call("icrl_chain_sync_bytes")), dtype=torch.uint8, device=dev)
            # [0:3] loss, mean reward, mean advantage; [3] mean entropy (entropy bonus only); [4:20] joint-check words of
            # the tc chain launches (value forward 4..7, reward forward 8..11, value backward 12..17): read together in ONE
            # device-to-host copy per step
            # [20:28] words of the policy's tcgen05 BPTT ([24] max |dL/dh|, [25] fp16-exchange overflow flag)
            self._stat_err = torch.zeros(28, dtype=torch.float32, device=dev)
        self._tc_err = self._stat_err[4:20]
        self._reward_versions = None
        self._dz_ld = None
        self._check_params()
        self._bind_flat_grads()

    # ------------------------------------------------------------------ parameters / gradients
    def _params(self):
        return list(self.a2c.parameters())

    def _check_params(self):
        for p in list(self.a2c.parameters()) + (list(self.reward.parameters()) if self.reward is not None else []):
            if p.dtype != torch.float32 or not p.is_contiguous() or p.device != self.device:
                raise _lib.IcrlError("parameters must be contiguous float32 on %s" % self.device)

    def _bind_flat_grads(self):
        """One flat fp32 bucket in a2c.parameters() order; every .grad is a view into it."""
        ps = [p for p in self._params() if p.requires_grad]
        # every tensor starts on a 256-byte boundary of the bucket (the kernels read parameters and write gradients with
        # 16-byte accesses; optim.FlatAdam lays the parameters out the same way): the padding floats stay zero
        self._flat_offsets, off = [], 0
        for p in ps:
            self._flat_offsets.append(off)
            off += -(-p.numel() // 64) * 64
        self.flat_grad = torch.zeros(off, dtype=torch.float32, device=self.device)
        self._grad_views = []
        for p, o in zip(ps, self._flat_offsets):
            self._grad_views.append((p, self.flat_grad[o:o + p.numel()].view_as(p)))
        self._attach_grads()

    def _attach_grads(self):
        for p, v in self._grad_views:
            if p.grad is None or p.grad.data_ptr() != v.data_ptr():
                p.grad = v

    def _g(self, p, optional=False):
        """Gradient destination for parameter p (frozen: a scratch buffer, or None where the ABI lets a gradient
        be skipped -- the frozen pretrained embeddings, models.py:61-63)."""
        for q, v in self._grad_views:
            if q is p:
                return v
        if optional:
            return None
        return self._buf("frozen_grad_%d" % id(p), p.numel())

    def _buf(self, name, numel, dtype=torch.float32):
        numel = int(max(numel, 1))
        t = self._bufs.get(name)
        if t is None or t.numel() < numel or t.dtype != dtype:
            t = torch.empty(numel, dtype=dtype, device=self.device)
            self._bufs[name] = t
        return t

    class _Phase:
        def __init__(self, eng, name):
            self.eng, self.name = eng, name

        def __enter__(self):
            if self.eng.phase_events is not None:
                self.t0 = torch.cuda.Event(enable_timing=True)
                self.t0.record(torch.cuda.current_stream(self.eng.device))

        def __exit__(self, *a):
            if self.eng.phase_events is not None:
                t1 = torch.cuda.Event(enable_timing=True)
                t1.record(torch.cuda.current_stream(self.eng.device))
                self.eng.phase_events.append((self.name, self.t0, t1))

    def _phase(self, name):
        return A2CEngine._Phase(self, name)

    def phase_times_ms(self):
        """Sum of CUDA-event durations per phase since phase_events was last reset (syncs)."""
        torch.cuda.synchronize(self.device)
        out = {}
        for name, a, b in self.phase_events or []:
            out.setdefault(name, []).append(a.elapsed_time(b))
        return out

    @property
    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ------------------------------------------------------------------ packing
    def pack_weights(self, reward=True):
        """Rebuild the derived operands from the current parameters (after every optimizer step):
        the three gate tables W_ih E + b and the collapsed value head."""
        st, L, V = self._stream, self.launches.ref, self.V
        P, Vn, R = self.policy, self.value, self.reward
        c = _lib.call
        c("icrl_pack_gate_table", st, V, 4 * H, 4 * H, P.caption_embedding.weight.shape[1], _p(P.caption_embedding.weight), _p(P.lstm.weight_ih_l0),
          _p(P.lstm.bias_ih_l0), _p(P.lstm.bias_hh_l0), _p(self._buf("p_table", V * 4 * H)), L)
        c("icrl_pack_gate_table", st, V, 4 * H, 4 * H, Vn.valrnn.caption_embedding.weight.shape[1], _p(Vn.valrnn.caption_embedding.weight),
          _p(Vn.valrnn.lstm.weight_ih_l0), _p(Vn.valrnn.lstm.bias_ih_l0), _p(Vn.valrnn.lstm.bias_hh_l0),
          _p(self._buf("v_table", V * 4 * H)), L)
        c("icrl_pack_value_head", st, _p(Vn.linear1.weight), _p(Vn.linear1.bias), _p(Vn.linear2.weight),
          _p(Vn.linear2.bias), _p(self._buf("v_weff", 2 * H)), _p(self._buf("v_beff", 1)), L)
        if self.use_tc:
            self._pack_policy_tc()
        if self.decode == "fused":
            n = int(_lib.call("icrl_decode_weight_halves"))
            _lib.call("icrl_pack_decode_weights", st, V, _p(P.lstm.weight_hh_l0), _p(P.linear2vocab.weight),
                      _p(self._buf("p_decode_pk", n, torch.float16)), L)
        if self._use_tc_chains():
            n = int(_lib.call("icrl_chain_tc_weight_halves", 0))
            _lib.call("icrl_pack_chain_tc_weights", st, 0, _p(Vn.valrnn.lstm.weight_hh_l0),
                      _p(self._buf("v_chain_pk", n, torch.float16)), L)
        if self.policy_bptt == "tc":
            n = int(_lib.call("icrl_chain_tc_weight_halves", 0))
            _lib.call("icrl_pack_chain_tc_weights", st, 0, _p(P.lstm.weight_hh_l0),
                      _p(self._buf("p_chain_pk", n, torch.float16)), L)
        if reward or self._reward_changed():
            self.pack_reward()

    def _use_tc_chains(self):
        return self.chain_segments > 1 and self.chain_shards == 1

    def _reward_changed(self):
        """The reward network is frozen during A2C training (trainers.py:372-373) and its derived operands are packed once;
        an in-place change of its parameters (load_state_dict, more reward pretraining on the same object) is noticed
        through the tensors' version counters."""
        v = tuple(p._version for p in self.reward.parameters()) + tuple(p.data_ptr() for p in self.reward.parameters())
        return v != self._reward_versions

    def _pack_policy_tc(self):
        """3-part bf16 splits of the two decode-step weight matrices (tensor-core operands)."""
        P = self.policy
        for name, w in (("whh", P.lstm.weight_hh_l0), ("wv", P.linear2vocab.weight)):
            n = w.numel()
            _lib.call("icrl_split_bf16x3", self._stream, n, _p(w), _p(self._buf("p_%s_parts" % name, 3 * n, torch.bfloat16)),
                      self.launches.ref)

    def pack_reward(self):
        R, V = self.reward, self.V
        _lib.call("icrl_pack_gate_table", self._stream, V, 3 * H, 2 * H, R.rewrnn.caption_embedding.weight.shape[1], _p(R.rewrnn.caption_embedding.weight),
                  _p(R.rewrnn.gru.weight_ih_l0), _p(R.rewrnn.gru.bias_ih_l0), _p(R.rewrnn.gru.bias_hh_l0),
                  _p(self._buf("r_table", V * 3 * H)), self.launches.ref)
        if self._use_tc_chains():
            n = int(_lib.call("icrl_chain_tc_weight_halves", 1))
            _lib.call("icrl_pack_chain_tc_weights", self._stream, 1, _p(R.rewrnn.gru.weight_hh_l0),
                      _p(self._buf("r_chain_pk", n, torch.float16)), self.launches.ref)
        # 3-part bf16 split of the sentence-embedding weight: the [S*B x 512] x [512 x 512] projection of the reward head
        # runs on the tensor-core GEMM of the decode step (gemm_tc.cu, fp32-grade) once it is large enough to fill tiles
        n = R.semantic_embed.weight.numel()
        _lib.call("icrl_split_bf16x3", self._stream, n, _p(R.semantic_embed.weight),
                  _p(self._buf("r_se_parts", 3 * n, torch.bfloat16)), self.launches.ref)
        self._reward_versions = tuple(p._version for p in R.parameters()) + tuple(p.data_ptr() for p in R.parameters())

    _TC_LINEAR_MIN_ROWS = 4096

    def _gemm(self, ta, tb, M, N, K, A, lda, B, ldb, C, ldc, bias=None, beta=0.0):
        _lib.call("icrl_gemm_f32", self._stream, ta, tb, M, N, K, _p(A), lda, _p(B), ldb, _p(C), ldc, _p(bias),
                  beta, None, 0, self.launches.ref)

    # ------------------------------------------------------------------ inputs
    def prepare(self, features, captions, uniforms=None, level=None, plan=None):
        """Host -> HBM staging of one minibatch (the copies the end-to-end timing includes)."""
        p0, S = plan if plan is not None else plan_rollout(captions, level)
        if p0 < 1:
            return None
        dev = self.device
        caps = captions.cpu().numpy() if isinstance(captions, torch.Tensor) else np.asarray(captions)
        B = caps.shape[0]
        f = torch.as_tensor(features)
        if f.dtype != torch.float32:
            f = f.float()
        f = f.to(dev, non_blocking=True).contiguous()
        pre = torch.from_numpy(np.ascontiguousarray(caps[:, :p0].T).astype(np.int32))
        prefix_cm = pre.to(dev, non_blocking=True)
        u = None
        if uniforms is not None:
            u = torch.as_tensor(uniforms, dtype=torch.float64).to(dev, non_blocking=True).contiguous()
            assert tuple(u.shape) == (S, B), "uniforms must be (S,B) float64"
        return Prepared(f, prefix_cm, u, B, p0, S)

    def gather_rows(self, matrix, rows):
        """matrix[rows] on the device: `matrix` (M,512) f32 resident in HBM, `rows` host integers (only they cross the
        bus).  The device-side half of the reference's minibatch generator (utilities.py:172-176)."""
        idx = torch.as_tensor(np.asarray(rows), dtype=torch.int32).to(self.device, non_blocking=True)
        out = torch.empty((idx.numel(), H), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.call("icrl_gather_rows", self._stream, idx.numel(), _p(matrix), _p(idx), 0, _p(out), self.launches.ref)
        return out

    def _stage_inputs(self, prep, forced):
        B, p0, S = prep.B, prep.p0, prep.S
        tokcm = self._buf("tokcm", (p0 + S) * B, torch.int32)
        tokcm[:p0 * B].copy_(prep.prefix_cm.reshape(-1), non_blocking=True)
        fo = None
        if forced is not None:
            fo = torch.as_tensor(np.asarray(forced), dtype=torch.int64).to(self.device).contiguous()
            assert tuple(fo.shape) == (B, S)
        return prep.f, tokcm, prep.u, fo, B

    # ------------------------------------------------------------------ phases
    def _policy_forward(self, f, tokcm, u, fo, B, p0, S, greedy):
        V, P = self.V, self.policy
        n_cell = p0 - 1 + S
        tokens = torch.empty((B, S), dtype=torch.int64, device=self.device)
        logp = torch.empty((B, S), dtype=torch.float32, device=self.device)
        Hs = self._buf("p_Hs", (n_cell + 1) * B * H)
        Cs = self._buf("p_Cs", (n_cell + 1) * B * H)
        Gs = self._buf("p_Gs", n_cell * B * 4 * H)
        logits = self._buf("p_logits", S * B * V)
        gpre = self._buf("p_gpre", B * 4 * H)
        b = self._bufs
        with self._phase("policy_fwd"):
          if self.decode == "fused":
            _lib.call("icrl_policy_rollout_fwd_fused", self._stream, B, V, p0, S, int(bool(greedy)), _p(f),
                  _p(P.cnn2linear.weight), _p(P.cnn2linear.bias), _p(b["p_table"]), _p(b["p_decode_pk"]),
                  _p(P.linear2vocab.bias), _p(u), _p(fo), _p(tokcm), _p(tokens), _p(logp), _p(Hs), _p(Cs), _p(Gs),
                  _p(logits), None, _p(self._buf("p_hparts", 4 * B * H, torch.float16)), self.launches.ref)
          elif self.use_tc:
            _lib.call("icrl_policy_rollout_fwd_tc", self._stream, B, V, p0, S, int(bool(greedy)), _p(f),
                  _p(P.cnn2linear.weight), _p(P.cnn2linear.bias), _p(b["p_table"]), _p(b["p_whh_parts"]),
                  _p(b["p_wv_parts"]), _p(P.linear2vocab.bias), _p(u), _p(fo), _p(tokcm), _p(tokens),
                  _p(logp), _p(Hs), _p(Cs), _p(Gs), _p(logits), _p(gpre),
                  _p(self._buf("p_h_parts", 3 * B * H, torch.bfloat16)), self.launches.ref)
          else:
            _lib.call("icrl_policy_rollout_fwd", self._stream, B, V, p0, S, int(bool(greedy)), _p(f),
                  _p(P.cnn2linear.weight), _p(P.cnn2linear.bias), _p(b["p_table"]),
                  _p(P.lstm.weight_hh_l0), _p(P.linear2vocab.weight), _p(P.linear2vocab.bias), _p(u), _p(fo),
                  _p(tokcm), _p(tokens), _p(logp), _p(Hs), _p(Cs), _p(Gs), _p(logits), _p(gpre), self.launches.ref)
        return tokens, logp

    def _streams(self, tokcm, B, p0, S, serial=False):
        st, L = self._stream, self.launches.ref
        K = self.chain_shards
        i32 = torch.int32
        if K > 1:
            if B % K:
                raise ValueError("batch of %d rows does not split into %d chain shards" % (B, K))
            Tv = int(_lib.call("icrl_stream_len", B // K, p0, S, 0))
            Tr = int(_lib.call("icrl_stream_len", B // K, p0, S, 1))
            v_stream, v_take = self._buf("v_stream", K * (Tv + 1), i32), self._buf("v_take", K * (Tv + 1), i32)
            r_stream = self._buf("r_stream", K * (Tr + 1), i32)
            v_pos, r_pos = self._buf("v_pos", S * B, i32), self._buf("r_pos", S * B, i32)
            _lib.call("icrl_build_stream_sharded", st, B, p0, S, 0, K, _p(tokcm), _p(v_stream), _p(v_take), _p(v_pos), L)
            _lib.call("icrl_build_stream_sharded", st, B, p0, S, 1, K, _p(tokcm), _p(r_stream), None, _p(r_pos), L)
            return Tv, Tr
        Tv = int(_lib.call("icrl_stream_len", B, p0, S, 0))
        Tr = int(_lib.call("icrl_stream_len", B, p0, S, 1))
        self._tc = self._pick_pieces(Tv, Tr) if not serial and self._use_tc_chains() else None
        nv, nr = self._padded(Tv, 0), self._padded(Tr, 1)
        v_stream, v_take, v_pos = self._buf("v_stream", nv, i32), self._buf("v_take", nv, i32), self._buf("v_pos", S * B, i32)
        r_stream, r_pos = self._buf("r_stream", nr, i32), self._buf("r_pos", S * B, i32)
        _lib.call("icrl_build_stream", st, B, p0, S, 0, _p(tokcm), _p(v_stream), _p(v_take), _p(v_pos), L)
        _lib.call("icrl_build_stream", st, B, p0, S, 1, _p(tokcm), _p(r_stream), None, _p(r_pos), L)
        if self._tc is not None:          # the last piece runs past the end of the chain: pad with token 0 / "no output"
            v_stream[Tv:nv].zero_()
            v_take[Tv:nv].fill_(-1)
            r_stream[Tr:nr].zero_()
        return Tv, Tr

    def _pieces_for(self, T, warm, pmax=None):
        """(P, seg) for a chain of T positions cut into tcgen05 pieces with a `warm`-position warm-up, or None when it is
        too short.  As many pieces as are co-resident (whole clusters of 128 once there is more than one), each at least
        max(warm / 4, 8) live positions long: the wall time of a launch is seg + warm kernel steps."""
        pmax = self.chain_pieces or pmax or int(_lib.call("icrl_chain_tc_max_pieces"))
        min_seg = max(warm // 4, 8)
        if T <= warm + 2 * min_seg:
            return None
        P = min(pmax, (T - warm) // min_seg)
        if P > 128 and self.chain_pieces is None:
            P -= P % 128
        if P < 2:
            return None
        return P, -(-(T - warm) // P)

    # relative cost of one kernel step of the value LSTM / reward GRU forward kernels (measured: 31.1 K / 22.2 K cycles at 128
    # pieces per cluster); only their ratio matters for splitting the clusters of the fused forward launch
    _STEP_COST = {"v": 1.4, "r": 1.0}

    def _pick_pieces(self, Tv, Tr):
        """Piece layout of the two forward chains.  Sequential: each chain gets every co-resident cluster in its own launch.
        Fused ("fused": True): ONE launch, the clusters split so that the two chains end together -- fewer, longer pieces
        each, but the discarded warm-up is paid once in wall time; chosen when the cost model says it is faster (always in
        the warm-up-dominated regime of small per-rank batches)."""
        wv, wr = self.warm["v"], self.warm["r"]
        r = self._pieces_for(Tr, wr)
        v = self._pieces_for(Tv, wv) if Tv > 0 else None
        if r is None or (Tv > 0 and v is None):
            return None
        # "b": the backward recurrence of the value chain always gets every co-resident cluster (its own launch); it may
        # be cut differently from the forward as long as the arrays cover both layouts (the stash rows past the forward's
        # end are zeroed: padding positions, whose gate gradients are exactly zero)
        wb = self.warm["b"]
        bw = None if v is None else self._pieces_for(Tv, wb, int(_lib.call("icrl_chain_tc_bwd_max_pieces")))
        if v is not None and bw is None:
            bw, wb = v, wv
        lay = {"v": None if v is None else (v[0], v[1], wv), "r": (r[0], r[1], wr), "fused": False,
               "b": None if bw is None else (bw[0], bw[1], wb)}
        if v is None or not self.chain_fuse_fwd or self.chain_pieces is not None:
            return lay
        C = int(_lib.call("icrl_chain_tc_max_pieces")) // 128
        cv, cr = self._STEP_COST["v"], self._STEP_COST["r"]
        best = (cv * (v[1] + wv) + cr * (r[1] + wr), None)
        for nv in range(1, C):
            Pv, Pr = min(128 * nv, v[0]), min(128 * (C - nv), r[0])
            if Pv < 2 or Pr < 2:
                continue
            sv, sr = -(-(Tv - wv) // Pv), -(-(Tr - wr) // Pr)
            t = max(cv * (sv + wv), cr * (sr + wr))
            if t < best[0]:
                best = (t, (Pv, sv, Pr, sr))
        if best[1] is not None:
            Pv, sv, Pr, sr = best[1]
            lay = dict(lay, v=(Pv, sv, wv), r=(Pr, sr, wr), fused=True)
        return lay

    def _padded(self, T, which):
        """Positions the arrays of a chain must hold (which: 0 = value, 1 = reward)."""
        if self._tc is None:
            return T
        lays = [self._tc["r"]] if which else [self._tc["v"], self._tc.get("b")]
        return max([T] + [l[0] * l[1] + l[2] for l in lays if l is not None])

    def _tc_scratch(self, key, P):
        """(ws, cp_state) of a tc chain launch; the tensors stay referenced by the engine."""
        ws = self._buf("tc_ws_" + key, (int(_lib.call("icrl_chain_tc_ws_bytes", P)) + 3) // 4)
        cp = self._buf("tc_cp_" + key, int(_lib.call("icrl_chain_tc_cp_floats", P)))
        return ws, cp

    def _chains_forward(self, f, B, S, Tv, Tr, train):
        st, L, b = self._stream, self.launches.ref, self._bufs
        Vn, R = self.value, self.reward
        K = self.chain_shards
        nv, nr = self._padded(Tv, 0), self._padded(Tr, 1)
        v_h = self._buf("v_stash_h", K * (nv + 1) * H)
        v_c = self._buf("v_stash_c", K * (nv + 1) * H)
        v_g = self._buf("v_stash_g", K * (nv + 1) * 4 * H)
        r_h = self._buf("r_stash_h", K * (nr + 1) * H)
        with self._phase("chains_fwd_fused"):
          if self._tc is not None:
            Pv, seg_v, warm_v = self._tc["v"]
            Pr, seg_r, warm_r = self._tc["r"]
            ws_v, cp_v = self._tc_scratch("v", Pv)
            ws_r, cp_r = self._tc_scratch("r", Pr)
            if self._tc.get("fused"):
                _lib.call("icrl_chains_tc_fwd_fused", st, Pv, seg_v, warm_v, _p(b["v_stream"]), _p(b["v_table"]), _p(b["v_chain_pk"]),
                          _p(v_h), _p(v_c), _p(v_g), _p(ws_v), _p(cp_v), _p(self._tc_err[0:]), Pr, seg_r, warm_r, _p(b["r_stream"]),
                          _p(b["r_table"]), _p(b["r_chain_pk"]), _p(R.rewrnn.gru.bias_hh_l0[2 * H:]), _p(r_h), _p(ws_r), _p(cp_r),
                          _p(self._tc_err[4:]), L)
            else:
                _lib.call("icrl_chain_tc_fwd", st, 0, Pv, seg_v, warm_v, _p(b["v_stream"]), _p(b["v_table"]), _p(b["v_chain_pk"]),
                          None, _p(v_h), _p(v_c), _p(v_g), _p(ws_v), _p(cp_v), _p(self._tc_err[0:]), L)
                _lib.call("icrl_chain_tc_fwd", st, 1, Pr, seg_r, warm_r, _p(b["r_stream"]), _p(b["r_table"]), _p(b["r_chain_pk"]),
                          _p(R.rewrnn.gru.bias_hh_l0[2 * H:]), _p(r_h), None, None, _p(ws_r), _p(cp_r), _p(self._tc_err[4:]), L)
          elif K > 1:
            _lib.call("icrl_chains_fwd_fused_sharded", st, K, _p(b["v_stream"]), Tv, _p(b["v_table"]),
                  _p(Vn.valrnn.lstm.weight_hh_l0), _p(v_h), _p(v_c), _p(v_g), _p(b["r_stream"]), Tr, _p(b["r_table"]),
                  _p(R.rewrnn.gru.weight_hh_l0), _p(R.rewrnn.gru.bias_hh_l0[2 * H:]), _p(r_h), _p(self.sync_state), L)
          else:
            _lib.call("icrl_chains_fwd_fused", st, _p(b["v_stream"]), Tv, _p(b["v_table"]), _p(Vn.valrnn.lstm.weight_hh_l0),
                  _p(v_h), _p(v_c), _p(v_g), _p(b["r_stream"]), Tr, _p(b["r_table"]), _p(R.rewrnn.gru.weight_hh_l0),
                  _p(R.rewrnn.gru.bias_hh_l0[2 * H:]), _p(r_h), _p(self.sync_state), L)
          if self._tc is not None and self._tc["v"] is not None:
            Pv, seg_v, warm_v = self._tc["v"]
            end_f = Pv * seg_v + warm_v
            if nv > end_f:                # rows only the backward layout reaches: finite (zero) stash, zero gradients
                v_g[end_f * 4 * H: nv * 4 * H].zero_()
                v_c[(end_f + 1) * H: (nv + 1) * H].zero_()
        SB = S * B
        v_take_h = self._buf("v_take_h", SB * H)
        r_take_h = self._buf("r_take_h", SB * H)
        _lib.call("icrl_gather_rows", st, SB, _p(v_h), _p(b["v_pos"]), 1, _p(v_take_h), L)
        _lib.call("icrl_gather_rows", st, SB, _p(r_h), _p(b["r_pos"]), 1, _p(r_take_h), L)
        values = torch.empty((B, S), dtype=torch.float32, device=self.device)
        rewards = torch.empty((B, S), dtype=torch.float32, device=self.device)
        _lib.call("icrl_value_head_fwd", st, B, S, _p(f), _p(v_take_h), _p(b["v_weff"]), _p(b["v_beff"]), _p(values), L)
        se = self._buf("r_se", SB * H)
        ve = self._buf("r_ve", B * H)
        if SB >= self._TC_LINEAR_MIN_ROWS:
            parts = self._buf("r_take_parts", 3 * SB * H, torch.bfloat16)
            _lib.call("icrl_split_bf16x3", st, SB * H, _p(r_take_h), _p(parts), L)
            _lib.call("icrl_gemm_bf16x3", st, SB, H, H, _p(parts), _p(b["r_se_parts"]), _p(se), H, _p(R.semantic_embed.bias), L)
        else:
            self._gemm(0, 1, SB, H, H, r_take_h, H, R.semantic_embed.weight, H, se, H, R.semantic_embed.bias)
        self._gemm(0, 1, B, H, H, f, H, R.visual_embed.weight, H, ve, H, R.visual_embed.bias)
        _lib.call("icrl_reward_cosine_fwd", st, B, S, _p(ve), _p(se), _p(rewards), L)
        return values, rewards

    def _backward(self, f, tokcm, tokens, B, p0, S, Tv, ent=None):
        """Backward of the minibatch.  The policy's backward depends only on dL/dlogp (and the entropy bonus, `ent` =
        (entropy [B][S], entropy_coef * inv_denom) or None); the value network's only on
        dL/dvalues: with overlap_backward the policy side runs on a second stream (own workspaces) while the main stream
        walks the value chain backwards -- the chain kernels occupy 120 of the 148 SMs (clusters of 8 cannot span GPCs),
        the policy's contractions fill the rest and whatever the chain kernel leaves in time."""
        main = torch.cuda.current_stream(self.device)
        if self.overlap_backward:
            if self._side_stream is None:
                self._side_stream = torch.cuda.Stream(device=self.device)
            fork = torch.cuda.Event()
            fork.record(main)
            self._backward_value(f, B, p0, S, Tv, launch_only_chain=True)
            self._side_stream.wait_event(fork)
            h_packed = None
            with torch.cuda.stream(self._side_stream):
                if self.wgrad == "tc" and self.chain_shards == 1:
                    # the h stash is final since the forward: its split (B operand of dW_hh = dgates^T h) leaves the
                    # critical path and runs beside the chain backward
                    _, gemm_ws, gemm_ws_floats, _ = self._bwd_workspaces(B, S, Tv, "")
                    _lib.call("icrl_wgrad_tc_pack_b", self._stream, 4 * H, H, Tv, _p(self._bufs["v_stash_h"]), H, _p(gemm_ws),
                              gemm_ws_floats * 4, 2, self.launches.ref)
                    h_packed = torch.cuda.Event()
                    h_packed.record(self._side_stream)
                self._backward_policy(f, tokcm, tokens, B, p0, S, "_p", ent)
                join = torch.cuda.Event()
                join.record(self._side_stream)
            if h_packed is not None:
                main.wait_event(h_packed)
            self._backward_value(f, B, p0, S, Tv, launch_only_chain=False, h_packed=h_packed is not None)
            main.wait_event(join)
        else:
            self._backward_value(f, B, p0, S, Tv, launch_only_chain=True)
            self._backward_value(f, B, p0, S, Tv, launch_only_chain=False)
            self._backward_policy(f, tokcm, tokens, B, p0, S, "", ent)

    def _bwd_workspaces(self, B, S, Tv, tag):
        """(colsum_ws, gemm_ws, gemm_ws_floats, dtable) of the value side (tag "") or the policy side on its own stream."""
        V = self.V
        SB = S * B
        cs_rows = max(SB, V, B)
        colsum_ws = self._buf("colsum_ws" + tag, int(_lib.call("icrl_colsum_ws_floats", cs_rows, 4 * H)) + 2 * H + 4 * H * 8)
        gemm_ws_floats = 24 * 4 * H * H
        if self.wgrad == "tc" or (not tag and self._tc is not None):
            if tag:       # policy side: dW_v (M = 1024) and dW_hh (M = 2048) contractions over S*B resp. n_cell*B rows
                n = max(int(_lib.call("icrl_wgrad_tc_ws_bytes", 4 * H, H, (self._n_cell_max) * B, 2)),
                        int(_lib.call("icrl_wgrad_tc_ws_bytes", 1024, H, SB, 2)))
            else:
                T_total = Tv if self.chain_shards == 1 else self.chain_shards * (Tv + 1)
                n = int(_lib.call("icrl_wgrad_tc_ws_bytes", 4 * H, H, T_total, 2))
                if not self.overlap_backward:
                    n = max(n, int(_lib.call("icrl_wgrad_tc_ws_bytes", 1024, H, SB, 2)))
            gemm_ws_floats = max(gemm_ws_floats, (n + 3) // 4)
        return colsum_ws, self._buf("gemm_ws" + tag, gemm_ws_floats), gemm_ws_floats, self._buf("dtable" + tag, V * 4 * H)

    def _backward_value(self, f, B, p0, S, Tv, launch_only_chain, h_packed=False):
        st, L, b, V = self._stream, self.launches.ref, self._bufs, self.V
        Vn = self.value
        SB = S * B
        g = self._g
        colsum_ws, gemm_ws, gemm_ws_floats, dtable = self._bwd_workspaces(B, S, Tv, "")
        K = self.chain_shards
        # fp32 gate gradients [rows][2048] (serial and shard kernels), or the tcgen05 pieces' fp16 pairs
        # [2][rows][2048] (same bytes) with their inverse scale in v_dg_scale
        rows = K * (self._padded(Tv, 0) + 1)
        dgates = self._buf("v_dgates", rows * 4 * H)
        dg_scale = self._buf("v_dg_scale", 1)
        if not launch_only_chain:
            lstm = Vn.valrnn.lstm
            D = Vn.valrnn.caption_embedding.weight.shape[1]
            tail = (_p(b["v_stash_h"]), _p(Vn.valrnn.caption_embedding.weight), _p(lstm.weight_ih_l0), _p(dtable), _p(colsum_ws),
                    _p(gemm_ws), gemm_ws_floats * 4, _p(g(Vn.valrnn.caption_embedding.weight, True)), _p(g(lstm.weight_ih_l0)),
                    _p(g(lstm.weight_hh_l0)), _p(g(lstm.bias_ih_l0)), _p(g(lstm.bias_hh_l0)))
            with self._phase("value_param_grads"):
              if self._tc is not None:
                _lib.call("icrl_value_chain_param_grads_pairs", st, Tv, V, D, _p(b["v_stream"]), _p(dgates), rows, _p(dg_scale),
                          *tail, B, p0, S, int(bool(h_packed)), L)
              else:
                _lib.call("icrl_value_chain_param_grads", st, Tv if K == 1 else K * (Tv + 1), V, D, _p(b["v_stream"]), _p(dgates),
                          *tail, B if K == 1 else 0, p0, S, int(bool(h_packed)), L)
            return
        # value head -> dh at the take positions + head gradients
        dh_take = self._buf("v_dh_take", SB * H)
        _lib.call("icrl_value_head_bwd", st, B, S, _p(f), _p(b["v_take_h"]), _p(b["dv_sb"]), _p(b["sum_dv"]),
                  _p(Vn.linear1.weight), _p(Vn.linear1.bias), _p(Vn.linear2.weight), _p(b["v_weff"]), _p(dh_take),
                  _p(g(Vn.linear1.weight)), _p(g(Vn.linear1.bias)), _p(g(Vn.linear2.weight)), _p(g(Vn.linear2.bias)),
                  _p(colsum_ws), L)
        # value chain BPTT and (second call) its parameter gradients (contractions over all T steps)
        with self._phase("chain_lstm_bwd"):
          if self._tc is not None:
            Pv, seg_v, warm_v = self._tc["b"]
            ws, _ = self._tc_scratch("v", Pv)
            cp = self._buf("tc_cp_b", int(_lib.call("icrl_chain_tc_cp_floats", Pv)))
            _lib.call("icrl_chain_tc_lstm_bwd", st, Pv, seg_v, warm_v, _p(b["v_chain_pk"]), _p(b["v_stash_g"]), _p(b["v_stash_c"]),
                      _p(b["v_take"]), _p(dh_take), SB, _p(dgates), rows, _p(dg_scale), _p(ws), _p(cp), _p(self._tc_err[8:]), L)
          elif K > 1:
            _lib.call("icrl_chain_lstm_bwd_sharded", st, K, Tv, _p(Vn.valrnn.lstm.weight_hh_l0), _p(b["v_stash_g"]),
                  _p(b["v_stash_c"]), _p(b["v_take"]), _p(dh_take), _p(dgates), _p(self.sync_state), L)
          else:
            _lib.call("icrl_chain_lstm_bwd", st, Tv, _p(Vn.valrnn.lstm.weight_hh_l0), _p(b["v_stash_g"]), _p(b["v_stash_c"]),
                  _p(b["v_take"]), _p(dh_take), _p(dgates), _p(self.sync_state), None, None, None, None, L)

    def _backward_policy(self, f, tokcm, tokens, B, p0, S, tag, ent=None, seed=None, bptt=None):
        # policy BPTT.  icrl_policy_rollout_bwd turns the logits into dL/dlogits IN PLACE; a step whose chains are re-run
        # (longer warm-up, serial fall-back) runs this backward again with slightly different dL/dlogp, so it works on a
        # copy and the rollout's logits stay intact.  seed(dz, ldz), when given, writes dL/dlogits into the [S*B][ldz]
        # buffer itself (padding columns included) and the backward starts from it (dlogp = NULL); bptt overrides
        # policy_bptt for this call.
        st, L, b, V = self._stream, self.launches.ref, self._bufs, self.V
        P = self.policy
        SB = S * B
        n_cell = p0 - 1 + S
        self._n_cell_max = max(self._n_cell_max, n_cell)
        g = self._g
        colsum_ws, gemm_ws, gemm_ws_floats, dtable = self._bwd_workspaces(B, S, 0, tag)
        pl = P.lstm
        tc = (bptt or self.policy_bptt) == "tc"
        ldz = int(_lib.call("icrl_vocab_pad")) if tc and V <= 1024 else V      # padded rows: vocabulary contractions on tcgen05
        dz = self._bufs.get("p_dlogits")
        if dz is None or dz.numel() < SB * ldz or self._dz_ld != ldz:
            dz = self._bufs["p_dlogits"] = torch.zeros(SB * ldz, dtype=torch.float32, device=self.device)   # padding stays zero
            self._dz_ld = ldz
        with self._phase("policy_bwd"):
          if seed is not None:
            seed(dz, ldz)
            dlogp = None
          else:
            dz[:SB * ldz].view(SB, ldz)[:, :V].copy_(b["p_logits"][:SB * V].view(SB, V))
            dlogp = b["dlogp"]
          if ent is not None:
            # dL/dlogits with the entropy bonus's term, in place; the rollout backward then starts from it (dlogp = NULL)
            _lib.call("icrl_softmax_entropy_bwd", st, B, S, V, _p(dz), ldz, _p(tokens), _p(dlogp), _p(ent[0]), ent[1], L)
            dlogp = None
          args = [st, B, V, p0, S, P.caption_embedding.weight.shape[1], _p(f), _p(P.caption_embedding.weight), _p(pl.weight_ih_l0),
                  _p(pl.weight_hh_l0), _p(P.linear2vocab.weight), _p(tokcm), _p(tokens), _p(dlogp), _p(b["p_Hs"]),
                  _p(b["p_Cs"]), _p(b["p_Gs"]), _p(dz), _p(self._buf("p_dHv", SB * H)),
                  _p(self._buf("p_DG", n_cell * B * 4 * H)), _p(self._buf("p_dh", 2 * B * H)), _p(self._buf("p_dc", B * H)),
                  _p(dtable), _p(colsum_ws), _p(gemm_ws), gemm_ws_floats * 4, _p(g(P.caption_embedding.weight, True)),
                  _p(g(P.cnn2linear.weight)), _p(g(P.cnn2linear.bias)), _p(g(pl.weight_ih_l0)), _p(g(pl.weight_hh_l0)),
                  _p(g(pl.bias_ih_l0)), _p(g(pl.bias_hh_l0)), _p(g(P.linear2vocab.weight)), _p(g(P.linear2vocab.bias))]
          if tc:
            # the n_cell serial cell-backward steps as ONE launch of the tcgen05 chain-backward kernel (rows = MMA rows)
            ws = self._buf("p_bptt_ws", (int(_lib.call("icrl_policy_bwd_tc_ws_bytes", B, S, n_cell)) + 3) // 4)
            _lib.call("icrl_policy_rollout_bwd_tc", *args, _p(b["p_chain_pk"]), _p(ws), _p(self._stat_err[20:]), ldz, L)
          else:
            _lib.call("icrl_policy_rollout_bwd", *args, L)

    # ------------------------------------------------------------------ public API
    def step(self, features, captions=None, uniforms=None, level=None, greedy=False, backward=True,
             global_rows=None, forced_tokens=None, repack=True, check=True, plan=None):
        """One A2C minibatch.  `features` may be a Prepared batch (already in HBM) or host/device data:
        features (B,512) f32, captions (B,L) int (host), uniforms (S,B) f64 or None
        (None draws them from numpy's global MT19937 stream exactly as np.random.choice would,
        trainers.py:447-450).  Returns StepResult or None when the curriculum level does not fit
        (trainers.py:550).  Gradients are written to the parameters' .grad (flat bucket)."""
        with torch.cuda.device(self.device):
            if isinstance(features, Prepared):
                prep = features
            else:
                p0, S = plan if plan is not None else plan_rollout(captions, level)
                if p0 < 1:
                    return None
                if S < 1:
                    raise ValueError("rollout needs at least one sampled step")
                B = int(captions.shape[0])
                if uniforms is None and not greedy and forced_tokens is None:
                    uniforms = np.random.random_sample(S * B).reshape(S, B)
                prep = self.prepare(features, captions, uniforms, plan=(p0, S))
            p0, S = prep.p0, prep.S
            self._attach_grads()
            if repack:
                self.pack_weights(reward="r_table" not in self._bufs)
            f, tokcm, u, fo, B = self._stage_inputs(prep, forced_tokens)
            tokens, logp = self._policy_forward(f, tokcm, u, fo, B, p0, S, greedy)
            dv_sb = self._buf("dv_sb", S * B)
            dlogp = self._buf("dlogp", S * B)
            sum_dv = self._buf("sum_dv", 1)
            inv = 1.0 / float((global_rows or B) * S)
            ent = None
            if self.entropy_coef:
                # the entropy of every sampled step's softmax, from the logits stash; a chain re-run leaves it as it is
                entropy = self._buf("p_entropy", S * B)
                with self._phase("policy_entropy"):
                    _lib.call("icrl_policy_entropy", self._stream, B, S, self.V, _p(self._bufs["p_logits"]), self.V, _p(entropy),
                              self.launches.ref)
                ent = (entropy, self.entropy_coef * inv)

            def run_chains(serial):
                Tv, Tr = self._streams(tokcm, B, p0, S, serial=serial)
                values, rewards = self._chains_forward(f, B, S, Tv, Tr, backward)
                if ent is None:
                    _lib.call("icrl_a2c_loss_fwd_bwd", self._stream, B, S, _p(values), _p(rewards), _p(logp), inv, _p(self._stat_err),
                              _p(dv_sb), _p(dlogp), _p(sum_dv), self.launches.ref)
                else:             # _stat_err[3] = mean entropy, brought over with the joint-check words
                    _lib.call("icrl_a2c_loss_entropy_fwd_bwd", self._stream, B, S, _p(values), _p(rewards), _p(logp), _p(ent[0]),
                              self.entropy_coef, inv, _p(self._stat_err), _p(dv_sb), _p(dlogp), _p(sum_dv), self.launches.ref)
                if backward:
                    self._backward(f, tokcm, tokens, B, p0, S, Tv, ent)
                self.segment_stats["steps"] += 1
                return Tv, Tr, values, rewards

            # Attempts 0 .. _TC_ATTEMPTS-1 run the chains cut into pieces; a failed joint check lengthens the warm-up and
            # tries again; the last attempt is always the serial kernels, the guaranteed floor.  Gradients are
            # overwritten, not accumulated, by a re-run.
            host, serial = None, False
            for attempt in range(self._TC_ATTEMPTS + 1):
                serial = serial or attempt == self._TC_ATTEMPTS
                Tv, Tr, values, rewards = run_chains(serial)
                if self._tc is None:
                    break
                self.segment_stats["segmented_steps"] += 1
                if not check:
                    self._seg_unverified = True       # the caller owes a segments_verified() before trusting the steps
                    break
                ok, host = self._tc_ok()
                if ok:
                    break
                host = None
                serial = self._tc_force_serial or attempt + 1 == self._TC_ATTEMPTS
                if serial:
                    self.segment_stats["fallbacks"] += 1
            n_stats = 3 if ent is None else 4
            stats = self._stat_err[:n_stats].clone()
            if check and self._tc is None:
                _lib.call("icrl_chain_check", self._stream, _p(self.sync_state))
        res = StepResult(tokens=tokens, logp=logp, values=values, rewards=rewards, stats=stats, p0=p0, S=S, B=B,
                         Tv=Tv, Tr=Tr)
        if host is not None:
            res.host_stats = host[:n_stats]
        return res

    _TC_ATTEMPTS = 3
    _SHRINK_AFTER = 2
    _HOLD_AFTER_GROWTH = 64
    _tc_force_serial = False

    def _adapt_warm(self, key, e_half, e_full):
        """Size the next warm-up of chain `key` from the joint errors half-way through / at the end of this one.
        The two errors give the contraction rate of the recurrence under the current weights: the warm-up GROWS as soon
        as the end-of-warm-up error passes chain_tol / 4 (before the check can fail; by the measured rate, at least
        x1.25, at most x4), and SHRINKS to 5/8 once the half-way error alone has been below that target on
        _SHRINK_AFTER consecutive steps (the new end point then lies beyond a point already measured clean); after a
        growth it is held for _HOLD_AFTER_GROWTH steps.  (A finer shrink by the positions the measured rate predicts can be
        given back was tried: 2 % faster on one GPU, but with 512 rows per rank the value chain then needed growth inside
        the next ten optimizer steps and paid for it with re-runs -- the half-way rule is the one with a measured point
        behind it.)  Returns False when the step failed its check (end-of-warm-up
        error above chain_tol, or not a number)."""
        tol = self.chain_tol
        target = tol / 4.0
        warm = self.warm[key]
        failed = not (e_full <= tol)
        self._hold[key] = max(0, self._hold[key] - 1)
        if failed or (self.chain_adapt and not (e_full <= target)):
            need = 2.0 * warm
            if e_half > e_full > 0.0 and np.isfinite(e_half):
                rate = np.log(e_half / e_full) / float(warm - warm // 2)         # nats forgotten per position
                need = warm + np.log(e_full / (target / 4.0)) / rate
            new = min(max(need, (1.5 if failed else 1.25) * warm), 4.0 * warm)
            self.warm[key] = int(-(-int(np.ceil(new)) // 32) * 32)
            self._clean[key] = 0
            self._hold[key] = self._HOLD_AFTER_GROWTH
        elif self.chain_adapt and warm >= 8 and e_half <= target and self._hold[key] == 0:
            self._clean[key] += 1
            if self._clean[key] >= self._SHRINK_AFTER and warm > self.chain_warmup_min:
                self.warm[key] = max(self.chain_warmup_min, int(-(-int(0.625 * warm) // 32) * 32))
                self._clean[key] = 0
        else:
            self._clean[key] = 0
        if self.warm[key] != warm:
            self.segment_stats["warm_history"].append((self.segment_stats["steps"], key, warm, self.warm[key]))
        return not failed

    def _tc_ok(self):
        """Joint checks of the tc chain launches of this step, read together with the three step statistics in ONE
        device-to-host copy (synchronises), and re-armed.  Returns (ok, host words)."""
        host = self._stat_err.tolist()
        self._tc_err.zero_()
        self._seg_unverified = False
        e = host[4:]
        st = self.segment_stats
        st["tc_max_err"] = [max(a, b) if b == b else float("nan") for a, b in zip(st["tc_max_err"], e)]
        nanmax = lambda xs: float("nan") if any(x != x for x in xs) else max(xs)
        self._tc_force_serial = e[13] != 0.0          # the fp16 exchange of the backward recurrence overflowed
        ok_v = ok_b = True
        if self._tc["v"] is not None:
            ok_v = self._adapt_warm("v", nanmax(e[2:4]), nanmax(e[0:2]))
            if e[12] != 0.0 or any(x != 0.0 for x in e[8:12]):        # the backward recurrence ran in this step
                ok_b = self._adapt_warm("b", nanmax(e[10:12]), nanmax(e[8:10]))
        ok_r = self._tc.get("r") is None or self._adapt_warm("r", e[6], e[4])
        ok = ok_v and ok_b and ok_r and not self._tc_force_serial
        if not ok:
            import warnings
            st["reruns"] += 1
            warnings.warn("chain segments did not converge onto the single chain within %g after the warm-up (value chain "
                          "forward |dh| %.3g |dc| %.3g, backward %.3g %.3g; reward chain |dh| %.3g%s): re-running with "
                          "warm-ups %s" % (self.chain_tol, e[0], e[1], e[8], e[9], e[4],
                                           "; gate gradients overflowed the fp16 exchange" if self._tc_force_serial else "",
                                           " / ".join("%d" % w for w in self.warm.values())))
        return ok, host

    @property
    def segment_layout(self):
        """(pieces, value-chain piece length, reward-chain piece length, warm-up) of the last step, or None when it ran on
        the serial kernels (chain too short, chain_segments = 1, or a failed warm-up check)."""
        if self._tc is None:
            return None
        v, r = self._tc["v"], self._tc["r"]
        return (r[0] if v is None else v[0], 0 if v is None else v[1], r[1], max(r[2], 0 if v is None else v[2]))

    @property
    def piece_layout(self):
        """{"v": (pieces, positions per piece, warm-up) | None, "r": (...)} of the last step on the tcgen05 chain kernels,
        or None."""
        return self._tc

    def segments_verified(self):
        """For callers that ran step(check=False): True when every segmented launch since the last check passed."""
        if not self._seg_unverified:
            return True
        with torch.cuda.device(self.device):
            return self._tc_ok()[0]

    def get_rewards(self, features, captions):
        """GetRewards on whole captions from zero state (trainers.py:108-121): (B,1) tensor."""
        caps = np.asarray(captions)
        B, Lc = caps.shape
        with torch.cuda.device(self.device):
            if "r_table" not in self._bufs or self._reward_changed():
                self.pack_reward()
            f, tokcm, _, _, _ = self._stage_inputs(self.prepare(features, caps, plan=(Lc, 0)), None)
            st, L, b, R = self._stream, self.launches.ref, self._bufs, self.reward
            T = int(_lib.call("icrl_stream_len", B, Lc, 1, 0))
            serial = False
            for attempt in range(self._TC_ATTEMPTS + 1):
                serial = serial or attempt == self._TC_ATTEMPTS
                self._tc = self._pick_pieces(0, T) if not serial and self._use_tc_chains() else None
                n = self._padded(T, 1)
                r_stream, r_pos = self._buf("r_stream", n, torch.int32), self._buf("r_pos", B, torch.int32)
                _lib.call("icrl_build_stream", st, B, Lc, 1, 0, _p(tokcm), _p(r_stream), None, _p(r_pos), L)
                r_h = self._buf("r_stash_h", (n + 1) * H)
                if self._tc is not None:
                    Pr, seg_r, warm_r = self._tc["r"]
                    r_stream[T:n].zero_()
                    ws, cp = self._tc_scratch("r", Pr)
                    _lib.call("icrl_chain_tc_fwd", st, 1, Pr, seg_r, warm_r, _p(r_stream), _p(b["r_table"]), _p(b["r_chain_pk"]),
                              _p(R.rewrnn.gru.bias_hh_l0[2 * H:]), _p(r_h), None, None, _p(ws), _p(cp), _p(self._tc_err[4:]), L)
                    ok, _ = self._tc_ok()
                    if ok:
                        break
                    serial = attempt + 1 == self._TC_ATTEMPTS
                    if serial:
                        self.segment_stats["fallbacks"] += 1
                else:
                    _lib.call("icrl_chain_gru_fwd", st, _p(r_stream), T, _p(b["r_table"]), _p(R.rewrnn.gru.weight_hh_l0),
                              _p(R.rewrnn.gru.bias_hh_l0[2 * H:]), None, _p(r_h), None, _p(self.sync_state), None, L)
                    break
            r_take_h = self._buf("r_take_h", B * H)
            _lib.call("icrl_gather_rows", st, B, _p(r_h), _p(r_pos), 1, _p(r_take_h), L)
            se, ve = self._buf("r_se", B * H), self._buf("r_ve", B * H)
            self._gemm(0, 1, B, H, H, r_take_h, H, R.semantic_embed.weight, H, se, H, R.semantic_embed.bias)
            self._gemm(0, 1, B, H, H, f, H, R.visual_embed.weight, H, ve, H, R.visual_embed.bias)
            rewards = torch.empty((B, 1), dtype=torch.float32, device=self.device)
            _lib.call("icrl_reward_cosine_fwd", st, B, 1, _p(ve), _p(se), _p(rewards), L)
            _lib.call("icrl_chain_check", st, _p(self.sync_state))
        return rewards

    def greedy_decode(self, features, first_col, steps=16):
        """GenerateCaptionsGreedy (trainers.py:57-70): (B, steps+1) int64 tokens and last-step logits."""
        first = np.asarray(first_col, dtype=np.int64).reshape(-1, 1)
        B = first.shape[0]
        with torch.cuda.device(self.device):
            self.pack_weights(reward=False)
            f, tokcm, _, _, _ = self._stage_inputs(self.prepare(features, first, plan=(1, steps)), None)
            tokens, _ = self._policy_forward(f, tokcm, None, None, B, 1, steps, True)
            last = self._bufs["p_logits"][(steps - 1) * B * self.V: steps * B * self.V].view(B, self.V).clone()
            out = torch.cat((torch.from_numpy(first).to(self.device), tokens), dim=1)
        return out, last


class PolicyOnlyEngine(A2CEngine):
    """A2CEngine restricted to the policy (greedy decode needs no value / reward network)."""

    def __init__(self, policy_network):
        self.policy, self.value, self.reward, self.a2c = policy_network, None, None, policy_network
        dev = policy_network.linear2vocab.weight.device
        if dev.type != "cuda":
            raise _lib.IcrlError("the policy engine needs the policy on a CUDA device (no CPU fallback)")
        _lib.load()
        self.device, self.V = dev, policy_network.linear2vocab.weight.shape[0]
        self._bufs, self.launches, self.phase_events = {}, _lib.Launches(), None
        self.decode, self.use_tc = ("fused" if self.V <= 1024 and self.V % 4 == 0 else "simt"), False

    def pack_weights(self, reward=False):
        P = self.policy
        _lib.call("icrl_pack_gate_table", self._stream, self.V, 4 * H, 4 * H, P.caption_embedding.weight.shape[1], _p(P.caption_embedding.weight),
                  _p(P.lstm.weight_ih_l0), _p(P.lstm.bias_ih_l0), _p(P.lstm.bias_hh_l0),
                  _p(self._buf("p_table", self.V * 4 * H)), self.launches.ref)
        if self.decode == "fused":
            n = int(_lib.call("icrl_decode_weight_halves"))
            _lib.call("icrl_pack_decode_weights", self._stream, self.V, _p(P.lstm.weight_hh_l0), _p(P.linear2vocab.weight),
                      _p(self._buf("p_decode_pk", n, torch.float16)), self.launches.ref)


class PolicyPretrainEngine(PolicyOnlyEngine):
    """Cross-entropy pretraining of the unidirectional policy (train_policy_network, trainers.py:202-257) on the fused
    engine: per minibatch the teacher-forced decode of A2CEngine (the persistent tcgen05 kernel with forced tokens; the
    per-step kernels where A2CEngine takes them), the fused masked cross entropy (icrl_policy_xent_fwd_bwd) and the
    policy backward of A2CEngine started from its dL/dlogits.  Gradients land in the flat bucket over
    policy.parameters() that the parameters' .grad alias, so optim.FlatAdam(engine) steps them.

    policy_bptt: "tc" runs the serial cell-backward steps on the tcgen05 chain-backward kernel; when its fp16 exchange
    overflows, the minibatch's backward is re-run on the fp32 kernels ("simt", which can also be chosen outright)."""

    def __init__(self, policy_network, policy_bptt="tc"):
        super().__init__(policy_network)
        if getattr(policy_network, "bidirectional", False):
            raise NotImplementedError("the fused pretraining engine is built for the unidirectional policy; bidirectional=True "
                                      "runs on the module (autograd) route")
        if policy_bptt not in ("tc", "simt"):
            raise ValueError("policy_bptt must be 'tc' or 'simt'")
        self.policy_bptt, self.wgrad, self._n_cell_max, self._dz_ld = policy_bptt, "tc", 1, None
        self.bptt_reruns = 0          # minibatches whose backward fell back to the fp32 kernels
        with torch.cuda.device(self.device):
            # [0] the loss; [20:28] words of the policy's tcgen05 BPTT ([25] fp16-exchange overflow flag): ONE copy per step
            self._stat_err = torch.zeros(28, dtype=torch.float32, device=self.device)
        self._check_params()
        self._bind_flat_grads()

    def pack_weights(self, reward=False):
        super().pack_weights()
        if self.policy_bptt == "tc":
            n = int(_lib.call("icrl_chain_tc_weight_halves", 0))
            _lib.call("icrl_pack_chain_tc_weights", self._stream, 0, _p(self.policy.lstm.weight_hh_l0),
                      _p(self._buf("p_chain_pk", n, torch.float16)), self.launches.ref)

    def xent_step(self, features, captions):
        """One minibatch of train_policy_network: features (B,512) f32 (host or device), captions (B,L) int (host).
        Leaves the gradients of the reference's loss in the parameters' .grad (flat bucket) and returns the loss (one
        device-to-host copy, which also brings the BPTT's overflow flag)."""
        caps = captions.cpu().numpy() if isinstance(captions, torch.Tensor) else np.asarray(captions)
        n, w, S = plan_xent(caps)
        if caps.min() < 0 or caps.max() >= self.V:
            raise ValueError("caption tokens must lie in [0, %d)" % self.V)
        B, V = caps.shape[0], self.V
        with torch.cuda.device(self.device):
            self._attach_grads()
            self.pack_weights()
            prep = self.prepare(features, caps, plan=(1, S))
            f, tokcm, _, fo, _ = self._stage_inputs(prep, caps[:, 1:1 + S])
            tokens, _ = self._policy_forward(f, tokcm, None, fo, B, 1, S, False)
            n_rows = torch.from_numpy(n.astype(np.int32)).to(self.device, non_blocking=True)
            w_rows = torch.from_numpy(w.astype(np.float64)).to(self.device, non_blocking=True)
            ce = self._buf("p_xent_ce", S * B)

            def seed(dz, ldz):
                _lib.call("icrl_policy_xent_fwd_bwd", self._stream, B, S, V, _p(self._bufs["p_logits"]), _p(fo), _p(n_rows),
                          _p(w_rows), _p(dz), ldz, _p(ce), _p(self._stat_err), self.launches.ref)

            self._backward_policy(f, tokcm, tokens, B, 1, S, "_p", seed=seed)
            host = self._stat_err[:26].tolist()
            if self.policy_bptt == "tc" and host[25] != 0.0:
                # the gate gradients overflowed the tcgen05 BPTT's fp16 exchange: the same backward on the fp32 kernels
                self.bptt_reruns += 1
                self._backward_policy(f, tokcm, tokens, B, 1, S, "_p", seed=seed, bptt="simt")
        return host[0]


class LookAheadEngine(A2CEngine):
    """The value-guided look-ahead decoder of the reference's evaluation path (GenerateCaptionsWithActorCriticLookAhead,
    trainers.py:73-105) on the fused engine; no reward network.

    Per beam step the K candidates' policy states advance by one cell on the tensor-core GEMMs (icrl_lookahead_policy_step:
    the reference re-runs every full prefix), and the K*k value calls of the step -- known before any value is needed,
    because the policy's top-k does not depend on them -- are ONE carried-state chain launch: tcgen05 pieces from the
    carried (h, c) (icrl_chain_tc_lstm_fwd_from) with the joint checks, re-runs with a longer warm-up and the serial floor of
    A2CEngine.step.  The value state starts from value_network.valrnn.hidden_cell and is written back to it (Q1)."""

    def __init__(self, policy_network, value_network, chain_segments=32, chain_warmup=256, chain_tol=1e-5, chain_pieces=None,
                 chain_adapt=True, chain_warmup_min=32):
        self.policy, self.value, self.reward, self.a2c = policy_network, value_network, None, policy_network
        if getattr(policy_network, "bidirectional", False) or getattr(value_network, "bidirectional", False):
            raise NotImplementedError("the look-ahead engine is built for the unidirectional networks")
        dev = policy_network.linear2vocab.weight.device
        if dev.type != "cuda" or value_network.linear1.weight.device != dev:
            raise _lib.IcrlError("the look-ahead engine needs both networks on one CUDA device (no CPU fallback)")
        _lib.load()
        self.device, self.V = dev, policy_network.linear2vocab.weight.shape[0]
        self._bufs, self.launches, self.phase_events = {}, _lib.Launches(), None
        self.chain_shards, self.chain_segments = 1, int(chain_segments)
        self.chain_pieces = None if chain_pieces is None else int(chain_pieces)
        self.chain_warmup, self.chain_tol = int(chain_warmup), float(chain_tol)
        self.chain_adapt, self.chain_warmup_min = bool(chain_adapt), int(chain_warmup_min)
        self.warm, self._clean, self._hold = {"v": self.chain_warmup}, {"v": 0}, {"v": 0}
        self._tc = None
        self.segment_stats = {"steps": 0, "segmented_steps": 0, "fallbacks": 0, "reruns": 0, "tc_max_err": [0.0] * 16,
                              "warm_history": []}
        self._seg_unverified = False
        # per beam step: "pieces", "fallback" (pieces failed their checks, the serial kernels finished) or "serial" (too
        # short to cut)
        self.step_paths = []
        with torch.cuda.device(dev):
            self.sync_state = torch.zeros(int(_lib.call("icrl_chain_sync_bytes")), dtype=torch.uint8, device=dev)
            # [4:20] joint-check words of the chain launch, [28:28+K*k] the children's batch means: ONE copy per beam step
            self._stat_err = torch.zeros(28 + 16 * 16, dtype=torch.float32, device=dev)
        self._tc_err = self._stat_err[4:20]

    def pack_weights(self, reward=False):
        """The operands of both networks, once per look_ahead call: gate tables, bf16x3 splits of the policy's W_hh and
        W_v, the collapsed value head and the value chain's tcgen05 W_hh."""
        st, L, V, c = self._stream, self.launches.ref, self.V, _lib.call
        P, Vn = self.policy, self.value
        for key, emb, lstm in (("p", P.caption_embedding, P.lstm), ("v", Vn.valrnn.caption_embedding, Vn.valrnn.lstm)):
            c("icrl_pack_gate_table", st, V, 4 * H, 4 * H, emb.weight.shape[1], _p(emb.weight), _p(lstm.weight_ih_l0),
              _p(lstm.bias_ih_l0), _p(lstm.bias_hh_l0), _p(self._buf(key + "_table", V * 4 * H)), L)
        self._pack_policy_tc()
        c("icrl_pack_value_head", st, _p(Vn.linear1.weight), _p(Vn.linear1.bias), _p(Vn.linear2.weight), _p(Vn.linear2.bias),
          _p(self._buf("v_weff", 2 * H)), _p(self._buf("v_beff", 1)), L)
        if self._use_tc_chains():
            c("icrl_pack_chain_tc_weights", st, 0, _p(Vn.valrnn.lstm.weight_hh_l0),
              _p(self._buf("v_chain_pk", int(c("icrl_chain_tc_weight_halves", 0)), torch.float16)), L)

    def _value_chain(self, B, n, Kc, K, cand_tok, words, h0, c0):
        """The value calls of one beam step as one chain from (h0, c0): values [B][Kc*K] and the chain's final (h, c) rows.
        Pieces first; a failed joint check re-runs with the grown warm-up, then the serial kernels (A2CEngine.step)."""
        st, L, b, Vn = self._stream, self.launches.ref, self._bufs, self.value
        S = Kc * K
        T = S * (n + 1) * B
        serial, tried = False, False
        for attempt in range(self._TC_ATTEMPTS + 1):
            serial = serial or attempt == self._TC_ATTEMPTS
            lay = None if serial or not self._use_tc_chains() else self._pieces_for(T, self.warm["v"])
            self._tc = None if lay is None else {"v": (lay[0], lay[1], self.warm["v"]), "r": None}
            npad = T if lay is None else max(T, lay[0] * lay[1] + self.warm["v"])
            v_stream, take_pos = self._buf("la_stream", npad, torch.int32), self._buf("la_take_pos", S * B, torch.int32)
            stash_h, stash_c = self._buf("la_stash_h", (npad + 1) * H), self._buf("la_stash_c", (npad + 1) * H)
            _lib.call("icrl_lookahead_stream", st, B, n, Kc, K, _p(cand_tok), _p(words), _p(v_stream), _p(take_pos), L)
            with self._phase("lookahead_value_chain"):
              if lay is not None:
                v_stream[T:npad].zero_()          # the last piece runs past the end of the chain
                ws, cp = self._tc_scratch("v", lay[0])
                _lib.call("icrl_chain_tc_lstm_fwd_from", st, lay[0], lay[1], self.warm["v"], _p(v_stream), _p(b["v_table"]),
                          _p(b["v_chain_pk"]), _p(h0), _p(c0), _p(stash_h), _p(stash_c), None, _p(ws), _p(cp),
                          _p(self._tc_err), L)
              else:
                _lib.call("icrl_chain_lstm_fwd", st, _p(v_stream), T, _p(b["v_table"]), _p(Vn.valrnn.lstm.weight_hh_l0), _p(h0),
                          _p(c0), _p(stash_h), _p(stash_c), None, None, None, _p(self.sync_state), L)
            take_h = self._buf("la_take_h", S * B * H)
            _lib.call("icrl_gather_rows", st, S * B, _p(stash_h), _p(take_pos), 1, _p(take_h), L)
            values = self._buf("la_values", B * S)
            _lib.call("icrl_value_head_fwd", st, B, S, _p(self._la_f), _p(take_h), _p(b["v_weff"]), _p(b["v_beff"]), _p(values), L)
            self.segment_stats["steps"] += 1
            if lay is None:
                break
            tried = True
            self.segment_stats["segmented_steps"] += 1
            _lib.call("icrl_lookahead_score", st, B, Kc, K, _p(self._la_parent_score), _p(values), _p(self._la_top_val),
                      _p(self._la_child), _p(self._stat_err[28:]), L)
            ok, host = self._tc_ok()
            if ok:
                self.step_paths.append("pieces")
                return stash_h[T * H:(T + 1) * H], stash_c[T * H:(T + 1) * H], host
            serial = attempt + 1 == self._TC_ATTEMPTS
        if tried:
            self.segment_stats["fallbacks"] += 1
        self.step_paths.append("fallback" if tried else "serial")
        _lib.call("icrl_lookahead_score", st, B, Kc, K, _p(self._la_parent_score), _p(values), _p(self._la_top_val),
                  _p(self._la_child), _p(self._stat_err[28:]), L)
        _lib.call("icrl_chain_check", st, _p(self.sync_state))
        return stash_h[T * H:(T + 1) * H], stash_c[T * H:(T + 1) * H], self._stat_err.tolist()

    def look_ahead(self, features, first_col, beam=5, steps=16):
        """GenerateCaptionsWithActorCriticLookAhead(most_likely=False) from the caption column `first_col` (B,): the
        reference's list of `beam` (captions (B, steps+1) int64, score (B,1) f32) device tensors, best first."""
        K = int(beam)
        if not 1 <= K <= 16:
            raise ValueError("the fused look-ahead keeps 1 to 16 candidates")
        first = torch.as_tensor(np.asarray(first_col).reshape(-1).astype(np.int32))
        B, V = first.numel(), self.V
        dev, i32 = self.device, torch.int32
        with torch.cuda.device(dev):
            st, L = self._stream, self.launches.ref
            P, rnn = self.policy, self.value.valrnn
            self.pack_weights()
            self._la_f = torch.as_tensor(features).to(dev, torch.float32).reshape(B, H).contiguous()
            hc = rnn.hidden_cell
            h0 = hc[0].to(dev, torch.float32).reshape(H).clone()
            c0 = hc[1].to(dev, torch.float32).reshape(H).clone()
            cand_tok = first.to(dev).view(1, 1, B)                  # [candidates][columns][B]
            tok, parent = cand_tok.reshape(-1), None
            score = torch.zeros((1, B), dtype=torch.float32, device=dev)
            h_st = c_st = None
            rows_b = torch.arange(B, dtype=i32, device=dev)
            for t in range(steps):
                Kc, n = cand_tok.shape[0], cand_tok.shape[1]
                R, S = Kc * B, Kc * K
                h_out, c_out = torch.empty((R, H), device=dev), torch.empty((R, H), device=dev)
                self._la_top_val = torch.empty((R, K), dtype=torch.float32, device=dev)
                top_idx = torch.empty((R, K), dtype=i32, device=dev)
                ws = self._buf("la_policy_ws", (R * (46 * H + 4 * V) + 3) // 4)
                with self._phase("lookahead_policy"):
                    _lib.call("icrl_lookahead_policy_step", st, R, V, K, int(t == 0), _p(self._la_f), _p(P.cnn2linear.weight),
                              _p(P.cnn2linear.bias), _p(self._bufs["p_table"]), _p(parent), _p(h_st), _p(c_st), _p(tok),
                              _p(self._bufs["p_whh_parts"]), _p(self._bufs["p_wv_parts"]), _p(P.linear2vocab.bias), _p(h_out),
                              _p(c_out), None, _p(self._la_top_val), _p(top_idx), _p(ws), L)
                self._la_parent_score = score
                self._la_child = torch.empty((S, B), dtype=torch.float32, device=dev)
                h_fin, c_fin, host = self._value_chain(B, n, Kc, K, cand_tok, top_idx, h0, c0)
                h0.copy_(h_fin)
                c0.copy_(c_fin)
                # trainers.py:93-94: a stable sort of the K*k children on their batch means, in the reference's list order
                means = host[28:28 + S]
                keep = sorted(range(S), key=lambda s: means[s])[:K]
                sel = torch.tensor(keep, dtype=torch.int64).to(dev, non_blocking=True)
                cand, word = sel // K, sel % K
                words = top_idx.view(Kc, B, K)[cand, :, word]                          # [K][B]
                cand_tok = torch.cat((cand_tok[cand], words.unsqueeze(1)), dim=1).contiguous()
                score = self._la_child[sel].contiguous()
                parent = (cand.to(i32).unsqueeze(1) * B + rows_b).reshape(-1).contiguous()
                tok = words.reshape(-1).contiguous()
                h_st, c_st = h_out, c_out
            rnn.hidden_cell = (h0.view(1, 1, H), c0.view(1, 1, H))
            caps = cand_tok.permute(0, 2, 1).to(torch.int64).contiguous()
            return [(caps[j], score[j].view(B, 1)) for j in range(cand_tok.shape[0])]
