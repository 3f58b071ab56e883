"""ctypes binding of libicrl_b200.so (the C ABI declared in include/icrl_b200.h).

There is no CPU fallback: if the shared library is missing or a call fails, this raises.
Build with ``python -c "import __graft_entry__ as g; g.build()"`` or ``make -C csrc``.
"""
import ctypes
import os
from ctypes import c_char_p, c_double, c_float, c_int, c_longlong, c_size_t, c_void_p, POINTER

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ICRL_LIB_PATH") or os.path.join(_HERE, "libicrl_b200.so")   # override: A/B builds only

P = c_void_p          # device pointer / stream
I = c_int
L = c_longlong
F = c_float
Z = c_size_t
LP = POINTER(c_int)   # host int* launch counter

# name -> argtypes (restype is int unless listed in _RESTYPES)
SIGNATURES = {
    "icrl_last_error": [],
    "icrl_version": [],
    "icrl_device_info": [LP],
    "icrl_gemm_f32": [P, I, I, I, I, I, P, I, P, I, P, I, P, F, P, Z, LP],
    "icrl_split_bf16x3": [P, L, P, P, LP],
    "icrl_gemm_bf16x3": [P, I, I, I, P, P, P, I, P, LP],
    "icrl_policy_rollout_fwd_tc": [P, I, I, I, I, I] + [P] * 18 + [LP],
    "icrl_wgrad_tc_ws_bytes": [I, I, L, I],
    "icrl_wgrad_tc": [P, I, I, L, P, I, P, I, P, I, P, Z, I, LP],
    "icrl_decode_weight_halves": [],
    "icrl_decode_set_profile": [P],
    "icrl_pack_decode_weights": [P, I, P, P, P, LP],
    "icrl_policy_rollout_fwd_fused": [P, I, I, I, I, I] + [P] * 17 + [LP],
    "icrl_pack_gate_table": [P, I, I, I, I, P, P, P, P, P, LP],
    "icrl_pack_value_head": [P, P, P, P, P, P, P, LP],
    "icrl_policy_rollout_fwd": [P, I, I, I, I, I] + [P] * 17 + [LP],
    "icrl_policy_rollout_bwd": [P, I, I, I, I, I] + [P] * 19 + [Z] + [P] * 9 + [LP],
    "icrl_policy_rollout_bwd_tc": [P, I, I, I, I, I] + [P] * 19 + [Z] + [P] * 9 + [P, P, P, I, LP],
    "icrl_policy_bwd_tc_ws_bytes": [I, I, I],
    "icrl_vocab_pad": [],
    "icrl_colsum_ws_floats": [L, I],
    "icrl_lstm_seq_fwd": [P, I, I] + [P] * 8 + [LP],
    "icrl_lstm_seq_bwd": [P, I, I, I, I] + [P] * 14 + [Z] + [P] * 6 + [LP],
    "icrl_stream_len": [I, I, I, I],
    "icrl_build_stream": [P, I, I, I, I, P, P, P, P, LP],
    "icrl_build_stream_sharded": [P, I, I, I, I, I, P, P, P, P, LP],
    "icrl_chains_fwd_fused_sharded": [P, I, P, I, P, P, P, P, P, P, I, P, P, P, P, P, LP],
    "icrl_chain_lstm_bwd_sharded": [P, I, I, P, P, P, P, P, P, P, LP],
    "icrl_chain_tc_max_pieces": [],
    "icrl_chain_tc_weight_halves": [I],
    "icrl_chain_tc_ws_bytes": [I],
    "icrl_chain_tc_cp_floats": [I],
    "icrl_pack_chain_tc_weights": [P, I, P, P, LP],
    "icrl_chain_tc_fwd": [P, I, I, L, I] + [P] * 10 + [LP],
    "icrl_chains_tc_fwd_fused": [P, I, L, I] + [P] * 9 + [I, L, I] + [P] * 8 + [LP],
    "icrl_chain_tc_lstm_bwd": [P, I, L, I, P, P, P, P, P, L, P, L, P, P, P, P, LP],
    "icrl_chain_tc_lstm_fwd_from": [P, I, L, I] + [P] * 11 + [LP],
    "icrl_lookahead_stream": [P, I, I, I, I, P, P, P, P, LP],
    "icrl_lookahead_policy_step": [P, I, I, I, I] + [P] * 17 + [LP],
    "icrl_lookahead_score": [P, I, I, I, P, P, P, P, P, LP],
    "icrl_chain_tc_set_profile": [P],
    "icrl_chain_tc_set_bias": [F, F],
    "icrl_chain_tc_bwd_max_pieces": [],
    "icrl_chain_tc_set_tma_store": [I],
    "icrl_chain_set_profile": [P],
    "icrl_chain_sync_bytes": [],
    "icrl_chain_lstm_fwd": [P, P, I] + [P] * 10 + [LP],
    "icrl_chain_gru_fwd": [P, P, I] + [P] * 8 + [LP],
    "icrl_chain_gru_bwd": [P, I] + [P] * 10 + [LP],
    "icrl_reward_chain_param_grads": [P, I, I, I] + [P] * 9 + [Z] + [P] * 5 + [LP],
    "icrl_linear_bwd": [P, I, I, I] + [P] * 8 + [Z, LP],
    "icrl_chains_fwd_fused": [P, P, I, P, P, P, P, P, P, I, P, P, P, P, P, LP],
    "icrl_chain_lstm_bwd": [P, I, P, P, P, P, P, P, P, P, P, P, P, LP],
    "icrl_adam_flat": [P, L, P, P, P, P, F, F, F, F, I, LP],
    "icrl_chain_check": [P, P],
    "icrl_gather_rows": [P, L, P, P, L, P, LP],
    "icrl_value_head_fwd": [P, I, I, P, P, P, P, P, LP],
    "icrl_value_head_bwd": [P, I, I] + [P] * 14 + [LP],
    "icrl_value_chain_param_grads": [P, I, I, I] + [P] * 8 + [Z] + [P] * 5 + [I, I, I, I, LP],
    "icrl_value_chain_param_grads_pairs": [P, I, I, I, P, P, L] + [P] * 7 + [Z] + [P] * 5 + [I, I, I, I, LP],
    "icrl_wgrad_tc_pack_b": [P, I, I, L, P, I, P, Z, I, LP],
    "icrl_reward_cosine_fwd": [P, I, I, P, P, P, LP],
    "icrl_a2c_loss_fwd_bwd": [P, I, I, P, P, P, F, P, P, P, P, LP],
    "icrl_policy_entropy": [P, I, I, I, P, I, P, LP],
    "icrl_a2c_loss_entropy_fwd_bwd": [P, I, I, P, P, P, P, F, F, P, P, P, P, LP],
    "icrl_softmax_entropy_bwd": [P, I, I, I, P, I, P, P, P, F, LP],
    "icrl_policy_xent_fwd_bwd": [P, I, I, I, P, P, P, P, P, I, P, P, LP],
}
_RESTYPES = {"icrl_last_error": c_char_p, "icrl_wgrad_tc_ws_bytes": c_size_t, "icrl_decode_weight_halves": c_size_t, "icrl_colsum_ws_floats": c_size_t, "icrl_stream_len": c_longlong,
             "icrl_chain_sync_bytes": c_size_t, "icrl_chain_tc_weight_halves": c_size_t, "icrl_chain_tc_ws_bytes": c_size_t, "icrl_chain_tc_cp_floats": c_size_t,
             "icrl_policy_bwd_tc_ws_bytes": c_size_t}
_NO_STATUS = set(_RESTYPES) | {"icrl_version", "icrl_chain_tc_max_pieces", "icrl_chain_tc_bwd_max_pieces", "icrl_vocab_pad"}


class IcrlError(RuntimeError):
    pass


_lib = None


def load():
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise IcrlError("libicrl_b200.so is missing (%s): build it with __graft_entry__.build(); "
                            "there is no CPU fallback" % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH)
        for name, args in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.argtypes = args
            fn.restype = _RESTYPES.get(name, c_int)
        _lib = lib
    return _lib


class Launches:
    """Host-side launch counter handed to the C ABI (gpu_launches in bench.py)."""

    def __init__(self):
        self.c = c_int(0)

    @property
    def ref(self):
        return ctypes.byref(self.c)

    @property
    def value(self):
        return self.c.value


def call(name, *args):
    """Invoke an entry point; raise IcrlError with icrl_last_error() on a non-zero status."""
    lib = load()
    rc = getattr(lib, name)(*args)
    if name in _NO_STATUS:
        return rc
    if rc != 0:
        raise IcrlError("%s failed (code %d): %s" % (name, rc, lib.icrl_last_error().decode()))
    return rc
