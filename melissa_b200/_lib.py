"""ctypes binding of libmelissa_b200.so (include/melissa_b200.h).

There is NO CPU fallback: if the library cannot be loaded every entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libmelissa_b200.so")

MLS_EP_SOURCE, MLS_EP_WORLD_MSGS, MLS_EP_NUM_MOVES, MLS_EP_GRAPH, MLS_EP_N_RESETS, MLS_EP_STRIDE = 0, 1, 2, 3, 4, 8
F_HAS_MESSAGE, F_INTERESTED, F_SCRIPTED, F_ORIGIN, F_HAS_TAKEN_ACTION, F_TRUNCATED, F_ACTIVE = 1, 2, 4, 8, 16, 32, 64
NODE_STEPS_SHIFT, NODE_MSGS_SHIFT = 8, 16

HEURISTIC_IDS = {None: 0, "silent": 1, "simple_broadcast": 2, "broadcast_if_any_interested": 3,
                 "probabilistic_gossip": 4, "probabilistic_relay": 5, "mpr": 6}
NET_KINDS = {"dgn_r": 0, "l_dgn": 1, "hl_dgn": 2}
POOLS = {"mean": 0, "add": 1, "max": 2}
PRECISIONS = {"fp32": 0, "bf16": 1}

vp = C.c_void_p


class MlsEnvDesc(C.Structure):
    _fields_ = [("n_episodes", C.c_int32), ("n_nodes", C.c_int32), ("dynamic", C.c_int32), ("is_testing", C.c_int32),
                ("heuristic", C.c_int32), ("episode_offset", C.c_int32), ("batch_episodes", C.c_int32),
                ("reserved", C.c_int32)]


class MlsEnvState(C.Structure):
    _fields_ = [("node", vp), ("recv_count", vp), ("recv_from", vp), ("episode", vp), ("rewards_sum", vp),
                ("adj", vp), ("pos", vp), ("pool_adj", vp), ("pool_pos", vp), ("pool_size", C.c_int32), ("pad_", C.c_int32)]


class MlsResetTuples(C.Structure):
    _fields_ = [("graph_index", vp), ("source", vp), ("interested", vp), ("scripted", vp), ("count", C.c_int32),
                ("pad_", C.c_int32)]


class MlsEpisodeSampler(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("pool_size", C.c_int32), ("n_scripted", C.c_int32),
                ("drop_source_from_scripted", C.c_int32), ("slot_offset", C.c_int32)]


class MlsInfo(C.Structure):
    _fields_ = [(k, C.c_int32) for k in (
        "total_messages_transmitted", "covered", "messages_sent", "messages_received", "n_neighbours",
        "interested_agents", "coverage_interested_count", "uninterested_with_message", "num_moves", "n_acted",
        "episodes_started", "reserved")] + [("episode_rewards_sum", C.c_double)]


INFO_INT_FIELDS = [f[0] for f in MlsInfo._fields_[:12]]


class MlsRoundInputs(C.Structure):
    _fields_ = [("actions", vp), ("move_offsets", vp), ("gossip_bits", vp), ("relay_bits", vp), ("philox_seed", C.c_uint64)]


class MlsRoundOutputs(C.Structure):
    _fields_ = [("obs", vp), ("reward", vp), ("active", vp), ("terminated", vp), ("done", vp), ("info", vp),
                ("transitions", vp)]


class MlsNetDesc(C.Structure):
    _fields_ = [("kind", C.c_int32), ("n_nodes", C.c_int32), ("hidden", C.c_int32), ("heads", C.c_int32),
                ("input_dim", C.c_int32), ("pool", C.c_int32), ("precision", C.c_int32), ("head_hidden", C.c_int32)]


WEIGHT_FIELDS = ["enc_w0", "enc_b0", "enc_w1", "enc_b1",
                 "c1_wa", "c1_ba", "c1_wb", "c1_bb", "c1_wc", "c1_bc", "c1_att", "c1_bias",
                 "c2_wa", "c2_ba", "c2_wb", "c2_bb", "c2_wc", "c2_bc", "c2_att", "c2_bias",
                 "q_w0", "q_b0", "q_w1", "q_b1", "q_w2", "q_b2", "v_w0", "v_b0", "v_w1", "v_b1", "v_w2", "v_b2",
                 "out_w", "out_b"]


class MlsNetWeights(C.Structure):
    _fields_ = [(k, vp) for k in WEIGHT_FIELDS]


class MlsForwardArgs(C.Structure):
    _fields_ = [("obs", vp), ("obs_stride", C.c_int64), ("n_graphs", C.c_int32), ("ctrl_mode", C.c_int32),
                ("ctrl_mask", vp), ("q", vp), ("act", vp), ("eps", C.c_float), ("flags", C.c_int32),
                ("philox_seed", C.c_uint64), ("philox_offset", C.c_uint64), ("rand3", vp), ("workspace", vp),
                ("workspace_bytes", C.c_size_t), ("prof_start", vp), ("prof_stop", vp), ("prof_kernel", C.c_int32),
                ("pad2_", C.c_int32), ("philox_offset_dev", vp), ("feature_errors", vp),
                ("graph_ids", vp), ("graph_id_stride", C.c_int32), ("csr_cache_graphs", C.c_int32), ("csr_cache", vp),
                ("philox_row0", C.c_uint64)]


FWD_DISCRETE_FEATURES = 1
FWD_PREPARED = 2
PROF_KERNELS = {None: 0, "proj1": 1, "proj2": 2, "edge1": 3, "edge2": 4, "head0": 5}


EXPORTS = ["mls_version", "mls_last_error", "mls_device_info", "mls_words_per_row", "mls_launch_count", "mls_set_option", "mls_get_option", "mls_env_reset", "mls_env_step",
           "mls_env_info", "mls_dgn_workspace_bytes", "mls_dgn_chunk_graphs", "mls_dgn_forward", "mls_dgn_prepare",
           "mls_dgn_csr_cache_bytes", "mls_dgn_csr_cache_build", "mls_obs_pack", "mls_obs_unpack", "mls_nstep_returns",
           "mls_adam_step", "mls_train_list_capacity", "mls_train_lists", "mls_gatv2_edge_fwd", "mls_gatv2_edge_bwd_blocks",
           "mls_gatv2_edge_bwd", "mls_transformer_edge_fwd", "mls_transformer_edge_bwd", "mls_per_tree_size",
           "mls_per_build", "mls_per_sample", "mls_per_update", "mls_linear_bf16_workspace_bytes", "mls_linear_bf16_fwd",
           "mls_linear_bf16_bwd", "mls_env_reset_sampled", "mls_env_step_sampled", "mls_episode_sample"]
PACKED_NODE_BYTES = 12

_lib = None


class MelissaLibraryError(RuntimeError):
    pass


def lib():
    """The loaded library.  Raises (never falls back) if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MelissaLibraryError(
            f"{LIB_PATH} not found: build it with `python -m melissa_b200.build` "
            "(there is no CPU fallback for the CUDA hot path)")
    L = C.CDLL(LIB_PATH)
    L.mls_version.restype = C.c_int
    L.mls_last_error.restype = C.c_char_p
    L.mls_device_info.argtypes = [C.POINTER(C.c_int32)] * 3
    L.mls_words_per_row.argtypes = [C.c_int]
    L.mls_launch_count.restype = C.c_ulonglong
    L.mls_set_option.argtypes = [C.c_char_p, C.c_int]
    L.mls_get_option.argtypes = [C.c_char_p]
    P = C.POINTER
    L.mls_env_reset.argtypes = [P(MlsEnvDesc), P(MlsEnvState), vp, P(MlsResetTuples), P(MlsRoundInputs),
                                P(MlsRoundOutputs), vp]
    L.mls_env_step.argtypes = [P(MlsEnvDesc), P(MlsEnvState), P(MlsRoundInputs), P(MlsRoundOutputs),
                               P(MlsResetTuples), vp]
    L.mls_env_info.argtypes = [P(MlsEnvDesc), P(MlsEnvState), vp, vp]
    L.mls_env_reset_sampled.argtypes = [P(MlsEnvDesc), P(MlsEnvState), vp, C.c_int32, P(MlsEpisodeSampler),
                                        P(MlsRoundInputs), P(MlsRoundOutputs), vp]
    L.mls_env_step_sampled.argtypes = [P(MlsEnvDesc), P(MlsEnvState), P(MlsRoundInputs), P(MlsRoundOutputs),
                                       P(MlsEpisodeSampler), vp]
    L.mls_episode_sample.argtypes = [P(MlsEpisodeSampler), C.c_int32, vp, vp, C.c_int32, vp, vp, vp, vp, vp]
    L.mls_dgn_workspace_bytes.argtypes = [P(MlsNetDesc), C.c_int32]
    L.mls_dgn_workspace_bytes.restype = C.c_size_t
    L.mls_dgn_chunk_graphs.argtypes = [P(MlsNetDesc), C.c_int32]
    L.mls_dgn_forward.argtypes = [P(MlsNetDesc), P(MlsNetWeights), P(MlsForwardArgs), vp]
    L.mls_dgn_prepare.argtypes = [P(MlsNetDesc), P(MlsNetWeights), C.c_int32, vp, C.c_size_t, vp]
    L.mls_dgn_csr_cache_bytes.argtypes = [P(MlsNetDesc), C.c_int32]
    L.mls_dgn_csr_cache_bytes.restype = C.c_size_t
    L.mls_dgn_csr_cache_build.argtypes = [P(MlsNetDesc), vp, C.c_int64, C.c_int32, vp, C.c_size_t, vp]
    L.mls_obs_pack.argtypes = [vp, C.c_int64, vp, vp, vp]
    L.mls_obs_unpack.argtypes = [vp, vp, vp, C.c_int32, C.c_int64, C.c_int64, vp, vp]
    L.mls_nstep_returns.argtypes = [vp, vp, C.c_int32, C.c_int64, C.c_int32, vp, vp, vp, C.c_int32, C.c_int32, C.c_double,
                                    vp, vp, vp, vp]
    L.mls_adam_step.argtypes = [vp, vp, vp, vp, C.c_int64, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float,
                                C.c_int64, C.c_float, vp]
    L.mls_train_lists.argtypes = [vp, C.c_int64, C.c_int32, C.c_int32, C.c_float, C.c_int32, vp, vp, vp, vp, vp, vp, vp]
    L.mls_gatv2_edge_fwd.argtypes = [vp, C.c_int64, vp, C.c_int64, vp, vp, vp, vp, C.c_int32, C.c_int32, vp, vp, vp]
    L.mls_gatv2_edge_bwd_blocks.argtypes = [C.c_int32]
    L.mls_gatv2_edge_bwd.argtypes = [vp, C.c_int64, vp, C.c_int64, vp, vp, vp, vp, C.c_int32, C.c_int32, vp, vp, vp, vp, vp, vp]
    L.mls_transformer_edge_fwd.argtypes = [vp, vp, C.c_int64, vp, C.c_int64, vp, vp, vp, C.c_int32, C.c_int32, vp, vp, vp]
    L.mls_transformer_edge_bwd.argtypes = [vp, vp, C.c_int64, vp, C.c_int64, vp, vp, vp, C.c_int32, C.c_int32, vp, vp, vp, vp, vp, vp]
    L.mls_per_tree_size.argtypes = [C.c_int64]
    L.mls_per_tree_size.restype = C.c_int64
    L.mls_per_build.argtypes = [vp, C.c_int64, C.c_int32, vp, C.c_double, vp, vp]
    L.mls_per_sample.argtypes = [vp, C.c_int32, C.c_int64, C.c_int32, C.c_int32, C.c_int32, vp, C.c_int32, vp, vp, vp, vp, vp]
    L.mls_per_update.argtypes = [vp, C.c_int32, C.c_int64, C.c_int32, vp, vp, vp, vp, C.c_int32, C.c_double, C.c_double,
                                 vp, vp, vp]
    L.mls_linear_bf16_workspace_bytes.argtypes = [C.c_int64, C.c_int32, C.c_int32]
    L.mls_linear_bf16_workspace_bytes.restype = C.c_size_t
    L.mls_linear_bf16_fwd.argtypes = [vp, C.c_int64, vp, vp, C.c_int64, C.c_int32, C.c_int32, vp, C.c_int64, vp, C.c_size_t, vp]
    L.mls_linear_bf16_bwd.argtypes = [vp, C.c_int64, vp, vp, C.c_int64, C.c_int64, C.c_int32, C.c_int32, vp, C.c_int64, vp, vp, vp,
                                      C.c_size_t, vp]
    for name in EXPORTS:
        getattr(L, name)
    _lib = L
    return L


def check(rc: int):
    if rc == 0:
        return
    msg = lib().mls_last_error().decode("utf-8", "replace")
    if rc == -1:
        raise ValueError(msg)
    raise MelissaLibraryError(f"libmelissa_b200 error {rc}: {msg}")


def words_per_row(n_nodes: int) -> int:
    w = (n_nodes + 31) // 32
    return 1 if w <= 1 else (2 if w <= 2 else (4 if w <= 4 else 8))


def ptr(t):
    """Device pointer of a torch tensor (or None)."""
    if t is None:
        return None
    assert t.is_contiguous(), "tensor must be contiguous"
    return t.data_ptr()


def current_stream_ptr():
    import torch
    return torch.cuda.current_stream().cuda_stream


def set_option(key: str, value: int) -> None:
    check(lib().mls_set_option(key.encode(), int(value)))


def get_option(key: str) -> int:
    return lib().mls_get_option(key.encode())
