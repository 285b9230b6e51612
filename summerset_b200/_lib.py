"""ctypes binding of libsummerset_b200.so (the C ABI in include/summerset_b200.h).

Fails loudly when the shared library is missing: there is no Python / CPU fallback for any
compute entry point.  Build it with `python -m summerset_b200.build` (or __graft_entry__.build()).
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

_PKG = Path(__file__).resolve().parent
LIB_PATH = _PKG / "libsummerset_b200.so"

# error codes (include/summerset_b200.h)
SS_OK = 0
SS_ERR_TOO_FEW_SHARDS = -1
SS_ERR_TOO_MANY_SHARDS = -2
SS_ERR_TOO_FEW_DATA_SHARDS = -3
SS_ERR_TOO_MANY_DATA_SHARDS = -4
SS_ERR_TOO_FEW_PARITY_SHARDS = -5
SS_ERR_TOO_MANY_PARITY_SHARDS = -6
SS_ERR_INCORRECT_SHARD_SIZE = -9
SS_ERR_TOO_FEW_SHARDS_PRESENT = -10
SS_ERR_EMPTY_SHARD = -11
SS_ERR_INVALID_SHARD_FLAGS = -12
SS_ERR_INVALID_INDEX = -13
SS_ERR_INVALID_ARG = -20
SS_ERR_UNSUPPORTED = -21
SS_ERR_OUT_OF_MEMORY = -22
SS_ERR_NO_DEVICE = -30
SS_ERR_CUDA = -31
SS_RS_OUT_PADDED16 = 1

_vp, _u8p, _u32, _u64, _i = C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint64, C.c_int
_sz = C.c_size_t

# name -> (restype, argtypes); every symbol the header declares
SIGNATURES = {
    "ss_version": (_i, []),
    "ss_last_error": (C.c_char_p, []),
    "ss_strerror": (C.c_char_p, [_i]),
    "ss_ctx_create": (_i, [_i, C.POINTER(_vp)]),
    "ss_ctx_create_on_stream": (_i, [_i, _vp, C.POINTER(_vp)]),
    "ss_ctx_destroy": (_i, [_vp]),
    "ss_ctx_sync": (_i, [_vp]),
    "ss_ctx_stream": (_vp, [_vp]),
    "ss_ctx_sm_count": (_i, [_vp]),
    "ss_ctx_launch_count": (_u64, [_vp]),
    "ss_dev_alloc": (_i, [_vp, _sz, C.POINTER(_vp)]),
    "ss_dev_free": (_i, [_vp, _vp]),
    "ss_dev_memset": (_i, [_vp, _vp, _i, _sz]),
    "ss_host_alloc": (_i, [_vp, _sz, C.POINTER(_vp)]),
    "ss_host_alloc_wc": (_i, [_vp, _sz, C.POINTER(_vp)]),
    "ss_host_free": (_i, [_vp, _vp]),
    "ss_copy_h2d": (_i, [_vp, _vp, _vp, _sz]),
    "ss_copy_d2h": (_i, [_vp, _vp, _vp, _sz]),
    "ss_copy_d2d": (_i, [_vp, _vp, _vp, _sz]),
    "ss_ipc_export": (_i, [_vp, _vp, _vp]),
    "ss_ipc_open": (_i, [_vp, _vp, C.POINTER(_vp)]),
    "ss_ipc_close": (_i, [_vp, _vp]),
    "ss_accept_step_replicate_dev": (_i, [_vp, _vp, _u64, _u32, _u64, C.POINTER(_vp), _u64, _vp, _u32, _u32, _vp, _vp, _vp]),
    "ss_follower_ack_dev": (_i, [_vp, _vp, C.POINTER(_vp), _u32, _u64, _vp]),
    "ss_ctx_device_status": (_i, [_vp, C.POINTER(_u32)]),
    "ss_flags_wait_dev": (_i, [_vp, _vp]),
    "ss_flags_signal_dev": (_i, [_vp, _vp]),
    "ss_event_create": (_i, [_vp, C.POINTER(_vp)]),
    "ss_event_destroy": (_i, [_vp, _vp]),
    "ss_event_record": (_i, [_vp, _vp]),
    "ss_event_wait": (_i, [_vp, _vp]),
    "ss_rs_coder_create": (_i, [_vp, _i, _i, C.POINTER(_vp)]),
    "ss_rs_coder_destroy": (_i, [_vp]),
    "ss_rs_data_shard_count": (_i, [_vp]),
    "ss_rs_parity_shard_count": (_i, [_vp]),
    "ss_rs_total_shard_count": (_i, [_vp]),
    "ss_rs_coder_matrix": (_i, [_vp, _u8p]),
    "ss_rs_encode": (_i, [_vp, C.POINTER(_vp), _sz, _sz]),
    "ss_rs_reconstruct": (_i, [_vp, C.POINTER(_vp), _u8p, _sz, _sz]),
    "ss_rs_reconstruct_data": (_i, [_vp, C.POINTER(_vp), _u8p, _sz, _sz]),
    "ss_rs_verify": (_i, [_vp, C.POINTER(_vp), _sz, _sz, C.POINTER(_i)]),
    "ss_rs_encode_batch_dev": (_i, [_vp, _vp, _vp, _vp, _u64, _vp, _u64, _vp, _u32]),
    "ss_rs_encode_uniform_dev": (_i, [_vp, _vp, _u64, _u32, _u64, _vp, _u64, _u64, _u32]),
    "ss_rs_reconstruct_batch_dev": (_i, [_vp, _vp, _u64, _vp, _vp, _vp, _u64, _i, _vp, _u32]),
    "ss_rs_reconstruct_uniform_dev": (_i, [_vp, _vp, _u64, _u64, _u32, _vp, _u64, _i, _vp]),
    "ss_rs_encode_uniform": (_i, [_vp, _vp, _u64, _u32, _u64, _vp, _u64, _u64]),
    "ss_tally_planes_dev": (_i, [_vp, _vp, _u32, _u64, _u32, _vp, _vp]),
    "ss_tally_planes": (_i, [_vp, _vp, _u32, _u64, _u32, _vp, _vp]),
    "ss_tally_masks_dev": (_i, [_vp, _vp, _u32, _u64, _u32, _vp]),
    "ss_ack_ingest_dev": (_i, [_vp, _vp, _vp, _vp, _vp, _u64, _vp, _vp, _vp, _u32, _u64, _vp]),
    "ss_tally_crossword_dev": (_i, [_vp, _vp, _u32, _vp, _u64, _vp, _u32, _u32, _u32, _u32, _u32, _u32, _i, _vp]),
    "ss_raft_commit_scan_dev": (_i, [_vp, _vp, _u32, _u64, _vp, _vp, _vp, _vp, _u32, _u32, _vp, _vp]),
    "ss_crossword_distribute_dev": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _u64, C.POINTER(_vp), _u32]),
    "ss_frame_accept_batch_dev": (_i, [_vp, _vp, _u64, _u32, _u32, _u32, _u32, _u32, _vp, _vp, _u64, _vp, _u64, _vp, _vp]),
    "ss_gossip_plan_dev": (_i, [_vp, _u32, _u32, _u32, _vp, _vp, _vp, _vp, _u32, _u32, _u64, _vp, _vp]),
    "ss_raft_kth_match_dev": (_i, [_vp, _vp, _u32, _u64, _u32, _vp]),
    "ss_prepare_merge_dev": (_i, [_vp, _vp, _vp, _u32, _u64, _vp, _u32, _u32, _u32, _vp, _vp, _vp]),
    "ss_accept_step_fused_dev": (_i, [_vp, _vp, _u64, _u32, _u64, _vp, _u64, _u64, _u32, _vp, _u32, _u32, _vp, _vp]),
    "ss_accept_step_fused": (_i, [_vp, _vp, _u64, _u32, _u64, _vp, _u64, _u64, _vp, _u32, _u32, _vp, _vp]),
    "ss_frame_accept_max_len": (_u64, [_vp, _u32]),
    "ss_frame_accept_pack_dev": (_i, [_vp, _vp, _vp, _u64, _u64, _vp, _u32, _vp, _u32, _vp, _vp, _u64, _vp, _u64, _vp, _vp]),
    "ss_accept_reply_parse_dev": (_i, [_vp, _vp, _u64, _vp, _vp, _vp, _vp, _u64, _u64, _u32, _i, _vp, _vp, _vp, _vp, _vp]),
    "ss_wal_commit_pack_dev": (_i, [_vp, _vp, _vp, _u64, _u32, _vp, _vp, _vp, _u64, _vp]),
    "ss_reconstruct_serve_dev": (_i, [_vp, _vp, _u64, _u64, _u32, _u32, _vp, _vp, _vp, _vp, _vp, _u64, _vp, _vp]),
    "ss_reconstruct_reply_dev": (_i, [_vp, _vp, _u64, _u64, _u32, _u64, _u32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                      _u64, _vp, _vp]),
    "ss_engine_create": (_i, [_vp, _vp, _u64, C.POINTER(_vp)]),
    "ss_engine_destroy": (_i, [_vp]),
    "ss_engine_view_get": (_i, [_vp, _vp]),
    "ss_engine_set_prepared_ballots": (_i, [_vp, _vp]),
    "ss_engine_set_policies": (_i, [_vp, _vp, _u32, _i]),
    "ss_engine_propose": (_i, [_vp, _u32, _vp, _u64, _vp, C.POINTER(_vp)]),
    "ss_engine_ingest": (_i, [_vp, _vp, _vp, _vp, _vp, _u64]),
    "ss_engine_tick": (_i, [_vp, _vp]),
    "ss_engine_raft_append": (_i, [_vp, _vp]),
    "ss_engine_raft_ingest": (_i, [_vp, _vp, _vp, _vp, _u64]),
    "ss_rs_set_variant": (_i, [_vp, _i]),
    "ss_rs_last_kernel": (C.c_char_p, [_vp]),
    "ss_rs_jit_status": (C.c_char_p, [_vp]),
    "ss_jit_selftest": (C.c_long, [_i, _i, C.c_char_p, _sz]),
}


class StepSync(C.Structure):
    """ss_step_sync (include/summerset_b200.h): device-side wait / signal flags of one multi-GPU step call."""
    _fields_ = [("wait_flags", C.c_void_p), ("n_wait", C.c_uint32), ("wait_value", C.c_uint64),
                ("signal_flags", C.POINTER(C.c_void_p)), ("n_signal", C.c_uint32), ("signal_value", C.c_uint64)]


SS_PROTO_MULTIPAXOS, SS_PROTO_RSPAXOS, SS_PROTO_CROSSWORD, SS_PROTO_RAFT, SS_PROTO_CRAFT = range(5)


class FrameSpec(C.Structure):
    """ss_frame_spec"""
    _fields_ = [("kind", C.c_uint32), ("msg_variant", C.c_uint32), ("data_shards", C.c_uint32), ("parity_shards", C.c_uint32),
                ("data_len", C.c_uint32), ("population", C.c_uint32), ("with_assignment", C.c_uint32), ("assign_size", C.c_uint32)]


class EngineConfig(C.Structure):
    """ss_engine_config"""
    _fields_ = [("protocol", C.c_uint32), ("population", C.c_uint32), ("fault_tolerance", C.c_uint32), ("data_len", C.c_uint32),
                ("rs_total_shards", C.c_uint32), ("rs_data_shards", C.c_uint32), ("keep_slots", C.c_uint32),
                ("raft_window", C.c_uint32)]


class EngineView(C.Structure):
    """ss_engine_view"""
    _fields_ = [("n_groups", C.c_uint64), ("population", C.c_uint32), ("threshold", C.c_uint32), ("data_shards", C.c_uint32),
                ("total_shards", C.c_uint32), ("shard_len", C.c_uint32), ("shard_stride", C.c_uint32), ("raft_window", C.c_uint32),
                ("pad0", C.c_uint32), ("plane_stride", C.c_uint64), ("slot_stride", C.c_uint64),
                ("planes", C.c_void_p), ("bal_prepared", C.c_void_p), ("inst_bal", C.c_void_p), ("accepting", C.c_void_p),
                ("committed", C.c_void_p), ("commit_bar", C.c_void_p), ("shards", C.c_void_p), ("policy_idx", C.c_void_p),
                ("match", C.c_void_p), ("next_slot", C.c_void_p), ("last_commit", C.c_void_p), ("log_end", C.c_void_p),
                ("curr_term", C.c_void_p), ("last_snap", C.c_void_p), ("terms", C.c_void_p)]


class SummersetError(RuntimeError):
    """Mirror of `SummersetError(String)` (src/utils/error.rs:6-14): message + the C error code."""

    def __init__(self, code: int, msg: str):
        super().__init__(f"[{code}] {msg}")
        self.code = code
        self.msg = msg


_lib = None


def load() -> C.CDLL:
    """Loads the shared library and binds every declared symbol. Raises if anything is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise ImportError(
            f"{LIB_PATH} is missing: build the CUDA extension first "
            "(`python -m summerset_b200.build`); there is no CPU fallback")
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != SS_OK:
        lib = load()
        msg = lib.ss_last_error().decode("utf-8", "replace")
        raise SummersetError(rc, msg or lib.ss_strerror(rc).decode())
