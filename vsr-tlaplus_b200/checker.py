"""ctypes binding of libvsr_b200.so (include/vsr_b200.h) and the Python mirror of TLC's CLI surface.

TLC reference invocation this mirrors (SURVEY §8b):
    java -cp tla2tools.jar tlc2.TLC [-deadlock] [-depth N] -config VSR.cfg VSR.tla
The BFS itself runs in hand-written CUDA behind ``vsr_bfs``; nothing here computes successors or
fingerprints in Python, and there is no CPU fallback: without the built library importing fails,
without a GPU ``check()`` raises.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass, field
from typing import List, Optional, Sequence, Tuple

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libvsr_b200.so")

VSR_MAX_R, VSR_MAX_V, VSR_MAX_C, VSR_MAX_MSGS = 7, 7, 2, 240
VSR_MAX_LEVELS = 512
VSR_NUM_ACTIONS = 20

ACTION_NAMES = [
    "Initial predicate", "TimerSendSVC", "ReceiveHigherSVC", "ReceiveMatchingSVC", "SendDVC", "ReceiveHigherDVC",
    "ReceiveMatchingDVC", "SendSV", "ReceiveSV", "ReceiveClientRequest", "ReceivePrepareMsg", "ReceivePrepareOkMsg",
    "ExecuteOp", "SendGetState", "ReceiveGetState", "ReceiveNewState", "RestartEmpty", "ReceivesRecoveryMsg",
    "ReceivesRecoveryResponseMsg", "CompleteRecovery",
]
INVARIANT_BITS = {
    "AcknowledgedWriteNotLost": 1,
    "AcknowledgedWritesExistOnMajority": 2,
    "NoLogDivergence": 4,
    "TestInv": 8,
}


class VsrError(RuntimeError):
    def __init__(self, rc: int, msg: str):
        super().__init__(f"[rc {rc}] {msg}")
        self.rc = rc


# ---- struct mirrors of include/vsr_flat.h / include/vsr_b200.h -------------------------------------

class VsrEntry(C.Structure):
    _fields_ = [("view", C.c_uint8), ("operation", C.c_uint8), ("client", C.c_uint8), ("req", C.c_uint8)]


class VsrMsg(C.Structure):
    _fields_ = [
        ("type", C.c_uint8), ("view", C.c_uint8), ("src", C.c_uint8), ("dest", C.c_uint8),
        ("op", C.c_uint8), ("commit", C.c_uint8), ("lnv", C.c_uint8), ("first_op", C.c_uint8),
        ("x", C.c_uint8), ("has_entry", C.c_uint8), ("has_log", C.c_uint8), ("log_lo", C.c_uint8),
        ("log_n", C.c_uint8), ("count", C.c_uint8), ("_pad", C.c_uint8 * 2),
        ("entry", VsrEntry), ("log", VsrEntry * VSR_MAX_V),
    ]


class VsrClientRow(C.Structure):
    _fields_ = [("req", C.c_uint8), ("op", C.c_uint8), ("executed", C.c_uint8), ("_pad", C.c_uint8)]


class VsrReplica(C.Structure):
    _fields_ = [
        ("status", C.c_uint8), ("view", C.c_uint8), ("op", C.c_uint8), ("commit", C.c_uint8),
        ("lnv", C.c_uint8), ("sent_dvc", C.c_uint8), ("sent_sv", C.c_uint8), ("rec_number", C.c_uint8),
        ("log_n", C.c_uint8), ("n_svc", C.c_uint8), ("n_dvc", C.c_uint8), ("n_rec", C.c_uint8),
        ("log", VsrEntry * VSR_MAX_V), ("peer_op", C.c_uint8 * (VSR_MAX_R + 1)),
        ("client_table", VsrClientRow * VSR_MAX_C),
        ("svc_recv", VsrMsg * VSR_MAX_R), ("dvc_recv", VsrMsg * VSR_MAX_R), ("rec_recv", VsrMsg * VSR_MAX_R),
    ]


class VsrFlatState(C.Structure):
    _fields_ = [
        ("R", C.c_uint8), ("C", C.c_uint8), ("V", C.c_uint8), ("aux_svc", C.c_uint8), ("aux_restart", C.c_uint8),
        ("acked", C.c_uint8 * VSR_MAX_V), ("_pad", C.c_uint8), ("n_msgs", C.c_uint16),
        ("rep", VsrReplica * VSR_MAX_R), ("msgs", VsrMsg * VSR_MAX_MSGS),
    ]


class VsrModelInfo(C.Structure):
    _fields_ = [
        ("replica_count", C.c_int32), ("client_count", C.c_int32), ("value_count", C.c_int32),
        ("start_view_on_timer_limit", C.c_int32), ("restart_empty_limit", C.c_int32),
        ("symmetry", C.c_int32), ("view", C.c_int32), ("invariant", C.c_int32),
        ("state_bytes", C.c_int32), ("state_bits", C.c_int32), ("num_candidates", C.c_int32),
        ("spec_verified", C.c_int32), ("spec_hash", C.c_uint64), ("value_names", (C.c_char * 32) * VSR_MAX_V),
        ("check_deadlock", C.c_int32), ("_pad", C.c_int32),
    ]


class VsrRunOpts(C.Structure):
    _fields_ = [
        ("device", C.c_int32), ("check_deadlock", C.c_int32), ("max_depth", C.c_int32),
        ("stop_on_violation", C.c_int32), ("keep_trace", C.c_int32), ("verbose", C.c_int32),
        ("table_capacity", C.c_uint64), ("frontier_capacity", C.c_uint64), ("max_states", C.c_uint64),
        ("max_seconds", C.c_double), ("collect_levels", C.c_int32), ("_reserved0", C.c_int32),
        ("frontier_host_capacity", C.c_uint64), ("checkpoint_path", C.c_char_p), ("recover_path", C.c_char_p),
        ("checkpoint_seconds", C.c_double),
    ]


class VsrStats(C.Structure):
    _fields_ = [
        ("generated", C.c_uint64), ("distinct", C.c_uint64), ("queue", C.c_uint64),
        ("depth", C.c_int32), ("rc", C.c_int32), ("complete", C.c_int32), ("num_levels", C.c_int32),
        ("level_sizes", C.c_uint64 * VSR_MAX_LEVELS), ("level_generated", C.c_uint64 * VSR_MAX_LEVELS),
        ("level_ms", C.c_double * VSR_MAX_LEVELS),
        ("h2_ties", C.c_uint64), ("fp_collisions", C.c_uint64), ("probe_total", C.c_uint64),
        ("kernel_launches", C.c_uint64), ("seconds_total", C.c_double), ("seconds_kernels", C.c_double),
        ("violation_level", C.c_int32), ("trace_len", C.c_int32), ("error_code", C.c_int32), ("violation_mask", C.c_int32),
        ("violation_id", C.c_uint64), ("table_capacity", C.c_uint64), ("frontier_capacity", C.c_uint64),
        ("bytes_table", C.c_uint64), ("bytes_frontier", C.c_uint64),
        ("bytes_h2d", C.c_uint64), ("bytes_d2h", C.c_uint64), ("seconds_setup", C.c_double),
        ("records_sent", C.c_uint64), ("records_received", C.c_uint64), ("seconds_insert", C.c_double),
        ("levels_expanded", C.c_int32), ("_pad", C.c_int32),
    ]


class VsrSimOpts(C.Structure):
    _fields_ = [("device", C.c_int32), ("depth", C.c_int32), ("num_walks", C.c_uint64), ("seed", C.c_uint64),
                ("probe_walks", C.c_uint64), ("probe_out", C.POINTER(C.c_uint64))]


class VsrSimStats(C.Structure):
    _fields_ = [("walks", C.c_uint64), ("steps", C.c_uint64), ("dead_ends", C.c_uint64), ("violating_walk", C.c_uint64),
                ("rc", C.c_int32), ("violation_depth", C.c_int32), ("trace_len", C.c_int32), ("_pad", C.c_int32),
                ("kernel_ms", C.c_double), ("seconds_total", C.c_double)]


class VsrLevelInfo(C.Structure):
    _fields_ = [
        ("new_states", C.c_uint64), ("generated", C.c_uint64), ("frontier_in", C.c_uint64), ("ties", C.c_uint64),
        ("collisions", C.c_uint64), ("violation", C.c_int32), ("deadlock", C.c_int32), ("error_code", C.c_int32),
        ("overflow", C.c_int32), ("violation_id", C.c_uint64), ("deadlock_id", C.c_uint64), ("ms", C.c_double),
        ("ms_insert", C.c_double), ("violation_mask", C.c_int32), ("_pad", C.c_int32),
    ]


# every symbol include/vsr_b200.h declares (tests check the library exports all of them)
EXPORTED_SYMBOLS = [
    "vsr_load", "vsr_load_cfg_text", "vsr_model_create", "vsr_model_free", "vsr_model_info", "vsr_init", "vsr_successors", "vsr_enabled_candidates",
    "vsr_canon", "vsr_fingerprint", "vsr_fingerprint_bytewise", "vsr_aux_key", "vsr_owner_rank", "vsr_invariant", "vsr_unpack", "vsr_pack", "vsr_state_to_tla",
    "vsr_flat_to_tla", "vsr_action_name", "vsr_action_location", "vsr_bfs", "vsr_engine_create", "vsr_engine_destroy",
    "vsr_engine_record_bytes", "vsr_engine_seed_init", "vsr_engine_expand", "vsr_engine_step",
    "vsr_engine_insert_records", "vsr_engine_finish_level", "vsr_engine_frontier_size", "vsr_engine_read_frontier",
    "vsr_engine_trace_record", "vsr_engine_stats", "vsr_engine_reset", "vsr_engine_checkpoint", "vsr_engine_recover", "vsr_engine_lookup", "vsr_engine_last_error", "vsr_engine_collected",
    "vsr_replay_candidates", "vsr_probe_bench", "vsr_simulate", "vsr_walk", "vsr_version",
    "vsr_group_open", "vsr_group_open_local", "vsr_group_close", "vsr_group_barrier", "vsr_group_allgather", "vsr_group_abort",
    "vsr_group_set_timeout", "vsr_group_rank", "vsr_group_world", "vsr_group_last_error",
    "vsr_engine_attach_group", "vsr_engine_attach_staged", "vsr_engine_detach", "vsr_engine_default_inbox_records",
    "vsr_bfs_sharded", "vsr_bfs_multi",
]

_lib = None


def load_library(path: Optional[str] = None) -> C.CDLL:
    """Load libvsr_b200.so.  Fails loudly if the CUDA extension has not been built."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or os.environ.get("VSR_B200_LIB") or LIB_PATH  # VSR_B200_LIB: tuning experiments with a variant build
    if not os.path.exists(p):
        raise VsrError(153, f"{p} not found: build it first (python -c 'import __graft_entry__ as g; g.build()'); "
                            "there is no Python/CPU fallback for the CUDA path")
    lib = C.CDLL(p)
    vp, cp, u64 = C.c_void_p, C.c_char_p, C.c_uint64
    lib.vsr_version.restype = cp
    lib.vsr_load.argtypes = [cp, cp, C.POINTER(vp), cp, C.c_size_t]
    lib.vsr_load_cfg_text.argtypes = [cp, cp, C.POINTER(vp), cp, C.c_size_t]
    lib.vsr_model_create.argtypes = [C.c_int] * 8 + [C.POINTER(vp), cp, C.c_size_t]
    lib.vsr_model_free.argtypes = [vp]
    lib.vsr_model_info.argtypes = [vp, C.POINTER(VsrModelInfo)]
    lib.vsr_init.argtypes = [vp, vp]
    lib.vsr_successors.argtypes = [vp, vp, vp, C.c_size_t, C.POINTER(C.c_uint8), C.POINTER(C.c_uint32)]
    lib.vsr_canon.argtypes = [vp, vp]
    lib.vsr_fingerprint.argtypes = [vp, vp]
    lib.vsr_fingerprint.restype = u64
    lib.vsr_fingerprint_bytewise.argtypes = [vp, vp]
    lib.vsr_fingerprint_bytewise.restype = u64
    lib.vsr_aux_key.argtypes = [vp, vp]
    lib.vsr_owner_rank.argtypes = [u64, C.c_int]
    lib.vsr_aux_key.restype = C.c_uint32
    lib.vsr_invariant.argtypes = [vp, vp]
    lib.vsr_unpack.argtypes = [vp, vp, C.POINTER(VsrFlatState)]
    lib.vsr_pack.argtypes = [vp, C.POINTER(VsrFlatState), vp]
    lib.vsr_state_to_tla.argtypes = [vp, vp, cp, C.c_size_t]
    lib.vsr_flat_to_tla.argtypes = [vp, C.POINTER(VsrFlatState), cp, C.c_size_t]
    lib.vsr_action_name.argtypes = [C.c_int]
    lib.vsr_action_name.restype = cp
    lib.vsr_action_location.argtypes = [vp, C.c_int, cp, C.c_size_t]
    lib.vsr_bfs.argtypes = [vp, C.POINTER(VsrRunOpts), C.POINTER(VsrStats), vp, C.POINTER(C.c_uint8), C.c_size_t]
    lib.vsr_engine_create.argtypes = [vp, C.POINTER(VsrRunOpts), C.c_int, C.c_int, C.POINTER(vp), cp, C.c_size_t]
    lib.vsr_engine_destroy.argtypes = [vp]
    lib.vsr_engine_record_bytes.argtypes = [vp]
    lib.vsr_engine_step.argtypes = [vp, u64, u64, C.c_int, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
    lib.vsr_group_open.argtypes = [cp, C.c_int, C.c_int, C.c_double, C.POINTER(vp), cp, C.c_size_t]
    lib.vsr_group_open_local.argtypes = [C.c_int, C.POINTER(vp)]
    lib.vsr_group_close.argtypes = [vp]
    lib.vsr_group_barrier.argtypes = [vp]
    lib.vsr_group_allgather.argtypes = [vp, vp, C.c_size_t, vp]
    lib.vsr_group_abort.argtypes = [vp]
    lib.vsr_group_set_timeout.argtypes = [vp, C.c_double]
    lib.vsr_group_rank.argtypes = [vp]
    lib.vsr_group_world.argtypes = [vp]
    lib.vsr_group_last_error.argtypes = [vp]
    lib.vsr_group_last_error.restype = cp
    lib.vsr_engine_attach_group.argtypes = [vp, vp, u64]
    lib.vsr_engine_attach_staged.argtypes = [vp, u64, C.POINTER(vp), C.POINTER(vp), C.POINTER(u64)]
    lib.vsr_engine_detach.argtypes = [vp]
    lib.vsr_engine_default_inbox_records.argtypes = [vp]
    lib.vsr_engine_default_inbox_records.restype = u64
    lib.vsr_bfs_sharded.argtypes = [vp, C.POINTER(VsrRunOpts), u64, C.POINTER(VsrStats), C.POINTER(C.c_uint32), C.POINTER(C.c_int), C.c_size_t]
    lib.vsr_bfs_multi.argtypes = [vp, C.POINTER(VsrRunOpts), C.c_int, u64, u64, C.POINTER(VsrStats), vp, C.POINTER(C.c_uint8), C.c_size_t, cp,
                                  C.c_size_t]
    lib.vsr_engine_seed_init.argtypes = [vp]
    lib.vsr_engine_expand.argtypes = [vp]
    lib.vsr_engine_insert_records.argtypes = [vp, vp, u64]
    lib.vsr_engine_finish_level.argtypes = [vp, C.POINTER(VsrLevelInfo)]
    lib.vsr_engine_frontier_size.argtypes = [vp]
    lib.vsr_engine_frontier_size.restype = u64
    lib.vsr_engine_read_frontier.argtypes = [vp, u64, u64, vp]
    lib.vsr_engine_trace_record.argtypes = [vp, u64, C.POINTER(u64), C.POINTER(C.c_uint32)]
    lib.vsr_engine_stats.argtypes = [vp, C.POINTER(VsrStats)]
    lib.vsr_engine_reset.argtypes = [vp]
    lib.vsr_engine_checkpoint.argtypes = [vp, cp, C.POINTER(VsrStats)]
    lib.vsr_engine_recover.argtypes = [vp, cp, C.POINTER(VsrStats)]
    lib.vsr_engine_lookup.argtypes = [vp, vp, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.vsr_engine_last_error.argtypes = [vp]
    lib.vsr_engine_last_error.restype = cp
    lib.vsr_engine_collected.argtypes = [vp, C.c_int, vp, u64]
    lib.vsr_engine_collected.restype = u64
    lib.vsr_replay_candidates.argtypes = [vp, C.POINTER(C.c_uint32), C.c_int, vp, C.POINTER(C.c_uint8), C.c_size_t]
    lib.vsr_simulate.argtypes = [vp, C.POINTER(VsrSimOpts), C.POINTER(VsrSimStats), vp, C.POINTER(C.c_uint8), C.c_size_t]
    lib.vsr_walk.argtypes = [vp, u64, u64, C.c_int, C.POINTER(C.c_uint32), C.POINTER(C.c_int)]
    lib.vsr_probe_bench.argtypes = [C.c_int, u64, u64, C.c_double, C.c_int, C.POINTER(C.c_double)]
    if path is None:
        _lib = lib
    return lib


def cfg_text(replica_count: int, values: Sequence[str], start_view_on_timer_limit: int, client_count: int = 1,
             restart_empty_limit: int = 0, view: bool = True, symmetry: bool = True,
             invariants: Sequence[str] = ("AcknowledgedWriteNotLost",)) -> str:
    """Text of a TLC config for VSR.tla with the given constants (same grammar as the shipped VSR.cfg)."""
    mv = ["Normal", "ViewChange", "Recovering", "RequestMsg", "ReplyMsg", "PrepareMsg", "PrepareOkMsg", "CommitMsg",
          "StartViewChangeMsg", "DoViewChangeMsg", "StartViewMsg", "GetStateMsg", "NewStateMsg", "RecoveryMsg",
          "RecoveryResponseMsg", "Nil"]
    lines = ["CONSTANTS",
             f"    ReplicaCount = {replica_count}",
             f"    ClientCount = {client_count}",
             "    Values = {" + ", ".join(values) + "}",
             f"    StartViewOnTimerLimit = {start_view_on_timer_limit}",
             f"    RestartEmptyLimit = {restart_empty_limit}"]
    lines += [f"    {n} = {n}" for n in mv]
    lines += ["", "INIT Init", "NEXT Next", ""]
    if view:
        lines += ["VIEW view"]
    if symmetry:
        lines += ["SYMMETRY symmValues"]
    if invariants:
        lines += ["", "INVARIANT"] + list(invariants)
    return "\n".join(lines) + "\n"


@dataclass
class CheckResult:
    """What a TLC run reports (SURVEY §5 'Metrics'): the four scalars, the verdict, the trace."""
    rc: int
    generated: int
    distinct: int
    queue: int
    depth: int
    complete: bool
    level_sizes: List[int]
    level_generated: List[int]
    level_ms: List[float]
    h2_ties: int
    fp_collisions: int
    probe_total: int
    kernel_launches: int
    seconds_total: float
    seconds_kernels: float
    violation_level: int
    error_code: int
    table_capacity: int
    frontier_capacity: int
    bytes_h2d: int = 0
    bytes_d2h: int = 0
    seconds_setup: float = 0.0
    violated_invariants: List[str] = field(default_factory=list)  # names of the INVARIANTs the reported state violates
    records_sent: int = 0        # several GPUs: records this rank pushed to peers / drained from its inbox
    records_received: int = 0
    seconds_insert: float = 0.0
    trace: List[Tuple[str, bytes]] = field(default_factory=list)  # (action name, packed state)
    levels: List[bytes] = field(default_factory=list)             # collect_levels: raw states per depth

    @property
    def violated(self) -> bool:
        return self.rc == 12


class ModelChecker:
    """``tlc2.TLC -config VSR.cfg VSR.tla`` for the one spec this repo lowers by hand."""

    def __init__(self, handle: C.c_void_p, lib: C.CDLL):
        self._h = handle
        self._lib = lib
        self.info = VsrModelInfo()
        lib.vsr_model_info(handle, C.byref(self.info))
        self.state_bytes = int(self.info.state_bytes)

    # -- construction ---------------------------------------------------------------------------
    @classmethod
    def from_cfg(cls, cfg_path: str, tla_path: Optional[str] = None) -> "ModelChecker":
        lib = load_library()
        h = C.c_void_p()
        err = C.create_string_buffer(1024)
        rc = lib.vsr_load(cfg_path.encode(), tla_path.encode() if tla_path else None, C.byref(h), err, len(err))
        if rc:
            raise VsrError(rc, err.value.decode())
        return cls(h, lib)

    @classmethod
    def from_cfg_text(cls, text: str, tla_path: Optional[str] = None) -> "ModelChecker":
        lib = load_library()
        h = C.c_void_p()
        err = C.create_string_buffer(1024)
        rc = lib.vsr_load_cfg_text(text.encode(), tla_path.encode() if tla_path else None, C.byref(h), err, len(err))
        if rc:
            raise VsrError(rc, err.value.decode())
        return cls(h, lib)

    @classmethod
    def from_constants(cls, replica_count: int, value_count: int, start_view_on_timer_limit: int, symmetry: bool = True,
                       view: bool = True, invariants: Sequence[str] = ("AcknowledgedWriteNotLost",),
                       client_count: int = 1, restart_empty_limit: int = 0) -> "ModelChecker":
        lib = load_library()
        h = C.c_void_p()
        err = C.create_string_buffer(1024)
        mask = 0
        for n in invariants:
            mask |= INVARIANT_BITS[n]
        rc = lib.vsr_model_create(replica_count, client_count, value_count, start_view_on_timer_limit, restart_empty_limit,
                                  int(symmetry), int(view), mask, C.byref(h), err, len(err))
        if rc:
            raise VsrError(rc, err.value.decode())
        return cls(h, lib)

    def close(self):
        if self._h:
            self._lib.vsr_model_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- single-state operations (host) -----------------------------------------------------------
    def _buf(self, n: int = 1):
        return (C.c_uint8 * (self.state_bytes * n))()

    def init_state(self) -> bytes:
        b = self._buf()
        self._lib.vsr_init(self._h, b)
        return bytes(b)

    def successors(self, state: bytes) -> List[Tuple[bytes, int, int]]:
        cap = 1024
        out = self._buf(cap)
        acts = (C.c_uint8 * cap)()
        mult = (C.c_uint32 * cap)()
        src = (C.c_uint8 * self.state_bytes).from_buffer_copy(state)
        n = self._lib.vsr_successors(self._h, src, out, cap, acts, mult)
        if n < 0:
            raise VsrError(255, f"vsr_successors: state not representable (code {n})")
        raw = bytes(out)
        sb = self.state_bytes
        return [(raw[i * sb:(i + 1) * sb], int(acts[i]), int(mult[i])) for i in range(n)]

    def fingerprint(self, state: bytes) -> int:
        return int(self._lib.vsr_fingerprint(self._h, (C.c_uint8 * self.state_bytes).from_buffer_copy(state)))

    def aux_key(self, state: bytes) -> int:
        return int(self._lib.vsr_aux_key(self._h, (C.c_uint8 * self.state_bytes).from_buffer_copy(state)))

    def invariant(self, state: bytes) -> int:
        return int(self._lib.vsr_invariant(self._h, (C.c_uint8 * self.state_bytes).from_buffer_copy(state)))

    def canon(self, state: bytes) -> bytes:
        b = (C.c_uint8 * self.state_bytes).from_buffer_copy(state)
        rc = self._lib.vsr_canon(self._h, b)
        if rc:
            raise VsrError(255, f"vsr_canon failed ({rc})")
        return bytes(b)

    def unpack(self, state: bytes) -> VsrFlatState:
        f = VsrFlatState()
        rc = self._lib.vsr_unpack(self._h, (C.c_uint8 * self.state_bytes).from_buffer_copy(state), C.byref(f))
        if rc:
            raise VsrError(255, f"vsr_unpack failed ({rc})")
        return f

    def pack(self, flat: VsrFlatState) -> bytes:
        b = self._buf()
        rc = self._lib.vsr_pack(self._h, C.byref(flat), b)
        if rc:
            raise VsrError(255, f"vsr_pack: state not representable in the slot encoding (code {rc})")
        return bytes(b)

    def to_tla(self, state: bytes) -> str:
        buf = C.create_string_buffer(1 << 18)
        n = self._lib.vsr_state_to_tla(self._h, (C.c_uint8 * self.state_bytes).from_buffer_copy(state), buf, len(buf))
        if n < 0:
            raise VsrError(255, "vsr_state_to_tla failed")
        return buf.value.decode()

    def flat_to_tla(self, flat: VsrFlatState) -> str:
        buf = C.create_string_buffer(1 << 18)
        n = self._lib.vsr_flat_to_tla(self._h, C.byref(flat), buf, len(buf))
        if n < 0:
            raise VsrError(255, "vsr_flat_to_tla failed")
        return buf.value.decode()

    def action_location(self, action_id: int) -> str:
        buf = C.create_string_buffer(256)
        self._lib.vsr_action_location(self._h, action_id, buf, len(buf))
        return buf.value.decode()

    def dump_trace_tlc(self, trace: Sequence[Tuple[str, bytes]]) -> str:
        """Text of TLC's `-dumpTrace tlc FILE` for a counterexample (format of state_transfer_violation_trace.txt)."""
        parts = []
        for i, (name, st) in enumerate(trace):
            loc = self.action_location(ACTION_NAMES.index(name))
            parts.append("[\n _TEAction |-> [\n   position |-> %d,\n   name |-> \"%s\",\n   location |-> \"%s\"\n ],\n%s]"
                         % (i + 1, name, loc, self.to_tla(st)))
        return "<<\n" + ",\n".join(parts) + "\n>>"

    # -- the BFS (GPU) ----------------------------------------------------------------------------
    def run_opts(self, deadlock: Optional[bool] = None, max_depth: int = 0, device: int = 0, table_capacity: int = 0,
                 frontier_capacity: int = 0, keep_trace: bool = True, collect_levels: bool = False, max_states: int = 0,
                 max_seconds: float = 0.0, stop_on_violation: bool = True, verbose: bool = False,
                 frontier_host_capacity: int = 0, checkpoint_path: Optional[str] = None, recover_path: Optional[str] = None,
                 checkpoint_seconds: float = 0.0) -> VsrRunOpts:
        """checkpoint_path / recover_path / checkpoint_seconds: TLC's -checkpoint / -recover (a file per rank at level
        boundaries; see include/vsr_b200.h VsrRunOpts)"""
        o = VsrRunOpts()
        o.device = device
        if deadlock is None:  # CHECK_DEADLOCK of the cfg when it has one; otherwise off (VSR.tla has terminal states)
            deadlock = int(self.info.check_deadlock) == 1
        o.check_deadlock = int(deadlock)
        o.max_depth = max_depth
        o.stop_on_violation = int(stop_on_violation)
        o.keep_trace = int(keep_trace)
        o.verbose = int(verbose)
        o.table_capacity = table_capacity
        o.frontier_capacity = frontier_capacity
        o.max_states = max_states
        o.max_seconds = max_seconds
        o.collect_levels = int(collect_levels)
        o.frontier_host_capacity = frontier_host_capacity
        o.checkpoint_path = checkpoint_path.encode() if checkpoint_path else None
        o.recover_path = recover_path.encode() if recover_path else None
        o.checkpoint_seconds = checkpoint_seconds
        return o

    @staticmethod
    def result_from_stats(st: VsrStats, rc: int, trace=None, levels=None) -> CheckResult:
        n = int(st.num_levels)
        return CheckResult(
            rc=rc, generated=int(st.generated), distinct=int(st.distinct), queue=int(st.queue), depth=int(st.depth),
            complete=bool(st.complete), level_sizes=[int(st.level_sizes[i]) for i in range(n)],
            level_generated=[int(st.level_generated[i]) for i in range(n)], level_ms=[float(st.level_ms[i]) for i in range(n)],
            h2_ties=int(st.h2_ties), fp_collisions=int(st.fp_collisions), probe_total=int(st.probe_total),
            kernel_launches=int(st.kernel_launches), seconds_total=float(st.seconds_total),
            seconds_kernels=float(st.seconds_kernels), violation_level=int(st.violation_level), error_code=int(st.error_code),
            table_capacity=int(st.table_capacity), frontier_capacity=int(st.frontier_capacity), bytes_h2d=int(st.bytes_h2d),
            bytes_d2h=int(st.bytes_d2h), seconds_setup=float(st.seconds_setup),
            violated_invariants=[n for n, b in INVARIANT_BITS.items() if int(st.violation_mask) & b],
            records_sent=int(st.records_sent), records_received=int(st.records_received), seconds_insert=float(st.seconds_insert),
            trace=trace or [], levels=levels or [])

    def check(self, **kw) -> CheckResult:
        """One-GPU BFS through the single C-ABI call ``vsr_bfs`` (counterexample included).  With collect_levels=True the
        same loop, ``vsr_bfs_sharded`` on a one-rank engine, runs on an engine kept open to read every level's states back."""
        o = self.run_opts(**kw)
        if o.collect_levels:
            return self._check_collecting_levels(o)
        st = VsrStats()
        cap = 512
        tr = self._buf(cap)
        acts = (C.c_uint8 * cap)()
        rc = self._lib.vsr_bfs(self._h, C.byref(o), C.byref(st), tr, acts, cap)
        if rc == 153:
            raise VsrError(rc, "no usable CUDA device / CUDA failure (the BFS has no CPU fallback), or a checkpoint file could not be read / written")
        return self.result_from_stats(st, rc, self._trace(tr, acts, int(st.trace_len)))

    def _check_collecting_levels(self, o: VsrRunOpts) -> CheckResult:
        lib = self._lib
        e = C.c_void_p()
        err = C.create_string_buffer(512)
        rc = lib.vsr_engine_create(self._h, C.byref(o), 0, 1, C.byref(e), err, len(err))
        if rc:
            raise VsrError(rc, err.value.decode())
        try:
            st = VsrStats()
            cap = 4096
            cands = (C.c_uint32 * cap)()
            n = C.c_int(0)
            rc = lib.vsr_bfs_sharded(e, C.byref(o), 0, C.byref(st), cands, C.byref(n), cap)
            if rc not in (0, 11, 12, 152, 255):
                raise VsrError(rc, lib.vsr_engine_last_error(e).decode())
            levels = []
            sb = self.state_bytes
            for lv in range(1, int(st.num_levels) + 1):
                k = lib.vsr_engine_collected(e, lv, None, 0)
                buf = (C.c_uint8 * (k * sb))()
                lib.vsr_engine_collected(e, lv, buf, k)
                levels.append(bytes(buf))
        finally:
            lib.vsr_engine_destroy(e)
        trace = replay_trace(self, cands[:n.value]) if st.trace_len else []
        if trace:  # as vsr_bfs reports it: the INVARIANT bits the counterexample's last state violates
            st.violation_mask = self.invariant(trace[-1][1])
        return self.result_from_stats(st, rc, trace, levels)

    def _trace(self, buf, acts, n: int) -> List[Tuple[str, bytes]]:
        """the first n (action name, packed state) pairs of a trace buffer the library filled"""
        raw, sb = bytes(buf), self.state_bytes
        return [(ACTION_NAMES[acts[i]], raw[i * sb:(i + 1) * sb]) for i in range(n)]

    def check_multi(self, gpus: int, inbox_records: int = 0, part_states: int = 0, **kw) -> CheckResult:
        """The BFS sharded over `gpus` GPUs from THIS process (one thread per GPU): ``vsr_bfs_multi``, what `vsrmc -gpus N` runs."""
        o = self.run_opts(**kw)
        st = VsrStats()
        cap = 512
        tr = self._buf(cap)
        acts = (C.c_uint8 * cap)()
        err = C.create_string_buffer(512)
        rc = self._lib.vsr_bfs_multi(self._h, C.byref(o), gpus, inbox_records, part_states, C.byref(st), tr, acts, cap, err, len(err))
        if rc in (151, 153):
            raise VsrError(rc, err.value.decode() or "no usable CUDA devices: the BFS has no CPU fallback")
        return self.result_from_stats(st, rc, self._trace(tr, acts, int(st.trace_len)))

    def simulate(self, num_walks: int = 1 << 20, depth: int = 100, seed: int = 1, device: int = 0, probe_walks: int = 0):
        """TLC's `-simulate -depth N`: random behaviours on the GPU.  Returns (VsrSimStats, trace) — the trace is the
        violating behaviour [(action name, packed state)] when rc == 12, else []."""
        o = VsrSimOpts(device=device, depth=depth, num_walks=num_walks, seed=seed)
        probe = (C.c_uint64 * max(2 * probe_walks, 1))()
        if probe_walks:
            o.probe_walks, o.probe_out = probe_walks, probe
        st = VsrSimStats()
        self.last_probe = [(int(probe[2 * i]), int(probe[2 * i + 1])) for i in range(0)]
        cap = max(depth + 1, 2)
        tr = self._buf(cap)
        acts = (C.c_uint8 * cap)()
        rc = self._lib.vsr_simulate(self._h, C.byref(o), C.byref(st), tr, acts, cap)
        if rc == 153:
            raise VsrError(rc, "no usable CUDA device: simulation runs on the GPU only")
        raw, sb = bytes(tr), self.state_bytes
        self.last_probe = [(int(probe[2 * i]), int(probe[2 * i + 1])) for i in range(probe_walks)]  # (fp of last state, transitions)
        return st, [(ACTION_NAMES[acts[i]], raw[i * sb:(i + 1) * sb]) for i in range(int(st.trace_len))]

    def walk(self, seed: int, walk: int, depth: int):
        """the same random walk on the host: (candidate indices, depth of the first violating state or 0)"""
        cands = (C.c_uint32 * max(depth, 1))()
        va = C.c_int()
        n = self._lib.vsr_walk(self._h, seed, walk, depth, cands, C.byref(va))
        return [int(cands[i]) for i in range(n)], int(va.value)


def replay_trace(mc: ModelChecker, cands: Sequence[int]) -> List[Tuple[str, bytes]]:
    """Literal behaviour (fixed value names) from the candidate chain of a counterexample."""
    n = len(cands)
    cap = n + 1
    out = mc._buf(cap)
    acts = (C.c_uint8 * cap)()
    m = mc._lib.vsr_replay_candidates(mc._h, (C.c_uint32 * max(n, 1))(*cands), n, out, acts, cap)
    if m < 0:
        raise VsrError(255, "trace replay failed")
    return mc._trace(out, acts, m)
