"""The BFS on several GPUs of one node (SURVEY §8e): one rank per GPU, the reachable set sharded by the high bits of the
64-bit fingerprint.

Two ways to move a successor to the rank that owns it, both behind the same CUDA kernel (csrc/vsr_gpu.cuh ``push_records``:
the lanes of a batch lay their outgoing records out by destination in shared memory and each run leaves as one TMA bulk
store):

``exchange="p2p"`` (default, what bench.py measures) — the kernel's store goes straight into the owner's inbox over NVLink
    (the inbox is mapped into this process with CUDA IPC) and the owner inserts it at the end of its next launch.  The level
    loop is C++ (``vsr_bfs_sharded``): per step one launch, one 32-byte read-back and one shared-memory all-gather between
    the ranks (``Group``); no collective, no staging copy, no Python on the path.  torch.distributed is only used by the
    caller to agree on the group's name and to time the run.

``exchange="staged"`` — the kernel's store goes into a local staging buffer and this file moves the records with
    torch.distributed (NCCL grouped send/recv over NVLink, or gloo through host memory in tests): ``ShardedBfs``, a
    level loop in Python.  It is the textbook "all-to-all after each wavefront" and the baseline the fused path is
    measured against; it is engine-agnostic so that tests can drive it over gloo with a host engine built from the C ABI's
    single-state functions (tests/host_engine.py) and exercise the N>1 control flow without a GPU.
"""
from __future__ import annotations

import ctypes as C
import os
import time
import uuid
from dataclasses import dataclass, field
from typing import List, Optional, Tuple

import torch
import torch.distributed as dist

from . import checker as ck
from .checker import replay_trace  # noqa: F401  (part of this module's interface: check_sharded, bench.py and the tests use it)

I64_MAX = (1 << 63) - 1
GID_SHIFT = 40             # global state id = rank << 40 | local id (vsr_gpu.cuh make_gid)
ROOT_PARENT = (1 << 44) - 1  # "no parent" (Init): vsr_gpu.cuh ROOT_GID
MAX_WORLD = 8


class Group:
    """The ranks of one job on this node: a shared-memory barrier and small all-gather (csrc/vsr_group.cpp)."""

    def __init__(self, name: str, rank: int, world: int, timeout_s: float = 120.0, lib=None):
        self.lib = lib or ck.load_library()
        self.rank, self.world, self.name = rank, world, name
        self._g = C.c_void_p()
        err = C.create_string_buffer(512)
        rc = self.lib.vsr_group_open(name.encode(), rank, world, float(timeout_s), C.byref(self._g), err, len(err))
        if rc:
            raise ck.VsrError(rc, err.value.decode())

    @classmethod
    def from_torch(cls, pg=None, timeout_s: float = 120.0) -> "Group":
        """every rank of an initialised torch.distributed job calls this: rank 0 picks a fresh name, broadcasts it"""
        rank, world = dist.get_rank(pg), dist.get_world_size(pg)
        box = ["/vsr-b200-%d-%s" % (os.getpid(), uuid.uuid4().hex[:12])] if rank == 0 else [None]
        dist.broadcast_object_list(box, src=0, group=pg)
        return cls(box[0], rank, world, timeout_s)

    def barrier(self):
        if self.lib.vsr_group_barrier(self._g):
            raise ck.VsrError(153, self.lib.vsr_group_last_error(self._g).decode())

    def allgather(self, payload: bytes) -> List[bytes]:
        n = len(payload)
        out = (C.c_uint8 * (n * self.world))()
        src = (C.c_uint8 * max(n, 1)).from_buffer_copy(payload or b"\0")
        if self.lib.vsr_group_allgather(self._g, src, n, out):
            raise ck.VsrError(153, self.lib.vsr_group_last_error(self._g).decode())
        raw = bytes(out)
        return [raw[i * n:(i + 1) * n] for i in range(self.world)]

    def set_timeout(self, seconds: float):
        self.lib.vsr_group_set_timeout(self._g, float(seconds))

    def abort(self):
        self.lib.vsr_group_abort(self._g)

    def close(self):
        if self._g:
            self.lib.vsr_group_close(self._g)
            self._g = None


class _DevMem:
    """a raw device pointer as something torch.as_tensor understands"""

    def __init__(self, ptr: int, nbytes: int):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}


@dataclass
class ShardedResult:
    rc: int = 0
    generated: int = 0
    distinct: int = 0
    queue: int = 0
    depth: int = 0
    complete: bool = False
    level_sizes: List[int] = field(default_factory=list)
    level_generated: List[int] = field(default_factory=list)
    level_ms: List[float] = field(default_factory=list)   # slowest rank's kernel time per level
    h2_ties: int = 0
    fp_collisions: int = 0
    violation_level: int = 0
    violation_gid: int = -1
    seconds: float = 0.0
    kernel_ms_max: float = 0.0       # sum over levels of the slowest rank's kernel time
    insert_ms_max: float = 0.0       # of which launches that only drained records from peers, slowest rank per level
    exchanged_records: int = 0       # records this rank sent
    received_records: int = 0
    # staged pump only: this rank's host wall clock by phase
    phase_seconds: dict = field(default_factory=lambda: {"expand": 0.0, "exchange": 0.0, "finish": 0.0})
    launches: int = 0
    bytes_h2d: int = 0               # host<->device bytes this rank's engine moved (inputs, per-step counters, trace reads)
    bytes_d2h: int = 0
    trace_cands: List[int] = field(default_factory=list)
    trace: List[Tuple[str, bytes]] = field(default_factory=list)
    # check_sharded only: this rank's wall clock of the one-call API by part (engine creation = allocation + clearing the
    # seen-set; attach = inbox allocation + CUDA IPC mapping of the peers; bfs; replay of the counterexample; teardown)
    call_seconds: dict = field(default_factory=dict)


class GpuEngine:
    """The C-ABI engine of one rank, with its exchange attached."""

    def __init__(self, mc: "ck.ModelChecker", rank: int, world: int, device: int = 0, table_capacity: int = 0,
                 frontier_capacity: int = 0, inbox_records: int = 0, keep_trace: bool = True, check_deadlock: bool = False,
                 collect_levels: bool = False, group: Optional[Group] = None, exchange: str = "p2p", frontier_host_capacity: int = 0):
        self.mc, self.rank, self.world = mc, rank, world
        self.lib = mc._lib
        self.dev = torch.device("cuda", device)
        self.exchange = exchange if world > 1 else "none"
        self._opts = mc.run_opts(deadlock=check_deadlock, device=device, table_capacity=table_capacity,
                                 frontier_capacity=frontier_capacity, keep_trace=keep_trace, collect_levels=collect_levels,
                                 frontier_host_capacity=frontier_host_capacity)
        self._e = C.c_void_p()
        err = C.create_string_buffer(512)
        t0 = time.time()
        rc = self.lib.vsr_engine_create(mc._h, C.byref(self._opts), rank, world, C.byref(self._e), err, len(err))
        self.seconds_create = time.time() - t0
        if rc:
            if group is not None:
                group.abort()
            raise ck.VsrError(rc, err.value.decode())
        self.record_bytes = int(self.lib.vsr_engine_record_bytes(self._e))
        self.group = group
        self.inbox_records = 0
        if world > 1 and self.exchange == "p2p":
            if group is None:
                raise ck.VsrError(255, "exchange='p2p' needs a Group")
            t0 = time.time()
            self._ck(self.lib.vsr_engine_attach_group(self._e, group._g, inbox_records))
            self.seconds_attach = time.time() - t0
            self.inbox_records = inbox_records or int(self.lib.vsr_engine_default_inbox_records(self._e))
        elif world > 1:
            stage, inbox, cap = C.c_void_p(), C.c_void_p(), C.c_uint64()
            self._ck(self.lib.vsr_engine_attach_staged(self._e, inbox_records, C.byref(stage), C.byref(inbox), C.byref(cap)))
            self.inbox_records = int(cap.value)
            seg = self.inbox_records * self.record_bytes
            self._stage = torch.as_tensor(_DevMem(stage.value, world * seg), device=self.dev).view(world, seg)
            self._inbox = torch.as_tensor(_DevMem(inbox.value, 2 * world * seg), device=self.dev).view(2, world, seg)

    def _ck(self, rc):
        if rc:
            raise ck.VsrError(rc, self.lib.vsr_engine_last_error(self._e).decode())

    # -- the fused path: the whole BFS in C++ ---------------------------------------------------------
    def run(self, max_depth: int = 0, max_seconds: float = 0.0, max_states: int = 0, stop_on_violation: bool = True,
            want_trace: bool = True, part_states: int = 0, verbose: bool = False, checkpoint_path: Optional[str] = None,
            recover_path: Optional[str] = None, checkpoint_seconds: float = 0.0) -> ShardedResult:
        """checkpoint_path / recover_path: TLC -checkpoint / -recover at level boundaries; with several ranks every rank writes /
        reads ``<path>.rank<r>``, one rank ``<path>`` itself"""
        o = self._opts
        o.max_depth, o.max_seconds, o.max_states = max_depth, max_seconds, max_states
        o.stop_on_violation, o.verbose = int(stop_on_violation), int(verbose)
        o.checkpoint_path = checkpoint_path.encode() if checkpoint_path else None
        o.recover_path = recover_path.encode() if recover_path else None
        o.checkpoint_seconds = checkpoint_seconds
        st = ck.VsrStats()
        cap = 4096
        cands = (C.c_uint32 * cap)()
        n = C.c_int(0)
        rc = self.lib.vsr_bfs_sharded(self._e, C.byref(o), part_states, C.byref(st), cands if want_trace else None, C.byref(n), cap)
        if rc not in (0, 11, 12, 152, 255):
            raise ck.VsrError(rc, self.lib.vsr_engine_last_error(self._e).decode())
        nl, ne = int(st.num_levels), int(st.levels_expanded)
        r = ShardedResult(rc=rc, generated=int(st.generated), distinct=int(st.distinct), queue=int(st.queue), depth=int(st.depth),
                          complete=bool(st.complete), level_sizes=[int(st.level_sizes[i]) for i in range(nl)],
                          level_generated=[int(st.level_generated[i]) for i in range(ne)],
                          level_ms=[float(st.level_ms[i]) for i in range(ne)], h2_ties=int(st.h2_ties),
                          fp_collisions=int(st.fp_collisions), violation_level=int(st.violation_level),
                          violation_gid=int(st.violation_id) if st.violation_level else -1, seconds=float(st.seconds_total),
                          kernel_ms_max=float(st.seconds_kernels) * 1e3, insert_ms_max=float(st.seconds_insert) * 1e3,
                          exchanged_records=int(st.records_sent), received_records=int(st.records_received),
                          launches=int(st.kernel_launches), bytes_h2d=int(st.bytes_h2d), bytes_d2h=int(st.bytes_d2h))
        if want_trace and (rc in (11, 12) or r.violation_level):
            r.trace_cands = [int(cands[i]) for i in range(int(n.value))]
        return r

    # -- the stepwise interface (staged pump, tests) ----------------------------------------------------
    def reset(self):
        self._ck(self.lib.vsr_engine_reset(self._e))

    def seed(self):
        self._ck(self.lib.vsr_engine_seed_init(self._e))

    def expand(self):
        self._ck(self.lib.vsr_engine_expand(self._e))

    def step(self, first: int, count: int, parity: int, drain_counts: Optional[List[int]]) -> List[int]:
        sent = (C.c_uint32 * MAX_WORLD)()
        dc = (C.c_uint32 * MAX_WORLD)(*drain_counts) if drain_counts is not None else None
        self._ck(self.lib.vsr_engine_step(self._e, first, count, parity, dc, sent))
        return [int(sent[i]) for i in range(self.world)]

    def outgoing(self, dest: int, n: int) -> torch.Tensor:
        """the n records the last step produced for rank `dest` (device bytes)"""
        return self._stage[dest, : n * self.record_bytes]

    def incoming_view(self, parity: int, src: int, n: int) -> torch.Tensor:
        """where n records from rank `src` pushed in a step of this parity must land"""
        return self._inbox[parity & 1, src, : n * self.record_bytes]

    def put_incoming(self, parity: int, src: int, data: torch.Tensor, n: int):
        self.incoming_view(parity, src, n).copy_(data.reshape(-1)[: n * self.record_bytes])
        torch.cuda.current_stream(self.dev).synchronize()

    def insert(self, recs: torch.Tensor, n: int):
        if n:
            torch.cuda.current_stream(self.dev).synchronize()
            self._ck(self.lib.vsr_engine_insert_records(self._e, recs.data_ptr(), n))

    def finish(self) -> "ck.VsrLevelInfo":
        li = ck.VsrLevelInfo()
        self._ck(self.lib.vsr_engine_finish_level(self._e, C.byref(li)))
        return li

    def frontier_size(self) -> int:
        return int(self.lib.vsr_engine_frontier_size(self._e))

    def stats(self) -> "ck.VsrStats":
        st = ck.VsrStats()
        self.lib.vsr_engine_stats(self._e, C.byref(st))
        return st

    def trace_record(self, local_id: int) -> Tuple[int, int]:
        parent, cand = C.c_uint64(), C.c_uint32()
        self._ck(self.lib.vsr_engine_trace_record(self._e, local_id, C.byref(parent), C.byref(cand)))
        return int(parent.value), int(cand.value)

    def lookup(self, state: bytes) -> Tuple[int, int]:
        """(depth at which this canonical packed state was first seen on THIS rank's shard or 0, owner rank)"""
        lvl, owner = C.c_int(), C.c_int()
        buf = (C.c_uint8 * self.mc.state_bytes).from_buffer_copy(state)
        self._ck(self.lib.vsr_engine_lookup(self._e, buf, C.byref(lvl), C.byref(owner)))
        return int(lvl.value), int(owner.value)

    def collected(self, level: int) -> bytes:
        n = int(self.lib.vsr_engine_collected(self._e, level, None, 0))
        buf = (C.c_uint8 * max(n * self.mc.state_bytes, 1))()
        if n:
            self.lib.vsr_engine_collected(self._e, level, buf, n)
        return bytes(buf)[: n * self.mc.state_bytes]

    def close(self):
        """collective when a group is attached (the peers' mappings of this rank's inbox are closed before it is freed)"""
        if self._e:
            self._stage = self._inbox = None
            self.lib.vsr_engine_destroy(self._e)
            self._e = None

    def sync(self):
        torch.cuda.synchronize(self.dev)


def check_sharded(mc: "ck.ModelChecker", group: Group, device: int = 0, table_capacity: int = 0, frontier_capacity: int = 0,
                  inbox_records: int = 0, part_states: int = 0, keep_trace: bool = True, check_deadlock: bool = False,
                  **run_kw) -> ShardedResult:
    """One call per rank: engine + inbox + BFS + teardown; on a violation rank 0's result carries the literal trace."""
    eng = GpuEngine(mc, group.rank, group.world, device=device, table_capacity=table_capacity, frontier_capacity=frontier_capacity,
                    inbox_records=inbox_records, keep_trace=keep_trace, check_deadlock=check_deadlock, group=group)
    res = None
    try:
        t0 = time.time()
        res = eng.run(part_states=part_states, **run_kw)
        t1 = time.time()
        if res.trace_cands or res.rc in (11, 12):
            res.trace = replay_trace(mc, res.trace_cands)
        res.call_seconds = {"create": eng.seconds_create, "attach": getattr(eng, "seconds_attach", 0.0), "bfs": t1 - t0, "replay": time.time() - t1}
        return res
    finally:
        t2 = time.time()
        eng.close()
        if res is not None:
            res.call_seconds["teardown"] = time.time() - t2


class ShardedBfs:
    """Level-synchronous BFS over `world` engines with the records moved by torch.distributed (exchange="staged");
    every rank runs this same loop."""

    ROOT_PARENT = ROOT_PARENT

    def __init__(self, engine, rank: int, world: int, group=None, part_states: int = 0):
        self.e, self.rank, self.world, self.group = engine, rank, world, group
        self.part_states = part_states  # frontier states per step and rank (0 = from the engine's inbox size)
        # NCCL moves device tensors; gloo (CPU tests, and ranks that share one GPU in a test) gets host tensors
        self._nccl = world > 1 and dist.get_backend(group) == "nccl"
        self._cdev = getattr(engine, "dev", torch.device("cpu")) if self._nccl else torch.device("cpu")
        self._phase = {"expand": 0.0, "exchange": 0.0, "finish": 0.0}

    # -- collectives (no-ops when world == 1) ---------------------------------------------------
    def _allreduce(self, vals: List[int], op) -> List[int]:
        if self.world == 1:
            return list(vals)
        t = torch.tensor(vals, dtype=torch.int64, device=self._cdev)
        dist.all_reduce(t, op=op, group=self.group)
        return [int(x) for x in t.cpu().tolist()]

    def _reduce_level(self, sums: List[int], mins: List[int], maxs: List[int]):
        """the level's sums, minima and maxima over ranks in ONE collective (an all-gather of a short vector reduced on the host)"""
        if self.world == 1:
            return list(sums), list(mins), list(maxs)
        v = torch.tensor(list(sums) + list(mins) + list(maxs), dtype=torch.int64, device=self._cdev)
        parts = [torch.empty_like(v) for _ in range(self.world)]
        dist.all_gather(parts, v, group=self.group)
        h = torch.stack(parts).cpu()
        ns, nm = len(sums), len(mins)
        return (h[:, :ns].sum(0).tolist(), h[:, ns:ns + nm].min(0).values.tolist(), h[:, ns + nm:].max(0).values.tolist())

    def _exchange(self, sent: List[int], parity: int) -> List[int]:
        """counts all-to-all, then the records: segment d of the staging buffer -> rank d's inbox, half `parity`, segment
        <this rank>.  Returns what this rank received from each peer (the next step's drain counts)."""
        counts = torch.tensor(sent, dtype=torch.int64, device=self._cdev)
        recv_counts = torch.empty_like(counts)
        dist.all_to_all_single(recv_counts, counts, group=self.group)
        rcnt = [int(x) for x in recv_counts.cpu().tolist()]
        cap = getattr(self.e, "inbox_records", 0)
        if cap:  # an overflowing sender has set its overflow flag (the level reduce stops everybody): never move more than fits
            sent = [min(c, cap) for c in sent]
            rcnt = [min(c, cap) for c in rcnt]
        rb = self.e.record_bytes
        if self._nccl:
            ops = []
            for p in range(self.world):
                if p == self.rank:
                    continue
                if rcnt[p]:
                    ops.append(dist.P2POp(dist.irecv, self.e.incoming_view(parity, p, rcnt[p]), p, self.group))
                if sent[p]:
                    ops.append(dist.P2POp(dist.isend, self.e.outgoing(p, sent[p]), p, self.group))
            if ops:
                for w in dist.batch_isend_irecv(ops):
                    w.wait()
            torch.cuda.current_stream(self._cdev).synchronize()
        else:
            parts = [self.e.outgoing(p, sent[p]).to("cpu") if p != self.rank and sent[p] else torch.empty(0, dtype=torch.uint8)
                     for p in range(self.world)]
            inp = torch.cat(parts) if sum(len(x) for x in parts) else torch.empty(0, dtype=torch.uint8)
            out = torch.empty(sum(rcnt[p] for p in range(self.world) if p != self.rank) * rb, dtype=torch.uint8)
            dist.all_to_all_single(out, inp, output_split_sizes=[0 if p == self.rank else rcnt[p] * rb for p in range(self.world)],
                                   input_split_sizes=[len(x) for x in parts], group=self.group)
            off = 0
            for p in range(self.world):
                if p != self.rank and rcnt[p]:
                    self.e.put_incoming(parity, p, out[off:off + rcnt[p] * rb], rcnt[p])
                    off += rcnt[p] * rb
        rcnt[self.rank] = 0
        return rcnt

    # -- the loop -----------------------------------------------------------------------------------
    def run(self, max_depth: int = 0, max_seconds: float = 0.0, max_states: int = 0, stop_on_violation: bool = True,
            want_trace: bool = True) -> ShardedResult:
        r = ShardedResult()
        SUM, MAX = dist.ReduceOp.SUM, dist.ReduceOp.MAX
        t0 = time.time()
        self.e.reset()
        self.e.seed()
        self._phase = r.phase_seconds
        level = 0
        bad_gid, result = -1, 0
        part = self.part_states or max(1024, getattr(self.e, "inbox_records", 1 << 20) * self.world // 8)
        while True:
            tf = time.time()
            li = self.e.finish()
            level += 1
            (new, gen, ties, coll, viol, dead, err, ovf), (vmin, dmin), (kms, ims, fmax) = self._reduce_level(
                [int(li.new_states), int(li.generated), int(li.ties), int(li.collisions), int(li.violation), int(li.deadlock),
                 1 if li.error_code else 0, 1 if li.overflow else 0],
                [(self.rank << GID_SHIFT) | int(li.violation_id) if li.violation else I64_MAX,
                 (self.rank << GID_SHIFT) | int(li.deadlock_id) if li.deadlock else I64_MAX],
                [int(li.ms * 1e6), int(getattr(li, "ms_insert", 0.0) * 1e6), int(self.e.frontier_size())])
            r.kernel_ms_max += kms / 1e6
            r.insert_ms_max += ims / 1e6
            self._phase["finish"] += time.time() - tf
            r.generated += gen
            r.distinct += new
            r.h2_ties += ties
            r.fp_collisions += coll
            if level >= 2:
                r.level_generated.append(gen)
                r.level_ms.append(kms / 1e3)
            if new:
                r.level_sizes.append(new)
            if err:
                result = 255
                break
            if ovf:
                result = 152
                break
            if viol and not r.violation_level:
                r.violation_level, r.violation_gid = level, vmin
                result, bad_gid = 12, vmin
                if stop_on_violation:
                    break
            if dead:
                result, bad_gid = 11, dmin
                break
            if fmax == 0:
                r.complete = True
                break
            if max_depth and level >= max_depth:
                break
            if level >= 254:  # the seen-set tags entries with an 8-bit depth
                result = 152
                break
            if max_states and r.distinct >= max_states:
                break
            if max_seconds:
                (late,) = self._allreduce([1 if time.time() - t0 >= max_seconds else 0], MAX)
                if late:
                    break
            if self.world == 1:
                te = time.time()
                self.e.expand()
                self._phase["expand"] += time.time() - te
                continue
            # the level in steps: step k pushes into half k & 1 and drains what arrived for half (k - 1) & 1
            nparts = max(1, (fmax + part - 1) // part)
            drain = None
            for k in range(nparts + 1):
                if k == nparts and not (drain and any(drain)):
                    break
                te = time.time()
                sent = self.e.step(k * part, part if k < nparts else 0, k & 1, drain)
                self._phase["expand"] += time.time() - te
                if k == nparts:
                    break
                tx = time.time()
                r.exchanged_records += sum(sent)
                drain = self._exchange(sent, k & 1)
                r.received_records += sum(drain)
                self._phase["exchange"] += time.time() - tx
        r.rc = result
        r.depth = len(r.level_sizes)
        (r.queue,) = self._allreduce([0 if r.complete else self.e.frontier_size()], SUM)
        if bad_gid >= 0 and want_trace:
            r.trace_cands = self._walk_trace(bad_gid)
        r.seconds = time.time() - t0
        return r

    def _walk_trace(self, gid: int) -> List[int]:
        """follow (parent, candidate) records across ranks from a state back to Init"""
        cands: List[int] = []
        for _ in range(4096):
            owner = gid >> GID_SHIFT
            buf = torch.zeros(2, dtype=torch.int64, device=self._cdev)
            if owner == self.rank:
                parent, cand = self.e.trace_record(gid & ((1 << GID_SHIFT) - 1))
                buf[0], buf[1] = parent, cand
            if self.world > 1:
                dist.broadcast(buf, src=owner, group=self.group)
            parent, cand = int(buf[0]), int(buf[1])
            if parent == self.ROOT_PARENT:
                break
            cands.append(cand)
            gid = parent
        return cands[::-1]
