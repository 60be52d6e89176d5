/*
 * vsr_shard.cu — the BFS on several GPUs of one node (SURVEY §8e): the reachable set is sharded by the high bits of the
 * 64-bit fingerprint, every rank (one per GPU) owns its shard of the seen-set, of the frontier and of the trace.
 *
 * The exchange is fused into the wavefront kernel: a successor owned by another rank is stored by expand_kernel straight
 * into that rank's inbox over NVLink (the inbox is mapped into this process with CUDA IPC, or is a peer pointer when the
 * ranks are threads of one process), and the owner inserts it at the end of its NEXT launch (drain).  A level is pumped in
 * steps of `part_states` frontier states; step k pushes into inbox half k & 1 while it drains half (k - 1) & 1, so the
 * transfer of one step and the insertion of the previous one overlap its expansion — no collective, no staging copy and no
 * Python on this path.  The host side is this file: per step one launch, one 32-byte read-back, one shared-memory
 * all-gather of the counts (vsr_group.cpp); per level one more all-gather of the level's totals.
 *
 *   vsr_engine_attach_group   allocate the inbox, exchange IPC handles through the group, map the peers
 *   vsr_engine_attach_staged  the same kernel writing into a LOCAL staging buffer, for a host that moves the records with
 *                             a collective instead (dist.ShardedBfs over torch.distributed: NCCL all-to-all, or gloo in tests)
 *   vsr_bfs_sharded           the level loop, called by every rank; all ranks return the same totals.  It is also the loop of
 *                             one GPU: with world 1 there is no group, and one step expands the whole frontier
 *   vsr_bfs                   one GPU: a world-1 engine, vsr_bfs_sharded, the counterexample replayed
 *   vsr_bfs_multi             one process, one thread per GPU (vsrmc -gpus N)
 */
#include <stdlib.h>
#include <unistd.h>

#include <algorithm>
#include <string>
#include <thread>
#include <vector>

#include "vsr_engine.h"

using namespace vsr;

namespace {

struct AttachMsg {
    cudaIpcMemHandle_t handle;
    uint64_t raw;       /* the pointer itself: valid for ranks of the same process */
    int64_t pid;
    int32_t device, ok;
    uint64_t cap;
};
static_assert(sizeof(AttachMsg) <= VSR_GROUP_MSG_BYTES, "all-gather slot");

struct StepMsg {
    uint32_t sent[MAX_WORLD];
    int32_t failed;
};

struct LevelMsg {
    uint64_t new_states, generated, ties, collisions, frontier, viol_id, dead_id, sent, received;
    double ms, ms_insert;
    int32_t violation, deadlock, error_code, overflow, late, failed, ckpt, _pad;
};
static_assert(sizeof(LevelMsg) <= VSR_GROUP_MSG_BYTES, "all-gather slot");

struct WalkMsg {
    uint64_t parent;
    uint32_t cand, ok;
};

int set_error(VsrEngine* e, const char* fmt, const char* a = "") {
    snprintf(e->last_error, sizeof e->last_error, fmt, a);
    return VSR_RC_SYSTEM;
}

} // namespace

extern "C" {

int vsr_engine_detach(VsrEngine* e) {
    if (!e) return 0;
    cudaSetDevice(e->device);
    if (e->stream) cudaStreamSynchronize(e->stream);
    if (e->group && e->inbox) vsr_group_barrier(e->group); /* nobody may still be storing into an inbox that is about to go */
    for (int r = 0; r < MAX_WORLD; r++) {
        if (e->peer_inbox[r] && e->peer_is_ipc[r]) cudaIpcCloseMemHandle(e->peer_inbox[r]);
        e->peer_inbox[r] = nullptr;
        e->peer_is_ipc[r] = false;
    }
    if (e->group && e->inbox) vsr_group_barrier(e->group); /* every mapping of my inbox is closed before it is freed */
    if (e->inbox) cudaFree(e->inbox);
    if (e->stage) cudaFree(e->stage);
    e->inbox = e->stage = nullptr;
    e->inbox_cap = 0;
    e->group = nullptr;
    return 0;
}

uint64_t vsr_engine_default_inbox_records(const VsrEngine* e) {
    /* a step of S frontier states per rank pushes about S * (successor records per state) / world records into each peer
       segment.  frontier capacity / (2 x world) records per segment, at most 2^25 / world: the inbox (2 halves x world
       segments) stays a fraction of the frontier's memory, steps are still hundreds of thousands to millions of states (the
       per-step host round trip — launch, 32-byte read-back, shared-memory all-gather: ~50 us — stays a few per cent), and what
       every peer has to map over CUDA IPC when the exchange is attached stays small: with 8 ranks mapping 7 inboxes of 2.7 GB
       (21 GB for the README constants) was most of the one-call API's 0.9 s around an 0.08 s BFS */
    const uint64_t w = (uint64_t)(e->world > 1 ? e->world : 1);
    uint64_t cap = e->frontier_cap / (2 * w);
    if (cap > (1ull << 25) / w) cap = (1ull << 25) / w;
    if (cap < 4096) cap = 4096;
    return cap;
}

static int alloc_inbox(VsrEngine* e, uint64_t inbox_records) {
    if (e->world < 2) return set_error(e, "an exchange needs world > 1");
    if (e->inbox) return set_error(e, "the engine already has an exchange attached");
    if (!inbox_records) inbox_records = vsr_engine_default_inbox_records(e);
    if (inbox_records > 0xFFFFFF00ull) inbox_records = 0xFFFFFF00ull; /* 32-bit slot counters */
    CK(cudaSetDevice(e->device));
    const uint64_t bytes = 2ull * e->world * inbox_records * (uint64_t)e->g->rec_bytes;
    /* plain cudaMalloc: memory from the stream-ordered pool cannot be exported with cudaIpcGetMemHandle */
    CK(cudaMalloc((void**)&e->inbox, bytes));
    e->inbox_cap = inbox_records;
    return 0;
}

int vsr_engine_attach_group(VsrEngine* e, VsrGroup* g, uint64_t inbox_records) {
    if (!e || !g) return VSR_RC_ERROR;
    if (g->world != e->world || g->rank != e->rank) return set_error(e, "group and engine disagree on rank / world");
    AttachMsg mine;
    memset(&mine, 0, sizeof mine);
    int rc = alloc_inbox(e, inbox_records);
    mine.ok = rc == 0;
    mine.pid = (int64_t)getpid();
    mine.device = e->device;
    if (!rc) {
        mine.raw = (uint64_t)(uintptr_t)e->inbox;
        mine.cap = e->inbox_cap;
        if (cudaIpcGetMemHandle(&mine.handle, e->inbox) != cudaSuccess) { /* ranks of other processes will report it */
            cudaGetLastError();
            memset(&mine.handle, 0, sizeof mine.handle);
        }
    }
    AttachMsg all[MAX_WORLD];
    if (vsr_group_allgather(g, &mine, sizeof mine, all)) return set_error(e, "attach: %s", g->last_error);
    e->group = g;
    std::string problem;
    for (int r = 0; r < e->world && problem.empty(); r++) {
        if (!all[r].ok) problem = "rank " + std::to_string(r) + " could not allocate its inbox";
        else if (all[r].cap != all[e->rank].cap) problem = "ranks disagree on the inbox size";
    }
    for (int r = 0; r < e->world && problem.empty(); r++) {
        if (r == e->rank) { e->peer_inbox[r] = e->inbox; continue; }
        if (all[r].pid == mine.pid) { /* same process (one thread per GPU): the pointer is valid here once peer access is on */
            if (all[r].device != e->device) {
                int can = 0;
                cudaDeviceCanAccessPeer(&can, e->device, all[r].device);
                if (!can) { problem = "device " + std::to_string(e->device) + " cannot access device " + std::to_string(all[r].device) + " (no P2P)"; break; }
                cudaError_t ce = cudaDeviceEnablePeerAccess(all[r].device, 0);
                if (ce != cudaSuccess && ce != cudaErrorPeerAccessAlreadyEnabled) { problem = std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(ce); break; }
                cudaGetLastError();
            }
            e->peer_inbox[r] = (uint8_t*)(uintptr_t)all[r].raw;
        } else {
            void* p = nullptr;
            cudaError_t ce = cudaIpcOpenMemHandle(&p, all[r].handle, cudaIpcMemLazyEnablePeerAccess);
            if (ce != cudaSuccess) { cudaGetLastError(); problem = std::string("cudaIpcOpenMemHandle(rank ") + std::to_string(r) + "): " + cudaGetErrorString(ce); break; }
            e->peer_inbox[r] = (uint8_t*)p;
            e->peer_is_ipc[r] = true;
        }
    }
    /* agree on the outcome: a rank that could not map a peer must not leave the others waiting in the first step */
    StepMsg v, vs[MAX_WORLD];
    memset(&v, 0, sizeof v);
    v.failed = problem.empty() ? 0 : 1;
    if (vsr_group_allgather(g, &v, sizeof v, vs)) return set_error(e, "attach: %s", g->last_error);
    int bad = 0;
    for (int r = 0; r < e->world; r++) bad |= vs[r].failed;
    if (bad) {
        if (problem.empty()) problem = "another rank could not map its peers";
        const std::string msg = problem; /* detach clears nothing of last_error, but keep a copy anyway */
        vsr_engine_detach(e);
        return set_error(e, "exchange over peer memory unavailable: %s", msg.c_str());
    }
    return 0;
}

int vsr_engine_attach_staged(VsrEngine* e, uint64_t inbox_records, void** stage_out, void** inbox_out, uint64_t* cap_out) {
    if (!e) return VSR_RC_ERROR;
    int rc = alloc_inbox(e, inbox_records);
    if (rc) return rc;
    CK(cudaMalloc((void**)&e->stage, (uint64_t)e->world * e->inbox_cap * (uint64_t)e->g->rec_bytes));
    if (stage_out) *stage_out = e->stage;
    if (inbox_out) *inbox_out = e->inbox;
    if (cap_out) *cap_out = e->inbox_cap;
    return 0;
}

/* The level loop on every rank of the group, or on a world-1 engine without one.  All ranks take every decision from the
   same all-gathered numbers, so they leave the loop together and report the same totals.  trace_cands / trace_len: the
   candidate chain from Init to the violating (or deadlocked) state, walked across ranks; replay it with
   vsr_replay_candidates.  *stats is written only when the search reaches a verdict, not when it fails (CUDA, checkpoint). */
int vsr_bfs_sharded(VsrEngine* e, const VsrRunOpts* opts, uint64_t part_states, VsrStats* stats, uint32_t* trace_cands, int* trace_len, size_t trace_cap) {
    if (!e || !opts || !stats) return VSR_RC_ERROR;
    if (trace_len) *trace_len = 0;
    VsrGroup* g = e->group;
    if (e->world > 1 && (!g || !e->inbox || e->stage)) return set_error(e, "vsr_bfs_sharded needs vsr_engine_attach_group first");
    const int W = e->world, me = e->rank;
    const double t0 = now_s();
    /* a step of S states per rank fills each peer segment with about S * (successor records per state) / W records.  The
       fan-out is measured, not assumed (2.7 per state on the shipped VSR.cfg, 16 with five replicas): each level's steps are
       sized from the previous level's ratio with a factor of two to spare (an overflow is detected, never silent) */
    const bool auto_part = part_states == 0 || W == 1; /* one rank: no inbox, one step expands the whole frontier */
    double fanout = 16.0, seg_ratio = 0;
    uint64_t prev_frontier_total = 0;
    VsrStats tot;
    memset(&tot, 0, sizeof tot);
    int result = 0, level = 0;
    bool complete = false, bounded = false;
    uint64_t bad_gid = ~0ull;
    double kernel_ms = 0, insert_ms = 0;
    /* checkpoints: every rank writes / reads <path>.rank<r> at the same level boundary (rank 0's clock decides when); one
       rank uses <path> itself */
    const std::string rank_suffix = W > 1 ? ".rank" + std::to_string(me) : std::string();
    const std::string ckpt_path = opts->checkpoint_path ? opts->checkpoint_path + rank_suffix : std::string();
    double last_ckpt = now_s();
    bool resumed = false;
    int rc;
    if (opts->recover_path) {
        rc = vsr_engine_recover(e, (opts->recover_path + rank_suffix).c_str(), &tot);
        if (!rc) {
            resumed = true;
            level = e->level - 1; /* the loop's first pass stands at the checkpoint's level boundary without finishing a level */
            kernel_ms = tot.seconds_kernels * 1e3;
            insert_ms = tot.seconds_insert * 1e3;
            if (tot.violation_level) { result = VSR_RC_VIOLATION; bad_gid = tot.violation_id; }
        }
    } else {
        rc = vsr_engine_reset(e);
        if (!rc) rc = vsr_engine_seed_init(e);
    }
    auto fail_all = [&](int code) { /* tell the others (they are, or will be, in a barrier) and leave */
        if (g) vsr_group_abort(g);
        return code;
    };
    if (rc) return fail_all(rc);
    std::vector<LevelMsg> all(W);
    int step_rc = 0; /* a failure inside the level's steps travels to everybody in the level's all-gather */
    for (;;) {
        VsrLevelInfo li;
        memset(&li, 0, sizeof li);
        if (!resumed) rc = vsr_engine_finish_level(e, &li);
        level++;
        LevelMsg mine;
        memset(&mine, 0, sizeof mine);
        mine.failed = step_rc ? step_rc : rc;
        mine.new_states = li.new_states; mine.generated = li.generated; mine.ties = li.ties; mine.collisions = li.collisions;
        mine.frontier = e->n_cur;
        mine.violation = li.violation; mine.deadlock = li.deadlock; mine.error_code = li.error_code; mine.overflow = li.overflow;
        mine.viol_id = li.violation ? make_gid(me, li.violation_id) : ~0ull;
        mine.dead_id = li.deadlock ? make_gid(me, li.deadlock_id) : ~0ull;
        mine.ms = li.ms; mine.ms_insert = li.ms_insert;
        mine.late = opts->max_seconds > 0 && now_s() - t0 >= opts->max_seconds;
        mine.ckpt = !ckpt_path.empty() && now_s() - last_ckpt >= opts->checkpoint_seconds;
        if (W > 1) {
            if (vsr_group_allgather(g, &mine, sizeof mine, all.data())) return set_error(e, "%s", g->last_error);
        } else all[0] = mine;
        uint64_t n_new = 0, n_gen = 0, max_frontier = 0, vmin = ~0ull, dmin = ~0ull;
        int viol = 0, dead = 0, err = 0, ovf = 0, failed = 0;
        double ms = 0, msi = 0;
        for (int r = 0; r < W; r++) {
            n_new += all[r].new_states; n_gen += all[r].generated;
            tot.h2_ties += all[r].ties; tot.fp_collisions += all[r].collisions;
            max_frontier = std::max(max_frontier, all[r].frontier);
            viol |= all[r].violation; dead |= all[r].deadlock;
            if (all[r].error_code && !err) err = all[r].error_code;
            if (all[r].overflow && !ovf) ovf = all[r].overflow;
            if (all[r].failed && !failed) failed = all[r].failed;
            vmin = std::min(vmin, all[r].viol_id); dmin = std::min(dmin, all[r].dead_id);
            ms = std::max(ms, all[r].ms); msi = std::max(msi, all[r].ms_insert);
        }
        if (failed) { rc = failed; break; }
        kernel_ms += ms;
        insert_ms += msi;
        tot.generated += n_gen;
        tot.distinct += n_new;
        const bool boundary_only = resumed; /* first pass after a recovery: stands at the checkpoint's level boundary */
        if (resumed) { /* the totals, level tables and verdicts up to this boundary came with the checkpoint */
            resumed = false;
        } else if (level >= 2 && level - 2 < VSR_MAX_LEVELS) {
            tot.level_generated[level - 2] = n_gen;
            tot.level_ms[level - 2] = ms; /* slowest rank */
            tot.levels_expanded = level - 1;
        }
        if (n_new && level - 1 < VSR_MAX_LEVELS) {
            tot.level_sizes[level - 1] = n_new;
            tot.num_levels = level;
        }
        if (opts->verbose && me == 0 && level >= 2 && !boundary_only) {
            fprintf(stderr, "depth %3d: %12llu new  %12llu generated  %8.3f ms", level, (unsigned long long)n_new, (unsigned long long)n_gen, ms);
            if (W > 1) fprintf(stderr, " (slowest of %d GPUs)", W);
            fprintf(stderr, "\n");
        }
        if (err) { result = VSR_RC_ERROR; tot.error_code = err; break; }
        if (ovf) { result = VSR_RC_TOO_LARGE; break; }
        if (viol && !tot.violation_level) {
            tot.violation_level = level;
            tot.violation_id = vmin;
            result = VSR_RC_VIOLATION;
            bad_gid = vmin;
            if (opts->stop_on_violation) break;
        }
        if (dead) { result = VSR_RC_DEADLOCK; bad_gid = dmin; break; }
        if (max_frontier == 0) { complete = true; break; }
        if (opts->max_depth && level >= opts->max_depth) { bounded = true; break; }
        if (opts->max_states && tot.distinct >= opts->max_states) { bounded = true; break; }
        if (all[0].late) { bounded = true; break; } /* rank 0's clock decides for everybody */
        if (level >= 254) { result = VSR_RC_TOO_LARGE; break; } /* 8-bit level tag in the seen-set */
        if (all[0].ckpt) { /* TLC -checkpoint: nothing is in flight at a level boundary, every rank saves its shard */
            tot.seconds_kernels = kernel_ms * 1e-3;
            tot.seconds_insert = insert_ms * 1e-3;
            step_rc = vsr_engine_checkpoint(e, ckpt_path.c_str(), &tot); /* a failure travels to everybody in the next all-gather */
            last_ckpt = now_s();
            if (opts->verbose && me == 0 && !step_rc)
                fprintf(stderr, "Checkpointing of run %s%s completed (depth %d, %llu distinct states).\n", opts->checkpoint_path, W > 1 ? ".rank*" : "", level,
                        (unsigned long long)tot.distinct);
        }
        /* ---- the next level, in steps: step k expands part k and pushes into inbox half k & 1, and drains what the
           peers pushed here in step k - 1; one more launch drains the last part's records */
        if (auto_part) {
            if (prev_frontier_total && level >= 4) fanout = std::max(4.0, 2.0 * (double)n_gen / (double)prev_frontier_total);
            /* records per expanded state into ONE (sender, owner) segment: twice the average, or twice the fullest segment
               the last level's steps measured — whichever is larger (owner_of spreads the owners evenly, but the inbox must
               hold whatever distribution a model produces) */
            double per_state = fanout / W;
            if (seg_ratio > 0) per_state = std::max(per_state, 2.0 * seg_ratio);
            part_states = e->inbox_cap ? std::max<uint64_t>(1024, (uint64_t)((double)e->inbox_cap / per_state)) : ~0ull;
        }
        prev_frontier_total = 0;
        for (int r = 0; r < W; r++) prev_frontier_total += all[r].frontier;
        uint32_t drain_counts[MAX_WORLD] = {0};
        bool have_drain = false;
        StepMsg sm, sms[MAX_WORLD];
        double level_ratio = 0;
        uint64_t first = 0;
        for (uint64_t k = 0; !step_rc; k++) {
            const bool expanding = first < max_frontier; /* some rank still has frontier states from `first` on */
            if (!expanding && (W == 1 || !have_drain)) break;
            memset(&sm, 0, sizeof sm);
            const uint64_t count = (expanding && first < e->n_cur) ? std::min(part_states, e->n_cur - first) : 0;
            sm.failed = vsr_engine_step(e, first, count, (int)(k & 1), have_drain ? drain_counts : nullptr, sm.sent);
            if (W == 1 || !expanding) { /* the last launch only drains: nothing was pushed, the level's all-gather follows */
                step_rc = sm.failed;
                break;
            }
            if (vsr_group_allgather(g, &sm, sizeof sm, sms)) return set_error(e, "%s", g->last_error);
            have_drain = false;
            for (int r = 0; r < W; r++) {
                if (sms[r].failed && !step_rc) step_rc = sms[r].failed;
                drain_counts[r] = r == me ? 0 : sms[r].sent[me];
                have_drain |= drain_counts[r] != 0;
            }
            /* what this step really put into the fullest segment, per expanded state (every rank sees the whole matrix and
               every rank's frontier size, so all take the same decision); the next step is sized from it */
            uint64_t next_part = part_states;
            if (auto_part) {
                for (int sr = 0; sr < W; sr++) {
                    const uint64_t cnt = all[sr].frontier > first ? std::min(part_states, all[sr].frontier - first) : 0;
                    if (cnt < 4096) continue;
                    for (int d = 0; d < W; d++)
                        if (d != sr) level_ratio = std::max(level_ratio, (double)sms[sr].sent[d] / (double)cnt);
                }
                if (level_ratio > 0) {
                    const double per_state = std::max(fanout / W, 2.0 * level_ratio);
                    next_part = std::max<uint64_t>(1024, (uint64_t)((double)e->inbox_cap / per_state));
                }
            }
            first = part_states >= max_frontier - first ? max_frontier : first + part_states;
            part_states = next_part;
        }
        if (level_ratio > 0) seg_ratio = level_ratio;
    }
    if (rc) {
        fail_all(rc);
        return rc;
    }
    if (bounded && !ckpt_path.empty()) { /* a run that stops on a bound leaves a checkpoint to continue from */
        tot.seconds_kernels = kernel_ms * 1e-3;
        tot.seconds_insert = insert_ms * 1e-3;
        int crc = vsr_engine_checkpoint(e, ckpt_path.c_str(), &tot), crcs[MAX_WORLD];
        if (W > 1) {
            if (vsr_group_allgather(g, &crc, sizeof crc, crcs)) return set_error(e, "%s", g->last_error);
            for (int r = 0; r < W; r++)
                if (crcs[r] && !crc) crc = crcs[r];
        }
        if (crc) return crc;
    }
    tot.rc = result;
    tot.complete = complete ? 1 : 0;
    tot.depth = tot.num_levels;
    tot.seconds_kernels = kernel_ms * 1e-3;
    /* queue: states left unexplored */
    {
        uint64_t q = complete ? 0 : e->n_cur, qs[MAX_WORLD];
        if (W > 1) {
            if (vsr_group_allgather(g, &q, sizeof q, qs)) return set_error(e, "%s", g->last_error);
            q = 0;
            for (int r = 0; r < W; r++) q += qs[r];
        }
        tot.queue = q;
    }
    /* counterexample: follow (parent, candidate) records across ranks back to Init */
    if (bad_gid != ~0ull && trace_cands && e->trace && opts->keep_trace) {
        std::vector<uint32_t> cands;
        uint64_t gid = bad_gid;
        for (int guard = 0; guard < 4096; guard++) {
            const int owner = (int)(gid >> 40);
            WalkMsg wm, wms[MAX_WORLD];
            memset(&wm, 0, sizeof wm);
            if (owner == me) {
                uint64_t parent = 0;
                uint32_t cand = 0;
                wm.ok = vsr_engine_trace_record(e, gid & ((1ull << 40) - 1), &parent, &cand) == 0;
                wm.parent = parent;
                wm.cand = cand;
            }
            if (W > 1) {
                if (vsr_group_allgather(g, &wm, sizeof wm, wms)) return set_error(e, "%s", g->last_error);
                wm = wms[owner < W ? owner : 0];
            }
            if (!wm.ok) break;
            if (wm.parent == ROOT_GID) break;
            cands.push_back(wm.cand);
            gid = wm.parent;
        }
        std::reverse(cands.begin(), cands.end());
        const size_t n = std::min(cands.size(), trace_cap);
        memcpy(trace_cands, cands.data(), n * sizeof(uint32_t));
        if (trace_len) *trace_len = (int)n;
        tot.trace_len = (int)n + 1;
    }
    tot.kernel_launches = e->st.kernel_launches;
    tot.probe_total = e->st.probe_total;
    tot.table_capacity = e->st.table_capacity;
    tot.frontier_capacity = e->st.frontier_capacity;
    tot.bytes_table = e->st.bytes_table;
    tot.bytes_frontier = e->st.bytes_frontier;
    tot.bytes_h2d = e->st.bytes_h2d;
    tot.bytes_d2h = e->st.bytes_d2h;
    tot.records_sent = e->records_sent;
    tot.records_received = e->records_received;
    tot.seconds_insert = insert_ms * 1e-3;
    tot.seconds_total = now_s() - t0;
    *stats = tot;
    return result;
}

/* the literal counterexample of a finished search from the candidate chain vsr_bfs_sharded walked (it set stats->trace_len
   when it walked one): its length and the INVARIANT bits its last state violates */
static void replay_counterexample(const VsrModel* m, const uint32_t* cands, int n, VsrStats* stats, void* trace_out, uint8_t* trace_actions,
                                  size_t trace_cap) {
    const int len = trace_out && stats->trace_len > 0 ? vsr_replay_candidates(m, cands, n, trace_out, trace_actions, trace_cap) : 0;
    stats->trace_len = len > 0 ? len : 0;
    if (len > 0) stats->violation_mask = m->ops->invariant(&m->run, (const uint32_t*)((const uint8_t*)trace_out + (size_t)(len - 1) * m->ops->bytes));
}

int vsr_bfs(const VsrModel* m, const VsrRunOpts* opts, VsrStats* stats, void* trace_out, uint8_t* trace_actions, size_t trace_cap) {
    if (!m || !opts || !stats) return VSR_RC_ERROR;
    const double t0 = now_s();
    memset(stats, 0, sizeof *stats);
    VsrEngine* e = nullptr;
    char err[256];
    int rc = vsr_engine_create(m, opts, 0, 1, &e, err, sizeof err);
    if (rc) {
        stats->rc = rc;
        if (opts->verbose) fprintf(stderr, "vsr_bfs: %s\n", err);
        return rc;
    }
    const double t_setup = now_s() - t0;
    std::vector<uint32_t> cands(4096);
    int n = 0;
    rc = vsr_bfs_sharded(e, opts, 0, stats, trace_out ? cands.data() : nullptr, &n, cands.size());
    if (stats->rc != rc) { /* failed before a verdict: *stats is still all zero */
        stats->rc = rc;
        if (opts->verbose) fprintf(stderr, "vsr_bfs: %s\n", e->last_error);
    } else {
        replay_counterexample(m, cands.data(), n, stats, trace_out, trace_actions, trace_cap);
        stats->seconds_setup = t_setup;
        stats->seconds_total = now_s() - t0;
    }
    vsr_engine_destroy(e);
    return rc;
}

/* vsrmc -gpus N: one process, one thread per GPU; devices opts->device .. opts->device + ngpus - 1 */
int vsr_bfs_multi(const VsrModel* m, const VsrRunOpts* opts, int ngpus, uint64_t inbox_records, uint64_t part_states, VsrStats* stats, void* trace_out,
                  uint8_t* trace_actions, size_t trace_cap, char* err, size_t errcap) {
    if (!m || !opts || !stats) return VSR_RC_ERROR;
    if (ngpus == 1) return vsr_bfs(m, opts, stats, trace_out, trace_actions, trace_cap);
    if (ngpus < 1 || ngpus > MAX_WORLD || (ngpus & (ngpus - 1))) {
        if (err && errcap) snprintf(err, errcap, "-gpus must be 1, 2, 4 or 8");
        return VSR_RC_CONFIG_ERROR;
    }
    const char* one = getenv("VSR_B200_MULTI_ONE_DEVICE"); /* test hook: every rank on opts->device (a one-GPU box) */
    const bool one_device = one && one[0] == '1';
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < opts->device + (one_device ? 1 : ngpus)) {
        if (err && errcap) snprintf(err, errcap, "%d GPUs requested from device %d on, %d visible: the BFS runs on GPUs only, there is no CPU fallback", ngpus, opts->device, ndev);
        return VSR_RC_SYSTEM;
    }
    const double t0 = now_s();
    VsrGroup* groups[MAX_WORLD] = {nullptr};
    if (vsr_group_open_local(ngpus, groups)) return VSR_RC_SYSTEM;
    std::vector<VsrStats> st(ngpus);
    std::vector<int> rcs(ngpus, 0), lens(ngpus, 0);
    std::vector<std::vector<uint32_t>> cands(ngpus, std::vector<uint32_t>(4096));
    std::vector<std::string> errors(ngpus);
    std::vector<std::thread> threads;
    for (int r = 0; r < ngpus; r++) {
        threads.emplace_back([&, r]() {
            VsrRunOpts o = *opts;
            o.device = opts->device + (one_device ? 0 : r);
            char msg[256] = {0};
            VsrEngine* e = nullptr;
            int rc = vsr_engine_create(m, &o, r, ngpus, &e, msg, sizeof msg);
            if (rc) {
                errors[r] = msg;
                vsr_group_abort(groups[r]);
                rcs[r] = rc;
                return;
            }
            rc = vsr_engine_attach_group(e, groups[r], inbox_records);
            if (!rc) rc = vsr_bfs_sharded(e, &o, part_states, &st[r], cands[r].data(), &lens[r], cands[r].size());
            if (rc && rc != VSR_RC_VIOLATION && rc != VSR_RC_DEADLOCK && rc != VSR_RC_TOO_LARGE && rc != VSR_RC_ERROR) {
                errors[r] = vsr_engine_last_error(e);
                vsr_group_abort(groups[r]);
            } else if (rc == VSR_RC_TOO_LARGE) errors[r] = vsr_engine_last_error(e);
            rcs[r] = rc;
            vsr_engine_destroy(e);
        });
    }
    for (auto& t : threads) t.join();
    for (int r = 0; r < ngpus; r++) vsr_group_close(groups[r]);
    int rc = rcs[0];
    for (int r = 0; r < ngpus; r++)
        if (rcs[r] == VSR_RC_SYSTEM || rcs[r] == VSR_RC_CONFIG_ERROR) rc = rcs[r];
    if (err && errcap) {
        err[0] = 0;
        for (int r = 0; r < ngpus; r++)
            if (!errors[r].empty()) { snprintf(err, errcap, "GPU %d: %s", opts->device + r, errors[r].c_str()); break; }
    }
    *stats = st[0];
    replay_counterexample(m, cands[0].data(), lens[0], stats, trace_out, trace_actions, trace_cap);
    stats->seconds_total = now_s() - t0;
    return rc;
}

} /* extern "C" */
