/*
 * vsr_ckpt.cu — checkpoint / recover of one rank's shard of the BFS (include/vsr_b200.h: vsr_engine_checkpoint,
 * vsr_engine_recover).  Stands in for TLC's `-checkpoint <minutes>` / `-recover <dir>` (SURVEY §8f item 4; the reference's
 * .gitignore:1 ignores TLC's states/ metadir): a multi-hour run of the README constants can be stopped and continued.
 *
 * A checkpoint is taken at a level boundary — every state of depth <= level is in the seen-set, the current frontier holds
 * exactly the states of depth `level`, nothing is in flight between ranks — and is ONE file per rank:
 *
 *   CkptHeader | VsrStats of this rank | VsrStats totals of the job | frontier: n_cur packed states | seen-set: n_entries x {fp, meta} | trace: next_base x 8 B
 *
 * The seen-set is written as its non-empty entries (compacted on the device into the idle frontier buffer, chunk by chunk)
 * and re-inserted on recovery with the BFS's own insert routine, so the table a run continues with may have another
 * capacity (or bucket layout) than the one it was checkpointed from.
 */
#include <errno.h>
#include <stdio.h>
#include <string.h>
#include <unistd.h>

#include <algorithm>
#include <string>
#include <vector>

#include "vsr_engine.h"

using namespace vsr;

namespace {

constexpr uint64_t CKPT_MAGIC = 0x3154504B43525356ull; /* "VSRCKPT1" */

struct CkptHeader {
    uint64_t magic;
    uint32_t version, header_bytes, stats_bytes, state_bytes;
    int32_t R, V, K;                      /* layout */
    int32_t symmetry, use_view, invariant; /* RunCfg: another VIEW / SYMMETRY setting is another state graph */
    int32_t rank, world;
    int32_t level, keep_trace;
    uint64_t n_cur, cur_base, next_base;  /* frontier of depth `level`: local ids [cur_base, cur_base + n_cur) */
    uint64_t n_entries;                   /* seen-set entries that follow */
    uint64_t n_trace;                     /* trace records that follow (0 without keep_trace) */
    uint64_t records_sent, records_received;
};

/* non-empty entries of table slots [first, first + n) appended to out[] (order is irrelevant); one atomic per warp */
__global__ void ckpt_compact_kernel(const uint64_t* __restrict__ table, unsigned long long first, unsigned long long n, uint64_t* __restrict__ out,
                                    unsigned long long* count) {
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    const unsigned long long rounds = (n + stride - 1) / stride;
    unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    for (unsigned long long r = 0; r < rounds; r++, i += stride) { /* whole warps stay in the loop: the ballot below is warp-wide */
        uint64_t e0 = 0, e1 = 0;
        if (i < n) {
            e0 = table[2 * (first + i)];
            e1 = table[2 * (first + i) + 1];
        }
        const unsigned m = __ballot_sync(0xffffffffu, e0 != 0);
        if (!m) continue;
        unsigned long long base = 0;
        const int leader = __ffs(m) - 1;
        if (lane == leader) base = atomicAdd(count, (unsigned long long)__popc(m));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (e0) {
            const unsigned long long pos = base + __popc(m & ((1u << lane) - 1u));
            out[2 * pos] = e0;
            out[2 * pos + 1] = e1;
        }
    }
}

/* entries of a checkpoint back into a (fresh) table: every one must be new */
__global__ void ckpt_reinsert_kernel(uint64_t* table, unsigned long long cap, const uint64_t* __restrict__ ents, unsigned long long n,
                                     unsigned long long* not_new) {
    unsigned long long bad = 0;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x) {
        unsigned probes = 0, coll = 0;
        if (table_insert(table, cap, ents[2 * i], ents[2 * i + 1], probes, coll) != INS_NEW) bad++;
    }
    if (bad) atomicAdd(not_new, bad);
}

struct File {
    FILE* f = nullptr;
    ~File() { if (f) fclose(f); }
};

int io_error(VsrEngine* e, const char* what, const char* path) {
    snprintf(e->last_error, sizeof e->last_error, "checkpoint: %s %s: %s", what, path, strerror(errno));
    return VSR_RC_SYSTEM;
}

/* frontier states [first, first + n) of buffer `buf` <-> host: the part in HBM by cudaMemcpy, the spilled part directly */
int frontier_to_host(VsrEngine* e, int buf, uint64_t first, uint64_t n, uint8_t* host) {
    const uint64_t S = (uint64_t)e->g->bytes;
    const uint64_t in_dev = first < e->frontier_cap ? std::min(n, e->frontier_cap - first) : 0;
    if (in_dev) CK(cudaMemcpy(host, (const uint8_t*)e->frontier[buf] + first * S, in_dev * S, cudaMemcpyDeviceToHost));
    if (n > in_dev) memcpy(host + in_dev * S, (const uint8_t*)e->frontier_host[buf] + (first + in_dev - e->frontier_cap) * S, (n - in_dev) * S);
    return 0;
}
int frontier_from_host(VsrEngine* e, int buf, uint64_t first, uint64_t n, const uint8_t* host) {
    const uint64_t S = (uint64_t)e->g->bytes;
    const uint64_t in_dev = first < e->frontier_cap ? std::min(n, e->frontier_cap - first) : 0;
    if (in_dev) CK(cudaMemcpy((uint8_t*)e->frontier[buf] + first * S, host, in_dev * S, cudaMemcpyHostToDevice));
    if (n > in_dev) memcpy((uint8_t*)e->frontier_host[buf] + (first + in_dev - e->frontier_cap) * S, host + in_dev * S, (n - in_dev) * S);
    return 0;
}

constexpr uint64_t IO_CHUNK = 64ull << 20; /* bytes per host staging round */

} // namespace

extern "C" {

int vsr_engine_checkpoint(VsrEngine* e, const char* path, const VsrStats* totals) {
    if (!e || !path) return VSR_RC_ERROR;
    if (e->level_open) {
        snprintf(e->last_error, sizeof e->last_error, "checkpoint: only at a level boundary (after vsr_engine_finish_level)");
        return VSR_RC_ERROR;
    }
    CK(cudaSetDevice(e->device));
    CK(cudaStreamSynchronize(e->stream));
    const uint64_t S = (uint64_t)e->g->bytes;
    const std::string tmp = std::string(path) + ".tmp";
    File out;
    out.f = fopen(tmp.c_str(), "wb");
    if (!out.f) return io_error(e, "cannot create", tmp.c_str());
    CkptHeader h;
    memset(&h, 0, sizeof h);
    h.magic = CKPT_MAGIC;
    h.version = 1;
    h.header_bytes = sizeof h;
    h.stats_bytes = sizeof(VsrStats);
    h.state_bytes = (uint32_t)S;
    h.R = e->g->R; h.V = e->g->V; h.K = e->g->K;
    h.symmetry = e->m->run.symmetry; h.use_view = e->m->run.use_view; h.invariant = e->m->run.invariant;
    h.rank = e->rank; h.world = e->world;
    h.level = e->level;
    h.keep_trace = e->trace ? 1 : 0;
    h.n_cur = e->n_cur; h.cur_base = e->cur_base; h.next_base = e->next_base;
    h.n_entries = e->st.distinct; /* checked against what the compaction finds */
    h.n_trace = e->trace ? std::min<uint64_t>(e->next_base, e->trace_cap) : 0;
    h.records_sent = e->records_sent; h.records_received = e->records_received;
    const VsrStats& tot = totals ? *totals : e->st;
    if (fwrite(&h, sizeof h, 1, out.f) != 1 || fwrite(&e->st, sizeof(VsrStats), 1, out.f) != 1 || fwrite(&tot, sizeof(VsrStats), 1, out.f) != 1)
        return io_error(e, "cannot write", tmp.c_str());
    std::vector<uint8_t> host;
    /* 1. the frontier of depth `level` */
    {
        const uint64_t per = std::max<uint64_t>(1, IO_CHUNK / S);
        host.resize(per * S);
        for (uint64_t first = 0; first < e->n_cur; first += per) {
            const uint64_t n = std::min(per, e->n_cur - first);
            int rc = frontier_to_host(e, e->cur, first, n, host.data());
            if (rc) return rc;
            if (fwrite(host.data(), S, n, out.f) != n) return io_error(e, "cannot write", tmp.c_str());
        }
    }
    /* 2. the seen-set's entries, compacted into the idle frontier buffer (its HBM part) chunk by chunk */
    {
        uint64_t* scratch = (uint64_t*)e->frontier[e->cur ^ 1];
        const uint64_t slots_per_pass = std::max<uint64_t>(64, e->frontier_cap * S / 16);
        unsigned long long* dcount = &e->ctr->work_next; /* scratch word: the level's counters are reset when it opens */
        uint64_t written = 0;
        for (uint64_t first = 0; first < e->table_cap; first += slots_per_pass) {
            const uint64_t n = std::min(slots_per_pass, e->table_cap - first);
            CK(cudaMemsetAsync(dcount, 0, 8, e->stream));
            ckpt_compact_kernel<<<e->sms * 8, 256, 0, e->stream>>>(e->table, first, n, scratch, dcount);
            CK(cudaGetLastError());
            unsigned long long cnt = 0;
            CK(cudaMemcpyAsync(&cnt, dcount, 8, cudaMemcpyDeviceToHost, e->stream));
            CK(cudaStreamSynchronize(e->stream));
            const uint64_t per = IO_CHUNK / 16;
            host.resize(std::min<uint64_t>(per, std::max<uint64_t>(cnt, 1)) * 16);
            for (uint64_t o = 0; o < cnt; o += per) {
                const uint64_t k = std::min<uint64_t>(per, cnt - o);
                CK(cudaMemcpy(host.data(), scratch + 2 * o, k * 16, cudaMemcpyDeviceToHost));
                if (fwrite(host.data(), 16, k, out.f) != k) return io_error(e, "cannot write", tmp.c_str());
            }
            written += cnt;
        }
        if (written != h.n_entries) {
            snprintf(e->last_error, sizeof e->last_error, "checkpoint: the seen-set holds %llu entries, the run counted %llu distinct states",
                     (unsigned long long)written, (unsigned long long)h.n_entries);
            return VSR_RC_ERROR;
        }
        e->st.bytes_d2h += written * 16;
    }
    /* 3. the trace records */
    if (h.n_trace) {
        const uint64_t per = IO_CHUNK / 8;
        host.resize(std::min(per, h.n_trace) * 8);
        for (uint64_t o = 0; o < h.n_trace; o += per) {
            const uint64_t k = std::min(per, h.n_trace - o);
            CK(cudaMemcpy(host.data(), e->trace + o, k * 8, cudaMemcpyDeviceToHost));
            if (fwrite(host.data(), 8, k, out.f) != k) return io_error(e, "cannot write", tmp.c_str());
        }
        e->st.bytes_d2h += h.n_trace * 8;
    }
    e->st.bytes_d2h += e->n_cur * S;
    if (fflush(out.f) != 0 || fsync(fileno(out.f)) != 0) return io_error(e, "cannot write", tmp.c_str()); /* on disk before it replaces the previous one */
    fclose(out.f);
    out.f = nullptr;
    if (rename(tmp.c_str(), path) != 0) return io_error(e, "cannot rename to", path);
    return 0;
}

int vsr_engine_recover(VsrEngine* e, const char* path, VsrStats* totals_out) {
    if (!e || !path) return VSR_RC_ERROR;
    CK(cudaSetDevice(e->device));
    File in;
    in.f = fopen(path, "rb");
    if (!in.f) return io_error(e, "cannot open", path);
    CkptHeader h;
    VsrStats mine, tot;
    if (fread(&h, sizeof h, 1, in.f) != 1 || h.magic != CKPT_MAGIC || h.version != 1 || h.header_bytes != sizeof h || h.stats_bytes != sizeof(VsrStats)) {
        snprintf(e->last_error, sizeof e->last_error, "recover: %s is not a checkpoint of this build", path);
        return VSR_RC_SPEC_ERROR;
    }
    if (fread(&mine, sizeof mine, 1, in.f) != 1 || fread(&tot, sizeof tot, 1, in.f) != 1) return io_error(e, "truncated", path);
    const uint64_t S = (uint64_t)e->g->bytes;
    if (h.state_bytes != S || h.R != e->g->R || h.V != e->g->V || h.K != e->g->K || h.symmetry != e->m->run.symmetry || h.use_view != e->m->run.use_view ||
        h.invariant != e->m->run.invariant) {
        snprintf(e->last_error, sizeof e->last_error,
                 "recover: %s was written for ReplicaCount=%d |Values|=%d StartViewOnTimerLimit=%d symmetry=%d view=%d invariants=%d: not this model", path,
                 h.R, h.V, h.K - 1, h.symmetry, h.use_view, h.invariant);
        return VSR_RC_SPEC_ERROR;
    }
    if (h.rank != e->rank || h.world != e->world) {
        snprintf(e->last_error, sizeof e->last_error, "recover: %s is rank %d of %d, this engine is rank %d of %d", path, h.rank, h.world, e->rank, e->world);
        return VSR_RC_CONFIG_ERROR;
    }
    if (h.n_cur > e->frontier_cap + e->frontier_host_cap || h.n_entries > e->table_cap - e->table_cap / 8 || (h.n_trace && e->trace && h.n_trace > e->trace_cap)) {
        snprintf(e->last_error, sizeof e->last_error, "capacity exceeded (recover): the checkpoint holds %llu frontier states and %llu seen-set entries",
                 (unsigned long long)h.n_cur, (unsigned long long)h.n_entries);
        return VSR_RC_TOO_LARGE;
    }
    if (e->trace && !h.n_trace && h.next_base) {
        snprintf(e->last_error, sizeof e->last_error, "recover: %s was written without trace records; continue it with keep_trace off (vsrmc -notrace)", path);
        return VSR_RC_CONFIG_ERROR;
    }
    int rc = vsr_engine_reset(e);
    if (rc) return rc;
    e->table_clean = false;
    CK(cudaStreamSynchronize(e->stream));
    std::vector<uint8_t> host;
    /* 1. the frontier, into buffer 0 */
    e->cur = 0;
    {
        const uint64_t per = std::max<uint64_t>(1, IO_CHUNK / S);
        host.resize(per * S);
        for (uint64_t first = 0; first < h.n_cur; first += per) {
            const uint64_t n = std::min(per, h.n_cur - first);
            if (fread(host.data(), S, n, in.f) != n) return io_error(e, "truncated", path);
            rc = frontier_from_host(e, 0, first, n, host.data());
            if (rc) return rc;
        }
    }
    /* 2. the seen-set, re-inserted through the idle frontier buffer */
    {
        uint64_t* scratch = (uint64_t*)e->frontier[1];
        const uint64_t per = std::max<uint64_t>(1, std::min<uint64_t>(IO_CHUNK / 16, e->frontier_cap * S / 16));
        unsigned long long* dbad = &e->ctr->work_next;
        CK(cudaMemsetAsync(dbad, 0, 8, e->stream));
        host.resize(per * 16);
        for (uint64_t o = 0; o < h.n_entries; o += per) {
            const uint64_t k = std::min(per, h.n_entries - o);
            if (fread(host.data(), 16, k, in.f) != k) return io_error(e, "truncated", path);
            CK(cudaMemcpyAsync(scratch, host.data(), k * 16, cudaMemcpyHostToDevice, e->stream));
            ckpt_reinsert_kernel<<<e->sms * 8, 256, 0, e->stream>>>(e->table, e->table_cap, scratch, k, dbad);
            CK(cudaGetLastError());
            CK(cudaStreamSynchronize(e->stream)); /* `host` is reused by the next round */
        }
        unsigned long long bad = 0;
        CK(cudaMemcpy(&bad, dbad, 8, cudaMemcpyDeviceToHost));
        if (bad) {
            snprintf(e->last_error, sizeof e->last_error, "recover: %llu seen-set entries of %s could not be inserted as new (corrupt file?)", bad, path);
            return VSR_RC_ERROR;
        }
    }
    /* 3. the trace records */
    if (h.n_trace) {
        const uint64_t per = IO_CHUNK / 8;
        host.resize(std::min(per, h.n_trace) * 8);
        for (uint64_t o = 0; o < h.n_trace; o += per) {
            const uint64_t k = std::min(per, h.n_trace - o);
            if (fread(host.data(), 8, k, in.f) != k) return io_error(e, "truncated", path);
            if (e->trace) CK(cudaMemcpy(e->trace + o, host.data(), k * 8, cudaMemcpyHostToDevice));
        }
    }
    /* the BFS position and this rank's statistics continue where they were; capacities are this engine's */
    const uint64_t tc = e->st.table_capacity, fc = e->st.frontier_capacity, bt = e->st.bytes_table, bf = e->st.bytes_frontier;
    e->st = mine;
    e->st.table_capacity = tc; e->st.frontier_capacity = fc; e->st.bytes_table = bt; e->st.bytes_frontier = bf;
    e->st.bytes_h2d += h.n_cur * S + h.n_entries * 16 + h.n_trace * 8;
    e->n_cur = h.n_cur; e->cur_base = h.cur_base; e->next_base = h.next_base;
    e->level = h.level;
    e->level_open = false;
    e->records_sent = h.records_sent; e->records_received = h.records_received;
    if (totals_out) *totals_out = tot;
    return 0;
}

} /* extern "C" */
