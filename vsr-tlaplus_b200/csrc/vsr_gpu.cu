/*
 * vsr_gpu.cu — the engine's steps behind the C ABI (vsr_engine_*; include/vsr_b200.h), vsr_simulate and vsr_probe_bench.
 * Per level one expand launch on each step (which also inserts the records peer ranks pushed here), one small counter
 * read-back, swap frontiers.  The level loop that drives these steps is vsr_bfs_sharded (vsr_shard.cu).  Kernels: vsr_gpu.cuh.
 * There is NO CPU fallback: without a usable CUDA device every entry point returns 153.
 */
#include <stddef.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <chrono>
#include <string>
#include <vector>

#include "vsr_engine.h"

namespace vsr {

const GpuOps* find_gpu_ops(int R, int V, int K) {
#define X(r, v, k) \
    if (R == r && V == v && K == k) return GpuThunks<Layout<r, v, k>>::get();
    VSR_FOR_EACH_CONFIG(X)
#undef X
    return nullptr;
}

} // namespace vsr

using namespace vsr;

int engine_reset_level(VsrEngine* e) {
    CK(cudaMemsetAsync(e->ctr, 0, sizeof(DevCounters), e->stream));
    static const unsigned long long ones = ~0ull;
    CK(cudaMemcpyAsync(&e->ctr->viol_id, &ones, 8, cudaMemcpyHostToDevice, e->stream));
    CK(cudaMemcpyAsync(&e->ctr->dead_id, &ones, 8, cudaMemcpyHostToDevice, e->stream));
    e->level_open = true;
    e->level_ms_acc = 0;
    e->level_ms_insert_acc = 0;
    return 0;
}

void fill_params(VsrEngine* e, ExpandParams& p) {
    memset(&p, 0, sizeof p);
    p.in = e->frontier[e->cur];
    p.n_in = e->n_cur;
    p.in_base = e->cur_base;
    p.in_hi = e->frontier_host[e->cur];
    p.in_split = e->frontier_host_cap ? e->frontier_cap : ~0ull;
    p.out = e->frontier[e->cur ^ 1];
    p.out_hi = e->frontier_host[e->cur ^ 1];
    p.out_split = e->frontier_host_cap ? e->frontier_cap : ~0ull;
    p.out_cap = e->frontier_cap + e->frontier_host_cap;
    p.out_base = e->next_base;
    p.table = e->table;
    p.table_cap = e->table_cap;
    p.trace = e->trace;
    p.trace_cap = e->trace_cap;
    p.ctr = e->ctr;
    p.ties = e->ties;
    p.tie_cap = e->tie_cap;
    p.fp_tab = e->fp_tab;
    p.run = e->m->run;
    p.level = e->level + 1;
    p.check_deadlock = e->opts.check_deadlock;
    p.rank = e->rank;
    p.world = e->world;
    p.owner_shift = e->owner_shift;
    p.push_cap = e->inbox_cap;
    p.push_direct = e->push_direct;
}

extern "C" {

int vsr_gpu_abi(void) { return vsr::gpu_abi_value(); } /* compared with a layout plug-in's vsr_plugin_abi() before it is used */

int vsr_engine_create(const VsrModel* m, const VsrRunOpts* opts, int rank, int world, VsrEngine** out, char* err, size_t errcap) {
    auto fail = [&](int rc, const std::string& msg) {
        if (err && errcap) snprintf(err, errcap, "%s", msg.c_str());
        return rc;
    };
    if (!m || !opts || !out) return fail(VSR_RC_ERROR, "null argument");
    if (!m->gpu) return fail(VSR_RC_CONFIG_ERROR, "no GPU kernels compiled for this configuration");
    if (world < 1 || world > MAX_WORLD || (world & (world - 1)) || rank < 0 || rank >= world)
        return fail(VSR_RC_CONFIG_ERROR, "world must be 1, 2, 4 or 8 and 0 <= rank < world");
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev == 0)
        return fail(VSR_RC_SYSTEM, std::string("no usable CUDA device (") + cudaGetErrorString(ce) + "): the BFS runs on the GPU only, there is no CPU fallback");
    VsrEngine* e = new VsrEngine();
    e->m = m;
    e->g = m->gpu;
    e->opts = *opts;
    e->rank = rank;
    e->world = world;
    int lg = 0;
    while ((1 << lg) < world) lg++;
    e->owner_shift = world > 1 ? 64 - lg : 64;
    e->device = opts->device;
    if (const char* pm = getenv("VSR_B200_PUSH")) e->push_direct = strcmp(pm, "direct") == 0;
    memset(&e->st, 0, sizeof e->st);
    auto bail = [&](const char* what, cudaError_t c) {
        std::string msg = std::string(what) + ": " + cudaGetErrorString(c);
        vsr_engine_destroy(e);
        return fail(VSR_RC_SYSTEM, msg);
    };
    if ((ce = cudaSetDevice(e->device)) != cudaSuccess) return bail("cudaSetDevice", ce);
    cudaDeviceProp prop;
    if ((ce = cudaGetDeviceProperties(&prop, e->device)) != cudaSuccess) return bail("cudaGetDeviceProperties", ce);
    e->sms = prop.multiProcessorCount;
    if ((ce = cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking)) != cudaSuccess) return bail("cudaStreamCreate", ce);
    { /* keep freed device memory in the driver's pool: a process that checks one model after another (bench e2e, a service)
         does not pay the page-mapping cost of tens of GB again */
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, e->device) == cudaSuccess) {
            uint64_t keep = ~0ull;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
    }
    cudaEventCreate(&e->ev0);
    cudaEventCreate(&e->ev1);
    if ((ce = e->g->prepare(&e->blocks_per_sm)) != cudaSuccess) return bail("kernel attributes", ce);
    if (e->blocks_per_sm < 1) e->blocks_per_sm = 1;
    /* capacities */
    size_t free_b = 0, total_b = 0;
    cudaMemGetInfo(&free_b, &total_b);
    uint64_t tcap = opts->table_capacity, fcap = opts->frontier_capacity;
    const uint64_t S = (uint64_t)e->g->bytes;
    if (!tcap) tcap = (uint64_t)(free_b * 0.45) / 23; /* table 16 B/slot + trace 8 B per state at load <= 7/8  ->  23 B per slot; ~45% of free memory */
    tcap = (tcap + 63) & ~63ull; /* any size (whole buckets / cache lines), not only powers of two */
    if (!fcap) fcap = (uint64_t)(free_b * 0.40) / (2 * S);
    if (fcap < 64) fcap = 64;
    e->table_cap = tcap;
    e->frontier_cap = fcap;
    e->trace_cap = opts->keep_trace ? tcap - tcap / 8 + 64 : 0; /* one record per distinct state, up to the seen-set's load limit */
    e->tie_cap = 1 << 16;
    if ((ce = cudaMallocAsync((void**)&e->table, tcap * 16, e->stream)) != cudaSuccess) return bail("cudaMalloc(seen-set)", ce);
    if ((ce = cudaMemsetAsync(e->table, 0, tcap * 16, e->stream)) != cudaSuccess) return bail("memset", ce);
    for (int i = 0; i < 2; i++)
        if ((ce = cudaMallocAsync((void**)&e->frontier[i], fcap * S, e->stream)) != cudaSuccess) return bail("cudaMalloc(frontier)", ce);
    if (opts->frontier_host_capacity) { /* spill: each frontier buffer continues in pinned, device-mapped host memory */
        e->frontier_host_cap = opts->frontier_host_capacity;
        for (int i = 0; i < 2; i++)
            if ((ce = cudaHostAlloc((void**)&e->frontier_host[i], e->frontier_host_cap * S, cudaHostAllocPortable | cudaHostAllocMapped)) != cudaSuccess)
                return bail("cudaHostAlloc(frontier spill)", ce);
    }
    if (e->trace_cap && (ce = cudaMallocAsync((void**)&e->trace, e->trace_cap * 8, e->stream)) != cudaSuccess) return bail("cudaMalloc(trace)", ce);
    if ((ce = cudaMallocAsync((void**)&e->ctr, sizeof(DevCounters), e->stream)) != cudaSuccess) return bail("cudaMalloc", ce);
    if ((ce = cudaMallocAsync((void**)&e->ties, e->tie_cap * (size_t)e->g->tie_bytes, e->stream)) != cudaSuccess) return bail("cudaMalloc", ce);
    if ((ce = cudaMallocAsync((void**)&e->fp_tab, 8 * 256 * 8, e->stream)) != cudaSuccess) return bail("cudaMalloc", ce);
    if ((ce = cudaMallocAsync((void**)&e->init_rec, e->g->rec_bytes, e->stream)) != cudaSuccess) return bail("cudaMalloc", ce);
    if ((ce = cudaMemcpyAsync(e->fp_tab, fp64_table(), 8 * 256 * 8, cudaMemcpyHostToDevice, e->stream)) != cudaSuccess) return bail("memcpy", ce);
    e->st.table_capacity = tcap;
    e->st.frontier_capacity = fcap + e->frontier_host_cap;
    e->st.bytes_table = tcap * 16;
    e->st.bytes_frontier = 2 * fcap * S;
    e->st.bytes_h2d += 8 * 256 * 8;
    if ((ce = cudaStreamSynchronize(e->stream)) != cudaSuccess) return bail("sync", ce);
    e->table_clean = true;
    *out = e;
    return 0;
}

void vsr_engine_destroy(VsrEngine* e) {
    if (!e) return;
    if (e->stream) cudaFreeAsync(e->table, e->stream); else cudaFree(e->table);
    if (e->stream) cudaFreeAsync(e->frontier[0], e->stream); else cudaFree(e->frontier[0]);
    if (e->stream) cudaFreeAsync(e->frontier[1], e->stream); else cudaFree(e->frontier[1]);
    for (int i = 0; i < 2; i++)
        if (e->frontier_host[i]) cudaFreeHost(e->frontier_host[i]);
    if (e->stream) cudaFreeAsync(e->trace, e->stream); else cudaFree(e->trace);
    if (e->stream) cudaFreeAsync(e->ctr, e->stream); else cudaFree(e->ctr);
    if (e->stream) cudaFreeAsync(e->ties, e->stream); else cudaFree(e->ties);
    if (e->stream) cudaFreeAsync(e->fp_tab, e->stream); else cudaFree(e->fp_tab);
    if (e->stream) cudaFreeAsync(e->init_rec, e->stream); else cudaFree(e->init_rec);
    vsr_engine_detach(e);
    if (e->ev0) cudaEventDestroy(e->ev0);
    if (e->ev1) cudaEventDestroy(e->ev1);
    if (e->stream) { cudaStreamSynchronize(e->stream); cudaStreamDestroy(e->stream); }
    delete e;
}

int vsr_engine_record_bytes(const VsrEngine* e) { return e->g->rec_bytes; }

/* Level 1: the single initial state (VSR.tla:323-348), inserted by the rank that owns its fingerprint.
   The "current frontier" is empty and the "next" frontier receives Init; finish_level() then advances. */
int vsr_engine_seed_init(VsrEngine* e) {
    const ModelOps* ops = e->m->ops;
    std::vector<uint8_t> rec(e->g->rec_bytes, 0);
    ops->init((uint32_t*)rec.data());
    uint64_t fp = ops->fingerprint((const uint32_t*)rec.data(), e->m->run.use_view);
    if (fp == 0) fp = 1;
    const int owner = e->world > 1 ? owner_of(fp, e->owner_shift) : e->rank;
    e->level = 0;
    e->n_cur = 0;
    e->cur_base = 0;
    e->next_base = 0;
    int rc = engine_reset_level(e);
    if (rc) return rc;
    if (owner != e->rank) return 0;
    e->table_clean = false;
    RecHdr* h = (RecHdr*)(rec.data() + e->g->bytes);
    h->fp = fp;
    h->tm = make_trec(ROOT_GID, 0) | (1ull << 56); /* no parent; stands for one generated state */
    CK(cudaMemcpyAsync(e->init_rec, rec.data(), rec.size(), cudaMemcpyHostToDevice, e->stream));
    e->st.bytes_h2d += rec.size();
    InsertParams q;
    fill_params(e, q.e);
    q.e.level = 1;
    q.recs = e->init_rec;
    q.n = 1;
    CK(e->g->launch_insert(q, e->stream));
    e->st.kernel_launches++;
    return 0;
}

/* One launch of the wavefront kernel: expand frontier states [first, first + count) of the current level (count = 0:
   nothing to expand on this rank) — successors this rank owns are inserted, the others are pushed into their owners'
   inboxes, half `parity` — and then insert the records peers pushed HERE in the previous step (the other half):
   drain_counts[s] records from rank s (NULL = none).  sent_out[d] = records pushed to rank d by this launch. */
int vsr_engine_step(VsrEngine* e, uint64_t first, uint64_t count, int parity, const uint32_t* drain_counts, uint32_t* sent_out) {
    if (!e->level_open) {
        int rc = engine_reset_level(e);
        if (rc) return rc;
    }
    if (first >= e->n_cur) { first = e->n_cur; count = 0; } /* this rank's frontier ends before the part (or the launch only drains) */
    else if (count > e->n_cur - first) count = e->n_cur - first;
    ExpandParams p;
    fill_params(e, p);
    if (first < p.in_split || !e->frontier_host_cap) {
        p.in += first * (uint64_t)e->g->nw;
        if (e->frontier_host_cap) p.in_split -= first;
    } else { /* this part lies entirely in the host part of the frontier */
        p.in = p.in_hi + (first - p.in_split) * (uint64_t)e->g->nw;
        p.in_hi = nullptr;
        p.in_split = ~0ull;
    }
    p.n_in = count;
    p.in_base += first;
    uint64_t drain_total = 0;
    if (e->world > 1) {
        if (!e->inbox) {
            snprintf(e->last_error, sizeof e->last_error, "world > 1 without an exchange: call vsr_engine_attach_group or vsr_engine_attach_staged first");
            return VSR_RC_ERROR;
        }
        const uint64_t seg = e->inbox_cap * (uint64_t)e->g->rec_bytes;
        parity &= 1;
        for (int r = 0; r < e->world; r++) {
            p.push[r] = e->stage ? e->stage + (uint64_t)r * seg : (e->peer_inbox[r] ? e->peer_inbox[r] + ((uint64_t)parity * e->world + e->rank) * seg : nullptr);
            p.drain[r] = e->inbox + ((uint64_t)(parity ^ 1) * e->world + r) * seg;
            uint32_t n = (drain_counts && r != e->rank) ? drain_counts[r] : 0;
            if (n > e->inbox_cap) n = (uint32_t)e->inbox_cap; /* the sender reported the overflow; never read past the segment */
            p.drain_n[r] = n;
            drain_total += n;
        }
        p.drain_total = drain_total;
    }
    if (sent_out) memset(sent_out, 0, sizeof(uint32_t) * e->world);
    if (count == 0 && drain_total == 0) return 0;
    e->table_clean = false;
    CK(cudaMemsetAsync(&e->ctr->work_next, 0, sizeof(DevCounters) - offsetof(DevCounters, work_next), e->stream)); /* work_next, drain_next, send_count[] */
    const uint64_t spb = (uint64_t)e->g->states_per_block;
    uint64_t want_blocks = (count + spb - 1) / spb;
    const uint64_t drain_blocks = (drain_total + spb - 1) / spb;
    if (drain_blocks > want_blocks) want_blocks = drain_blocks;
    const uint64_t max_blocks = (uint64_t)e->sms * e->blocks_per_sm; /* persistent: whole multiples of the SM count */
    int grid = (int)(want_blocks < max_blocks ? want_blocks : max_blocks);
    if (grid < 1) grid = 1;
    CK(cudaEventRecord(e->ev0, e->stream));
    CK(e->g->launch_expand(p, grid, e->stream));
    CK(cudaEventRecord(e->ev1, e->stream));
    e->st.kernel_launches++;
    if (e->world > 1 && sent_out) {
        CK(cudaMemcpyAsync(sent_out, e->ctr->send_count, sizeof(uint32_t) * e->world, cudaMemcpyDeviceToHost, e->stream));
        e->st.bytes_d2h += sizeof(uint32_t) * e->world;
    }
    CK(cudaStreamSynchronize(e->stream)); /* the pushed records have landed (kernel completion) before the host tells anybody */
    float ms = 0;
    cudaEventElapsedTime(&ms, e->ev0, e->ev1);
    e->level_ms_acc += ms;
    if (count == 0) e->level_ms_insert_acc += ms;
    if (sent_out)
        for (int r = 0; r < e->world; r++) e->records_sent += sent_out[r];
    e->records_received += drain_total;
    return 0;
}

int vsr_engine_expand(VsrEngine* e) { return vsr_engine_step(e, 0, e->n_cur, 0, nullptr, nullptr); }

int vsr_engine_insert_records(VsrEngine* e, const void* dev_records, uint64_t n) {
    if (!e->level_open) {
        int rc = engine_reset_level(e);
        if (rc) return rc;
    }
    if (n == 0) return 0;
    e->table_clean = false;
    InsertParams q;
    fill_params(e, q.e);
    q.recs = (const uint8_t*)dev_records;
    q.n = n;
    CK(cudaEventRecord(e->ev0, e->stream));
    CK(e->g->launch_insert(q, e->stream));
    CK(cudaEventRecord(e->ev1, e->stream));
    e->st.kernel_launches++;
    CK(cudaEventSynchronize(e->ev1));
    float ms = 0;
    cudaEventElapsedTime(&ms, e->ev0, e->ev1);
    e->level_ms_acc += ms;
    e->level_ms_insert_acc += ms;
    return 0;
}

int vsr_engine_finish_level(VsrEngine* e, VsrLevelInfo* out) {
    DevCounters c;
    CK(cudaMemcpyAsync(&c, e->ctr, sizeof c, cudaMemcpyDeviceToHost, e->stream));
    e->st.bytes_d2h += sizeof c;
    CK(cudaStreamSynchronize(e->stream));
    const uint64_t fcap_total = e->frontier_cap + e->frontier_host_cap;
    if (c.tie_count > 0 && c.tie_count <= e->tie_cap && !c.overflow && c.out_count <= fcap_total) {
        /* SURVEY H2: same-level states with equal VIEW but different aux variables.  Keep, per fingerprint, the
           smallest (aux_key, parent, candidate) among the late arrivals, sorted by fingerprint, and let the patch
           kernel replace first arrivals that lose; the level's violation verdict is recomputed from scratch. */
        const size_t tb = (size_t)e->g->tie_bytes;
        std::vector<uint8_t> host(c.tie_count * tb);
        CK(cudaMemcpyAsync(host.data(), e->ties, host.size(), cudaMemcpyDeviceToHost, e->stream));
        CK(cudaStreamSynchronize(e->stream));
        std::vector<const uint8_t*> recs;
        for (uint64_t i = 0; i < c.tie_count; i++) recs.push_back(host.data() + i * tb);
        auto key = [](const uint8_t* r) { return (const TieRec*)r; };
        std::sort(recs.begin(), recs.end(), [&](const uint8_t* a, const uint8_t* b) {
            const TieRec *x = key(a), *y = key(b);
            if (x->fp != y->fp) return x->fp < y->fp;
            if (x->check != y->check) return x->check < y->check;
            if (x->auxkey != y->auxkey) return x->auxkey < y->auxkey;
            if (x->parent != y->parent) return x->parent < y->parent;
            return x->cand < y->cand;
        });
        std::vector<uint8_t> best;
        uint64_t nbest = 0;
        for (size_t i = 0; i < recs.size(); i++) {
            if (i && key(recs[i])->fp == key(recs[i - 1])->fp && key(recs[i])->check == key(recs[i - 1])->check) continue;
            best.insert(best.end(), recs[i], recs[i] + tb);
            nbest++;
        }
        /* everything on the engine's stream (it does not synchronise with the legacy stream); `best` and `ones` outlive
           the copies: the stream is synchronised below before they go out of scope */
        CK(cudaMemcpyAsync(e->ties, best.data(), best.size(), cudaMemcpyHostToDevice, e->stream));
        static const unsigned long long ones = ~0ull;
        CK(cudaMemcpyAsync(&e->ctr->viol_id, &ones, 8, cudaMemcpyHostToDevice, e->stream));
        CK(cudaMemsetAsync(&e->ctr->viol_which, 0, sizeof(int), e->stream));
        ExpandParams p;
        fill_params(e, p);
        CK(e->g->launch_patch(p, e->ties, nbest, c.out_count, e->stream));
        e->st.kernel_launches++;
        CK(cudaMemcpyAsync(&c, e->ctr, sizeof c, cudaMemcpyDeviceToHost, e->stream));
        CK(cudaStreamSynchronize(e->stream));
        e->st.bytes_d2h += host.size() + sizeof c;
        e->st.bytes_h2d += best.size();
    }
    VsrLevelInfo li;
    memset(&li, 0, sizeof li);
    li.new_states = c.out_count;
    li.generated = c.generated;
    li.frontier_in = e->n_cur;
    li.ties = c.ties;
    li.collisions = c.collisions;
    li.violation = c.viol_id != ~0ull;
    li.violation_id = c.viol_id;
    li.violation_mask = c.viol_which;
    li.deadlock = c.dead_id != ~0ull;
    li.deadlock_id = c.dead_id;
    li.error_code = c.error;
    li.overflow = c.overflow;
    li.ms = e->level_ms_acc;
    li.ms_insert = e->level_ms_insert_acc;
    if (c.overflow) {
        snprintf(e->last_error, sizeof e->last_error, "capacity exceeded (%s): %llu new states this level, frontier capacity %llu",
                 c.overflow == 1 ? "frontier" : (c.overflow == 2 ? "tie list" : (c.overflow == 3 ? "send buffer" : "seen-set")), (unsigned long long)c.out_count,
                 (unsigned long long)fcap_total);
    }
    if (!li.overflow && e->st.distinct + c.out_count > e->table_cap - e->table_cap / 8) {
        li.overflow = 4; /* seen-set load above 7/8: probe chains explode long before it is literally full */
        snprintf(e->last_error, sizeof e->last_error, "capacity exceeded (seen-set): %llu distinct states in %llu slots",
                 (unsigned long long)(e->st.distinct + c.out_count), (unsigned long long)e->table_cap);
    }
    /* advance */
    const uint64_t n_new = c.out_count <= fcap_total ? c.out_count : fcap_total;
    e->st.generated += c.generated;
    e->st.distinct += n_new;
    e->st.h2_ties += c.ties;
    e->st.fp_collisions += c.collisions;
    e->st.probe_total += c.probes;
    e->st.seconds_kernels += e->level_ms_acc * 1e-3;
    if (c.error && !e->st.error_code) e->st.error_code = c.error;
    const int gen_level = e->level + 1; /* depth of the states just generated */
    if (e->level >= 1 && e->level - 1 < VSR_MAX_LEVELS) {
        e->st.level_generated[e->level - 1] = c.generated;
        e->st.level_ms[e->level - 1] = e->level_ms_acc;
        e->st.levels_expanded = e->level;
    }
    if (n_new > 0 && gen_level - 1 < VSR_MAX_LEVELS) {
        e->st.level_sizes[gen_level - 1] = n_new;
        e->st.num_levels = gen_level;
    }
    if (li.violation && e->st.violation_level == 0) {
        e->st.violation_level = gen_level;
        e->st.violation_id = c.viol_id;
    }
    e->cur ^= 1;
    e->cur_base = e->next_base;
    e->n_cur = n_new;
    e->next_base += n_new;
    e->level = gen_level;
    e->level_open = false;
    if (e->opts.collect_levels) { /* one entry per level, empty when this rank found nothing at that depth (several ranks) */
        std::vector<uint8_t> host((size_t)n_new * e->g->bytes);
        if (n_new && vsr_engine_read_frontier(e, 0, n_new, host.data())) return VSR_RC_SYSTEM;
        e->collected.push_back(std::move(host));
    }
    if (out) *out = li;
    return 0;
}

uint64_t vsr_engine_frontier_size(const VsrEngine* e) { return e->n_cur; }

int vsr_engine_read_frontier(VsrEngine* e, uint64_t first, uint64_t n, void* host_out) {
    if (first + n > e->n_cur) return VSR_RC_ERROR;
    const uint64_t S = (uint64_t)e->g->bytes;
    const uint64_t in_dev = first < e->frontier_cap ? std::min(n, e->frontier_cap - first) : 0; /* the rest is in the host part (spill) */
    if (in_dev) CK(cudaMemcpy(host_out, (const uint8_t*)e->frontier[e->cur] + first * S, in_dev * S, cudaMemcpyDeviceToHost));
    if (n > in_dev) memcpy((uint8_t*)host_out + in_dev * S, (const uint8_t*)e->frontier_host[e->cur] + (first + in_dev - e->frontier_cap) * S, (n - in_dev) * S);
    return 0;
}

int vsr_engine_trace_record(VsrEngine* e, uint64_t local_id, uint64_t* parent_out, uint32_t* cand_out) {
    if (!e->trace || local_id >= e->trace_cap) return VSR_RC_ERROR;
    uint64_t t = 0;
    CK(cudaMemcpy(&t, e->trace + local_id, 8, cudaMemcpyDeviceToHost));
    e->st.bytes_d2h += 8;
    *parent_out = (t >> 12) & GID_MASK;
    *cand_out = (uint32_t)(t & 0xFFF);
    return 0;
}

int vsr_engine_lookup(VsrEngine* e, const void* state, int* level_out, int* owner_out) {
    const ModelOps* ops = e->m->ops;
    uint64_t fp = ops->fingerprint((const uint32_t*)state, e->m->run.use_view);
    if (fp == 0) fp = 1;
    const int owner = e->world > 1 ? owner_of(fp, e->owner_shift) : e->rank;
    if (owner_out) *owner_out = owner;
    *level_out = 0;
    if (owner != e->rank) return 0;
    const uint32_t chk = e->g->check_hash((const uint32_t*)state, e->m->run.use_view);
    unsigned long long* d = (unsigned long long*)&e->ctr->work_next; /* scratch word; counters are reset per level */
    lookup_kernel<<<1, 1, 0, e->stream>>>(e->table, e->table_cap, fp, chk, d);
    CK(cudaGetLastError());
    unsigned long long meta = 0;
    CK(cudaMemcpyAsync(&meta, d, 8, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    *level_out = (int)(meta >> 56);
    return 0;
}

int vsr_engine_reset(VsrEngine* e) {
    if (!e->table_clean) CK(cudaMemsetAsync(e->table, 0, e->table_cap * 16, e->stream)); /* tens of GB: once per run, not twice */
    e->table_clean = true;
    const uint64_t tc = e->st.table_capacity, fc = e->st.frontier_capacity, bt = e->st.bytes_table, bf = e->st.bytes_frontier;
    memset(&e->st, 0, sizeof e->st);
    e->st.table_capacity = tc; e->st.frontier_capacity = fc; e->st.bytes_table = bt; e->st.bytes_frontier = bf;
    e->cur = 0; e->n_cur = 0; e->cur_base = 0; e->next_base = 0; e->level = 0; e->level_open = false;
    e->records_sent = e->records_received = 0;
    e->collected.clear();
    return 0;
}

int vsr_engine_stats(const VsrEngine* e, VsrStats* out) {
    *out = e->st;
    return 0;
}

const char* vsr_engine_last_error(const VsrEngine* e) { return e->last_error; }

/* number of states collected for `level` (1-based) and a copy of them (tests) */
uint64_t vsr_engine_collected(const VsrEngine* e, int level, void* host_out, uint64_t cap_states) {
    if (level < 1 || (size_t)level > e->collected.size()) return 0;
    const std::vector<uint8_t>& v = e->collected[level - 1];
    const uint64_t n = v.size() / e->g->bytes;
    if (host_out && cap_states >= n) memcpy(host_out, v.data(), v.size());
    return n;
}

/* TLC `-simulate`: random walks on the GPU; a violating walk is re-walked on the host (same generator, same step
   function) and returned as a literal behaviour. */
int vsr_simulate(const VsrModel* m, const VsrSimOpts* o, VsrSimStats* out, void* trace_out, uint8_t* trace_actions, size_t trace_cap) {
    if (!m || !o || !out) return VSR_RC_ERROR;
    memset(out, 0, sizeof *out);
    if (!m->gpu) return VSR_RC_CONFIG_ERROR;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return VSR_RC_SYSTEM;
    if (cudaSetDevice(o->device) != cudaSuccess) return VSR_RC_SYSTEM;
    const double t0 = now_s();
    unsigned long long* d = nullptr;
    if (cudaMalloc(&d, 24) != cudaSuccess) return VSR_RC_SYSTEM;
    unsigned long long init[3] = {~0ull, 0, 0};
    cudaMemcpy(d, init, 24, cudaMemcpyHostToDevice);
    SimParams q;
    q.num_walks = o->num_walks;
    q.seed = o->seed;
    q.depth = o->depth > 0 ? o->depth : 100; /* TLC's default simulation depth */
    q.run = m->run;
    q.first_bad = d;
    q.steps = d + 1;
    q.dead_ends = d + 2;
    unsigned long long* dprobe = nullptr;
    uint64_t* dtab = nullptr;
    q.probe_walks = (o->probe_out && o->probe_walks) ? o->probe_walks : 0;
    if (q.probe_walks > o->num_walks) q.probe_walks = o->num_walks;
    if (q.probe_walks) {
        if (cudaMalloc(&dprobe, q.probe_walks * 16) != cudaSuccess || cudaMalloc(&dtab, 8 * 256 * 8) != cudaSuccess) { cudaFree(d); return VSR_RC_SYSTEM; }
        cudaMemcpy(dtab, fp64_table(), 8 * 256 * 8, cudaMemcpyHostToDevice);
    }
    q.probe_out = dprobe;
    q.fp_tab = dtab;
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, o->device);
    cudaEvent_t a, b;
    cudaEventCreate(&a);
    cudaEventCreate(&b);
    cudaEventRecord(a);
    cudaError_t ce = m->gpu->launch_simulate(q, prop.multiProcessorCount * 16, 0);
    cudaEventRecord(b);
    if (ce != cudaSuccess || cudaEventSynchronize(b) != cudaSuccess) { cudaFree(d); return VSR_RC_SYSTEM; }
    float ms = 0;
    cudaEventElapsedTime(&ms, a, b);
    unsigned long long h[3];
    cudaMemcpy(h, d, 24, cudaMemcpyDeviceToHost);
    if (q.probe_walks) cudaMemcpy(o->probe_out, dprobe, q.probe_walks * 16, cudaMemcpyDeviceToHost);
    cudaFree(dprobe);
    cudaFree(dtab);
    cudaFree(d);
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    out->walks = o->num_walks;
    out->steps = h[1];
    out->dead_ends = h[2];
    out->kernel_ms = ms;
    int rc = 0;
    if (h[0] != ~0ull) {
        rc = VSR_RC_VIOLATION;
        out->violating_walk = h[0] >> 16;
        out->violation_depth = (int)(h[0] & 0xFFFF);
        /* re-walk on the host */
        const ModelOps* ops = m->ops;
        std::vector<uint32_t> cands;
        uint32_t cur[VSR_MAX_STATE_BYTES / 4], nxt[VSR_MAX_STATE_BYTES / 4];
        ops->init(cur);
        uint64_t rng = o->seed ^ (out->violating_walk * 0xD1B54A32D192ED03ULL);
        for (int dd = 2; dd <= out->violation_depth; dd++) {
            const int c = ops->random_enabled(&m->run, cur, &rng);
            if (c < 0 || ops->step(&m->run, cur, c, nxt) <= 0) { rc = VSR_RC_ERROR; break; }
            memcpy(cur, nxt, ops->bytes);
            cands.push_back((uint32_t)c);
        }
        if (rc == VSR_RC_VIOLATION && !ops->invariant(&m->run, cur)) rc = VSR_RC_ERROR; /* host and device disagree */
        if (rc == VSR_RC_VIOLATION && trace_out) {
            const int n = vsr_replay_candidates(m, cands.data(), (int)cands.size(), trace_out, trace_actions, trace_cap);
            out->trace_len = n > 0 ? n : 0;
        }
    }
    out->rc = rc;
    out->seconds_total = now_s() - t0;
    return rc;
}

int vsr_probe_bench(int device, uint64_t capacity, uint64_t n, double dup_frac, int iters, double* ms_out) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return VSR_RC_SYSTEM;
    if (capacity < 64 || (capacity & 63)) return VSR_RC_ERROR;
    cudaSetDevice(device);
    uint64_t* table = nullptr;
    unsigned long long* cnt = nullptr;
    if (cudaMalloc(&table, capacity * 16) != cudaSuccess) return VSR_RC_SYSTEM;
    if (cudaMalloc(&cnt, 16) != cudaSuccess) { cudaFree(table); return VSR_RC_SYSTEM; }
    cudaEvent_t a, b;
    cudaEventCreate(&a);
    cudaEventCreate(&b);
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, device);
    const unsigned long long distinct = (unsigned long long)((double)n * (1.0 - dup_frac)) + 1;
    double best = 1e30;
    unsigned long long h[2] = {0, 0};
    for (int it = 0; it < iters + 1; it++) { /* first pass is warm-up */
        cudaMemset(table, 0, capacity * 16);
        cudaMemset(cnt, 0, 16);
        cudaEventRecord(a);
        probe_bench_kernel<<<prop.multiProcessorCount * 8, 256>>>(table, capacity, n, distinct, 1 + it, cnt, cnt + 1);
        cudaEventRecord(b);
        if (cudaEventSynchronize(b) != cudaSuccess) { cudaFree(table); cudaFree(cnt); return VSR_RC_SYSTEM; }
        float ms = 0;
        cudaEventElapsedTime(&ms, a, b);
        if (it > 0 && ms < best) best = ms;
        cudaMemcpy(h, cnt, 16, cudaMemcpyDeviceToHost);
    }
    cudaFree(table);
    cudaFree(cnt);
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    if (ms_out) { ms_out[0] = best; ms_out[1] = (double)h[0]; ms_out[2] = (double)h[1]; }
    return h[0] == (distinct < n ? distinct : n) ? 0 : VSR_RC_ERROR;
}

} /* extern "C" */
