/*
 * vsr_engine.h — internal: the engine object behind the opaque VsrEngine of include/vsr_b200.h, shared by vsr_gpu.cu (the
 * engine's steps: create / seed / step / finish_level / reset), vsr_shard.cu (the exchange between ranks and the level loop
 * vsr_bfs_sharded with its wrappers vsr_bfs / vsr_bfs_multi) and vsr_ckpt.cu (checkpoint / recover).
 */
#ifndef VSR_ENGINE_H
#define VSR_ENGINE_H

#include <stdio.h>
#include <string.h>

#include <chrono>
#include <vector>

#include "vsr_gpu_thunks.cuh"
#include "vsr_group.h"
#include "vsr_thunks.h"

namespace vsr {
inline double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
}

#define CK(call)                                                                                        \
    do {                                                                                                \
        cudaError_t _e = (call);                                                                        \
        if (_e != cudaSuccess) {                                                                        \
            snprintf(e->last_error, sizeof e->last_error, "%s failed: %s", #call, cudaGetErrorString(_e)); \
            return VSR_RC_SYSTEM;                                                                       \
        }                                                                                               \
    } while (0)

struct VsrEngine {
    const VsrModel* m = nullptr;
    const vsr::GpuOps* g = nullptr;
    VsrRunOpts opts;
    int rank = 0, world = 1, owner_shift = 64;
    int device = 0, sms = 0, blocks_per_sm = 1;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    /* device memory */
    uint64_t* table = nullptr;
    uint64_t table_cap = 0;
    uint32_t* frontier[2] = {nullptr, nullptr};
    uint64_t frontier_cap = 0;        /* states per buffer in HBM */
    uint32_t* frontier_host[2] = {nullptr, nullptr}; /* continuation of each buffer in pinned host memory (spill) */
    uint64_t frontier_host_cap = 0;
    uint64_t* trace = nullptr;
    uint64_t trace_cap = 0;
    vsr::DevCounters* ctr = nullptr;
    uint8_t* ties = nullptr;
    uint64_t tie_cap = 0;
    uint64_t* fp_tab = nullptr;
    uint8_t* init_rec = nullptr;
    /* world > 1: the exchange.  inbox = 2 halves x world segments x inbox_cap records; half h, segment s holds what rank s
       pushed here in a step of parity h.  peer_inbox[d] = rank d's inbox as seen from this device (CUDA IPC mapping or a
       peer pointer of the same process); staged mode: stage = world segments of outgoing records a collective moves */
    uint8_t* inbox = nullptr;
    uint64_t inbox_cap = 0;
    uint8_t* peer_inbox[vsr::MAX_WORLD] = {nullptr};
    bool peer_is_ipc[vsr::MAX_WORLD] = {false};
    uint8_t* stage = nullptr;
    VsrGroup* group = nullptr;
    int push_direct = 0;         /* VSR_B200_PUSH=direct */
    /* BFS position */
    int cur = 0;                 /* which frontier buffer is the current level */
    uint64_t n_cur = 0;          /* states in it */
    uint64_t cur_base = 0;       /* local id of its first state */
    uint64_t next_base = 0;      /* local id the next level starts at */
    int level = 0;               /* depth of the current frontier (Init = 1) */
    bool level_open = false;     /* counters reset for the level being generated */
    bool table_clean = false;    /* the seen-set is all zero (since create or reset, nothing inserted): reset skips the memset */
    VsrStats st;
    double level_ms_acc = 0;
    double level_ms_insert_acc = 0; /* the part of level_ms_acc spent in launches that only insert records from peers */
    uint64_t records_sent = 0, records_received = 0;
    std::vector<std::vector<uint8_t>> collected; /* per level states (collect_levels) */
    char last_error[256] = {0};
};

int engine_reset_level(VsrEngine* e);
void fill_params(VsrEngine* e, vsr::ExpandParams& p);

#endif
