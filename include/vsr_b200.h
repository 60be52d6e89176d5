/*
 * vsr_b200.h — C ABI of the B200-native explicit-state model checker for
 * vsr-revisited/paper/VSR.tla (reference: Vanlightly/vsr-tlaplus @ 7566e8af).
 *
 * What this replaces.  The reference has no plugin/operator ABI: TLA+ has no FFI and the path
 * "model-check VSR.tla under VSR.cfg" is executed by the external TLC tool
 *     java -cp tla2tools.jar tlc2.TLC [-deadlock] [-workers N] [-fp N] [-dumpTrace tlc F] -config VSR.cfg VSR.tla
 * so the drop-in boundary is TLC's file + CLI surface (SURVEY §8b).  Each entry point below cites
 * the part of the reference it stands in for.  Plain pointers and sizes; caller owns every buffer;
 * no torch / C++ types.  Return codes follow TLC's exit statuses where one exists:
 *     0 ok, 11 deadlock, 12 safety (invariant) violation, 150 spec error, 151 config error,
 *     152 state space too large for the configured capacity, 153 system (CUDA) error, 255 other.
 */
#ifndef VSR_B200_H
#define VSR_B200_H

#include <stddef.h>
#include <stdint.h>

#include "vsr_flat.h"

#ifdef __cplusplus
extern "C" {
#endif

#define VSR_RC_OK 0
#define VSR_RC_DEADLOCK 11
#define VSR_RC_VIOLATION 12
#define VSR_RC_SPEC_ERROR 150
#define VSR_RC_CONFIG_ERROR 151
#define VSR_RC_TOO_LARGE 152
#define VSR_RC_SYSTEM 153
#define VSR_RC_ERROR 255

#define VSR_MAX_STATE_BYTES 256

typedef struct VsrModel VsrModel; /* opaque: parsed config + selected packed layout */

typedef struct VsrModelInfo {
    int32_t replica_count, client_count, value_count;   /* VSR.cfg:4-6 */
    int32_t start_view_on_timer_limit, restart_empty_limit; /* VSR.cfg:7-8 */
    int32_t symmetry, view;                             /* SYMMETRY symmValues / VIEW view present (VSR.cfg:29,31) */
    int32_t invariant;                                  /* bitmask of INVARIANT names (VSR.cfg:36-39): 1 AcknowledgedWriteNotLost
                                                           2 AcknowledgedWritesExistOnMajority 4 NoLogDivergence 8 TestInv */
    int32_t state_bytes;                                /* size of one packed state */
    int32_t state_bits;                                 /* bits in use */
    int32_t num_candidates;                             /* (action, binding) pairs tried per state */
    int32_t spec_verified;                              /* 1 if a .tla was given and matched VSR.tla's structure */
    uint64_t spec_hash;                                 /* FNV-1a 64 of the .tla bytes (0 if none) */
    char value_names[VSR_MAX_V][32];                    /* model values of Values, cfg order */
    int32_t check_deadlock;                             /* CHECK_DEADLOCK in the cfg: 1 TRUE, 0 FALSE, -1 absent (TLC's default: check) */
    int32_t _pad;
} VsrModelInfo;

/* ---- loading: TLC's `-config VSR.cfg VSR.tla` (SURVEY §8b; grammar of vsr-revisited/paper/VSR.cfg:1-39).
 * tla_path may be NULL (the spec is hand-lowered; when given, it is verified to BE VSR.tla: module
 * name :1, the 20 VARIABLES :119-138, the 19 disjuncts of Next :896-918).  On failure returns
 * 150/151 and writes a message to err.
 * Constants: ReplicaCount 2..7, |Values| 1..7, StartViewOnTimerLimit 0..14, ClientCount 1, RestartEmptyLimit 0.  The
 * packed layouts of the reference's configurations and their neighbours are built in; any other combination is
 * compiled on first use into <library dir>/layouts/ (needs nvcc; VSR_B200_JIT=0 turns that into a 151). */
int vsr_load(const char* cfg_path, const char* tla_path, VsrModel** out, char* err, size_t errcap);
/* same, from the text of a cfg file */
int vsr_load_cfg_text(const char* cfg_text, const char* tla_path, VsrModel** out, char* err, size_t errcap);
/* same, straight from constants (CONSTANTS of VSR.tla:92-96) */
int vsr_model_create(int replica_count, int client_count, int value_count, int start_view_on_timer_limit,
                     int restart_empty_limit, int symmetry, int view, int invariant, VsrModel** out, char* err,
                     size_t errcap);
void vsr_model_free(VsrModel* m);
int vsr_model_info(const VsrModel* m, VsrModelInfo* out);

/* ---- single-state operations on packed states (host; re-entrant).  A packed state is
 * info.state_bytes bytes, 16-byte aligned. */
int vsr_init(const VsrModel* m, void* state_out);                        /* Init, VSR.tla:323-348 */
/* Next, VSR.tla:896-918: writes up to cap successors (state_bytes apart) in TLC's binding order,
 * action_ids[i] = VSR_ACT_*, mult[i] = TLC bindings that successor stands for; returns the number
 * of successors, or a negative E_* code if one cannot be represented. */
int vsr_successors(const VsrModel* m, const void* state, void* out, size_t cap, uint8_t* action_ids, uint32_t* mult);
/* candidate (action, binding) indices whose guard holds in `state`, in the order vsr_successors emits them.  Evaluates the
 * guards in both of their forms (one candidate at a time, and the register-mask form of the GPU scan); -100 if they
 * ever disagree */
int vsr_enabled_candidates(const VsrModel* m, const void* state, uint32_t* out, size_t cap);
int vsr_canon(const VsrModel* m, void* state);                           /* SYMMETRY representative, VSR.tla:151 */
uint64_t vsr_fingerprint(const VsrModel* m, const void* state);          /* FP64 of the VIEW projection, VSR.tla:149-150 */
/* the same fingerprint by its byte-at-a-time definition (vsr_fingerprint and the GPU use the slicing-by-8 form) */
uint64_t vsr_fingerprint_bytewise(const VsrModel* m, const void* state);
uint32_t vsr_aux_key(const VsrModel* m, const void* state);
/* rank (GPU) that owns a fingerprint when the state space is sharded over `world` = 1, 2, 4 or 8 ranks: the high bits of
 * fingerprint x an odd constant (FP64 is GF(2)-linear: its own high bits would route a rank's successors to a few peers only) */
int vsr_owner_rank(uint64_t fingerprint, int world);
int vsr_invariant(const VsrModel* m, const void* state);                 /* 0 = all hold, else mask bit of the violated one; VSR.tla:926-952 */
int vsr_unpack(const VsrModel* m, const void* state, VsrFlatState* out);
int vsr_pack(const VsrModel* m, const VsrFlatState* in, void* state_out);
/* TLC value text of one state, format of state_transfer_violation_trace.txt (variables
 * alphabetical, records in first-interned field order); returns length or -needed. */
int vsr_state_to_tla(const VsrModel* m, const void* state, char* buf, size_t cap);
int vsr_flat_to_tla(const VsrModel* m, const VsrFlatState* f, char* buf, size_t cap);
const char* vsr_action_name(int action_id);
/* "line A, col B to line C, col D of module VSR" for an action when a .tla was loaded, else "Unknown location" */
int vsr_action_location(const VsrModel* m, int action_id, char* buf, size_t cap);

/* ---- the BFS (TLC's worker loop; SURVEY §3.1, stages E1-E9) on the GPU */
typedef struct VsrRunOpts {
    int32_t device;              /* CUDA device ordinal */
    int32_t check_deadlock;      /* TLC default is on; `-deadlock` turns it off.  Here default 0 (VSR has terminal states) */
    int32_t max_depth;           /* TLC `-depth`-like bound for BFS (0 = none) */
    int32_t stop_on_violation;   /* 1: stop at the first violating level (TLC behaviour) */
    int32_t keep_trace;          /* 1: keep (parent, binding) per distinct state so a counterexample can be rebuilt */
    int32_t verbose;
    uint64_t table_capacity;     /* seen-set slots (any number, rounded up to 64; 0 = auto from free memory) */
    uint64_t frontier_capacity;  /* states per frontier buffer (0 = auto) */
    uint64_t max_states;         /* stop after the level that crosses this many distinct states (0 = none) */
    double max_seconds;          /* stop after the level that crosses this much time (0 = none) */
    int32_t collect_levels;      /* 1: keep every level's states on the host (tests) */
    int32_t _reserved0;
    /* frontier spill (BASELINE configs[3], "spill to pinned host DRAM"): each of the two frontier buffers continues, after
       its frontier_capacity states in HBM, with this many states in pinned host memory mapped into the device; the kernels
       write and read that part over PCIe / C2C.  0 = no spill: a level that does not fit is a 152. */
    uint64_t frontier_host_capacity;
    /* checkpoint / recover: TLC's `-checkpoint <minutes>` and `-recover <dir>` (the reference's .gitignore:1 ignores TLC's
       states/ metadir, i.e. its users run with checkpoints).  checkpoint_path: file written at the first level boundary after
       checkpoint_seconds since the last one (0 = after every level; written to <path>.tmp and renamed, so an interrupted write
       leaves the previous checkpoint intact); recover_path: continue the BFS from that file instead of Init.  One rank uses
       <path> itself; with several ranks every rank uses <path>.rank<r>.  NULL = off. */
    const char* checkpoint_path;
    const char* recover_path;
    double checkpoint_seconds;
} VsrRunOpts;

#define VSR_MAX_LEVELS 512
typedef struct VsrStats {
    uint64_t generated, distinct, queue;  /* TLC's "N states generated, M distinct states found, Q left on queue" */
    int32_t depth;                        /* TLC's "depth of the complete state graph search" (Init = 1) */
    int32_t rc;
    int32_t complete;
    int32_t num_levels;
    uint64_t level_sizes[VSR_MAX_LEVELS];
    uint64_t level_generated[VSR_MAX_LEVELS];
    double level_ms[VSR_MAX_LEVELS];      /* device time of each level's kernels (CUDA events) */
    uint64_t h2_ties;                     /* same-level VIEW ties with different aux variables */
    uint64_t fp_collisions;               /* equal 64-bit fingerprints told apart by the check hash */
    uint64_t probe_total;                 /* table slots inspected */
    uint64_t kernel_launches;
    double seconds_total, seconds_kernels;
    int32_t violation_level;              /* depth of the violating state */
    int32_t trace_len;
    int32_t error_code;                   /* first E_* raised on the device (0 = none) */
    int32_t violation_mask;               /* INVARIANT bits violated by the reported state (0 = none reported) */
    uint64_t violation_id;
    uint64_t table_capacity, frontier_capacity;
    uint64_t bytes_table, bytes_frontier;
    uint64_t bytes_h2d, bytes_d2h;         /* host<->device bytes moved by the engine (inputs, per-level counters, trace reads) */
    double seconds_setup;                 /* engine creation: allocation + clearing the seen-set */
    uint64_t records_sent, records_received; /* several GPUs: records this rank pushed to / drained from peers */
    double seconds_insert;                /* several GPUs: part of seconds_kernels spent in drain-only launches */
    int32_t levels_expanded;              /* frontiers expanded = valid entries of level_generated / level_ms */
    int32_t _pad;
} VsrStats;

typedef struct VsrEngine VsrEngine;

/* One-call BFS on one GPU: a world-1 engine running vsr_bfs_sharded.  Fails loudly (153) when no CUDA device is usable —
 * there is no CPU fallback; a run that fails (CUDA, checkpoint file) returns its status with *stats all zero but rc.
 * If trace_out != NULL and a violation/deadlock is found, writes the counterexample (packed states, trace_cap capacity)
 * with its action ids; stats.trace_len is its length. */
int vsr_bfs(const VsrModel* m, const VsrRunOpts* opts, VsrStats* stats, void* trace_out, uint8_t* trace_actions,
            size_t trace_cap);

/* Stepwise engine (what vsr_bfs_sharded, and through it vsr_bfs, is made of).
 * rank/world: this engine owns the fingerprints f with owner(f) == rank (world = 1, 2, 4 or 8: the high bits of f). */
int vsr_engine_create(const VsrModel* m, const VsrRunOpts* opts, int rank, int world, VsrEngine** out, char* err,
                      size_t errcap);
void vsr_engine_destroy(VsrEngine* e);
/* bytes of one record that travels between ranks or into vsr_engine_insert_records: the packed state, then
 * { uint64 fingerprint; uint64 parent global id << 12 | candidate index | mult << 56 } */
int vsr_engine_record_bytes(const VsrEngine* e);
int vsr_engine_seed_init(VsrEngine* e);                       /* inserts Init if this rank owns it */
/* one launch of the wavefront kernel over the whole current frontier (world = 1: that is the level) */
int vsr_engine_expand(VsrEngine* e);
/* world > 1, one step = one launch: expand frontier states [first, first + count) — successors owned here are inserted,
 * the others are stored into their owners' inboxes (half `parity` of the double buffer) by the kernel itself — then insert
 * the records the peers stored HERE in the previous step: drain_counts[s] from rank s (NULL = none).  sent_out[d] = records
 * this launch pushed to rank d (tell rank d: it is its drain_counts[this rank] of the next step).  Returns after the
 * kernel has completed, i.e. after the pushed records have landed. */
int vsr_engine_step(VsrEngine* e, uint64_t first, uint64_t count, int parity, const uint32_t* drain_counts, uint32_t* sent_out);
/* inserts records (device pointer, layout above) as states of the level being generated (Init; tests) */
int vsr_engine_insert_records(VsrEngine* e, const void* dev_records, uint64_t n);
/* finishes the level: resolves ties, swaps frontiers; writes this rank's level numbers */
typedef struct VsrLevelInfo {
    uint64_t new_states, generated, frontier_in, ties, collisions;
    int32_t violation, deadlock, error_code, overflow;
    uint64_t violation_id, deadlock_id;
    double ms;        /* kernel time of the level on this rank (expand + insert), CUDA events on the launch stream */
    double ms_insert; /* of which launches that only inserted records received from peers */
    int32_t violation_mask, _pad; /* INVARIANT bits (VsrModelInfo.invariant) violated by some new state of the level */
} VsrLevelInfo;
int vsr_engine_finish_level(VsrEngine* e, VsrLevelInfo* out);
uint64_t vsr_engine_frontier_size(const VsrEngine* e);
/* copies `n` states of the current frontier starting at `first` to a host buffer */
int vsr_engine_read_frontier(VsrEngine* e, uint64_t first, uint64_t n, void* host_out);
/* trace record of a locally owned state id: parent global id (rank << 40 | local id; 2^44 - 1 = none: Init) and candidate index */
int vsr_engine_trace_record(VsrEngine* e, uint64_t local_id, uint64_t* parent_out, uint32_t* cand_out);
int vsr_engine_stats(const VsrEngine* e, VsrStats* out);
/* membership query: *level_out = BFS depth at which `state` (a canonical packed state) was first seen, 0 if it is not
 * in this rank's shard of the seen-set; *owner_out = the rank owning its fingerprint */
int vsr_engine_lookup(VsrEngine* e, const void* state, int* level_out, int* owner_out);
/* Checkpoint of this rank's shard at a level boundary (after vsr_engine_finish_level, before the next expansion): the
 * current frontier, every seen-set entry {fingerprint, meta}, the trace records and the run's statistics, to one file.
 * vsr_engine_recover loads it into a fresh (or reset) engine of the same model, rank and world; the seen-set is re-inserted
 * entry by entry, so its capacity may differ from the one the checkpoint was written with.  `totals` (may be NULL) travels
 * with the file: vsr_bfs / vsr_bfs_sharded store the job's running totals there.  150 = not a checkpoint of this model. */
int vsr_engine_checkpoint(VsrEngine* e, const char* path, const VsrStats* totals);
int vsr_engine_recover(VsrEngine* e, const char* path, VsrStats* totals_out);
/* forget everything explored (clears the seen-set unless nothing was inserted since create or the last reset, keeps the
 * allocations): ready for seed_init again */
int vsr_engine_reset(VsrEngine* e);
const char* vsr_engine_last_error(const VsrEngine* e);
/* with opts.collect_levels: number of states first seen at depth `level` (1-based) and, if host_out has room, a copy */
uint64_t vsr_engine_collected(const VsrEngine* e, int level, void* host_out, uint64_t cap_states);

/* ---- several GPUs of one node (SURVEY §8e: TLC's `-workers` / distributed mode).  One rank per GPU — processes
 * (torchrun) or threads of one process — fingerprint space split by its high bits.  The ranks coordinate through a
 * VsrGroup: a block of shared memory with a barrier and an all-gather of one small message per rank (a few per wavefront,
 * about a microsecond each).  The states do not pass through it: expand_kernel stores a successor owned by a peer straight
 * into that peer's inbox over NVLink (CUDA IPC mapping / peer access) and the peer inserts it in its next launch. */
typedef struct VsrGroup VsrGroup;
#define VSR_GROUP_MSG_BYTES 256
/* processes: `name` is a POSIX shared-memory name ("/vsr-<job>") every rank of the job passes and nobody else uses; rank 0
 * creates it, the others wait for it up to timeout_s; the name is unlinked once all have attached */
int vsr_group_open(const char* name, int rank, int world, double timeout_s, VsrGroup** out, char* err, size_t errcap);
/* threads of one process: `world` handles on one heap block */
int vsr_group_open_local(int world, VsrGroup** out_handles);
void vsr_group_close(VsrGroup* g);
int vsr_group_barrier(VsrGroup* g);                                  /* 0, or 153 when a rank aborted / timed out */
int vsr_group_allgather(VsrGroup* g, const void* mine, size_t bytes, void* all_out); /* bytes <= VSR_GROUP_MSG_BYTES */
void vsr_group_abort(VsrGroup* g);                                   /* make every pending and future wait fail */
void vsr_group_set_timeout(VsrGroup* g, double seconds);
int vsr_group_rank(const VsrGroup* g);
int vsr_group_world(const VsrGroup* g);
const char* vsr_group_last_error(const VsrGroup* g);
/* collective over the group: allocate this rank's inbox (2 halves x world segments x inbox_records records; 0 = default
 * from the frontier capacity) and map every peer's.  153 with a message if peer memory is unavailable. */
int vsr_engine_attach_group(VsrEngine* e, VsrGroup* g, uint64_t inbox_records);
/* the same kernels with the outgoing records in a LOCAL staging buffer (world segments of inbox_records records, destination
 * major) for a host that moves them with its own collective: segment d of *stage_out goes to segment <this rank> of half
 * `parity` of rank d's *inbox_out (2 halves x world segments).  Used by dist.ShardedBfs (torch.distributed all-to-all). */
int vsr_engine_attach_staged(VsrEngine* e, uint64_t inbox_records, void** stage_out, void** inbox_out, uint64_t* cap_out);
int vsr_engine_detach(VsrEngine* e);                                 /* collective when attached to a group */
uint64_t vsr_engine_default_inbox_records(const VsrEngine* e);
/* The whole BFS, called by every rank of the group with the same opts — or on a world-1 engine, which needs no group; all
 * ranks return the same rc and the same totals (records_sent / received, bytes_* and kernel_launches are this rank's).
 * part_states = frontier states per rank and step (0 = from the inbox size; one rank expands its whole frontier in one
 * step).  On a violation / deadlock trace_cands[0 .. *trace_len) is the candidate chain from Init, walked across ranks:
 * vsr_replay_candidates turns it into the literal behaviour.  *stats is written when the search reaches a verdict; a run
 * that fails (CUDA, the group, a checkpoint file) returns its status and leaves *stats untouched. */
int vsr_bfs_sharded(VsrEngine* e, const VsrRunOpts* opts, uint64_t part_states, VsrStats* stats, uint32_t* trace_cands, int* trace_len,
                    size_t trace_cap);
/* `vsrmc -gpus N`: the same from ONE process, one thread per GPU (devices opts->device ... + ngpus - 1) */
int vsr_bfs_multi(const VsrModel* m, const VsrRunOpts* opts, int ngpus, uint64_t inbox_records, uint64_t part_states, VsrStats* stats,
                  void* trace_out, uint8_t* trace_actions, size_t trace_cap, char* err, size_t errcap);

/* Host replay helper for multi-rank traces: given a chain of candidate indices from Init, re-executes
 * them (canonicalising as the engine does) and writes the literal states. */
int vsr_replay_candidates(const VsrModel* m, const uint32_t* cands, int n, void* trace_out, uint8_t* trace_actions,
                          size_t trace_cap);

/* ---- simulation mode: TLC `-simulate [-depth N]` (the reference's README.md:22 recommends it for the defect).
 * num_walks random behaviours from Init of at most `depth` states (TLC's default 100), uniformly random among the
 * enabled (action, binding) pairs at every step, invariant checked on every state; one GPU thread per walk.  Returns 12
 * and the violating behaviour (literal value names, re-walked on the host) if one walk hits a violation. */
typedef struct VsrSimOpts {
    int32_t device, depth;
    uint64_t num_walks, seed;
    uint64_t probe_walks;   /* optional cross-check: for walks 0 .. probe_walks-1 the device reports ... */
    uint64_t* probe_out;    /* ... [2w] = bytewise FP64 of the walk's last state (all words), [2w+1] = transitions taken; NULL = off */
} VsrSimOpts;
typedef struct VsrSimStats {
    uint64_t walks, steps, dead_ends, violating_walk;
    int32_t rc, violation_depth, trace_len, _pad;
    double kernel_ms, seconds_total;
} VsrSimStats;
int vsr_simulate(const VsrModel* m, const VsrSimOpts* opts, VsrSimStats* out, void* trace_out, uint8_t* trace_actions,
                 size_t trace_cap);

/* the same walk on the host (walk index `walk` of vsr_simulate with this seed): chosen candidate indices, number of
 * transitions, and the depth of the first violating state (0 = none) */
int vsr_walk(const VsrModel* m, uint64_t seed, uint64_t walk, int depth, uint32_t* cands_out, int* violated_at);

/* seen-set micro-benchmark (SURVEY §8d): inserts n splitmix64 keys (a fraction dup_frac of them repeats) into a fresh
 * table of `capacity` slots (power of two) with the BFS's own insert routine; best of `iters` launches.
 * out[0] = device ms per launch, out[1] = keys found new (must equal the number of distinct keys), out[2] = slots probed. */
int vsr_probe_bench(int device, uint64_t capacity, uint64_t n, double dup_frac, int iters, double* out);

const char* vsr_version(void);

#ifdef __cplusplus
}
#endif
#endif /* VSR_B200_H */
