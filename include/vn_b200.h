/*
 * vn_b200.h - C ABI of the B200-native cached-graph navigation hot path (libvn_b200.so).
 *
 * The reference (felipefelixarias/a2cat-vn-pytorch) is pure Python and has NO plugin / FFI surface
 * for this path; its seam is the gym Env / baselines-style VecEnv duck type built in
 * experiments/thor_cached_auxiliary.py:58-71.  This header is therefore the boundary a Python
 * VecEnv (ours: a2cat-vn-pytorch_b200/vec_env.py, bound with ctypes) or any other host binds to.
 * Each entry point names the reference code it replaces (paths relative to the reference root).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; no exceptions cross the boundary.
 *   - every function returns 0 on success or a negative VN_E* code; vn_last_error() returns a
 *     thread-local human-readable message for the last failure on the calling thread.
 *   - all data pointers are CALLER-OWNED DEVICE pointers (e.g. torch tensor.data_ptr()) unless
 *     marked [host]; the descriptor structs themselves are read on the host during the call.
 *   - no allocation, no implicit synchronisation: kernels are enqueued on the caller's
 *     cudaStream_t (passed as void*; NULL = legacy default stream) and the call returns.
 *   - re-entrant.  The global state is: the thread-local error string, a launch counter kept for
 *     statistics (vn_launch_count), the development trace buffer of vn_debug_gather_trace, per-device
 *     caches of the SM count and of the dynamic shared-memory limit set on each kernel, and a
 *     per-thread cache of host pointers already found pinned and device-mapped.  No environment
 *     variable is read: how a call runs follows from its arguments and the device alone.
 *
 * State numbering: oriented scenes use state = free_cell_rank * 4 + rotation (the numbering of
 * graph/util.py:208-210,229-237 save_graph_as_h5), un-oriented ones state = free_cell_rank; with
 * several scenes resident the indices are global (scene_base + local).
 */
#ifndef VN_B200_H
#define VN_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VN_ABI_VERSION 6
#define VN_MAX_PLANES 6 /* rgb, depth, segmentation (+ the 3 third-person planes of graph/thor_graph.py:25-31) */

/* error codes */
#define VN_OK 0
#define VN_EINVAL (-1)    /* bad argument (null pointer, size, alignment) */
#define VN_ECUDA (-2)     /* CUDA runtime error at launch */
#define VN_EUNSUPPORTED (-3)

/* vn_rules_t.flags */
#define VN_RULE_COLLISION_SKIPS_GOAL 0x01 /* gym_graph/graph.py:69-72: collision returns before the goal test */
#define VN_RULE_NEG_STEP_REWARD 0x02      /* gym_ai2thor/envs/cached.py:84: reward = -cfg[1] */
#define VN_RULE_COLLISION_OVERRIDES 0x04  /* cached.py:87-88: collided reward overrides the terminal reward */
#define VN_RULE_TERM_PREV_OBS 0x08        /* cached.py:90-97: terminal step returns the previous observation */
#define VN_RULE_TWO_LEVEL 0x10            /* graph/util.py:103-116: 0.9 / 0.1 curriculum buckets */
#define VN_RULE_NOOP_ACTION 0x20          /* graph/env.py:118-120: action -1 is a no-op with reward 0.0 */
#define VN_RULE_AUTO_RESET 0x40           /* baselines VecEnv worker: if done: ob = env.reset() */

/* vn_step_out_t.flags */
#define VN_STEP_ACTIONS_READY 0x01 /* the caller guarantees that the action buffer was complete before the PREVIOUS
                                      call's gather was enqueued (e.g. a pre-computed action stream, or host actions
                                      written after the previous ready_event): with gather_desc set, the scalar
                                      kernel then overlaps the previous gather instead of waiting for it */
#define VN_STEP_NO_OVERLAP 0x04 /* with VN_STEP_ACTIONS_READY: the step is still part of a pipelined loop (which decides how
                                   VN_GATHER_AUTO runs it) but must NOT overlap the launch before it - that launch was not the
                                   gather half of these envs' previous two-kernel step (it was a reset, a one-launch step, a
                                   graph replay, ...) and may still be writing the env state this step reads */
#define VN_STEP_SKIP_UNCHANGED 0x02 /* the caller guarantees that out->obs[] are the SAME buffers as in the previous
                                       reset / step call on these envs and that nothing else wrote to them: the row of
                                       an env whose record did not change (collision, no-op action) is then not copied
                                       again - the reference returns the same frame view in that case
                                       (gym_graph/graph.py:69-72).  Honoured when gather_desc is set or the launch is
                                       fused; out->obs_state must persist between calls.  Counted in
                                       VN_STAT_ROWS_SKIPPED. */

/* vn_rules_t.goal_compare */
#define VN_GOAL_FULL 0     /* gym_graph/graph.py:60-61 position and rotation; cached.py:83 index equality */
#define VN_GOAL_POSITION 1 /* position only (state >> 2) */
#define VN_GOAL_NEVER 2    /* graph/env.py:61 as written: never true (SURVEY.md A4) */

/* indices into the device statistics vector (vn_step_out_t.stats, uint64 each; [1] is a double) */
#define VN_STAT_EPISODES 0
#define VN_STAT_RETURN_SUM 1 /* double, bit pattern stored in the uint64 slot */
#define VN_STAT_LENGTH_SUM 2
#define VN_STAT_SUCCESSES 3
#define VN_STAT_COLLISIONS 4
#define VN_STAT_STEPS 5
#define VN_STAT_TRUNCATIONS 6
#define VN_STAT_RESETS 7
#define VN_STAT_ROWS_SKIPPED 8 /* observation rows not re-copied under VN_STEP_SKIP_UNCHANGED */
#define VN_N_STATS 9

/* The cached-observation store resident in HBM.  Replaces the numpy arrays
 * ThorGridWorld._observations/_depths/_segmentations [X,Y,4,H,W,C] (graph/multi_graph_no_tp.py:6-25,
 * 141-144) and the h5 'observation' dataset (graph/util.py:224): one record per state holding all
 * planes, record pitch and plane offsets multiples of 128 B, plane sizes multiples of 16 B: plane_bytes is
 * H * W * C rounded up to 16 (84 x 84 frames need no rounding, the reference's native 174 x 174 ones get 4 / 12
 * padding bytes), and the rows of an observation batch are plane_bytes apart as well. */
typedef struct vn_store {
    const uint8_t *base;               /* [n_states][state_pitch] */
    int64_t state_pitch;
    int32_t n_states;
    int32_t n_planes;
    int32_t plane_off[VN_MAX_PLANES];
    int32_t plane_bytes[VN_MAX_PLANES];
} vn_store_t;

/* Transition + reset tables.  adj replaces graph.util.step + is_valid_state (graph/util.py:15-37)
 * and the h5 'graph' dataset (graph/util.py:212-233); the candidate lists replace the per-reset
 * Python loops of sample_initial_state / sample_initial_position (graph/util.py:88-143). */
typedef struct vn_tables {
    const int32_t *adj;           /* [n_states][4] next state, -1 = collision */
    const int32_t *task_goal;     /* [n_tasks] goal state */
    const int32_t *task_cand_off; /* [n_tasks + 1] CSR offsets into cand_state */
    const int32_t *task_prefix;   /* [n_tasks] number of leading candidates eligible under the curriculum */
    const int32_t *cand_state;    /* candidates of each task sorted by curriculum distance */
    int32_t n_states;
    int32_t n_tasks;
} vn_tables_t;

/* Per-env mutable state (struct of arrays, n_envs each). */
typedef struct vn_envs {
    int32_t n_envs;
    int32_t env_id_base;     /* global id of env 0 of this shard: keys the RNG so results do not depend on sharding */
    int32_t *state;
    int32_t *goal;           /* goal state of the current episode */
    int32_t *task;           /* task of the current episode */
    int32_t *elapsed;        /* steps since reset (gym TimeLimit) */
    uint32_t *epoch;         /* resets so far = RNG counter = index into the injected stream */
    float *ep_return;        /* RewardCollector accumulators */
    int32_t *ep_length;
    const int32_t *task_lo;  /* [n_envs] first task this env may draw (gym_graph/graph.py:47 goals list) */
    const int32_t *task_cnt; /* [n_envs] number of tasks it draws from */
} vn_envs_t;

typedef struct vn_rules {
    float reward_goal, reward_step, reward_collision; /* rewards = [1.0, 0.0, 0.0] gym_graph/graph.py:10 */
    int32_t max_episode_steps;                        /* gym TimeLimit; <= 0 disables */
    int32_t goal_compare;
    int32_t flags;
    int32_t n_actions;                                /* 4 */
    int32_t reserved;
    uint64_t seed;
} vn_rules_t;

/* Optional injected reset stream (parity runs): reset k of env i uses task_lo[i] + task[i*stride + k]
 * and start state start[i*stride + k] instead of the Philox draw.  NULL pointers = Philox. */
typedef struct vn_inject {
    const int32_t *task;
    const int32_t *start;
    int32_t stride;
    int32_t reserved;
} vn_inject_t;

/* One float observation leaf (see vn_gather_leaves_f32_chw and vn_step_out_t.float_leaves). */
typedef struct vn_float_leaf {
    int32_t plane;
    int32_t source;   /* 0 observation record, 1 goal record */
    int32_t channels; /* 1 or 3 */
    int32_t reserved;
    float *out;       /* [n][channels][h][w] */
} vn_float_leaf_t;

/* Outputs of one vectorised step.  Any pointer may be NULL to skip that output. */
typedef struct vn_step_out {
    uint8_t *obs[VN_MAX_PLANES];      /* [n_envs][plane_bytes[p]] observation batch, rows plane_bytes[p] apart */
    uint8_t *goal_obs[VN_MAX_PLANES]; /* persistent goal batch: rows rewritten only for envs that reset */
    float *reward;                    /* [n_envs] */
    uint8_t *done;                    /* [n_envs] env done OR time-limit */
    uint8_t *truncated;               /* [n_envs] gym TimeLimit: 0 limit not reached (no info key), 1 info['TimeLimit.truncated']
                                         = True, 2 limit reached on a step that was terminal anyway (= False) */
    uint8_t *win;                     /* [n_envs] info['win'] */
    uint8_t *did_reset;               /* [n_envs] */
    float *last_action_reward;        /* [n_envs][n_actions + 1] UnrealEnvBaseWrapper vector */
    float *episode_return;            /* [n_envs] info['episode']['r'], valid where done */
    int32_t *episode_length;          /* [n_envs] info['episode']['l'], valid where done */
    int32_t *info_state;              /* [n_envs] info['state']: state after the move, before auto-reset */
    int32_t *obs_state;               /* [n_envs] state whose frames were gathered (scratch, required) */
    uint64_t *stats;                  /* [VN_N_STATS] running sums, see VN_STAT_* */
    int32_t *gather_desc;             /* optional scratch [2][n_envs][2] int32: double-buffered (record, goal record or -1)
                                         descriptors handed from the scalar half to the gather half of step `parity` */
    int32_t parity;                   /* step counter (only bit 0 is used); the caller increments it every reset / step */
    int32_t flags;                    /* VN_STEP_* */
    uint32_t *sched;                  /* optional scratch of 4 uint32, zeroed once by the caller: [parity & 1] is the ticket
                                         counter of this step's gather (zeroed by the step's scalar half, so
                                         vn_env_gather runs exactly ONCE after each vn_env_step_scalar), [2] the arrival
                                         counter of the persistent launch's host signal (self re-arming), [3] reserved; one
                                         scratch per env batch / stream */
    uint8_t *host_pack;               /* optional MAPPED PINNED HOST block of 20 * n_envs bytes ("host pack") that the
                                         scalar kernel also writes, n = n_envs:
                                           [0, 4n) reward f32 | [4n, 8n) episode_return f32 | [8n, 12n) episode_length i32
                                           | [12n, 16n) info_state i32 | [16n, 17n) done | [17n, 18n) truncated
                                           | [18n, 19n) win | [19n, 20n) did_reset */
    uint32_t *host_seq;               /* optional MAPPED PINNED HOST words, one per thread block of the scalar half
                                         (vn_env_host_seq_words of them): a block stores `seq` into its word once the scalars
                                         of ITS envs are in host_pack (system-scope fence first); the host polls the words
                                         with vn_host_wait_seq instead of waiting on an event - no stream operation between
                                         the two halves, so the gather stays programmatically chained to the scalar half */
    uint32_t seq;                     /* value to store; the caller changes it every call */
    uint32_t reserved;
    /* Optional rollout record of this step, [n_envs] each, typically row t of a caller-owned [T, n_envs] rollout
     * storage (deep_rl RolloutStorage.insert): written by the step itself instead of by copy kernels afterwards. */
    int32_t *rec_action;              /* the action taken */
    float *rec_reward;                /* = reward */
    uint8_t *rec_done;                /* = done */
    int32_t *rec_state;               /* state whose frames the NEXT observation shows (= obs_state, post auto-reset) */
    int32_t *rec_goal;                /* goal state of the next observation's episode */
    /* Optional float observation mode (TransposeImage + ScaledFloatFrame, thor_cached_auxiliary.py:61-62, as part of the
     * step): after the scalar half (and the uint8 gather, if obs[] are set) vn_env_reset / vn_env_step /
     * vn_env_step_host* enqueue ONE more kernel that converts the records named by this step's descriptors into the
     * persistent float32 CHW batches of these leaves (rows whose record did not change - and goal rows of envs that
     * did not reset - keep their content).  Same restrictions as vn_gather_leaves_f32_chw; needs gather_desc. */
    const vn_float_leaf_t *float_leaves; /* [host] n_float_leaves descriptors, read during the call; NULL = off */
    int32_t n_float_leaves;
    int32_t float_h, float_w;         /* frame geometry of the leaves */
    int32_t reserved2;
} vn_step_out_t;

/* gather kernel variants (all bit-identical; see DESIGN.md) */
#define VN_GATHER_AUTO 0
#define VN_GATHER_LDG 1      /* 16-byte vector loads/stores through registers */
#define VN_GATHER_BULK 2     /* cp.async.bulk (TMA engine) global->shared->global, mbarrier-tracked */
#define VN_GATHER_FUSED 3    /* vn_env_reset / vn_env_step / vn_env_step_host as ONE launch (CTA per env: scalar half, then
                                bulk copies); what VN_GATHER_AUTO picks for batches that fit in one wave of CTAs (as many
                                envs per SM as shared memory holds records, at most 4), where the step is bound by launch
                                latency.  Elsewhere it means VN_GATHER_BULK. */
#define VN_GATHER_PERSISTENT 4 /* vn_env_reset / vn_env_step / vn_env_step_host as ONE launch for batches of any size: a
                                persistent grid of one-warp CTAs, each owning a fixed set of envs - its lanes step them,
                                then lane 0 moves their records with bulk copies.  Needs out->gather_desc and out->sched
                                and plane sets of at most 52 KB per env; a host caller polls ONE host_seq word.  In the
                                gather-only entry points it means VN_GATHER_BULK.  VN_GATHER_AUTO picks it beyond the
                                fused launch's wave for device callers: serial steps (no VN_STEP_ACTIONS_READY) of up to
                                four envs per CTA, pipelined steps of up to 3/4 of a wave; a host caller (out->host_pack)
                                and everything larger run as scalar kernel + gather kernel.  vn_env_step_mode tells. */

int32_t vn_abi_version(void);
/* sizeof of the descriptor structs as compiled into the library (0 store, 1 tables, 2 envs, 3 rules, 4 inject,
 * 5 step_out, 6 replay, 7 float_leaf, 8 host_call, 9 u8_frames; -1 otherwise): a binding checks its mirrors against these at load
 * time. */
int32_t vn_abi_struct_size(int32_t which);
const char *vn_last_error(void);
/* Kernels enqueued by the library so far (process-wide, monotonically increasing; statistics only). */
int64_t vn_launch_count(void);

/* Fills the store with the synthetic frame hash (a2cat-vn-pytorch_b200/scenes.py frame_bytes):
 * record r of this call holds local state state0 + r of scene `scene`.  Stands in for loading
 * the pickled scene (graph/util.py:69-79) when no AI2-THOR data exists. */
int32_t vn_fill_store(const vn_store_t *store, int32_t record0, int32_t n_records, uint64_t seed, int32_t scene,
                      int32_t state0, const int32_t *plane_ids /* [host][n_planes] */, void *stream);

/* VecEnv.reset(): (re)starts every env (mask == NULL) or the masked ones, gathers observation and
 * goal frames.  Replaces OrientedGraphEnv.reset (gym_graph/graph.py:46-54), sample_initial_state,
 * THORDiscreteCachedEnv.reset (cached.py:47-57) for the whole batch. */
int32_t vn_env_reset(const vn_store_t *store, const vn_tables_t *tables, const vn_envs_t *envs,
                     const vn_rules_t *rules, const vn_inject_t *inject, const uint8_t *mask,
                     const vn_step_out_t *out, int32_t gather_variant, void *stream);

/* VecEnv.step(actions): adjacency lookup, collision / goal test, reward, time limit, done,
 * auto-reset, episode statistics, last_action_reward and the frame gather, for all envs.
 * Replaces OrientedGraphEnv.step (gym_graph/graph.py:67-79), SimpleGraphEnv.step (graph/env.py:117-133),
 * THORDiscreteCachedEnv.step (cached.py:74-99), ThorGridWorld.render (graph/multi_graph_no_tp.py:12-25),
 * GoalGymGraphAuxiliaryEnv.observe (gym_graph/graph.py:110-120) and the SubprocVecEnv worker loop. */
int32_t vn_env_step(const vn_store_t *store, const vn_tables_t *tables, const vn_envs_t *envs,
                    const vn_rules_t *rules, const vn_inject_t *inject, const int32_t *actions,
                    const vn_step_out_t *out, int32_t gather_variant, void *stream);

/* The two halves of vn_env_step as separate launches (vn_env_step == scalar half then gather half on
 * the same stream).  Exposed so a host can time the gather kernel on its own or overlap the scalar
 * half of one batch with the gather of another. */
int32_t vn_env_step_scalar(const vn_tables_t *tables, const vn_envs_t *envs, const vn_rules_t *rules,
                           const vn_inject_t *inject, const int32_t *actions, const vn_step_out_t *out, void *stream);
int32_t vn_env_gather(const vn_store_t *store, const vn_envs_t *envs, const vn_step_out_t *out,
                      int32_t gather_variant, void *stream);

/* The reference-facing call with HOST buffers: VecEnv.step(actions) as deep_rl's trainer makes it
 * (numpy actions in, numpy rewards / dones / infos out; experiments/thor_cached_auxiliary.py:67 +
 * SubprocVecEnv.step).  host_actions and out->host_pack are PINNED host memory (device-mapped under
 * UVA).  Enqueues, in stream order: the scalar half - which reads the actions straight from
 * host_actions and mirrors the per-env scalars into out->host_pack over PCIe, so no copy-engine
 * operation sits on the critical path -; a record of ready_event (optional); the gather half.  The
 * host waits for the scalars only - on out->host_seq (vn_host_wait_seq, preferred: nothing sits between the
 * two kernels) or on ready_event (vn_event_wait) - while the gather keeps running; the
 * observations stay in HBM, ordered before any later work on the same stream.  dev_actions_copy
 * (optional) receives a device copy of the actions for device-side consumers (rollout buffer). */
int32_t vn_env_step_host(const vn_store_t *store, const vn_tables_t *tables, const vn_envs_t *envs,
                         const vn_rules_t *rules, const vn_inject_t *inject, const int32_t *host_actions,
                         int32_t *dev_actions_copy, const vn_step_out_t *out, void *ready_event,
                         int32_t gather_variant, void *stream);
/* How vn_env_reset / vn_env_step / vn_env_step_host would run for these arguments (out->flags and out->host_pack
 * matter under VN_GATHER_AUTO): 0 = scalar kernel + gather kernel, 1 = CTA-per-env fused launch, 2 = persistent launch;
 * negative on error.  A caller that pipelines steps (VN_STEP_ACTIONS_READY) uses it to know whether the PREVIOUS call
 * ended in a gather kernel it may overlap (mode 0) or not (then it adds VN_STEP_NO_OVERLAP). */
int32_t vn_env_step_mode(const vn_store_t *store, const vn_envs_t *envs, const vn_step_out_t *out,
                         int32_t gather_variant);

/* Number of host_seq words vn_env_step_host will publish for this batch (= thread blocks of its scalar half:
 * one per env when the step runs as the fused launch, ONE for the persistent launch, one per 128 envs otherwise);
 * <= 0 on error. */
int32_t vn_env_host_seq_words(const vn_store_t *store, const vn_envs_t *envs, const vn_step_out_t *out,
                              int32_t gather_variant);
/* Spins (pause loop, no GIL under ctypes) until host_seq[0 .. words) all equal seq.  Every ~50 us it looks at the
 * stream: a CUDA error, or a stream that drained without the words ever arriving, ends the wait with VN_ECUDA; so
 * does timeout_us (> 0). */
int32_t vn_host_wait_seq(const uint32_t *host_seq, int32_t words, uint32_t seq, void *stream, int64_t timeout_us);
/* VecEnv.step(actions) in ONE call for a host caller: vn_env_step_host (out->host_pack and out->host_seq are
 * required, no event), vn_host_wait_seq on out->host_seq / out->seq, then copies [host, pageable is fine; each
 * optional] so that the caller owns the results while a later step overwrites the pinned block: pack_copy receives
 * the whole 20 * n_envs host pack, reward_copy the n_envs rewards, done_copy the n_envs done bytes.  A caller that
 * alternates between two host packs only needs rewards and dones copied (20 KB instead of 80 KB at 4,096 envs): the
 * rest of the pack - what `infos` is built from - stays readable in place until the step after next.
 * seq_words = vn_env_host_seq_words(...).  The gather of this step is still running on return. */
int32_t vn_env_step_host_sync(const vn_store_t *store, const vn_tables_t *tables, const vn_envs_t *envs,
                              const vn_rules_t *rules, const vn_inject_t *inject, const int32_t *host_actions,
                              int32_t *dev_actions_copy, const vn_step_out_t *out, uint8_t *pack_copy,
                              float *reward_copy, uint8_t *done_copy, int32_t seq_words, int32_t gather_variant,
                              void *stream, int64_t timeout_us);
/* The same call with its constant arguments bound once: a host loop that steps the same env batch thousands of times per
 * second (a Python binding pays per argument it converts) fills this descriptor once, updates out->parity / flags / seq /
 * host_pack in place between calls and passes four arguments per step.  All pointers are [host]; the structs they point
 * to must outlive the calls. */
typedef struct vn_host_call {
    const vn_store_t *store;
    const vn_tables_t *tables;
    const vn_envs_t *envs;
    const vn_rules_t *rules;
    const vn_inject_t *inject;        /* may be NULL */
    const int32_t *host_actions;      /* pinned */
    int32_t *dev_actions_copy;        /* device, may be NULL */
    const vn_step_out_t *out;
    int32_t seq_words;
    int32_t gather_variant;
    int64_t timeout_us;
} vn_host_call_t;
int32_t vn_env_step_host_call(const vn_host_call_t *call, float *reward_copy, uint8_t *done_copy, void *stream);

/* Development aid: when device_buffer is not NULL every CTA of the step path's bulk gather writes 16 uint64 there
 * ([grid][16]: globaltimer ns when resident, when its predecessor had completed, after its first and last unit, when its
 * shared memory had drained; [5] = units it handled, [6] = SM id, [8..15] = time after each of its first 8 units, bit 63
 * set when the unit copied nothing) - tools/gather_timeline.py.  NULL switches it off.  Process-wide. */
int32_t vn_debug_gather_trace(uint64_t *device_buffer);

int32_t vn_event_create(void **event);   /* cudaEventDisableTiming */
int32_t vn_event_destroy(void *event);
int32_t vn_event_wait(void *event);      /* cudaEventSynchronize; releases the GIL under ctypes */

/* out[i] = plane `plane` of store record idx[i] (replay / sample_sequence gathers,
 * experiments/ai2_auxiliary/trainer.py:29).  idx may be live env state (envs->state, out->obs_state, envs->goal): the
 * kernel does not release its stream successor early, so a following vn_env_step* call - even one with
 * VN_STEP_ACTIONS_READY - only starts rewriting those arrays after this gather has completed. */
int32_t vn_gather_plane(const vn_store_t *store, int32_t plane, const int32_t *idx, int32_t n, uint8_t *out,
                        int32_t gather_variant, void *stream);

/* TransposeImage + ScaledFloatFrame (deep_rl.common.env, used at thor_cached_auxiliary.py:61-62)
 * fused with the gather: out[i] = float32 CHW of plane / 255. */
int32_t vn_gather_plane_f32_chw(const vn_store_t *store, int32_t plane, const int32_t *idx, int32_t n, int32_t h,
                                int32_t w, int32_t c, float *out, void *stream);
/* The same into a PERSISTENT float batch: row i is rewritten from record idx[i * idx_stride] unless that entry is
 * negative.  With idx = gather_desc of the step just enqueued (stride 2; + 1 for the goal record) only the rows
 * whose observation changed - and only the goal rows of envs that reset - are converted again. */
int32_t vn_gather_plane_f32_chw_rows(const vn_store_t *store, int32_t plane, const int32_t *idx, int32_t idx_stride,
                                     int32_t n, int32_t h, int32_t w, int32_t c, float *out, void *stream);

/* All float leaves of one step in ONE launch (the observation tuple the reference's wrappers produce,
 * thor_cached_auxiliary.py:59-64): leaf l is plane leaves[l].plane of the observation record (source 0) or of the
 * goal record (source 1) named by desc[i] = (record or -1, goal record or -1) - the gather_desc half of the step
 * just enqueued - written as float32 CHW / 255 into row i of the persistent batch leaves[l].out; negative records
 * leave the row untouched.  VN_EUNSUPPORTED when H * W is not a multiple of 4 or a plane has neither 1 nor 3
 * channels (use vn_gather_plane_f32_chw_rows per leaf then).  At most 6 leaves. */
int32_t vn_gather_leaves_f32_chw(const vn_store_t *store, const vn_float_leaf_t *leaves /* [host] */, int32_t n_leaves,
                                 const int32_t *desc /* [n][2] */, int32_t n, int32_t h, int32_t w, void *stream);

/* Index conventions of the rollout builders.  A rollout storage is TIME-major (row t of a [T, n_envs] array is
 * what one env step appends; deep_rl RolloutStorage), the tensors a loss consumes are BATCH-major ([B, T, ...] like
 * the reference's).  Every builder therefore takes its INPUT arrays with explicit element strides - element (n, t)
 * lives at n * stride_n + t * stride_t: (T, 1) for batch-major, (1, n_envs) for time-major storage - and writes its
 * output batch-major, so no transpose kernel ever runs between the storage and the loss. */

/* A2C n-step returns (deep_rl RolloutStorage.batch, SURVEY.md D4):
 *   R_T = (1 - done[T-1]) * last_value;  R_t = reward[t] + gamma * (1 - done[t]) * R_{t+1}.
 * Element (n, t) of reward / done lives at n * stride_n + t * stride_t, of out at n * out_stride_n + t * out_stride_t. */
int32_t vn_nstep_returns(const float *reward, const uint8_t *done, const float *last_value, float gamma, int32_t n,
                         int32_t t, int64_t stride_n, int64_t stride_t, float *out, int64_t out_stride_n,
                         int64_t out_stride_t, void *stream);

/* The same returns by a warp-level scan (one warp per env, 32 steps per pass, affine maps composed with shuffles):
 * for few envs and long rollouts.  Re-associates the float operations: within ~1e-6 relative of vn_nstep_returns,
 * not bit-identical. */
int32_t vn_nstep_returns_scan(const float *reward, const uint8_t *done, const float *last_value, float gamma,
                              int32_t n, int32_t t, int64_t stride_n, int64_t stride_t, float *out,
                              int64_t out_stride_n, int64_t out_stride_t, void *stream);

/* Backward discounted scan with a trailing feature axis of width d (pixel-control returns):
 *   R_T = bootstrap;  R_t = reward[t] + gamma * (1 - done[t]) * R_{t+1};  reward / out are [n][t][d], bootstrap [n][d],
 * done(n, t) lives at n * done_stride_n + t * done_stride_t. */
int32_t vn_discounted_backup(const float *reward, const uint8_t *done, int64_t done_stride_n, int64_t done_stride_t,
                             const float *bootstrap, float gamma, int32_t n, int32_t t, int32_t d, float *out,
                             void *stream);

/* UNREAL pixel-control reward (deep_rl.a2c_unreal.util.pixel_control_reward, SURVEY.md D5) computed
 * straight from the store: for the t + 1 observations states(n, 0..t) of every env (element (n, k) at
 * n * state_stride_n + k * state_stride_t)
 *   out[n][k] = mean_c avg_pool_cell( | f(states(n, k+1)) - f(states(n, k)) | ),  f = plane / 255 in fp32,
 * centred crop to (out_h*cell, out_w*cell).  out is [n][t][out_h][out_w] float32. */
int32_t vn_pixel_control(const vn_store_t *store, int32_t plane, const int32_t *states, int32_t n, int32_t t,
                         int64_t state_stride_n, int64_t state_stride_t, int32_t h, int32_t w, int32_t c, int32_t cell,
                         int32_t out_h, int32_t out_w, float *out, void *stream);

/* Table-driven pixel control.  On a cached graph the pixel-control reward of a transition is a pure
 * function of the state pair, so it is computed ONCE per (state, action) into a table
 * pc_table[n_states * 4][out_h * out_w] (vn_pixel_control over the pairs (s, adj[s][a])) and a rollout's
 * rewards become row gathers:
 *   vn_transition_rows   rows(n, k) = s*4 + a with adj[s][a] == s' (element (n, k) of the scratch lives at
 *                        n * row_stride_n + k * row_stride_t: give it the layout of `states` and both are accessed
 *                        coalesced); -1 (zeros) when s' == s (collision /
 *                        no-op: identical frames); -(2 + m) for transitions the table cannot serve (resets):
 *                        their positions n*t + k are appended to miss_pos[m] and counted in miss_count[0]
 *   vn_gather_rows       out[i] = table[idx(i)] (rows of row_bytes, multiple of 16); idx -1 writes zeros,
 *                        idx <= -2 leaves the row untouched.  Output row i = (a, k) of a batch-major
 *                        [n / idx_t][idx_t] result reads idx[a * idx_stride_n + k * idx_stride_t] (a flat index
 *                        list is idx_t = 1, strides (1, 0)).  Also serves the auxiliary-target tables.
 *   vn_pixel_control_list direct computation for the listed positions (count read from device memory,
 *                        at most max_count), written into row p of the same [n][t][out_h][out_w] output, or
 *                        (compact != 0) into row m of a side buffer [max_count][out_h][out_w]
 *   vn_pixel_control_returns  the discounted back-up (gamma_pc = 0.9 from max_a Q(s_T), SURVEY.md D5) fused with
 *                        the row gather: R_T = bootstrap; R_k = pc(n, k) + gamma (1 - done(n, k)) R_{k+1} with
 *                        pc(n, k) = table[rows] | 0 | miss_rows[m] read on the fly; out_returns [n][t][cells],
 *                        out_reward (optional) receives pc itself.  cells must be a multiple of 4. */
int32_t vn_transition_rows(const int32_t *adj, const int32_t *states, int32_t n, int32_t t, int64_t state_stride_n,
                           int64_t state_stride_t, int32_t *rows, int64_t row_stride_n, int64_t row_stride_t,
                           int32_t *miss_pos, int32_t *miss_count, void *stream);
int32_t vn_gather_rows(const void *table, int64_t row_bytes, const int32_t *idx, int64_t n, int32_t idx_t,
                       int64_t idx_stride_n, int64_t idx_stride_t, void *out, void *stream);
int32_t vn_pixel_control_list(const vn_store_t *store, int32_t plane, const int32_t *states, int32_t n, int32_t t,
                              int64_t state_stride_n, int64_t state_stride_t, int32_t h, int32_t w, int32_t c,
                              int32_t cell, int32_t out_h, int32_t out_w, const int32_t *pos, const int32_t *count,
                              int32_t max_count, int32_t compact, float *out, void *stream);
int32_t vn_pixel_control_returns(const float *pc_table, int32_t cells, const int32_t *rows, int64_t row_stride_n,
                                 int64_t row_stride_t, const float *miss_rows, const uint8_t *done,
                                 int64_t done_stride_n, int64_t done_stride_t,
                                 const float *bootstrap, float gamma, int32_t n, int32_t t, float *out_returns,
                                 float *out_reward, void *stream);
/* The three steps above as ONE call for a rollout's states: vn_transition_rows, vn_pixel_control_list (compact, into
 * miss_rows [max_miss][cells]) and vn_pixel_control_returns, chained with programmatic dependent launches (each kernel's
 * launch latency hides behind its predecessor).  rows / miss_pos are int32 scratch of n * t entries; *miss_count must be
 * 0 on entry - zero it once when the scratch is allocated, the last kernel re-arms it for the next call. */
int32_t vn_pixel_control_returns_from_states(const vn_store_t *store, int32_t plane, const int32_t *adj,
                                             const float *pc_table, const int32_t *states, int64_t state_stride_n,
                                             int64_t state_stride_t, const uint8_t *done, int64_t done_stride_n,
                                             int64_t done_stride_t, const float *bootstrap, float gamma, int32_t n,
                                             int32_t t, int32_t h, int32_t w, int32_t c, int32_t cell, int32_t out_h,
                                             int32_t out_w, int32_t *rows, int32_t *miss_pos, int32_t *miss_count,
                                             float *miss_rows, int32_t max_miss, float *out_returns, float *out_reward,
                                             void *stream);

/* Device-side UNREAL experience replay (deep_rl's replay behind `self.replay.sample_sequence()`,
 * experiments/ai2_auxiliary/trainer.py:29, and sample_rp_sequence; SURVEY.md D6 / section 8(f) rank 1).
 * The ring holds state INDICES, not frames: per inserted env step the state observed before the action,
 * the state observed after it (post auto-reset), the goal of each of the two observations (they differ when
 * the step ended an episode and the env drew a new task), action, reward, done; time-major [cap][n]. */
typedef struct vn_replay {
    const int32_t *before, *after, *goal, *goal_before, *action;
    const float *reward;
    const uint8_t *done;
    int32_t n, cap;
    int32_t head;  /* next slot to be written */
    int32_t count; /* filled slots, <= cap */
} vn_replay_t;

/* One window per env, uniform over the env's valid windows (inside the ring, no episode end except on
 * the last transition), drawn with Philox keyed by (seed, env_id_base + env, call).
 *   mode 0: `length` transitions -> o_states/o_goals [n][length+1], o_actions/o_rewards/o_dones [n][length]
 *   mode 1: reward prediction - 3 history transitions + the transition whose reward is classified
 *           (length ignored, windows of 4), zero / non-zero reward classes drawn 50/50 (the other class
 *           when one is empty); o_label [n] = 0 zero, 1 positive, 2 negative.
 * o_start[n] = chronological index of the window, -1 when the env has no valid window (outputs untouched). */
int32_t vn_replay_sample(const vn_replay_t *ring, int32_t length, int32_t mode, uint64_t seed, uint32_t call,
                         int32_t env_id_base, int32_t *o_states, int32_t *o_goals, int32_t *o_actions,
                         float *o_rewards, uint8_t *o_dones, int32_t *o_start, int8_t *o_label, void *stream);

/* compute_auxiliary_target (experiments/ai2_auxiliary/trainer.py:9-15) from the store:
 * out[i] = avg_pool_cell(crop(plane(idx[i]) / 255)), [m][c][out_h][out_w] float32. */
int32_t vn_aux_target(const vn_store_t *store, int32_t plane, const int32_t *idx, int32_t m, int32_t h, int32_t w,
                      int32_t c, int32_t cell, int32_t out_h, int32_t out_w, float *out, void *stream);

/* Reward-prediction classes (0 zero, 1 positive, 2 negative) and the ascending position lists of
 * zero / non-zero rewards the 50/50 sampler draws from (SURVEY.md D6).  n positions in all; position
 * i = (a, k) of the batch-major [n / t][t] result reads reward[a * stride_n + k * stride_t] (flat input: t = 1,
 * strides (1, 0)).  counts[0..1] receive the list lengths (always written).  Ballot / warp-scan compaction in three
 * small launches, order preserving, up to 2^24 positions per call; scratch is int32 [(n + 1023) / 1024]
 * caller-owned device memory. */
int32_t vn_rp_labels(const float *reward, int32_t n, int32_t t, int64_t stride_n, int64_t stride_t, int8_t *labels,
                     int32_t *zero_idx, int32_t *nonzero_idx, int32_t *counts, int32_t *scratch, void *stream);

/* The policy's first convolution read straight from uint8 frames.  Replaces TransposeImage + ScaledFloatFrame
 * (deep_rl.common.env, thor_cached_auxiliary.py:61-62) + the model's first Conv2d (models/goal.py:36-41):
 *   y = conv2d(x / 255, weight, bias, stride), x = frame i as [c][h][w] (the frame is stored HWC), padding 0.
 * The frames are never written as float32: the forward reads each uint8 frame once, and the weight gradient reads it
 * again, so an update pass keeps only the state indices alive between its forward and its backward.
 *
 * Frame source.  Frame i of a batch (idx == NULL) is row i: base + i * pitch.  With idx it is record
 * idx[a * idx_stride_n + k * idx_stride_t], a = i / idx_t, k = i % idx_t (vn_gather_rows' convention: a [B, T] view of
 * time-major rollout states is read in place), at base + record * pitch.  base is a store plane
 * (store->base + plane_off[p], pitch state_pitch) or a uint8 observation batch (pitch plane_bytes); base and pitch are
 * multiples of 16, pitch >= h * w * c, and idx holds valid record indices. */
typedef struct vn_u8_frames {
    const uint8_t *base;
    int64_t pitch;
    const int32_t *idx;
    int64_t idx_stride_n, idx_stride_t;
    int32_t n, idx_t, h, w, c, reserved;
} vn_u8_frames_t;

/* Supported: c 1 or 3, 1 <= k <= 8, 1 <= stride <= k, cout a multiple of 8 up to 64, k <= h, w <= 174; anything else
 * is VN_EUNSUPPORTED.  n == 0 launches nothing (and writes nothing).  The kernels run on the tensor cores with the fp32
 * operand split into three exact bf16 terms: fp32-class results (see vn_conv.cu).  A programmatic launch that waits for
 * its predecessor before it reads anything and does not release its successor early: like vn_gather_plane, idx may be
 * live env state (out->obs_state), and a batch row may be one a following vn_env_step* call rewrites. */
/* out [n][cout][oh][ow] float32, oh = (h - k) / stride + 1; weight [cout][c][k][k]; bias [cout] or NULL. */
int32_t vn_conv_u8_forward(const vn_u8_frames_t *src, const float *weight, const float *bias, int32_t cout, int32_t k,
                           int32_t stride, float *out, void *stream);
/* Bytes of device scratch vn_conv_u8_backward needs: ceil(n / 32) * cout * (c * k * k + 1) * 4 (one partial gradient
 * per chunk of 32 frames); -1 for negative or zero sizes.  Host only.  With c the set's channel count, also the
 * scratch of vn_conv_u8_planes_backward[_lp]. */
int64_t vn_conv_u8_wgrad_scratch_bytes(int32_t n, int32_t c, int32_t cout, int32_t k);
/* The weight and bias gradient of vn_conv_u8_forward for grad_out [n][cout][oh][ow]:
 *   grad_weight[co][ci][ky][kx] = sum_{i, oy, ox} grad_out[i][co][oy][ox] * x_i[ci][oy * stride + ky][ox * stride + kx] / 255,
 *   grad_bias[co] (optional) = sum_{i, oy, ox} grad_out[i][co][oy][ox].
 * Both are written, not accumulated.  Two kernels: partial sums per chunk of 32 frames into scratch, then a reduction
 * over the chunks in a fixed order - no atomics, the same bits on every run and every device size. */
int32_t vn_conv_u8_backward(const vn_u8_frames_t *src, const float *grad_out, int32_t cout, int32_t k, int32_t stride,
                            float *grad_weight, float *grad_bias, void *scratch, int64_t scratch_bytes, void *stream);

/* The same layer under torch.autocast with a 16-bit dtype (mixed precision).  out and grad_out are of `dtype`, weight,
 * bias, grad_weight and grad_bias stay float32.  The forward computes
 *   out = round_to_dtype(fp32(conv2d(x / 255, round_to_dtype(weight), round_to_dtype(bias), stride)))
 * with the weight and bias rounded to nearest-even in its prologue (autocast's cast), the pixel NOT rounded (0..255 is
 * exact in both types; 1/255 is applied in fp32 as in vn_conv_u8_forward), every product exact on the tensor cores
 * with one term per operand, fp32 accumulation, and one rounding of the result (fp16 overflows to +-inf).  The backward
 * takes grad_out in `dtype`, forms every product exactly, and writes the fp32 weight / bias gradient with the two
 * kernels and the scratch (vn_conv_u8_wgrad_scratch_bytes) of vn_conv_u8_backward; a non-finite grad_out element makes
 * its output channel's gradients non-finite.  Arguments, limits and launch behaviour are those of the fp32 entry
 * points; in addition out and grad_out must be 2-byte aligned (any oh * ow, odd ones included), and a dtype other
 * than VN_DTYPE_F16 / VN_DTYPE_BF16 is VN_EUNSUPPORTED. */
#define VN_DTYPE_F16 1
#define VN_DTYPE_BF16 2
int32_t vn_conv_u8_forward_lp(const vn_u8_frames_t *src, const float *weight, const float *bias, int32_t cout,
                              int32_t k, int32_t stride, int32_t dtype, void *out, void *stream);
int32_t vn_conv_u8_backward_lp(const vn_u8_frames_t *src, const void *grad_out, int32_t dtype, int32_t cout,
                               int32_t k, int32_t stride, float *grad_weight, float *grad_bias,
                               void *scratch, int64_t scratch_bytes, void *stream);

/* The same layer over a plane set: the frames of n_srcs sources stacked along channels in source order (RGB-D:
 * {rgb, depth}; early-fused goal: {obs rgb, goal rgb}):
 *   y = conv2d(cat_c(x_0, ..., x_{n_srcs-1}) / 255, weight, bias, stride), weight [cout][C][k][k], C = sum of srcs[s].c.
 * Every source has its own base, pitch, idx and index strides (the observation and the goal may come from two index
 * tensors, or a store plane and an observation batch); all share n, idx_t, h and w (a mismatch is VN_EINVAL).
 * Supported: 1 to 4 sources of 1 or 3 channels, 8 channels in all, the kernel, stride and cout of vn_conv_u8_forward,
 * and frames whose set (sum of h * w * c rounded up to 16 bytes per source) fits in shared memory beside the kernels'
 * tables: every such set on frames up to 84 x 84, and up to 5 channels (e.g. RGB-D) on the reference's 174 x 174;
 * anything else is VN_EUNSUPPORTED.  Numerics, results (one source gives the bits of vn_conv_u8_forward / _backward),
 * scratch (vn_conv_u8_wgrad_scratch_bytes with c = C), alignment and launch behaviour are those of the one-source entry
 * points above, in fp32 and in fp16 / bf16 (_lp). */
int32_t vn_conv_u8_planes_forward(const vn_u8_frames_t *srcs, int32_t n_srcs, const float *weight, const float *bias,
                                  int32_t cout, int32_t k, int32_t stride, float *out, void *stream);
int32_t vn_conv_u8_planes_forward_lp(const vn_u8_frames_t *srcs, int32_t n_srcs, const float *weight,
                                     const float *bias, int32_t cout, int32_t k, int32_t stride, int32_t dtype,
                                     void *out, void *stream);
int32_t vn_conv_u8_planes_backward(const vn_u8_frames_t *srcs, int32_t n_srcs, const float *grad_out, int32_t cout,
                                   int32_t k, int32_t stride, float *grad_weight, float *grad_bias, void *scratch,
                                   int64_t scratch_bytes, void *stream);
int32_t vn_conv_u8_planes_backward_lp(const vn_u8_frames_t *srcs, int32_t n_srcs, const void *grad_out, int32_t dtype,
                                      int32_t cout, int32_t k, int32_t stride, float *grad_weight, float *grad_bias,
                                      void *scratch, int64_t scratch_bytes, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* VN_B200_H */
