// Vectorised env step / reset and the frame gather (sm_100a).
//
// A vectorised step is, in stream order, programmatically chained:
//   K1 vn_step_kernel   one thread per env: adjacency lookup, collision + goal test, reward, TimeLimit,
//                       done, auto-reset (Philox4x32-10, injected stream or a fixed episode list whose results it
//                       records), RewardCollector accumulators,
//                       last_action_reward, warp-aggregated episode statistics.  ~40 B per env.
//   K2 vn_gather_*      copies each env's observation planes (and, only if the env just reset, its goal planes)
//                       from the HBM store into the contiguous policy batch.  >99.9 % of the bytes; HBM-bound; two
//                       variants: LDG.128 through registers (one CTA per env) and bulk async copies (persistent
//                       one-warp CTAs that take (env, slice) units, see vn_gather_bulk_kernel).
// or ONE launch that does both: vn_step_fused_kernel (a CTA per env, batches of one wave) and vn_step_gather_kernel
// (a persistent grid, mid-size batches); choose_mode decides.
#include <atomic>
#include <chrono>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <utility>

#include "vn_common.cuh"

namespace vn {

static thread_local std::string g_error;
static unsigned long long *g_gather_trace = nullptr;  // development: vn_debug_gather_trace
static std::atomic<long long> g_launches{0};  // statistics only: kernels enqueued by this library, all threads

void set_error(const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_error = buf;
}

int32_t launch_result(const char *what, cudaError_t e) {
    if (e != cudaSuccess) {
        set_error("%s: %s", what, cudaGetErrorString(e));
        return VN_ECUDA;
    }
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return VN_OK;
}

// =====================================================================================================
// K1: step / reset
// =====================================================================================================
struct StepParams {
    vn_tables_t tab;
    vn_envs_t env;
    vn_rules_t rules;
    vn_inject_t inj;
    vn_step_out_t out;
    vn_episodes_t eps;       // copy of *env.episodes; eps.cursor == NULL: no list
    const int32_t *actions;  // NULL in reset mode
    const uint8_t *mask;     // reset mode only
    int32_t *actions_copy;   // optional device copy of the actions (host-actions path)
    int32_t skip_rows;       // VN_STEP_SKIP_UNCHANGED is set AND the gather half can honour it (descriptors / fused)
};

constexpr int kStepThreads = 128;  // envs per block of the scalar half (= envs per host_seq word)

// Programmatic dependent launch: every kernel of the step path lets its successor be scheduled early
// (launch latency overlaps this kernel's execution) and waits for its predecessor's memory to be visible
// before touching any env data.  Both are no-ops when the launch was not programmatic.
__device__ __forceinline__ void pdl_wait_then_release() {
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}

// Per-env statistics contributions of one step (summed over a warp, or added directly by the fused kernel).
struct EnvStats {
    uint32_t episodes = 0, len = 0, succ = 0, coll = 0, steps = 0, trunc = 0, resets = 0, skipped = 0;
    float ret = 0.f;

    __device__ __forceinline__ EnvStats &operator+=(const EnvStats &o) {
        episodes += o.episodes;
        len += o.len;
        succ += o.succ;
        coll += o.coll;
        steps += o.steps;
        trunc += o.trunc;
        resets += o.resets;
        skipped += o.skipped;
        ret += o.ret;
        return *this;
    }
};

// Sum over the (full) warp; every lane receives it.
__device__ __forceinline__ EnvStats warp_reduce(const EnvStats &s) {
    EnvStats w;
    w.episodes = __reduce_add_sync(0xffffffffu, s.episodes);
    w.len = __reduce_add_sync(0xffffffffu, s.len);
    w.succ = __reduce_add_sync(0xffffffffu, s.succ);
    w.coll = __reduce_add_sync(0xffffffffu, s.coll);
    w.steps = __reduce_add_sync(0xffffffffu, s.steps);
    w.trunc = __reduce_add_sync(0xffffffffu, s.trunc);
    w.resets = __reduce_add_sync(0xffffffffu, s.resets);
    w.skipped = __reduce_add_sync(0xffffffffu, s.skipped);
    w.ret = s.ret;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) w.ret += __shfl_xor_sync(0xffffffffu, w.ret, o);
    return w;
}

// One env, one step (or reset): everything the reference does between receiving the action and calling
// observe().  Returns the store record whose frames must be in the batch (rec; -1 = the batch row already
// holds it, VN_STEP_SKIP_UNCHANGED) and the goal record to (re)write (grec; -1 = none).
template <bool kReset>
__device__ __forceinline__ void step_env(const StepParams &p, const int i, EnvStats &st, int &rec, int &grec) {
    const int flags = p.rules.flags;
    int s = p.env.state[i];
    int g = p.env.goal[i];
    float ep_ret = p.env.ep_return[i];
    int ep_len = p.env.ep_length[i];
    int elapsed = p.env.elapsed[i];
    // record gathered by the previous call (the scratch is persistent): only read when rows may be skipped
    const bool may_skip = !kReset && p.skip_rows;
    const int prev_obs = may_skip ? p.out.obs_state[i] : -1;
    int obs_s = s;
    int listed = -1;  // listed episode (vn_episodes_t) that ended on this step, -1 = none
    bool do_reset;

    if (kReset) {
        do_reset = p.mask ? (p.mask[i] != 0) : true;
    } else {
        // may live in mapped pinned host memory (vn_env_step_host).  Carrying the host's actions in the kernel parameters
        // instead (one byte per env, packed by the CPU) was measured: no PCIe read in front of the dependent loads, but
        // packing + an 8 KB parameter block cost more than that saved (RGB-only e2e 145.4 -> 141.2 M env-steps/s)
        const int a = p.actions[i];
        if (p.actions_copy) p.actions_copy[i] = a;
        const int s_old = s;
        bool terminal = false, collided = false;
        float r;
        if ((flags & VN_RULE_NOOP_ACTION) && a < 0) {
            r = 0.0f;  // graph/env.py:118-120: latest observation, 0.0, not done
        } else {
            // graph.util.step + is_valid_state folded into one table lookup; an action outside
            // [0, 4) has no transition in the reference (step() returns None) and is a collision here
            const int nxt = (a >= 0 && a < 4) ? __ldg(p.tab.adj + (size_t)s * 4 + a) : -1;
            collided = nxt < 0;
            if (!collided) s = nxt;
            bool at_goal;
            if (p.rules.goal_compare == VN_GOAL_FULL)
                at_goal = (s == g);
            else if (p.rules.goal_compare == VN_GOAL_POSITION)
                at_goal = ((s >> 2) == (g >> 2));
            else
                at_goal = false;
            terminal = at_goal && !(collided && (flags & VN_RULE_COLLISION_SKIPS_GOAL));
            r = (flags & VN_RULE_NEG_STEP_REWARD) ? -p.rules.reward_step : p.rules.reward_step;
            if (terminal) r = p.rules.reward_goal;
            if (collided) r = p.rules.reward_collision;
        }
        if (p.rules.reward_progress != 0.0f) {
            // geodesic progress (vn_b200.h, vn_rules_t.reward_progress): distance of the current task's goal from the
            // state the action was taken in minus that from the state it led to, before any auto-reset
            const int32_t *dist = p.tab.task_dist + (size_t)p.env.task[i] * p.tab.n_states;
            const int d_prev = __ldg(dist + s_old);
            const int d_next = s == s_old ? d_prev : __ldg(dist + s);
            const int delta = (d_prev < 0 || d_next < 0) ? 0 : d_prev - d_next;
            r = __fadd_rn(r, __fmul_rn(p.rules.reward_progress, (float)delta));
        }
        bool done = terminal, trunc = false, at_limit = false;
        elapsed += 1;
        ep_ret += r;
        ep_len += 1;
        if (p.rules.max_episode_steps > 0 && elapsed >= p.rules.max_episode_steps) {
            at_limit = true;  // gym TimeLimit: info['TimeLimit.truncated'] = not done; done = True
            trunc = !done;
            done = true;
        }
        do_reset = done && (flags & VN_RULE_AUTO_RESET);
        obs_s = (terminal && (flags & VN_RULE_TERM_PREV_OBS) && !do_reset) ? s_old : s;

        const uint8_t trunc_code = at_limit ? (trunc ? 1 : 2) : 0;
        if (p.out.reward) p.out.reward[i] = r;
        if (p.out.done) p.out.done[i] = done;
        if (p.out.rec_action) p.out.rec_action[i] = a;
        if (p.out.rec_reward) p.out.rec_reward[i] = r;
        if (p.out.rec_done) p.out.rec_done[i] = done;
        if (p.out.truncated) p.out.truncated[i] = trunc_code;
        if (p.out.win) p.out.win[i] = terminal;
        if (p.out.info_state) p.out.info_state[i] = s;
        if (p.out.host_pack) {
            // mirror of the per-env scalars written straight into mapped pinned host memory
            // (layout: vn_b200.h "host pack"): the host reads them after the event that follows
            // this kernel, with no copy-engine operation on the critical path
            uint8_t *hp = p.out.host_pack;
            const size_t n = (size_t)p.env.n_envs;
            reinterpret_cast<float *>(hp)[i] = r;
            reinterpret_cast<int32_t *>(hp + 12 * n)[i] = s;
            hp[16 * n + i] = done;
            hp[17 * n + i] = trunc_code;
            hp[18 * n + i] = terminal;
            hp[19 * n + i] = do_reset;
            if (done) {
                reinterpret_cast<float *>(hp + 4 * n)[i] = ep_ret;
                reinterpret_cast<int32_t *>(hp + 8 * n)[i] = ep_len;
            }
        }
        if (done) {
            if (p.out.episode_return) p.out.episode_return[i] = ep_ret;
            if (p.out.episode_length) p.out.episode_length[i] = ep_len;
            st.episodes = 1;
            st.len = (uint32_t)ep_len;
            st.ret = ep_ret;
            st.succ = terminal;
            st.trunc = trunc;
            if (p.eps.cursor) {
                // the result of a listed episode, written once, by the step that ends it (vn_b200.h, vn_episodes_t)
                listed = p.eps.cursor[i];
                if (listed >= 0) {
                    p.eps.length[listed] = ep_len;
                    p.eps.ret[listed] = ep_ret;
                    p.eps.win[listed] = terminal;
                    p.eps.truncated[listed] = trunc;
                    p.eps.final_state[listed] = s;
                    atomicAdd(p.eps.count, 1u);
                }
            }
        }
        st.coll = collided;
        st.steps = 1;
        if (p.out.last_action_reward) {
            // UnrealEnvBaseWrapper: one_hot(action) ++ [clip(r, -1, 1)]; zeros right after a reset
            float *lar = p.out.last_action_reward + (size_t)i * (p.rules.n_actions + 1);
            for (int k = 0; k < p.rules.n_actions; ++k) lar[k] = (!do_reset && k == a) ? 1.0f : 0.0f;
            lar[p.rules.n_actions] = do_reset ? 0.0f : fminf(fmaxf(r, -1.0f), 1.0f);
        }
    }

    if (do_reset) {
        const uint32_t e = p.env.epoch[i];
        const int tlo = p.env.task_lo[i];
        int t, start;
        int next = -1;  // listed episode this reset starts, -1 = the ordinary source
        if (p.eps.cursor) {
            // the env's first listed episode is its global id, each later one `stride` further on (vn_episodes_t)
            const int64_t j = kReset ? (int64_t)p.env.env_id_base + i
                                     : (listed >= 0 ? (int64_t)listed + p.eps.stride : (int64_t)-1);
            next = (j >= 0 && j < p.eps.n_episodes) ? (int)j : -1;
            p.eps.cursor[i] = next;
        }
        if (next >= 0) {
            t = __ldg(p.eps.task + next);
            start = __ldg(p.eps.start + next);
        } else if (p.inj.start) {
            const uint32_t k = e < (uint32_t)p.inj.stride ? e : (uint32_t)p.inj.stride - 1;
            const size_t at = (size_t)i * p.inj.stride + k;
            t = tlo + (p.inj.task ? p.inj.task[at] : 0);
            start = p.inj.start[at];
        } else {
            const Philox4 d = philox4x32_10((uint32_t)(p.env.env_id_base + i), e, 0u, 0u, (uint32_t)p.rules.seed,
                                            (uint32_t)(p.rules.seed >> 32));
            t = tlo + (int)__umulhi(d.v[0], (uint32_t)p.env.task_cnt[i]);
            const int lo = __ldg(p.tab.task_cand_off + t);
            const int cnt = __ldg(p.tab.task_cand_off + t + 1) - lo;
            const int pre = __ldg(p.tab.task_prefix + t);
            int idx;
            if ((flags & VN_RULE_TWO_LEVEL) && pre < cnt && d.v[1] >= 3865470566u) {
                idx = pre + (int)__umulhi(d.v[2], (uint32_t)(cnt - pre));  // the 0.1 bucket, util.py:112-113
            } else {
                idx = (int)__umulhi(d.v[2], (uint32_t)pre);
            }
            start = __ldg(p.tab.cand_state + lo + idx);
        }
        s = start;
        g = __ldg(p.tab.task_goal + t);
        p.env.task[i] = t;
        p.env.goal[i] = g;
        p.env.epoch[i] = e + 1;
        elapsed = 0;
        ep_ret = 0.f;
        ep_len = 0;
        obs_s = s;
        st.resets = 1;
        if (kReset && p.out.last_action_reward) {
            float *lar = p.out.last_action_reward + (size_t)i * (p.rules.n_actions + 1);
            for (int k = 0; k <= p.rules.n_actions; ++k) lar[k] = 0.0f;
        }
    }
    p.env.state[i] = s;
    p.env.elapsed[i] = elapsed;
    p.env.ep_return[i] = ep_ret;
    p.env.ep_length[i] = ep_len;
    p.out.obs_state[i] = obs_s;
    if (p.out.did_reset) p.out.did_reset[i] = do_reset;
    if (!kReset) {  // rollout record of this step (RolloutStorage.insert without copy kernels)
        if (p.out.rec_state) p.out.rec_state[i] = obs_s;
        if (p.out.rec_goal) p.out.rec_goal[i] = g;
    }
    // the batch row of an env whose record did not change (collision, no-op) already holds the right frames
    const bool same = may_skip && obs_s == prev_obs;
    st.skipped = same;
    rec = same ? -1 : obs_s;
    grec = do_reset ? g : -1;
}

__device__ __forceinline__ void add_stats(uint64_t *stats, const EnvStats &s) {
    unsigned long long *st = reinterpret_cast<unsigned long long *>(stats);
    if (s.episodes) {
        atomicAdd(st + VN_STAT_EPISODES, (unsigned long long)s.episodes);
        atomicAdd(reinterpret_cast<double *>(st + VN_STAT_RETURN_SUM), (double)s.ret);
        atomicAdd(st + VN_STAT_LENGTH_SUM, (unsigned long long)s.len);
        if (s.succ) atomicAdd(st + VN_STAT_SUCCESSES, (unsigned long long)s.succ);
        if (s.trunc) atomicAdd(st + VN_STAT_TRUNCATIONS, (unsigned long long)s.trunc);
    }
    if (s.coll) atomicAdd(st + VN_STAT_COLLISIONS, (unsigned long long)s.coll);
    if (s.steps) atomicAdd(st + VN_STAT_STEPS, (unsigned long long)s.steps);
    if (s.resets) atomicAdd(st + VN_STAT_RESETS, (unsigned long long)s.resets);
    if (s.skipped) atomicAdd(st + VN_STAT_ROWS_SKIPPED, (unsigned long long)s.skipped);
}

// Every thread of a block calls this after its writes to the mapped host pack.  The block meets, then ONE thread
// issues the system-scope fence and publishes `seq` in the block's host word: the barrier orders the other threads'
// writes before that thread's fence, and the fence is cumulative over what happened before it - the pattern of a
// cooperative-groups grid barrier (bar.sync; one thread: fence; flag).  One fence per block instead of one per thread:
// the per-thread version cost ~6 us of the host-facing step.  The host has the scalars of all envs once every
// block's word shows `seq` (vn_host_wait_seq).
__device__ __forceinline__ void signal_host(const vn_step_out_t &out) {
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence_system();
        *reinterpret_cast<volatile uint32_t *>(out.host_seq + blockIdx.x) = out.seq;
    }
}

template <bool kReset>
__global__ void __launch_bounds__(kStepThreads) vn_step_kernel(const StepParams p) {
    // Pipelined mode (VN_STEP_ACTIONS_READY + gather_desc): nothing this kernel reads was produced by its
    // immediate predecessor - the previous gather - and what it writes for the next gather goes to the other
    // half of the double-buffered descriptor, so it runs WHILE the previous gather is still copying and only
    // waits for it at the very end (which also orders the next gather behind the previous one).
    const bool defer_wait = (p.out.flags & VN_STEP_ACTIONS_READY) && !(p.out.flags & VN_STEP_NO_OVERLAP) &&
                            p.out.gather_desc != nullptr;
    if (!defer_wait) asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    // the ticket counter the gather of THIS step draws from (the previous gather, possibly still running, uses the
    // other one; the last launch that used this one completed before the previous scalar half did)
    if (i == 0 && p.out.sched) p.out.sched[p.out.parity & 1] = 0u;
    EnvStats st;
    if (i < p.env.n_envs) {
        int rec, grec;
        step_env<kReset>(p, i, st, rec, grec);
        if (p.out.gather_desc)  // what the gather of THIS step needs: record to copy (or -1), goal record (or -1)
            reinterpret_cast<int2 *>(p.out.gather_desc)[(size_t)(p.out.parity & 1) * p.env.n_envs + i] =
                make_int2(rec, grec);
    }

    if (p.out.stats) {
        // warp-aggregated statistics: one atomic per counter per warp
        const EnvStats w = warp_reduce(st);
        if ((threadIdx.x & 31) == 0) add_stats(p.out.stats, w);
    }
    if (p.out.host_seq) signal_host(p.out);
    if (defer_wait) asm volatile("griddepcontrol.wait;" ::: "memory");
}

// =====================================================================================================
// K2: frame gather
// =====================================================================================================
struct GatherParams {
    vn_store_t store;
    const int2 *desc;          // [n] (record, goal record or -1) written by the step kernel; overrides the three below
    const int32_t *obs_state;  // [n] record to gather for the observation planes
    const int32_t *goal;       // [n] record of the goal planes (may be NULL)
    const uint8_t *did_reset;  // [n] goal planes are rewritten only where set (NULL = always)
    uint8_t *obs[VN_MAX_PLANES];
    uint8_t *goal_obs[VN_MAX_PLANES];
    unsigned int *sched;  // optional ticket counters (dynamic scheduling), see vn_gather_bulk_kernel
    int32_t n;
    int32_t parity;  // which of the two ticket counters (sched[0..1]) this launch draws from
    // 1: let the next kernel in the stream be scheduled while this one runs (the step path, where the successor is the
    // next scalar kernel and never writes what this gather reads).  0 (vn_gather_plane): the index list is caller
    // memory - often env.state / obs_state / goal themselves - that a following step kernel REWRITES, so the successor
    // must not start before this grid has completed.
    int32_t early_release;
    // development: per-CTA timeline (vn_debug_gather_trace): [grid][16] words, see vn_gather_bulk_kernel; NULL = off
    unsigned long long *trace;
};

__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}

// ---- variant A: 16-byte vector loads / stores through registers -------------------------------------
template <int kThreads, int kUnroll>
__device__ __forceinline__ void copy_segment16(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst, int n16) {
    const int4 *s = reinterpret_cast<const int4 *>(src);
    int4 *d = reinterpret_cast<int4 *>(dst);
    int base = threadIdx.x;
    // full batches: kUnroll independent 16 B loads in flight per thread before the first store
    for (; base + (kUnroll - 1) * kThreads < n16; base += kUnroll * kThreads) {
        int4 v[kUnroll];
#pragma unroll
        for (int k = 0; k < kUnroll; ++k) v[k] = ld_stream16(s + base + k * kThreads);
#pragma unroll
        for (int k = 0; k < kUnroll; ++k) st_stream16(d + base + k * kThreads, v[k]);
    }
    // tail: still issue all loads first
    int4 v[kUnroll];
#pragma unroll
    for (int k = 0; k < kUnroll; ++k)
        if (base + k * kThreads < n16) v[k] = ld_stream16(s + base + k * kThreads);
#pragma unroll
    for (int k = 0; k < kUnroll; ++k)
        if (base + k * kThreads < n16) st_stream16(d + base + k * kThreads, v[k]);
}

template <int kThreads, int kUnroll>
__global__ void __launch_bounds__(kThreads) vn_gather_ldg_kernel(const GatherParams p) {
    asm volatile("griddepcontrol.wait;" ::: "memory");
    if (p.early_release) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    for (int env = blockIdx.x; env < p.n; env += gridDim.x) {
        int rec, grec = -1;
        if (p.desc) {
            const int2 d = __ldg(p.desc + env);
            rec = d.x;
            grec = d.y;
        } else {
            rec = __ldg(p.obs_state + env);
            if (p.goal && (!p.did_reset || __ldg(p.did_reset + env))) grec = __ldg(p.goal + env);
        }
        if (rec >= 0) {  // rec < 0: the row already holds this record (VN_STEP_SKIP_UNCHANGED)
            const uint8_t *src = p.store.base + (size_t)rec * p.store.state_pitch;
#pragma unroll 1
            for (int pl = 0; pl < p.store.n_planes; ++pl) {
                if (p.obs[pl])
                    copy_segment16<kThreads, kUnroll>(src + p.store.plane_off[pl],
                                                      p.obs[pl] + (size_t)env * p.store.plane_bytes[pl],
                                                      p.store.plane_bytes[pl] >> 4);
            }
        }
        if (grec >= 0) {
            const uint8_t *gsrc = p.store.base + (size_t)grec * p.store.state_pitch;
#pragma unroll 1
            for (int pl = 0; pl < p.store.n_planes; ++pl) {
                if (p.goal_obs[pl])
                    copy_segment16<kThreads, kUnroll>(gsrc + p.store.plane_off[pl],
                                                      p.goal_obs[pl] + (size_t)env * p.store.plane_bytes[pl],
                                                      p.store.plane_bytes[pl] >> 4);
            }
        }
    }
}

// ---- variant B: bulk async copies (TMA engine), global -> shared -> global ---------------------------
// One warp per CTA; lane 0 issues one cp.async.bulk per plane into shared memory (completion counted in
// bytes on an mbarrier), then one cp.async.bulk per plane from shared memory to the batch rows.  No data
// passes through registers; several CTAs per SM keep ~200 KB of copies in flight.
//
// Work unit = (env, slice): each plane is cut into `split` slices of whole 16-byte units, so that
// split > 1 gives more, smaller CTAs per SM.  Units are handed out by an atomic ticket counter
// (persistent CTAs, dynamic scheduling): no CTA idles while another still has a queue of records.
// The ticket counter is CALLER-OWNED scratch (vn_step_out_t.sched[parity & 1]), zero before the first launch and
// zeroed again by the scalar half of the step that next uses it, so gathers of different env batches on different
// streams never share a counter.  Without scratch the units are dealt statically.
//
// L2 policies of the copies: the store is re-read across envs and steps, a batch row is written once and read by a
// later kernel, so loads are evict_last and stores evict_first (measured +2.5 % C2, +4 % at hardness 0.01,
// profiles/r1b_l2_hint_sweep.txt).
struct L2Policies {
    uint64_t load, store;
};

// One record slice through shared memory: all its loads complete on one mbarrier, then its stores go out.
// `while_loading()` runs after the loads have been issued and before the wait for them: the place to fetch whatever the
// NEXT unit needs (ticket, descriptor) so that its latency hides behind this transfer.  whole: the plane set is
// contiguous in the record and shared memory was sized for its SPAN (plane_set_bytes), so one load brings the record.
template <typename F>
__device__ __forceinline__ void bulk_copy_slice(const vn_store_t &st, const uint8_t *src, uint8_t *const *dst, int env,
                                                int slice, int split, uint8_t *smem, uint64_t *bar, uint32_t &parity,
                                                const L2Policies &pol, F while_loading, bool whole) {
    // the previous shared->global reads of this buffer must have drained before it is refilled
    bulk_wait_read<0>();
    int total = 0;
#pragma unroll 1
    for (int pl = 0; pl < st.n_planes; ++pl)
        if (dst[pl]) {
            const int n16 = st.plane_bytes[pl] >> 4, per = (n16 + split - 1) / split;
            const int lo = min(slice * per, n16), hi = min(lo + per, n16);
            total += hi - lo;
        }
    if (total == 0) return;
    if (whole && split == 1) {
        // The requested planes sit next to each other in the store record (128-byte aligned offsets, a few padding bytes
        // between them): ONE load brings the whole span, one store per plane sends it out - bulk copies are cheaper the
        // fewer and larger they are (every extra operation per record cost 0.2 - 1 us per step, profiles/r2_gather_groups.txt)
        int first = -1, last = -1;
        for (int pl = 0; pl < st.n_planes; ++pl)
            if (dst[pl]) {
                if (first < 0) first = pl;
                last = pl;
            }
        const uint32_t base = (uint32_t)st.plane_off[first];
        const uint32_t span = (uint32_t)st.plane_off[last] + (uint32_t)st.plane_bytes[last] - base;
        mbar_expect_tx(bar, span);
        bulk_g2s_hint(smem, src + base, span, bar, pol.load);
        while_loading();
        mbar_wait(bar, parity & 1u);
        parity ^= 1u;
        for (int pl = first; pl <= last; ++pl)
            if (dst[pl])
                bulk_s2g_hint(dst[pl] + (size_t)env * st.plane_bytes[pl], smem + ((uint32_t)st.plane_off[pl] - base),
                              (uint32_t)st.plane_bytes[pl], pol.store);
        bulk_commit();
        return;
    }
    // the slices of the planes, packed back to back in shared memory
    mbar_expect_tx(bar, (uint32_t)total << 4);
    int off = 0;
#pragma unroll 1
    for (int pl = 0; pl < st.n_planes; ++pl)
        if (dst[pl]) {
            const int n16 = st.plane_bytes[pl] >> 4, per = (n16 + split - 1) / split;
            const int lo = min(slice * per, n16), hi = min(lo + per, n16);
            if (hi > lo)
                bulk_g2s_hint(smem + ((size_t)off << 4), src + st.plane_off[pl] + ((size_t)lo << 4),
                              (uint32_t)(hi - lo) << 4, bar, pol.load);
            off += hi - lo;
        }
    while_loading();
    mbar_wait(bar, parity & 1u);
    parity ^= 1u;
    off = 0;
#pragma unroll 1
    for (int pl = 0; pl < st.n_planes; ++pl)
        if (dst[pl]) {
            const int n16 = st.plane_bytes[pl] >> 4, per = (n16 + split - 1) / split;
            const int lo = min(slice * per, n16), hi = min(lo + per, n16);
            if (hi > lo)
                bulk_s2g_hint(dst[pl] + (size_t)env * st.plane_bytes[pl] + ((size_t)lo << 4), smem + ((size_t)off << 4),
                              (uint32_t)(hi - lo) << 4, pol.store);
            off += hi - lo;
        }
    bulk_commit();
}

// whole: bit 0 / 1 = the observation / goal plane set is loaded as one span (bulk_copy_slice), only with split == 1.
// Trace record of a CTA (16 words): [0] resident, [1] predecessor complete, [2] first unit issued, [3] last unit
// issued, [4] shared memory drained, [5] units, [6] SM id, [8 + k] unit k issued (bit 63: nothing copied), k < 8.
__global__ void __launch_bounds__(32) vn_gather_bulk_kernel(const GatherParams p, int split, unsigned int *sched,
                                                            int whole) {
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ uint64_t bar;
    if (threadIdx.x != 0) return;
    unsigned long long *tr = p.trace ? p.trace + (size_t)blockIdx.x * 16 : nullptr;
    if (tr) {
        tr[0] = globaltimer_ns();
        unsigned int smid;
        asm volatile("mov.u32 %0, %smid;" : "=r"(smid));
        tr[6] = smid;
    }
    mbar_init(&bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    // the prologue above overlapped the scalar kernel; its results are needed from here on
    asm volatile("griddepcontrol.wait;" ::: "memory");
    if (p.early_release) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (tr) tr[1] = globaltimer_ns();
    int n_units = 0;
    uint32_t parity = 0;
    const L2Policies pol{l2_policy_evict_last(), l2_policy_evict_first()};
    const int units = p.n * split;
    const bool dynamic = sched != nullptr;
    // (record, goal record) of a unit; -1 = nothing to copy (row unchanged / no reset / past the end)
    auto unit_desc = [&](int u) -> int2 {
        if (u >= units) return make_int2(-1, -1);
        const int env = split == 1 ? u : u / split;
        if (p.desc) return p.desc[env];
        int2 d = make_int2(p.obs_state[env], -1);
        if (p.goal && (!p.did_reset || p.did_reset[env])) d.y = p.goal[env];
        return d;
    };
    // the first unit of every CTA is its block index (no atomic round trip before the first copy); the units
    // beyond the grid are handed out by the ticket counter.  The NEXT unit - its ticket and its descriptor, two
    // dependent round trips through L2 - is fetched while the copies of the current one are in flight.
    int u = (int)blockIdx.x;
    int2 d = unit_desc(u);
    while (u < units) {
        const int env = split == 1 ? u : u / split;
        const int slice = split == 1 ? 0 : u - env * split;
        int u_next = 0;
        int2 d_next = make_int2(-1, -1);
        bool have_next = false;
        auto fetch_next = [&]() {
            if (have_next) return;
            u_next = dynamic ? (int)gridDim.x + (int)atomicAdd(sched, 1u) : u + (int)gridDim.x;
            d_next = unit_desc(u_next);
            have_next = true;
        };
        if (d.x >= 0) {  // < 0: the row already holds this record (VN_STEP_SKIP_UNCHANGED)
            const uint8_t *src = p.store.base + (size_t)d.x * p.store.state_pitch;
            bulk_copy_slice(p.store, src, p.obs, env, slice, split, smem, &bar, parity, pol, fetch_next,
                            (whole & 1) != 0);
        }
        if (d.y >= 0) {
            const uint8_t *gsrc = p.store.base + (size_t)d.y * p.store.state_pitch;
            bulk_copy_slice(p.store, gsrc, p.goal_obs, env, slice, split, smem, &bar, parity, pol, fetch_next,
                            (whole & 2) != 0);
        }
        fetch_next();
        if (tr) {
            if (n_units == 0) tr[2] = globaltimer_ns();
            tr[3] = globaltimer_ns();
            if (n_units < 8) tr[8 + n_units] = tr[3] | ((unsigned long long)(d.x < 0 && d.y < 0) << 63);
            ++n_units;
        }
        u = u_next;
        d = d_next;
    }
    bulk_wait_read<0>();
    if (tr) {
        tr[4] = globaltimer_ns();
        tr[5] = (unsigned long long)n_units;
    }
    // no epilogue: the ticket counter of this launch (sched[parity]) is zeroed by the scalar half of the step that
    // next uses it - a fence + atomic + re-arm here sat on the critical path of every launch (~1 us)
}

// ---- fused single launch for small batches ----------------------------------------------------------
// A batch that fits in one wave of CTAs (C1: 16 envs; up to 444 envs for C2's records, see choose_fused) is bound
// by launch latency and by the chain of dependent memory round trips, not by bandwidth, so ONE kernel does both
// halves: one CTA per env, thread 0 steps the
// env, then lane 0 of warp w moves slice w of every plane - the observation record and, after a reset, the goal
// record, both in flight at once - with bulk async copies through a record-shaped region of shared memory.
constexpr int kFusedWarps = 4;
// VN_GATHER_AUTO runs a batch fused up to this many envs per SM (fewer when shared memory holds fewer records): beyond,
// the step is no longer bound by launch latency and the two-kernel path (pipelined, bandwidth-tuned) wins
constexpr int kFusedPerSm = 4;

template <bool kReset>
__global__ void __launch_bounds__(kFusedWarps * 32) vn_step_fused_kernel(const StepParams sp, const GatherParams gp) {
    extern __shared__ __align__(128) uint8_t smem[];  // [state_pitch] observation record (+ [state_pitch] goal record)
    __shared__ uint64_t bar[kFusedWarps];
    __shared__ int s_rec, s_grec;
    const int warp = threadIdx.x >> 5;
    if (threadIdx.x < kFusedWarps) mbar_init(&bar[threadIdx.x], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    const int env = blockIdx.x;
    if (threadIdx.x == 0) {
        EnvStats st;
        int rec, grec;
        step_env<kReset>(sp, env, st, rec, grec);
        if (sp.out.stats) add_stats(sp.out.stats, st);
        if (sp.out.gather_desc)  // for consumers after this launch (float batches, vn_gather_plane_f32_chw_rows)
            reinterpret_cast<int2 *>(sp.out.gather_desc)[(size_t)(sp.out.parity & 1) * sp.env.n_envs + env] =
                make_int2(rec, grec);
        s_rec = rec;
        s_grec = gp.goal ? grec : -1;
    }
    if (sp.out.host_seq)
        signal_host(sp.out);  // contains the block barrier
    else
        __syncthreads();
    if ((threadIdx.x & 31) != 0) return;
    const vn_store_t &S = gp.store;
    const uint8_t *src[2] = {s_rec >= 0 ? S.base + (size_t)s_rec * S.state_pitch : nullptr,
                             s_grec >= 0 ? S.base + (size_t)s_grec * S.state_pitch : nullptr};
    uint8_t *const *dst[2] = {gp.obs, gp.goal_obs};
    uint32_t total = 0;
    for (int k = 0; k < 2; ++k)
        if (src[k])
            for (int pl = 0; pl < S.n_planes; ++pl)
                if (dst[k][pl]) {
                    const int n16 = S.plane_bytes[pl] >> 4, per = (n16 + kFusedWarps - 1) / kFusedWarps;
                    const int lo = min(warp * per, n16), hi = min(lo + per, n16);
                    total += (uint32_t)(hi - lo) << 4;
                }
    if (total == 0) return;
    mbar_expect_tx(&bar[warp], total);
    for (int k = 0; k < 2; ++k)
        if (src[k])
            for (int pl = 0; pl < S.n_planes; ++pl)
                if (dst[k][pl]) {
                    const int n16 = S.plane_bytes[pl] >> 4, per = (n16 + kFusedWarps - 1) / kFusedWarps;
                    const int lo = min(warp * per, n16), hi = min(lo + per, n16);
                    if (hi > lo)
                        bulk_g2s(smem + (size_t)k * S.state_pitch + S.plane_off[pl] + ((size_t)lo << 4),
                                 src[k] + S.plane_off[pl] + ((size_t)lo << 4), (uint32_t)(hi - lo) << 4, &bar[warp]);
                }
    mbar_wait(&bar[warp], 0);
    for (int k = 0; k < 2; ++k)
        if (src[k])
            for (int pl = 0; pl < S.n_planes; ++pl)
                if (dst[k][pl]) {
                    const int n16 = S.plane_bytes[pl] >> 4, per = (n16 + kFusedWarps - 1) / kFusedWarps;
                    const int lo = min(warp * per, n16), hi = min(lo + per, n16);
                    if (hi > lo)
                        bulk_s2g(dst[k][pl] + (size_t)env * S.plane_bytes[pl] + ((size_t)lo << 4),
                                 smem + (size_t)k * S.state_pitch + S.plane_off[pl] + ((size_t)lo << 4),
                                 (uint32_t)(hi - lo) << 4);
                }
    bulk_commit();
    bulk_wait_read<0>();
}

// ---- persistent single launch for large batches -----------------------------------------------------
// ONE launch per vectorised step for batches beyond one wave of CTAs: a persistent grid of one-warp CTAs (as many per
// SM as shared memory holds records).  CTA b OWNS the envs b, b + G, b + 2G, ... for the whole launch:
//   phase A  its lanes step those envs (step_env, one env per lane and round) - every env of the batch is stepped
//            within the first microseconds of the launch, so a host caller gets rewards / dones while the copies run:
//            lane 1 issues ONE system-scope fence for the CTA's writes to the mapped host pack and arrives on a
//            device counter; the last CTA to arrive publishes `seq` in host_seq[0];
//   phase B  lane 0 moves the records of the same envs with bulk async copies (global -> shared -> global), reading
//            the (record, goal record) pairs its own warp just wrote to the gather descriptors.
// No CTA ever waits for another one (ownership is static), nothing goes through a second launch, and there is no
// descriptor hand-off between kernels: the scalar kernel, the PDL hand-off and the ticket counter of the two-kernel
// path are gone.  Records that need slicing (split > 1) stay on the two-kernel path.
// whole: as for vn_gather_bulk_kernel.
template <bool kReset>
__global__ void __launch_bounds__(32) vn_step_gather_kernel(const StepParams sp, const GatherParams gp, int whole) {
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ uint64_t bar;
    const int lane = threadIdx.x;
    if (lane == 0) {
        mbar_init(&bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // everything above overlapped the previous kernel of the stream; its env state is needed from here on
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    const int n = sp.env.n_envs, G = (int)gridDim.x, b = (int)blockIdx.x;
    int2 *desc = reinterpret_cast<int2 *>(sp.out.gather_desc) + (size_t)(sp.out.parity & 1) * n;

    // ---- phase A: step the envs this CTA owns
    EnvStats acc;
    for (int base = b; base < n; base += 32 * G) {   // uniform trip count across the warp
        const int e = base + lane * G;
        if (e < n) {
            EnvStats st;
            int rec, grec;
            step_env<kReset>(sp, e, st, rec, grec);
            desc[e] = make_int2(rec, grec);
            acc += st;
        }
    }
    if (sp.out.stats) {
        const EnvStats w = warp_reduce(acc);
        if (lane == 0) add_stats(sp.out.stats, w);
    }
    __syncwarp();   // the lanes' descriptor / host-pack writes are ordered before what lanes 0 and 1 do next
    if (lane == 1 && sp.out.host_seq) {
        // one system-scope fence per CTA (cumulative over the warp's writes ordered by the barrier above), then arrive;
        // the last CTA publishes the sequence word the host spins on and re-arms the counter
        __threadfence_system();
        unsigned int *arrive = sp.out.sched + 2;
        if (atomicAdd(arrive, 1u) == (unsigned int)G - 1u) {
            *arrive = 0u;
            __threadfence_system();
            *reinterpret_cast<volatile uint32_t *>(sp.out.host_seq) = sp.out.seq;
        }
    }
    if (lane != 0) return;

    // ---- phase B: copy the records of the same envs
    uint32_t parity = 0;
    const L2Policies pol{l2_policy_evict_last(), l2_policy_evict_first()};
    int2 d = desc[b];
    for (int e = b; e < n; e += G) {
        int2 d_next = make_int2(-1, -1);
        bool have_next = false;
        auto fetch_next = [&]() {  // the next descriptor is read while this env's copies are in flight
            if (!have_next && e + G < n) d_next = desc[e + G];
            have_next = true;
        };
        if (d.x >= 0)  // < 0: the row already holds this record (VN_STEP_SKIP_UNCHANGED)
            bulk_copy_slice(gp.store, gp.store.base + (size_t)d.x * gp.store.state_pitch, gp.obs, e, 0, 1, smem, &bar,
                            parity, pol, fetch_next, (whole & 1) != 0);
        if (d.y >= 0 && gp.goal)
            bulk_copy_slice(gp.store, gp.store.base + (size_t)d.y * gp.store.state_pitch, gp.goal_obs, e, 0, 1, smem,
                            &bar, parity, pol, fetch_next, (whole & 2) != 0);
        fetch_next();
        d = d_next;
    }
    bulk_wait_read<0>();
}

// =====================================================================================================
// synthetic store fill
// =====================================================================================================
struct FillParams {
    vn_store_t store;
    int32_t plane_ids[VN_MAX_PLANES];
    int32_t record0, n_records, scene, state0;
    uint64_t seed;
};

__global__ void __launch_bounds__(256) vn_fill_kernel(const FillParams p) {
    const int64_t words_per_rec = p.store.state_pitch >> 3;
    const int64_t total = words_per_rec * p.n_records;
    for (int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; w < total; w += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = w / words_per_rec;
        const int32_t byte = (int32_t)((w - r * words_per_rec) << 3);
        uint64_t val = 0;  // padding between planes is zero
#pragma unroll 1
        for (int pl = 0; pl < p.store.n_planes; ++pl) {
            const int32_t o = byte - p.store.plane_off[pl];
            if (o >= 0 && o < p.store.plane_bytes[pl]) {
                const uint64_t key = frame_key(p.seed, (uint32_t)p.scene, (uint64_t)(p.state0 + r), p.plane_ids[pl]);
                val = splitmix64(key + (uint64_t)(o >> 3));
            }
        }
        *reinterpret_cast<uint64_t *>(const_cast<uint8_t *>(p.store.base) + (p.record0 + r) * p.store.state_pitch +
                                      byte) = val;
    }
}

// =====================================================================================================
// host side
// =====================================================================================================
static int32_t validate_store(const vn_store_t *s) {
    VN_REQUIRE(s && s->base, "store: null");
    VN_REQUIRE(s->n_planes >= 1 && s->n_planes <= VN_MAX_PLANES, "store: n_planes=%d", s->n_planes);
    VN_REQUIRE((reinterpret_cast<uintptr_t>(s->base) & 127) == 0, "store: base must be 128-byte aligned");
    VN_REQUIRE(s->state_pitch > 0 && (s->state_pitch & 127) == 0, "store: state_pitch must be a multiple of 128");
    for (int i = 0; i < s->n_planes; ++i) {
        VN_REQUIRE(s->plane_bytes[i] > 0 && (s->plane_bytes[i] & 15) == 0,
                   "store: plane %d size %d is not a multiple of 16", i, s->plane_bytes[i]);
        VN_REQUIRE((s->plane_off[i] & 127) == 0 && s->plane_off[i] + (int64_t)s->plane_bytes[i] <= s->state_pitch,
                   "store: plane %d offset %d", i, s->plane_off[i]);
    }
    return VN_OK;
}

constexpr int kMaxDevices = 64;
static int current_device() {
    int dev = 0;
    cudaGetDevice(&dev);
    return dev >= 0 && dev < kMaxDevices ? dev : 0;
}
int sm_count() {
    static int cached[kMaxDevices] = {0};
    const int dev = current_device();
    if (!cached[dev]) {
        cudaDeviceGetAttribute(&cached[dev], cudaDevAttrMultiProcessorCount, dev);
        if (cached[dev] <= 0) cached[dev] = 148;
    }
    return cached[dev];
}

int32_t ensure_smem(const void *kernel, int bytes) {
    static std::mutex mu;
    static std::map<std::pair<const void *, int>, int> configured;  // (kernel, device) -> bytes
    const int dev = current_device();
    std::lock_guard<std::mutex> lock(mu);
    int &have = configured[{kernel, dev}];
    if (bytes <= have) return VN_OK;
    const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e != cudaSuccess) {
        cudaGetLastError();
        set_error("%d bytes of dynamic shared memory: %s", bytes, cudaGetErrorString(e));
        return VN_ECUDA;
    }
    have = bytes;
    return VN_OK;
}

static int32_t check_rows_aligned(const GatherParams &gp) {
    for (int pl = 0; pl < gp.store.n_planes; ++pl) {
        VN_REQUIRE(aligned16(gp.obs[pl]), "gather: obs[%d] must be 16-byte aligned", pl);
        VN_REQUIRE(aligned16(gp.goal_obs[pl]), "gather: goal_obs[%d] must be 16-byte aligned", pl);
    }
    return VN_OK;
}

// Shared memory a CTA needs for one whole record of a plane set, and whether that set is CONTIGUOUS in the record
// (nothing but alignment padding between its planes): then *span covers it with one load.
static int plane_set_bytes(const vn_store_t &st, uint8_t *const *dst, bool use, int *span, bool *contiguous) {
    int sum = 0, first = -1, last = -1;
    for (int pl = 0; pl < st.n_planes; ++pl)
        if (use && dst[pl]) {
            sum += st.plane_bytes[pl];
            if (first < 0) first = pl;
            last = pl;
        }
    *span = first < 0 ? 0 : st.plane_off[last] + st.plane_bytes[last] - st.plane_off[first];
    *contiguous = first >= 0 && last > first && *span - sum <= 128 * (last - first);
    return sum;
}

// The gather half of a two-kernel step, and the gather-only entry points (vn_env_gather, vn_gather_plane): there is
// no scalar half here, so the one-launch modes mean VN_GATHER_BULK.
static int32_t launch_gather(const GatherParams &gp, int32_t variant, cudaStream_t stream) {
    if (gp.n == 0) return VN_OK;
    int32_t rc = check_rows_aligned(gp);
    if (rc) return rc;
    // measured on B200 (profiles/): the bulk-copy variant reaches 94 % of the copy peak, LDG.128 86 %
    if (variant == VN_GATHER_AUTO || variant == VN_GATHER_FUSED || variant == VN_GATHER_PERSISTENT)
        variant = VN_GATHER_BULK;
    if (variant == VN_GATHER_LDG) {
        constexpr int kThreads = 256;
        return launch(vn_gather_ldg_kernel<kThreads, 4>, "vn_gather_ldg_kernel", dim3(gp.n), dim3(kThreads), 0, stream,
                      true, gp);
    }
    if (variant != VN_GATHER_BULK) {
        set_error("gather: unknown variant %d", variant);
        return VN_EINVAL;
    }
    // small batches (C1: 16 envs) cannot fill 148 SMs with one record per CTA: cut each record into
    // slices until there are ~2 units per SM (latency-bound regime; one slice >= 2 KB)
    int split = gp.n < 2 * sm_count() ? min(16, (2 * sm_count() + gp.n - 1) / gp.n) : 1;
    // large records (the reference's native 174 x 174 frames: 212 KB for rgb + depth + segmentation) are
    // cut into slices of at most 52 KB so that at least 4 CTAs stay resident per SM (84 x 84 rgb + depth +
    // segmentation = 49.6 KB stays whole: one load per record instead of two slices of three)
    int per_env = 0, per_goal = 0;
    for (int pl = 0; pl < gp.store.n_planes; ++pl) {
        if (gp.obs[pl]) per_env += gp.store.plane_bytes[pl];
        if (gp.goal && gp.goal_obs[pl]) per_goal += gp.store.plane_bytes[pl];
    }
    split = max(split, (max(per_env, per_goal) + 52 * 1024 - 1) / (52 * 1024));
    int smem_obs = 0, smem_goal = 0;
    for (int pl = 0; pl < gp.store.n_planes; ++pl) {
        const int n16 = gp.store.plane_bytes[pl] >> 4, per = (n16 + split - 1) / split;
        if (gp.obs[pl]) smem_obs += per << 4;
        if (gp.goal && gp.goal_obs[pl]) smem_goal += per << 4;
    }
    int smem = max(smem_obs, smem_goal), whole = 0;
    if (split == 1) {
        int span_o, span_g;
        bool co, cg;
        plane_set_bytes(gp.store, gp.obs, true, &span_o, &co);
        plane_set_bytes(gp.store, gp.goal_obs, gp.goal != nullptr, &span_g, &cg);
        if (co) smem = max(smem, span_o);
        if (cg) smem = max(smem, span_g);
        whole = (co ? 1 : 0) | (cg ? 2 : 0);
    }
    VN_REQUIRE(smem <= 200 * 1024, "gather(bulk): %d bytes of planes per env exceed shared memory", smem);
    rc = ensure_smem(vn_gather_bulk_kernel, smem);
    if (rc) return rc;
    const int grid = (int)min((int64_t)gp.n * split, (int64_t)sm_count() * ctas_per_sm(smem));
    return launch(vn_gather_bulk_kernel, "vn_gather_bulk_kernel", dim3(grid), dim3(32), (size_t)smem, stream, true, gp,
                  split, gp.sched ? gp.sched + (gp.parity & 1) : nullptr, whole);
}

static int32_t make_step_params(StepParams &sp, const vn_tables_t *tab, const vn_envs_t *envs, const vn_rules_t *rules,
                                const vn_inject_t *inj, const int32_t *actions, const uint8_t *mask,
                                const vn_step_out_t *out, bool reset, int32_t *actions_copy) {
    VN_REQUIRE(tab && tab->adj && tab->task_goal && tab->task_cand_off && tab->task_prefix && tab->cand_state,
               "tables: null pointer");
    VN_REQUIRE(tab->n_tasks > 0, "tables: n_tasks=%d", tab->n_tasks);
    VN_REQUIRE(envs->state && envs->goal && envs->task && envs->elapsed && envs->epoch && envs->ep_return &&
                   envs->ep_length && envs->task_lo && envs->task_cnt,
               "envs: null pointer");
    VN_REQUIRE(rules && rules->n_actions >= 1 && rules->n_actions <= 16, "rules: n_actions");
    VN_REQUIRE(rules->goal_compare >= 0 && rules->goal_compare <= 2, "rules: goal_compare=%d", rules->goal_compare);
    VN_REQUIRE(isfinite(rules->reward_progress), "rules: reward_progress=%g is not finite", (double)rules->reward_progress);
    VN_REQUIRE(rules->reward_progress == 0.0f || tab->task_dist,
               "rules: reward_progress=%g needs tables->task_dist (the [n_tasks][n_states] distance table)",
               (double)rules->reward_progress);
    VN_REQUIRE(out && out->obs_state, "out: obs_state scratch is required");
    VN_REQUIRE(reset || actions, "step: actions is null");
    VN_REQUIRE(!inj || !inj->start || inj->stride > 0, "inject: stride=%d", inj ? inj->stride : 0);
    const vn_episodes_t *ep = envs->episodes;
    if (ep) {
        VN_REQUIRE(!inj || !inj->start, "episodes: a list cannot be combined with an injected reset stream (inject)");
        VN_REQUIRE(rules->flags & VN_RULE_AUTO_RESET, "episodes: a list needs VN_RULE_AUTO_RESET in rules->flags");
        VN_REQUIRE(!(reset && mask), "episodes: a masked reset cannot run while a list is installed");
        VN_REQUIRE(ep->n_episodes >= 0, "episodes: n_episodes=%d", ep->n_episodes);
        VN_REQUIRE(ep->cursor && ep->count, "episodes: cursor and count are required");
        VN_REQUIRE(ep->n_episodes == 0 || (ep->task && ep->start && ep->length && ep->ret && ep->win &&
                                           ep->truncated && ep->final_state),
                   "episodes: null list or result pointer with n_episodes=%d", ep->n_episodes);
        VN_REQUIRE(envs->env_id_base >= 0 && ep->stride >= (int64_t)envs->env_id_base + envs->n_envs,
                   "episodes: stride=%d is less than env_id_base + n_envs = %d + %d", ep->stride, envs->env_id_base,
                   envs->n_envs);
        sp.eps = *ep;
    } else {
        memset(&sp.eps, 0, sizeof(sp.eps));
    }
    sp.tab = *tab;
    sp.env = *envs;
    sp.rules = *rules;
    if (inj)
        sp.inj = *inj;
    else
        sp.inj = vn_inject_t{nullptr, nullptr, 0, 0};
    sp.out = *out;
    sp.actions = actions;
    sp.mask = mask;
    sp.actions_copy = actions_copy;
    // rows can only be skipped when the gather half learns about it through the descriptors
    sp.skip_rows = (out->flags & VN_STEP_SKIP_UNCHANGED) && out->gather_desc != nullptr;
    return VN_OK;
}

static int32_t run_scalar(const vn_tables_t *tab, const vn_envs_t *envs, const vn_rules_t *rules,
                          const vn_inject_t *inj, const int32_t *actions, const uint8_t *mask,
                          const vn_step_out_t *out, void *stream, bool reset, int32_t *actions_copy = nullptr) {
    VN_REQUIRE(envs && envs->n_envs >= 0, "envs: null or negative n_envs");
    if (envs->n_envs == 0) return VN_OK;  // an empty shard (more ranks than envs): nothing to do, nothing to check
    StepParams sp;
    int32_t rc = make_step_params(sp, tab, envs, rules, inj, actions, mask, out, reset, actions_copy);
    if (rc) return rc;
    const int blocks = (envs->n_envs + kStepThreads - 1) / kStepThreads;
    return launch(reset ? vn_step_kernel<true> : vn_step_kernel<false>, "vn_step_kernel", dim3(blocks),
                  dim3(kStepThreads), 0, static_cast<cudaStream_t>(stream), true, sp);
}

// *any = whether there is anything to gather at all
static int32_t make_gather_params(GatherParams &gp, const vn_store_t *store, const vn_envs_t *envs,
                                  const vn_step_out_t *out, bool *any) {
    int32_t rc = validate_store(store);
    if (rc) return rc;
    VN_REQUIRE(envs->goal, "envs: null pointer");
    VN_REQUIRE(out && out->obs_state, "out: obs_state is required");
    gp.store = *store;
    gp.obs_state = out->obs_state;
    gp.n = envs->n_envs;
    bool any_goal = false, any_obs = false;
    for (int pl = 0; pl < VN_MAX_PLANES; ++pl) {
        gp.obs[pl] = pl < store->n_planes ? out->obs[pl] : nullptr;
        gp.goal_obs[pl] = pl < store->n_planes ? out->goal_obs[pl] : nullptr;
        any_goal |= gp.goal_obs[pl] != nullptr;
        any_obs |= gp.obs[pl] != nullptr;
    }
    gp.goal = any_goal ? envs->goal : nullptr;
    gp.did_reset = out->did_reset;
    gp.sched = out->sched;
    gp.parity = out->parity;
    gp.early_release = 1;
    gp.trace = g_gather_trace;
    gp.desc = out->gather_desc
                  ? reinterpret_cast<const int2 *>(out->gather_desc) + (size_t)(out->parity & 1) * envs->n_envs
                  : nullptr;
    VN_REQUIRE(!any_goal || out->did_reset, "out: did_reset is required when goal planes are emitted");
    *any = any_goal || any_obs;
    return VN_OK;
}

static int32_t run_gather(const vn_store_t *store, const vn_envs_t *envs, const vn_step_out_t *out, int32_t variant,
                          void *stream) {
    VN_REQUIRE(envs && envs->n_envs >= 0, "envs: null or negative n_envs");
    if (envs->n_envs == 0) return VN_OK;
    GatherParams gp;
    bool any = false;
    int32_t rc = make_gather_params(gp, store, envs, out, &any);
    if (rc) return rc;
    if (!any) return VN_OK;
    return launch_gather(gp, variant, static_cast<cudaStream_t>(stream));
}

// Whether vn_env_step / vn_env_reset / vn_env_step_host run as the single fused launch: on request
// (VN_GATHER_FUSED), or by default (VN_GATHER_AUTO) for batches of at most one env per SM.
static int32_t fused_smem_bytes(const vn_store_t *store, const vn_step_out_t *out) {
    bool any_goal = false;
    for (int pl = 0; pl < store->n_planes; ++pl) any_goal |= out->goal_obs[pl] != nullptr;
    const int64_t smem = store->state_pitch * (any_goal ? 2 : 1);
    return smem <= 200 * 1024 ? (int32_t)smem : -1;
}

static int32_t run_fused(const vn_store_t *store, const vn_tables_t *tab, const vn_envs_t *envs, const vn_rules_t *rules,
                         const vn_inject_t *inj, const int32_t *actions, const uint8_t *mask, const vn_step_out_t *out,
                         void *stream, bool reset, int32_t *actions_copy, int32_t smem) {
    StepParams sp;
    int32_t rc = make_step_params(sp, tab, envs, rules, inj, actions, mask, out, reset, actions_copy);
    if (rc) return rc;
    sp.skip_rows = (out->flags & VN_STEP_SKIP_UNCHANGED) != 0;  // the record index never leaves the kernel
    GatherParams gp;
    bool any = false;
    rc = make_gather_params(gp, store, envs, out, &any);
    if (!rc) rc = check_rows_aligned(gp);
    if (rc) return rc;
    const auto kernel = reset ? vn_step_fused_kernel<true> : vn_step_fused_kernel<false>;
    rc = ensure_smem(kernel, smem);
    if (rc) return rc;
    return launch(kernel, "vn_step_fused_kernel", dim3(envs->n_envs), dim3(kFusedWarps * 32), (size_t)smem,
                  static_cast<cudaStream_t>(stream), true, sp, gp);
}

// Shared memory of one CTA of the persistent single launch (largest of the observation / goal plane sets), or 0 when
// the batch does not qualify: needs the descriptor and scheduler scratch, whole records per CTA (no slicing) and at
// least two CTAs per SM.
static int32_t persistent_smem_bytes(const vn_store_t *store, const vn_step_out_t *out, int *whole = nullptr) {
    if (!out || !out->gather_desc || !out->sched) return 0;
    int span_o, span_g;
    bool co, cg;
    const int obs = plane_set_bytes(*store, out->obs, true, &span_o, &co);
    const int goal = plane_set_bytes(*store, out->goal_obs, true, &span_g, &cg);
    int smem = max(obs, goal);
    if (co) smem = max(smem, span_o);
    if (cg) smem = max(smem, span_g);
    if (whole) *whole = (co ? 1 : 0) | (cg ? 2 : 0);
    if (smem == 0 || smem > 52 * 1024) return 0;   // >= 4 CTAs per SM; larger records are sliced by the two-kernel path
    return smem;
}

static int32_t run_persistent(const vn_store_t *store, const vn_tables_t *tab, const vn_envs_t *envs,
                              const vn_rules_t *rules, const vn_inject_t *inj, const int32_t *actions, const uint8_t *mask,
                              const vn_step_out_t *out, void *stream, bool reset, int32_t *actions_copy, int32_t smem) {
    StepParams sp;
    int32_t rc = make_step_params(sp, tab, envs, rules, inj, actions, mask, out, reset, actions_copy);
    if (rc) return rc;
    GatherParams gp;
    bool any = false;
    rc = make_gather_params(gp, store, envs, out, &any);
    if (!rc) rc = check_rows_aligned(gp);
    if (rc) return rc;
    const auto kernel = reset ? vn_step_gather_kernel<true> : vn_step_gather_kernel<false>;
    rc = ensure_smem(kernel, smem);
    if (rc) return rc;
    int whole = 0;
    persistent_smem_bytes(store, out, &whole);
    const int grid = (int)min((int64_t)envs->n_envs, (int64_t)sm_count() * ctas_per_sm(smem));
    return launch(kernel, "vn_step_gather_kernel", dim3(grid), dim3(32), (size_t)smem, static_cast<cudaStream_t>(stream),
                  true, sp, gp, whole);
}

enum StepMode { kModeError = -1, kModeSplit = 0, kModeFused = 1, kModePersistent = 2 };

// How vn_env_reset / vn_env_step / vn_env_step_host run: *smem receives the dynamic shared memory of the one-launch
// modes.  VN_GATHER_AUTO: the CTA-per-env fused launch for batches of one wave, the persistent launch beyond that when
// the batch qualifies, else scalar kernel + gather kernel.
static StepMode choose_mode(const vn_store_t *store, const vn_envs_t *envs, const vn_step_out_t *out, int32_t variant,
                            int32_t *smem);

// -1: error already set; 0: two launches; > 0: fused, shared memory bytes
static int32_t choose_fused(const vn_store_t *store, const vn_envs_t *envs, const vn_step_out_t *out, int32_t variant) {
    if (variant != VN_GATHER_FUSED && variant != VN_GATHER_AUTO) return 0;
    if (!out) return 0;  // reported by the parameter checks
    const int32_t smem = fused_smem_bytes(store, out);
    if (smem < 0) {
        if (variant == VN_GATHER_AUTO) return 0;
        set_error("gather(fused): a %lld-byte record (x2 with goal planes) exceeds shared memory",
                  (long long)store->state_pitch);
        return -1;
    }
    // one wave of CTAs: as many envs as fit at once, at most kFusedPerSm per SM
    if (variant == VN_GATHER_AUTO && envs->n_envs > sm_count() * ctas_per_sm(smem, kFusedPerSm)) return 0;
    return smem;
}

// Float observation mode as part of the step: one more kernel converts this step's records into the float leaves.
static int32_t run_float_leaves(const vn_store_t *store, const vn_envs_t *envs, const vn_step_out_t *out, void *stream) {
    if (!out->float_leaves || out->n_float_leaves <= 0) return VN_OK;
    VN_REQUIRE(out->gather_desc, "float_leaves: out->gather_desc is required");
    const int32_t *desc = out->gather_desc + (size_t)(out->parity & 1) * envs->n_envs * 2;
    return launch_float_leaves(store, out->float_leaves, out->n_float_leaves, desc, envs->n_envs, out->float_h,
                               out->float_w, stream, true);
}

static StepMode choose_mode(const vn_store_t *store, const vn_envs_t *envs, const vn_step_out_t *out, int32_t variant,
                            int32_t *smem) {
    *smem = 0;
    if (variant == VN_GATHER_PERSISTENT) {
        *smem = persistent_smem_bytes(store, out);
        if (*smem <= 0) {
            set_error("gather(persistent): needs out->gather_desc, out->sched and plane sets of at most 52 KB per env");
            return kModeError;
        }
        return kModePersistent;
    }
    const int32_t fused = choose_fused(store, envs, out, variant);
    if (fused < 0) return kModeError;
    if (fused > 0) {
        *smem = fused;
        return kModeFused;
    }
    if (variant == VN_GATHER_AUTO) {
        // Measured on B200 (profiles/r2a_launch_modes.txt, r2c_small_batches.txt, r2_serial_modes.txt; C2 records):
        //  * PIPELINED steps (VN_STEP_ACTIONS_READY: the scalar kernel of the two-kernel path hides behind the previous
        //    gather): the persistent launch wins while the batch fills at most ~3/4 of one wave of its CTAs (300 envs
        //    9.3 -> 6.8 us per step, 512: 9.1 -> 7.1, 768: 9.2 -> 9.0) and loses beyond (1,024: 9.5 vs 9.9 us; 4,096: 33.3
        //    vs 35.8) - its stepping phase is exposed;
        //  * SERIAL steps (the actions were produced just now, e.g. by a policy kernel between two steps - nothing can
        //    overlap the previous gather): one launch beats scalar kernel + hand-off + gather up to about four envs per CTA
        //    (1,024 envs: 11.8 -> 10.1 us, 2,048: 19.2 -> 16.6, 4,096: 37.4 -> 36.9, RGB-only 4,096: 27.4 -> 24.9) and
        //    loses beyond (8,192: 66.0 vs 70.2, 16,384: 122.6 vs 135.5): the two-kernel path's tickets balance skipped rows
        //    and L2 hits, the persistent launch owns envs statically.
        // A HOST caller (out->host_pack) always takes two kernels: the stepping phase of a persistent grid cannot become
        // resident before the previous launch's CTAs release their shared memory, so the host would get its rewards a
        // whole gather late, and lanes that own strided envs read / write the mapped host buffers 4 bytes at a time.
        const int32_t ps = persistent_smem_bytes(store, out);
        if (ps > 0) {
            const int64_t wave = (int64_t)sm_count() * ctas_per_sm(ps), n = envs->n_envs;
            const bool pipelined = (out->flags & VN_STEP_ACTIONS_READY) != 0;
            if (!out->host_pack && (pipelined ? 4 * n <= 3 * wave : n <= 4 * wave)) {
                *smem = ps;
                return kModePersistent;
            }
        }
    }
    return kModeSplit;
}

static int32_t run_step(const vn_store_t *store, const vn_tables_t *tab, const vn_envs_t *envs, const vn_rules_t *rules,
                        const vn_inject_t *inj, const int32_t *actions, const uint8_t *mask, const vn_step_out_t *out,
                        int32_t variant, void *stream, bool reset) {
    VN_REQUIRE(envs && envs->n_envs >= 0, "envs: null or negative n_envs");
    if (envs->n_envs == 0) return VN_OK;
    int32_t rc = validate_store(store);  // fail before anything is enqueued
    if (rc) return rc;
    int32_t smem = 0;
    const StepMode mode = choose_mode(store, envs, out, variant, &smem);
    if (mode == kModeError) return VN_EINVAL;
    if (mode == kModeFused)
        rc = run_fused(store, tab, envs, rules, inj, actions, mask, out, stream, reset, nullptr, smem);
    else if (mode == kModePersistent)
        rc = run_persistent(store, tab, envs, rules, inj, actions, mask, out, stream, reset, nullptr, smem);
    else {
        rc = run_scalar(tab, envs, rules, inj, actions, mask, out, stream, reset);
        if (rc) return rc;
        rc = run_gather(store, envs, out, variant, stream);
    }
    if (rc) return rc;
    return run_float_leaves(store, envs, out, stream);
}

// Pinned + device-mapped?  The answer for the last few pointers is remembered per thread: the query costs about
// a microsecond and the host-facing step asks about the same three buffers every call.  (A buffer that is freed and
// whose address comes back as pageable memory would pass from the cache; the kernel then faults on the unmapped
// address - a loud failure, and only for callers that free the staging buffers of a live env.)
static bool is_mapped_host(const void *p) {
    constexpr int kSlots = 8;
    static thread_local const void *known[kSlots] = {nullptr};
    static thread_local int next = 0;
    for (int i = 0; i < kSlots; ++i)
        if (known[i] == p) return true;
    cudaPointerAttributes pa;
    if (cudaPointerGetAttributes(&pa, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    if (pa.type != cudaMemoryTypeHost || pa.devicePointer == nullptr) return false;
    known[next] = p;
    next = (next + 1) % kSlots;
    return true;
}

}  // namespace vn

// =====================================================================================================
// C ABI
// =====================================================================================================
extern "C" {

int32_t vn_abi_version(void) { return VN_ABI_VERSION; }

int32_t vn_abi_struct_size(int32_t which) {
    switch (which) {
        case 0: return (int32_t)sizeof(vn_store_t);
        case 1: return (int32_t)sizeof(vn_tables_t);
        case 2: return (int32_t)sizeof(vn_envs_t);
        case 3: return (int32_t)sizeof(vn_rules_t);
        case 4: return (int32_t)sizeof(vn_inject_t);
        case 5: return (int32_t)sizeof(vn_step_out_t);
        case 6: return (int32_t)sizeof(vn_replay_t);
        case 7: return (int32_t)sizeof(vn_float_leaf_t);
        case 8: return (int32_t)sizeof(vn_host_call_t);
        case 9: return (int32_t)sizeof(vn_u8_frames_t);
        case 10: return (int32_t)sizeof(vn_episodes_t);
        default: return -1;
    }
}
const char *vn_last_error(void) { return vn::g_error.c_str(); }
int64_t vn_launch_count(void) { return (int64_t)vn::g_launches.load(std::memory_order_relaxed); }

int32_t vn_fill_store(const vn_store_t *store, int32_t record0, int32_t n_records, uint64_t seed, int32_t scene,
                      int32_t state0, const int32_t *plane_ids, void *stream) {
    int32_t rc = vn::validate_store(store);
    if (rc) return rc;
    VN_REQUIRE(plane_ids, "fill: plane_ids is null");
    VN_REQUIRE(record0 >= 0 && n_records >= 0 && record0 + (int64_t)n_records <= store->n_states,
               "fill: records [%d, %d) outside the store (%d)", record0, record0 + n_records, store->n_states);
    if (n_records == 0) return VN_OK;
    vn::FillParams fp;
    fp.store = *store;
    for (int i = 0; i < VN_MAX_PLANES; ++i) fp.plane_ids[i] = i < store->n_planes ? plane_ids[i] : 0;
    fp.record0 = record0;
    fp.n_records = n_records;
    fp.scene = scene;
    fp.state0 = state0;
    fp.seed = seed;
    const int64_t total = (store->state_pitch >> 3) * n_records;
    const int blocks = (int)((total + 255) / 256 < (int64_t)vn::sm_count() * 32 ? (total + 255) / 256
                                                                                 : (int64_t)vn::sm_count() * 32);
    return vn::launch(vn::vn_fill_kernel, "vn_fill_kernel", dim3(blocks), dim3(256), 0, static_cast<cudaStream_t>(stream),
                      false, fp);
}

int32_t vn_env_reset(const vn_store_t *store, const vn_tables_t *tables, const vn_envs_t *envs,
                     const vn_rules_t *rules, const vn_inject_t *inject, const uint8_t *mask,
                     const vn_step_out_t *out, int32_t gather_variant, void *stream) {
    return vn::run_step(store, tables, envs, rules, inject, nullptr, mask, out, gather_variant, stream, true);
}

int32_t vn_env_step(const vn_store_t *store, const vn_tables_t *tables, const vn_envs_t *envs,
                    const vn_rules_t *rules, const vn_inject_t *inject, const int32_t *actions,
                    const vn_step_out_t *out, int32_t gather_variant, void *stream) {
    return vn::run_step(store, tables, envs, rules, inject, actions, nullptr, out, gather_variant, stream, false);
}

int32_t vn_env_step_scalar(const vn_tables_t *tables, const vn_envs_t *envs, const vn_rules_t *rules,
                           const vn_inject_t *inject, const int32_t *actions, const vn_step_out_t *out, void *stream) {
    return vn::run_scalar(tables, envs, rules, inject, actions, nullptr, out, stream, false);
}

int32_t vn_env_gather(const vn_store_t *store, const vn_envs_t *envs, const vn_step_out_t *out,
                      int32_t gather_variant, void *stream) {
    return vn::run_gather(store, envs, out, gather_variant, stream);
}

int32_t vn_env_step_host(const vn_store_t *store, const vn_tables_t *tables, const vn_envs_t *envs,
                         const vn_rules_t *rules, const vn_inject_t *inject, const int32_t *host_actions,
                         int32_t *dev_actions_copy, const vn_step_out_t *out, void *ready_event,
                         int32_t gather_variant, void *stream) {
    VN_REQUIRE(envs && envs->n_envs >= 0, "envs: null or negative n_envs");
    if (envs->n_envs == 0) return VN_OK;
    int32_t rc = vn::validate_store(store);
    if (rc) return rc;
    VN_REQUIRE(host_actions, "step_host: host_actions is null");
    VN_REQUIRE(vn::is_mapped_host(host_actions),
               "step_host: host_actions must be pinned (page-locked, device-mapped) host memory");
    VN_REQUIRE(!out || !out->host_pack || vn::is_mapped_host(out->host_pack),
               "step_host: out->host_pack must be pinned (page-locked, device-mapped) host memory");
    VN_REQUIRE(!out || !out->host_seq || vn::is_mapped_host(out->host_seq),
               "step_host: out->host_seq must be pinned (page-locked, device-mapped) host memory");
    int32_t smem = 0;
    const vn::StepMode mode = vn::choose_mode(store, envs, out, gather_variant, &smem);
    if (mode == vn::kModeError) return VN_EINVAL;
    const bool one_launch = mode != vn::kModeSplit;
    // the scalar part reads the actions from, and mirrors its per-env results to, mapped host memory
    if (mode == vn::kModeFused)
        rc = vn::run_fused(store, tables, envs, rules, inject, host_actions, nullptr, out, stream, false,
                           dev_actions_copy, smem);
    else if (mode == vn::kModePersistent)
        rc = vn::run_persistent(store, tables, envs, rules, inject, host_actions, nullptr, out, stream, false,
                                dev_actions_copy, smem);
    else
        rc = vn::run_scalar(tables, envs, rules, inject, host_actions, nullptr, out, stream, false, dev_actions_copy);
    if (rc) return rc;
    if (ready_event) {
        cudaError_t e = cudaEventRecord(static_cast<cudaEvent_t>(ready_event), static_cast<cudaStream_t>(stream));
        if (e != cudaSuccess) {
            vn::set_error("step_host: event record: %s", cudaGetErrorString(e));
            return VN_ECUDA;
        }
    }
    if (!one_launch) {
        rc = vn::run_gather(store, envs, out, gather_variant, stream);
        if (rc) return rc;
    }
    return vn::run_float_leaves(store, envs, out, stream);
}

int32_t vn_env_step_mode(const vn_store_t *store, const vn_envs_t *envs, const vn_step_out_t *out,
                         int32_t gather_variant) {
    VN_REQUIRE(envs && envs->n_envs >= 0, "envs: null or negative n_envs");
    int32_t rc = vn::validate_store(store);
    if (rc) return rc;
    int32_t smem = 0;
    const vn::StepMode mode = vn::choose_mode(store, envs, out, gather_variant, &smem);
    return mode == vn::kModeError ? VN_EINVAL : (int32_t)mode;
}

int32_t vn_env_host_seq_words(const vn_store_t *store, const vn_envs_t *envs, const vn_step_out_t *out,
                              int32_t gather_variant) {
    VN_REQUIRE(envs && envs->n_envs >= 0, "envs: null or negative n_envs");
    int32_t rc = vn::validate_store(store);
    if (rc) return rc;
    int32_t smem = 0;
    const vn::StepMode mode = vn::choose_mode(store, envs, out, gather_variant, &smem);
    if (mode == vn::kModeError) return VN_EINVAL;
    if (envs->n_envs == 0 || mode == vn::kModePersistent) return 1;
    return mode == vn::kModeFused ? envs->n_envs : (envs->n_envs + vn::kStepThreads - 1) / vn::kStepThreads;
}

int32_t vn_host_wait_seq(const uint32_t *host_seq, int32_t words, uint32_t seq, void *stream, int64_t timeout_us) {
    VN_REQUIRE(host_seq && words >= 1, "host_wait_seq: null or no words");
    const volatile uint32_t *flag = host_seq;
    const auto t0 = std::chrono::steady_clock::now();
    int64_t next_query_us = 50;
    int32_t have = 0;  // words [0, have) have been seen with the new value (they do not change back)
    for (uint64_t spin = 0;; ++spin) {
        while (have < words && flag[have] == seq) ++have;
        if (have == words) {
            std::atomic_thread_fence(std::memory_order_acquire);
            return VN_OK;
        }
#if defined(__x86_64__) || defined(__i386__)
        __builtin_ia32_pause();
#endif
        if ((spin & 255) != 255) continue;
        const int64_t us =
            std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t0).count();
        if (us >= next_query_us) {
            next_query_us = us + 50;
            const cudaError_t e = cudaStreamQuery(static_cast<cudaStream_t>(stream));
            if (e == cudaSuccess) {  // everything enqueued has run: the words must have been written by now
                while (have < words && flag[have] == seq) ++have;
                if (have == words) return VN_OK;
                vn::set_error("host_wait_seq: the stream drained but word %d is %u, not %u", have, flag[have], seq);
                return VN_ECUDA;
            }
            if (e != cudaErrorNotReady) {
                vn::set_error("host_wait_seq: %s", cudaGetErrorString(e));
                return VN_ECUDA;
            }
        }
        if (timeout_us > 0 && us > timeout_us) {
            vn::set_error("host_wait_seq: timed out after %lld us", (long long)us);
            return VN_ECUDA;
        }
    }
}

int32_t vn_env_step_host_sync(const vn_store_t *store, const vn_tables_t *tables, const vn_envs_t *envs,
                              const vn_rules_t *rules, const vn_inject_t *inject, const int32_t *host_actions,
                              int32_t *dev_actions_copy, const vn_step_out_t *out, uint8_t *pack_copy,
                              float *reward_copy, uint8_t *done_copy, int32_t seq_words, int32_t gather_variant,
                              void *stream, int64_t timeout_us) {
    VN_REQUIRE(out && out->host_pack && out->host_seq, "step_host_sync: out->host_pack and out->host_seq are required");
    VN_REQUIRE(envs && envs->n_envs >= 0, "envs: null or negative n_envs");
    int32_t rc = vn_env_step_host(store, tables, envs, rules, inject, host_actions, dev_actions_copy, out, nullptr,
                                  gather_variant, stream);
    if (rc || envs->n_envs == 0) return rc;
    rc = vn_host_wait_seq(out->host_seq, seq_words, out->seq, stream, timeout_us);
    if (rc) return rc;
    const size_t n = (size_t)envs->n_envs;
    if (pack_copy) memcpy(pack_copy, out->host_pack, 20 * n);
    if (reward_copy) memcpy(reward_copy, out->host_pack, 4 * n);
    if (done_copy) memcpy(done_copy, out->host_pack + 16 * n, n);
    return VN_OK;
}

int32_t vn_env_step_host_call(const vn_host_call_t *call, float *reward_copy, uint8_t *done_copy, void *stream) {
    VN_REQUIRE(call, "step_host_call: null descriptor");
    return vn_env_step_host_sync(call->store, call->tables, call->envs, call->rules, call->inject, call->host_actions,
                                 call->dev_actions_copy, call->out, nullptr, reward_copy, done_copy, call->seq_words,
                                 call->gather_variant, stream, call->timeout_us);
}

int32_t vn_debug_gather_trace(uint64_t *device_buffer) {
    vn::g_gather_trace = reinterpret_cast<unsigned long long *>(device_buffer);
    return VN_OK;
}

int32_t vn_event_create(void **event) {
    VN_REQUIRE(event, "event_create: null");
    cudaEvent_t ev;
    cudaError_t e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
    if (e != cudaSuccess) {
        vn::set_error("event_create: %s", cudaGetErrorString(e));
        return VN_ECUDA;
    }
    *event = ev;
    return VN_OK;
}

int32_t vn_event_destroy(void *event) {
    if (event) cudaEventDestroy(static_cast<cudaEvent_t>(event));
    return VN_OK;
}

int32_t vn_event_wait(void *event) {
    VN_REQUIRE(event, "event_wait: null");
    cudaError_t e = cudaEventSynchronize(static_cast<cudaEvent_t>(event));
    if (e != cudaSuccess) {
        vn::set_error("event_wait: %s", cudaGetErrorString(e));
        return VN_ECUDA;
    }
    return VN_OK;
}

int32_t vn_gather_plane(const vn_store_t *store, int32_t plane, const int32_t *idx, int32_t n, uint8_t *out,
                        int32_t gather_variant, void *stream) {
    int32_t rc = vn::validate_store(store);
    if (rc) return rc;
    VN_REQUIRE(plane >= 0 && plane < store->n_planes, "gather_plane: plane=%d", plane);
    VN_REQUIRE(idx && out && n >= 0, "gather_plane: null pointer");
    vn::GatherParams gp;
    gp.store = *store;
    gp.obs_state = idx;
    gp.goal = nullptr;
    gp.did_reset = nullptr;
    gp.desc = nullptr;
    gp.sched = nullptr;  // static unit assignment: no scratch in this signature
    gp.parity = 0;
    gp.early_release = 0;  // idx is caller memory a following step may rewrite: no early start of the successor
    gp.trace = nullptr;
    gp.n = n;
    for (int pl = 0; pl < VN_MAX_PLANES; ++pl) {
        gp.obs[pl] = (pl == plane) ? out : nullptr;
        gp.goal_obs[pl] = nullptr;
    }
    return vn::launch_gather(gp, gather_variant, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
