// Rollout / target builders (sm_100a): n-step returns, discounted back-up, pixel-control reward and
// auxiliary targets computed straight from the HBM frame store, reward-prediction labels + compaction,
// and the fused gather -> float32 CHW conversion for the policy input.
#include <climits>

#include "vn_common.cuh"

namespace vn {

// Programmatic dependent launch inside a builder CHAIN (several kernels enqueued by one C call): every kernel waits for
// its predecessor's memory before touching data; a kernel whose successor is the next kernel of the SAME chain lets it
// be scheduled early (its launch latency and prologue then overlap this kernel).  The LAST kernel of a call never
// releases early: what follows it in the stream is unknown (a step kernel that rewrites the rollout rows just read).
__device__ __forceinline__ void chain_wait(int release_successor) {
    asm volatile("griddepcontrol.wait;" ::: "memory");
    if (release_successor) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}

// =====================================================================================================
// n-step returns: one thread per env, serial backward recurrence over T (parallel across envs)
// =====================================================================================================
__global__ void __launch_bounds__(64) vn_nstep_returns_kernel(const float *__restrict__ reward,
                                                               const uint8_t *__restrict__ done,
                                                               const float *__restrict__ last_value, float gamma, int n,
                                                               int t, int64_t stride_n, int64_t stride_t,
                                                               float *__restrict__ out, int64_t ostride_n,
                                                               int64_t ostride_t) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t base = (int64_t)i * stride_n, obase = (int64_t)i * ostride_n;
    // R_T = (1 - done[T-1]) * V(s_T)
    float ret = (1.0f - (float)done[base + (int64_t)(t - 1) * stride_t]) * last_value[i];
    for (int k = t - 1; k >= 0; --k) {
        const int64_t at = base + (int64_t)k * stride_t;
        const float nd = 1.0f - (float)done[at];
        // r + (gamma * R) * nd, evaluated in this order without contraction (nd is 0 or 1, so the
        // product by nd is exact and an FMA could not change the result either)
        ret = __fadd_rn(reward[at], __fmul_rn(__fmul_rn(gamma, ret), nd));
        out[obase + (int64_t)k * ostride_t] = ret;
    }
}

// The same recurrence as a warp-level scan: one warp per env, 32 time steps per pass.  Step t is the affine map
// f_t(x) = b_t + a_t x with a_t = gamma (1 - done_t), b_t = r_t; R_t = (f_t o f_{t+1} o ... o f_{T-1})(R_T).  An
// inclusive SUFFIX scan of the maps under composition (5 shuffle rounds) gives every R_t of the chunk from the carry
// R_{chunk end + 1}.  Re-associates the float operations: equal to the serial kernel within ~1e-6 relative, not bit
// for bit - which is why the serial kernel stays the default (the north-star bound is 1e-5).
__global__ void __launch_bounds__(128) vn_nstep_returns_scan_kernel(const float *__restrict__ reward,
                                                                    const uint8_t *__restrict__ done,
                                                                    const float *__restrict__ last_value, float gamma,
                                                                    int n, int t, int64_t stride_n, int64_t stride_t,
                                                                    float *__restrict__ out, int64_t ostride_n,
                                                                    int64_t ostride_t) {
    const int lane = threadIdx.x & 31;
    const int warps = (gridDim.x * blockDim.x) >> 5;
    for (int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += warps) {
        const int64_t base = (int64_t)i * stride_n;
        float carry = (1.0f - (float)done[base + (int64_t)(t - 1) * stride_t]) * last_value[i];
        for (int hi = t; hi > 0; hi -= 32) {          // chunk [hi - 32, hi), lane L <-> step hi - 32 + L
            const int k = hi - 32 + lane;
            float a = 1.0f, b = 0.0f;                 // identity map for lanes before step 0
            if (k >= 0) {
                const int64_t at = base + (int64_t)k * stride_t;
                a = gamma * (1.0f - (float)done[at]);
                b = reward[at];
            }
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const float a2 = __shfl_down_sync(0xffffffffu, a, o), b2 = __shfl_down_sync(0xffffffffu, b, o);
                if (lane + o < 32) {                  // f <- f o g with g the composed map of the lanes after this one
                    b = fmaf(a, b2, b);
                    a = a * a2;
                }
            }
            const float r = fmaf(a, carry, b);
            if (k >= 0) out[(int64_t)i * ostride_n + (int64_t)k * ostride_t] = r;
            carry = __shfl_sync(0xffffffffu, r, hi >= 32 ? 0 : 32 - hi);   // R at the first real step of the chunk
        }
    }
}

// [n][t][d] with trailing feature axis: one thread per (env, feature), coalesced over d
__global__ void __launch_bounds__(256) vn_backup_kernel(const float *__restrict__ reward,
                                                        const uint8_t *__restrict__ done,
                                                        const float *__restrict__ bootstrap, float gamma, int n, int t,
                                                        int d, int64_t dstride_n, int64_t dstride_t,
                                                        float *__restrict__ out) {
    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= (int64_t)n * d) return;
    const int i = (int)(gid / d), f = (int)(gid - (int64_t)i * d);
    float ret = bootstrap[(int64_t)i * d + f];
    for (int k = t - 1; k >= 0; --k) {
        const int64_t at = ((int64_t)i * t + k) * d + f;
        const float nd = 1.0f - (float)done[(int64_t)i * dstride_n + (int64_t)k * dstride_t];
        ret = __fadd_rn(reward[at], __fmul_rn(__fmul_rn(gamma, ret), nd));
        out[at] = ret;
    }
}

// =====================================================================================================
// pixel-control reward and auxiliary targets from the store
// =====================================================================================================
// float(v) / 255.0f, correctly rounded, without a division or a table: q = v * r with r = fl(1 / 255), one Newton
// step on the exact residual e = fma(-q, 255, v), q' = fma(e, r, q).  Equal to __fdiv_rn(v, 255) for all 256 byte
// values (checked exhaustively on the host and, bit for bit, by the policy_input parity tests).
__device__ __forceinline__ float u8_over_255_f(float x) {
    const float r = 1.0f / 255.0f;
    const float q = __fmul_rn(x, r);
    const float e = __fmaf_rn(-q, 255.0f, x);
    return __fmaf_rn(e, r, q);
}

// Byte k of word w as a float without the (quarter-rate) integer-to-float conversion: one byte permute builds
// 0x4B0000vv = 2^23 + v, one exact subtraction removes the 2^23.
__device__ __forceinline__ float byte_as_float(uint32_t w, uint32_t k) {
    return __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7540u | k)) - 8388608.0f;
}

__device__ __forceinline__ float u8_over_255(uint32_t v) { return u8_over_255_f(byte_as_float(v, 0)); }

__device__ __forceinline__ void load_frame(uint8_t *dst_smem, const uint8_t *src, int nbytes) {
    const int4 *s = reinterpret_cast<const int4 *>(src);
    int4 *d = reinterpret_cast<int4 *>(dst_smem);
    // whole 16-byte units: a frame that is not a multiple of 16 bytes is padded in the store (and in dst_smem)
    for (int k = threadIdx.x; k < ((nbytes + 15) >> 4); k += blockDim.x) d[k] = ld_stream16(s + k);
}

struct PoolGeom {
    int h, w, c, cell, out_h, out_w, top, left;
};

// F.avg_pool2d's window sum for output cell (oi, oj) of channel ch: value(byte offset of the pixel in the HWC frame)
// summed in row-major order
template <typename Value>
__device__ __forceinline__ float window_sum(const PoolGeom &g, int oi, int oj, int ch, Value value) {
    const int row_bytes = g.w * g.c;
    float acc = 0.f;
    for (int dy = 0; dy < g.cell; ++dy) {
        const int rowoff = (g.top + oi * g.cell + dy) * row_bytes + (g.left + oj * g.cell) * g.c + ch;
        for (int dx = 0; dx < g.cell; ++dx) acc = __fadd_rn(acc, value(rowoff + dx * g.c));
    }
    return acc;
}

// out[cell] = mean_c avg_pool_cell(|nxt/255 - cur/255|) for one transition; frames in shared memory
__device__ __forceinline__ void pc_cells(const uint8_t *cur, const uint8_t *nxt, const PoolGeom &g,
                                         float *__restrict__ out_row) {
    const int cells = g.out_h * g.out_w;
    for (int cidx = threadIdx.x; cidx < cells; cidx += blockDim.x) {
        const int oi = cidx / g.out_w, oj = cidx - oi * g.out_w;
        float chan_sum = 0.f;
        for (int ch = 0; ch < g.c; ++ch) {
            const float acc = window_sum(g, oi, oj, ch, [&](int at) {
                return fabsf(__fsub_rn(u8_over_255(nxt[at]), u8_over_255(cur[at])));
            });
            chan_sum = __fadd_rn(chan_sum, __fdiv_rn(acc, (float)(g.cell * g.cell)));
        }
        out_row[cidx] = __fdiv_rn(chan_sum, (float)g.c);  // mean over channels
    }
}

// The two frames a pixel-control CTA stages in shared memory: frame 1 starts at the 16-byte boundary after frame 0
struct TwoFrames {
    uint8_t *f0, *f1;
    int bytes;
};
__device__ __forceinline__ TwoFrames two_frames(uint8_t *smem, const PoolGeom &g) {
    const int bytes = g.h * g.w * g.c;
    return {smem, smem + ((bytes + 15) & ~15), bytes};
}

// CTA per (env n, chunk of time steps).  Frames of consecutive steps are kept in a 2-slot shared ring so
// each frame is read from HBM/L2 once per chunk: (chunk + 1) / chunk reads per output.  8 CTAs per SM caps ptxas at
// 32 registers, which it reaches without spills; left free it takes 40 and runs slower (B200, 1,000 W: 131.8 vs
// 122.5 us for tools/bench_targets.py's pixel_control_direct).
template <int kChunk>
__global__ void __launch_bounds__(256, 8) vn_pixel_control_kernel(const uint8_t *__restrict__ pbase,
                                                                  int64_t pitch, const int32_t *__restrict__ states,
                                                                  int n, int t, int64_t sn, int64_t st, PoolGeom g,
                                                                  float *__restrict__ out) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    const TwoFrames fr = two_frames(smem_raw, g);
    const int chunks = (t + kChunk - 1) / kChunk;
    const int env = blockIdx.x / chunks;
    const int k0 = (blockIdx.x - env * chunks) * kChunk;
    const int k1 = min(t, k0 + kChunk);
    const int32_t *srow = states + (int64_t)env * sn;   // observation k of this env lives at srow[k * st]

    load_frame(fr.f0, pbase + (size_t)srow[(int64_t)k0 * st] * pitch, fr.bytes);
    uint8_t *cur = fr.f0, *nxt = fr.f1;
    const int cells = g.out_h * g.out_w;
    for (int k = k0; k < k1; ++k) {
        load_frame(nxt, pbase + (size_t)srow[(int64_t)(k + 1) * st] * pitch, fr.bytes);
        __syncthreads();
        pc_cells(cur, nxt, g, out + ((int64_t)env * t + k) * cells);
        __syncthreads();
        uint8_t *tmp = cur;
        cur = nxt;
        nxt = tmp;
    }
}

// Direct pixel-control reward for a device-resident LIST of transitions (the reset transitions that the
// per-scene transition table cannot serve).  Persistent CTAs loop over the list; its length is read from
// device memory, so no host synchronisation is needed between the lookup pass and this one.
__global__ void __launch_bounds__(512) vn_pixel_control_list_kernel(const uint8_t *__restrict__ pbase,
                                                                    int64_t pitch, const int32_t *__restrict__ states,
                                                                    int t, int64_t sn, int64_t st, PoolGeom g,
                                                                    const int32_t *__restrict__ pos,
                                                                    const int32_t *__restrict__ count, int max_count,
                                                                    int compact, float *__restrict__ out, int chained) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    chain_wait(chained);
    const TwoFrames fr = two_frames(smem_raw, g);
    const int m_total = min(*count, max_count);
    if ((int)blockIdx.x >= m_total) return;
    const int cells = g.out_h * g.out_w;
    for (int m = blockIdx.x; m < m_total; m += gridDim.x) {
        const int p = pos[m];
        const int env = p / t, k = p - env * t;
        const int32_t *srow = states + (int64_t)env * sn;
        __syncthreads();
        load_frame(fr.f0, pbase + (size_t)srow[(int64_t)k * st] * pitch, fr.bytes);
        load_frame(fr.f1, pbase + (size_t)srow[(int64_t)(k + 1) * st] * pitch, fr.bytes);
        __syncthreads();
        // compact: row m of a side buffer (consumed by vn_pixel_control_returns); else row p of the [n][t] output
        pc_cells(fr.f0, fr.f1, g, out + (int64_t)(compact ? m : p) * cells);
    }
}

// rows[n][k] = pixel-control table row of transition states[n][k] -> states[n][k+1]
constexpr int kRowZero = -1, kRowMiss = -2;   // a miss is stored as -(2 + m), m = its index in the miss list
// Thread q handles transition (env, k).  The thread order follows the faster axis of `states` so that a warp reads
// consecutive addresses: time-major storage (st > sn: rollout buffers) -> env fastest, batch-major -> k fastest.  The
// row index of (env, k) is written to rows[env * rsn + k * rst] (the caller picks the matching scratch layout).
__global__ void __launch_bounds__(256) vn_transition_rows_kernel(const int32_t *__restrict__ adj,
                                                                 const int32_t *__restrict__ states, int n, int t,
                                                                 int64_t sn, int64_t st, int64_t rsn, int64_t rst,
                                                                 int32_t *__restrict__ rows,
                                                                 int32_t *__restrict__ miss_pos,
                                                                 int32_t *__restrict__ miss_count, int chained) {
    chain_wait(chained);
    const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool miss = false;
    int64_t p = 0, at = 0;
    if (q < (int64_t)n * t) {
        int env, k;
        if (st > sn) {
            k = (int)(q / n);
            env = (int)(q - (int64_t)k * n);
        } else {
            env = (int)(q / t);
            k = (int)(q - (int64_t)env * t);
        }
        p = (int64_t)env * t + k;          // batch-major position: what the miss list and the outputs are indexed by
        at = (int64_t)env * rsn + (int64_t)k * rst;
        const int s = states[(int64_t)env * sn + (int64_t)k * st], s2 = states[(int64_t)env * sn + (int64_t)(k + 1) * st];
        int row = kRowMiss;
        if (s2 == s) {
            row = kRowZero;  // collision / no-op: identical frames, |x - x| = 0 exactly
        } else {
            const int4 nb = __ldg(reinterpret_cast<const int4 *>(adj) + s);
            if (nb.x == s2)
                row = s * 4;
            else if (nb.y == s2)
                row = s * 4 + 1;
            else if (nb.z == s2)
                row = s * 4 + 2;
            else if (nb.w == s2)
                row = s * 4 + 3;
        }
        if (row != kRowMiss) rows[at] = row;
        miss = row == kRowMiss;
    }
    // warp-aggregated append of the misses (ballot + one atomic per warp)
    const unsigned b = __ballot_sync(0xffffffffu, miss);
    if (b) {
        const int lane = threadIdx.x & 31;
        int base = 0;
        if (lane == __ffs(b) - 1) base = atomicAdd(miss_count, __popc(b));
        base = __shfl_sync(0xffffffffu, base, __ffs(b) - 1);
        if (miss) {
            const int m = base + __popc(b & ((1u << lane) - 1u));
            miss_pos[m] = (int32_t)p;
            rows[at] = kRowMiss - m;
        }
    }
}

// out[i] = table[idx[i]] (rows of row16 16-byte units); idx < 0 writes zeros (kRowZero) or leaves the row
// untouched (kRowMiss: the list kernel fills it).  One warp per row, grid-stride.
__global__ void __launch_bounds__(256) vn_gather_rows_kernel(const int4 *__restrict__ table, int row16,
                                                             const int32_t *__restrict__ idx, int64_t n,
                                                             int idx_t, int64_t sn, int64_t st,
                                                             int4 *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t i = warp0; i < n; i += nwarps) {
        // output row i = (a, k) of an [n / idx_t][idx_t] batch-major result reads idx[a * sn + k * st]
        const int64_t a = i / idx_t, k = i - a * idx_t;
        const int r = __ldg(idx + a * sn + k * st);
        if (r <= kRowMiss) continue;
        int4 *dst = out + i * row16;
        if (r < 0) {
            for (int k = lane; k < row16; k += 32) st_stream16(dst + k, make_int4(0, 0, 0, 0));
        } else {
            const int4 *src = table + (int64_t)r * row16;
            int k = lane;
            for (; k + 96 < row16; k += 128) {  // 4 independent 16-byte loads in flight per lane
                const int4 v0 = __ldg(src + k), v1 = __ldg(src + k + 32), v2 = __ldg(src + k + 64),
                           v3 = __ldg(src + k + 96);
                st_stream16(dst + k, v0);
                st_stream16(dst + k + 32, v1);
                st_stream16(dst + k + 64, v2);
                st_stream16(dst + k + 96, v3);
            }
            for (; k < row16; k += 32) st_stream16(dst + k, __ldg(src + k));
        }
    }
}

// CTA per gathered frame: out[m][c][out_h][out_w] = avg_pool(crop(frame / 255))
__global__ void __launch_bounds__(256) vn_aux_target_kernel(const uint8_t *__restrict__ pbase, int64_t pitch,
                                                            const int32_t *__restrict__ idx, int m, PoolGeom g,
                                                            float *__restrict__ out) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    const int fbytes = g.h * g.w * g.c;
    const uint8_t *frame = smem_raw;
    const int cells = g.out_h * g.out_w;
    for (int f = blockIdx.x; f < m; f += gridDim.x) {
        __syncthreads();
        load_frame(smem_raw, pbase + (size_t)idx[f] * pitch, fbytes);
        __syncthreads();
        for (int o = threadIdx.x; o < cells * g.c; o += blockDim.x) {
            const int ch = o / cells, cidx = o - ch * cells;
            const int oi = cidx / g.out_w, oj = cidx - oi * g.out_w;
            const float acc = window_sum(g, oi, oj, ch, [&](int at) { return u8_over_255(frame[at]); });
            out[(int64_t)f * cells * g.c + o] = __fdiv_rn(acc, (float)(g.cell * g.cell));
        }
    }
}

// gather + TransposeImage + ScaledFloatFrame: out[i][c][h][w] = float(frame[h][w][c]) / 255
__global__ void __launch_bounds__(256) vn_gather_f32_chw_kernel(const uint8_t *__restrict__ pbase,
                                                                int64_t pitch, const int32_t *__restrict__ idx,
                                                                int idx_stride, int n, int h, int w, int c,
                                                                float *__restrict__ out) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    const int fbytes = h * w * c;
    const int hw = h * w;
    for (int f = blockIdx.x; f < n; f += gridDim.x) {
        const int rec = idx[(int64_t)f * idx_stride];
        if (rec < 0) continue;  // uniform over the block: row f keeps its content
        __syncthreads();
        load_frame(smem_raw, pbase + (size_t)rec * pitch, fbytes);
        __syncthreads();
        float *o = out + (int64_t)f * fbytes;
        for (int k = threadIdx.x; k < fbytes; k += blockDim.x) {  // k indexes the CHW output: coalesced stores
            const int ch = k / hw, px = k - ch * hw;
            o[k] = __fdiv_rn((float)smem_raw[px * c + ch], 255.0f);
        }
    }
}

// One group of 4 pixels as float32 CHW / 255: w holds the group's 4 * C bytes (pixel-major, channel-minor, as in the
// HWC frame); one streaming 16-byte store per channel plane of the output, o pointing at the group in plane 0.
template <int C>
__device__ __forceinline__ void store_group(float *o, const uint32_t *w, int hw) {
#pragma unroll
    for (int ch = 0; ch < C; ++ch) {
        float v[4];
#pragma unroll
        for (int px = 0; px < 4; ++px) {
            const int b = px * C + ch;
            v[px] = u8_over_255_f(byte_as_float(w[b >> 2], b & 3));
        }
        asm volatile("st.global.cs.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(o + (int64_t)ch * hw), "f"(v[0]), "f"(v[1]),
                     "f"(v[2]), "f"(v[3])
                     : "memory");
    }
}

// Vectorised form of the same conversion for frames whose pixel count is a multiple of 4 (84 x 84, 174 x 174):
// one thread per GROUP of 4 pixels.  It reads the group's 4 * C bytes as C aligned 32-bit words straight from the
// store (no staging, no shared memory, no block barrier), scales every byte with u8_over_255 and writes one
// 16-byte vector per channel plane - a warp writes 512 contiguous bytes of each plane.  Grid-stride over
// (frame, group), 4 groups per thread in flight.
template <int C>
__global__ void __launch_bounds__(256) vn_gather_f32_chw_vec_kernel(const uint8_t *__restrict__ pbase, int64_t pitch,
                                                                    const int32_t *__restrict__ idx, int idx_stride,
                                                                    int n, int hw, float *__restrict__ out) {
    const int groups = hw >> 2;
    const int64_t total = (int64_t)n * groups;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    constexpr int kUnroll = 4;  // groups per thread and iteration: 4 * C independent loads in flight
    for (int64_t g0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g0 < total; g0 += kUnroll * stride) {
        uint32_t w[kUnroll][C];
        float *o[kUnroll];
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) {
            const int64_t g = g0 + u * stride;
            o[u] = nullptr;
            if (g < total) {
                const int f = (int)(g / groups), q = (int)(g - (int64_t)f * groups);
                const int rec = __ldg(idx + (int64_t)f * idx_stride);
                if (rec >= 0) {  // negative: row f keeps its content
                    const uint32_t *src = reinterpret_cast<const uint32_t *>(pbase + (size_t)rec * pitch) + (size_t)q * C;
#pragma unroll
                    for (int j = 0; j < C; ++j) w[u][j] = __ldg(src + j);
                    o[u] = out + ((int64_t)f * C) * hw + 4 * q;
                }
            }
        }
#pragma unroll
        for (int u = 0; u < kUnroll; ++u)
            if (o[u]) store_group<C>(o[u], w[u], hw);
    }
}

// All float leaves of one step in ONE launch: thread per (env, group of 4 pixels); for every leaf the record comes
// from the step's gather descriptor (x = observation record or -1, y = goal record or -1).  The loads of all
// leaves are issued before the first conversion, so one thread keeps up to 18 independent 4-byte loads in flight.
constexpr int kMaxFloatLeaves = 6;
struct FloatLeaves {
    const uint8_t *pbase[kMaxFloatLeaves];  // store base + plane offset
    float *out[kMaxFloatLeaves];
    int32_t c[kMaxFloatLeaves];             // 1 or 3
    int32_t goal[kMaxFloatLeaves];          // 0: descriptor x, 1: descriptor y
    int32_t n_leaves;
};

// kLeaves = number of leaves (sizes the register arrays), kUnroll = groups per thread and iteration: chosen on the
// host so that a thread has about a dozen independent loads in flight without running out of registers.
template <int kLeaves, int kUnroll>
__global__ void __launch_bounds__(256) vn_gather_leaves_f32_kernel(const FloatLeaves L, int64_t pitch,
                                                                   const int2 *__restrict__ desc, int n, int hw,
                                                                   int early_release) {
    // as part of a step (programmatic launch) the scalar half's descriptors are needed from here on, and the next
    // step's scalar kernel - which touches nothing this kernel reads - may be scheduled while this one runs
    chain_wait(early_release);
    const int groups = hw >> 2;
    const int64_t total = (int64_t)n * groups;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t g0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g0 < total; g0 += kUnroll * stride) {
        uint32_t w[kUnroll][kLeaves][3];
        bool live[kUnroll][kLeaves];
        int fq[kUnroll][2];
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) {
            const int64_t g = g0 + u * stride;
            const bool in = g < total;
            const int f = in ? (int)(g / groups) : 0, q = in ? (int)(g - (int64_t)f * groups) : 0;
            fq[u][0] = f;
            fq[u][1] = q;
            int2 d = make_int2(-1, -1);
            if (in) d = __ldg(desc + f);
#pragma unroll
            for (int l = 0; l < kLeaves; ++l) {
                const int rec = L.goal[l] ? d.y : d.x;
                live[u][l] = rec >= 0;
                if (rec >= 0) {
                    const uint32_t *src =
                        reinterpret_cast<const uint32_t *>(L.pbase[l] + (size_t)rec * pitch) + (size_t)q * L.c[l];
                    w[u][l][0] = __ldg(src);
                    if (L.c[l] == 3) {
                        w[u][l][1] = __ldg(src + 1);
                        w[u][l][2] = __ldg(src + 2);
                    }
                }
            }
        }
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) {
#pragma unroll
            for (int l = 0; l < kLeaves; ++l) {
                if (!live[u][l]) continue;
                float *o = L.out[l] + ((int64_t)fq[u][0] * L.c[l]) * hw + 4 * fq[u][1];
                if (L.c[l] == 3)
                    store_group<3>(o, w[u][l], hw);
                else
                    store_group<1>(o, w[u][l], hw);
            }
        }
    }
}

// Pixel-control returns in ONE pass over the table rows: thread per (env, group of 4 cells), backward over t,
//   pc(n, k) = table[rows[n][k]] | 0 (rows == -1: identical frames) | miss_rows[m] (rows == -(2 + m): reset transition,
//              computed directly by vn_pixel_control_list in compact mode) | NaN (m >= max_miss: no side-buffer row)
//   R_T = bootstrap;  R_k = pc(n, k) + gamma * (1 - done(n, k)) * R_{k+1}     (same operation order as vn_backup_kernel)
// The rewards are never written to memory unless out_reward is given: 1,600 B read + 1,600 B written per transition
// instead of twice that for gather + back-up.
// The float4 a miss past the side buffer reads (m >= max_miss: the list kernel computed no row for it).  Selecting its
// address keeps the miss branch one unconditional load: a select of the loaded value cost 1.8 % of the fused chain.
__device__ __align__(16) const uint32_t kQuietNaN4[4] = {0x7fc00000u, 0x7fc00000u, 0x7fc00000u, 0x7fc00000u};

__global__ void __launch_bounds__(256) vn_pc_returns_kernel(const float4 *__restrict__ table,
                                                            const int32_t *__restrict__ rows, int64_t rsn, int64_t rst,
                                                            const float4 *__restrict__ miss_rows, int max_miss,
                                                            const uint8_t *__restrict__ done, int64_t dsn, int64_t dst,
                                                            const float4 *__restrict__ bootstrap, float gamma, int n,
                                                            int t, int d4, float4 *__restrict__ out,
                                                            float4 *__restrict__ out_reward, int32_t *reset_counter) {
    chain_wait(0);
    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    // the miss counter of the chain (read by the list kernel, which has completed) is re-armed for the next call
    if (gid == 0 && reset_counter) *reset_counter = 0;
    if (gid >= (int64_t)n * d4) return;
    const int i = (int)(gid / d4), f = (int)(gid - (int64_t)i * d4);
    float4 ret = bootstrap[(int64_t)i * d4 + f];
    constexpr int kAhead = 4;   // loads of kAhead steps are issued before the dependent chain consumes them
    for (int hi = t; hi > 0; hi -= kAhead) {
        float4 v[kAhead];
        float nd[kAhead];
#pragma unroll
        for (int u = 0; u < kAhead; ++u) {
            const int k = hi - 1 - u;
            v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
            nd[u] = 0.f;
            if (k >= 0) {
                const int r = __ldg(rows + (int64_t)i * rsn + (int64_t)k * rst);
                if (r >= 0)
                    v[u] = __ldg(table + (int64_t)r * d4 + f);
                else if (r <= kRowMiss)
                    v[u] = __ldg(kRowMiss - r < max_miss ? miss_rows + (int64_t)(kRowMiss - r) * d4 + f
                                                         : reinterpret_cast<const float4 *>(kQuietNaN4));
                nd[u] = 1.0f - (float)done[(int64_t)i * dsn + (int64_t)k * dst];
            }
        }
#pragma unroll
        for (int u = 0; u < kAhead; ++u) {
            const int k = hi - 1 - u;
            if (k < 0) break;
            ret.x = __fadd_rn(v[u].x, __fmul_rn(__fmul_rn(gamma, ret.x), nd[u]));
            ret.y = __fadd_rn(v[u].y, __fmul_rn(__fmul_rn(gamma, ret.y), nd[u]));
            ret.z = __fadd_rn(v[u].z, __fmul_rn(__fmul_rn(gamma, ret.z), nd[u]));
            ret.w = __fadd_rn(v[u].w, __fmul_rn(__fmul_rn(gamma, ret.w), nd[u]));
            const int64_t at = ((int64_t)i * t + k) * d4 + f;
            __stcs(out + at, ret);
            if (out_reward) __stcs(out_reward + at, v[u]);
        }
    }
}

// =====================================================================================================
// reward-prediction labels + order-preserving compaction of zero / non-zero positions
// =====================================================================================================
constexpr int kRpBlock = 1024;

// Position i = (a, k) of the batch-major [n / t][t] result reads reward[a * sn + k * st] (t = 1, sn = 1: flat input).
__device__ __forceinline__ float rp_reward(const float *__restrict__ reward, int i, int t, int64_t sn, int64_t st) {
    const int a = i / t, k = i - a * t;
    return reward[(int64_t)a * sn + (int64_t)k * st];
}

__global__ void __launch_bounds__(kRpBlock) vn_rp_count_kernel(const float *__restrict__ reward, int n, int t,
                                                               int64_t sn, int64_t st, int8_t *__restrict__ labels,
                                                               int32_t *__restrict__ block_counts) {
    __shared__ int warp_nz[kRpBlock / 32];
    chain_wait(1);   // always followed by the scan or scatter kernel of the same call
    const int i = blockIdx.x * kRpBlock + threadIdx.x;
    const float r = i < n ? rp_reward(reward, i, t, sn, st) : 0.f;
    const bool nz = i < n && r != 0.f;
    if (i < n && labels) labels[i] = r > 0.f ? 1 : (r < 0.f ? 2 : 0);
    const unsigned b = __ballot_sync(0xffffffffu, nz);
    if ((threadIdx.x & 31) == 0) warp_nz[threadIdx.x >> 5] = __popc(b);
    __syncthreads();
    if (threadIdx.x == 0) {
        int s = 0;
        for (int k = 0; k < kRpBlock / 32; ++k) s += warp_nz[k];
        block_counts[blockIdx.x] = s;
    }
}

// exclusive scan of the per-block non-zero counts (single block; blocks <= 2^24 / 1024 = 16384)
__global__ void __launch_bounds__(1024) vn_rp_scan_kernel(int32_t *__restrict__ block_counts, int blocks, int n,
                                                          int32_t *__restrict__ counts) {
    __shared__ int warp_tot[32];
    __shared__ int carry;
    chain_wait(0);
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int base = 0; base < blocks; base += 1024) {
        const int k = base + threadIdx.x;
        const int v = k < blocks ? block_counts[k] : 0;
        int x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += y;
        }
        if (lane == 31) warp_tot[wid] = x;
        __syncthreads();
        if (wid == 0) {
            int wv = warp_tot[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int y = __shfl_up_sync(0xffffffffu, wv, o);
                if (lane >= o) wv += y;
            }
            warp_tot[lane] = wv;
        }
        __syncthreads();
        const int incl = x + (wid ? warp_tot[wid - 1] : 0);
        if (k < blocks) block_counts[k] = carry + incl - v;
        __syncthreads();
        if (threadIdx.x == 1023) carry += incl;
        __syncthreads();
    }
    if (threadIdx.x == 0 && counts) {
        counts[1] = carry;
        counts[0] = n - carry;
    }
}

// scanned != 0: block_offsets holds the exclusive scan of the per-block counts (vn_rp_scan_kernel ran).  scanned == 0
// (few blocks): it still holds the raw counts and every block sums the counts of the blocks before it itself - one
// launch less; the last block also writes the two totals.
__global__ void __launch_bounds__(kRpBlock) vn_rp_scatter_kernel(const float *__restrict__ reward, int n, int t,
                                                                 int64_t sn, int64_t st,
                                                                 const int32_t *__restrict__ block_offsets, int scanned,
                                                                 int32_t *__restrict__ counts,
                                                                 int32_t *__restrict__ zero_idx,
                                                                 int32_t *__restrict__ nonzero_idx) {
    __shared__ int warp_nz[kRpBlock / 32];
    __shared__ int s_offset;
    chain_wait(0);
    const int i = blockIdx.x * kRpBlock + threadIdx.x;
    const bool valid = i < n;
    const bool nz = valid && rp_reward(reward, i, t, sn, st) != 0.f;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const unsigned b = __ballot_sync(0xffffffffu, nz);
    if (lane == 0) warp_nz[wid] = __popc(b);
    if (wid == 0) {
        int off;
        if (scanned) {
            off = block_offsets[blockIdx.x];
        } else {
            off = 0;
            for (int k = lane; k < (int)blockIdx.x; k += 32) off += block_offsets[k];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) off += __shfl_xor_sync(0xffffffffu, off, o);
        }
        if (lane == 0) s_offset = off;
    }
    __syncthreads();
    if (!scanned && counts && blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) {
        const int total_nz = s_offset + block_offsets[blockIdx.x];
        counts[1] = total_nz;
        counts[0] = n - total_nz;
    }
    if (!zero_idx && !nonzero_idx) return;
    int before = 0;  // non-zeros in earlier warps of this block
    for (int k = 0; k < wid; ++k) before += warp_nz[k];
    const int nz_rank = s_offset + before + __popc(b & ((1u << lane) - 1u));
    if (!valid) return;
    if (nz) {
        if (nonzero_idx) nonzero_idx[nz_rank] = i;
    } else if (zero_idx) {
        zero_idx[i - nz_rank] = i;  // zeros before i = i - (non-zeros before i)
    }
}

// =====================================================================================================
// device-side UNREAL replay ring: uniform sampling of valid windows, one thread per env
// =====================================================================================================
struct ReplayParams {
    vn_replay_t ring;                                // [cap][n] time-major ring, as the caller described it
    int32_t length;                                  // transitions per sampled window
    int32_t mode;                                    // 0 sequence, 1 reward-prediction (length is 3 history steps)
    int32_t env_id_base;
    uint32_t call;                                   // sample counter (RNG counter word)
    uint64_t seed;
    int32_t *o_states, *o_goals, *o_actions;         // [n][length+1], [n][length+1], [n][length]
    float *o_rewards;                                // [n][length]
    uint8_t *o_dones;                                // [n][length]
    int32_t *o_start;                                // [n] chronological index of the window start, -1 if none
    int8_t *o_label;                                 // [n] RP class of the predicted reward (mode 1)
};

// A window of L transitions starting at chronological index i is valid when it lies inside the ring and no
// transition except possibly the last one ends an episode (sequences never straddle an episode boundary).
// In RP mode the window is 3 history transitions + the transition whose reward is classified, and the
// candidates are split by that reward being zero / non-zero (50/50 skewed sampling, SURVEY.md D6).
//
// One WARP per env: the ring column is scanned 32 slots at a time.  A window ending at transition i is valid iff
// i >= L - 1 and the last episode end strictly before i lies before the window (index < i - L + 1); "the last episode
// end before i" is a prefix maximum, taken inside a chunk from the ballot of the done bits (31 - clz of the bits below
// the lane) and across chunks from a carried index.  Pass 0 counts the valid windows per class with ballot + popc, pass
// 1 walks the chunks again until the running count passes the drawn rank and picks the bit with __fns - the k-th valid
// window in chronological order, exactly what the one-thread-per-env loop of round 1 selected, in O(cap / 32) steps
// instead of O(cap).
__global__ void __launch_bounds__(128) vn_replay_sample_kernel(const ReplayParams p) {
    const int lane = threadIdx.x & 31;
    const int e = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (e >= p.ring.n) return;   // whole warps leave together
    const int L = p.mode == 1 ? 4 : p.length;
    const int oldest = (p.ring.head - p.ring.count + p.ring.cap) % p.ring.cap;
    const Philox4 d = philox4x32_10((uint32_t)(p.env_id_base + e), p.call, 0x5EB1A7u, (uint32_t)p.mode,
                                    (uint32_t)p.seed, (uint32_t)(p.seed >> 32));
    int n_valid[2] = {0, 0};  // [0] all (mode 0) or zero-reward (mode 1); [1] non-zero reward (mode 1)
    int start = -1, cls = 0;
    for (int pass = 0; pass < 2; ++pass) {
        int want = -1;
        if (pass == 1) {
            if (p.mode == 1) {
                cls = (d.v[1] & 1u) ? 1 : 0;                   // fair coin between the two classes
                if (n_valid[cls] == 0) cls ^= 1;               // fall back to the non-empty class
                if (n_valid[cls] == 0) break;                  // nothing to sample ("could not sample")
            } else if (n_valid[0] == 0) {
                break;
            }
            want = (int)__umulhi(d.v[0], (uint32_t)n_valid[cls]);
        }
        int carry = -1;   // chronological index of the last episode end seen in earlier chunks
        int seen = 0;     // valid windows of class `cls` in earlier chunks (pass 1)
        for (int base = 0; base < p.ring.count; base += 32) {
            const int i = base + lane;
            const bool in = i < p.ring.count;
            const size_t at = (size_t)((oldest + (in ? i : 0)) % p.ring.cap) * p.ring.n + e;
            const bool dn = in && p.ring.done[at] != 0;
            const unsigned m = __ballot_sync(0xffffffffu, dn);
            const unsigned below = m & ((1u << lane) - 1u);
            const int last = below ? base + 31 - __clz((int)below) : carry;
            const bool valid = in && i >= L - 1 && last < i - L + 1;
            const int c = (p.mode == 1 && valid) ? (p.ring.reward[at] != 0.0f) : 0;
            if (pass == 0) {
                n_valid[0] += __popc(__ballot_sync(0xffffffffu, valid && c == 0));
                n_valid[1] += __popc(__ballot_sync(0xffffffffu, valid && c == 1));
            } else {
                const unsigned b = __ballot_sync(0xffffffffu, valid && c == cls);
                const int here = __popc(b);
                if (seen + here > want) {
                    start = base + (int)__fns(b, 0, want - seen + 1) - L + 1;
                    break;
                }
                seen += here;
            }
            if (m) carry = base + 31 - __clz((int)m);
        }
    }
    if (lane == 0) p.o_start[e] = start;
    if (start < 0) return;
    // lanes write the L transitions (and the closing observation) of the window
    for (int k = lane; k < L; k += 32) {
        const size_t at = (size_t)((oldest + start + k) % p.ring.cap) * p.ring.n + e;
        p.o_states[(size_t)e * (L + 1) + k] = p.ring.before[at];
        // goal of the episode the BEFORE observation belongs to (ring.goal is the goal after the step, i.e. the next
        // episode's goal when the step ended one and the env auto-reset)
        p.o_goals[(size_t)e * (L + 1) + k] = p.ring.goal_before[at];
        p.o_actions[(size_t)e * L + k] = p.ring.action[at];
        p.o_rewards[(size_t)e * L + k] = p.ring.reward[at];
        p.o_dones[(size_t)e * L + k] = p.ring.done[at];
        if (k == L - 1) {
            p.o_states[(size_t)e * (L + 1) + L] = p.ring.after[at];
            p.o_goals[(size_t)e * (L + 1) + L] = p.ring.goal[at];
            if (p.o_label) {
                const float r = p.ring.reward[at];
                p.o_label[e] = r > 0.f ? 1 : (r < 0.f ? 2 : 0);
            }
        }
    }
}


// =====================================================================================================
// host side
// =====================================================================================================
constexpr int kMaxSmem = 220 * 1024;   // dynamic shared memory one CTA can have

// A store plane as the frame kernels read it.
struct FrameArgs {
    const uint8_t *pbase;   // store base + plane offset
    int64_t pitch;          // bytes from one record to the next
    PoolGeom g;             // h, w, c; the pool fields as well when a pool applies
    int smem;               // bytes of the frames a CTA stages, each padded to 16 bytes
};

// Validates plane `plane` of the store against the frame geometry (h, w, c) and, when `pool` = {cell, out_h, out_w} is
// given, the centred pool; `frames` frames are staged in shared memory.  Their size is checked by frame_smem() when a
// call has work to launch.
static int32_t frame_args(const vn_store_t *store, int32_t plane, int h, int w, int c, const int *pool, int frames,
                          const char *who, FrameArgs *f) {
    VN_REQUIRE(store && store->base, "%s: store is null", who);
    VN_REQUIRE(plane >= 0 && plane < store->n_planes, "%s: plane=%d", who, plane);
    const int fb = (h * w * c + 15) & ~15;
    VN_REQUIRE(store->plane_bytes[plane] == fb, "%s: plane holds %d bytes, geometry says %d (rounded up to 16)", who,
               store->plane_bytes[plane], h * w * c);
    VN_REQUIRE((store->plane_bytes[plane] & 15) == 0 && (store->state_pitch & 15) == 0 &&
                   (store->plane_off[plane] & 15) == 0,
               "%s: store is not 16-byte aligned", who);
    f->pbase = store->base + store->plane_off[plane];
    f->pitch = store->state_pitch;
    f->smem = frames * fb;
    f->g = PoolGeom{h, w, c, 1, h, w, 0, 0};
    if (!pool) return VN_OK;
    const int cell = pool[0], out_h = pool[1], out_w = pool[2];
    VN_REQUIRE(h > 0 && w > 0 && c > 0 && cell > 0 && out_h > 0 && out_w > 0, "%s: bad pool geometry", who);
    VN_REQUIRE(out_h * cell <= h && out_w * cell <= w, "%s: pool output %dx%d * cell %d exceeds frame %dx%d", who, out_h,
               out_w, cell, h, w);
    // autocrop_observations: centred, top margin (H - H') // 2
    f->g = PoolGeom{h, w, c, cell, out_h, out_w, (h - out_h * cell) / 2, (w - out_w * cell) / 2};
    return VN_OK;
}

// The frames `kernel` stages must fit one CTA's shared memory; raises the kernel's limit to their size.
template <typename... KArgs>
static int32_t frame_smem(void (*kernel)(KArgs...), const FrameArgs &f, const char *who) {
    VN_REQUIRE(f.smem <= kMaxSmem, "%s: frame too large for shared memory", who);
    return ensure_smem(kernel, f.smem);
}

// chained: the first kernel of vn_pixel_control_returns_from_states (programmatic launch, releases the list kernel
// early); otherwise an ordinary launch.
static int32_t launch_transition_rows(const int32_t *adj, const int32_t *states, int n, int t, int64_t sn, int64_t st,
                                      int64_t rsn, int64_t rst, int32_t *rows, int32_t *miss_pos, int32_t *miss_count,
                                      cudaStream_t stream, bool chained) {
    const int64_t total = (int64_t)n * t;
    return launch(vn_transition_rows_kernel, "vn_transition_rows_kernel", dim3((unsigned)((total + 255) / 256)),
                  dim3(256), 0, stream, chained, adj, states, n, t, sn, st, rsn, rst, rows, miss_pos, miss_count,
                  chained ? 1 : 0);
}

// The list kernel loops over a device-resident list (episode resets: ~0.1 % of an A2C rollout's transitions, ~2 % at
// C5's short episodes).  512 threads: one per output cell (20 x 20) in a single round - the kernel sits on the critical
// path between the row lookup and the back-up.  chained: the second kernel of vn_pixel_control_returns_from_states.
static int32_t launch_pc_list(const FrameArgs &f, const int32_t *states, int t, int64_t sn, int64_t st,
                              const int32_t *pos, const int32_t *count, int max_count, int compact, float *out,
                              cudaStream_t stream, bool chained, const char *who) {
    int32_t rc = frame_smem(vn_pixel_control_list_kernel, f, who);
    if (rc) return rc;
    const int want = sm_count() * ctas_per_sm(f.smem, 4);
    const int grid = max_count < want ? max_count : want;
    return launch(vn_pixel_control_list_kernel, "vn_pixel_control_list_kernel", dim3(grid), dim3(512), (size_t)f.smem,
                  stream, true, f.pbase, f.pitch, states, t, sn, st, f.g, pos, count, max_count, compact, out,
                  chained ? 1 : 0);
}

// chained: the last kernel of vn_pixel_control_returns_from_states (programmatic launch), which re-arms the chain's
// miss counter reset_counter; otherwise an ordinary launch and reset_counter is null.
static int32_t launch_pc_returns(const float *pc_table, int cells, const int32_t *rows, int64_t rsn, int64_t rst,
                                 const float *miss_rows, int max_miss, const uint8_t *done, int64_t dsn, int64_t dst,
                                 const float *bootstrap, float gamma, int n, int t, float *out_returns,
                                 float *out_reward, int32_t *reset_counter, cudaStream_t stream, bool chained) {
    const int d4 = cells >> 2;
    const int64_t threads = (int64_t)n * d4;
    return launch(vn_pc_returns_kernel, "vn_pc_returns_kernel", dim3((unsigned)((threads + 255) / 256)), dim3(256), 0,
                  stream, chained, reinterpret_cast<const float4 *>(pc_table), rows, rsn, rst,
                  reinterpret_cast<const float4 *>(miss_rows), max_miss, done, dsn, dst,
                  reinterpret_cast<const float4 *>(bootstrap), gamma, n, t, d4, reinterpret_cast<float4 *>(out_returns),
                  reinterpret_cast<float4 *>(out_reward), reset_counter);
}

int32_t launch_float_leaves(const vn_store_t *store, const vn_float_leaf_t *leaves, int32_t n_leaves, const int32_t *desc,
                            int32_t n, int32_t h, int32_t w, void *stream, bool in_step) {
    VN_REQUIRE(store && store->base && leaves && desc && n >= 0, "gather_leaves_f32_chw: null pointer");
    VN_REQUIRE(n_leaves >= 1 && n_leaves <= kMaxFloatLeaves, "gather_leaves_f32_chw: n_leaves=%d (max %d)", n_leaves,
               kMaxFloatLeaves);
    if ((h * w) % 4 != 0) {
        set_error("gather_leaves_f32_chw: %d x %d pixels are not whole groups of 4 (use the per-leaf call)", h, w);
        return VN_EUNSUPPORTED;
    }
    FloatLeaves L = {};
    L.n_leaves = n_leaves;
    for (int l = 0; l < n_leaves; ++l) {
        FrameArgs f;
        int32_t rc = frame_args(store, leaves[l].plane, h, w, leaves[l].channels, nullptr, 0, "gather_leaves_f32_chw", &f);
        if (rc) return rc;
        if (leaves[l].channels != 1 && leaves[l].channels != 3) {
            set_error("gather_leaves_f32_chw: %d channels (use the per-leaf call)", leaves[l].channels);
            return VN_EUNSUPPORTED;
        }
        VN_REQUIRE(leaves[l].out && aligned16(leaves[l].out), "gather_leaves_f32_chw: out[%d] must be 16-byte aligned",
                   l);
        VN_REQUIRE(leaves[l].source == 0 || leaves[l].source == 1, "gather_leaves_f32_chw: source=%d", leaves[l].source);
        L.pbase[l] = f.pbase;
        L.out[l] = leaves[l].out;
        L.c[l] = leaves[l].channels;
        L.goal[l] = leaves[l].source;
    }
    if (n == 0) return VN_OK;
    const int64_t total = (int64_t)n * (h * w / 4);
    const int unroll = n_leaves == 1 ? 4 : (n_leaves <= 3 ? 2 : 1);
    const int64_t want = (total + unroll * 256 - 1) / (unroll * 256), cap = (int64_t)sm_count() * 16;
    const int grid = (int)(want < cap ? want : cap);
    void (*const kernels[])(FloatLeaves, int64_t, const int2 *, int, int, int) = {
        vn_gather_leaves_f32_kernel<1, 4>, vn_gather_leaves_f32_kernel<2, 2>, vn_gather_leaves_f32_kernel<3, 2>,
        vn_gather_leaves_f32_kernel<4, 1>, vn_gather_leaves_f32_kernel<5, 1>, vn_gather_leaves_f32_kernel<6, 1>};
    // programmatic launch only as part of a step: there the predecessor is the step's own scalar / gather kernel
    return launch(kernels[n_leaves - 1], "vn_gather_leaves_f32_kernel", dim3(grid), dim3(256), 0,
                  static_cast<cudaStream_t>(stream), in_step, L, store->state_pitch, reinterpret_cast<const int2 *>(desc),
                  n, h * w, in_step ? 1 : 0);
}

}  // namespace vn

extern "C" {

int32_t vn_nstep_returns(const float *reward, const uint8_t *done, const float *last_value, float gamma, int32_t n,
                         int32_t t, int64_t stride_n, int64_t stride_t, float *out, int64_t out_stride_n,
                         int64_t out_stride_t, void *stream) {
    VN_REQUIRE(reward && done && last_value && out, "nstep_returns: null pointer");
    VN_REQUIRE(n >= 0 && t >= 1, "nstep_returns: n=%d t=%d", n, t);
    if (n == 0) return VN_OK;
    // 64-thread blocks: 4,096 envs spread over 64 SMs instead of 16 (the loop over T is a chain of dependent FMAs)
    return vn::launch(vn::vn_nstep_returns_kernel, "vn_nstep_returns_kernel", dim3((n + 63) / 64), dim3(64), 0,
                      static_cast<cudaStream_t>(stream), false, reward, done, last_value, gamma, n, t, stride_n,
                      stride_t, out, out_stride_n, out_stride_t);
}

int32_t vn_nstep_returns_scan(const float *reward, const uint8_t *done, const float *last_value, float gamma,
                              int32_t n, int32_t t, int64_t stride_n, int64_t stride_t, float *out,
                              int64_t out_stride_n, int64_t out_stride_t, void *stream) {
    VN_REQUIRE(reward && done && last_value && out, "nstep_returns_scan: null pointer");
    VN_REQUIRE(n >= 0 && t >= 1, "nstep_returns_scan: n=%d t=%d", n, t);
    if (n == 0) return VN_OK;
    const int64_t want = ((int64_t)n * 32 + 127) / 128, cap = (int64_t)vn::sm_count() * 16;
    return vn::launch(vn::vn_nstep_returns_scan_kernel, "vn_nstep_returns_scan_kernel",
                      dim3((unsigned)(want < cap ? want : cap)), dim3(128), 0, static_cast<cudaStream_t>(stream), false,
                      reward, done, last_value, gamma, n, t, stride_n, stride_t, out, out_stride_n, out_stride_t);
}

int32_t vn_discounted_backup(const float *reward, const uint8_t *done, int64_t done_stride_n, int64_t done_stride_t,
                             const float *bootstrap, float gamma, int32_t n, int32_t t, int32_t d, float *out,
                             void *stream) {
    VN_REQUIRE(reward && done && bootstrap && out, "discounted_backup: null pointer");
    VN_REQUIRE(n >= 0 && t >= 1 && d >= 1, "discounted_backup: n=%d t=%d d=%d", n, t, d);
    if (n == 0) return VN_OK;
    const int64_t total = (int64_t)n * d;
    return vn::launch(vn::vn_backup_kernel, "vn_backup_kernel", dim3((unsigned)((total + 255) / 256)), dim3(256), 0,
                      static_cast<cudaStream_t>(stream), false, reward, done, bootstrap, gamma, n, t, d, done_stride_n,
                      done_stride_t, out);
}

int32_t vn_pixel_control_returns(const float *pc_table, int32_t cells, const int32_t *rows, int64_t row_stride_n,
                                 int64_t row_stride_t, const float *miss_rows, const uint8_t *done,
                                 int64_t done_stride_n, int64_t done_stride_t,
                                 const float *bootstrap, float gamma, int32_t n, int32_t t, float *out_returns,
                                 float *out_reward, void *stream) {
    VN_REQUIRE(pc_table && rows && miss_rows && done && bootstrap && out_returns, "pixel_control_returns: null pointer");
    VN_REQUIRE(n >= 0 && t >= 1 && cells >= 4 && (cells & 3) == 0, "pixel_control_returns: n=%d t=%d cells=%d", n, t,
               cells);
    VN_REQUIRE(vn::aligned16(pc_table, miss_rows, bootstrap, out_returns, out_reward),
               "pixel_control_returns: arrays must be 16-byte aligned");
    if (n == 0) return VN_OK;
    // the caller built rows and miss_rows: every miss index it wrote has its row
    return vn::launch_pc_returns(pc_table, cells, rows, row_stride_n, row_stride_t, miss_rows, INT_MAX, done,
                                 done_stride_n, done_stride_t, bootstrap, gamma, n, t, out_returns, out_reward, nullptr,
                                 static_cast<cudaStream_t>(stream), false);
}

int32_t vn_pixel_control_returns_from_states(const vn_store_t *store, int32_t plane, const int32_t *adj,
                                             const float *pc_table, const int32_t *states, int64_t state_stride_n,
                                             int64_t state_stride_t, const uint8_t *done, int64_t done_stride_n,
                                             int64_t done_stride_t, const float *bootstrap, float gamma, int32_t n,
                                             int32_t t, int32_t h, int32_t w, int32_t c, int32_t cell, int32_t out_h,
                                             int32_t out_w, int32_t *rows, int32_t *miss_pos, int32_t *miss_count,
                                             float *miss_rows, int32_t max_miss, float *out_returns, float *out_reward,
                                             void *stream) {
    const char *who = "pixel_control_returns";
    const int pool[] = {cell, out_h, out_w};
    vn::FrameArgs f;
    int32_t rc = vn::frame_args(store, plane, h, w, c, pool, 2, who, &f);
    if (rc) return rc;
    const int32_t cells = out_h * out_w;
    VN_REQUIRE(adj && pc_table && states && done && bootstrap && rows && miss_pos && miss_count && miss_rows && out_returns,
               "pixel_control_returns: null pointer");
    VN_REQUIRE(n >= 0 && t >= 1 && cells >= 4 && (cells & 3) == 0 && max_miss >= 1,
               "pixel_control_returns: n=%d t=%d cells=%d max_miss=%d", n, t, cells, max_miss);
    VN_REQUIRE(vn::aligned16(adj), "pixel_control_returns: adj must be 16-byte aligned");
    VN_REQUIRE(vn::aligned16(pc_table, miss_rows, bootstrap, out_returns, out_reward),
               "pixel_control_returns: arrays must be 16-byte aligned");
    if (n == 0) return VN_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    // (1) table row of every transition; the misses (episode resets) go to a list.  *miss_count must be 0 on entry:
    //     zero it once when the scratch is allocated - kernel (3) re-arms it for the next call
    // `rows` is written batch-major whatever the layout of `states` (the lookup kernel orders its threads for coalesced
    // state READS; its 4-byte row writes are then scattered for time-major input, which costs nothing next to what a
    // time-major `rows` costs the back-up kernel: there every step's row index is a dependent load in front of the table
    // load, and batch-major keeps an env's T indices in one or two cache lines - 42 vs 58 us at 4,096 x 20)
    const int64_t rsn = t, rst = 1;
    rc = vn::launch_transition_rows(adj, states, n, t, state_stride_n, state_stride_t, rsn, rst, rows, miss_pos,
                                    miss_count, st, true);
    if (rc) return rc;
    // (2) the misses computed directly from their two frames into the compact side buffer
    rc = vn::launch_pc_list(f, states, t, state_stride_n, state_stride_t, miss_pos, miss_count, max_miss, 1, miss_rows, st,
                            true, who);
    if (rc) return rc;
    // (3) rewards gathered on the fly + discounted back-up; a miss past the side buffer (m >= max_miss: kernel (2)
    //     computed no row for it) contributes NaN instead of a read past miss_rows
    return vn::launch_pc_returns(pc_table, cells, rows, rsn, rst, miss_rows, max_miss, done, done_stride_n, done_stride_t,
                                 bootstrap, gamma, n, t, out_returns, out_reward, miss_count, st, true);
}

int32_t vn_pixel_control(const vn_store_t *store, int32_t plane, const int32_t *states, int32_t n, int32_t t,
                         int64_t state_stride_n, int64_t state_stride_t, int32_t h, int32_t w, int32_t c, int32_t cell,
                         int32_t out_h, int32_t out_w, float *out, void *stream) {
    const int pool[] = {cell, out_h, out_w};
    vn::FrameArgs f;
    int32_t rc = vn::frame_args(store, plane, h, w, c, pool, 2, "pixel_control", &f);
    if (rc) return rc;
    VN_REQUIRE(states && out && n >= 0 && t >= 1, "pixel_control: bad arguments");
    if (n == 0) return VN_OK;
    constexpr int kChunk = 16;
    rc = vn::frame_smem(vn::vn_pixel_control_kernel<kChunk>, f, "pixel_control");
    if (rc) return rc;
    const int64_t blocks = (int64_t)n * ((t + kChunk - 1) / kChunk);
    VN_REQUIRE(blocks < (1ll << 31), "pixel_control: too many blocks");
    return vn::launch(vn::vn_pixel_control_kernel<kChunk>, "vn_pixel_control_kernel", dim3((unsigned)blocks), dim3(256),
                      (size_t)f.smem, static_cast<cudaStream_t>(stream), false, f.pbase, f.pitch, states, n, t,
                      state_stride_n, state_stride_t, f.g, out);
}

int32_t vn_transition_rows(const int32_t *adj, const int32_t *states, int32_t n, int32_t t, int64_t state_stride_n,
                           int64_t state_stride_t, int32_t *rows, int64_t row_stride_n, int64_t row_stride_t,
                           int32_t *miss_pos, int32_t *miss_count, void *stream) {
    VN_REQUIRE(adj && states && rows && miss_pos && miss_count, "transition_rows: null pointer");
    VN_REQUIRE(n >= 0 && t >= 1, "transition_rows: n=%d t=%d", n, t);
    VN_REQUIRE(vn::aligned16(adj), "transition_rows: adj must be 16-byte aligned");
    if (n == 0) return VN_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const cudaError_t e = cudaMemsetAsync(miss_count, 0, sizeof(int32_t), st);
    if (e != cudaSuccess) {
        cudaGetLastError();
        vn::set_error("transition_rows: zeroing miss_count: %s", cudaGetErrorString(e));
        return VN_ECUDA;
    }
    return vn::launch_transition_rows(adj, states, n, t, state_stride_n, state_stride_t, row_stride_n, row_stride_t, rows,
                                      miss_pos, miss_count, st, false);
}

int32_t vn_gather_rows(const void *table, int64_t row_bytes, const int32_t *idx, int64_t n, int32_t idx_t,
                       int64_t idx_stride_n, int64_t idx_stride_t, void *out, void *stream) {
    VN_REQUIRE(table && idx && out, "gather_rows: null pointer");
    VN_REQUIRE(idx_t >= 1 && n % idx_t == 0, "gather_rows: n=%lld is not a multiple of idx_t=%d", (long long)n, idx_t);
    VN_REQUIRE(row_bytes > 0 && (row_bytes & 15) == 0, "gather_rows: row_bytes=%lld must be a multiple of 16",
               (long long)row_bytes);
    VN_REQUIRE(vn::aligned16(table, out), "gather_rows: table and out must be 16-byte aligned");
    if (n <= 0) return VN_OK;
    const int64_t cap = (int64_t)vn::sm_count() * 64, warps = n < cap ? n : cap;
    return vn::launch(vn::vn_gather_rows_kernel, "vn_gather_rows_kernel", dim3((unsigned)((warps * 32 + 255) / 256)),
                      dim3(256), 0, static_cast<cudaStream_t>(stream), false, static_cast<const int4 *>(table),
                      (int)(row_bytes >> 4), idx, n, idx_t, idx_stride_n, idx_stride_t, static_cast<int4 *>(out));
}

int32_t vn_pixel_control_list(const vn_store_t *store, int32_t plane, const int32_t *states, int32_t n, int32_t t,
                              int64_t state_stride_n, int64_t state_stride_t, int32_t h, int32_t w, int32_t c,
                              int32_t cell, int32_t out_h, int32_t out_w, const int32_t *pos, const int32_t *count,
                              int32_t max_count, int32_t compact, float *out, void *stream) {
    const int pool[] = {cell, out_h, out_w};
    vn::FrameArgs f;
    int32_t rc = vn::frame_args(store, plane, h, w, c, pool, 2, "pixel_control_list", &f);
    if (rc) return rc;
    VN_REQUIRE(states && pos && count && out && n >= 0 && t >= 1 && max_count >= 0, "pixel_control_list: bad arguments");
    if (n == 0 || max_count == 0) return VN_OK;
    return vn::launch_pc_list(f, states, t, state_stride_n, state_stride_t, pos, count, max_count, compact, out,
                              static_cast<cudaStream_t>(stream), false, "pixel_control_list");
}

int32_t vn_replay_sample(const vn_replay_t *ring, int32_t length, int32_t mode, uint64_t seed, uint32_t call,
                         int32_t env_id_base, int32_t *o_states, int32_t *o_goals, int32_t *o_actions,
                         float *o_rewards, uint8_t *o_dones, int32_t *o_start, int8_t *o_label, void *stream) {
    VN_REQUIRE(ring && ring->before && ring->after && ring->goal && ring->goal_before && ring->action && ring->reward &&
                   ring->done,
               "replay_sample: null ring pointer");
    VN_REQUIRE(ring->n >= 0 && ring->cap > 0 && ring->count >= 0 && ring->count <= ring->cap && ring->head >= 0 &&
                   ring->head < ring->cap,
               "replay_sample: bad ring geometry");
    VN_REQUIRE(mode == 0 || mode == 1, "replay_sample: mode=%d", mode);
    VN_REQUIRE(mode == 1 || length >= 1, "replay_sample: length=%d", length);
    VN_REQUIRE(o_states && o_goals && o_actions && o_rewards && o_dones && o_start, "replay_sample: null output");
    if (ring->n == 0) return VN_OK;
    const vn::ReplayParams p = {*ring,    length,    mode,      env_id_base, call,    seed,   o_states,
                                o_goals, o_actions, o_rewards, o_dones,     o_start, o_label};
    return vn::launch(vn::vn_replay_sample_kernel, "vn_replay_sample_kernel", dim3((ring->n + 3) / 4), dim3(128), 0,
                      static_cast<cudaStream_t>(stream), false, p);   // warp per env
}

int32_t vn_aux_target(const vn_store_t *store, int32_t plane, const int32_t *idx, int32_t m, int32_t h, int32_t w,
                      int32_t c, int32_t cell, int32_t out_h, int32_t out_w, float *out, void *stream) {
    const int pool[] = {cell, out_h, out_w};
    vn::FrameArgs f;
    int32_t rc = vn::frame_args(store, plane, h, w, c, pool, 1, "aux_target", &f);
    if (rc) return rc;
    VN_REQUIRE(idx && out && m >= 0, "aux_target: bad arguments");
    if (m == 0) return VN_OK;
    rc = vn::frame_smem(vn::vn_aux_target_kernel, f, "aux_target");
    if (rc) return rc;
    const int grid = m < vn::sm_count() * 8 ? m : vn::sm_count() * 8;
    return vn::launch(vn::vn_aux_target_kernel, "vn_aux_target_kernel", dim3(grid), dim3(256), (size_t)f.smem,
                      static_cast<cudaStream_t>(stream), false, f.pbase, f.pitch, idx, m, f.g, out);
}

int32_t vn_gather_plane_f32_chw(const vn_store_t *store, int32_t plane, const int32_t *idx, int32_t n, int32_t h,
                                int32_t w, int32_t c, float *out, void *stream) {
    return vn_gather_plane_f32_chw_rows(store, plane, idx, 1, n, h, w, c, out, stream);
}

int32_t vn_gather_plane_f32_chw_rows(const vn_store_t *store, int32_t plane, const int32_t *idx, int32_t idx_stride,
                                     int32_t n, int32_t h, int32_t w, int32_t c, float *out, void *stream) {
    vn::FrameArgs f;
    int32_t rc = vn::frame_args(store, plane, h, w, c, nullptr, 1, "gather_plane_f32_chw", &f);
    if (rc) return rc;
    VN_REQUIRE(idx && out && n >= 0 && idx_stride >= 1, "gather_plane_f32_chw: bad arguments");
    if (n == 0) return VN_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if ((h * w) % 4 == 0 && (c == 1 || c == 3) && vn::aligned16(out)) {
        // whole 4-pixel groups: the vectorised kernel (0.36 -> see DESIGN.md of the copy peak for the staged one)
        const int64_t total = (int64_t)n * (h * w / 4);
        const int64_t want = (total + 4 * 256 - 1) / (4 * 256), cap = (int64_t)vn::sm_count() * 16;
        return vn::launch(c == 1 ? vn::vn_gather_f32_chw_vec_kernel<1> : vn::vn_gather_f32_chw_vec_kernel<3>,
                          "vn_gather_f32_chw_vec_kernel", dim3((unsigned)(want < cap ? want : cap)), dim3(256), 0, st,
                          false, f.pbase, f.pitch, idx, idx_stride, n, h * w, out);
    }
    rc = vn::frame_smem(vn::vn_gather_f32_chw_kernel, f, "gather_plane_f32_chw");
    if (rc) return rc;
    const int grid = n < vn::sm_count() * 8 ? n : vn::sm_count() * 8;
    return vn::launch(vn::vn_gather_f32_chw_kernel, "vn_gather_f32_chw_kernel", dim3(grid), dim3(256), (size_t)f.smem, st,
                      false, f.pbase, f.pitch, idx, idx_stride, n, h, w, c, out);
}

int32_t vn_gather_leaves_f32_chw(const vn_store_t *store, const vn_float_leaf_t *leaves, int32_t n_leaves,
                                 const int32_t *desc, int32_t n, int32_t h, int32_t w, void *stream) {
    return vn::launch_float_leaves(store, leaves, n_leaves, desc, n, h, w, stream, false);
}

int32_t vn_rp_labels(const float *reward, int32_t n, int32_t t, int64_t stride_n, int64_t stride_t, int8_t *labels,
                     int32_t *zero_idx, int32_t *nonzero_idx, int32_t *counts, int32_t *scratch, void *stream) {
    VN_REQUIRE(reward && scratch, "rp_labels: reward and scratch are required");
    VN_REQUIRE(n >= 0 && n <= (1 << 24), "rp_labels: n=%d (max 2^24 per call)", n);
    VN_REQUIRE(t >= 1 && n % t == 0, "rp_labels: n=%d is not a multiple of t=%d", n, t);
    if (n == 0) return VN_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int blocks = (n + vn::kRpBlock - 1) / vn::kRpBlock;
    int32_t rc = vn::launch(vn::vn_rp_count_kernel, "vn_rp_count_kernel", dim3(blocks), dim3(vn::kRpBlock), 0, st, true,
                            reward, n, t, stride_n, stride_t, labels, scratch);
    if (rc) return rc;
    // few blocks (an A2C rollout: 80 blocks at 4,096 envs x 20 steps): no separate scan launch, the scatter kernel
    // sums the block counts itself and writes the totals
    const bool scan = blocks > 256;
    if (scan) {
        rc = vn::launch(vn::vn_rp_scan_kernel, "vn_rp_scan_kernel", dim3(1), dim3(1024), 0, st, true, scratch, blocks, n,
                        counts);
        if (rc || !(zero_idx || nonzero_idx)) return rc;
    }
    return vn::launch(vn::vn_rp_scatter_kernel, "vn_rp_scatter_kernel", dim3(blocks), dim3(vn::kRpBlock), 0, st, true,
                      reward, n, t, stride_n, stride_t, scratch, scan ? 1 : 0, scan ? nullptr : counts, zero_idx,
                      nonzero_idx);
}

}  // extern "C"
