// libvn_b200 - the policy's first convolution read straight from uint8 frames (sm_100a).
//
// Replaces TransposeImage + ScaledFloatFrame (deep_rl.common.env, thor_cached_auxiliary.py:61-62) + the model's first
// Conv2d (models/goal.py:36-41): y = conv2d(x / 255, weight, bias, stride) with x the uint8 HWC frame of an observation
// batch row or of a store record, and the weight / bias gradient of that layer.  No float copy of a frame is written.
//
// Numerics.  A pixel is an integer 0..255, exact in bf16.  The fp32 operand (the weight in the forward, grad_out in the
// weight gradient) is split into three bf16 terms hi + mid + lo (24 significant bits in all), so every product on the
// tensor cores is exact.  Per 16-deep k-step the three terms are chained through one mma.sync accumulator started at
// zero, and that k-step's sum is added to an fp32 register accumulator with a round-to-nearest FADD; the 1/255 scale is
// one division at the end.  The weight gradient's partial sums per fixed chunk of frames are reduced in a fixed order
// by a second kernel: no float atomics, the same bits on any number of SMs.
//
// The 16-bit variants (the *_lp entry points, torch.autocast) have fp16 or bf16 as the element type T.  The weight is
// rounded to T once (round-to-nearest-even, as autocast's cast), grad_out arrives in T, and a pixel is exact in either
// type, so every product is exact with ONE term: one mma.sync per k-step instead of three.  Accumulation, the 1/255
// scale and the reduction are those of the fp32 kernels; the forward rounds its fp32 result to T once.
//
// Plane sets (the vn_conv_u8_planes_* entry points, S = kMaxSrcs) read the frames of up to four sources (RGB-D,
// observation + goal) as one input of C = sum c_s channels in source order.  Each source's frame has its own region of
// the frame buffer, filled by its own bulk copy on the buffer's one mbarrier; a tap of the table is packed as
// (region byte offset of its channel at pixel (ky, kx)) << 2 | c_s, so the byte of output pixel p is at
// off + pixel(p) * c_s.  K = C * k * k grows to 512, so the forward splits the output channels into groups of NT * 8
// whose weight fragments fit in shared memory (a CTA keeps one group for its whole life and reads every frame it owns
// once per group), and the weight gradient splits the (cout, tap) tiles into groups of at most kWgradWarps * kWgradTiles
// (a CTA keeps one group and sums its chunks' frames for that group).  Both kernels keep the k-step and frame order of
// the single-frame kernels, so every output element is computed with the same operations in the same order.  The S = 1
// instantiations behind vn_conv_u8_forward / vn_conv_u8_backward compile none of this.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <type_traits>

#include "vn_common.cuh"

namespace vn {

constexpr int kMaxSmemConv = 220 * 1024;  // dynamic shared memory one CTA can have
constexpr int kMaxFrameSide = 174;        // the reference's native frame (INTEGRATION.md section 1)
constexpr int kFwdWarps = 4;
constexpr int kWgradWarps = 8;
constexpr int kWgradTiles = 13;    // (cout, tap) tiles of 16 x 8 per warp: 4 x 25 at most over 8 warps
constexpr int kWgradChunk = 32;    // frames per partial gradient
constexpr int kReduceLanes = 32;   // chunks summed in parallel per output of the reduce kernel
constexpr int kMaxSrcs = 4;        // frame sources of a plane set
constexpr int kMaxSetChannels = 8; // channels of a plane set

// ---------------------------------------------------------------- device helpers
__device__ __forceinline__ const uint8_t *frame_src(const vn_u8_frames_t &f, int i) {
    int64_t rec = i;
    if (f.idx) {
        const int a = i / f.idx_t, k = i - a * f.idx_t;
        rec = f.idx[a * f.idx_stride_n + k * f.idx_stride_t];
    }
    return f.base + rec * f.pitch;
}
// byte -> float, exact, without the integer-conversion pipe
__device__ __forceinline__ float u8f(uint32_t v) { return __int_as_float(0x4B000000u | v) - 8388608.f; }
// two floats of at most 8 significant bits as bf16x2 (exact truncation), lo in the low half
__device__ __forceinline__ uint32_t pack_exact(float lo, float hi) {
    return __byte_perm(__float_as_uint(lo), __float_as_uint(hi), 0x7632);
}
__device__ __forceinline__ uint32_t bf2_bits(__nv_bfloat162 v) { return *reinterpret_cast<uint32_t *>(&v); }
// (a, b) = hi + mid + lo, each a bf16x2 with a in the low half; every residual is exact in fp32
__device__ __forceinline__ void split3(float a, float b, uint32_t &hi, uint32_t &mid, uint32_t &lo) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    const float2 hf = __bfloat1622float2(h);
    const float ra = __fsub_rn(a, hf.x), rb = __fsub_rn(b, hf.y);
    const __nv_bfloat162 m = __floats2bfloat162_rn(ra, rb);
    const float2 mf = __bfloat1622float2(m);
    hi = bf2_bits(h);
    mid = bf2_bits(m);
    lo = bf2_bits(__floats2bfloat162_rn(__fsub_rn(ra, mf.x), __fsub_rn(rb, mf.y)));
}
// Element type T of a kernel: float = the fp32 operand split into three bf16 terms, __half / __nv_bfloat16 = one term.
template <typename T>
constexpr int kTerms = std::is_same_v<T, float> ? 3 : 1;
// two floats rounded to T x2 (round-to-nearest-even), lo in the low half
template <typename T>
__device__ __forceinline__ uint32_t pack_rn(float lo, float hi) {
    if constexpr (std::is_same_v<T, __half>) {
        const __half2 v = __floats2half2_rn(lo, hi);
        return *reinterpret_cast<const uint32_t *>(&v);
    } else {
        return bf2_bits(__floats2bfloat162_rn(lo, hi));
    }
}
// two pixels 0..255 as the mma operand type of T, exactly
template <typename T>
__device__ __forceinline__ uint32_t pack_px(float lo, float hi) {
    if constexpr (std::is_same_v<T, __half>)
        return pack_rn<__half>(lo, hi);
    else
        return pack_exact(lo, hi);
}
// x rounded to T and back (the value autocast's cast gives)
template <typename T>
__device__ __forceinline__ float round_to(float x) {
    if constexpr (std::is_same_v<T, __half>)
        return __half2float(__float2half_rn(x));
    else if constexpr (std::is_same_v<T, __nv_bfloat16>)
        return __bfloat162float(__float2bfloat16_rn(x));
    else
        return x;
}
// the output element of x: x itself, or x rounded once to T (fp16 overflows to +-inf)
template <typename T>
__device__ __forceinline__ T to_out(float x) {
    if constexpr (std::is_same_v<T, __half>)
        return __float2half_rn(x);
    else if constexpr (std::is_same_v<T, __nv_bfloat16>)
        return __float2bfloat16_rn(x);
    else
        return x;
}
// d = a * b + c, m16n8k16, fp32 accumulate; f16 operands for T = __half, bf16 otherwise
template <typename T = float>
__device__ __forceinline__ void mma16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1,
                                         const float (&c)[4]) {
    if constexpr (std::is_same_v<T, __half>)
        asm volatile(
            "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, "
            "{%10,%11,%12,%13};"
            : "=f"(d[0]), "=f"(d[1]), "=f"(d[2]), "=f"(d[3])
            : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1), "f"(c[0]), "f"(c[1]), "f"(c[2]), "f"(c[3]));
    else
        asm volatile(
            "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, "
            "{%10,%11,%12,%13};"
            : "=f"(d[0]), "=f"(d[1]), "=f"(d[2]), "=f"(d[3])
            : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1), "f"(c[0]), "f"(c[1]), "f"(c[2]), "f"(c[3]));
}
// acc += a * b over one k-step, one term of type T
template <typename T>
__device__ __forceinline__ void mma_one(float (&acc)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    const float z[4] = {0.f, 0.f, 0.f, 0.f};
    float d[4];
    mma16816<T>(d, a, b0, b1, z);
#pragma unroll
    for (int q = 0; q < 4; ++q) acc[q] = __fadd_rn(acc[q], d[q]);
}
// acc += (a_hi + a_mid + a_lo) * b over one k-step (operand split on A)
__device__ __forceinline__ void mma_split_a(float (&acc)[4], const uint32_t (&ah)[4], const uint32_t (&am)[4],
                                            const uint32_t (&al)[4], uint32_t b0, uint32_t b1) {
    const float z[4] = {0.f, 0.f, 0.f, 0.f};
    float d[4];
    mma16816(d, al, b0, b1, z);
    mma16816(d, am, b0, b1, d);
    mma16816(d, ah, b0, b1, d);
#pragma unroll
    for (int q = 0; q < 4; ++q) acc[q] = __fadd_rn(acc[q], d[q]);
}
// acc += a * (b_hi + b_mid + b_lo) over one k-step (operand split on B)
__device__ __forceinline__ void mma_split_b(float (&acc)[4], const uint32_t (&a)[4], uint2 bh, uint2 bm, uint2 bl) {
    const float z[4] = {0.f, 0.f, 0.f, 0.f};
    float d[4];
    mma16816(d, a, bl.x, bl.y, z);
    mma16816(d, a, bm.x, bm.y, d);
    mma16816(d, a, bh.x, bh.y, d);
#pragma unroll
    for (int q = 0; q < 4; ++q) acc[q] = __fadd_rn(acc[q], d[q]);
}
// byte offset of output pixel p's window corner inside an HWC frame
__device__ __forceinline__ int pix_base(int p, int ow, int stride, int w, int c) {
    const int oy = p / ow, ox = p - oy * ow;
    return (oy * stride * w + ox * stride) * c;
}
// the packed plane-set tap of input channel ci (of the set) at window pixel pix = ky * w + kx; 0 (byte 0) past the set
template <int S>
__device__ __forceinline__ int set_tap(const vn_u8_frames_t (&src)[S], const int (&region)[S + 1], int n_srcs, int ci,
                                       int pix) {
    int t = 0;
#pragma unroll
    for (int s = 0; s < S; ++s)
        if (s < n_srcs) {
            const int cs = src[s].c;
            if (ci >= 0 && ci < cs) t = (region[s] + pix * cs + ci) << 2 | cs;
            ci -= cs;
        }
    return t;
}
// the plane-set byte of tap t for the output pixel whose window corner is pixel pp of the frame
__device__ __forceinline__ uint32_t set_px(const uint8_t *x, int pp, int t) { return x[(t >> 2) + pp * (t & 3)]; }

// The frames of a CTA, double-buffered in shared memory (one buffer when two do not fit): frame number `it` of the
// CTA's sequence sits in buffer it % nbuf and completes phase it / nbuf of that buffer's mbarrier.
struct FramePipe {
    uint8_t *buf;
    uint64_t *bar;
    int fb, nbuf;
    __device__ void load(int slot, const uint8_t *src) const {
        mbar_expect_tx(&bar[slot], (uint32_t)fb);
        bulk_g2s(buf + (size_t)slot * fb, src, (uint32_t)fb, &bar[slot]);
    }
    __device__ const uint8_t *wait(int it) const {
        const int slot = nbuf == 2 ? (it & 1) : 0;
        mbar_wait(&bar[slot], (uint32_t)((nbuf == 2 ? it >> 1 : it) & 1));
        return buf + (size_t)slot * fb;
    }
    __device__ int slot(int it) const { return nbuf == 2 ? (it & 1) : 0; }
    // a plane set's frame f: one bulk copy per source into its region, all on the slot's one transaction
    template <int S>
    __device__ void load_set(int slot, const vn_u8_frames_t (&src)[S], const int (&region)[S + 1], int n_srcs,
                             int f) const {
        mbar_expect_tx(&bar[slot], (uint32_t)fb);
        uint8_t *dst = buf + (size_t)slot * fb;
#pragma unroll
        for (int s = 0; s < S; ++s)
            if (s < n_srcs)
                bulk_g2s(dst + region[s], frame_src(src[s], f), (uint32_t)(region[s + 1] - region[s]), &bar[slot]);
    }
};

// The frame sources of a kernel: one (S = 1), or a plane set of n_srcs <= S sources whose frames sit at region[s] of a
// frame buffer (region[n_srcs] = fb), their output channels or tiles split into `groups` groups.
template <int S>
struct FwdArgs {
    vn_u8_frames_t src[S];
    const float *weight;   // [cout][K], K = c * k * k
    const float *bias;     // [cout] or null
    void *out;             // [n][cout][oh][ow] of the kernel's element type
    int k, stride, oh, ow, K, ksteps, nbuf, fb;
    int n_srcs, groups, cout;
    int region[S + 1];
};

template <int S>
__device__ __forceinline__ void load_frame(const FramePipe &pipe, int slot, const FwdArgs<S> &a, int f) {
    if constexpr (S == 1)
        pipe.load(slot, frame_src(a.src[0], f));
    else
        pipe.load_set(slot, a.src, a.region, a.n_srcs, f);
}

// Persistent grid; a CTA owns whole frames.  Its prologue splits (fp32) or rounds (16-bit T) the weights into shared
// memory in mma B-fragment order ([k-step][n-tile][hi, mid, lo or the one term][lane] uint2).  A warp owns two 16-pixel
// m-tiles of a frame and every output channel; the A fragments are the frame's bytes picked through a tap-offset table
// (implicit im2col).  Each C fragment row is 8 consecutive pixels of one channel, so every fp32 store instruction
// writes whole 32-byte sectors of the NCHW output (16-bit ones write half sectors, which L2 joins: the other half is
// the same thread's row g + 8).  A plane-set CTA owns output channels [grp * NT * 8, ...) of its frames.
template <int NT, typename T, int S>   // output channels of a CTA / 8, element type, frame sources
__global__ void __launch_bounds__(kFwdWarps * 32, 1) vn_conv_u8_fwd_kernel(const FwdArgs<S> a) {
    constexpr int TERMS = kTerms<T>;
    constexpr bool SET = S > 1;
    extern __shared__ __align__(128) uint8_t smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, tig = lane & 3;
    const int w = a.src[0].w, c = a.src[0].c, K = a.K, ksteps = a.ksteps;
    // a plane-set CTA's first frame, frame step and first output channel (blockIdx.x, gridDim.x and 0 otherwise)
    const auto f0 = [&] { if constexpr (SET) return (int)blockIdx.x / a.groups; else return blockIdx.x; };
    const auto fstep = [&] { if constexpr (SET) return (int)gridDim.x / a.groups; else return gridDim.x; };
    const auto co0 = [&] { if constexpr (SET) return (int)blockIdx.x % a.groups * NT * 8; else return 0; };
    uint2 *wfrag = reinterpret_cast<uint2 *>(smem + (size_t)a.nbuf * a.fb);
    int *tap = reinterpret_cast<int *>(wfrag + ksteps * NT * TERMS * 32);
    float *sbias = reinterpret_cast<float *>(tap + ksteps * 16);
    uint64_t *bar = reinterpret_cast<uint64_t *>(sbias + NT * 8);
    const FramePipe pipe{smem, bar, a.fb, a.nbuf};

    const int kk2 = a.k * a.k;
    for (int t = tid; t < ksteps * 16; t += blockDim.x) {
        int off = 0;   // padding taps read byte 0: their weight is zero
        if (t < K) {
            const int ci = t / kk2, r = t - ci * kk2, ky = r / a.k, kx = r - ky * a.k;
            if constexpr (SET)
                off = set_tap(a.src, a.region, a.n_srcs, ci, ky * w + kx);
            else
                off = (ky * w + kx) * c + ci;
        }
        tap[t] = off;
    }
    if (tid == 0) {
        mbar_init(&bar[0], 1);
        mbar_init(&bar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // the weights, indices and frames may be written by the kernels before this one; nothing is released early, so a
    // following env step cannot rewrite the batch rows or obs_state while they are read here
    asm volatile("griddepcontrol.wait;" ::: "memory");
    for (int e = tid; e < ksteps * NT * 32; e += blockDim.x) {
        const int ln = e & 31, j = (e >> 5) % NT, ks = (e >> 5) / NT;
        const int n = j * 8 + (ln >> 2), k0 = ks * 16 + (ln & 3) * 2;
        const float *wr = a.weight + (size_t)(co0() + n) * K;
        const float v0 = k0 < K ? wr[k0] : 0.f, v1 = k0 + 1 < K ? wr[k0 + 1] : 0.f;
        const float v8 = k0 + 8 < K ? wr[k0 + 8] : 0.f, v9 = k0 + 9 < K ? wr[k0 + 9] : 0.f;
        if constexpr (TERMS == 3) {
            uint32_t h0, m0, l0, h1, m1, l1;
            split3(v0, v1, h0, m0, l0);
            split3(v8, v9, h1, m1, l1);
            uint2 *dst = wfrag + (size_t)(ks * NT + j) * 96 + ln;
            dst[0] = make_uint2(h0, h1);
            dst[32] = make_uint2(m0, m1);
            dst[64] = make_uint2(l0, l1);
        } else {
            wfrag[(size_t)(ks * NT + j) * 32 + ln] = make_uint2(pack_rn<T>(v0, v1), pack_rn<T>(v8, v9));
        }
    }
    for (int co = tid; co < NT * 8; co += blockDim.x) sbias[co] = a.bias ? round_to<T>(a.bias[co0() + co]) : 0.f;
    const int n = a.src[0].n;
    if (tid == 0)
        for (int s = 0; s < a.nbuf; ++s) {
            const int f = f0() + s * fstep();
            if (f < n) load_frame(pipe, s, a, f);
        }
    __syncthreads();

    const int P = a.oh * a.ow, tasks = ((P + 15) / 16 + 1) / 2;
    int it = 0;
    for (int f = f0(); f < n; f += fstep(), ++it) {
        const uint8_t *x = pipe.wait(it);
        T *out = static_cast<T *>(a.out) + (int64_t)f * (SET ? a.cout : NT * 8) * P;
        if constexpr (SET) out += (int64_t)co0() * P;
        for (int task = warp; task < tasks; task += kFwdWarps) {
            int pb[2][2];
#pragma unroll
            for (int mt = 0; mt < 2; ++mt)
#pragma unroll
                for (int r = 0; r < 2; ++r) {
                    const int p = (task * 2 + mt) * 16 + g + r * 8;
                    pb[mt][r] = p < P ? pix_base(p, a.ow, a.stride, w, SET ? 1 : c) : 0;
                }
            float acc[2][NT][4];
#pragma unroll
            for (int mt = 0; mt < 2; ++mt)
#pragma unroll
                for (int j = 0; j < NT; ++j)
#pragma unroll
                    for (int q = 0; q < 4; ++q) acc[mt][j][q] = 0.f;
#pragma unroll 1
            for (int ks = 0; ks < ksteps; ++ks) {
                const int2 t01 = *reinterpret_cast<const int2 *>(tap + ks * 16 + tig * 2);
                const int2 t89 = *reinterpret_cast<const int2 *>(tap + ks * 16 + tig * 2 + 8);
                uint32_t af[2][4];
#pragma unroll
                for (int mt = 0; mt < 2; ++mt)
#pragma unroll
                    for (int r = 0; r < 2; ++r) {
                        if constexpr (SET) {
                            const int pp = pb[mt][r];
                            af[mt][r] = pack_px<T>(u8f(set_px(x, pp, t01.x)), u8f(set_px(x, pp, t01.y)));
                            af[mt][2 + r] = pack_px<T>(u8f(set_px(x, pp, t89.x)), u8f(set_px(x, pp, t89.y)));
                        } else {
                            const uint8_t *row = x + pb[mt][r];
                            af[mt][r] = pack_px<T>(u8f(row[t01.x]), u8f(row[t01.y]));
                            af[mt][2 + r] = pack_px<T>(u8f(row[t89.x]), u8f(row[t89.y]));
                        }
                    }
                const uint2 *wf = wfrag + (size_t)ks * NT * TERMS * 32 + lane;
#pragma unroll
                for (int j = 0; j < NT; ++j) {
                    if constexpr (TERMS == 3) {
                        const uint2 bh = wf[j * 96], bm = wf[j * 96 + 32], bl = wf[j * 96 + 64];
                        mma_split_b(acc[0][j], af[0], bh, bm, bl);
                        mma_split_b(acc[1][j], af[1], bh, bm, bl);
                    } else {
                        const uint2 b = wf[j * 32];
                        mma_one<T>(acc[0][j], af[0], b.x, b.y);
                        mma_one<T>(acc[1][j], af[1], b.x, b.y);
                    }
                }
            }
#pragma unroll
            for (int mt = 0; mt < 2; ++mt)
#pragma unroll
                for (int r = 0; r < 2; ++r) {
                    const int p = (task * 2 + mt) * 16 + g + r * 8;
                    if (p >= P) continue;
#pragma unroll
                    for (int j = 0; j < NT; ++j) {
                        const int co = j * 8 + tig * 2;
                        out[(int64_t)co * P + p] = to_out<T>(__fadd_rn(__fdiv_rn(acc[mt][j][2 * r], 255.f), sbias[co]));
                        out[(int64_t)(co + 1) * P + p] =
                            to_out<T>(__fadd_rn(__fdiv_rn(acc[mt][j][2 * r + 1], 255.f), sbias[co + 1]));
                    }
                }
        }
        __syncthreads();   // every warp is done with this buffer
        const int next = f + a.nbuf * fstep();
        if (tid == 0 && next < n) {
            fence_proxy_async();
            load_frame(pipe, pipe.slot(it), a, next);
        }
    }
}

template <int S>
struct WgradArgs {
    vn_u8_frames_t src[S];
    const void *grad_out;    // [n][cout][oh][ow] of the kernel's element type
    float *partial;          // [chunks][cout][K + 1]
    int cout, k, stride, oh, ow, K, mtiles, ntiles, nbuf, fb;
    int n_srcs, groups, group_tiles;
    int region[S + 1];
};

template <int S>
__device__ __forceinline__ void load_frame(const FramePipe &pipe, int slot, const WgradArgs<S> &a, int f) {
    if constexpr (S == 1)
        pipe.load(slot, frame_src(a.src[0], f));
    else
        pipe.load_set(slot, a.src, a.region, a.n_srcs, f);
}

// The frames of chunk q are [q * kWgradChunk, ...): the CTA's next frame after f, its chunks `cstep` apart.
__device__ __forceinline__ int next_frame(int f, int n, int cstep) {
    const int chunk_end = min(n, (f / kWgradChunk + 1) * kWgradChunk);
    return f + 1 < chunk_end ? f + 1 : (f / kWgradChunk + cstep) * kWgradChunk;
}

// dW[co][t] = sum over the chunk's frames and output pixels p of g[co][p] * x[tap t of p]: an implicit GEMM with
// M = cout, N = taps + 1 (the last tap reads 1: the bias gradient), K = pixels.  grad_out is A (read from global: each
// fragment row is 8 consecutive elements of one channel), split into three terms when it is fp32, and the frame's bytes
// are B.  A warp owns up to kWgradTiles (16 x 8) output tiles for the whole chunk.  Its registers sum one frame; the
// frame sums are added into the thread's own shared-memory column, and the chunk's raw sums go to partial[chunk].
// 16-bit grad_out is read one element at a time: a channel row is only 2-byte aligned when oh * ow is odd.
// A plane-set CTA owns tiles [grp * group_tiles, ...) of its chunks.
template <typename T, int S>
__global__ void __launch_bounds__(kWgradWarps * 32) vn_conv_u8_wgrad_kernel(const WgradArgs<S> a) {
    constexpr int TERMS = kTerms<T>;
    constexpr bool SET = S > 1;
    extern __shared__ __align__(128) uint8_t smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, tig = lane & 3;
    const int w = a.src[0].w, c = a.src[0].c, K = a.K, K1 = a.K + 1, cout = a.cout;
    // a plane-set CTA's first chunk and chunk step (blockIdx.x and gridDim.x otherwise)
    const auto chunk0 = [&] { if constexpr (SET) return (int)blockIdx.x / a.groups; else return blockIdx.x; };
    const auto cstep = [&] { if constexpr (SET) return (int)gridDim.x / a.groups; else return (int)gridDim.x; };
    int *tap = reinterpret_cast<int *>(smem + (size_t)a.nbuf * a.fb);
    uint64_t *bar = reinterpret_cast<uint64_t *>(tap + a.ntiles * 8);
    float *chunk_acc = reinterpret_cast<float *>(bar + 2) + tid;   // this thread's [kWgradTiles * 4] column
    const FramePipe pipe{smem, bar, a.fb, a.nbuf};

    const int kk2 = a.k * a.k;
    for (int t = tid; t < a.ntiles * 8; t += blockDim.x) {
        int off = t == K ? -1 : -2;   // -1: the bias tap (reads 1), -2: padding (reads 0)
        if (t < K) {
            const int ci = t / kk2, r = t - ci * kk2, ky = r / a.k, kx = r - ky * a.k;
            if constexpr (SET)
                off = set_tap(a.src, a.region, a.n_srcs, ci, ky * w + kx);
            else
                off = (ky * w + kx) * c + ci;
        }
        tap[t] = off;
    }
    if (tid == 0) {
        mbar_init(&bar[0], 1);
        mbar_init(&bar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    asm volatile("griddepcontrol.wait;" ::: "memory");
    __syncthreads();

    int tiles = a.mtiles * a.ntiles, g0 = 0;   // this CTA's tiles: [g0, tiles)
    if constexpr (SET) {
        g0 = (int)blockIdx.x % a.groups * a.group_tiles;
        tiles = min(tiles, g0 + a.group_tiles);
    }
    const int per = (tiles - g0 + kWgradWarps - 1) / kWgradWarps;
    const int t0 = g0 + warp * per, cnt = max(0, min(per, tiles - t0));
    int tmi[kWgradTiles], toff[kWgradTiles];
#pragma unroll
    for (int i = 0; i < kWgradTiles; ++i) {
        const int tl = i < cnt ? t0 + i : 0, mi = tl / a.ntiles;
        tmi[i] = mi;
        toff[i] = tap[(tl - mi * a.ntiles) * 8 + g];
    }

    const int n = a.src[0].n, P = a.oh * a.ow, ksteps = (P + 15) / 16;
    int f = chunk0() * kWgradChunk;
    if (tid == 0 && f < n) {
        load_frame(pipe, 0, a, f);
        const int f1 = next_frame(f, n, cstep());
        if (a.nbuf == 2 && f1 < n) load_frame(pipe, 1, a, f1);
    }
    int it = 0;
    for (int chunk = chunk0(); chunk * kWgradChunk < n; chunk += cstep()) {
        float acc[kWgradTiles][4];
#pragma unroll
        for (int i = 0; i < kWgradTiles; ++i)
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                acc[i][q] = 0.f;
                chunk_acc[(i * 4 + q) * kWgradWarps * 32] = 0.f;
            }
        const int end = min(n, (chunk + 1) * kWgradChunk);
        for (; f < end; f = next_frame(f, n, cstep()), ++it) {
            const uint8_t *x = pipe.wait(it);
            const T *gf = static_cast<const T *>(a.grad_out) + (int64_t)f * cout * P;
#pragma unroll 1
            for (int ks = 0; ks < ksteps; ++ks) {
                const int p0 = ks * 16 + tig * 2, cp = SET ? 1 : c;
                const int pb0 = p0 < P ? pix_base(p0, a.ow, a.stride, w, cp) : 0;
                const int pb1 = p0 + 1 < P ? pix_base(p0 + 1, a.ow, a.stride, w, cp) : 0;
                const int pb8 = p0 + 8 < P ? pix_base(p0 + 8, a.ow, a.stride, w, cp) : 0;
                const int pb9 = p0 + 9 < P ? pix_base(p0 + 9, a.ow, a.stride, w, cp) : 0;
                int cur = -1;
                uint32_t ah[4], am[4], al[4];
#pragma unroll
                for (int i = 0; i < kWgradTiles; ++i) {
                    if (i >= cnt) break;
                    if (tmi[i] != cur) {   // warp-uniform: the warp's tiles are sorted by m-tile
                        cur = tmi[i];
#pragma unroll
                        for (int r = 0; r < 2; ++r) {
                            const int co = cur * 16 + g + r * 8;
                            const bool ok = co < cout;
                            if constexpr (TERMS == 3) {
                                const float *gr = gf + (int64_t)co * P;
                                const float v0 = ok && p0 < P ? gr[p0] : 0.f, v1 = ok && p0 + 1 < P ? gr[p0 + 1] : 0.f;
                                const float v8 = ok && p0 + 8 < P ? gr[p0 + 8] : 0.f;
                                const float v9 = ok && p0 + 9 < P ? gr[p0 + 9] : 0.f;
                                split3(v0, v1, ah[r], am[r], al[r]);
                                split3(v8, v9, ah[2 + r], am[2 + r], al[2 + r]);
                            } else {   // the raw 16-bit patterns; 0 is +0 in both types
                                const uint16_t *gr = reinterpret_cast<const uint16_t *>(gf) + (int64_t)co * P;
                                const uint32_t v0 = ok && p0 < P ? gr[p0] : 0u, v1 = ok && p0 + 1 < P ? gr[p0 + 1] : 0u;
                                const uint32_t v8 = ok && p0 + 8 < P ? gr[p0 + 8] : 0u;
                                const uint32_t v9 = ok && p0 + 9 < P ? gr[p0 + 9] : 0u;
                                ah[r] = v0 | v1 << 16;
                                ah[2 + r] = v8 | v9 << 16;
                            }
                        }
                    }
                    const int o = toff[i];
                    float b0, b1, b8, b9;
                    if (o >= 0) {
                        if constexpr (SET) {
                            b0 = u8f(set_px(x, pb0, o));
                            b1 = u8f(set_px(x, pb1, o));
                            b8 = u8f(set_px(x, pb8, o));
                            b9 = u8f(set_px(x, pb9, o));
                        } else {
                            b0 = u8f(x[pb0 + o]);
                            b1 = u8f(x[pb1 + o]);
                            b8 = u8f(x[pb8 + o]);
                            b9 = u8f(x[pb9 + o]);
                        }
                    } else {
                        b0 = b1 = b8 = b9 = o == -1 ? 1.f : 0.f;
                    }
                    if constexpr (TERMS == 3)
                        mma_split_a(acc[i], ah, am, al, pack_exact(b0, b1), pack_exact(b8, b9));
                    else
                        mma_one<T>(acc[i], ah, pack_px<T>(b0, b1), pack_px<T>(b8, b9));
                }
            }
            // the frame's sums join the chunk's in shared memory: no register sum runs over more than one frame
#pragma unroll
            for (int i = 0; i < kWgradTiles; ++i)
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    float &s = chunk_acc[(i * 4 + q) * kWgradWarps * 32];
                    s = __fadd_rn(s, acc[i][q]);
                    acc[i][q] = 0.f;
                }
            __syncthreads();   // every warp is done with this buffer
            if (tid == 0) {
                int nx = next_frame(f, n, cstep());
                if (a.nbuf == 2 && nx < n) nx = next_frame(nx, n, cstep());
                if (nx < n) {
                    fence_proxy_async();
                    load_frame(pipe, pipe.slot(it), a, nx);
                }
            }
        }
        float *part = a.partial + (int64_t)chunk * cout * K1;
#pragma unroll
        for (int i = 0; i < kWgradTiles; ++i) {
            if (i >= cnt) break;
            const int tl = t0 + i, mi = tmi[i], nj = tl - mi * a.ntiles;
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                const int co = mi * 16 + g + r * 8, t = nj * 8 + tig * 2;
                if (co >= cout) continue;
                if (t < K1) part[(int64_t)co * K1 + t] = chunk_acc[(i * 4 + 2 * r) * kWgradWarps * 32];
                if (t + 1 < K1) part[(int64_t)co * K1 + t + 1] = chunk_acc[(i * 4 + 2 * r + 1) * kWgradWarps * 32];
            }
        }
    }
}

// out[o] = sum over chunks of partial[chunk][o], o = co * (K + 1) + t: lane ty of a column sums chunks ty, ty + 32, ...
// in order, then the 32 lane sums are added in a fixed tree.  Weight columns are scaled by 1/255, the bias column
// (t == K) is the bias gradient.
__global__ void __launch_bounds__(kReduceLanes * 32) vn_conv_u8_wgrad_reduce_kernel(const float *__restrict__ partial,
                                                                                   int chunks, int cout, int K,
                                                                                   float *__restrict__ grad_weight,
                                                                                   float *__restrict__ grad_bias) {
    __shared__ float red[kReduceLanes][33];
    asm volatile("griddepcontrol.wait;" ::: "memory");
    const int K1 = K + 1, total = cout * K1;
    const int tx = threadIdx.x, ty = threadIdx.y, o = blockIdx.x * 32 + tx;
    float s = 0.f;
    if (o < total)
        for (int q = ty; q < chunks; q += kReduceLanes) s = __fadd_rn(s, partial[(int64_t)q * total + o]);
    red[ty][tx] = s;
    __syncthreads();
#pragma unroll
    for (int st = kReduceLanes / 2; st > 0; st >>= 1) {
        if (ty < st) red[ty][tx] = __fadd_rn(red[ty][tx], red[ty + st][tx]);
        __syncthreads();
    }
    if (ty != 0 || o >= total) return;
    const int co = o / K1, t = o - co * K1;
    if (t < K)
        grad_weight[(int64_t)co * K + t] = __fdiv_rn(red[0][tx], 255.f);
    else if (grad_bias)
        grad_bias[co] = red[0][tx];
}

// ---------------------------------------------------------------- host side
struct ConvGeom {
    int oh, ow, K, fb;
    int c;                      // input channels (of the whole set)
    int region[kMaxSrcs + 1];   // plane sets: byte offset of each source's frame in a frame buffer
};

static bool aligned4(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 3) == 0; }
static bool aligned2(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 1) == 0; }

// Checks one frame source up to its channel count.
static int32_t source_args(const vn_u8_frames_t *src, const char *who) {
    VN_REQUIRE(src->n >= 0, "%s: n=%d", who, src->n);
    VN_REQUIRE(src->base, "%s: frame base is null", who);
    VN_REQUIRE(aligned16(src->base) && (src->pitch & 15) == 0, "%s: frame base and pitch (%lld) must be 16-byte aligned",
               who, (long long)src->pitch);
    VN_REQUIRE(src->h > 0 && src->w > 0 && src->c > 0, "%s: frame %d x %d x %d", who, src->h, src->w, src->c);
    VN_REQUIRE(src->pitch >= (int64_t)src->h * src->w * src->c, "%s: pitch %lld is less than a %d x %d x %d frame", who,
               (long long)src->pitch, src->h, src->w, src->c);
    VN_REQUIRE(!src->idx || (src->idx_t >= 1 && src->n % src->idx_t == 0), "%s: idx_t=%d does not divide n=%d", who,
               src->idx_t, src->n);
    if (src->c != 1 && src->c != 3) {
        set_error("%s: %d channels (1 or 3 are supported)", who, src->c);
        return VN_EUNSUPPORTED;
    }
    return VN_OK;
}

// Checks the layer shape for frames of `src`'s size with c input channels in all.
static int32_t layer_args(const vn_u8_frames_t *src, int c, int32_t cout, int32_t k, int32_t stride, const char *who,
                          ConvGeom *g) {
    if (k < 1 || k > 8 || stride < 1 || stride > k) {
        set_error("%s: kernel %d, stride %d (1 <= stride <= kernel <= 8 are supported)", who, k, stride);
        return VN_EUNSUPPORTED;
    }
    if (cout < 8 || cout > 64 || cout % 8) {
        set_error("%s: %d output channels (multiples of 8 up to 64 are supported)", who, cout);
        return VN_EUNSUPPORTED;
    }
    if (src->h < k || src->w < k || src->h > kMaxFrameSide || src->w > kMaxFrameSide) {
        set_error("%s: %d x %d frame with kernel %d (frames of kernel .. %d pixels a side are supported)", who, src->h,
                  src->w, k, kMaxFrameSide);
        return VN_EUNSUPPORTED;
    }
    g->oh = (src->h - k) / stride + 1;
    g->ow = (src->w - k) / stride + 1;
    g->K = c * k * k;
    g->c = c;
    return VN_OK;
}

// Checks the frame source and the layer shape shared by the forward and the backward.
static int32_t conv_args(const vn_u8_frames_t *src, int32_t cout, int32_t k, int32_t stride, const char *who, ConvGeom *g) {
    VN_REQUIRE(src, "%s: src is null", who);
    int32_t rc = source_args(src, who);
    if (rc) return rc;
    rc = layer_args(src, src->c, cout, k, stride, who, g);
    if (rc) return rc;
    g->fb = (src->h * src->w * src->c + 15) & ~15;
    g->region[0] = 0;
    g->region[1] = g->fb;
    return VN_OK;
}

// Shared memory past the frame buffers: the forward's weight fragments of nt n-tiles, tap table and bias, and the
// weight gradient's tap table and per-thread chunk sums.
template <typename T>
static int fwd_rest(int ksteps, int nt) { return ksteps * nt * kTerms<T> * 32 * 8 + ksteps * 16 * 4 + nt * 8 * 4 + 16; }
static int wgrad_rest(int ntiles) { return ntiles * 8 * 4 + 16 + kWgradTiles * 4 * kWgradWarps * 32 * 4; }

// Checks a plane set (1 .. kMaxSrcs sources of one size and index shape, 1 or 3 channels each, kMaxSetChannels in all)
// and the layer shape, and that one frame buffer of the set fits beside the tables of both kernels.
static int32_t set_args(const vn_u8_frames_t *srcs, int32_t n_srcs, int32_t cout, int32_t k, int32_t stride,
                        const char *who, ConvGeom *g) {
    VN_REQUIRE(srcs, "%s: srcs is null", who);
    VN_REQUIRE(n_srcs >= 1, "%s: %d sources", who, n_srcs);
    if (n_srcs > kMaxSrcs) {
        set_error("%s: %d sources (1 to %d are supported)", who, n_srcs, kMaxSrcs);
        return VN_EUNSUPPORTED;
    }
    int c = 0;
    g->region[0] = 0;
    for (int s = 0; s < n_srcs; ++s) {
        const vn_u8_frames_t *f = &srcs[s];
        char whos[96];
        snprintf(whos, sizeof whos, "%s: source %d", who, s);
        const int32_t rc = source_args(f, whos);
        if (rc) return rc;
        VN_REQUIRE(f->n == srcs[0].n && f->idx_t == srcs[0].idx_t && f->h == srcs[0].h && f->w == srcs[0].w,
                   "%s: n, idx_t, h, w (%d, %d, %d, %d) differ from source 0's (%d, %d, %d, %d)", whos, f->n, f->idx_t,
                   f->h, f->w, srcs[0].n, srcs[0].idx_t, srcs[0].h, srcs[0].w);
        c += f->c;
        g->region[s + 1] = g->region[s] + ((f->h * f->w * f->c + 15) & ~15);
    }
    if (c > kMaxSetChannels) {
        set_error("%s: %d channels in all (at most %d are supported)", who, c, kMaxSetChannels);
        return VN_EUNSUPPORTED;
    }
    const int32_t rc = layer_args(srcs, c, cout, k, stride, who, g);
    if (rc) return rc;
    g->fb = g->region[n_srcs];
    const int ksteps = (g->K + 15) / 16, ntiles = (g->K + 1 + 7) / 8;
    if (g->fb + fwd_rest<float>(ksteps, 1) > kMaxSmemConv || g->fb + wgrad_rest(ntiles) > kMaxSmemConv) {
        set_error("%s: a %d x %d frame set of %d channels (%d bytes) does not fit in shared memory", who, srcs->h,
                  srcs->w, c, g->fb);
        return VN_EUNSUPPORTED;
    }
    return VN_OK;
}

static int64_t chunks_of(int64_t n) { return (n + kWgradChunk - 1) / kWgradChunk; }

template <typename T, int S>
using FwdKernel = void (*)(const FwdArgs<S>);
template <typename T, int S>
static const FwdKernel<T, S> kFwdKernels[8] = {
    vn_conv_u8_fwd_kernel<1, T, S>, vn_conv_u8_fwd_kernel<2, T, S>, vn_conv_u8_fwd_kernel<3, T, S>,
    vn_conv_u8_fwd_kernel<4, T, S>, vn_conv_u8_fwd_kernel<5, T, S>, vn_conv_u8_fwd_kernel<6, T, S>,
    vn_conv_u8_fwd_kernel<7, T, S>, vn_conv_u8_fwd_kernel<8, T, S>};

// Shared memory of `frames_bytes` frame buffers plus `rest`: two buffers when they fit, else one.
static int frame_buffers(int fb, int rest) { return 2 * fb + rest <= kMaxSmemConv ? 2 : 1; }

// A persistent grid: as many CTAs of `kernel` as are resident at once (registers and shared memory), at most `work`,
// a multiple of `groups` (work is).
template <typename... KArgs>
static int32_t persistent_grid(void (*kernel)(KArgs...), int threads, int smem, int64_t work, const char *who,
                               int *grid, int groups = 1) {
    int per_sm = 0;
    const cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem);
    if (e != cudaSuccess || per_sm < 1) {
        cudaGetLastError();
        set_error("%s: occupancy query: %s", who, cudaGetErrorString(e));
        return VN_ECUDA;
    }
    const int64_t cap = (int64_t)sm_count() * per_sm / groups * groups;
    *grid = (int)(work < cap ? work : cap);
    return VN_OK;
}

template <typename A>
static void set_sources(A &a, const vn_u8_frames_t *src, int n_srcs, const ConvGeom &g) {
    for (int s = 0; s < n_srcs; ++s) a.src[s] = src[s];
    a.n_srcs = n_srcs;
    for (int s = 0; s <= n_srcs; ++s) a.region[s] = g.region[s];
}

// The forward launch of element type T and S frame sources for checked arguments and n > 0.  A plane set splits its
// output channels into the fewest groups whose weight fragments fit beside two frame buffers, else beside one.
template <typename T, int S>
static int32_t conv_forward(const vn_u8_frames_t *src, int n_srcs, const ConvGeom &g, const float *weight,
                            const float *bias, int32_t cout, int32_t k, int32_t stride, void *out, void *stream,
                            const char *who) {
    const int ksteps = (g.K + 15) / 16;
    int NT = cout / 8, groups = 1;
    if (S > 1) {
        int pick = 0;
        for (int nbuf = 2; nbuf >= 1 && !pick; --nbuf)
            for (int gr = 1; gr <= NT && !pick; ++gr)
                if (NT % gr == 0 && nbuf * g.fb + fwd_rest<T>(ksteps, NT / gr) <= kMaxSmemConv) pick = gr;
        groups = pick;   // set_args checked that one n-tile fits beside one buffer
        NT /= groups;
    }
    const int rest = fwd_rest<T>(ksteps, NT);
    const int nbuf = frame_buffers(g.fb, rest), smem = nbuf * g.fb + rest;
    const FwdKernel<T, S> kernel = kFwdKernels<T, S>[NT - 1];
    int32_t rc = ensure_smem(kernel, smem);
    if (rc) return rc;
    int grid;
    rc = persistent_grid(kernel, kFwdWarps * 32, smem, (int64_t)src->n * groups, who, &grid, groups);
    if (rc) return rc;
    FwdArgs<S> a{};
    set_sources(a, src, n_srcs, g);
    a.weight = weight;
    a.bias = bias;
    a.out = out;
    a.k = k;
    a.stride = stride;
    a.oh = g.oh;
    a.ow = g.ow;
    a.K = g.K;
    a.ksteps = ksteps;
    a.nbuf = nbuf;
    a.fb = g.fb;
    a.groups = groups;
    a.cout = cout;
    return launch(kernel, "vn_conv_u8_fwd_kernel", dim3(grid), dim3(kFwdWarps * 32), (size_t)smem,
                  (cudaStream_t)stream, true, a);
}

// Checks the weight-gradient scratch shared by the backward entry points.
static int32_t scratch_args(const vn_u8_frames_t *src, const ConvGeom &g, int32_t cout, int32_t k,
                            const void *scratch, int64_t scratch_bytes, const char *who) {
    const int64_t need = vn_conv_u8_wgrad_scratch_bytes(src->n, g.c, cout, k);
    VN_REQUIRE(scratch_bytes >= need, "%s: %lld scratch bytes, %lld needed", who, (long long)scratch_bytes,
               (long long)need);
    VN_REQUIRE(need == 0 || (scratch && aligned16(scratch)), "%s: scratch must be a 16-byte aligned device buffer",
               who);
    return VN_OK;
}

// The two backward launches of element type T and S frame sources for checked arguments and n > 0.  A plane set
// splits its (cout, tap) tiles into the fewest groups of at most kWgradWarps * kWgradTiles.
template <typename T, int S>
static int32_t conv_backward(const vn_u8_frames_t *src, int n_srcs, const ConvGeom &g, const void *grad_out,
                             int32_t cout, int32_t k, int32_t stride, float *grad_weight, float *grad_bias,
                             void *scratch, void *stream, const char *who) {
    const int mtiles = (cout + 15) / 16, ntiles = (g.K + 1 + 7) / 8, tiles = mtiles * ntiles;
    const int groups = S > 1 ? (tiles + kWgradWarps * kWgradTiles - 1) / (kWgradWarps * kWgradTiles) : 1;
    const int rest = wgrad_rest(ntiles);
    const int nbuf = frame_buffers(g.fb, rest), smem = nbuf * g.fb + rest;
    int32_t rc = ensure_smem(vn_conv_u8_wgrad_kernel<T, S>, smem);
    if (rc) return rc;
    const int64_t chunks = chunks_of(src->n);
    int grid;
    rc = persistent_grid(vn_conv_u8_wgrad_kernel<T, S>, kWgradWarps * 32, smem, chunks * groups, who, &grid, groups);
    if (rc) return rc;
    WgradArgs<S> a{};
    set_sources(a, src, n_srcs, g);
    a.grad_out = grad_out;
    a.partial = (float *)scratch;
    a.cout = cout;
    a.k = k;
    a.stride = stride;
    a.oh = g.oh;
    a.ow = g.ow;
    a.K = g.K;
    a.mtiles = mtiles;
    a.ntiles = ntiles;
    a.nbuf = nbuf;
    a.fb = g.fb;
    a.groups = groups;
    a.group_tiles = (tiles + groups - 1) / groups;
    rc = launch(vn_conv_u8_wgrad_kernel<T, S>, "vn_conv_u8_wgrad_kernel", dim3(grid), dim3(kWgradWarps * 32),
                (size_t)smem, (cudaStream_t)stream, true, a);
    if (rc) return rc;
    const int outputs = cout * (g.K + 1);
    return launch(vn_conv_u8_wgrad_reduce_kernel, "vn_conv_u8_wgrad_reduce_kernel", dim3((outputs + 31) / 32),
                  dim3(32, kReduceLanes), 0, (cudaStream_t)stream, true, (const float *)scratch, (int)chunks,
                  (int)cout, g.K, grad_weight, grad_bias);
}

// The launch of S frame sources in fp32 (lp false) or in the checked 16-bit `dtype`.
template <int S>
static int32_t forward_of(const vn_u8_frames_t *src, int n_srcs, const ConvGeom &g, const float *weight,
                          const float *bias, int32_t cout, int32_t k, int32_t stride, bool lp, int32_t dtype, void *out,
                          void *stream, const char *who) {
    if (!lp) return conv_forward<float, S>(src, n_srcs, g, weight, bias, cout, k, stride, out, stream, who);
    if (dtype == VN_DTYPE_F16) return conv_forward<__half, S>(src, n_srcs, g, weight, bias, cout, k, stride, out, stream, who);
    return conv_forward<__nv_bfloat16, S>(src, n_srcs, g, weight, bias, cout, k, stride, out, stream, who);
}

template <int S>
static int32_t backward_of(const vn_u8_frames_t *src, int n_srcs, const ConvGeom &g, const void *grad_out,
                           int32_t cout, int32_t k, int32_t stride, float *grad_weight, float *grad_bias,
                           void *scratch, bool lp, int32_t dtype, void *stream, const char *who) {
    if (!lp)
        return conv_backward<float, S>(src, n_srcs, g, grad_out, cout, k, stride, grad_weight, grad_bias, scratch,
                                       stream, who);
    if (dtype == VN_DTYPE_F16)
        return conv_backward<__half, S>(src, n_srcs, g, grad_out, cout, k, stride, grad_weight, grad_bias, scratch,
                                        stream, who);
    return conv_backward<__nv_bfloat16, S>(src, n_srcs, g, grad_out, cout, k, stride, grad_weight, grad_bias, scratch,
                                           stream, who);
}

static int32_t dtype_arg(int32_t dtype, const char *who) {
    if (dtype != VN_DTYPE_F16 && dtype != VN_DTYPE_BF16) {
        set_error("%s: dtype %d (VN_DTYPE_F16 or VN_DTYPE_BF16 are supported)", who, dtype);
        return VN_EUNSUPPORTED;
    }
    return VN_OK;
}

// The argument checks and launch of every forward entry point: one source (set false) or a plane set of n_srcs, in
// fp32 (lp false) or in a 16-bit dtype (the _lp entry points).
static int32_t forward_entry(const vn_u8_frames_t *src, int32_t n_srcs, bool set, const float *weight,
                             const float *bias, int32_t cout, int32_t k, int32_t stride, bool lp, int32_t dtype,
                             void *out, void *stream, const char *who) {
    ConvGeom g;
    int32_t rc = set ? set_args(src, n_srcs, cout, k, stride, who, &g) : conv_args(src, cout, k, stride, who, &g);
    if (rc) return rc;
    if (!lp) {
        VN_REQUIRE(weight && out, "%s: weight and out must not be null", who);
        VN_REQUIRE(aligned4(weight) && aligned4(bias) && aligned4(out), "%s: weight, bias and out must be 4-byte aligned",
                   who);
    } else {
        rc = dtype_arg(dtype, who);
        if (rc) return rc;
        VN_REQUIRE(weight && out, "%s: weight and out must not be null", who);
        VN_REQUIRE(aligned4(weight) && aligned4(bias), "%s: weight and bias must be 4-byte aligned", who);
        VN_REQUIRE(aligned2(out), "%s: out must be 2-byte aligned", who);
    }
    if (src->n == 0) return VN_OK;
    return set ? forward_of<kMaxSrcs>(src, n_srcs, g, weight, bias, cout, k, stride, lp, dtype, out, stream, who)
               : forward_of<1>(src, 1, g, weight, bias, cout, k, stride, lp, dtype, out, stream, who);
}

// The argument checks and launches of every backward entry point (see forward_entry).
static int32_t backward_entry(const vn_u8_frames_t *src, int32_t n_srcs, bool set, const void *grad_out, bool lp,
                              int32_t dtype, int32_t cout, int32_t k, int32_t stride, float *grad_weight,
                              float *grad_bias, void *scratch, int64_t scratch_bytes, void *stream, const char *who) {
    ConvGeom g;
    int32_t rc = set ? set_args(src, n_srcs, cout, k, stride, who, &g) : conv_args(src, cout, k, stride, who, &g);
    if (rc) return rc;
    if (!lp) {
        VN_REQUIRE(grad_out && grad_weight, "%s: grad_out and grad_weight must not be null", who);
        VN_REQUIRE(aligned4(grad_out) && aligned4(grad_weight) && aligned4(grad_bias),
                   "%s: grad_out, grad_weight and grad_bias must be 4-byte aligned", who);
    } else {
        rc = dtype_arg(dtype, who);
        if (rc) return rc;
        VN_REQUIRE(grad_out && grad_weight, "%s: grad_out and grad_weight must not be null", who);
        VN_REQUIRE(aligned2(grad_out), "%s: grad_out must be 2-byte aligned", who);
        VN_REQUIRE(aligned4(grad_weight) && aligned4(grad_bias), "%s: grad_weight and grad_bias must be 4-byte aligned",
                   who);
    }
    rc = scratch_args(src, g, cout, k, scratch, scratch_bytes, who);
    if (rc) return rc;
    if (src->n == 0) return VN_OK;
    return set ? backward_of<kMaxSrcs>(src, n_srcs, g, grad_out, cout, k, stride, grad_weight, grad_bias, scratch, lp,
                                       dtype, stream, who)
               : backward_of<1>(src, 1, g, grad_out, cout, k, stride, grad_weight, grad_bias, scratch, lp, dtype,
                                stream, who);
}

}  // namespace vn

extern "C" {

int32_t vn_conv_u8_forward(const vn_u8_frames_t *src, const float *weight, const float *bias, int32_t cout, int32_t k,
                           int32_t stride, float *out, void *stream) {
    return vn::forward_entry(src, 1, false, weight, bias, cout, k, stride, false, 0, out, stream, "conv_u8_forward");
}

int32_t vn_conv_u8_forward_lp(const vn_u8_frames_t *src, const float *weight, const float *bias, int32_t cout,
                              int32_t k, int32_t stride, int32_t dtype, void *out, void *stream) {
    return vn::forward_entry(src, 1, false, weight, bias, cout, k, stride, true, dtype, out, stream, "conv_u8_forward_lp");
}

int64_t vn_conv_u8_wgrad_scratch_bytes(int32_t n, int32_t c, int32_t cout, int32_t k) {
    if (n < 0 || c < 1 || cout < 1 || k < 1) return -1;
    return vn::chunks_of(n) * cout * ((int64_t)c * k * k + 1) * (int64_t)sizeof(float);
}

int32_t vn_conv_u8_backward(const vn_u8_frames_t *src, const float *grad_out, int32_t cout, int32_t k, int32_t stride,
                            float *grad_weight, float *grad_bias, void *scratch, int64_t scratch_bytes, void *stream) {
    return vn::backward_entry(src, 1, false, grad_out, false, 0, cout, k, stride, grad_weight, grad_bias, scratch,
                              scratch_bytes, stream, "conv_u8_backward");
}

int32_t vn_conv_u8_backward_lp(const vn_u8_frames_t *src, const void *grad_out, int32_t dtype, int32_t cout,
                               int32_t k, int32_t stride, float *grad_weight, float *grad_bias, void *scratch,
                               int64_t scratch_bytes, void *stream) {
    return vn::backward_entry(src, 1, false, grad_out, true, dtype, cout, k, stride, grad_weight, grad_bias, scratch,
                              scratch_bytes, stream, "conv_u8_backward_lp");
}

int32_t vn_conv_u8_planes_forward(const vn_u8_frames_t *srcs, int32_t n_srcs, const float *weight, const float *bias,
                                  int32_t cout, int32_t k, int32_t stride, float *out, void *stream) {
    return vn::forward_entry(srcs, n_srcs, true, weight, bias, cout, k, stride, false, 0, out, stream,
                             "conv_u8_planes_forward");
}

int32_t vn_conv_u8_planes_forward_lp(const vn_u8_frames_t *srcs, int32_t n_srcs, const float *weight,
                                     const float *bias, int32_t cout, int32_t k, int32_t stride, int32_t dtype,
                                     void *out, void *stream) {
    return vn::forward_entry(srcs, n_srcs, true, weight, bias, cout, k, stride, true, dtype, out, stream,
                             "conv_u8_planes_forward_lp");
}

int32_t vn_conv_u8_planes_backward(const vn_u8_frames_t *srcs, int32_t n_srcs, const float *grad_out, int32_t cout,
                                   int32_t k, int32_t stride, float *grad_weight, float *grad_bias, void *scratch,
                                   int64_t scratch_bytes, void *stream) {
    return vn::backward_entry(srcs, n_srcs, true, grad_out, false, 0, cout, k, stride, grad_weight, grad_bias, scratch,
                              scratch_bytes, stream, "conv_u8_planes_backward");
}

int32_t vn_conv_u8_planes_backward_lp(const vn_u8_frames_t *srcs, int32_t n_srcs, const void *grad_out, int32_t dtype,
                                      int32_t cout, int32_t k, int32_t stride, float *grad_weight, float *grad_bias,
                                      void *scratch, int64_t scratch_bytes, void *stream) {
    return vn::backward_entry(srcs, n_srcs, true, grad_out, true, dtype, cout, k, stride, grad_weight, grad_bias, scratch,
                              scratch_bytes, stream, "conv_u8_planes_backward_lp");
}

}  // extern "C"
