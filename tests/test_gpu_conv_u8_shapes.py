"""Every uint8 first-convolution kernel and launch shape (vn_conv.cu) against exact and float64 references.

The host code picks one of 48 forward kernels ``vn_conv_u8_fwd_kernel<NT, T, S>`` (NT = output channels / 8 of a CTA,
T = float / __half / __nv_bfloat16, S = 1 source or a plane set), one of 6 ``vn_conv_u8_wgrad_kernel<T, S>``, and at
run time one or two shared-memory frame buffers, the number of output-channel or tile groups of a plane set, and how
many frames or 32-frame chunks each persistent CTA owns.  ``CASES`` names, for each launch shape, the branch it is there
for and the one-line derivation from ``fwd_rest``, ``wgrad_rest``, ``frame_buffers`` and ``kMaxSmemConv``;
``test_case_table_branches_and_operand_budget`` recomputes those branches on the CPU.

Exact family.  Pixels are integers and the weights (forward) and ``grad_out`` values (backward) are dyadic rationals
v * 2^-b with |v| < 2^b, exact in the operand type.  When x_max * count * max|v| * (1 + 2^-7) < 2^24 (count = K terms
per output in the forward, n * P per weight-gradient element; 2^-7 covers the three-term split's |hi| + |mid| + |lo|
exceeding |v|), every product on the tensor cores and every fp32 partial sum the kernels can form, in any order, is an
exact multiple of 2^-b.  The outputs are then fully determined: ``fp32(fp32(S / 255) + b)`` in the forward (b and the
result rounded to T for the 16-bit kernels), ``fp32(S_w / 255)`` and ``fp32(sum g)`` in the backward, with S and S_w
computed here in int64 by an unfold and an integer matmul (no cuDNN).  They are compared with ``torch.equal``, so a
dropped or doubled frame, a lost split term or a misplaced pixel shows as a wrong bit.  Regime "x255" takes pixels
0..255 (the pixel conversion), regime "x01" pixels in {0, 1} with as many significant bits in the weights / grad_out as
the budget allows (the mid and lo terms of the fp32 split).

Bound family.  Random uint8 frames, fp32 weights and grad_out, every element checked against float64 with the error
bound of the kernels' summation order, and each bound shown to reject three wrong answers on the same data."""
import ctypes as C
import importlib
import math
import re
import zlib
from collections import namedtuple

import pytest

torch = pytest.importorskip("torch")

vn = importlib.import_module("a2cat-vn-pytorch_b200")

F32, F16, BF16 = torch.float32, torch.float16, torch.bfloat16
ALL = (F32, F16, BF16)
DT_ID = {F32: "f32", F16: "f16", BF16: "bf16"}
T_NAME = {F32: "float", F16: "__half", BF16: "__nv_bfloat16"}
LP = {F16: vn.lib.DTYPE_F16, BF16: vn.lib.DTYPE_BF16}
B200_SMS = 148   # the budget check on the CPU sizes the SM-dependent batches for a B200

# vn_conv.cu's shared-memory plan, for the derivations in CASES
SMEM = 220 * 1024                                   # kMaxSmemConv
WGRAD_TILES, WGRAD_WARPS, CHUNK = 13, 8, 32         # kWgradTiles, kWgradWarps, kWgradChunk


def _cdiv(a, b):
    return -(-a // b)


def _fwd_rest(ksteps, nt, dtype):
    return ksteps * nt * (3 if dtype == F32 else 1) * 256 + ksteps * 64 + nt * 32 + 16


def _wgrad_rest(ntiles):
    return ntiles * 32 + 16 + WGRAD_TILES * 4 * WGRAD_WARPS * 32 * 4


def _plan(case, dtype):
    """What conv_forward / conv_backward pick for `case`: buffers, groups, NT; buffers, groups, tiles per warp."""
    h, w = case.hw
    fb = sum((h * w * c + 15) // 16 * 16 for c in case.planes)
    K = sum(case.planes) * case.k ** 2
    ksteps, nt, groups = (K + 15) // 16, case.cout // 8, 1
    if case.set:
        groups = next(gr for nbuf in (2, 1) for gr in range(1, nt + 1)
                      if nt % gr == 0 and nbuf * fb + _fwd_rest(ksteps, nt // gr, dtype) <= SMEM)
        nt //= groups
    fwd_nbuf = 2 if 2 * fb + _fwd_rest(ksteps, nt, dtype) <= SMEM else 1
    ntiles = (K + 1 + 7) // 8
    tiles = (case.cout + 15) // 16 * ntiles
    wgroups = _cdiv(tiles, WGRAD_WARPS * WGRAD_TILES) if case.set else 1
    return dict(fwd_nbuf=fwd_nbuf, fwd_groups=groups, nt=nt,
                wgrad_nbuf=2 if 2 * fb + _wgrad_rest(ntiles) <= SMEM else 1, wgrad_groups=wgroups,
                per_warp=_cdiv(_cdiv(tiles, wgroups), WGRAD_WARPS))


# n: an int, "many_frames" = 3 * 16 * SMs + 5 (more frames than 3 per resident 128-thread CTA, 16 of which fit an SM),
# or "many_chunks" = 32 * 8 * SMs + 17 (more 32-frame chunks than resident 256-thread CTAs, 8 of which fit an SM, and
# a partial last chunk).  via: "batch" (the nn layer on uint8 batches), "store" (forward_states on a [B, T] view of
# time-major indices), "abi" (the C ABI with guard bytes around out, grad_weight, grad_bias and the scratch).
# claims: {dtype: {plan key: value}} checked against _plan on the CPU.
Case = namedtuple("Case", "id planes set cout k s hw n via dtypes claims why")


def _f1(nt, set_):
    planes, k, s, hw = ((3, 1), 3, 2, (12, 12)) if set_ else ((3,), 4, 2, (14, 14))
    claims = {dt: dict(nt=nt, fwd_groups=1, fwd_nbuf=2) for dt in ALL}
    return Case("f1_%s_nt%d" % ("set" if set_ else "one", nt), planes, set_, 8 * nt, k, s, hw, 5, "batch", ALL, claims,
                "F1/W1: vn_conv_u8_fwd_kernel<%d, T, %d> (cout %d / 8, tiny frames: one group, two buffers) and "
                "vn_conv_u8_wgrad_kernel<T, %d>%s" % (nt, 4 if set_ else 1, 8 * nt, 4 if set_ else 1,
                                                      "; W4: cout 8 = half an m-tile" if nt == 1 else ""))


CASES = [_f1(nt, set_) for set_ in (False, True) for nt in range(1, 9)] + [
    Case("f2_rgb174_cout40", (3,), False, 40, 8, 4, (174, 174), 3, "abi", (F32,),
         {F32: dict(fwd_nbuf=1, wgrad_nbuf=1)},
         "F2: 174^2 x 3, k 8, cout 40, fp32: 2 * 90,832 + 47,024 > 225,280 -> one forward buffer; W2: "
         "2 * 90,832 + 54,064 > 225,280 -> one weight-gradient buffer"),
    Case("f2_rgb174_cout64", (3,), False, 64, 8, 4, (174, 174), 3, "abi", ALL,
         {F32: dict(fwd_nbuf=1, nt=8, wgrad_nbuf=1), F16: dict(fwd_nbuf=2, wgrad_nbuf=1)},
         "F2: cout 64 fp32: 2 * 90,832 + 74,768 > 225,280 -> one buffer, NT 8 (16-bit: + 25,616 fits -> two); W2: "
         "one weight-gradient buffer in every dtype"),
    Case("f3_c8_cout48", (3, 3, 1, 1), True, 48, 8, 4, (84, 84), 3, "abi", (F32,),
         {F32: dict(fwd_nbuf=2, fwd_groups=2, nt=3, wgrad_groups=2)},
         "F3: fb 56,448; 2 * 56,448 + fwd_rest(32, 6) = 262,608 > 225,280, + fwd_rest(32, 3) = 188,784 fits -> 2 "
         "groups of NT 3, two buffers; weight gradient 3 * 65 tiles -> 2 groups"),
    Case("f3_c8_cout48_n1", (3, 3, 1, 1), True, 48, 8, 4, (84, 84), 1, "batch", (F32,),
         {F32: dict(fwd_groups=2, nt=3)},
         "F4: n = 1 with 2 groups: the grid is n * groups = 2 CTAs sharing frame 0, the second buffer of each never "
         "filled; one 32-frame chunk of 1 frame"),
    Case("f3_rgbdd174_cout64", (3, 1, 1), True, 64, 8, 4, (174, 174), 2, "abi", (F32,),
         {F32: dict(fwd_nbuf=1, fwd_groups=2, nt=4, wgrad_nbuf=1, wgrad_groups=2)},
         "F3: fb 151,408: two buffers never fit; 151,408 + fwd_rest(20, 8) = 275,840 > 225,280, + fwd_rest(20, 4) "
         "= 214,272 fits -> one buffer, 2 groups of NT 4; weight gradient 4 * 41 tiles -> 2 groups, one buffer"),
    Case("f4_one_many_frames", (1,), False, 24, 3, 1, (5, 5), "many_frames", "batch", ALL, {},
         "F4: n > 3 * 16 * SMs >= 3 * grid: every forward CTA owns 3 or more frames and refills both buffers; "
         "NT 3 one source"),
    Case("f4_set_many_frames", (3, 1), True, 56, 2, 1, (3, 3), "many_frames", "batch", ALL, {F32: dict(nt=7)},
         "F4: as f4_one_many_frames for a plane set (groups 1, NT 7), 16-byte source regions"),
    Case("w2_rgbd174", (3, 1), True, 32, 8, 4, (174, 174), 3, "abi", ALL,
         {dt: dict(wgrad_nbuf=1, fwd_nbuf=1, fwd_groups=1) for dt in ALL},
         "W2: RGB-D 174^2: fb 121,120, 2 * 121,120 + 54,320 > 225,280 -> one weight-gradient buffer (and one "
         "forward buffer: two exceed it alone)"),
    Case("w3_one_many_chunks", (3,), False, 16, 2, 2, (2, 2), "many_chunks", "abi", ALL, {},
         "W3: ceil(n / 32) > 8 * SMs >= grid: CTAs sum 2 or more chunks (chunk += cstep, the prefetch across a "
         "chunk boundary, chunk_acc re-zeroed); n mod 32 = 17; side = k: P = 1; k 2 s 2"),
    Case("w3_set_many_chunks", (3, 1), True, 24, 2, 2, (2, 2), "many_chunks", "abi", ALL, {},
         "W3: as w3_one_many_chunks for a plane set"),
    Case("w4_cout64_k192", (3,), False, 64, 8, 4, (36, 36), 5, "batch", ALL, {F32: dict(per_warp=WGRAD_TILES)},
         "W4: cout 64, K 192: 4 m-tiles x 25 n-tiles = 100 tiles, 13 per warp = kWgradTiles"),
    Case("w4_k1_whole_ntile", (3, 3, 1), True, 16, 1, 1, (9, 7), 5, "batch", ALL, {},
         "W4: K + 1 = 8 = one whole n-tile (plane set (3, 3, 1), k 1); 9 x 7 frames, P = 63 odd"),
    Case("w4_tile_groups2", (3, 3), True, 64, 8, 4, (20, 20), 5, "batch", ALL, {F32: dict(wgrad_groups=2)},
         "W4: K 384: 4 x 49 = 196 tiles > 104 -> 2 tile groups"),
    Case("w4_tile_groups3", (3, 3, 1, 1), True, 64, 8, 4, (20, 20), 5, "batch", ALL, {F32: dict(wgrad_groups=3)},
         "W4: K 512: 4 x 65 = 260 tiles > 208 -> 3 tile groups"),
    Case("w5_depth85_odd_p", (1,), False, 16, 5, 4, (85, 85), 4, "abi", ALL, {},
         "W5: 85^2, k 5, s 4 -> 21 x 21, P = 441 odd (16-bit grad_out rows 2-byte aligned); E: 85 * 85 * 1 = 7,225 "
         "bytes in a padded 7,232-byte pitch"),
    Case("w5_rgbd85_odd_p", (3, 1), True, 24, 5, 4, (85, 85), 4, "abi", ALL, {},
         "W5: as w5_depth85_odd_p for a plane set; regions 21,680 + 7,232"),
    Case("e_wide_30x52", (3,), False, 16, 7, 3, (30, 52), 4, "batch", ALL, {}, "E: non-square 30 x 52 -> 8 x 16"),
    Case("e_tall_52x30", (3, 1), True, 16, 7, 3, (52, 30), 4, "batch", ALL, {}, "E: non-square 52 x 30 -> 16 x 8"),
    Case("e_k1s1", (3,), False, 16, 1, 1, (9, 11), 4, "batch", ALL, {},
         "E: k 1 s 1 (K 3, one mostly padded k-step); 9 * 11 * 3 = 297 bytes, not a multiple of 16"),
    Case("e_k8s8", (3,), False, 16, 8, 8, (40, 40), 4, "batch", ALL, {}, "E: k 8 s 8 -> 5 x 5"),
    Case("e_k5s3", (3, 1), True, 16, 5, 3, (23, 23), 4, "batch", ALL, {}, "E: k 5 s 3 -> 7 x 7"),
    Case("e_p9", (3,), False, 32, 8, 4, (16, 16), 4, "batch", ALL, {}, "E: P = 9 < 16: one masked m-tile / k-step"),
] + [Case("e_n%d" % n, (3,), False, 16, 4, 2, (14, 14), n, "batch", ALL, {},
          "E: backward with n = %d (%s)" % (n, {1: "one frame", 31: "one partial chunk", 32: "one whole chunk",
                                                 33: "a whole and a one-frame chunk"}[n]))
     for n in (1, 31, 32, 33)] + [
    Case("e_store_one", (3,), False, 24, 4, 2, (20, 28), 35, "store", ALL, {},
         "E: forward_states on a [7, 5] view of time-major [5, 7] indices, 20 x 28 maze store"),
    Case("e_store_set", (3, 1), True, 40, 3, 2, (20, 28), 35, "store", ALL, {},
         "E: U8PlanesConv2d.forward_states, rgb + depth of two index views, NT 5"),
]
CASE_IDS = [c.id for c in CASES]
REGIMES = ("x255", "x01")


def _n(case, sms):
    return {"many_frames": 3 * 16 * sms + 5, "many_chunks": 32 * 8 * sms + 17}.get(case.n, case.n)


def _geom(case):
    h, w = case.hw
    oh, ow = (h - case.k) // case.s + 1, (w - case.k) // case.s + 1
    return oh, ow, sum(case.planes) * case.k ** 2


# ---------------------------------------------------------------- exact family: operands and budget
_MANT = {F32: 24, F16: 11, BF16: 8}


def _value_bits(x_max, count, dtype):
    """The most significant bits b (up to T's precision) with x_max * count * (2^b - 1) * (1 + 2^-7) < 2^24."""
    b = _MANT[dtype]
    while b > 1 and x_max * count * (2 ** b - 1) * (1 + 2 ** -7) >= 2 ** 24:
        b -= 1
    return b


def _terms(v, dtype):
    """The operand terms the kernel multiplies: split3's bf16 hi + mid + lo of fp32 v, or v itself (16-bit)."""
    if dtype != F32:
        return [v]
    hi = v.bfloat16().float()
    r = v - hi
    mid = r.bfloat16().float()
    return [hi, mid, (r - mid).bfloat16().float()]


def _budget(x_max, count, ints, bits, dtype):
    """x_max * count * max over the values of sum |term|, in units of 2^-bits, over 2^24 (< 1: every partial sum is
    exact); also checks that the values are exact in T and that the split reproduces them."""
    v = ints.float() * 2.0 ** -bits
    terms = _terms(v, dtype)
    assert torch.equal(sum(terms[1:], terms[0]) if dtype == F32 else v.to(dtype).float(), v)
    worst = float(sum(t.abs() for t in terms).max()) * 2 ** bits if ints.numel() else 0.0
    return x_max * count * worst / 2 ** 24


Ops = namedtuple("Ops", "n x_max W bw G bg b xs")


def _operands(case, dtype, regime, sms):
    """Exact-family operands on the CPU: W [cout, K] and G [n, cout, P] int64 scaled by 2^-bw / 2^-bg, fp32 bias, and
    (batch / abi cases) uint8 frames [n, pitch] per plane, pad bytes random 0..255."""
    n = _n(case, sms)
    oh, ow, K = _geom(case)
    gen = torch.Generator().manual_seed(zlib.crc32(("%s/%s/%s" % (case.id, DT_ID[dtype], regime)).encode()))
    x_max = 255 if regime == "x255" else 1
    bw, bg = _value_bits(x_max, K, dtype), _value_bits(x_max, n * oh * ow, dtype)
    W = torch.randint(1 - 2 ** bw, 2 ** bw, (case.cout, K), generator=gen)
    G = torch.randint(1 - 2 ** bg, 2 ** bg, (n, case.cout, oh * ow), generator=gen)
    b = torch.randn(case.cout, generator=gen)
    xs = []
    if case.via != "store":
        h, w = case.hw
        for c in case.planes:
            pitch = (h * w * c + 15) // 16 * 16
            raw = torch.randint(0, 256, (max(n, 1), pitch), dtype=torch.uint8, generator=gen)
            raw[:, :h * w * c] = torch.randint(0, x_max + 1, (max(n, 1), h * w * c), dtype=torch.uint8, generator=gen)
            xs.append(raw)
    return Ops(n, x_max, W, bw, G, bg, b, xs)


def _budgets(case, dtype, ops):
    oh, ow, K = _geom(case)
    return (_budget(ops.x_max, K, ops.W, ops.bw, dtype),
            _budget(ops.x_max, ops.n * oh * ow, ops.G, ops.bg, dtype))


def _cols(x, k, s):
    """[n, c, h, w] (any dtype) -> [n, P, c * k * k] patches in the weight's (ci, ky, kx) order."""
    n, c = x.shape[:2]
    u = x.unfold(2, k, s).unfold(3, k, s)                      # [n, c, oh, ow, k, k]
    return u.permute(0, 2, 3, 1, 4, 5).reshape(n, -1, c * k * k)


def _exact_expected(case, dtype, ops, frames):
    """(y, grad_weight, grad_bias) the kernels must return bit for bit; frames: uint8 CPU [n, h, w, c] per plane."""
    oh, ow, K = _geom(case)
    n, cout = ops.n, case.cout
    cols = _cols(torch.cat([f.permute(0, 3, 1, 2).long() for f in frames], 1), case.k, case.s)   # [n, P, K]
    S = (cols.reshape(-1, K) @ ops.W.t()).view(n, oh * ow, cout).transpose(1, 2)                 # int64
    bias = ops.b.to(dtype).float()
    y = ((S.double() * 2.0 ** -ops.bw / 255).float() + bias[:, None]).to(dtype).view(n, cout, oh, ow)
    Sw = ops.G.transpose(0, 1).reshape(cout, -1) @ cols.reshape(-1, K)                          # int64 [cout, K]
    gw = (Sw.double() * 2.0 ** -ops.bg / 255).float().view(cout, -1, case.k, case.k)
    gb = (ops.G.sum((0, 2)).double() * 2.0 ** -ops.bg).float()
    return y, gw, gb


# ---------------------------------------------------------------- CPU check of the case table
def test_case_table_branches_and_operand_budget():
    """Every case's claimed launch branch is what vn_conv.cu's plan picks, every case's chosen operand ranges keep all
    partial sums exact in both regimes and every dtype (for a B200's SM count), and regime x01 puts bits into the fp32
    split's mid and lo terms where K is small."""
    assert len({c.id for c in CASES}) == len(CASES)
    for case in CASES:
        for dt, claim in case.claims.items():
            plan = _plan(case, dt)
            assert {key: plan[key] for key in claim} == claim, (case.id, DT_ID[dt], plan)
        for dt in case.dtypes:
            for regime in REGIMES[:1] if case.via == "store" else REGIMES:
                ops = _operands(case, dt, regime, B200_SMS)
                fwd, bwd = _budgets(case, dt, ops)
                assert fwd < 1 and bwd < 1, (case.id, DT_ID[dt], regime, fwd, bwd)
    ops = _operands(CASES[0], F32, "x01", B200_SMS)       # K = 48: 18 bits per weight
    hi, mid, lo = _terms(ops.W.float() * 2.0 ** -ops.bw, F32)
    assert ops.bw >= 17 and bool((mid != 0).any()) and bool((lo != 0).any())
    assert _value_bits(255, 32 * 8 * B200_SMS + 17, F32) == 1       # many_chunks at 0..255 still fits the budget


# ---------------------------------------------------------------- GPU side
def _sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


@pytest.fixture(scope="module")
def dw():
    scene = vn.scenes.make_maze_scene((10, 10), 0.25, 0, n_goals=2, frame_hw=(20, 28), planes=("rgb", "depth"))
    return vn.DeviceWorld(vn.compile_world([scene], vn.GYM_GRAPH), "cuda")


def _layer(case, W=None, b=None, seed=0):
    torch.manual_seed(seed)
    if case.set:
        layer = vn.nn.U8PlanesConv2d(case.planes, case.cout, case.k, stride=case.s).cuda()
    else:
        layer = vn.nn.U8Conv2d(case.planes[0], case.cout, case.k, stride=case.s).cuda()
    if W is not None:
        with torch.no_grad():
            layer.weight.copy_(W.view(layer.weight.shape))
            layer.bias.copy_(b)
    return layer


def _run_nn(layer, dtype, run, g):
    """(y, grad_weight, grad_bias) of `run()` under autocast to a 16-bit dtype (or none) and y.backward(g)."""
    with torch.autocast("cuda", dtype=BF16 if dtype == F32 else dtype, enabled=dtype != F32):
        y = run()
    assert y.dtype == dtype
    y.backward(g.view(y.shape))
    return y.detach().flatten(0, y.dim() - 4), layer.weight.grad, layer.bias.grad


def _guarded(count, dtype, shift=0, guard=1024):
    """(buffer, view) of `count` elements between NaN guards (fp32 / 16-bit) starting `shift` elements in."""
    buf = torch.full((guard + shift + count + guard,), float("nan"), dtype=dtype, device="cuda")
    return buf, buf[guard + shift:guard + shift + count]


def _assert_guarded(buf, view):
    start = view.storage_offset()
    assert bool(buf[:start].isnan().all()) and bool(buf[start + view.numel():].isnan().all()), "wrote outside"
    assert not bool(view.isnan().any()), "left an element unwritten"


def _run_abi(case, dtype, xs, W, b, g):
    """The forward and backward through the C ABI, every output and the scratch between guard bytes; 16-bit outputs
    and grad_out start 2 bytes past a 4-byte boundary."""
    lib = vn.lib.load()
    oh, ow, K = _geom(case)
    n, cout = xs[0].shape[0], case.cout
    shift = 0 if dtype == F32 else 1
    outb, out = _guarded(n * cout * oh * ow, dtype, shift)
    gob, go = _guarded(out.numel(), dtype, shift)
    go.copy_(g.flatten())
    gwb, gw = _guarded(W.numel(), F32)
    gbb, gb = _guarded(cout, F32)
    nbytes = lib.vn_conv_u8_wgrad_scratch_bytes(n, sum(case.planes), cout, case.k)
    pad = 4096
    scr = torch.full((pad + nbytes + pad,), 0x5A, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    srcs = [vn.nn._frames_of_batch(x) for x in xs]
    head = (vn.nn._frame_set(srcs), len(srcs)) if case.set else (C.byref(srcs[0]),)
    pre = "vn_conv_u8_planes_" if case.set else "vn_conv_u8_"
    lp = () if dtype == F32 else (LP[dtype],)
    sfx = "" if dtype == F32 else "_lp"
    vn.lib.check(getattr(lib, pre + "forward" + sfx)(*head, W.data_ptr(), b.data_ptr(), cout, case.k, case.s, *lp,
                                                     out.data_ptr(), stream))
    vn.lib.check(getattr(lib, pre + "backward" + sfx)(*head, go.data_ptr(), *lp, cout, case.k, case.s, gw.data_ptr(),
                                                      gb.data_ptr(), scr[pad:].data_ptr(), nbytes, stream))
    torch.cuda.synchronize()
    for buf, view in ((outb, out), (gwb, gw), (gbb, gb)):
        _assert_guarded(buf, view)
    assert bool((scr[:pad] == 0x5A).all()) and bool((scr[pad + nbytes:] == 0x5A).all()), "scratch overrun"
    return out.view(n, cout, oh, ow), gw.view(cout, -1, case.k, case.k), gb


def _same(got, want, what):
    got = got.cpu()
    if torch.equal(got, want):
        return
    bad = got != want
    idx = bad.nonzero()[0].tolist()
    raise AssertionError("%s: %d of %d elements differ, first at %s: %r != %r"
                         % (what, int(bad.sum()), want.numel(), idx, float(got[tuple(idx)]), float(want[tuple(idx)])))


def _run_exact(case, dtype, regime, dw=None):
    ops = _operands(case, dtype, regime, _sms())
    fwd, bwd = _budgets(case, dtype, ops)
    assert fwd < 1 and bwd < 1, (fwd, bwd)
    oh, ow, K = _geom(case)
    n, (h, w) = ops.n, case.hw
    W = (ops.W.float() * 2.0 ** -ops.bw).cuda()
    b = ops.b.cuda()
    g = (ops.G.float() * 2.0 ** -ops.bg).to(dtype).cuda()
    if case.via == "store":
        names = {3: "rgb", 1: "depth"}
        gen = torch.Generator(device="cuda").manual_seed(zlib.crc32(case.id.encode()))
        views = [torch.randint(0, dw.world.n_states, (5, 7), dtype=torch.int32, device="cuda", generator=gen).t()
                 for _ in case.planes]                                     # [7, 5] views of time-major storage
        sources = [(v, names[c]) for v, c in zip(views, case.planes)]
        frames = [dw.plane_view(p)[v.reshape(-1).long()].cpu() for v, p in sources]
        layer = _layer(case, W, b)
        if case.set:
            got = _run_nn(layer, dtype, lambda: layer.forward_states(dw, *sources), g)
        else:
            got = _run_nn(layer, dtype, lambda: layer.forward_states(dw, *sources[0]), g)
    else:
        xs = [raw.cuda().as_strided((n, h, w, c), (raw.shape[1], w * c, c, 1)) for raw, c in zip(ops.xs, case.planes)]
        frames = [x.cpu() for x in xs]
        if case.via == "abi":
            got = _run_abi(case, dtype, xs, W, b, g)
        else:
            layer = _layer(case, W, b)
            got = _run_nn(layer, dtype, lambda: layer(*xs) if case.set else layer(xs[0]), g)
    y, gw, gb = _exact_expected(case, dtype, ops, frames)
    _same(got[0], y, "forward")
    _same(got[1], gw, "weight gradient")
    _same(got[2], gb, "bias gradient")


@pytest.mark.gpu
@pytest.mark.parametrize("regime", REGIMES)
@pytest.mark.parametrize("dtype", ALL, ids=[DT_ID[d] for d in ALL])
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_exact_operands_bit_equal(case, dtype, regime, request):
    """Forward, weight gradient and bias gradient equal the exact result bit for bit (see the module docstring)."""
    if dtype not in case.dtypes:
        pytest.skip("%s runs in %s" % (case.id, ", ".join(DT_ID[d] for d in case.dtypes)))
    if case.via == "store" and regime != "x255":
        pytest.skip("store frames are whatever the scene renders: 0..255")
    _run_exact(case, dtype, regime, request.getfixturevalue("dw") if case.via == "store" else None)


@pytest.mark.gpu
@pytest.mark.parametrize("fresh", [False, True], ids=["sliced", "fresh"])
@pytest.mark.parametrize("dtype", ALL, ids=[DT_ID[d] for d in ALL])
@pytest.mark.parametrize("set_", [False, True], ids=["one", "set"])
def test_empty_batch_returns_zero_gradients_without_launching(set_, dtype, fresh):
    """n = 0: an empty output, zero gradients and no library launch, for a batch sliced to nothing and for a freshly
    allocated empty tensor (whose data pointer is null)."""
    case = next(c for c in CASES if c.id == ("f1_set_nt1" if set_ else "f1_one_nt1"))
    layer = _layer(case)
    h, w = case.hw
    if fresh:
        xs = [torch.empty((0, h, w, c), dtype=torch.uint8, device="cuda") for c in case.planes]
    else:
        xs = [torch.zeros((4, h, w, c), dtype=torch.uint8, device="cuda")[:0] for c in case.planes]
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        y, gw, gb = _run_nn(layer, dtype, lambda: layer(*xs), torch.zeros((0,), dtype=dtype, device="cuda"))
        torch.cuda.synchronize()
    assert y.shape[0] == 0
    assert torch.equal(gw, torch.zeros_like(gw)) and torch.equal(gb, torch.zeros_like(gb))
    launched = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    assert not any("vn_" in name for name in launched), launched


@pytest.mark.gpu
def test_every_kernel_instantiation_launches():
    """The F1 cases (forward and backward, three dtypes, one source and plane set) launch all 48 forward kernels, all 6
    weight-gradient kernels and the reduce kernel; each run is also checked bit for bit."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for case in CASES[:16]:
            for dt in ALL:
                _run_exact(case, dt, "x255")
    names = {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
    fwd = {m.groups() for nm in names for m in [re.search(r"vn_conv_u8_fwd_kernel<(\d+), ([\w]+), (\d+)>", nm)] if m}
    wgrad = {m.groups() for nm in names for m in [re.search(r"vn_conv_u8_wgrad_kernel<([\w]+), (\d+)>", nm)] if m}
    types = [T_NAME[d] for d in ALL]
    assert fwd == {(str(nt), t, s) for nt in range(1, 9) for t in types for s in ("1", "4")}, sorted(fwd)
    assert wgrad == {(t, s) for t in types for s in ("1", "4")}, sorted(wgrad)
    assert any("vn_conv_u8_wgrad_reduce_kernel" in nm for nm in names)


# ---------------------------------------------------------------- bound family
U = 2.0 ** -24
C_TC = 8    # the tensor cores' accumulation inside one k-step, the / 255 and the bias add
RAND = [c for c in CASES if c.id in ("f2_rgb174_cout40", "f3_c8_cout48", "w5_rgbd85_odd_p", "e_wide_30x52")] + [
    Case("rgb84_k8s4", (3,), False, 32, 8, 4, (84, 84), 64, "batch", ALL, {}, "the reference's layer at 84^2"),
    Case("multi_chunk", (3,), False, 16, 4, 2, (6, 6), "many_chunks", "batch", ALL, {},
         "CTAs sum several chunks (see w3_one_many_chunks), P = 4"),
]


def _ulp(v, dtype):
    fi = torch.finfo(dtype)
    return torch.exp2(torch.floor(torch.log2(v.abs())).clamp_min(math.log2(fi.tiny))) * fi.eps


def _rejects(wrong, ref, bound):
    return not bool(((wrong - ref).abs() <= bound).all())


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ALL, ids=[DT_ID[d] for d in ALL])
@pytest.mark.parametrize("case", RAND, ids=[c.id for c in RAND])
def test_random_values_within_error_bound(case, dtype):
    """Random frames, weights and grad_out: every element within its error bound of float64, and each bound rejects
    the operand rounded to bf16 (a lost split term), two input channels swapped, and the result shifted one pixel.

    A 16-bit forward's worst ratio is close to 1 by construction: its bound adds half an ulp of T for the one final
    rounding, which an output whose exact value lies near the midpoint of two T values nearly reaches (0.97 to 0.999 on
    a B200 at 1,000 W).  The printed accumulation part, the error beyond that half ulp over the summation bound, is
    the margin of the sums themselves."""
    n = _n(case, _sms())
    oh, ow, K = _geom(case)
    P, (h, w), cout, k = oh * ow, case.hw, case.cout, case.k
    gen = torch.Generator(device="cuda").manual_seed(zlib.crc32(case.id.encode()))
    xs = []
    for c in case.planes:
        pitch = (h * w * c + 15) // 16 * 16
        raw = torch.randint(0, 256, (n, pitch), dtype=torch.uint8, device="cuda", generator=gen)
        xs.append(raw.as_strided((n, h, w, c), (pitch, w * c, c, 1)))
    layer = _layer(case, seed=zlib.crc32(case.id.encode()))
    g = torch.randn((n, cout, oh, ow), device="cuda", generator=gen).to(dtype)
    y, gw, gb = _run_nn(layer, dtype, lambda: layer(*xs) if case.set else layer(xs[0]), g)

    wt = layer.weight.detach().to(dtype).double().view(cout, K)
    bt = layer.bias.detach().to(dtype).double()
    x64 = torch.cat([x.permute(0, 3, 1, 2).double() for x in xs], 1) / 255
    swapped = x64[:, [1, 0] + list(range(2, x64.shape[1]))]
    cols, cols_sw = _cols(x64, k, case.s), _cols(swapped, k, case.s)                # [n, P, K]

    def conv(cl, wm):
        return (cl @ wm.t()).transpose(1, 2).reshape(n, cout, oh, ow) + bt[:, None, None]

    y64 = conv(cols, wt)
    a = (cols @ wt.abs().t()).transpose(1, 2).reshape(n, cout, oh, ow) + bt.abs()[:, None, None]
    acc_bound = ((K + 15) // 16 + C_TC) * U * a
    half_ulp = 0 if dtype == F32 else 0.5 * torch.maximum(_ulp(y64, dtype), _ulp(y.double(), dtype))
    bound = acc_bound + half_ulp
    err = (y.double() - y64).abs()
    print("%s %s forward: worst |y - y64| / bound = %.3f, accumulation part %.3f"
          % (case.id, DT_ID[dtype], float((err / bound).max()), float(((err - half_ulp).clamp_min(0) / acc_bound).max())))
    assert bool((err <= bound).all()), float((err - bound).max())
    wrongs = {"swapped channels": conv(cols_sw, wt), "shifted pixel": y64.roll(1, -1)}
    if dtype != BF16:
        wrongs["bf16 weight"] = conv(cols, layer.weight.detach().bfloat16().double().view(cout, K))
    for what, wrong in wrongs.items():
        assert _rejects(wrong, y64, bound), what

    g64 = g.double().view(n, cout, P)
    gw64 = torch.einsum("ncp,npk->ck", g64, cols)
    aw = torch.einsum("ncp,npk->ck", g64.abs(), cols)
    steps = _cdiv(P, 16) + CHUNK + _cdiv(_cdiv(n, CHUNK), 32) + 5 + C_TC
    bound_w = steps * U * aw
    err_w = (gw.double().view(cout, K) - gw64).abs()
    gb64, bound_b = g64.sum((0, 2)), steps * U * g64.abs().sum((0, 2))
    err_b = (gb.double() - gb64).abs()
    print("%s %s backward: worst error / bound = %.3f (weight), %.3f (bias)"
          % (case.id, DT_ID[dtype], float((err_w / bound_w).max()), float((err_b / bound_b).max())))
    assert bool((err_w <= bound_w).all()), float((err_w - bound_w).max())
    assert bool((err_b <= bound_b).all()), float((err_b - bound_b).max())
    wrongs = {"swapped channels": torch.einsum("ncp,npk->ck", g64, cols_sw),
              "shifted pixel": gw64.view(cout, -1, k, k).roll(1, -1).reshape(cout, K)}
    if dtype != BF16:
        wrongs["bf16 grad_out"] = torch.einsum("ncp,npk->ck", g.bfloat16().double().view(n, cout, P), cols)
    for what, wrong in wrongs.items():
        assert _rejects(wrong, gw64, bound_w), what
