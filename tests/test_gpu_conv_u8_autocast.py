"""vn.nn.U8Conv2d under torch.autocast with fp16 / bf16: forward accuracy against float64 with the weight rounded like
autocast, the bitwise properties of the fp32 layer (two frame sources, halves, repeats, CUDA-graph replay) and the
fp32 path under a nested autocast(enabled=False), the weight / bias gradient from a 16-bit grad_out, non-finite
propagation for GradScaler, launches and synchronisation, guard bytes around every output of the 16-bit entry points,
and the update pass's peak memory."""
import ctypes as C
import importlib
import math
import os
import sys

import pytest

torch = pytest.importorskip("torch")
F = torch.nn.functional

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_gpu_conv_u8 import GEOM_IDS, GEOMS, _batch, _layer, _library_kernels, _rel, _thor  # noqa: E402

vn = importlib.import_module("a2cat-vn-pytorch_b200")

pytestmark = pytest.mark.gpu

DTYPES = [torch.float16, torch.bfloat16]
DTYPE_IDS = ["f16", "bf16"]
# plus one geometry with an odd number of output pixels: 41 x 41, so every other channel row of the 16-bit output and
# of grad_out starts on a 2-byte boundary
AC_GEOMS = GEOMS + [(3, 8, 3, 2, 84)]
AC_IDS = GEOM_IDS + ["odd_k3s2"]
LP = {torch.float16: vn.lib.DTYPE_F16, torch.bfloat16: vn.lib.DTYPE_BF16}


def _ulp(y64, dtype):
    """Spacing of `dtype` at |y64| (subnormal spacing below the smallest normal)."""
    fi = torch.finfo(dtype)
    e = torch.floor(torch.log2(y64.abs())).clamp_min(math.log2(fi.tiny))
    return torch.exp2(e) * fi.eps


@pytest.mark.parametrize("n", [1, 7, 4096])
@pytest.mark.parametrize("bias", [True, False])
@pytest.mark.parametrize("geom", AC_GEOMS, ids=AC_IDS)
@pytest.mark.parametrize("dtype", DTYPES, ids=DTYPE_IDS)
def test_forward_matches_float64(dtype, geom, bias, n):
    cin, cout, k, s, side = geom
    if side == 174 and n == 4096:
        n = 1024
    layer = _layer(cin, cout, k, s, bias, seed=n)
    x = _batch(n, side, cin, seed=n + 1)
    with torch.no_grad(), torch.autocast("cuda", dtype=dtype):
        y = layer(x)
        xf = x.permute(0, 3, 1, 2).float() / 255
        y_torch = F.conv2d(xf, layer.weight, layer.bias, s)
    torch.cuda.synchronize()
    assert y.dtype == dtype and y.shape == y_torch.shape
    w = layer.weight.detach().to(dtype).double()
    b = None if layer.bias is None else layer.bias.detach().to(dtype).double()
    x64 = x.permute(0, 3, 1, 2).double() / 255
    y64 = F.conv2d(x64, w, b, s)
    # Within one ulp of the exact value, up to the fp32 accumulation's own error: the k-step sums and the FADDs that join
    # them, (ksteps + 18) roundings of at most 2^-23 relative to the sum of |terms|.  That error only shows where the
    # sum cancels to far below its terms.
    ksteps = (cin * k * k + 15) // 16
    s_abs = F.conv2d(x64, w.abs(), None if b is None else b.abs(), s)
    err = (y.double() - y64).abs()
    bound = _ulp(y64, dtype) + (ksteps + 18) * 2.0 ** -23 * s_abs
    assert bool((err <= bound).all()), float((err - bound).max())
    exact = float((y == y64.to(dtype)).double().mean())
    assert exact >= 0.999, exact
    assert _rel(y, y64) <= _rel(y_torch, y64), (_rel(y, y64), _rel(y_torch, y64))


@pytest.fixture(scope="module")
def env():
    e = _thor()
    e.reset()
    yield e
    e.close()


@pytest.mark.parametrize("dtype", DTYPES, ids=DTYPE_IDS)
def test_batch_path_equals_store_path(env, dtype):
    layer = _layer(3, 32, 7, 4)
    for i in range(5):
        env.step(torch.full((env.num_envs,), i % 4, dtype=torch.int32, device="cuda"))
    with torch.no_grad(), torch.autocast("cuda", dtype=dtype):
        a = layer(env.obs_buf["rgb"])
        b = layer.forward_states(env.dw, env.obs_state)
    assert a.dtype == b.dtype == dtype and torch.equal(a, b)


@pytest.mark.parametrize("dtype", DTYPES, ids=DTYPE_IDS)
def test_batch_equals_its_halves_and_runs_repeat(dtype):
    layer = _layer(3, 32, 7, 4)
    x = _batch(1000, 84, 3, seed=9)
    with torch.no_grad(), torch.autocast("cuda", dtype=dtype):
        y = layer(x)
        halves = torch.cat([layer(x[:500]), layer(x[500:])])
        again = layer(x)
    assert torch.equal(y, halves) and torch.equal(y, again)


@pytest.mark.parametrize("dtype", DTYPES, ids=DTYPE_IDS)
def test_backward_repeats_bitwise(env, dtype):
    layer = _layer(3, 32, 7, 4)
    states = torch.randint(0, env.dw.world.n_states, (20, 300), dtype=torch.int32, device="cuda").t()
    go = torch.randn((300, 20, 32, 20, 20), device="cuda").to(dtype)
    grads = []
    for _ in range(2):
        layer.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=dtype):
            y = layer.forward_states(env.dw, states)
        y.backward(go)
        grads.append((y.detach(), layer.weight.grad.clone(), layer.bias.grad.clone()))
    assert grads[0][1].dtype == torch.float32
    assert all(torch.equal(a, b) for a, b in zip(*grads))


@pytest.mark.parametrize("dtype", DTYPES, ids=DTYPE_IDS)
def test_nested_disabled_autocast_is_the_fp32_layer(env, dtype):
    layer = _layer(3, 32, 7, 4)
    states = torch.randint(0, env.dw.world.n_states, (8, 50), dtype=torch.int32, device="cuda").t()
    go = torch.randn((50, 8, 32, 20, 20), device="cuda")
    y = layer.forward_states(env.dw, states)
    y.backward(go)
    plain = (y.detach(), layer.weight.grad.clone(), layer.bias.grad.clone())
    layer.zero_grad(set_to_none=True)
    with torch.autocast("cuda", dtype=dtype):
        with torch.autocast("cuda", enabled=False):
            y = layer.forward_states(env.dw, states)
    y.backward(go)
    assert y.dtype == torch.float32
    assert torch.equal(y, plain[0]) and torch.equal(layer.weight.grad, plain[1]) and torch.equal(layer.bias.grad, plain[2])


@pytest.mark.parametrize("geom", [g for g in AC_GEOMS if g[4] == 84], ids=[i for g, i in zip(AC_GEOMS, AC_IDS) if g[4] == 84])
@pytest.mark.parametrize("dtype", DTYPES, ids=DTYPE_IDS)
def test_weight_gradient_matches_float64(env, dtype, geom):
    cin, cout, k, s, _ = geom
    plane = "rgb" if cin == 3 else "depth"
    dw = env.dw
    g = torch.Generator(device="cuda").manual_seed(5)
    store_t = torch.randint(0, dw.world.n_states, (20, 410), dtype=torch.int32, device="cuda", generator=g)
    states = store_t.t()                                      # [410, 20] strided view of time-major storage: 8,200 frames
    layer = _layer(cin, cout, k, s, True, seed=1)
    with torch.autocast("cuda", dtype=dtype):
        y = layer.forward_states(dw, states, plane)
    assert y.dtype == dtype
    go = torch.randn(y.shape, device="cuda", generator=g).to(dtype)
    y.backward(go)
    assert layer.weight.grad.dtype == layer.bias.grad.dtype == torch.float32
    x = dw.plane_view(plane)[states.reshape(-1).long()]       # [N, H, W, C]
    w64 = layer.weight.detach().double().requires_grad_()
    b64 = layer.bias.detach().double().requires_grad_()
    F.conv2d(x.permute(0, 3, 1, 2).double() / 255, w64, b64, s).backward(go.double().flatten(0, 1))
    w32 = layer.weight.detach().clone().requires_grad_()
    b32 = layer.bias.detach().clone().requires_grad_()
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        F.conv2d(x.permute(0, 3, 1, 2).float() / 255, w32, b32, s).backward(go.float().flatten(0, 1))
    finally:
        torch.backends.cudnn.allow_tf32 = prev
    for got, ref, f32 in ((layer.weight.grad, w64.grad, w32.grad), (layer.bias.grad, b64.grad, b32.grad)):
        e, e_torch = _rel(got, ref), _rel(f32, ref)
        assert e <= 1e-5 and e <= 4 * e_torch + 1e-7, (e, e_torch)


@pytest.mark.parametrize("dtype", DTYPES, ids=DTYPE_IDS)
def test_non_finite_grad_out_reaches_its_channel_and_grad_scaler(dtype):
    layer = _layer(3, 32, 7, 4)
    x = _batch(64, 84, 3, seed=4)
    go = (torch.randn((64, 32, 20, 20), device="cuda") * 0.01).to(dtype)
    bad = go.clone()
    c = 5
    bad[17, c, 3, 11] = float("inf")
    grads = []
    for g in (go, bad):
        layer.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=dtype):
            y = layer(x)
        y.backward(g)
        grads.append((layer.weight.grad.clone(), layer.bias.grad.clone()))
    (gw, gb), (bw, bb) = grads
    assert not bool(torch.isfinite(bw[c]).any()) and not bool(torch.isfinite(bb[c]))
    others = torch.arange(32, device="cuda") != c
    assert bool(torch.isfinite(bw[others]).all()) and bool(torch.isfinite(bb[others]).all())
    assert torch.equal(bw[others], gw[others]) and torch.equal(bb[others], gb[others])

    opt = torch.optim.SGD(layer.parameters(), lr=0.1)
    scaler = torch.amp.GradScaler("cuda", init_scale=4.0)
    for g, moves in ((bad, False), (go, True)):
        before = layer.weight.detach().clone()
        opt.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=dtype):
            y = layer(x)
        scaler.scale(y).backward(g)
        scaler.step(opt)
        scaler.update()
        assert (not torch.equal(layer.weight.detach(), before)) == moves


@pytest.mark.parametrize("dtype", DTYPES, ids=DTYPE_IDS)
def test_launches_and_no_synchronisation(env, dtype):
    layer = _layer(3, 32, 7, 4)
    states = torch.randint(0, env.dw.world.n_states, (20, 256), dtype=torch.int32, device="cuda").t()
    go = torch.randn((256, 20, 32, 20, 20), device="cuda").to(dtype)
    with torch.autocast("cuda", dtype=dtype):
        y = layer.forward_states(env.dw, states)
    y.backward(go)                                        # warm-up (library load, shared-memory attributes)
    layer.zero_grad(set_to_none=True)
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.set_sync_debug_mode("error")
    try:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            with torch.autocast("cuda", dtype=dtype):
                y = layer.forward_states(env.dw, states)
        fwd = _library_kernels(prof.events())
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            y.backward(go)
        bwd = _library_kernels(prof.events())
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert len(fwd) == 1 and "vn_conv_u8_fwd_kernel" in fwd[0], fwd
    assert len(bwd) == 2 and "vn_conv_u8_wgrad_kernel" in bwd[0] and "vn_conv_u8_wgrad_reduce_kernel" in bwd[1], bwd


@pytest.mark.parametrize("dtype", DTYPES, ids=DTYPE_IDS)
def test_cuda_graph_replay_matches_eager(env, dtype):
    layer = _layer(3, 32, 7, 4)
    states = torch.randint(0, env.dw.world.n_states, (20, 128), dtype=torch.int32, device="cuda").t()
    go = torch.randn((128, 20, 32, 20, 20), device="cuda").to(dtype)

    def run():
        with torch.autocast("cuda", dtype=dtype):
            y = layer.forward_states(env.dw, states)
        y.backward(go)
        return y

    y = run()
    eager = (y.detach().clone(), layer.weight.grad.clone(), layer.bias.grad.clone())
    del y
    layer.zero_grad(set_to_none=True)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            layer.zero_grad(set_to_none=True)
            run()
        layer.zero_grad(set_to_none=True)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        gy = run()
    graph.replay()
    torch.cuda.synchronize()
    assert gy.dtype == dtype
    assert torch.equal(gy, eager[0]) and torch.equal(layer.weight.grad, eager[1]) and torch.equal(layer.bias.grad, eager[2])


@pytest.mark.parametrize("geom", AC_GEOMS, ids=AC_IDS)
@pytest.mark.parametrize("dtype", DTYPES, ids=DTYPE_IDS)
def test_outputs_stay_inside_their_buffers(dtype, geom):
    cin, cout, k, s, side = geom
    lib = vn.lib.load()
    n = 37
    x = _batch(n, side, cin, seed=2)
    oh = (side - k) // s + 1
    guard = 4096
    canary = -4096.0                  # exact in fp16, bf16 and fp32, and no output of these layers

    def guarded(count, dt, shift=0):
        """A canary-filled buffer and the view of `count` elements inside it, `shift` elements past the guard."""
        buf = torch.full((guard + shift + count + guard,), canary, dtype=dt, device="cuda")
        return buf, buf[guard + shift:guard + shift + count], guard + shift

    w = torch.randn(cout * cin * k * k, device="cuda") * 0.05
    b = torch.randn(cout, device="cuda")
    # the 16-bit output starts 2 bytes past a 4-byte boundary: 2-byte alignment is what the entry points require
    outb, out, out0 = guarded(n * cout * oh * oh, dtype, shift=1)
    src = vn.lib.U8Frames(x.data_ptr(), x.stride(0), None, 0, 0, n, 1, side, side, cin, 0)
    stream = torch.cuda.current_stream().cuda_stream
    vn.lib.check(lib.vn_conv_u8_forward_lp(C.byref(src), w.data_ptr(), b.data_ptr(), cout, k, s, LP[dtype],
                                           out.data_ptr(), stream))
    go_b, go, _ = guarded(n * cout * oh * oh, dtype, shift=1)
    go.copy_(torch.randn(go.numel(), device="cuda"))
    gwb, gw, gw0 = guarded(w.numel(), torch.float32)
    gbb, gb, gb0 = guarded(cout, torch.float32)
    nbytes = lib.vn_conv_u8_wgrad_scratch_bytes(n, cin, cout, k)
    scr = torch.full((guard * 4 + nbytes + guard * 4,), 0x5A, dtype=torch.uint8, device="cuda")
    vn.lib.check(lib.vn_conv_u8_backward_lp(C.byref(src), go.data_ptr(), LP[dtype], cout, k, s, gw.data_ptr(),
                                            gb.data_ptr(), scr[guard * 4:].data_ptr(), nbytes, stream))
    torch.cuda.synchronize()
    for buf, start, count in ((outb, out0, out.numel()), (gwb, gw0, gw.numel()), (gbb, gb0, gb.numel())):
        assert bool((buf[:start] == canary).all()) and bool((buf[start + count:] == canary).all())
        assert not bool((buf[start:start + count] == canary).any())
    assert bool((scr[:guard * 4] == 0x5A).all()) and bool((scr[guard * 4 + nbytes:] == 0x5A).all())


@pytest.mark.parametrize("dtype", DTYPES, ids=DTYPE_IDS)
def test_update_pass_peak_memory(env, dtype):
    """(3 -> 32, k7, s4) over 81,920 frames: the 16-bit output, the scratch and at most 1 MB more above the inputs."""
    layer = _layer(3, 32, 7, 4)
    states = torch.randint(0, env.dw.world.n_states, (20, 4096), dtype=torch.int32, device="cuda").t()
    go = torch.randn((4096, 20, 32, 20, 20), device="cuda", dtype=dtype)
    n = states.numel()
    out_bytes = n * 32 * 20 * 20 * 2
    scratch = vn.lib.load().vn_conv_u8_wgrad_scratch_bytes(n, 3, 32, 7)

    def update():
        layer.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=dtype):
            y = layer.forward_states(env.dw, states)
        y.backward(go)

    update()                                              # warm-up
    layer.zero_grad(set_to_none=True)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    update()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    assert peak <= out_bytes + scratch + (1 << 20), (peak, out_bytes, scratch)
