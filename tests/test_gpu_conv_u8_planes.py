"""vn.nn.U8PlanesConv2d on the GPU: forward and weight / bias gradient against float64 for plane sets of up to 8 channels,
bitwise equality with U8Conv2d for one plane, the batch and store paths, halves and repeats, autocast accuracy and
GradScaler, an RGB-D policy's gradients, launches and synchronisation, CUDA-graph replay, and guard bytes around every
output of the plane-set entry points."""
import ctypes as C
import importlib
import math
import os
import sys

import pytest

torch = pytest.importorskip("torch")
F = torch.nn.functional

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_gpu_conv_u8 import _Policy, _batch, _check, _library_kernels, _rel, _thor  # noqa: E402

vn = importlib.import_module("a2cat-vn-pytorch_b200")

pytestmark = pytest.mark.gpu

PLANES = [(3, 1), (3, 3), (1, 1), (3, 1, 3, 1), (3, 3, 1, 1)]
PLANE_IDS = ["rgbd", "obs_goal", "depth2", "rgbd2", "c8"]
DTYPES = [torch.float16, torch.bfloat16]
DTYPE_IDS = ["f16", "bf16"]
LP = {torch.float16: vn.lib.DTYPE_F16, torch.bfloat16: vn.lib.DTYPE_BF16}


def _layer(planes, cout=32, k=7, s=4, bias=True, seed=0):
    torch.manual_seed(seed)
    return vn.nn.U8PlanesConv2d(planes, cout, k, stride=s, bias=bias).cuda()


def _frames(n, side, planes, seed):
    return [_batch(n, side, c, seed=seed + 101 * i) for i, c in enumerate(planes)]


def _cat(xs, dtype=torch.float64):
    return torch.cat([x.permute(0, 3, 1, 2).to(dtype) for x in xs], 1) / 255


def _f64(xs, layer):
    return F.conv2d(_cat(xs), layer.weight.detach().double(),
                    None if layer.bias is None else layer.bias.detach().double(), layer.stride)


def _f32(xs, layer):
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        return F.conv2d(_cat(xs, torch.float32), layer.weight.detach(),
                        None if layer.bias is None else layer.bias.detach(), layer.stride)
    finally:
        torch.backends.cudnn.allow_tf32 = prev


@pytest.mark.parametrize("n", [1, 7, 4096])
@pytest.mark.parametrize("bias", [True, False])
@pytest.mark.parametrize("planes", PLANES, ids=PLANE_IDS)
def test_forward_matches_float64(planes, bias, n):
    layer = _layer(planes, bias=bias, seed=n)
    xs = _frames(n, 84, planes, seed=n + 1)
    with torch.no_grad():
        y = layer(*xs)
    y64 = _f64(xs, layer)
    assert y.shape == y64.shape and y.dtype == torch.float32
    _check(_rel(y, y64), _rel(_f32(xs, layer), y64))


# (planes, cout, k, stride, side): the widest layer on the widest set, and RGB-D on the reference's native frames
@pytest.mark.parametrize("geom", [((3, 3, 1, 1), 64, 8, 4, 84), ((3, 3, 1, 1), 64, 8, 1, 84), ((3, 1), 32, 7, 4, 174)],
                         ids=["c8_cout64_k8s4", "c8_cout64_k8s1", "native174_rgbd"])
def test_forward_wide_and_native(geom):
    planes, cout, k, s, side = geom
    layer = _layer(planes, cout, k, s, seed=3)
    xs = _frames(256, side, planes, seed=4)
    with torch.no_grad():
        y = layer(*xs)
    y64 = _f64(xs, layer)
    _check(_rel(y, y64), _rel(_f32(xs, layer), y64))


@pytest.fixture(scope="module")
def env():
    e = _thor()
    e.reset()
    yield e
    e.close()


@pytest.fixture(scope="module")
def buf(env):
    """A real rollout of 20 steps: states and goals time-major [21, 64]."""
    b = vn.rollout.RolloutBuffer(env.dw, env.num_envs, 20)
    b.start(env)
    g = torch.Generator(device="cuda").manual_seed(7)
    for _ in range(20):
        a = torch.randint(0, 4, (env.num_envs,), dtype=torch.int32, device="cuda", generator=g)
        env.step(a)
        b.insert(env, a)
    return b


def _grad_refs(layer, xs, go):
    """float64 and TF32-off float32 weight / bias gradients of F.conv2d on the concatenated frames."""
    out = []
    for dt in (torch.float64, torch.float32):
        w = layer.weight.detach().to(dt).requires_grad_()
        b = layer.bias.detach().to(dt).requires_grad_()
        prev = torch.backends.cudnn.allow_tf32
        torch.backends.cudnn.allow_tf32 = False
        try:
            F.conv2d(_cat(xs, dt), w, b, layer.stride).backward(go.to(dt))
        finally:
            torch.backends.cudnn.allow_tf32 = prev
        out.append((w.grad, b.grad))
    return out


@pytest.mark.parametrize("geom", [((3, 3), 32, 7, 4), ((3, 1), 16, 8, 4), ((3, 3, 1, 1), 64, 8, 4)],
                         ids=["obs_goal", "rgbd_k8", "c8_cout64"])
def test_weight_gradient_matches_float64(env, buf, geom):
    planes, cout, k, s = geom
    dw = env.dw
    names = {3: "rgb", 1: "depth"}
    views = [buf.states[:-1].t(), buf.goals[:-1].t()]       # [64, 20] strided views of time-major storage
    sources = [(views[i % 2], names[c]) for i, c in enumerate(planes)]
    layer = _layer(planes, cout, k, s, seed=1)
    y = layer.forward_states(dw, *sources)
    g = torch.Generator(device="cuda").manual_seed(5)
    go = torch.randn(y.shape, device="cuda", generator=g)
    y.backward(go)
    xs = [dw.plane_view(p)[st.reshape(-1).long()] for st, p in sources]
    (w64, b64), (w32, b32) = _grad_refs(layer, xs, go.flatten(0, 1))
    _check(_rel(layer.weight.grad, w64), _rel(w32, w64))
    _check(_rel(layer.bias.grad, b64), _rel(b32, b64))


@pytest.mark.parametrize("dtype", [None] + DTYPES, ids=["f32"] + DTYPE_IDS)
@pytest.mark.parametrize("plane", ["rgb", "depth"])
def test_one_plane_equals_u8conv2d(env, plane, dtype):
    c = 3 if plane == "rgb" else 1
    one = _layer((c,), seed=2)
    ref = vn.nn.U8Conv2d(c, 32, 7, stride=4).cuda()
    ref.load_state_dict(one.state_dict())
    states = torch.randint(0, env.dw.world.n_states, (20, 100), dtype=torch.int32, device="cuda").t()
    go = torch.randn((100, 20, 32, 20, 20), device="cuda")
    res = []
    for layer, run in ((one, lambda: one.forward_states(env.dw, (states, plane))),
                       (ref, lambda: ref.forward_states(env.dw, states, plane))):
        with torch.autocast("cuda", dtype=dtype or torch.float16, enabled=dtype is not None):
            y = run()
        y.backward(go if dtype is None else go.to(dtype))
        res.append((y.detach(), layer.weight.grad, layer.bias.grad))
    assert all(torch.equal(a, b) for a, b in zip(*res))
    x = env.obs_buf[plane]
    with torch.no_grad(), torch.autocast("cuda", dtype=dtype or torch.float16, enabled=dtype is not None):
        assert torch.equal(one(x), ref(x))


def test_batch_path_equals_store_path(env):
    layer = _layer((3, 1))
    for i in range(5):
        env.step(torch.full((env.num_envs,), i % 4, dtype=torch.int32, device="cuda"))
    with torch.no_grad():
        a = layer(env.obs_buf["rgb"], env.obs_buf["depth"])
        b = layer.forward_states(env.dw, (env.obs_state, "rgb"), (env.obs_state, "depth"))
    assert torch.equal(a, b)


def test_batch_equals_its_halves_and_runs_repeat():
    layer = _layer((3, 3, 1, 1), 64, 8, 4)
    xs = _frames(1000, 84, (3, 3, 1, 1), seed=9)
    with torch.no_grad():
        y = layer(*xs)
        halves = torch.cat([layer(*[x[:500] for x in xs]), layer(*[x[500:] for x in xs])])
        again = layer(*xs)
    assert torch.equal(y, halves) and torch.equal(y, again)


@pytest.mark.parametrize("planes", [(3, 3), (3, 3, 1, 1)], ids=["obs_goal", "c8"])
def test_backward_repeats_bitwise(env, buf, planes):
    layer = _layer(planes, 64, 8, 4)
    names = {3: "rgb", 1: "depth"}
    sources = [((buf.states if i % 2 == 0 else buf.goals)[:-1].t(), names[c]) for i, c in enumerate(planes)]
    go = torch.randn((64, 20, 64, 20, 20), device="cuda")
    grads = []
    for _ in range(2):
        layer.zero_grad(set_to_none=True)
        layer.forward_states(env.dw, *sources).backward(go)
        grads.append((layer.weight.grad.clone(), layer.bias.grad.clone()))
    assert all(torch.equal(a, b) for a, b in zip(*grads))


def _ulp(y64, dtype):
    fi = torch.finfo(dtype)
    e = torch.floor(torch.log2(y64.abs())).clamp_min(math.log2(fi.tiny))
    return torch.exp2(e) * fi.eps


@pytest.mark.parametrize("planes", [(3, 1), (3, 3, 1, 1)], ids=["rgbd", "c8"])
@pytest.mark.parametrize("dtype", DTYPES, ids=DTYPE_IDS)
def test_autocast_forward_matches_float64(dtype, planes):
    layer = _layer(planes, 64, 8, 4, seed=11)
    xs = _frames(512, 84, planes, seed=12)
    with torch.no_grad(), torch.autocast("cuda", dtype=dtype):
        y = layer(*xs)
    assert y.dtype == dtype
    w = layer.weight.detach().to(dtype).double()
    b = layer.bias.detach().to(dtype).double()
    x64 = _cat(xs)
    y64 = F.conv2d(x64, w, b, 4)
    ksteps = (sum(planes) * 64 + 15) // 16
    s_abs = F.conv2d(x64, w.abs(), b.abs(), 4)
    err = (y.double() - y64).abs()
    bound = _ulp(y64, dtype) + (ksteps + 18) * 2.0 ** -23 * s_abs
    assert bool((err <= bound).all()), float((err - bound).max())
    assert float((y == y64.to(dtype)).double().mean()) >= 0.999


@pytest.mark.parametrize("dtype", DTYPES, ids=DTYPE_IDS)
def test_autocast_weight_gradient_and_grad_scaler(env, buf, dtype):
    layer = _layer((3, 1), seed=13)
    sources = [(buf.states[:-1].t(), "rgb"), (buf.states[:-1].t(), "depth")]
    with torch.autocast("cuda", dtype=dtype):
        y = layer.forward_states(env.dw, *sources)
    assert y.dtype == dtype
    go = torch.randn(y.shape, device="cuda").to(dtype)
    y.backward(go)
    assert layer.weight.grad.dtype == torch.float32
    xs = [env.dw.plane_view(p)[st.reshape(-1).long()] for st, p in sources]
    (w64, b64), (w32, b32) = _grad_refs(layer, xs, go.float().flatten(0, 1))
    _check(_rel(layer.weight.grad, w64), _rel(w32, w64))
    _check(_rel(layer.bias.grad, b64), _rel(b32, b64))

    x = [_batch(64, 84, 3, seed=14), _batch(64, 84, 1, seed=15)]
    good = (torch.randn((64, 32, 20, 20), device="cuda") * 0.01).to(dtype)
    bad = good.clone()
    bad[17, 5, 3, 11] = float("inf")
    opt = torch.optim.SGD(layer.parameters(), lr=0.1)
    scaler = torch.amp.GradScaler("cuda", init_scale=4.0)
    for g, moves in ((bad, False), (good, True)):
        before = layer.weight.detach().clone()
        opt.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=dtype):
            y = layer(*x)
        scaler.scale(y).backward(g)
        if not moves:
            assert not bool(torch.isfinite(layer.weight.grad[5]).any())
        scaler.step(opt)
        scaler.update()
        assert (not torch.equal(layer.weight.detach(), before)) == moves


def test_drop_in_rgbd_policy_gradients(env, monkeypatch):
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)
    torch.manual_seed(0)
    ref = _Policy(torch.nn.Conv2d(4, 16, 8, stride=4)).cuda().double()
    fused = _Policy(torch.nn.Conv2d(4, 16, 8, stride=4)).cuda()
    fused.load_state_dict({k: v.float() for k, v in ref.state_dict().items()})
    fused.c1 = vn.nn.U8PlanesConv2d.from_conv2d(fused.c1, (3, 1))
    assert isinstance(fused.c1, torch.nn.Conv2d) and set(fused.state_dict()) == set(ref.state_dict())
    states = torch.randint(0, env.dw.world.n_states, (5, 64), dtype=torch.int32, device="cuda").t()
    target = torch.randn(64 * 5, 4, device="cuda", dtype=torch.float64)
    x = torch.cat([vn.rollout.policy_input(env.dw, states.contiguous(), p) for p in ("rgb", "depth")], 2)
    (ref.trunk(ref.c1(x.flatten(0, 1).double())) * target).sum().backward()
    y = fused.c1.forward_states(env.dw, (states, "rgb"), (states, "depth")).flatten(0, 1)
    (fused.trunk(y) * target.float()).sum().backward()
    for (name, p), (_, q) in zip(fused.named_parameters(), ref.named_parameters()):
        e = float((p.grad.double() - q.grad).abs().max() / q.grad.abs().max())
        assert e < 1e-4, (name, e)


@pytest.mark.parametrize("dtype", [None] + DTYPES, ids=["f32"] + DTYPE_IDS)
def test_launches_and_no_synchronisation(env, buf, dtype):
    layer = _layer((3, 3), 64, 8, 4)
    sources = [(buf.states[:-1].t(), "rgb"), (buf.goals[:-1].t(), "rgb")]
    go = torch.randn((64, 20, 64, 20, 20), device="cuda").to(dtype or torch.float32)

    def fwd():
        with torch.autocast("cuda", dtype=dtype or torch.float16, enabled=dtype is not None):
            return layer.forward_states(env.dw, *sources)

    fwd().backward(go)                                     # warm-up (library load, shared-memory attributes)
    layer.zero_grad(set_to_none=True)
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.set_sync_debug_mode("error")
    try:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            y = fwd()
        f = _library_kernels(prof.events())
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            y.backward(go)
        b = _library_kernels(prof.events())
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert len(f) == 1 and "vn_conv_u8_fwd_kernel" in f[0], f
    assert len(b) == 2 and "vn_conv_u8_wgrad_kernel" in b[0] and "vn_conv_u8_wgrad_reduce_kernel" in b[1], b


def test_cuda_graph_replay_matches_eager(env, buf):
    layer = _layer((3, 1, 3, 1), 64, 8, 4)
    sources = [(buf.states[:-1].t(), "rgb"), (buf.states[:-1].t(), "depth"), (buf.goals[:-1].t(), "rgb"),
               (buf.goals[:-1].t(), "depth")]
    go = torch.randn((64, 20, 64, 20, 20), device="cuda")
    y = layer.forward_states(env.dw, *sources)
    y.backward(go)
    eager = (y.detach().clone(), layer.weight.grad.clone(), layer.bias.grad.clone())
    del y
    layer.zero_grad(set_to_none=True)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            layer.zero_grad(set_to_none=True)
            layer.forward_states(env.dw, *sources).backward(go)
        layer.zero_grad(set_to_none=True)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        gy = layer.forward_states(env.dw, *sources)
        gy.backward(go)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(gy, eager[0]) and torch.equal(layer.weight.grad, eager[1]) and torch.equal(layer.bias.grad, eager[2])


@pytest.mark.parametrize("dtype", [None] + DTYPES, ids=["f32"] + DTYPE_IDS)
@pytest.mark.parametrize("geom", [((3, 1), 32, 7, 4, 84), ((3, 3, 1, 1), 64, 8, 4, 84), ((3, 1), 32, 7, 4, 174),
                                  ((1, 3), 8, 3, 2, 84)], ids=["rgbd", "c8_cout64", "native174_rgbd", "odd_k3s2"])
def test_outputs_stay_inside_their_buffers(geom, dtype):
    planes, cout, k, s, side = geom
    lib = vn.lib.load()
    n = 37
    xs = _frames(n, side, planes, seed=2)
    cin = sum(planes)
    oh = (side - k) // s + 1
    guard = 4096
    canary = -4096.0                  # exact in fp16, bf16 and fp32, and no output of these layers
    odt = dtype or torch.float32
    shift = 0 if dtype is None else 1   # 16-bit outputs start 2 bytes past a 4-byte boundary

    def guarded(count, dt, sh=0):
        buf = torch.full((guard + sh + count + guard,), canary, dtype=dt, device="cuda")
        return buf, buf[guard + sh:guard + sh + count], guard + sh

    w = torch.randn(cout * cin * k * k, device="cuda") * 0.05
    b = torch.randn(cout, device="cuda")
    srcs = vn.nn._frame_set([vn.nn._frames_of_batch(x) for x in xs])
    stream = torch.cuda.current_stream().cuda_stream
    outb, out, out0 = guarded(n * cout * oh * oh, odt, shift)
    go_b, go, _ = guarded(n * cout * oh * oh, odt, shift)
    go.copy_(torch.randn(go.numel(), device="cuda"))
    gwb, gw, gw0 = guarded(w.numel(), torch.float32)
    gbb, gb, gb0 = guarded(cout, torch.float32)
    nbytes = lib.vn_conv_u8_wgrad_scratch_bytes(n, cin, cout, k)
    scr = torch.full((guard * 4 + nbytes + guard * 4,), 0x5A, dtype=torch.uint8, device="cuda")
    if dtype is None:
        vn.lib.check(lib.vn_conv_u8_planes_forward(srcs, len(planes), w.data_ptr(), b.data_ptr(), cout, k, s,
                                                   out.data_ptr(), stream))
        vn.lib.check(lib.vn_conv_u8_planes_backward(srcs, len(planes), go.data_ptr(), cout, k, s, gw.data_ptr(),
                                                    gb.data_ptr(), scr[guard * 4:].data_ptr(), nbytes, stream))
    else:
        vn.lib.check(lib.vn_conv_u8_planes_forward_lp(srcs, len(planes), w.data_ptr(), b.data_ptr(), cout, k, s,
                                                      LP[dtype], out.data_ptr(), stream))
        vn.lib.check(lib.vn_conv_u8_planes_backward_lp(srcs, len(planes), go.data_ptr(), LP[dtype], cout, k, s,
                                                       gw.data_ptr(), gb.data_ptr(), scr[guard * 4:].data_ptr(),
                                                       nbytes, stream))
    torch.cuda.synchronize()
    for bf, start, count in ((outb, out0, out.numel()), (gwb, gw0, gw.numel()), (gbb, gb0, gb.numel())):
        assert bool((bf[:start] == canary).all()) and bool((bf[start + count:] == canary).all())
        assert not bool((bf[start:start + count] == canary).any())
    assert bool((scr[:guard * 4] == 0x5A).all()) and bool((scr[guard * 4 + nbytes:] == 0x5A).all())


def test_rejects_unsupported_layers_and_inputs(env):
    for kw in (dict(plane_channels=()), dict(plane_channels=(3, 1, 1, 1, 1)), dict(plane_channels=(2, 1)),
               dict(plane_channels=(3, 3, 3)), dict(padding=1), dict(kernel_size=9), dict(out_channels=12)):
        args = dict(plane_channels=(3, 1), out_channels=32, kernel_size=7, stride=4)
        args.update(kw)
        with pytest.raises(ValueError):
            vn.nn.U8PlanesConv2d(**args)
    with pytest.raises(ValueError):
        vn.nn.U8PlanesConv2d.from_conv2d(torch.nn.Conv2d(3, 32, 7, stride=4), (3, 1))
    layer = _layer((3, 1))
    rgb, depth = env.obs_buf["rgb"], env.obs_buf["depth"]
    with pytest.raises(TypeError):
        layer(rgb.float(), depth)
    with pytest.raises(TypeError):
        layer(rgb)
    with pytest.raises(ValueError):
        layer(depth, rgb)
    with pytest.raises(ValueError):
        layer(rgb, depth[:10])
    with pytest.raises(ValueError):
        layer.forward_states(env.dw, (env.obs_state, "depth"), (env.obs_state, "rgb"))
    with pytest.raises(ValueError):
        layer.forward_states(env.dw, (env.obs_state, "rgb"), (env.obs_state[:10], "depth"))
